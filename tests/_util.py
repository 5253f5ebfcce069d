"""Shared helpers for the parity tests (test infrastructure)."""
from __future__ import annotations

import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

if os.path.join(ROOT, "oracle") not in sys.path:
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
import synth  # noqa: E402  (oracle/synth.py: seeded scenes, cameras, the caller-preamble restatement)


def ref_module():
    """Oracle-A: the reference extension built in place under oracle/_ref (GPU only)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import build_ref
    return build_ref.load()


def ref_available() -> bool:
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import build_ref
    return build_ref.is_built()


def _align(off: int, a: int = 128) -> int:
    return (off + a - 1) // a * a


def parse_ref_buffers(P: int, W: int, H: int, R: int, geom: torch.Tensor, binning: torch.Tensor, img: torch.Tensor):
    """Unpack the reference's three opaque byte buffers with its `obtain` arithmetic
    (rasterizer_impl.h:21-27, rasterizer_impl.cu:155-194).  Only the arrays in front of the
    CUB-sized temp regions are addressable without knowing CUB's temp size -- enough for the gates."""
    out = {}
    g = geom.cpu().numpy()
    base = geom.data_ptr()
    off = _align(base) - base
    out["depths"] = g[off:off + 4 * P].view(np.float32).copy(); off += 4 * P
    off = _align(base + off) - base; off += 3 * P                       # clamped bool[3P]
    off = _align(base + off) - base; off += 4 * P                       # internal_radii
    off = _align(base + off) - base
    out["means2D"] = g[off:off + 8 * P].view(np.float32).reshape(P, 2).copy(); off += 8 * P
    off = _align(base + off) - base; off += 24 * P                      # cov3D
    off = _align(base + off) - base
    out["conic_opacity"] = g[off:off + 16 * P].view(np.float32).reshape(P, 4).copy(); off += 16 * P
    off = _align(base + off) - base; off += 12 * P                      # rgb 3P
    off = _align(base + off) - base
    out["tiles_touched"] = g[off:off + 4 * P].view(np.uint32).copy()

    b = binning.cpu().numpy()
    base = binning.data_ptr()
    off = _align(base) - base
    out["point_list"] = b[off:off + 4 * R].view(np.uint32).copy(); off += 4 * R
    off = _align(base + off) - base; off += 4 * R                       # point_list_unsorted
    off = _align(base + off) - base
    out["keys"] = b[off:off + 8 * R].view(np.uint64).copy(); off += 8 * R

    i = img.cpu().numpy()
    base = img.data_ptr()
    N = W * H
    off = _align(base) - base
    out["final_T"] = i[off:off + 4 * N].view(np.float32).copy(); off += 4 * N
    off = _align(base + off) - base
    out["n_contrib"] = i[off:off + 4 * N].view(np.uint32).copy(); off += 4 * N
    off = _align(base + off) - base
    T = ((W + 15) // 16) * ((H + 15) // 16)
    out["ranges"] = i[off:off + 8 * T].view(np.uint32).reshape(T, 2).copy()
    return out


def settings_tuple(mod, s: dict):
    return mod.GaussianRasterizationSettings(
        image_height=s["image_height"], image_width=s["image_width"], tanfovx=s["tanfovx"], tanfovy=s["tanfovy"],
        bg=s["bg"], scale_modifier=s["scale_modifier"], viewmatrix=s["viewmatrix"], projmatrix=s["projmatrix"],
        sh_degree=s["sh_degree"], campos=s["campos"], prefiltered=s["prefiltered"], debug=s["debug"])


def native_args(inp: dict, empty_device=None):
    """The 21 positional args of `_C.rasterize_gaussians` (reference __init__.py:63-85)."""
    kw, s = inp["kwargs"], inp["settings"]
    e = torch.Tensor([])
    g = lambda k: e if kw[k] is None else kw[k]  # noqa: E731
    return (s["bg"], kw["means3D"], kw["means2D"], g("colors_precomp"), kw["opacities"], g("scales"), g("rotations"),
            s["scale_modifier"], g("cov3D_precomp"), g("conic_precomp"), s["viewmatrix"], s["projmatrix"],
            s["tanfovx"], s["tanfovy"], s["image_height"], s["image_width"], e, s["sh_degree"], s["campos"],
            s["prefiltered"], s["debug"])


def backward_args(inp: dict, radii, dL, geom, R, binning, img):
    kw, s = inp["kwargs"], inp["settings"]
    e = torch.Tensor([])
    g = lambda k: e if kw[k] is None else kw[k]  # noqa: E731
    return (s["bg"], kw["means3D"], radii, g("colors_precomp"), g("scales"), g("rotations"), s["scale_modifier"],
            g("cov3D_precomp"), g("conic_precomp"), s["viewmatrix"], s["projmatrix"], s["tanfovx"], s["tanfovy"],
            dL, e, s["sh_degree"], s["campos"], geom, R, binning, img, s["debug"])


GRAD_NAMES = ("dL_dmeans2D", "dL_dcolors", "dL_dopacity", "dL_dmeans3D", "dL_dcov3D", "dL_dconic",
              "dL_dsh", "dL_dscales", "dL_drotations")


def rel_err(a: torch.Tensor, b: torch.Tensor) -> float:
    """norm-relative error ||a-b|| / ||b|| (0 if both are zero)."""
    a = a.double().flatten(); b = b.double().flatten()
    nb = b.norm().item()
    d = (a - b).norm().item()
    if nb == 0.0:
        return 0.0 if d == 0.0 else float("inf")
    return d / nb


# ------------------------------------------------------------------ stored reference results (tests/golden/reference/*.npz)
# The reference's outputs of the GPU parity tests are stored as fingerprints small enough to commit
# (tests/golden/make_golden_reference.py writes them): a digest of the bytes for the bit-exact checks, the
# exact norm and max|x|, a count sketch (the norm of a difference is estimated over EVERY element) and the
# values at a few seeded positions (element-wise checks).
SKETCH = 16
SAMPLE = 8
GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")


def _np(x) -> np.ndarray:
    if isinstance(x, torch.Tensor):
        x = x.detach().cpu().contiguous().numpy()
    return np.ascontiguousarray(np.asarray(x))


def digest(x) -> bytes:
    import hashlib
    return hashlib.sha256(_np(x).tobytes()).digest()[:16]


_hashes = {}


def _hash(n: int, device):
    """Seeded bucket, sign and sample position of every element of an n-element array."""
    key = (n, str(device))
    if key not in _hashes:
        g = torch.Generator().manual_seed(20240917)
        bucket = torch.randint(0, SKETCH, (n,), generator=g)
        sign = (torch.randint(0, 2, (n,), generator=g) * 2 - 1).double()
        pos = torch.randint(0, max(n, 1), (SAMPLE,), generator=g)
        _hashes.clear()
        _hashes[key] = (bucket.to(device), sign.to(device), pos)
    return _hashes[key]


def _flat64(x) -> torch.Tensor:
    if not isinstance(x, torch.Tensor):
        return torch.from_numpy(_np(x).astype(np.float64).reshape(-1))
    return x.detach().reshape(-1).double()


def sketch(x) -> torch.Tensor:
    v = _flat64(x)
    bucket, sign, _ = _hash(v.numel(), v.device)
    return torch.zeros(SKETCH, dtype=torch.float64, device=v.device).index_add_(0, bucket, v * sign).cpu()


def fingerprint(x) -> tuple:
    """(shape, digest, [numel, norm, max|x|, sketch..., sample...]) of a tensor or array."""
    v = _flat64(x)
    n = v.numel()
    sample = torch.zeros(SAMPLE, dtype=torch.float64)
    if n:
        sample = v[_hash(n, v.device)[2].to(v.device)].cpu()
    stats = [float(n), v.norm().item() if n else 0.0, v.abs().max().item() if n else 0.0]
    row = np.concatenate([np.array(stats), sketch(v).numpy(), sample.numpy()])
    return tuple(_np(x).shape), digest(x), row


def save_golden(path: str, records: dict) -> None:
    """records: key -> tensor/array (the reference's result)."""
    keys = sorted(records)
    fps = [fingerprint(records[k]) for k in keys]
    np.savez_compressed(path, keys=np.array(keys), shapes=np.array([",".join(map(str, f[0])) for f in fps]),
                        digests=np.frombuffer(b"".join(f[1] for f in fps), np.uint8).reshape(len(keys), 16),
                        rows=np.stack([f[2] for f in fps]))


class Ref:
    """A reference tensor known by its fingerprint."""

    def __init__(self, shape, dig, row):
        self.shape = shape
        self.digest = dig
        self.numel, self.norm, self.absmax = int(row[0]), float(row[1]), float(row[2])
        self.sketch = torch.from_numpy(row[3:3 + SKETCH].copy())
        self.sample = torch.from_numpy(row[3 + SKETCH:].copy())

    def equal(self, x) -> bool:
        """Bit-identical (same shape, dtype and bytes)."""
        return tuple(_np(x).shape) == self.shape and digest(x) == self.digest

    def rel_err(self, x) -> float:
        """||x - ref|| / ||ref||, the numerator estimated through the count sketch of the whole array."""
        assert tuple(_np(x).shape) == self.shape, f"shape {tuple(_np(x).shape)} vs {self.shape}"
        d = (sketch(x) - self.sketch).norm().item()
        if self.norm == 0.0:
            return 0.0 if _flat64(x).abs().max().item() == 0.0 else float("inf")
        return d / self.norm

    def sq_dist(self, x) -> float:
        """||x - ref||^2 estimated through the count sketch (for 0/1 flags: the number of differing elements)."""
        assert tuple(_np(x).shape) == self.shape, f"shape {tuple(_np(x).shape)} vs {self.shape}"
        return (sketch(x) - self.sketch).norm().item() ** 2

    def max_err(self, x) -> float:
        """max |x - ref| / max|ref| over the seeded sample positions."""
        v = _flat64(x)
        if self.numel == 0 or self.absmax == 0.0:
            return 0.0
        pos = _hash(v.numel(), v.device)[2].to(v.device)
        return (v[pos].cpu() - self.sample).abs().max().item() / self.absmax


def load_golden(name: str) -> dict:
    d = np.load(os.path.join(GOLDEN_DIR, name))
    return {str(k): Ref(tuple(int(s) for s in str(sh).split(",") if s), d["digests"][i].tobytes(), d["rows"][i])
            for i, (k, sh) in enumerate(zip(d["keys"], d["shapes"]))}


def make_inputs(scene_kind: str, n: int, W: int, H: int, mode: str, cam_k: int = 0, seed: int = 0,
                opacity_mode: str = "random", device=None, **cam_kw):
    if scene_kind == "strands":
        scene = synth.make_strand_scene(n, seed=seed, opacity_mode=opacity_mode)
        strand_dir = True
    else:
        scene = synth.make_blob_scene(n, seed=seed)
        strand_dir = False
    cam = synth.make_camera(cam_k, W, H, **cam_kw)
    if not strand_dir:
        # blobs: dir feature is whatever; keep the same preamble code path
        pass
    inp = synth.rasterizer_inputs(scene, cam, mode=mode, device=device)
    return inp
