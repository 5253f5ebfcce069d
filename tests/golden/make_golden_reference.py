"""Generate tests/golden/reference/*.npz: the reference's results that the GPU tests compare against.

Runs the reference itself on a B200: its CUDA extension compiled in place under oracle/_ref (oracle/build_ref.py)
and, for the densification and render() cases, its own Python (the copy build_ref stages under oracle/_ref/src).
Every result is stored as a fingerprint (tests/_util.py `save_golden`: digest, norm, max, count sketch, a seeded
sample), small enough to commit; the tests then need nothing outside the repository.

    python tests/golden/make_golden_reference.py OUT_DIR   # on the GPU, after build(); copy OUT_DIR/*.npz to tests/golden/reference/
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
for p in (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "oracle")):
    sys.path.insert(0, p)
import _util  # noqa: E402
import build_ref  # noqa: E402


def parity(dev):
    import test_gpu_parity as t
    ref = build_ref.load()
    rec = {}
    for key, make in t.INPUTS.items():
        inp = make(dev)
        s = inp["settings"]
        W, H = s["image_width"], s["image_height"]
        P = inp["kwargs"]["means3D"].shape[0]
        r = ref._C.rasterize_gaussians(*_util.native_args(inp))
        dL = _util.synth.upstream_gradient(W, H, 0).to(dev)
        g = ref._C.rasterize_gaussians_backward(*_util.backward_args(inp, r[2], dL, r[3], r[0], r[4], r[5]))
        torch.cuda.synchronize()
        state = _util.parse_ref_buffers(P, W, H, r[0], r[3], r[4], r[5])
        for name, v in t.observed(r[0], r[1], r[2], state, g).items():
            rec[f"{key}/{name}"] = v
        print(key, "R =", r[0], flush=True)
    rec["mark_visible/visible"] = ref._C.mark_visible(*t.mark_visible_args(dev))
    for mode in ("native", "render", "render_hair"):
        color, radii, grads = t.public_api_results(ref, mode, dev)
        key = t.case_key("public_api", mode)
        rec[f"{key}/color"], rec[f"{key}/radii"] = color, radii
        for k, v in grads.items():
            if v is not None:
                rec[f"{key}/grad.{k}"] = v
    return rec


def projection(dev):
    import ref_python
    import test_gpu_projection as t
    rec = {}
    gr = ref_python.load_renderer("ref")
    for case in t.FUSED_RENDER:
        key = t.case_key(*case)
        pkg, pc, cam = t.render_gaussian_model(gr.render, ref_python.make_gaussian_model, case, dev)
        for name, v in t.render_observed(pkg, pc, cam).items():
            rec[f"{key}/{name}"] = v
        print(key, flush=True)
    return rec


def densify(dev):
    import test_gpu_densify as t
    rec = {}
    for n, max_screen_size, train_conf in sorted({c[:3] for c in t.DENSIFY}, key=str):   # FusedAdam cases share the reference
        a = t.model(t.scene(n, seed=3), dev, train_conf, seed=7, reference=True)
        torch.manual_seed(123); torch.cuda.manual_seed(123)
        a.densify_and_prune(2e-4, 0.005, 2.0, max_screen_size)
        key = t.case_key(n, max_screen_size, train_conf)
        rec.update({f"{key}/{k}": v for k, v in t.densify_observed(a).items()})
    a = t.model(t.scene(5000, seed=5), dev, True, seed=2, reference=True)
    a.reset_opacity()
    rec.update({f"reset_opacity/{k}": v for k, v in t.densify_observed(a, step=False).items()})
    a = t.model(t.scene(2_000_000, seed=11), dev, True, seed=1, reference=True)
    torch.manual_seed(5); torch.cuda.manual_seed(5)
    a.densify_and_prune(2e-4, 0.005, 2.0, 20)
    rec.update({f"config5/{k}": v for k, v in t.densify_observed(a, step=False).items()})
    return rec


def main():
    out = sys.argv[1]
    os.makedirs(out, exist_ok=True)
    dev = torch.device("cuda:0")
    for name, fn in (("parity", parity), ("projection", projection), ("densify", densify)):
        rec = fn(dev)
        path = os.path.join(out, f"{name}.npz")
        _util.save_golden(path, rec)
        print(path, len(rec), "records", os.path.getsize(path), "bytes", flush=True)


if __name__ == "__main__":
    main()
