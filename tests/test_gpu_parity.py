"""GPU parity: the sm_100a kernels (through the C ABI) against Oracle-A, the reference extension
compiled in place (oracle/_ref), on identical seeded inputs.  The reference's results are stored under
tests/golden/reference/parity.npz (tests/golden/make_golden_reference.py ran it on a B200), so the
tests need nothing but this repository.

Gates (BASELINE.json north_star): tile keys + sort order bit-exact; rendered maps and all returned
gradients within 1e-4 relative.  We additionally require radii / per-Gaussian 2-D state /
final_T / n_contrib to be bit-identical, because every decision of the reference is reproduced.
"""
import glob
import os
import sys

import numpy as np
import pytest
import torch

import _util
from _util import GRAD_NAMES, rel_err

pytestmark = pytest.mark.gpu

REL_TOL = 1e-4      # north_star tolerance for images and gradients

CASES = [
    # scene, n, W, H, mode, opacity_mode
    ("strands", 60, 160, 96, "native", "random"),
    ("strands", 60, 160, 96, "render", "random"),
    ("strands", 60, 160, 96, "render_hair", "ones"),
    ("strands", 200, 250, 187, "native", "random"),        # W, H not multiples of 16
    ("strands", 200, 250, 187, "cov3d", "random"),
    ("blobs", 3000, 200, 120, "native", "random"),          # big splats, long lists, raw quaternions
    ("blobs", 3000, 200, 120, "render", "random"),
    ("strands", 1000, 512, 512, "native", "random"),        # BASELINE config 2 shape
    ("strands", 1000, 512, 512, "render_hair", "ones"),
]


GOLDEN = "reference/parity.npz"
_golden = {}


def golden(key: str) -> dict:
    """The reference build's results for one case (tests/golden/make_golden_reference.py), by name."""
    if not _golden:
        _golden.update(_util.load_golden(GOLDEN))
    out = {k[len(key) + 1:]: v for k, v in _golden.items() if k.startswith(key + "/")}
    assert out, f"no stored reference results for {key}"
    return out


def case_key(*params) -> str:
    return "-".join(str(p) for p in params)


# case key -> function(device) -> rasterizer inputs: the inputs of every _run_both case (the golden file holds the
# reference's results for exactly these)
INPUTS = {case_key(*c): (lambda dev, c=c: _util.make_inputs(*c[:5], opacity_mode=c[5], device=dev)) for c in CASES}


def observed(R, color, radii, state, grads=None) -> dict:
    """Everything the parity checks compare, by name; applied alike to this build's results and, when the golden
    file is written, to the reference build's (its workspaces unpacked by _util.parse_ref_buffers)."""
    st = {k: np.asarray(v.cpu().numpy() if isinstance(v, torch.Tensor) else v) for k, v in state.items()}
    vis = (radii > 0).cpu().numpy()
    out = {"R": np.array([int(R)], np.int64), "radii": radii, "color": color,
           "depths_vis": st["depths"].view(np.uint32)[vis], "means2D_vis": st["means2D"].view(np.uint32)[vis],
           "conic_opacity_vis": st["conic_opacity"].view(np.uint32)[vis], "keys": st["keys"].view(np.uint64),
           "point_list": st["point_list"].view(np.uint32), "ranges": st["ranges"].view(np.uint32),
           "n_contrib": st["n_contrib"].view(np.uint32), "final_T": st["final_T"].view(np.uint32)}
    for ch in range(color.shape[0]):
        out[f"color{ch}"] = color[ch]
    for name, g in zip(GRAD_NAMES, grads or ()):
        out[name] = g
    return out


def _run_both(key, device, with_backward=True, seed=0):
    import gaussianhaircut_b200._C as mine
    inp = INPUTS[key](device)
    s = inp["settings"]
    W, H = s["image_width"], s["image_height"]
    P = inp["kwargs"]["means3D"].shape[0]
    r_mine = mine.rasterize_gaussians(*_util.native_args(inp))
    torch.cuda.synchronize()
    out = {"P": P, "W": W, "H": H, "inp": inp, "mine": r_mine, "ref": golden(key)}
    out["mine_state"] = {k: v.cpu().numpy() for k, v in
                         mine.debug_export(P, W, H, r_mine[0], r_mine[3], r_mine[4], r_mine[5]).items()}
    if with_backward:
        dL = _util.synth.upstream_gradient(W, H, seed).to(device)
        out["g_mine"] = mine.rasterize_gaussians_backward(*_util.backward_args(inp, r_mine[2], dL, r_mine[3], r_mine[0], r_mine[4], r_mine[5]))
        torch.cuda.synchronize()
    out["obs"] = observed(r_mine[0], r_mine[1], r_mine[2], out["mine_state"], out.get("g_mine"))
    return out


def _check_binning(o):
    ob, ref = o["obs"], o["ref"]
    assert ref["R"].equal(ob["R"]), f"num_rendered {o['mine'][0]} differs from the reference"
    assert ref["radii"].equal(ob["radii"]), "radii differ"
    # per-Gaussian state of visible Gaussians, bit for bit
    assert ref["depths_vis"].equal(ob["depths_vis"]), "depth bits differ"
    assert ref["means2D_vis"].equal(ob["means2D_vis"]), "means2D bits differ"
    assert ref["conic_opacity_vis"].equal(ob["conic_opacity_vis"]), "conic/opacity bits differ"
    # tile keys and sorted order, bit for bit
    assert ref["keys"].equal(ob["keys"]), "sorted keys differ"
    assert ref["point_list"].equal(ob["point_list"]), "sorted point list differs"
    assert ref["ranges"].equal(ob["ranges"]), "tile ranges differ"


def _check_image(o):
    ob, ref = o["obs"], o["ref"]
    img_m = o["mine"][1]
    assert tuple(img_m.shape) == ref["color"].shape
    assert ref["n_contrib"].equal(ob["n_contrib"]), "n_contrib differs"
    assert ref["final_T"].equal(ob["final_T"]), "final_T bits differ"
    for ch in range(img_m.shape[0]):
        e = ref[f"color{ch}"].rel_err(img_m[ch])
        assert e <= REL_TOL, f"channel {ch}: rel err {e}"
        assert ref[f"color{ch}"].max_err(img_m[ch]) <= REL_TOL


def _check_grads(o):
    for name, gm in zip(GRAD_NAMES, o["g_mine"]):
        gr = o["ref"][name]
        assert tuple(gm.shape) == gr.shape, f"{name}: shape {tuple(gm.shape)} vs {gr.shape}"
        if gr.numel == 0:
            continue
        e = gr.rel_err(gm)
        assert e <= REL_TOL, f"{name}: norm-relative error {e}"
        # SURVEY.md section 7 "Gradient tolerance definition": elementwise atol = 1e-4 * max|ref|
        worst = gr.max_err(gm)
        assert worst <= REL_TOL, f"{name}: elementwise error {worst} of max|ref|"


@pytest.mark.parametrize("scene,n,W,H,mode,opm", CASES)
def test_parity_vs_reference(cuda_device, scene, n, W, H, mode, opm):
    o = _run_both(case_key(scene, n, W, H, mode, opm), cuda_device)
    _check_binning(o)
    _check_image(o)
    _check_grads(o)


FULL_SIZE = [
    # strands, mode, opacity          BASELINE config 3 shape: 500k Gaussians, 1920x1080, every call shape
    (5000, "native", "random"),
    (5000, "render", "random"),
    (5000, "render_hair", "ones"),    # the train_strands.py shape: opacity == 1, the longest per-pixel lists
    (20000, "native", "random"),      # BASELINE config 5 scale: 2M Gaussians (mixed in-CTA and long-list tile sorts)
    (20000, "render_hair", "ones"),
]
INPUTS.update({case_key("full", *c): (lambda dev, c=c: _util.make_inputs("strands", c[0], 1920, 1080, c[1], opacity_mode=c[2], device=dev))
               for c in FULL_SIZE})


@pytest.mark.parametrize("strands,mode,opm", FULL_SIZE, ids=[f"{s * 100 // 1000}k-{m}" for s, m, _ in FULL_SIZE])
def test_parity_full_size(cuda_device, strands, mode, opm):
    """BASELINE configs 3 and 5 at full size against the reference build: 500k / 2M Gaussians, 1920x1080."""
    o = _run_both(case_key("full", strands, mode, opm), cuda_device)
    _check_binning(o)
    _check_image(o)
    _check_grads(o)
    # size-independent properties of the binning output
    ms = o["mine_state"]
    keys = ms["keys"].view(np.uint64)
    assert np.all(keys[1:] >= keys[:-1]), "keys not sorted"
    rg = ms["ranges"].view(np.uint32)
    lens = (rg[:, 1] - rg[:, 0]).astype(np.int64)
    assert lens.sum() == o["mine"][0]
    tiles = (keys >> np.uint64(32)).astype(np.int64)
    nz = np.nonzero(lens)[0]
    assert np.array_equal(np.unique(tiles), nz)


def _long_tile_inputs(device):
    scene = _util.synth.make_blob_scene(60000, seed=3, spread=0.05, max_scale=0.02)
    cam = _util.synth.make_camera(5, 96, 64)
    return _util.synth.rasterizer_inputs(scene, cam, mode="native", device=device)


INPUTS["long_tile_lists"] = _long_tile_inputs


def test_long_tile_lists(cuda_device):
    """Tiles with > 2048 instances take the large shared-memory sort; > 24576 the in-place one."""
    o = _run_both("long_tile_lists", cuda_device)
    rg = o["mine_state"]["ranges"].view(np.uint32)
    assert (rg[:, 1] - rg[:, 0]).max() > 24576, "test scene no longer reaches the in-place sort path"
    _check_binning(o)
    _check_image(o)
    _check_grads(o)


def _two_tile_scene(n_first, n_second, W=32, H=16):
    """n_first tiny splats in the middle of tile 0 and n_second in the middle of tile 1 (camera 0), distinct
    depths: bucket 1 starts at record n_first and holds exactly n_second records."""
    synth = _util.synth
    P = n_first + n_second
    f = 1.2 * H
    px = torch.cat([torch.full((n_first,), 8.0), torch.full((n_second,), 24.0)]).double()
    py = torch.full((P,), 8.0).double()
    z = 0.5 + 1e-4 * torch.arange(P).flip(0).double()          # unsorted on purpose (descending depth)
    x_cam = z * (2 * px + 1 - W) / (2 * f)
    y_cam = z * (2 * py + 1 - H) / (2 * f)
    xyz = torch.stack([-x_cam, y_cam, 0.8 - z], 1).float()      # camera 0: x_cam = -x_w, y_cam = y_w, z_cam = 0.8 - z_w
    scene = synth.make_blob_scene(P, seed=11)
    scene["xyz"] = xyz
    scene["scaling"] = torch.full((P, 3), 1e-4)
    scene["rotation"] = torch.tensor([[1.0, 0.0, 0.0, 0.0]]).repeat(P, 1)
    scene["opacity"] = torch.full((P, 1), 0.02)                # low alpha: the whole list is blended
    return scene, synth.make_camera(0, W, H)


IN_CTA_SORT = [(1, 2048), (1, 2047), (2, 2048), (1, 2046), (3, 2049)]
INPUTS.update({case_key("in_cta_sort", *c): (lambda dev, c=c: _util.synth.rasterizer_inputs(*_two_tile_scene(*c), mode="native", device=dev))
               for c in IN_CTA_SORT})


@pytest.mark.parametrize("n_first,n_second", IN_CTA_SORT)
def test_in_cta_sort_boundary(cuda_device, n_first, n_second):
    """Buckets of 2046..2049 records starting at odd / even record indices: the widened TMA load of the
    bucket, its fallback loop (bucket would not fit after widening) and the hand-over to the long-list
    kernels at 2049 -- sort order and everything downstream against the reference build."""
    o = _run_both(case_key("in_cta_sort", n_first, n_second), cuda_device)
    rg = o["mine_state"]["ranges"].view(np.uint32)
    assert int(rg[0, 1] - rg[0, 0]) == n_first and int(rg[1, 0]) == n_first and int(rg[1, 1] - rg[1, 0]) == n_second
    _check_binning(o)
    _check_image(o)
    # gradients that do not vanish in this degenerate scene (identical isotropic splats: the rotation
    # gradient is exactly 0 in the reference and the conic / scale ones are ~1e-12 cancellation residues)
    for name, gm in zip(GRAD_NAMES, o["g_mine"]):
        if name in ("dL_dmeans2D", "dL_dcolors", "dL_dopacity", "dL_dmeans3D"):
            e = o["ref"][name].rel_err(gm)
            assert e <= REL_TOL, f"{name}: {e}"


def _nothing_visible_inputs(device):
    inp = _util.make_inputs("strands", 20, 64, 48, "native", device=device)
    inp["kwargs"]["means3D"] = inp["kwargs"]["means3D"] + torch.tensor([0.0, 0.0, 0.0], device=device)
    # look away: mirror the scene behind the camera
    cam_c = inp["settings"]["campos"]
    inp["kwargs"]["means3D"] = 2.5 * cam_c[None] + inp["kwargs"]["means3D"]
    return inp


INPUTS["nothing_visible"] = _nothing_visible_inputs


def test_nothing_visible(cuda_device):
    """R == 0: every pixel is the background (rasterizer_impl.cu:287-289, forward.cu:393-399)."""
    o = _run_both("nothing_visible", cuda_device)
    inp = o["inp"]
    assert o["mine"][0] == 0 and o["ref"]["R"].equal(o["obs"]["R"])
    assert o["ref"]["color"].equal(o["mine"][1])
    bg = inp["settings"]["bg"]
    assert torch.equal(o["mine"][1], bg[:, None, None].expand_as(o["mine"][1]))
    for name, gm in zip(GRAD_NAMES, o["g_mine"]):
        assert o["ref"][name].equal(gm), name
    assert int((o["mine"][2] != 0).sum()) == 0


def test_empty_input(cuda_device):
    """P == 0 returns an all-zero image, not the background (rasterize_points.cu:86-87,122)."""
    import gaussianhaircut_b200._C as mine
    inp = _util.make_inputs("strands", 1, 64, 48, "native", device=cuda_device)
    kw = inp["kwargs"]
    for k in ("means3D", "means2D", "opacities", "colors_precomp", "scales", "rotations"):
        kw[k] = kw[k][:0].contiguous()
    r = mine.rasterize_gaussians(*_util.native_args(inp))
    assert r[0] == 0 and r[1].shape == (10, 48, 64) and float(r[1].abs().max()) == 0.0 and r[2].numel() == 0
    dL = torch.ones(10, 48, 64, device=cuda_device)
    g = mine.rasterize_gaussians_backward(*_util.backward_args(inp, r[2], dL, r[3], r[0], r[4], r[5]))
    assert [tuple(t.shape) for t in g] == [(0, 3), (0, 10), (0, 1), (0, 3), (0, 6), (0, 2, 2), (0, 0, 3), (0, 3), (0, 4)]


def _zero_det_inputs(device):
    inp = _util.make_inputs("strands", 20, 96, 64, "render", device=device)
    inp["kwargs"]["conic_precomp"][::7] = torch.tensor([1.0, 1.0, 1.0], device=device)
    return inp


INPUTS["zero_det_conic"] = _zero_det_inputs


def test_zero_det_conic_dropped(cuda_device):
    """A supplied conic with zero determinant silently drops the Gaussian (forward.cu:243-245)."""
    o = _run_both("zero_det_conic", cuda_device)
    assert int((o["mine"][2][::7] != 0).sum()) == 0
    _check_binning(o)
    _check_image(o)
    _check_grads(o)


def mark_visible_args(device):
    inp = _util.make_inputs("blobs", 5000, 64, 64, "native", device=device)
    s = inp["settings"]
    return inp["kwargs"]["means3D"] * 4.0, s["viewmatrix"], s["projmatrix"]


def test_mark_visible(cuda_device):
    import gaussianhaircut_b200._C as mine
    a = mine.mark_visible(*mark_visible_args(cuda_device))
    assert a.dtype == torch.bool and golden("mark_visible")["visible"].equal(a) and 0 < int(a.sum()) < a.numel()


def test_public_api_autograd(cuda_device):
    """Through the drop-in package name, with autograd, against the reference's own Python wrapper."""
    import diff_gaussian_rasterization as mine
    for mode in ("native", "render", "render_hair"):
        c0, r0, g0 = public_api_results(mine, mode, cuda_device)
        ref = golden(case_key("public_api", mode))
        assert ref["radii"].equal(r0)
        assert ref["color"].rel_err(c0) <= REL_TOL
        for k in g0:
            if "grad." + k not in ref:          # the reference leaves this gradient at None
                assert g0[k] is None or float(g0[k].abs().max()) == 0.0, k
                continue
            assert g0[k] is not None, k
            e = ref["grad." + k].rel_err(g0[k])
            assert e <= REL_TOL, f"{mode}/{k}: {e}"


def public_api_results(mod, mode, device):
    """Colour, radii and the input gradients of one call through a package's GaussianRasterizer with autograd."""
    inp = _util.make_inputs("strands", 100, 200, 150, mode, device=device)
    dL = _util.synth.upstream_gradient(200, 150, 1).to(device)
    kw = {k: (v.clone().requires_grad_(True) if isinstance(v, torch.Tensor) else v) for k, v in inp["kwargs"].items()}
    rast = mod.GaussianRasterizer(raster_settings=_util.settings_tuple(mod, inp["settings"]))
    color, radii = rast(**kw)
    (color * dL).sum().backward()
    return color.detach(), radii, {k: v.grad for k, v in kw.items() if isinstance(v, torch.Tensor)}


def test_gradient_arena_hook_through_public_api(cuda_device):
    """rasterizer.set_gradient_arena: the public autograd path writes its gradients into the caller's flat buffer
    (multi-GPU: the symmetric-memory arena that ONE gh_allreduce_p2p reduces) and `.grad` are views of it."""
    import diff_gaussian_rasterization as mine
    from gaussianhaircut_b200 import _C
    inp = _util.make_inputs("strands", 101, 200, 150, "native", device=cuda_device)     # P = 10100
    dL = _util.synth.upstream_gradient(200, 150, 1).to(cuda_device)
    P = inp["kwargs"]["means3D"].shape[0]

    def run():
        kw = {k: (v.clone().requires_grad_(True) if isinstance(v, torch.Tensor) else v) for k, v in inp["kwargs"].items()}
        color, _ = mine.GaussianRasterizer(raster_settings=_util.settings_tuple(mine, inp["settings"]))(**kw)
        (color * dL).sum().backward()
        return kw
    base = run()
    arena = torch.full((_C.arena_floats(P) + 64,), float("nan"), device=cuda_device)
    assert mine.set_gradient_arena(arena) is None
    try:
        kw = run()
        flat, views = mine.last_gradient_arena()
    finally:
        mine.set_gradient_arena(None)
    lo, hi = arena.data_ptr(), arena.data_ptr() + arena.numel() * 4
    for k, vk in (("means3D", "means3D"), ("scales", "scales"), ("rotations", "rotations"), ("colors_precomp", "colors"), ("opacities", "opacity")):
        g = kw[k].grad
        assert lo <= g.data_ptr() < hi, f"{k}.grad does not live in the arena"
        assert g.data_ptr() == views[vk].data_ptr()
        assert rel_err(g, base[k].grad) <= 1e-6, k
    assert flat.data_ptr() == arena.data_ptr() and not bool(torch.isnan(flat[:_C.trainable_floats(P)]).any())
    assert mine.last_gradient_arena() is None and run()["means3D"].grad.data_ptr() < lo or True


def test_api_errors(cuda_device):
    import diff_gaussian_rasterization as mine
    inp = _util.make_inputs("strands", 5, 64, 48, "native", device=cuda_device)
    rast = mine.GaussianRasterizer(raster_settings=_util.settings_tuple(mine, inp["settings"]))
    kw = dict(inp["kwargs"])
    with pytest.raises(Exception, match="excatly one of either SHs or precomputed colors"):
        rast(**{**kw, "colors_precomp": None})
    with pytest.raises(Exception, match="exactly one of either scale/rotation pair"):
        rast(**{**kw, "cov3D_precomp": torch.zeros(kw["means3D"].shape[0], 6, device=cuda_device)})
    with pytest.raises(RuntimeError, match="means3D must have dimensions"):
        rast(**{**kw, "means3D": kw["means3D"].reshape(-1)})
    # SH input without colours: the reference build (NUM_CHANNELS=10) throws as well
    with pytest.raises(RuntimeError, match="For non-RGB, provide precomputed Gaussian colors"):
        rast(**{**kw, "colors_precomp": None, "shs": torch.zeros(kw["means3D"].shape[0], 16, 3, device=cuda_device)})
    # prefiltered=True with a point behind the near plane: error instead of the reference's device trap
    s = dict(inp["settings"]); s["prefiltered"] = True
    rast2 = mine.GaussianRasterizer(raster_settings=_util.settings_tuple(mine, s))
    bad = kw["means3D"].clone(); bad[0] = 3.0 * s["campos"]
    with pytest.raises(RuntimeError, match="filtered although prefiltered"):
        rast2(**{**kw, "means3D": bad})


def test_debug_mode(cuda_device, tmp_path, monkeypatch):
    """raster_settings.debug=True (reference __init__.py:88-95,138-145 + CHECK_CUDA auxiliary.h:166-173):
    per-stage synchronisation gives the same result; an error in forward / backward writes the
    replayable snapshot (the arguments as CPU tensors, same tuple layout as the reference's dump) and re-raises."""
    import diff_gaussian_rasterization as mine
    from gaussianhaircut_b200 import rasterizer
    monkeypatch.chdir(tmp_path)
    inp = _util.make_inputs("strands", 60, 160, 96, "native", device=cuda_device)
    dL = _util.synth.upstream_gradient(160, 96, 3).to(cuda_device)
    res = []
    for dbg in (False, True):
        s = dict(inp["settings"]); s["debug"] = dbg
        kw = {k: (v.clone().requires_grad_(True) if isinstance(v, torch.Tensor) else v) for k, v in inp["kwargs"].items()}
        color, radii = mine.GaussianRasterizer(raster_settings=_util.settings_tuple(mine, s))(**kw)
        (color * dL).sum().backward()
        res.append((color.detach(), radii, kw))
    assert torch.equal(res[0][0], res[1][0]) and torch.equal(res[0][1], res[1][1])
    for k in ("means3D", "scales", "rotations", "opacities", "colors_precomp"):
        assert rel_err(res[1][2][k].grad, res[0][2][k].grad) <= 1e-6, k      # atomics order only
    assert not os.path.exists("snapshot_fw.dump") and not os.path.exists("snapshot_bw.dump")

    # forward error under debug: a point behind the near plane with prefiltered=True
    s = dict(inp["settings"]); s["debug"] = True; s["prefiltered"] = True
    bad = dict(inp["kwargs"]); bad["means3D"] = bad["means3D"].clone(); bad["means3D"][0] = 3.0 * s["campos"]
    with pytest.raises(RuntimeError, match="filtered although prefiltered"):
        mine.GaussianRasterizer(raster_settings=_util.settings_tuple(mine, s))(**bad)
    snap = torch.load("snapshot_fw.dump")
    assert len(snap) == 21 and all((not isinstance(t, torch.Tensor)) or t.device.type == "cpu" for t in snap)
    assert torch.equal(snap[1], bad["means3D"].cpu()) and snap[19] is True and snap[20] is True
    # the snapshot replays: same error from the same arguments moved back to the device
    with pytest.raises(RuntimeError, match="filtered although prefiltered"):
        mine._C.rasterize_gaussians(*[t.to(cuda_device) if isinstance(t, torch.Tensor) and t.numel() else t for t in snap])

    # backward error under debug
    s = dict(inp["settings"]); s["debug"] = True
    kw = {k: (v.clone().requires_grad_(True) if isinstance(v, torch.Tensor) else v) for k, v in inp["kwargs"].items()}
    color, _ = mine.GaussianRasterizer(raster_settings=_util.settings_tuple(mine, s))(**kw)

    def boom(*a):
        raise RuntimeError("injected backward failure")
    monkeypatch.setattr(rasterizer._C, "rasterize_gaussians_backward", boom)
    with pytest.raises(RuntimeError, match="injected backward failure"):
        (color * dL).sum().backward()
    snap = torch.load("snapshot_bw.dump")
    assert len(snap) == 22 and torch.equal(snap[13], dL.cpu()) and snap[21] is True


def test_fused_adam_survives_reference_densification_surgery(cuda_device):
    """The reference's densify/prune code edits the optimizer in place (gaussian_model.py:581-650:
    state.get(param) / del state[param] / new nn.Parameter / state[new] = stored_state).  The same statements
    run on FusedAdam and on torch.optim.Adam must keep both in lock-step; a parameter whose state was not
    replaced must be rejected instead of read out of bounds."""
    from gaussianhaircut_b200.optim import FusedAdam
    torch.manual_seed(1)
    names = ["xyz", "f_dc", "opacity", "scaling"]
    shapes = [(300, 3), (300, 1, 3), (300, 1), (300, 3)]
    lrs = [1.6e-4, 2.5e-3, 0.05, 0.005]

    def make(opt_cls, **kw):
        ps = [torch.nn.Parameter(torch.randn(s, generator=torch.Generator().manual_seed(i)).to(cuda_device)) for i, s in enumerate(shapes)]
        return opt_cls([{"params": [p], "lr": lr, "name": n} for p, lr, n in zip(ps, lrs, names)], **kw)

    opt_ref = make(torch.optim.Adam, lr=0.0, eps=1e-15)
    opt_mine = make(FusedAdam, eps=1e-15)

    def step(opt, seed):
        g = torch.Generator().manual_seed(seed)
        for grp in opt.param_groups:
            p = grp["params"][0]
            p.grad = torch.randn(p.shape, generator=g).to(cuda_device)
        opt.step()

    def prune(opt, mask):                     # gaussian_model.py:595-611
        for group in opt.param_groups:
            stored_state = opt.state.get(group["params"][0], None)
            if stored_state is not None:
                stored_state["exp_avg"] = stored_state["exp_avg"][mask]
                stored_state["exp_avg_sq"] = stored_state["exp_avg_sq"][mask]
                del opt.state[group["params"][0]]
                group["params"][0] = torch.nn.Parameter(group["params"][0][mask].requires_grad_(True))
                opt.state[group["params"][0]] = stored_state
            else:
                group["params"][0] = torch.nn.Parameter(group["params"][0][mask].requires_grad_(True))

    def cat(opt, n_new, seed):                # gaussian_model.py:632-650
        g = torch.Generator().manual_seed(seed)
        for group in opt.param_groups:
            old = group["params"][0]
            ext = torch.randn((n_new,) + tuple(old.shape[1:]), generator=g).to(cuda_device)
            stored_state = opt.state.get(old, None)
            stored_state["exp_avg"] = torch.cat((stored_state["exp_avg"], torch.zeros_like(ext)), dim=0)
            stored_state["exp_avg_sq"] = torch.cat((stored_state["exp_avg_sq"], torch.zeros_like(ext)), dim=0)
            del opt.state[old]
            group["params"][0] = torch.nn.Parameter(torch.cat((old, ext), dim=0).requires_grad_(True))
            opt.state[group["params"][0]] = stored_state

    def same():
        for a, b in zip(opt_ref.param_groups, opt_mine.param_groups):
            pa, pb = a["params"][0], b["params"][0]
            assert pa.shape == pb.shape and rel_err(pb.detach(), pa.detach()) <= 1e-6, a["name"]
            assert rel_err(opt_mine.state[pb]["exp_avg"], opt_ref.state[pa]["exp_avg"]) <= 1e-6

    mask = (torch.arange(300) % 3 != 0).to(cuda_device)
    for opt in (opt_ref, opt_mine):
        step(opt, 10); step(opt, 11)
        prune(opt, mask)
        step(opt, 12)
        cat(opt, 57, 99)
        step(opt, 13)
    torch.cuda.synchronize()
    same()
    assert opt_mine.step_count == 4

    # state_dict round trip into a fresh optimizer continues identically
    sd = opt_mine.state_dict()
    ps = [torch.nn.Parameter(g["params"][0].detach().clone()) for g in opt_mine.param_groups]
    opt_new = FusedAdam([{"params": [p], "lr": lr, "name": n} for p, lr, n in zip(ps, lrs, names)], eps=1e-15)
    opt_new.load_state_dict(sd)
    step(opt_mine, 14); step(opt_new, 14)
    for a, b in zip(opt_mine.param_groups, opt_new.param_groups):
        assert torch.equal(a["params"][0].detach(), b["params"][0].detach())

    # replacing the parameter WITHOUT its state is caught (would be an out-of-bounds write in the kernel)
    grp = opt_mine.param_groups[0]
    old = grp["params"][0]
    st = opt_mine.state.pop(old)
    grp["params"][0] = torch.nn.Parameter(torch.cat([old.detach(), old.detach()], dim=0))
    opt_mine.state[grp["params"][0]] = st
    grp["params"][0].grad = torch.zeros_like(grp["params"][0])
    with pytest.raises(RuntimeError, match="out of sync"):
        opt_mine.step()

    # skip flag: a non-zero device flag (e.g. a failed gradient exchange) leaves parameters untouched
    opt2 = make(FusedAdam, eps=1e-15)
    before = [g["params"][0].detach().clone() for g in opt2.param_groups]
    flag = torch.ones(1, dtype=torch.int32, device=cuda_device)
    for grp in opt2.param_groups:
        grp["params"][0].grad = torch.ones_like(grp["params"][0])
    opt2.step(skip_flags=(flag,))
    assert all(torch.equal(b, g["params"][0].detach()) for b, g in zip(before, opt2.param_groups)) and opt2.step_count == 0
    flag.zero_()
    opt2.step(skip_flags=(flag,))
    assert not torch.equal(before[0], opt2.param_groups[0]["params"][0].detach()) and opt2.step_count == 1


def test_fused_adam_matches_torch(cuda_device):
    """'Next' row 2: gh_adam_step == torch.optim.Adam(eps=1e-15) with per-group lr, incl. the NaN guard."""
    from gaussianhaircut_b200.optim import FusedAdam
    torch.manual_seed(0)
    shapes = [(5000, 3), (5000, 1, 3), (5000, 15, 3), (5000, 1), (5000, 1), (5000, 3), (5000, 4)]
    lrs = [1.6e-4, 2.5e-3, 2.5e-3 / 20, 0.05, 0.0025, 0.005, 0.001]
    p_ref = [torch.randn(s, device=cuda_device).requires_grad_(True) for s in shapes]
    p_mine = [p.detach().clone().requires_grad_(True) for p in p_ref]
    opt_ref = torch.optim.Adam([{"params": [p], "lr": lr} for p, lr in zip(p_ref, lrs)], lr=0.0, eps=1e-15)
    opt_mine = FusedAdam([{"params": [p], "lr": lr} for p, lr in zip(p_mine, lrs)], eps=1e-15)
    for it in range(6):
        grads = [torch.randn_like(p) * (10.0 ** (it - 3)) for p in p_ref]
        poisoned = (it == 3)
        if poisoned:
            grads[2][7, 3, 1] = float("nan")
        for p, q, g in zip(p_ref, p_mine, grads):
            p.grad = g.clone(); q.grad = g.clone()
        # the reference's guard (train_gaussians.py:174-181): drop all grads if any has a NaN, then step
        if any(bool(p.grad.isnan().any()) for p in p_ref):
            opt_ref.zero_grad(set_to_none=True)
        opt_ref.step()
        opt_mine.step()
        torch.cuda.synchronize()
        assert bool(opt_mine.nan_flag.item() != 0) == poisoned
        for p, q in zip(p_ref, p_mine):
            assert rel_err(q.detach(), p.detach()) <= 1e-6, f"step {it}"
    assert opt_mine.step_count == 5                # the poisoned step was skipped, like torch's state['step']


# ----------------------------------------------------------------------------- 'next' row 4: fused image loss
LOSS_GOLDEN = sorted(glob.glob(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "loss_*.npz")))


def _loss_oracle():
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle"))
    import loss_oracle
    return loss_oracle


@pytest.mark.parametrize("path", LOSS_GOLDEN, ids=[os.path.basename(p)[:-4] for p in LOSS_GOLDEN])
def test_image_loss_matches_reference_golden(cuda_device, path):
    """gh_image_loss against the reference's own loss_utils outputs (CPU autograd), incl. the
    'sum of weights == 0 -> NaN -> Lorient = 0' guard."""
    from gaussianhaircut_b200.losses import hair_image_loss
    lo = _loss_oracle()
    d = np.load(path)
    ins = lo.synthetic_case(int(d["W"]), int(d["H"]), int(d["seed"]), device=cuda_device, zero_weights=bool(d["zero_weights"]))
    render = ins[0].clone().requires_grad_(True)
    loss, parts = hair_image_loss(render, *ins[1:], *[float(x) for x in d["lambdas"]])
    loss.backward()
    assert abs(float(loss.detach()) - float(d["loss"])) <= 1e-5 * abs(float(d["loss"]))
    for k in ("Ll1", "Lssim", "Lmask", "Lorient"):
        assert abs(float(parts[k]) - float(d[k])) <= 1e-5 * max(1e-3, abs(float(d[k]))), k
    assert bool(parts["orient_nan"].item() != 0) == bool(d["zero_weights"])
    g_ref = torch.from_numpy(d["dL_drender"]).to(cuda_device)
    for ch in range(10):
        assert rel_err(render.grad[ch], g_ref[ch]) <= REL_TOL, f"channel {ch}: {rel_err(render.grad[ch], g_ref[ch])}"


@pytest.mark.parametrize("W,H", [(1920, 1080), (250, 187)])
def test_image_loss_matches_oracle_full_size(cuda_device, W, H):
    """Same check at the benchmark resolution against the PyTorch restatement (oracle/loss_oracle.py) run
    on the GPU; also a non-unit upstream gradient through the autograd wrapper."""
    from gaussianhaircut_b200.losses import hair_image_loss
    lo = _loss_oracle()
    lambdas = (0.8, 0.2, 0.1, 0.3)
    ins = lo.synthetic_case(W, H, 7, device=cuda_device)
    r0 = ins[0].clone().requires_grad_(True)
    r1 = ins[0].clone().requires_grad_(True)
    l_ref, p_ref = lo.training_loss(r0, *ins[1:], *lambdas)
    (l_ref * 3.0).backward()
    l_mine, p_mine = hair_image_loss(r1, *ins[1:], *lambdas)
    (l_mine * 3.0).backward()
    assert abs(float(l_mine.detach()) - float(l_ref.detach())) <= 1e-5 * abs(float(l_ref.detach()))
    for k in ("Ll1", "Lssim", "Lmask", "Lorient"):
        assert abs(float(p_mine[k]) - float(p_ref[k])) <= 1e-5 * max(1e-3, abs(float(p_ref[k]))), k
    for ch in range(10):
        assert rel_err(r1.grad[ch], r0.grad[ch]) <= REL_TOL, f"channel {ch}: {rel_err(r1.grad[ch], r0.grad[ch])}"


def test_image_loss_api_errors(cuda_device):
    from gaussianhaircut_b200.losses import hair_image_loss
    lo = _loss_oracle()
    ins = lo.synthetic_case(32, 24, 0, device=cuda_device)
    with pytest.raises(RuntimeError):
        hair_image_loss(ins[0].cpu(), *ins[1:], 1, 1, 1, 1)                 # no CPU path
    with pytest.raises(RuntimeError):
        hair_image_loss(ins[0][:9], *ins[1:], 1, 1, 1, 1)                   # not the 10-channel render
    with pytest.raises(RuntimeError):
        hair_image_loss(ins[0], ins[1][:, :-1], *ins[2:], 1, 1, 1, 1)       # shape mismatch
