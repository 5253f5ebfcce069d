"""GPU tests of the fused projection preamble ("next" row 8f-1) and of the `render()` / `render_hair()` drop-ins built
on it (gaussianhaircut_b200/projection.py, renderer.py):

* the two kernels against PyTorch autograd of the restated preamble (oracle/synth.py `project_reference`, pinned on
  the reference's Python by tests/test_project_cpu.py) at 500k Gaussians: values, every parameter gradient and the
  camera gradients (view / projection matrix, camera centre, tan fov), in both incoming-gradient modes;
* `renderer.render` / `renderer.render_hair` against the reference's OWN functions imported unmodified and running
  on the reference's OWN rasterizer build (oracle/ref_python.py + oracle/_ref): everything a trainer reads back.
  The reference's render() results are stored under tests/golden/reference/projection.npz; render_hair() drives the
  reference's hair model classes and runs only where the reference is staged.
Tolerance: the north-star 1e-4 (norm-relative) on maps and gradients."""
import os
import sys

import pytest
import torch

import _util
from _util import rel_err

pytestmark = pytest.mark.gpu
REL_TOL = 1e-4

sys.path.insert(0, os.path.join(_util.ROOT, "oracle"))
import ref_python  # noqa: E402


def _leaves(raw, dev):
    return {k: v.clone().to(dev).requires_grad_(True) for k, v in raw.items()}


@pytest.mark.parametrize("flavour,strands,W,H,deg", [("gaussian_model", 5000, 1920, 1080, 3), ("hair", 5000, 1920, 1080, 3),
                                                     ("gaussian_model", 37, 250, 187, 1), ("gaussian_model", 37, 250, 187, 0)])
def test_projection_kernels_match_autograd(cuda_device, flavour, strands, W, H, deg):
    from gaussianhaircut_b200 import projection
    synth = _util.synth
    dev = cuda_device
    scene = synth.make_strand_scene(strands, seed=2)
    cam = dict(synth.make_camera(19, W, H))
    cfg = dict(synth.PROJECT_GAUSSIAN_MODEL if flavour == "gaussian_model" else synth.PROJECT_HAIR_MODEL)
    raw = synth.raw_params_from_scene(scene, flavour)
    if flavour == "gaussian_model":
        raw["rotation"] = raw["rotation"] * (0.5 + torch.rand(raw["rotation"].shape[0], 1, generator=torch.Generator().manual_seed(1)))
    leaves = _leaves(raw, dev)
    camg = dict(cam)
    for k in ("world_view_transform", "full_proj_transform", "camera_center"):
        camg[k] = cam[k].to(dev).requires_grad_(True)
    camg["tanfovx"] = torch.tensor(cam["tanfovx"], dtype=torch.float32, device=dev, requires_grad=True)
    camg["tanfovy"] = torch.tensor(cam["tanfovy"], dtype=torch.float32, device=dev, requires_grad=True)
    ref = synth.project_reference(leaves, camg, cfg, sh_degree=deg)
    mask = ref["mask"]

    pi = projection.pack_inputs(leaves["xyz"], leaves["scaling"], leaves["rotation"], leaves.get("dirs"), leaves["f_dc"],
                                leaves["f_rest"], leaves.get("opacity"), leaves.get("label"), leaves.get("conf"),
                                camg["world_view_transform"], camg["full_proj_transform"], camg["camera_center"],
                                cam["tanfovx"], cam["tanfovy"], W, H, deg, 1.0, cfg)
    out = projection.project_forward(pi, want_cov3D=True)
    torch.cuda.synchronize()
    flips = int((out["visible"].bool() != mask).sum())
    assert flips <= max(2, mask.numel() // 100000), f"{flips} prefilter decisions differ"       # image-border ties only
    both = out["visible"].bool() & mask
    assert rel_err(out["means2D"], ref["means2D"]) <= 1e-5
    assert rel_err(out["conic"][both], ref["conic"][both]) <= REL_TOL
    assert float(out["conic"][~out["visible"].bool()].abs().sum()) == 0.0
    assert rel_err(out["colors"], ref["colors"]) <= 1e-5
    assert rel_err(out["opacity"], ref["opacity"]) <= 1e-6
    assert rel_err(out["cov3D"], ref["cov3D"]) <= 1e-5

    g = torch.Generator().manual_seed(3)
    gin = {"means2D": torch.randn(ref["means2D"].shape, generator=g).to(dev), "conic": (torch.randn(ref["conic"].shape, generator=g) * 1e-3).to(dev),
           "colors": torch.randn(ref["colors"].shape, generator=g).to(dev), "opacity": torch.randn(ref["opacity"].shape, generator=g).to(dev)}
    gin["means2D"][:, 2] = 0.0
    m = out["visible"].bool()[:, None].float()          # gradients reach exactly the Gaussians the op kept
    loss = sum((ref[k] * gin[k] * m).sum() for k in gin)
    loss.backward()
    # the rasterizer's native conic-gradient layout: (P,2,2) with HALF the off-diagonal derivative at [0][1]
    conic4 = torch.zeros(mask.numel(), 2, 2, device=dev)
    conic4[:, 0, 0] = gin["conic"][:, 0]; conic4[:, 0, 1] = 0.5 * gin["conic"][:, 1]; conic4[:, 1, 1] = gin["conic"][:, 2]
    d = projection.project_backward(pi, out["visible"], dL_dmeans2D=gin["means2D"], dL_dconic4=conic4, dL_dcolors=gin["colors"],
                                    dL_dopacity=gin["opacity"], camera_grads=True, want_means2D_grad=True)
    torch.cuda.synchronize()
    names = {"xyz": "xyz", "scaling": "scaling", "rotation": "rotation", "f_dc": "f_dc", "f_rest": "f_rest", "conf": "conf"}
    names.update({"opacity": "opacity", "label": "label"} if flavour == "gaussian_model" else {"dirs": "dirs"})
    for k, src in names.items():
        gref = leaves[src].grad
        if gref is None:
            gref = torch.zeros_like(leaves[src])
        e = rel_err(d[k].reshape(gref.shape), gref)
        assert e <= REL_TOL, f"{k}: {e}"
    assert rel_err(d["viewmatrix"], camg["world_view_transform"].grad) <= REL_TOL
    assert rel_err(d["projmatrix"], camg["full_proj_transform"].grad) <= REL_TOL
    if deg > 0:
        assert rel_err(d["campos"], camg["camera_center"].grad) <= REL_TOL
    else:
        assert float(d["campos"].abs().max()) == 0.0
    gt = torch.stack([camg["tanfovx"].grad, camg["tanfovy"].grad])
    assert rel_err(d["tanfov"], gt) <= REL_TOL
    assert torch.equal(d["means2D"][:, :2], (gin["means2D"] * m)[:, :2])
    # deterministic camera reduction
    d2 = projection.project_backward(pi, out["visible"], dL_dmeans2D=gin["means2D"], dL_dconic4=conic4, dL_dcolors=gin["colors"],
                                     dL_dopacity=gin["opacity"], camera_grads=True)
    assert torch.equal(d2["viewmatrix"], d["viewmatrix"]) and torch.equal(d2["projmatrix"], d["projmatrix"])


@pytest.mark.parametrize("flavour,strands,W,H,view", [("gaussian_model", 5000, 1920, 1080, 19), ("hair", 5000, 1920, 1080, 3)])
def test_binned_projection_is_bit_identical_to_the_two_kernel_path(cuda_device, flavour, strands, W, H, view):
    """gh_project_forward_binned (projection + the rasterizer's first phase in one pass) against gh_project_forward
    followed by the rasterizer's own preprocess on its outputs: same radii, R, workspaces' content as seen by the
    second phase (the rendered image), bit for bit."""
    from gaussianhaircut_b200 import projection, _C
    synth = _util.synth
    dev = cuda_device
    scene = synth.make_strand_scene(strands, seed=4)
    cam = synth.make_camera(view, W, H)
    cfg = dict(synth.PROJECT_GAUSSIAN_MODEL if flavour == "gaussian_model" else synth.PROJECT_HAIR_MODEL)
    raw = {k: v.to(dev) for k, v in synth.raw_params_from_scene(scene, flavour).items()}
    if flavour == "gaussian_model":
        raw["xyz"][::97] += torch.tensor([0.0, 0.0, -5.0], device=dev)          # some Gaussians behind the camera / culled
    pi = projection.pack_inputs(raw["xyz"], raw["scaling"], raw["rotation"], raw.get("dirs"), raw["f_dc"], raw["f_rest"],
                                raw.get("opacity"), raw.get("label"), raw.get("conf"), cam["world_view_transform"].to(dev),
                                cam["full_proj_transform"].to(dev), cam["camera_center"].to(dev), cam["tanfovx"], cam["tanfovy"],
                                W, H, 3, 1.0, cfg)
    bg = torch.tensor(synth.BG_DEFAULT, device=dev)
    empty = torch.empty(0)
    a = projection.project_forward(pi)
    Ra, color_a, radii_a, geom_a, bin_a, img_a = _C.rasterize_gaussians(
        bg, pi.xyz, empty, a["colors"], a["opacity"], empty, empty, 1.0, empty, a["conic"], pi.V, pi.Pm, cam["tanfovx"], cam["tanfovy"],
        H, W, empty, 3, pi.campos, False, False)
    b, radii_b, geom_b, img_b, Rb, max_len = projection.project_forward_binned(pi)
    color_b, bin_b = _C.forward_render(bg, b["colors"], radii_b, geom_b, img_b, Rb, max_len, H, W)
    torch.cuda.synchronize()
    assert Ra == Rb and Ra > 0
    for k in ("means2D", "colors", "opacity", "conic", "visible"):
        assert torch.equal(a[k], b[k]), k
    assert torch.equal(radii_a, radii_b)
    if flavour == "gaussian_model":
        assert int((radii_a > 0).sum()) < radii_a.numel()                          # view 19 sees the displaced rows behind it: culled rows exist
    assert torch.equal(color_a, color_b)
    assert torch.equal(bin_a[:8 * Ra], bin_b[:8 * Rb])                             # sorted (depth | index) records of every tile


def _weights(H, W, device, seed):
    g = torch.Generator().manual_seed(seed)
    return {k: torch.rand(c, H, W, generator=g).to(device) for k, c in (("render", 3), ("mask", 2), ("orient_angle", 1), ("orient_conf", 1))}


def _loss(pkg, Wt):
    return sum((pkg[k] * Wt[k]).sum() for k in Wt)


def _need_reference():
    if not ref_python.available() or not _util.ref_available():
        pytest.skip("reference Python sources / oracle/_ref not staged")


FUSED_RENDER = [(300, 512, 384), (5000, 1920, 1080)]
GOLDEN = "reference/projection.npz"


def case_key(*params) -> str:
    return "-".join(str(p) for p in params)


def render_gaussian_model(fn, make_model, case, device):
    """One render(cam, pc, pipe, bg) call with `fn` on a model made by `make_model` and the backward of a fixed
    weighted sum of the four maps: (package, model, camera), gradients populated."""
    strands, W, H = case
    synth = _util.synth
    scene = synth.make_strand_scene(strands, seed=3)
    g = torch.Generator().manual_seed(4)
    scene["rotation"] = scene["rotation"] * (0.6 + 0.8 * torch.rand(scene["rotation"].shape[0], 1, generator=g))
    scene["scaling"] = scene["scaling"] * torch.tensor([1.0, 1.0, 1.5])        # three distinct scales: unambiguous arg-max
    cam_d = synth.make_camera(11, W, H)
    bg = torch.tensor(synth.BG_DEFAULT, device=device)
    Wt = _weights(H, W, device, 5)
    pc = make_model(scene, device)
    cam = ref_python.make_camera(cam_d, device, trainable=True)
    pkg = fn(cam, pc, ref_python.pipe(), bg)
    _loss(pkg, Wt).backward()
    torch.cuda.synchronize()
    return pkg, pc, cam


def render_observed(pkg, pc, cam) -> dict:
    """What a trainer reads back from render(), by name."""
    out = {k: pkg[k].detach() for k in ("render", "mask", "orient_conf", "orient_angle", "viewspace_points")}
    out["radii"] = pkg["radii"].int()
    out["visibility_filter"] = pkg["visibility_filter"].int()
    out["viewspace_points.grad"] = pkg["viewspace_points"].grad
    for name in ref_python.MODEL_PARAMS:
        out["grad" + name] = getattr(pc, name).grad
    for name in ("world_view_transform", "full_proj_transform", "camera_center"):
        out["camera." + name] = getattr(cam, name).grad
    return out


@pytest.mark.parametrize("strands,W,H", FUSED_RENDER, ids=["30k-512x384", "500k-1080p"])
def test_fused_render_matches_the_reference_pipeline(cuda_device, strands, W, H):
    """renderer.render (fused projection + this repository's rasterizer) against the reference's render() running
    on the reference's rasterizer: the whole reference pipeline, nothing of the product in it (its results stored
    under tests/golden/reference/projection.npz by tests/golden/make_golden_reference.py)."""
    from gaussianhaircut_b200 import renderer
    pkg, pc, cam = render_gaussian_model(renderer.render, ref_python.plain_gaussian_model, (strands, W, H), cuda_device)
    a = render_observed(pkg, pc, cam)
    every = _util.load_golden(GOLDEN)
    key = case_key(strands, W, H)
    ref = {k[len(key) + 1:]: v for k, v in every.items() if k.startswith(key + "/")}
    n = a["radii"].numel()
    # the number of differing flags, and of radii off by one, estimated through the stored sketches
    assert ref["visibility_filter"].sq_dist(a["visibility_filter"]) <= max(2, n // 100000)
    assert ref["radii"].sq_dist(a["radii"]) <= max(4, n // 20000)                 # ceil() of a radius computed two ways
    for k in ("render", "mask", "orient_conf"):
        e = ref[k].rel_err(a[k])
        assert e <= REL_TOL, f"{k}: {e}"
    assert ref["orient_angle"].rel_err(a["orient_angle"]) <= 1e-3
    assert ref["viewspace_points"].rel_err(a["viewspace_points"]) <= 1e-5
    for name in ref_python.MODEL_PARAMS:
        assert a["grad" + name] is not None, name
        e = ref["grad" + name].rel_err(a["grad" + name])
        assert e <= 2 * REL_TOL, f"{name}: {e}"
    for name in ("world_view_transform", "full_proj_transform", "camera_center"):
        e = ref["camera." + name].rel_err(a["camera." + name])
        assert e <= 2 * REL_TOL, f"camera {name}: {e}"
    assert ref["viewspace_points.grad"].rel_err(a["viewspace_points.grad"]) <= 2 * REL_TOL


def test_fused_render_hair_matches_the_reference_pipeline(cuda_device):
    _need_reference()
    from gaussianhaircut_b200 import renderer
    synth = _util.synth
    W, H = 512, 512
    head = synth.make_blob_scene(20000, seed=2, spread=0.08, max_scale=0.004)
    hair = synth.make_strand_scene(500, seed=4, opacity_mode="ones")
    cam_d = synth.make_camera(7, W, H)
    bg = torch.tensor(synth.BG_DEFAULT, device=cuda_device)
    Wt = _weights(H, W, cuda_device, 9)
    ref_mod = ref_python.load_renderer("ref")
    res = {}
    for which, fn in (("mine", renderer.render_hair), ("ref", ref_mod.render_hair)):
        pc, pc_hair = ref_python.make_hair_models(head, hair, cuda_device)
        cam = ref_python.make_camera(cam_d, cuda_device, trainable=True)
        pkg = fn(cam, pc, pc_hair, ref_python.pipe(), bg)
        _loss(pkg, Wt).backward()
        torch.cuda.synchronize()
        res[which] = (pkg, pc_hair, cam)
    (pa, ha, ca), (pb, hb, cb) = res["mine"], res["ref"]
    assert int((pa["visibility_filter"] != pb["visibility_filter"]).sum()) <= 2
    for k in ("render", "mask", "orient_conf"):
        assert rel_err(pa[k], pb[k]) <= REL_TOL, f"{k}: {rel_err(pa[k], pb[k])}"
    assert rel_err(pa["orient_angle"], pb["orient_angle"]) <= 1e-3
    for name in ref_python.HAIR_PARAMS:
        ga, gb = getattr(ha, name).grad, getattr(hb, name).grad
        assert ga is not None and gb is not None, name
        assert rel_err(ga, gb) <= 2 * REL_TOL, f"{name}: {rel_err(ga, gb)}"
    for name in ("world_view_transform", "full_proj_transform", "camera_center"):
        assert rel_err(getattr(ca, name).grad, getattr(cb, name).grad) <= 2 * REL_TOL, name
    assert rel_err(pa["viewspace_points"].grad, pb["viewspace_points"].grad) <= 2 * REL_TOL


def test_nan_guard_rides_on_the_projection_backward(cuda_device):
    """renderer.set_nan_flag: a NaN anywhere in the parameter gradients raises the device flag during the backward;
    FusedAdam(nan_flag_in=...) then skips the step like the reference trainer (train_gaussians.py:174-181), without a
    pass over the gradients and without a host sync."""
    import types
    from gaussianhaircut_b200 import renderer
    from gaussianhaircut_b200.optim import FusedAdam
    synth = _util.synth
    scene = synth.make_strand_scene(40, seed=6)
    raw = synth.raw_params_from_scene(scene, "gaussian_model")
    cam = ref_python.make_camera(synth.make_camera(3, 160, 96), cuda_device)
    bg = torch.tensor(synth.BG_DEFAULT, device=cuda_device)
    names = ("_xyz", "_features_dc", "_features_rest", "_opacity", "_label", "_scaling", "_rotation", "_orient_conf")
    keys = ("xyz", "f_dc", "f_rest", "opacity", "label", "scaling", "rotation", "conf")
    pc = types.SimpleNamespace(active_sh_degree=3, max_sh_degree=3)
    for n, k in zip(names, keys):
        setattr(pc, n, torch.nn.Parameter(raw[k].to(cuda_device).contiguous()))
    opt = FusedAdam([{"params": [getattr(pc, n)], "lr": 1e-3, "name": n} for n in names], eps=1e-15)
    flag = torch.zeros(1, dtype=torch.int32, device=cuda_device)
    renderer.set_nan_flag(flag)
    try:
        dL = torch.rand(10, 96, 160, device=cuda_device)
        for poisoned in (False, True, False):
            before = pc._xyz.detach().clone()
            renders, _r, _v = renderer.render_raw(cam, pc, types.SimpleNamespace(debug=False), bg)
            g = dL.clone()
            if poisoned:
                g[0, 40:60, 60:100] = float("nan")
            renders.backward(g)
            assert bool(flag.item() != 0) == poisoned
            opt.step(nan_flag_in=flag)
            opt.zero_grad()
            torch.cuda.synchronize()
            assert int(flag.item()) == 0                       # consumed
            assert torch.equal(before, pc._xyz.detach()) == poisoned, "a poisoned step must leave the parameters untouched"
        assert opt.step_count == 2
    finally:
        renderer.set_nan_flag(None)


def test_projection_api_errors(cuda_device):
    from gaussianhaircut_b200 import projection
    synth = _util.synth
    scene = synth.make_strand_scene(2, seed=0)
    raw = synth.raw_params_from_scene(scene, "gaussian_model")
    cam = synth.make_camera(0, 64, 48)
    args = lambda r, dev: (r["xyz"].to(dev), r["scaling"].to(dev), r["rotation"].to(dev), None, r["f_dc"].to(dev), r["f_rest"].to(dev),  # noqa: E731
                           r["opacity"].to(dev), r["label"].to(dev), r["conf"].to(dev), cam["world_view_transform"].to(dev),
                           cam["full_proj_transform"].to(dev), cam["camera_center"].to(dev), cam["tanfovx"], cam["tanfovy"], 64, 48, 3, 1.0,
                           projection.GAUSSIAN_MODEL)
    with pytest.raises(RuntimeError, match="no CPU path"):
        projection.pack_inputs(*args(raw, "cpu"))
    bad = dict(raw, xyz=raw["xyz"].reshape(-1))
    with pytest.raises(RuntimeError, match="means3D must have dimensions"):
        projection.pack_inputs(*args(bad, cuda_device))
    bad = dict(raw, f_rest=raw["f_rest"][:, :8])
    with pytest.raises(RuntimeError, match="features_rest"):
        projection.pack_inputs(*args(bad, cuda_device))
    pi = projection.pack_inputs(*args(raw, cuda_device))
    pi.sh_degree = 4
    with pytest.raises(RuntimeError, match="sh_degree must be 0..3"):
        projection.project_forward(pi)
