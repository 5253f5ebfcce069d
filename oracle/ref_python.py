"""TEST INFRASTRUCTURE ONLY -- runs the reference's own Python callers of the hot path UNMODIFIED.

`src/gaussian_renderer/__init__.py` (`render` :23, `render_hair` :116) and the model classes it drives
(`src/scene/gaussian_model.py:45`, `src/scene/gaussian_model_latent_strands.py:28`) are imported as they
are, from /root/reference/src in the build container, or from the copy that `oracle/build_ref.py`
stages under oracle/_ref/src (git-ignored build output, the pure-Python half of "installing" the
reference; it travels to the GPU box like oracle/_ref's compiled extension).  Nothing of it is part of
the product; only tests/, bench.py's reference arm and tools/ import this module.

* Third-party modules the reference imports at module scope but that the render path never calls are
  absent from the image (plyfile, simple_knn, pytorch3d, NeuS, trimesh, pysdf, src.hair_networks.*):
  they are stubbed in sys.modules.
* `gaussian_renderer` binds `diff_gaussian_rasterization` at import time, so it is loaded once per
  rasterizer under a private module name: "mine" = this repository's drop-in package, "ref" = the
  reference's own extension built in oracle/_ref.
"""
from __future__ import annotations

import importlib.util
import math
import os
import sys
import types

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REF_SRC_LIVE = "/root/reference/src"
REF_SRC_STAGED = os.path.join(HERE, "_ref", "src")

STUBS = ("plyfile", "simple_knn", "simple_knn._C", "pytorch3d", "pytorch3d.io", "pytorch3d.ops", "NeuS", "NeuS.models",
         "NeuS.models.dataset", "src", "src.hair_networks", "src.hair_networks.optimizable_textured_strands",
         "src.hair_networks.strand_prior", "trimesh", "pysdf", "lpips", "kaolin", "skimage", "matplotlib",
         "matplotlib.pyplot", "easydict", "pyhocon", "face_alignment")


def ref_src_dir():
    for d in (REF_SRC_LIVE, REF_SRC_STAGED):
        if os.path.isfile(os.path.join(d, "gaussian_renderer", "__init__.py")):
            return d
    return None


def available() -> bool:
    return ref_src_dir() is not None


class _AnyModule(types.ModuleType):
    """Stub: any attribute is an empty class (enough for `from x import Y` at module scope)."""

    def __getattr__(self, k):
        if k.startswith("__"):
            raise AttributeError(k)
        return type(k, (), {})


def install_stubs():
    for name in STUBS:
        if name in sys.modules:
            continue
        try:
            if importlib.util.find_spec(name) is not None:
                continue
        except (ImportError, ValueError, AttributeError):
            pass
        m = _AnyModule(name)
        m.__path__ = []
        sys.modules[name] = m


_renderers = {}


def load_renderer(which: str = "mine"):
    """The reference's `gaussian_renderer` module bound to the chosen rasterizer ("mine" | "ref")."""
    if which in _renderers:
        return _renderers[which]
    src = ref_src_dir()
    if src is None:
        raise RuntimeError("reference Python sources not available (neither /root/reference/src nor oracle/_ref/src)")
    install_stubs()
    if src not in sys.path:
        sys.path.insert(0, src)
    if ROOT not in sys.path:
        sys.path.insert(0, ROOT)
    if which == "mine":
        import diff_gaussian_rasterization as rast           # this repository's drop-in package
        assert os.path.dirname(os.path.dirname(os.path.abspath(rast.__file__))) == ROOT
    elif which == "ref":
        if HERE not in sys.path:
            sys.path.insert(0, HERE)
        import build_ref
        rast = build_ref.load()
    else:
        raise ValueError(which)
    saved = sys.modules.get("diff_gaussian_rasterization")
    sys.modules["diff_gaussian_rasterization"] = rast
    try:
        name = f"gh_ref_gaussian_renderer_{which}"
        spec = importlib.util.spec_from_file_location(name, os.path.join(src, "gaussian_renderer", "__init__.py"))
        mod = importlib.util.module_from_spec(spec)
        sys.modules[name] = mod
        spec.loader.exec_module(mod)
    finally:
        if saved is not None:
            sys.modules["diff_gaussian_rasterization"] = saved
        else:
            sys.modules.pop("diff_gaussian_rasterization", None)
    assert mod.GaussianRasterizer is rast.GaussianRasterizer
    _renderers[which] = mod
    return mod


# ------------------------------------------------------------------------------------------- model / camera builders
def make_camera(cam_d: dict, device, trainable: bool = False):
    """A duck-typed viewpoint camera with the attributes `render()` reads (src/scene/cameras.py:21-150):
    image_width/height, FoVx/FoVy (tensors), world_view_transform, full_proj_transform, camera_center.
    `trainable=True` makes the three matrices/vectors autograd leaves (the reference's trainable cameras
    produce them differentiably, cameras.py:124-150)."""
    import torch
    leaf = (lambda t: t.detach().clone().to(device).requires_grad_(True)) if trainable else (lambda t: t.to(device))
    return types.SimpleNamespace(
        image_width=int(cam_d["image_width"]), image_height=int(cam_d["image_height"]),
        FoVx=torch.tensor(float(cam_d["FoVx"]), device=device), FoVy=torch.tensor(float(cam_d["FoVy"]), device=device),
        world_view_transform=leaf(cam_d["world_view_transform"]), full_proj_transform=leaf(cam_d["full_proj_transform"]),
        camera_center=leaf(cam_d["camera_center"]))


def make_gaussian_model(scene: dict, device, sh_degree: int = 3, active_sh_degree: int = 3):
    """A real reference `GaussianModel` (scene/gaussian_model.py:45) whose parameters are set from a seeded
    synthetic scene the way `create_from_pcd` / `load_ply` set them (:409-419, :569-577): raw log-scales,
    raw quaternions, logit opacities / labels, log orientation confidences."""
    from scene.gaussian_model import GaussianModel
    return fill_gaussian_model(GaussianModel(sh_degree), scene, device, active_sh_degree)


def fill_gaussian_model(pc, scene: dict, device, active_sh_degree: int = 3):
    """Set the parameters of `pc` (a GaussianModel, or any object with its attribute names) from a seeded scene."""
    import torch
    from torch import nn
    P = lambda t: nn.Parameter(t.detach().clone().to(device).contiguous().requires_grad_(True))  # noqa: E731
    logit = lambda p: torch.log(p / (1 - p))  # noqa: E731
    pc._xyz = P(scene["xyz"])
    pc._features_dc = P(scene["f_dc"])
    pc._features_rest = P(scene["f_rest"])
    pc._scaling = P(torch.log(scene["scaling"]))
    pc._rotation = P(scene["rotation"])
    pc._opacity = P(logit(scene["opacity"].clamp(1e-6, 1 - 1e-6)))
    pc._label = P(logit(scene["label"].clamp(1e-6, 1 - 1e-6)))
    pc._orient_conf = P(torch.log(scene["orient_conf"]))
    pc.active_sh_degree = active_sh_degree
    pc.max_radii2D = torch.zeros(pc._xyz.shape[0], device=device)
    return pc


def plain_gaussian_model(scene: dict, device, sh_degree: int = 3):
    """The GaussianModel attributes that this repository's renderer and densification read, on a plain namespace
    (no reference sources needed)."""
    return fill_gaussian_model(types.SimpleNamespace(max_sh_degree=sh_degree), scene, device, sh_degree)


MODEL_PARAMS = ("_xyz", "_features_dc", "_features_rest", "_scaling", "_rotation", "_opacity", "_label", "_orient_conf")


def make_hair_models(head_scene: dict, hair_scene: dict, device, sh_degree: int = 3):
    """The two models `render_hair()` consumes (gaussian_renderer/__init__.py:116-236):
    `pc` = a frozen GaussianModel with the *_precomp attributes the strand trainers attach
    (train_strands.py:67-73) and `pc_hair` = a `GaussianModelHair` (scene/gaussian_model_latent_strands.py:28)
    whose per-Gaussian tensors are set directly the way `initialize_gaussians_hair` leaves them (:486-504)
    -- its strand-prior networks are external code that is absent, so `__init__` is bypassed."""
    import torch
    from scene.gaussian_model_latent_strands import GaussianModelHair
    pc = make_gaussian_model(head_scene, device, sh_degree)
    with torch.no_grad():
        pc.mask_precomp = pc.get_label[..., 0] < 0.5
        pc.xyz_precomp = pc.get_xyz[pc.mask_precomp].detach()
        pc.opacity_precomp = pc.get_opacity[pc.mask_precomp].detach()
        pc.scaling_precomp = pc.get_scaling[pc.mask_precomp].detach()
        pc.rotation_precomp = pc.get_rotation[pc.mask_precomp].detach()
        pc.shs_view = pc.get_features[pc.mask_precomp].detach().transpose(1, 2).view(-1, 3, (pc.max_sh_degree + 1) ** 2)
    hair = GaussianModelHair.__new__(GaussianModelHair)
    hair.setup_functions()
    hair.active_sh_degree = sh_degree
    hair.max_sh_degree = sh_degree
    leaf = lambda t: t.detach().clone().to(device).contiguous().requires_grad_(True)  # noqa: E731
    hair._xyz = leaf(hair_scene["xyz"])
    hair._dir = leaf(hair_scene["dir"])
    hair.scale = float(hair_scene["scaling"][0, 1]) * torch.ones(1, device=device)          # create_from_pcd :510-515
    from utils.general_utils import parallel_transport
    ex = torch.cat([torch.ones_like(hair._xyz[:, :1]), torch.zeros_like(hair._xyz[:, :2])], dim=-1)
    hair._rotation = parallel_transport(a=ex, b=hair._dir).view(-1, 4)                          # initialize_gaussians_hair :489-498
    hair._features_dc = leaf(hair_scene["f_dc"])
    hair._features_rest = leaf(hair_scene["f_rest"])
    hair._orient_conf = leaf(torch.log(hair_scene["orient_conf"]))
    return pc, hair


HAIR_PARAMS = ("_xyz", "_dir", "_features_dc", "_features_rest", "_orient_conf")


def pipe(debug: bool = False):
    return types.SimpleNamespace(debug=debug, convert_SHs_python=False, compute_cov3D_python=False)


def focal_fov(width: int, height: int, focal: float):
    return 2.0 * math.atan(width / (2.0 * focal)), 2.0 * math.atan(height / (2.0 * focal))
