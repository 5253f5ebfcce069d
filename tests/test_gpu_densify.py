"""Adaptive density control ("next" row 8f-3): gaussianhaircut_b200.densify against the reference's OWN
`GaussianModel.densify_and_prune` / `reset_opacity` (src/scene/gaussian_model.py:723-737, :516-519), imported unmodified
(oracle/ref_python.py) and run on the GPU with the same seed: every parameter tensor, both Adam moments of every group,
the statistics buffers and the resulting order of the Gaussians must agree -- with torch.optim.Adam (the reference's
optimizer) and with this repository's FusedAdam.  The reference's results are stored under
tests/golden/reference/densify.npz (tests/golden/make_golden_reference.py); the models here are plain namespaces with
the reference's attribute names and optimizer groups."""
import copy
import os
import sys
import types

import pytest
import torch

import _util
from _util import rel_err

pytestmark = pytest.mark.gpu

sys.path.insert(0, os.path.join(_util.ROOT, "oracle"))
import ref_python  # noqa: E402

TRAIN_ARGS = types.SimpleNamespace(percent_dense=0.01, position_lr_init=1.6e-4, position_lr_final=1.6e-6, position_lr_delay_mult=0.01,
                                   position_lr_max_steps=30000, feature_lr=2.5e-3, opacity_lr=0.05, label_lr=0.0025, scaling_lr=0.005,
                                   rotation_lr=0.001, train_orient_conf=True, orient_conf_lr=0.001)
NAMES = ("xyz", "f_dc", "f_rest", "opacity", "label", "scaling", "rotation", "orient_conf")


def model(scene, device, train_orient_conf=True, fused=False, seed=0, reference=False):
    """A GaussianModel with optimizer moments and densification statistics as after a stretch of training.
    reference=True: the reference's own class and optimizer construction (needs its staged sources); otherwise the
    same attributes on a plain namespace and the same Adam groups (gaussian_model.py:426-444)."""
    if reference:
        ref_python.install_stubs()
        src = ref_python.ref_src_dir()
        if src not in sys.path:
            sys.path.insert(0, src)
        pc = ref_python.make_gaussian_model(scene, device)
        pc.spatial_lr_scale = 1.0
        args = copy.copy(TRAIN_ARGS)
        args.train_orient_conf = train_orient_conf
        pc.training_setup(args)                              # the reference's own optimizer construction (:423-448)
    else:
        pc = ref_python.plain_gaussian_model(scene, device)
        pc.percent_dense = TRAIN_ARGS.percent_dense
        a = TRAIN_ARGS
        lrs = [("xyz", a.position_lr_init), ("f_dc", a.feature_lr), ("f_rest", a.feature_lr / 20.0), ("opacity", a.opacity_lr),
               ("label", a.label_lr), ("scaling", a.scaling_lr), ("rotation", a.rotation_lr)]
        if train_orient_conf:
            lrs.append(("orient_conf", a.orient_conf_lr))
        pc.optimizer = torch.optim.Adam([{"params": [getattr(pc, densify_groups()[n])], "lr": lr, "name": n} for n, lr in lrs],
                                        lr=0.0, eps=1e-15)
    if fused:
        from gaussianhaircut_b200.optim import FusedAdam
        pc.optimizer = FusedAdam([{"params": g["params"], "lr": g["lr"], "name": g["name"]} for g in pc.optimizer.param_groups], eps=1e-15)
    g = torch.Generator().manual_seed(seed)
    for it in range(3):                                      # populate exp_avg / exp_avg_sq
        for grp in pc.optimizer.param_groups:
            p = grp["params"][0]
            p.grad = (torch.randn(p.shape, generator=g) * 0.01).to(device)
        pc.optimizer.step()
    P = pc._xyz.shape[0]
    pc.xyz_gradient_accum = (torch.rand(P, 1, generator=g) * 6e-4).to(device)
    pc.denom = torch.randint(0, 3, (P, 1), generator=g).float().to(device)        # zeros included: 0/0 -> NaN -> 0
    pc.max_radii2D = (torch.rand(P, generator=g) * 40).to(device)
    return pc


def densify_groups():
    from gaussianhaircut_b200 import densify
    return densify.GROUPS


def scene(n, seed):
    synth = _util.synth
    sc = synth.make_blob_scene(n, seed=seed, spread=0.2, max_scale=0.02)
    g = torch.Generator().manual_seed(seed + 1)
    sc["scaling"] = sc["scaling"] * torch.exp(torch.randn(n, 1, generator=g))           # spread of sizes around the density threshold
    sc["opacity"] = torch.sigmoid(torch.randn(n, 1, generator=g) * 3 - 1)               # some below min_opacity
    return sc


def case_key(*params) -> str:
    return "-".join(str(p) for p in params)


def _step(pc):
    """One optimizer step with seeded gradients (the model must keep training after the surgery)."""
    g = torch.Generator().manual_seed(99)
    for grp in pc.optimizer.param_groups:
        grp["params"][0].grad = (torch.randn(grp["params"][0].shape, generator=g) * 0.01).to(grp["params"][0].device)
    pc.optimizer.step()
    torch.cuda.synchronize()


def densify_observed(pc, step=True) -> dict:
    """Every parameter and both Adam moments by group name, the statistics buffers and orient_conf; with step=True
    also the parameters after one more optimizer step ('stepped.<name>')."""
    out = {}
    for grp in pc.optimizer.param_groups:
        p = grp["params"][0]
        out[grp["name"]] = p.detach().clone()
        for k in ("exp_avg", "exp_avg_sq"):
            out[grp["name"] + "." + k] = pc.optimizer.state[p][k].clone()
    for n in ("xyz_gradient_accum", "denom", "max_radii2D"):
        out[n] = getattr(pc, n).clone()
    out["_orient_conf"] = pc._orient_conf.detach().clone()
    if step:
        _step(pc)
        for grp in pc.optimizer.param_groups:
            out["stepped." + grp["name"]] = grp["params"][0].detach().clone()
    return out


_golden = {}


def golden(key):
    """The reference's results of one case (tests/golden/reference/densify.npz, tests/golden/make_golden_reference.py)."""
    if not _golden:
        _golden.update(_util.load_golden("reference/densify.npz"))
    return {k[len(key) + 1:]: v for k, v in _golden.items() if k.startswith(key + "/")}


def _compare(ref, b, fused_b):
    assert ref["xyz"].shape == tuple(b._xyz.shape), f"{ref['xyz'].shape} vs {tuple(b._xyz.shape)}"
    gb = {g["name"]: g for g in b.optimizer.param_groups}
    assert set(gb) == {k for k in ref if "." not in k and k in densify_groups()}
    for n in gb:
        pb = gb[n]["params"][0]
        assert ref[n].shape == tuple(pb.shape), n
        e = ref[n].rel_err(pb.detach())
        assert e <= 1e-6, f"{n}: {e}"
        assert getattr(b, densify_groups()[n]) is pb
        sb = b.optimizer.state[pb]
        for k in ("exp_avg", "exp_avg_sq"):
            assert ref[n + "." + k].shape == tuple(sb[k].shape) == tuple(pb.shape)
            tol = 1e-6 if not fused_b else 5e-5          # FusedAdam's moments differ from torch's by rounding before the surgery
            e = ref[n + "." + k].rel_err(sb[k])
            assert e <= tol, f"{n}.{k}: {e}"
    for n in ("xyz_gradient_accum", "denom", "max_radii2D"):
        assert ref[n].shape == tuple(getattr(b, n).shape) and float(getattr(b, n).abs().sum()) == 0.0, n
    assert ref["_orient_conf"].shape == tuple(b._orient_conf.shape) and ref["_orient_conf"].rel_err(b._orient_conf.detach()) <= 1e-6


DENSIFY = [(20000, 20, True, False), (20000, None, True, False), (20000, 20, False, False), (20000, 20, True, True), (7, 20, True, False)]


@pytest.mark.parametrize("n,max_screen_size,train_conf,fused", DENSIFY)
def test_densify_and_prune_matches_the_reference(cuda_device, n, max_screen_size, train_conf, fused):
    from gaussianhaircut_b200 import densify
    b = model(scene(n, seed=3), cuda_device, train_conf, fused=fused, seed=7)
    torch.manual_seed(123); torch.cuda.manual_seed(123)
    counts = densify.densify_and_prune(b, 2e-4, 0.005, 2.0, max_screen_size)
    torch.cuda.synchronize()
    ref = golden(case_key(n, max_screen_size, train_conf))
    assert (counts["total"],) == ref["xyz"].shape[:1]
    if n >= 1000:
        assert counts["cloned"] > 0 and counts["children"] > 0 and counts["kept"] < n, counts     # every branch exercised
    _compare(ref, b, fused)
    # the model keeps training like the reference's afterwards (optimizer state re-keyed correctly)
    _step(b)
    for grp in b.optimizer.param_groups:
        assert ref["stepped." + grp["name"]].rel_err(grp["params"][0].detach()) <= 1e-6, grp["name"]


def test_reserved_pools_are_used_and_change_nothing(cuda_device):
    """densify.reserve_pools: the rebuilt tensors live in the buffers allocated up front (no allocation inside the
    call), results identical to the un-reserved path."""
    from gaussianhaircut_b200 import densify
    sc = scene(20000, seed=3)
    a = model(sc, cuda_device, True, fused=True, seed=7)
    b = model(sc, cuda_device, True, fused=True, seed=7)
    densify.reserve_pools(b, 400000)
    slots = {k: [t.data_ptr() for t in v] for k, v in b._gh_pools.items()}
    assert all(len(v) == 2 and v[0] != v[1] for v in slots.values()) and len(slots) == 3 * 8
    for rnd in range(3):                                   # source and destination alternate between the two slots
        for pc in (a, b):
            torch.manual_seed(5 + rnd); torch.cuda.manual_seed(5 + rnd)
            P = pc._xyz.shape[0]
            g = torch.Generator().manual_seed(rnd)
            pc.xyz_gradient_accum = (torch.rand(P, 1, generator=g) * 6e-4).to(cuda_device)
            pc.denom = torch.randint(1, 3, (P, 1), generator=g).float().to(cuda_device)
            densify.densify_and_prune(pc, 2e-4, 0.005, 2.0, 20)
        assert a._xyz.shape == b._xyz.shape
        for name in NAMES:
            pa = [g for g in a.optimizer.param_groups if g["name"] == name][0]["params"][0]
            pb = [g for g in b.optimizer.param_groups if g["name"] == name][0]["params"][0]
            assert torch.equal(pa.detach(), pb.detach()), name
            assert torch.equal(a.optimizer.state[pa]["exp_avg_sq"], b.optimizer.state[pb]["exp_avg_sq"]), name
            assert pb.data_ptr() in slots[name], name      # still inside the reserved buffers
            assert b.optimizer.state[pb]["exp_avg"].data_ptr() in slots[name + ".exp_avg"], name
    assert {k: [t.data_ptr() for t in v] for k, v in b._gh_pools.items()} == slots


def test_reset_opacity_matches_the_reference(cuda_device):
    from gaussianhaircut_b200 import densify
    b = model(scene(5000, seed=5), cuda_device, True, seed=2)
    densify.reset_opacity(b)
    ref = golden("reset_opacity")
    assert ref["opacity"].rel_err(b._opacity.detach()) <= 1e-6
    pb = [g for g in b.optimizer.param_groups if g["name"] == "opacity"][0]["params"][0]
    assert pb is b._opacity and float(b.optimizer.state[pb]["exp_avg"].abs().sum()) == 0.0
    assert ref["opacity.exp_avg_sq"].equal(b.optimizer.state[pb]["exp_avg_sq"])


def test_densify_at_config5_scale(cuda_device):
    """BASELINE config 5 scale (2M Gaussians): same outcome as the reference, and the time (informational)."""
    import time
    from gaussianhaircut_b200 import densify
    b = model(scene(2_000_000, seed=11), cuda_device, True, seed=1)
    torch.manual_seed(5); torch.cuda.manual_seed(5)
    torch.cuda.synchronize(); t0 = time.time()
    counts = densify.densify_and_prune(b, 2e-4, 0.005, 2.0, 20)
    torch.cuda.synchronize(); t_mine = time.time() - t0
    print(f"\\n[densify 2M] fused {t_mine * 1e3:.1f} ms, counts {counts}")
    _compare(golden("config5"), b, False)
