"""The rasterizer's forward and backward against Oracle-B (oracle/gh_oracle.c, the serial CPU restatement of the
reference rasterizer) at the shapes where the blend kernels are most likely to go wrong: image sizes that are
odd, smaller than a tile or one pixel past it; per-tile lists whose length sits on the forward's 256-record
staging chunks and the backward's 384-record windows; early termination at those positions; clamped and skipped
alphas; and small Gaussian counts.

The reference is computed at test time on the CPU for every case, so each check covers every element:
  * bit for bit: num_rendered, radii, tile keys, point list, ranges, n_contrib, and for visible Gaussians the
    depths, 2-D means and conic/opacity;
  * the maps: out_color within 1e-5 * max|ref| per channel, final_T within 1e-6 (the oracle's exp is correctly
    rounded, CUDA's is ex2.approx; the same bounds tests/test_oracle_cpu.py holds the oracle to);
  * the nine gradients: norm-relative <= 1e-4 and |delta| <= 1e-4 * max|ref| at every element; a gradient that
    is zero in the oracle must be exactly zero.
Every scene also checks that it reaches the path it is named for.
"""
import math

import numpy as np
import pytest
import torch

import _util
from _util import GRAD_NAMES

pytestmark = pytest.mark.gpu

synth = _util.synth
REL_TOL = 1e-4
MAP_TOL = 1e-5
FINAL_T_TOL = 1e-6


@pytest.fixture(scope="module")
def oracle():
    import oracle as _oracle
    _oracle.build()
    return _oracle


# ------------------------------------------------------------------------------------------------ scene builders
def pixel_scene(px, py, z, sx, sy, W, H, opacity, seed=0, focal=None, rotate=True):
    """Gaussians placed in pixel space for camera 0: centre (px, py) in pixels (the reference's pixel (x, y) has its
    centre at (x, y)), camera depth z, screen-space scales sx, sy in pixels.  Returns (scene, camera)."""
    P = len(px)
    f = float(focal if focal is not None else 1.2 * max(W, H))
    px, py, z = (torch.as_tensor(a, dtype=torch.float64) for a in (px, py, z))
    x_cam = z * (2 * px + 1 - W) / (2 * f)
    y_cam = z * (2 * py + 1 - H) / (2 * f)
    scene = synth.make_blob_scene(P, seed=seed)
    scene["xyz"] = torch.stack([-x_cam, y_cam, 0.8 - z], 1).float()     # camera 0: x_w = -x_cam, y_w = y_cam, z_w = 0.8 - z_cam
    s = torch.stack([torch.as_tensor(sx, dtype=torch.float64), torch.as_tensor(sy, dtype=torch.float64),
                     torch.full((P,), 0.5, dtype=torch.float64)], 1) * (z / f)[:, None]
    scene["scaling"] = s.float().contiguous()
    if not rotate:
        scene["rotation"] = torch.tensor([[1.0, 0.0, 0.0, 0.0]]).repeat(P, 1)
    scene["opacity"] = torch.as_tensor(opacity, dtype=torch.float32).reshape(P, 1).contiguous()
    return scene, synth.make_camera(0, W, H, focal_factor=f / H)


def inputs(scene, cam, mode, device, bg=None):
    inp = synth.rasterizer_inputs(scene, cam, mode=mode, device=device)
    if bg is not None:
        inp["settings"]["bg"] = torch.as_tensor(bg, dtype=torch.float32, device=device)
    return inp


def upstream(W, H, seed):
    """dL/d(out) with negative values, an all-zero channel and scattered zeros."""
    g = torch.Generator().manual_seed(500 + seed)
    dL = torch.rand(10, H, W, generator=g) * 2 - 1
    dL[4] = 0.0
    dL[torch.rand(10, H, W, generator=g) < 0.1] = 0.0
    return dL


def size_scene(W, H, seed):
    """Random splats over and around a W x H image: centres up to 8 pixels outside it, screen sizes from a fraction of
    a pixel to about a tile, some straddling tile borders."""
    g = np.random.default_rng(seed)
    P = int(min(300, 12 + W * H // 6))
    px = g.uniform(-8.0, W + 7.0, P)
    py = g.uniform(-8.0, H + 7.0, P)
    # one splat each just right of the last column, just below the last row and past the corner, reaching in
    px[:3] = [W + 1.5, g.uniform(0, W - 1), W + 2.0]
    py[:3] = [g.uniform(0, H - 1), H + 1.5, H + 2.0]
    sx = g.uniform(0.3, 6.0, P)
    sy = g.uniform(0.3, 6.0, P)
    z = 0.4 + 0.3 * g.permutation(P) / P
    op = g.uniform(0.05, 1.0, P)
    return pixel_scene(px, py, z, sx, sy, W, H, op, seed=seed)


def list_scene(L, seed=0):
    """One 16 x 16 tile holding L records, every one of which every pixel blends: wide splats (60..200 px) centred
    inside the tile with opacity 0.00405..0.0043, so alpha >= 0.00398 > 1/255 at every pixel and
    T >= (1 - 0.0043)^2048 > 1e-4 after the whole list."""
    g = np.random.default_rng(100 + seed)
    px = g.uniform(0.0, 15.0, L)
    py = g.uniform(0.0, 15.0, L)
    s = g.uniform(60.0, 200.0, (2, L))
    z = 0.4 + 0.3 * np.arange(L) / L
    op = g.uniform(0.00405, 0.0043, L)
    return pixel_scene(px, py, z, s[0], s[1], 16, 16, op, seed=seed, rotate=False)


def termination_inputs(targets, n_total, device, seed=0):
    """One 16 x 16 tile ('render' call shape): a haze of wide splats with alpha ~0.004 at every pixel, and for pixel i
    two opaque splats centred on it (alpha 0.99) whose supplied conic (40, 0, 40) leaves every other pixel alone.
    The second sits at list position targets[i] (depth order is list order), the first up to 40 positions earlier,
    so pixel i's test_T falls below 1e-4 at targets[i]."""
    g = np.random.default_rng(200 + seed)
    slot_px = np.full(n_total, 7.5); slot_py = np.full(n_total, 7.5)
    slot_s = np.full(n_total, 150.0); slot_op = np.full(n_total, 0.004)
    used = set(int(t) for t in targets)
    assert len(used) == len(targets)
    before = set(int(t) - 1 for t in targets)          # kept for the haze: the record before a target is blended
    sharp = np.zeros(n_total, bool)
    for i, t in enumerate(targets):
        first = int(t) - int(g.integers(2, 40))
        while first in used or first in before:
            first -= 1
        used.add(first)
        for slot in (first, int(t)):
            assert 0 <= slot < n_total
            slot_px[slot], slot_py[slot], slot_s[slot], slot_op[slot], sharp[slot] = i % 16, i // 16, 0.05, 1.0, True
    z = 0.4 + 0.3 * np.arange(n_total) / n_total
    scene, cam = pixel_scene(slot_px, slot_py, z, slot_s, slot_s, 16, 16, slot_op, seed=seed, rotate=False)
    inp = inputs(scene, cam, "render", device, bg=np.linspace(1.0, 0.1, 10))
    assert bool(inp["mask"].all())
    inp["kwargs"]["conic_precomp"][torch.from_numpy(sharp).to(device)] = torch.tensor([40.0, 0.0, 40.0], device=device)
    return inp


# ------------------------------------------------------------------------------------------------ running both
def _np(t):
    return None if t is None else t.detach().cpu().numpy()


def run_both(oracle, inp, dL):
    import gaussianhaircut_b200._C as native
    kw, s = inp["kwargs"], inp["settings"]
    W, H = s["image_width"], s["image_height"]
    P = kw["means3D"].shape[0]
    r = native.rasterize_gaussians(*_util.native_args(inp))
    dLd = dL.to(kw["means3D"].device)
    g = native.rasterize_gaussians_backward(*_util.backward_args(inp, r[2], dLd, r[3], r[0], r[4], r[5]))
    torch.cuda.synchronize()
    st = {k: v.cpu().numpy() for k, v in native.debug_export(P, W, H, r[0], r[3], r[4], r[5]).items()}
    mine = {"R": int(r[0]), "color": _np(r[1]), "radii": _np(r[2]), "state": st,
            "grads": {n: _np(t) for n, t in zip(GRAD_NAMES, g)}}
    okw = dict(scales=_np(kw["scales"]), rotations=_np(kw["rotations"]), cov3D_precomp=_np(kw["cov3D_precomp"]),
               conic_precomp=_np(kw["conic_precomp"]), scale_modifier=float(s["scale_modifier"]))
    args = (_np(s["viewmatrix"]), _np(s["projmatrix"]), s["tanfovx"], s["tanfovy"], W, H, _np(s["bg"]))
    fw = oracle.forward(_np(kw["means3D"]), _np(kw["opacities"]), _np(kw["colors_precomp"]), *args, **okw)
    bw = oracle.backward(fw, dL.numpy(), _np(kw["means3D"]), _np(kw["colors_precomp"]), *args, **okw)
    return mine, fw, bw


def _near_ties(fw, W, pix):
    """Records of pixel `pix`'s tile list whose alpha or test_T, evaluated in float32 from the oracle's state, lies
    within 2 ulp of the reference's thresholds 1/255 and 1e-4: decisions the CPU's exp cannot reproduce."""
    f32 = np.float32
    x, y = pix % W, pix // W
    gx = (W + 15) // 16
    lo, hi = fw["ranges"][(y // 16) * gx + x // 16]
    T = f32(1.0)
    found = []
    for k in range(int(lo), int(hi)):
        i = int(fw["point_list"][k])
        mx, my = fw["means2D"][i]
        a, b, c, o = fw["conic_opacity"][i]
        dx, dy = f32(mx - f32(x)), f32(my - f32(y))
        power = f32(f32(-0.5) * f32(f32(a * dx) * dx + f32(c * dy) * dy) - f32(b * dx) * dy)
        if power > 0:
            continue
        alpha = min(f32(0.99), f32(o * f32(math.exp(float(power)))))
        near_a = abs(alpha - f32(1 / 255.0)) <= 2 * np.spacing(f32(1 / 255.0))
        if alpha < f32(1 / 255.0) and not near_a:
            continue
        test_T = f32(T * f32(1 - alpha))
        near_t = abs(test_T - f32(1e-4)) <= 2 * np.spacing(f32(1e-4))
        if near_a or near_t:
            found.append(f"record {k - lo} (Gaussian {i}): alpha {alpha!r}{' ~ 1/255' if near_a else ''}, "
                         f"test_T {test_T!r}{' ~ 1e-4' if near_t else ''}")
        if test_T < f32(1e-4):
            break
        T = test_T
    return found


def check_all(mine, fw, bw, W, H):
    st = mine["state"]
    assert mine["R"] == fw["num_rendered"], f"num_rendered {mine['R']} vs oracle {fw['num_rendered']}"
    assert np.array_equal(mine["radii"], fw["radii"]), "radii differ"
    vis = fw["radii"] > 0
    for k in ("depths", "means2D", "conic_opacity"):
        assert np.array_equal(st[k].view(np.uint32)[vis], fw[k].view(np.uint32)[vis]), f"{k} bits differ"
    assert np.array_equal(st["keys"].view(np.uint64), fw["keys"]), "tile keys differ"
    assert np.array_equal(st["point_list"].view(np.uint32), fw["point_list"]), "point list differs"
    assert np.array_equal(st["ranges"].view(np.uint32).reshape(-1, 2), fw["ranges"]), "tile ranges differ"
    nc_m, nc_r = st["n_contrib"].view(np.uint32).reshape(-1), fw["n_contrib"]
    bad = np.nonzero(nc_m != nc_r)[0]
    if bad.size:
        lines = [f"pixel ({p % W}, {p // W}): n_contrib {nc_m[p]} vs oracle {nc_r[p]}; near ties: "
                 f"{_near_ties(fw, W, int(p)) or 'none'}" for p in bad[:4]]
        raise AssertionError(f"n_contrib differs at {bad.size} pixels (a near tie means: move the scene)\n" + "\n".join(lines))
    dT = np.abs(st["final_T"].reshape(-1) - fw["final_T"]).max()
    assert dT <= FINAL_T_TOL, f"final_T differs by {dT}"
    col_m, col_r = mine["color"].astype(np.float64), fw["out_color"].astype(np.float64)
    assert col_m.shape == (10, H, W)
    for ch in range(10):
        scale = max(np.abs(col_r[ch]).max(), 1e-12)
        e = np.abs(col_m[ch] - col_r[ch]).max() / scale
        assert e <= MAP_TOL, f"out_color channel {ch}: max error {e} of max|ref|"
    for name in GRAD_NAMES:
        gm, gr = mine["grads"][name], bw[name]
        assert gm.shape == gr.shape, f"{name}: shape {gm.shape} vs {gr.shape}"
        if gr.size == 0:
            continue
        gm, gr = gm.astype(np.float64), gr.astype(np.float64)
        if not gr.any():
            assert not gm.any(), f"{name}: the oracle's gradient is zero, the kernel's is not"
            continue
        e = np.linalg.norm(gm - gr) / np.linalg.norm(gr)
        assert e <= REL_TOL, f"{name}: norm-relative error {e}"
        worst = np.abs(gm - gr).max() / np.abs(gr).max()
        where = np.unravel_index(np.abs(gm - gr).argmax(), gr.shape)
        assert worst <= REL_TOL, f"{name}: element {where} off by {worst} of max|ref|"


# ------------------------------------------------------------------------------------------------ image sizes
SIZES = [(1, 1), (1, 37), (37, 1), (15, 15), (16, 16), (17, 17), (31, 33), (33, 31), (161, 97), (251, 187)]


@pytest.mark.parametrize("mode", ["native", "render", "cov3d"])
@pytest.mark.parametrize("W,H", SIZES, ids=[f"{w}x{h}" for w, h in SIZES])
def test_image_sizes(cuda_device, oracle, W, H, mode):
    """Odd widths and heights, images smaller than a tile and one pixel past it: the backward's 2 x 2 blocks in the
    right-hand column (odd W) or bottom row (odd H) lie half outside the image."""
    scene, cam = size_scene(W, H, seed=W * 1000 + H + 7)
    inp = inputs(scene, cam, mode, cuda_device, bg=np.linspace(-0.5, 2.0, 10))
    mine, fw, bw = run_both(oracle, inp, upstream(W, H, W + H))
    nc = fw["n_contrib"].reshape(H, W)
    assert nc[:, -1].any() and nc[-1, :].any(), "nothing is blended in the last row / column"
    vis = fw["radii"] > 0
    m2 = fw["means2D"]
    off = vis & ((m2[:, 0] < -0.5) | (m2[:, 0] > W - 0.5) | (m2[:, 1] < -0.5) | (m2[:, 1] > H - 0.5))
    assert off.any(), "no splat with its centre off-screen reaches into the image"
    if W > 16 or H > 16:
        assert (fw["tiles_touched"][vis] > 1).any(), "no splat straddles a tile border"
    check_all(mine, fw, bw, W, H)


# ------------------------------------------------------------------------------------------------ staging boundaries
LIST_LENGTHS = [1, 255, 256, 257, 383, 384, 385, 511, 512, 513, 767, 768, 769, 1151, 1152, 1153, 2047, 2048]


@pytest.mark.parametrize("L", LIST_LENGTHS)
def test_list_length_at_staging_boundaries(cuda_device, oracle, L):
    """One tile with L records, every one blended by every pixel: the forward stages 256-record chunks (double
    buffered, ids prefetched two chunks ahead), the backward walks 384-record windows from the last to the first,
    the last one holding n - 384 * (windows - 1) records."""
    scene, cam = list_scene(L)
    inp = inputs(scene, cam, "native", cuda_device, bg=np.linspace(0.25, 1.0, 10))
    # colours of one sign: the map is then not a small difference of up to 2048 terms, and the 1e-5 * max|ref| bound
    # measures the blend rather than cancellation
    inp["kwargs"]["colors_precomp"].abs_()
    mine, fw, bw = run_both(oracle, inp, upstream(16, 16, L))
    rg = fw["ranges"]
    assert int(rg[0, 1] - rg[0, 0]) == L, "the tile does not hold L records"
    assert int(fw["n_contrib"].max()) == L, f"max(n_contrib) {fw['n_contrib'].max()} != L"
    check_all(mine, fw, bw, 16, 16)


TERMINATION = [
    # end positions around the forward's chunk boundaries (256, 512, 768) and the backward's window boundaries
    # (384, 768, 1152); the remaining pixels end at random positions in [100, last)
    (np.r_[254:259:2, 382:387:2, 510:515:2, 766:771:2, 1150:1155:2], 1300),
    (np.r_[255:258:2, 383:386:2, 767:770:2], 900),
]


@pytest.mark.parametrize("case", range(len(TERMINATION)))
def test_early_termination_at_staging_boundaries(cuda_device, oracle, case):
    """Pixels of one tile stop blending (T < 1e-4) at list positions on both sides of the chunk and window
    boundaries, differently inside a 2 x 2 block and from one block to the next."""
    vals, n_total = TERMINATION[case]
    g = np.random.default_rng(7 + case)
    rest = np.setdiff1d(np.arange(100, n_total - 60), np.r_[vals, vals - 1])
    targets = g.permutation(np.r_[vals, g.choice(rest, 256 - len(vals), replace=False)])
    inp = termination_inputs(targets, n_total, cuda_device, seed=case)
    mine, fw, bw = run_both(oracle, inp, upstream(16, 16, 77 + case))
    nc = fw["n_contrib"].reshape(16, 16).astype(np.int64)
    vals_hit = set(nc.reshape(-1).tolist())
    assert vals_hit & {255, 256, 257}, "no pixel stops at the first chunk boundary"
    assert vals_hit & {383, 384, 385}, "no pixel stops at the first window boundary"
    blocks = nc.reshape(8, 2, 8, 2).transpose(0, 2, 1, 3).reshape(64, 4)
    assert (blocks.min(1) != blocks.max(1)).any(), "n_contrib does not vary inside a 2x2 block"
    # a property of the scene: the 2x2 blocks end at many different depths.  The backward hands blocks to its warps by
    # the rank of their list length, so which blocks share a warp is the kernel's choice, not this test's
    assert len(set(blocks.max(1).tolist())) >= 32, "the 2x2 blocks do not end at different depths"
    assert nc.max() // 384 > nc.min() // 384, "the deepest pixel is in the same backward window as the shallowest"
    assert int(nc.max()) < n_total - 60, "a pixel blended to the end of the list instead of terminating"
    check_all(mine, fw, bw, 16, 16)


# ------------------------------------------------------------------------------------------------ alpha decisions
def test_alpha_clamp_and_negative_determinant(cuda_device, oracle):
    """Opacity-1 splats centred on pixel centres: alpha = min(0.99, 1 * exp(0)) takes the clamp.  Supplied conics
    with a negative determinant: power > 0 on part of the footprint, which both passes skip."""
    W, H = 40, 24
    g = np.random.default_rng(3)
    P = 60
    px = np.r_[g.integers(0, W, 20).astype(np.float64), g.uniform(-3, W + 2, P - 20)]
    py = np.r_[g.integers(0, H, 20).astype(np.float64), g.uniform(-3, H + 2, P - 20)]
    s = g.uniform(0.5, 4.0, (2, P))
    op = np.r_[np.ones(20), g.uniform(0.1, 1.0, P - 20)]
    scene, cam = pixel_scene(px, py, 0.4 + 0.3 * g.permutation(P) / P, s[0], s[1], W, H, op, seed=3, rotate=False)
    inp = inputs(scene, cam, "render", cuda_device, bg=np.linspace(0.0, 3.0, 10))
    con = inp["kwargs"]["conic_precomp"]
    neg = torch.arange(con.shape[0], device=con.device) % 4 == 3
    con[neg, 1] = 1.5 * torch.sqrt(con[neg, 0] * con[neg, 2])       # b^2 > a c
    mine, fw, bw = run_both(oracle, inp, upstream(W, H, 9))

    vis = fw["radii"] > 0
    co, m2 = fw["conic_opacity"], fw["means2D"]
    centred = vis & (co[:, 3] == 1.0) & (m2[:, 0] == np.round(m2[:, 0])) & (m2[:, 1] == np.round(m2[:, 1]))
    inside = (m2[:, 0] >= 0) & (m2[:, 0] < W) & (m2[:, 1] >= 0) & (m2[:, 1] < H)
    assert (centred & inside).any(), "no opacity-1 splat is centred exactly on a pixel"
    negdet = vis & (co[:, 0] * co[:, 2] - co[:, 1] ** 2 < 0)
    assert negdet.any(), "no visible splat has a negative-determinant conic"
    # power > 0 somewhere within the radius of a negative-determinant splat
    i = int(np.nonzero(negdet)[0][0])
    ys, xs = np.mgrid[0:H, 0:W].astype(np.float32)
    dx, dy = m2[i, 0] - xs, m2[i, 1] - ys
    power = -0.5 * (co[i, 0] * dx * dx + co[i, 2] * dy * dy) - co[i, 1] * dx * dy
    assert (power > 0).any() and (power <= 0).any()
    check_all(mine, fw, bw, W, H)


# ------------------------------------------------------------------------------------------------ Gaussian counts
@pytest.mark.parametrize("P", [1, 31, 33, 257])
@pytest.mark.parametrize("mode", ["native", "render"])
def test_gaussian_counts(cuda_device, oracle, P, mode):
    """Gaussian counts around a warp (31, 33) and a CTA (257), a single Gaussian; non-zero background and an upstream
    gradient with negative values, zeros and an all-zero channel."""
    W, H = 48, 40
    g = np.random.default_rng(P)
    px, py = g.uniform(-2, W + 1, P), g.uniform(-2, H + 1, P)
    s = g.uniform(0.5, 8.0, (2, P))
    if P == 1:
        px[0], py[0] = 20.3, 17.8
    scene, cam = pixel_scene(px, py, 0.4 + 0.3 * g.permutation(P) / P, s[0], s[1], W, H, g.uniform(0.1, 1.0, P), seed=P)
    inp = inputs(scene, cam, mode, cuda_device, bg=np.linspace(-1.0, 1.0, 10))
    assert inp["kwargs"]["means3D"].shape[0] == P
    mine, fw, bw = run_both(oracle, inp, upstream(W, H, P))
    assert (fw["radii"] > 0).sum() > 0
    check_all(mine, fw, bw, W, H)
