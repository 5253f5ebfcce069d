"""The forward hands the backward one mask per list record over the tile's 64 blocks of 2 x 2 pixels, and the
backward stages only the records whose mask is not zero ("live" records).  These scenes check forward and backward
against Oracle-B, with the tolerances of test_gpu_blend_edges.py, where that hand-over is most likely to go wrong:

  * a tile where most records are dead: thin ellipses whose bounding square overlaps the tile but whose
    alpha >= 1/255 ellipse does not;
  * a tile where every record is dead;
  * every pixel of a tile terminating inside the first, a middle and the last 256-record forward chunk (the
    forward writes masks only up to the chunk where it stops);
  * a list longer than 2048 records, which the long-list sort orders through the scratch buffer that later holds
    the masks;
  * long lists in edge tiles of an image with odd width and height.

Besides the results, each scene reads the masks the forward wrote (in the binning workspace, after the sorted
records) and checks that they are conservative -- every block with a pixel that blends a record has that record's
bit -- and that the scene reaches its path.
"""
import numpy as np
import pytest
import torch

import _util
from test_gpu_blend_edges import check_all, inputs, pixel_scene, run_both, upstream

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def oracle():
    import oracle as _oracle
    _oracle.build()
    return _oracle


def _run(oracle, inp, dL):
    """run_both plus the forward's block masks: binning workspace = [R sorted records][R masks], each region
    aligned to 256 bytes (GhBinWS in gh_common.cuh)."""
    import gaussianhaircut_b200._C as native
    mine, fw, bw = run_both(oracle, inp, dL)
    r = native.rasterize_gaussians(*_util.native_args(inp))      # same inputs: same lists, same masks
    torch.cuda.synchronize()
    R, buf = int(r[0]), r[4]
    off = (-buf.data_ptr()) % 256
    moff = off + (8 * R + 255) // 256 * 256
    masks = buf[moff:moff + 8 * R].cpu().numpy().view(np.uint64) if R else np.zeros(0, np.uint64)
    return mine, fw, bw, masks


def _tile_stats(fw, masks, W, H):
    """Per non-empty tile: (list length, last blended position, live records before it); asserts that the masks
    cover every (record, pixel) pair the oracle blends."""
    gx = (W + 15) // 16
    nc = fw["n_contrib"].reshape(H, W).astype(np.int64)
    m2, co = fw["means2D"], fw["conic_opacity"]
    out = {}
    for t, (lo, hi) in enumerate(fw["ranges"].astype(np.int64)):
        if hi == lo:
            continue
        ty, tx = divmod(t, gx)
        x0, y0 = tx * 16, ty * 16
        ncl = nc[y0:y0 + 16, x0:x0 + 16]
        last = int(ncl.max())
        ids = fw["point_list"][lo:lo + last].astype(np.int64)
        mk = masks[lo:lo + last]
        ys, xs = np.mgrid[y0:y0 + ncl.shape[0], x0:x0 + ncl.shape[1]]
        dx = m2[ids, 0][:, None, None] - xs[None].astype(np.float32)
        dy = m2[ids, 1][:, None, None] - ys[None].astype(np.float32)
        a, b, c, o = (co[ids, k][:, None, None] for k in range(4))
        power = -0.5 * (a * dx * dx + c * dy * dy) - b * dx * dy
        alpha = np.minimum(0.99, o * np.exp(np.minimum(power, 0.0)))
        pos = np.arange(last)[:, None, None]
        blend = (power <= 0) & (alpha >= 1 / 255.0) & (pos < ncl[None])
        k, py, px = np.nonzero(blend)                 # tile-local pixel
        bit = (py // 2) * 8 + px // 2
        assert ((mk[k] >> bit.astype(np.uint64)) & np.uint64(1)).all(), \
            f"tile {t}: a record's mask misses a block in which it is blended"
        out[t] = (int(hi - lo), last, int((mk != 0).sum()))
    return out


def test_mostly_dead_records(cuda_device, oracle):
    """Thin rotated ellipses along the tile borders of a 64 x 48 image: each one's bounding square reaches several
    tiles, its alpha >= 1/255 footprint few of them.  'render' call shape (conics supplied): the gradients end at
    the 2-D quantities the blend kernels produce; through the projection, the scale and rotation gradients of such
    thin, overlapping splats are too ill-conditioned in float32 for the per-element bound."""
    W, H = 64, 48
    g = np.random.default_rng(11)
    P = 160
    px = np.r_[g.choice([15.5, 31.5, 47.5], P // 2) + g.normal(0, 0.6, P // 2), g.uniform(0, W, P // 2)]
    py = np.r_[g.uniform(0, H, P // 2), g.choice([15.5, 31.5], P // 2) + g.normal(0, 0.6, P // 2)]
    sx, sy = g.uniform(4.0, 9.0, P), g.uniform(0.8, 1.6, P)
    scene, cam = pixel_scene(px, py, 0.4 + 0.3 * g.permutation(P) / P, sx, sy, W, H, g.uniform(0.05, 0.6, P), seed=11)
    inp = inputs(scene, cam, "render", cuda_device, bg=np.linspace(0.5, -0.5, 10))
    mine, fw, bw, masks = _run(oracle, inp, upstream(W, H, 11))
    st = _tile_stats(fw, masks, W, H)
    assert any(live * 2 < last for _, last, live in st.values()), "no tile has most of its records dead"
    assert sum(live for *_, live in st.values()) < sum(last for _, last, _ in st.values())
    check_all(mine, fw, bw, W, H)


def test_tile_with_every_record_dead(cuda_device, oracle):
    """Faint splats (opacity 0.01: alpha >= 1/255 only within ~1.4 sigma) centred in the left tile of a 32 x 16
    image, 3 sigma reaching into the right tile: the right tile's list holds only dead records."""
    W, H = 32, 16
    g = np.random.default_rng(12)
    P = 40
    px, py = g.uniform(2.0, 9.0, P), g.uniform(2.0, 13.0, P)
    s = np.full(P, 3.0)
    scene, cam = pixel_scene(px, py, 0.4 + 0.3 * g.permutation(P) / P, s, s, W, H, np.full(P, 0.01), seed=12,
                             rotate=False)
    inp = inputs(scene, cam, "native", cuda_device, bg=np.linspace(0.0, 1.0, 10))
    mine, fw, bw, masks = _run(oracle, inp, upstream(W, H, 12))
    n1 = int(fw["ranges"][1, 1] - fw["ranges"][1, 0])
    assert n1 > 0, "the right tile holds no records"
    assert int(fw["n_contrib"].reshape(H, W)[:, 16:].max()) == 0, "a pixel of the right tile blends something"
    lo = int(fw["ranges"][1, 0])
    assert not masks[lo:lo + n1].any(), "a record of the right tile has a non-zero mask"
    st = _tile_stats(fw, masks, W, H)
    assert st[0][2] > 0
    check_all(mine, fw, bw, W, H)


def haze_scene(n, opacity, seed):
    """One 16 x 16 tile, n very wide splats (sigma 300..600 px, so alpha is the same at every pixel to 0.3 %)
    with opacities in `opacity`: every pixel terminates after about ln(1e-4) / ln(1 - opacity) records."""
    g = np.random.default_rng(300 + seed)
    s = g.uniform(300.0, 600.0, (2, n))
    return pixel_scene(g.uniform(0.0, 15.0, n), g.uniform(0.0, 15.0, n), 0.4 + 0.3 * np.arange(n) / n, s[0], s[1],
                       16, 16, g.uniform(*opacity, n), seed=seed, rotate=False)


# (records, opacity range, forward chunk in which every pixel stops)
TERMINATION = [(1100, (0.5, 0.6), 0), (1100, (0.0150, 0.0156), 2), (1100, (0.00860, 0.00875), 4)]


@pytest.mark.parametrize("case", range(len(TERMINATION)))
def test_termination_chunk(cuda_device, oracle, case):
    n, op, chunk = TERMINATION[case]
    scene, cam = haze_scene(n, op, case)
    inp = inputs(scene, cam, "native", cuda_device, bg=np.linspace(0.25, 1.0, 10))
    inp["kwargs"]["colors_precomp"].abs_()
    mine, fw, bw, masks = _run(oracle, inp, upstream(16, 16, 40 + case))
    nc = fw["n_contrib"]
    assert int(fw["ranges"][0, 1] - fw["ranges"][0, 0]) == n
    assert 256 * chunk < nc.min() and nc.max() <= min(n, 256 * (chunk + 1)), \
        f"pixels stop at {nc.min()}..{nc.max()}, not all inside chunk {chunk}"
    assert nc.max() < n, "a pixel blended the whole list"
    _tile_stats(fw, masks, 16, 16)
    check_all(mine, fw, bw, 16, 16)


def test_long_list_sorted_through_scratch(cuda_device, oracle):
    """2600 records in one tile: longer than the 2048 the forward sorts in shared memory, so the long-list sort runs
    through the scratch buffer before the forward writes the masks there.  Every pixel blends ~2300 of them."""
    scene, cam = haze_scene(2600, (0.0040, 0.0041), 7)
    inp = inputs(scene, cam, "native", cuda_device, bg=np.linspace(0.25, 1.0, 10))
    inp["kwargs"]["colors_precomp"].abs_()
    mine, fw, bw, masks = _run(oracle, inp, upstream(16, 16, 47))
    assert int(fw["ranges"][0, 1] - fw["ranges"][0, 0]) == 2600 > 2048
    assert int(fw["n_contrib"].min()) > 2048, "the pixels stop before the end of the in-kernel sort's reach"
    st = _tile_stats(fw, masks, 16, 16)
    assert st[0][2] == st[0][1], "a record every pixel blends has a zero mask"
    check_all(mine, fw, bw, 16, 16)


def test_heavy_edge_tiles(cuda_device, oracle):
    """A 41 x 37 image whose right column and bottom row of tiles (9 and 5 pixels wide) each hold lists of more than
    1000 records, most of them blended, a part dead.  'render' call shape, as in test_mostly_dead_records."""
    W, H = 41, 37
    g = np.random.default_rng(13)
    P = 1500
    px, py = g.uniform(20.0, W + 4.0, P), g.uniform(20.0, H + 4.0, P)
    sx, sy = g.uniform(3.0, 12.0, P), g.uniform(1.5, 12.0, P)
    scene, cam = pixel_scene(px, py, 0.4 + 0.3 * g.permutation(P) / P, sx, sy, W, H, g.uniform(0.004, 0.02, P), seed=13)
    inp = inputs(scene, cam, "render", cuda_device, bg=np.linspace(-1.0, 1.0, 10))
    mine, fw, bw, masks = _run(oracle, inp, upstream(W, H, 13))
    st = _tile_stats(fw, masks, W, H)
    gx = (W + 15) // 16
    edge = [t for t in st if t % gx == gx - 1 or t // gx == (H + 15) // 16 - 1]
    assert sum(st[t][0] > 1000 for t in edge) >= 3, "fewer than three edge tiles hold more than 1000 records"
    assert any(st[t][2] < st[t][1] for t in edge), "no edge tile has a dead record before its last blended one"
    check_all(mine, fw, bw, W, H)
