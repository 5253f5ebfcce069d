"""Per-tile work of the blend kernels on one view, counted on the CPU with Oracle-B (no GPU needed).

    python tools/tile_work.py [--strands 5000] [--width 1920] [--height 1080] [--camera 0]

Prints one JSON object:
  R                    records in all tile lists (num_rendered)
  before_last          records before their tile's last contributor (max n_contrib over the tile's pixels):
                       what the backward has to consider
  live                 of those, the records that reach alpha >= 1/255 (and power <= 0) on some pixel of their
                       tile, by the exact test.  The kernels' block masks are conservative, so they keep slightly more
  pairs                contributing (record, pixel) pairs
  tiles / nonempty     tile count, tiles with a non-empty list
  len_quantiles        list length at the 50/90/99/100 % quantiles of the non-empty tiles, and the top 5
  lpt                  for 740 (148 SMs x 5, the backward) and 592 (x 4, the forward) equal-speed CTA slots filled
                       heaviest tile first: the heaviest tile's work over the mean slot load, work counted in records
                       before the last contributor, in live records and in contributing pairs.  Above 1, one tile is
                       longer than a fair share of the whole launch.
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))


def tile_counts(fw, W, H):
    """-> per tile: (list length, records before the last contributor, live records, contributing pairs)."""
    gx = (W + 15) // 16
    nc = fw["n_contrib"].reshape(H, W).astype(np.int64)
    m2, co = fw["means2D"], fw["conic_opacity"]
    out = np.zeros((len(fw["ranges"]), 4), np.int64)
    for t, (lo, hi) in enumerate(fw["ranges"].astype(np.int64)):
        if hi == lo:
            continue
        ty, tx = divmod(t, gx)
        x0, y0 = tx * 16, ty * 16
        ncl = nc[y0:y0 + 16, x0:x0 + 16]
        last = int(ncl.max())
        ys, xs = np.mgrid[y0:y0 + ncl.shape[0], x0:x0 + ncl.shape[1]]
        xs, ys = xs.reshape(-1).astype(np.float32), ys.reshape(-1).astype(np.float32)
        live = pairs = 0
        for a0 in range(0, last, 512):                      # bounded memory on long lists
            ids = fw["point_list"][lo + a0:lo + min(last, a0 + 512)].astype(np.int64)
            dx = m2[ids, 0][:, None] - xs[None]
            dy = m2[ids, 1][:, None] - ys[None]
            a, b, c, o = (co[ids, k][:, None] for k in range(4))
            power = np.float32(-0.5) * (a * dx * dx + c * dy * dy) - b * dx * dy
            hit = (power <= 0) & (np.minimum(0.99, o * np.exp(np.minimum(power, 0))) >= np.float32(1 / 255.0))
            live += int(hit.any(1).sum())
            pos = np.arange(a0, a0 + len(ids))[:, None]
            pairs += int((hit & (pos < ncl.reshape(-1)[None])).sum())
        out[t] = (hi - lo, last, live, pairs)
    return out


def lpt_ratio(work, slots):
    """Heaviest tile over the mean slot load when the tiles go to `slots` equal slots heaviest first."""
    w = np.sort(work[work > 0])[::-1]
    if w.size == 0:
        return 0.0
    return float(w[0] / (w.sum() / slots))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--strands", type=int, default=5000)
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--height", type=int, default=1080)
    ap.add_argument("--camera", type=int, default=0)
    args = ap.parse_args()
    import torch
    import oracle
    import synth
    oracle.build()
    W, H = args.width, args.height
    scene = synth.make_strand_scene(args.strands, seed=0)
    inp = synth.rasterizer_inputs(scene, synth.make_camera(args.camera, W, H), mode="native", device=torch.device("cpu"))
    kw, s = inp["kwargs"], inp["settings"]
    npy = lambda t: None if t is None else t.detach().cpu().numpy()  # noqa: E731
    fw = oracle.forward(npy(kw["means3D"]), npy(kw["opacities"]), npy(kw["colors_precomp"]), npy(s["viewmatrix"]),
                        npy(s["projmatrix"]), s["tanfovx"], s["tanfovy"], W, H, npy(s["bg"]),
                        scales=npy(kw["scales"]), rotations=npy(kw["rotations"]),
                        cov3D_precomp=npy(kw["cov3D_precomp"]), conic_precomp=npy(kw["conic_precomp"]))
    tc = tile_counts(fw, W, H)
    lens = tc[:, 0][tc[:, 0] > 0]
    res = {
        "view": {"strands": args.strands, "width": W, "height": H, "camera": args.camera},
        "R": int(fw["num_rendered"]),
        "before_last": int(tc[:, 1].sum()),
        "live": int(tc[:, 2].sum()),
        "pairs": int(tc[:, 3].sum()),
        "tiles": int(len(tc)),
        "nonempty": int(lens.size),
        "len_quantiles": {q: int(np.quantile(lens, q / 100.0, method="lower")) for q in (50, 90, 99, 100)} if lens.size else {},
        "len_top5": sorted(lens.tolist(), reverse=True)[:5],
        "lpt": {str(slots): {"records": round(lpt_ratio(tc[:, 1], slots), 3), "live": round(lpt_ratio(tc[:, 2], slots), 3),
                             "pairs": round(lpt_ratio(tc[:, 3], slots), 3)} for slots in (740, 592)},
    }
    print(json.dumps(res))


if __name__ == "__main__":
    main()
