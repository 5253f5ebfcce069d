"""Per-stage device times of one library build on the benchmark scene; without a path, the in-tree build.
   python tools/stage_times.py [path/to/libgh_raster.so] [--strands 5000] [--mode native]"""
import argparse, json, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "oracle"))
ap = argparse.ArgumentParser()
ap.add_argument("lib", nargs="?", default=None)
ap.add_argument("--strands", type=int, default=5000)
ap.add_argument("--mode", default="native")
ap.add_argument("--steps", type=int, default=30)
ap.add_argument("--opacity", default="random")
args = ap.parse_args()
import torch
from gaussianhaircut_b200 import _capi
if args.lib:
    _capi.LIB_PATH = os.path.abspath(args.lib)      # development only: measure another build of the library
from gaussianhaircut_b200 import _C
import synth
dev = torch.device("cuda:0")
W, H = 1920, 1080
scene = synth.make_strand_scene(args.strands, seed=0, opacity_mode=args.opacity)
views = [synth.rasterizer_inputs(scene, synth.make_camera((v * 8) % 64, W, H), mode=args.mode, device=dev) for v in range(8)]
dL = synth.upstream_gradient(W, H, 0).to(dev)
e = torch.Tensor([])

def step(i):
    inp = views[i % 8]; kw, s = inp["kwargs"], inp["settings"]
    g = lambda k: e if kw[k] is None else kw[k]
    R, color, radii, geom, binning, img = _C.rasterize_gaussians(
        s["bg"], kw["means3D"], kw["means2D"], g("colors_precomp"), kw["opacities"], g("scales"), g("rotations"), 1.0,
        g("cov3D_precomp"), g("conic_precomp"), s["viewmatrix"], s["projmatrix"], s["tanfovx"], s["tanfovy"], H, W, e, 3, s["campos"],
        s["prefiltered"], False)
    _C.rasterize_gaussians_backward_arena(s["bg"], kw["means3D"], radii, g("colors_precomp"), g("scales"), g("rotations"), 1.0,
                                          g("cov3D_precomp"), g("conic_precomp"), s["viewmatrix"], s["projmatrix"], s["tanfovx"], s["tanfovy"],
                                          dL, e, 3, s["campos"], geom, R, binning, img, False)
    return R

for i in range(8):
    step(i)
torch.cuda.synchronize()
reps = []
for r in range(5):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        step(i)
    e1.record(); torch.cuda.synchronize()
    reps.append(e0.elapsed_time(e1) / args.steps)
lib = _capi.load()
lib.gh_stage_timing_enable(1)
for i in range(16):
    step(i)
torch.cuda.synchronize()
st = _capi.stage_timing_read()
lib.gh_stage_timing_enable(0)
reps.sort()
print(json.dumps({"lib": os.path.basename(_capi.LIB_PATH), "ms_per_step": reps[len(reps) // 2], "ms_min": reps[0],
                  "stages_us": {k: round(1e3 * ms / c, 1) for k, (ms, c) in st.items() if c}}))
