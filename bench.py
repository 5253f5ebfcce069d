#!/usr/bin/env python
"""bench.py -- forward+backward Gaussians/s of the strand-aligned rasterizer hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl mine|reference] [--mode native|render|render_hair]
                    [--dump-outputs DIR]

Workload (BASELINE.json configs[2], the one `metric` is quoted on): 500 000 synthetic strand-aligned
Gaussians (SURVEY.md 8d scene "strands(5000)"), 1920x1080, one ring camera per step, forward +
backward with a fixed random upstream gradient.  A *step* is one pass of the hot path (forward
rasterize -> backward) over one view.  Inputs are resident in HBM for `value`; `e2e` goes through
the public Python API (`GaussianRasterizer` + autograd) with the per-view camera and supervision
tensor copied from pinned host memory and the loss read back every step.

N > 1 (torchrun, one rank per GPU): views shard one per rank per step (weak scaling), the flat
gradient arena is summed with ONE NCCL all-reduce per step; time is the max over ranks.

`--impl reference` times Oracle-A: the reference's own CUDA extension compiled in place for sm_100a
(oracle/_ref) -- the reference ships no CPU rasterizer, so that build is the baseline
(BASELINE.json north_star).  It prints the same JSON line with "impl": "reference".

Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "fwd+bwd Gaussians/s at 500k G, 1080p"
UNIT = "Gaussians/s"


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="mine", choices=["mine", "reference"])
    ap.add_argument("--mode", default="native", choices=["native", "render", "render_hair", "cov3d"])
    ap.add_argument("--strands", type=int, default=5000)
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--height", type=int, default=1080)
    ap.add_argument("--views", type=int, default=8, help="distinct camera views cycled per rank")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-roofline", action="store_true")
    ap.add_argument("--ref-steps", type=int, default=10)
    ap.add_argument("--repeats", type=int, default=1, help="how many times the timed K-step window is repeated (median reported)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (image, radii, gradients) as DIR/<name>.npy")
    ap.add_argument("--collective", default="auto", choices=["auto", "peer-mc", "peer-nomc", "nccl"],
                    help="N>1: gh_allreduce_p2p over symmetric memory (auto: peer ld/st up to 4 GPUs, NVLS multimem from 8) or NCCL")
    return ap.parse_args()


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.path = f"/tmp/gh_clocks_{os.getpid()}.csv"

    def start(self):
        try:
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.f.close()
        sm, smax, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in open(self.path):
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1])); smax = float(parts[2])
            except ValueError:
                continue
            for nm, v in zip(names, parts[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        try:
            os.remove(self.path)
        except OSError:
            pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": smax,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def algorithmic_bytes(P, R, W, H, T, mode):
    """Compulsory HBM bytes per stage and for the whole fwd+bwd path (DESIGN.md section 4;
    path total = SURVEY.md 8(d): 400P + 52R + 96WH + 24T native, 344P when the conic is supplied)."""
    native = mode in ("native", "cov3d")
    stage = {
        "preprocess": (84 if native else 68) * P,
        "tile_scan": 16 * T,
        "emit": 24 * P + 8 * R,
        "tile_sort": 16 * R + 8 * T,
        "blend_forward": 8 * R + 72 * P + 48 * W * H + 8 * T,
        "blend_backward": 8 * R + 144 * P + 48 * W * H + 8 * T,
        "preprocess_backward": 136 * P if native else 0,
    }
    path = (400 if native else 344) * P + 52 * R + 96 * W * H + 24 * T
    return stage, path


DUMP_BYTES = 60 << 20
# positions of the rasterizer's 9 gradients in the tuple `rasterize_gaussians_backward` returns
GRAD_TUPLE = ("means2D", "colors", "opacity", "means3D", "cov3D", "conic", "sh", "scales", "rotations")


def dump_outputs(out_dir, last):
    """The arrays the last timed step handed to its caller -- the rendered image, radii, num_rendered and every
    gradient -- as float32 `.npy` files (num_rendered float64).  An array larger than its share of DUMP_BYTES is
    replaced by the values at a fixed, seeded set of positions, so that two builds can be compared file by file."""
    import numpy as np
    import torch
    grads = last["views"] if "views" in last else dict(zip(GRAD_TUPLE, last["grads"]))
    arrays = {"color": last["color"], "radii": last["radii"]}
    arrays.update({f"grad_{k}": v for k, v in grads.items() if v is not None and v.numel() > 0})
    cap = DUMP_BYTES // 4 // len(arrays)
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        v = t.detach().reshape(-1).float()
        if v.numel() > cap:
            idx = torch.randperm(v.numel(), generator=torch.Generator().manual_seed(0))[:cap].sort().values
            v = v[idx.to(v.device)]
        np.save(os.path.join(out_dir, name + ".npy"), v.cpu().numpy())
    np.save(os.path.join(out_dir, "num_rendered.npy"), np.array([float(last["R"])], np.float64))
    log(f"[bench] outputs of the last timed step written to {out_dir} ({len(arrays) + 1} arrays)")


def main():
    args = parse_args()
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.gpus != world and world > 1:
        log(f"[bench] note: --gpus {args.gpus} but WORLD_SIZE {world}; using WORLD_SIZE")
    N = world

    if args.impl == "reference" and rank != 0:
        return 0     # reference arm: rank 0 alone runs and prints

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU path exists for this product)")
    device = torch.device("cuda", local_rank)
    torch.cuda.set_device(device)
    use_dist = (N > 1 and args.impl == "mine")
    if use_dist:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=device)

    from gaussianhaircut_b200 import dist as ghdist
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import build_ref
    import synth          # seeded scene / camera generator (test infrastructure, oracle/synth.py)

    if args.impl == "mine":
        import gaussianhaircut_b200._C as native
        import gaussianhaircut_b200 as pkg
        from gaussianhaircut_b200 import _capi
        _capi.load()
    else:
        if not build_ref.is_built():
            print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref not built (python oracle/build_ref.py)"}))
            return 0
        pkg = build_ref.load()
        native = pkg._C

    W, H = args.width, args.height
    gx, gy = (W + 15) // 16, (H + 15) // 16
    T = gx * gy
    t0 = time.time()
    scene = synth.make_strand_scene(args.strands, seed=0)
    P_total = scene["xyz"].shape[0]
    views = []
    for v in range(args.views):
        cam_k = (rank * args.views + v) % 64 if N > 1 else (v * 8) % 64
        cam = synth.make_camera(cam_k, W, H)
        inp = synth.rasterizer_inputs(scene, cam, mode=args.mode, device=device)
        views.append(inp)
    dL = synth.upstream_gradient(W, H, 0).to(device)
    P = views[0]["kwargs"]["means3D"].shape[0]
    log(f"[bench] rank {rank}: scene P={P_total} (passed to op: {P}), {args.views} views, mode={args.mode}, "
        f"setup {time.time() - t0:.1f}s")

    def pack_args(inp):
        kw, s = inp["kwargs"], inp["settings"]
        e = torch.Tensor([])
        g = lambda k: e if kw[k] is None else kw[k]  # noqa: E731
        fw = (s["bg"], kw["means3D"], kw["means2D"], g("colors_precomp"), kw["opacities"], g("scales"), g("rotations"),
              s["scale_modifier"], g("cov3D_precomp"), g("conic_precomp"), s["viewmatrix"], s["projmatrix"],
              s["tanfovx"], s["tanfovy"], s["image_height"], s["image_width"], e, s["sh_degree"], s["campos"],
              s["prefiltered"], False)
        return fw, kw, s, e, g

    packed = [pack_args(v) for v in views]
    last = {}
    par = None
    collective = "none"
    allreduce_check = None
    if use_dist and args.impl == "mine":
        collective = "nccl all_reduce"
        n_arena, n_train = native.arena_floats(P), native.trainable_floats(P)
        if args.collective != "nccl":
            try:
                par = ghdist.PeerAllReduce(n_arena, device, use_multicast={"auto": None, "peer-mc": True, "peer-nomc": False}[args.collective])
                collective = "gh_allreduce_p2p (" + ("NVLS multimem" if par.multicast else "peer loads/stores") + ")"
            except Exception as exc:      # symmetric memory unavailable on this box: NCCL
                log(f"[bench] rank {rank}: peer all-reduce unavailable ({exc}); using NCCL")
                par = None
        log(f"[bench] rank {rank}: collective = {collective}")
        if par is not None:
            # correctness of the hand-written collective where the driver runs it: both data paths against
            # NCCL on the same arena contents, bit-identical across ranks; any mismatch aborts the bench
            def check_path(p_obj, label):
                g = torch.Generator(device="cpu").manual_seed(4242 + rank)
                for rnd, nfl in enumerate((n_train, n_arena)):
                    x = (torch.randn(n_arena, generator=g) * (10.0 ** (rnd - 1))).to(device)
                    p_obj.buffer[:n_arena].copy_(x)
                    ref = x.clone()
                    dist.all_reduce(ref[:nfl], op=dist.ReduceOp.SUM)
                    p_obj.all_reduce(n_floats=nfl)
                    torch.cuda.synchronize(device)
                    if not p_obj.ok():
                        raise SystemExit(f"[bench] rank {rank}: gh_allreduce_p2p ({label}): a peer did not arrive")
                    err = float((p_obj.buffer[:n_arena] - ref).abs().max() / ref.abs().max().clamp_min(1e-30))
                    if not err <= 1e-6:
                        raise SystemExit(f"[bench] rank {rank}: gh_allreduce_p2p ({label}) differs from NCCL all_reduce: rel err {err}")
                    if nfl < n_arena and not torch.equal(p_obj.buffer[nfl:n_arena], x[nfl:]):
                        raise SystemExit(f"[bench] rank {rank}: gh_allreduce_p2p ({label}) touched floats outside the requested range")
                    digest = p_obj.buffer[:nfl].view(torch.int32).to(torch.int64).sum().reshape(1)      # the reduced range only
                    every = [torch.zeros_like(digest) for _ in range(N)]
                    dist.all_gather(every, digest)
                    if any(int(t) != int(every[0]) for t in every):
                        raise SystemExit(f"[bench] gh_allreduce_p2p ({label}): ranks hold different sums")
                    if int(p_obj.nan_flag.item()) != 0:
                        raise SystemExit(f"[bench] gh_allreduce_p2p ({label}): spurious NaN flag")
                return label

            checked = [check_path(par, "NVLS multimem" if par.multicast else "peer loads/stores")]
            try:
                other = ghdist.PeerAllReduce(n_arena, device, use_multicast=not bool(par.multicast))
                if bool(other.multicast) != bool(par.multicast):
                    checked.append(check_path(other, "NVLS multimem" if other.multicast else "peer loads/stores"))
                del other
            except Exception as exc:
                log(f"[bench] rank {rank}: second data path not checked ({exc})")
            allreduce_check = "ok (" + ", ".join(checked) + " == NCCL all_reduce <= 1e-6, bit-identical across ranks)"
            log(f"[bench] rank {rank}: allreduce_check = {allreduce_check}")

    def step(i, mod=native, arena=(args.impl == "mine"), plist=None):
        fw, kw, s, e, g = (plist or packed)[i % len(packed)]
        R, color, radii, geom, binning, img = mod.rasterize_gaussians(*fw)
        last["color"], last["radii"] = color, radii
        bw = (s["bg"], kw["means3D"], radii, g("colors_precomp"), g("scales"), g("rotations"), s["scale_modifier"],
              g("cov3D_precomp"), g("conic_precomp"), s["viewmatrix"], s["projmatrix"], s["tanfovx"], s["tanfovy"],
              dL, e, s["sh_degree"], s["campos"], geom, R, binning, img, False)
        if arena:
            flat, grads, _ = mod.rasterize_gaussians_backward_arena(*bw, arena_storage=(par.buffer if par is not None else None))
            if use_dist:
                # one collective per step, over the part of the arena the optimizer reads
                sl = ghdist.trainable_slice(flat, P, "native" if args.mode == "native" else "any")
                if par is not None:
                    par.all_reduce(n_floats=sl.numel())
                else:
                    dist.all_reduce(sl, op=dist.ReduceOp.SUM)
            last["grads"] = flat
            last["views"] = grads
        else:
            last["grads"] = mod.rasterize_gaussians_backward(*bw)
        last["R"] = R
        return R

    def timed(nsteps, fn):
        if use_dist:
            dist.barrier()
        torch.cuda.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for i in range(nsteps):
            fn(i)
        ev1.record()
        torch.cuda.synchronize()
        ms = ev0.elapsed_time(ev1)
        if use_dist:
            t = torch.tensor([ms], device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    # ---------------------------------------------------------------- device-resident throughput
    for i in range(args.warmup):
        step(i)
    torch.cuda.synchronize()
    launches0 = None
    if args.impl == "mine":
        launches0 = _capi.load().gh_kernel_launch_count()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    # the K-step window is timed `--repeats` times back to back (each bracketed by barrier + synchronize, max over
    # ranks) and the MEDIAN window is reported; every window is listed in `ms_per_step_repeats`
    windows = []
    gpu_launches = None
    for rep in range(max(1, args.repeats)):
        windows.append(timed(args.steps, step))
        if rep == 0 and args.impl == "mine":
            gpu_launches = int(_capi.load().gh_kernel_launch_count() - launches0)
    clocks = sampler.stop() if rank == 0 else None
    ms_total = statistics.median(windows)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last)
    ms_per_step = ms_total / args.steps
    n_eff = N if args.impl == "mine" else 1       # reference arm: rank 0 alone runs (one GPU's worth of work)
    value = (args.steps * P * n_eff) / (ms_total * 1e-3)
    R_mean = float(last["R"])
    log(f"[bench] {args.impl}: {ms_per_step:.3f} ms/step  -> {value / 1e6:.1f} M Gaussians/s  (R={last['R']})")

    # ---------------------------------------------------------------- the call shapes of the reference trainers (M-call)
    # render(): cov3D_precomp + conic_precomp; render_hair(): scales/rotations + conic_precomp (SURVEY.md 8d)
    call_shapes = None
    if args.mode == "native" and not use_dist:
        call_shapes = {}
        for m in ("render", "render_hair"):
            vm = []
            for v in range(args.views):
                cam = synth.make_camera((v * 8) % 64, W, H)
                vm.append(pack_args(synth.rasterizer_inputs(scene, cam, mode=m, device=device)))
            P_m = vm[0][1]["means3D"].shape[0]
            fn = (lambda i, vm=vm: step(i, arena=False, plist=vm)) if args.impl == "mine" else (lambda i, vm=vm: step(i, mod=native, arena=False, plist=vm))
            for i in range(max(3, len(vm))):
                fn(i)
            ms_m = timed(args.steps, fn) / args.steps
            call_shapes[m] = {"ms_per_step": ms_m, "value": P_m / (ms_m * 1e-3), "unit": UNIT, "gaussians_per_view": int(P_m)}
            log(f"[bench] call shape {m}: {ms_m:.3f} ms/step -> {P_m / ms_m / 1e3:.1f} M Gaussians/s (P={P_m})")
            del vm
        last["R"] = int(R_mean)

    # ---------------------------------------------------------------- end to end through the public API
    # One step = what a trainer does around the op for one view (src/train_gaussians.py:103-140), through the public
    # Python API: the view's camera and its SUPERVISION MAPS arrive from pinned host memory in the dtypes the dataset
    # stores them in (image 3 + masks 2 + orientation angle 1 planes of uint8 -- they are 8-bit PNGs,
    # src/utils/camera_utils.py:53-66 -- and the float32 orientation confidence), are widened on the device,
    # GaussianRasterizer(settings)(**tensors) renders, the trainer's image loss (L1 + SSIM + mask + orientation) is
    # evaluated on the render, loss.backward() runs the rasterizer backward, and loss.item() comes back to the host.
    # mine: gaussianhaircut_b200.losses.hair_image_loss (fused kernels); reference arm: the same harness with the
    # reference rasterizer build and the PyTorch loss functions its trainer runs.  At N > 1 the gradients of the op are
    # summed with ONE gh_allreduce_p2p over the arena the backward wrote into (rasterizer.set_gradient_arena).
    e2e = None
    if not args.no_e2e:
        mod = pkg
        gen = torch.Generator(device="cpu").manual_seed(77)
        host_views = []
        for inp in views:
            s = inp["settings"]
            host_views.append({
                "view": s["viewmatrix"].cpu().pin_memory(), "proj": s["projmatrix"].cpu().pin_memory(),
                "campos": s["campos"].cpu().pin_memory(),
                # 8-bit maps as the dataset stores them + float32 confidence
                "u8": torch.randint(0, 256, (6, H, W), dtype=torch.uint8, generator=gen).pin_memory(),
                "conf": torch.rand(1, H, W, generator=gen).pin_memory(),
            })
        params = []
        for inp in views:
            kw = {k: (v.detach().clone().requires_grad_(True) if isinstance(v, torch.Tensor) else v)
                  for k, v in inp["kwargs"].items()}
            params.append(kw)
        h2d = sum(t.numel() * t.element_size() for t in host_views[0].values())
        lambdas = (0.8, 0.2, 0.1, 0.1)      # lambda_dl1, lambda_dssim, lambda_dmask, lambda_dorient (arguments/__init__.py defaults' order)
        if args.impl == "mine":
            from gaussianhaircut_b200 import losses as ghl
            from gaussianhaircut_b200 import rasterizer as ghr

            def image_loss(color, gi, gm, ga, gc):
                return ghl.hair_image_loss(color, gi, gm, ga, gc, *lambdas)[0]
            if par is not None:
                ghr.set_gradient_arena(par.buffer)
        else:
            import loss_oracle

            def image_loss(color, gi, gm, ga, gc):
                return loss_oracle.training_loss(color, gi, gm, ga, gc, *lambdas)[0]

        # A data loader feeds the step: the NEXT step's per-view inputs are copied host->device on a side stream into
        # one of two device slots while the current step computes (same harness for both arms); every copy of every
        # step lies inside the timed region.
        copy_stream = torch.cuda.Stream(device=device)
        slots = [{"u8": torch.empty((6, H, W), dtype=torch.uint8, device=device), "conf": torch.empty((1, H, W), device=device),
                  "view": torch.empty(4, 4, device=device), "proj": torch.empty(4, 4, device=device),
                  "campos": torch.empty(3, device=device), "ready": torch.cuda.Event(), "free": torch.cuda.Event()} for _ in range(2)]
        for sl in slots:
            sl["free"].record(torch.cuda.current_stream(device))

        def copy_in(sl, hv):
            for k in ("u8", "conf", "view", "proj", "campos"):
                sl[k].copy_(hv[k], non_blocking=True)

        def prefetch(i):
            sl, hv = slots[i % 2], host_views[i % len(views)]
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(sl["free"])                # the step that last used this slot is done
                copy_in(sl, hv)
                sl["ready"].record(copy_stream)

        e2e_state = {"next": 0, "overlap": True}

        def e2e_step(i):
            j = i % len(views)
            s = views[j]["settings"]
            sl = slots[i % 2]
            cur = torch.cuda.current_stream(device)
            if e2e_state["overlap"]:
                if e2e_state["next"] <= i:                        # first step of a timed run: nothing prefetched yet
                    prefetch(i)
                    e2e_state["next"] = i + 1
                cur.wait_event(sl["ready"])
                prefetch(i + 1)                                   # overlaps with this step's compute
                e2e_state["next"] = i + 2
            else:                                                 # serial loader: copy, then compute, on one stream
                copy_in(sl, host_views[j])
            settings = mod.GaussianRasterizationSettings(
                image_height=s["image_height"], image_width=s["image_width"], tanfovx=s["tanfovx"],
                tanfovy=s["tanfovy"], bg=s["bg"], scale_modifier=1.0, viewmatrix=sl["view"], projmatrix=sl["proj"],
                sh_degree=s["sh_degree"], campos=sl["campos"], prefiltered=s["prefiltered"], debug=False)
            rast = mod.GaussianRasterizer(raster_settings=settings)
            kw = params[j]
            for v in kw.values():
                if isinstance(v, torch.Tensor):
                    v.grad = None
            # widen the 8-bit maps on the device (what `PILtoTorch(...)/255` did once on the host in the reference loader)
            maps = sl["u8"].float().mul_(1.0 / 255.0)
            color, _radii = rast(**kw)
            loss = image_loss(color, maps[0:3], maps[3:5], maps[5:6], sl["conf"])
            loss.backward()
            sl["free"].record(cur)
            if use_dist:
                if par is not None:
                    par.all_reduce(n_floats=native.trainable_floats(P) if args.mode == "native" else native.arena_floats(P))
                else:
                    for v in kw.values():
                        if isinstance(v, torch.Tensor) and v.grad is not None:
                            dist.all_reduce(v.grad, op=dist.ReduceOp.SUM)
            last["loss"] = float(loss.item())          # device -> host read of the step's result

        # warm-up must visit every cycled view once: workspace sizes depend on the view (R varies), and a
        # first-use cudaMalloc inside the timed region would be charged to the step
        for i in range(len(views) + max(3, args.warmup)):
            e2e_step(i)
        e2e_steps = max(2 * len(views), args.steps // 2)
        # both loader styles are measured and the faster one is reported for this arm (the reference's
        # synchronous cudaMemcpy/cudaMemset inside its forward serialise against a concurrent H2D stream)
        results = {}
        for overlap in (True, False):
            e2e_state["overlap"] = overlap
            torch.cuda.synchronize(); copy_stream.synchronize()
            e2e_state["next"] = 0
            for sl in slots:
                sl["free"].record(torch.cuda.current_stream(device))
            for i in range(3):
                e2e_step(i)
            torch.cuda.synchronize(); copy_stream.synchronize()
            e2e_state["next"] = 0
            reps = [timed(e2e_steps, e2e_step) for _ in range(3)]
            results[overlap] = statistics.median(reps)
            copy_stream.synchronize()
        if args.impl == "mine" and par is not None:
            ghr.set_gradient_arena(None)
        best_overlap = min(results, key=results.get)
        ms_e2e = results[best_overlap]
        e2e_value = (e2e_steps * P * n_eff) / (ms_e2e * 1e-3)
        e2e = {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": 4,
               "ms_per_step": ms_e2e / e2e_steps, "steps": e2e_steps, "repeats": 3,
               "loader": "prefetch on a copy stream" if best_overlap else "serial copy on the compute stream",
               "ms_per_step_prefetch": results[True] / e2e_steps, "ms_per_step_serial": results[False] / e2e_steps,
               "image_loss": "gh_image_loss (hair_image_loss)" if args.impl == "mine" else "PyTorch loss functions of the reference trainer (oracle/loss_oracle.py)",
               "api": "per step: camera + the view's supervision maps (6 uint8 planes + float32 confidence) from pinned host memory "
                      "(double-buffered on a copy stream), GaussianRasterizer(...)(**tensors), the trainer's image loss on the "
                      "render, autograd backward" + (", one gh_allreduce_p2p over the gradient arena" if (use_dist and par is not None) else "") +
                      ", loss.item() read back"}
        log(f"[bench] e2e: {ms_e2e / e2e_steps:.3f} ms/step -> {e2e_value / 1e6:.1f} M Gaussians/s (loss {last['loss']:.4g})")

    # ---------------------------------------------------------------- per-stage timing -> roofline
    roofline = None
    stages = None
    peak, peak_src = measured_peak_gbs()
    stage_bytes, path_bytes = algorithmic_bytes(P, last["R"], W, H, T, args.mode)
    if args.impl == "mine" and rank == 0 and not args.no_roofline:
        lib = _capi.load()
        lib.gh_stage_timing_enable(1)
        nrf = max(5, args.steps // 2)
        for i in range(nrf):
            step(i, arena=False)
        torch.cuda.synchronize()
        st = _capi.stage_timing_read()
        lib.gh_stage_timing_enable(0)
        stages = {}
        if st.get("tile_sort", (0.0, 0))[1] == 0:
            # every tile list fitted the forward CTA's shared memory: the sort (read + write back of the
            # 8-byte records) ran inside blend_forward, so its bytes belong to that kernel
            stage_bytes["blend_forward"] += 8 * last["R"]
        for name, (ms, calls) in st.items():
            if calls == 0:
                continue
            avg = ms / calls
            gbs = stage_bytes[name] / (avg * 1e-3) / 1e9 if avg > 0 else 0.0
            stages[name] = {"ms": avg, "alg_bytes": int(stage_bytes[name]), "gbs": gbs, "frac": gbs / peak}
        dom = max(stages, key=lambda k: stages[k]["ms"])
        traffic = None
        try:     # DRAM bytes per launch of that kernel from the committed ncu --set full capture
            import glob
            tf = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_traffic.json")))[-1]
            traffic = json.load(open(tf)).get(dom) if args.mode == "native" else None
        except Exception:
            traffic = None
        roofline = {"bound": "hbm", "kernel": dom, "achieved": stages[dom]["gbs"], "peak": peak, "unit": "GB/s",
                    "frac": stages[dom]["frac"], "traffic": traffic, "peak_source": peak_src,
                    "ms": stages[dom]["ms"], "alg_bytes": stages[dom]["alg_bytes"],
                    "timing": f"CUDA events around each stage on the launching stream, {nrf} steps after the timed region"}
    if use_dist:
        dist.barrier()

    # ---------------------------------------------------------------- baseline: the reference CUDA build
    cpu_baseline = None
    sm_count = torch.cuda.get_device_properties(device).multi_processor_count
    if args.impl == "mine" and rank == 0 and N == 1 and not args.no_cpu_baseline:
        if build_ref.is_built():
            refmod = build_ref.load()._C
            for i in range(3):
                step(i, mod=refmod, arena=False)
            ms_ref = timed(args.ref_steps, lambda i: step(i, mod=refmod, arena=False))
            ref_value = args.ref_steps * P / (ms_ref * 1e-3)
            cpu_baseline = {"value": ref_value, "unit": UNIT, "cores": sm_count, "kind": "reference",
                            "ms_per_step": ms_ref / args.ref_steps,
                            "sample": f"{args.ref_steps} steps of the same workload; the reference has no CPU rasterizer, "
                                      f"this is its own CUDA extension (oracle/_ref, sm_100a) on the same B200, {sm_count} SMs"}
            log(f"[bench] reference CUDA build: {ms_ref / args.ref_steps:.3f} ms/step -> {ref_value / 1e6:.1f} M Gaussians/s")
        else:
            cpu_baseline = {"value": None, "unit": UNIT, "cores": sm_count, "kind": "reference",
                            "sample": "oracle/_ref not built on this box"}
    # (the optimizer / training-iteration figures run LAST so that they cannot perturb the headline sections: the
    #  reference leg measured 2x slower when it ran after them in the same process)
    # ---------------------------------------------------------------- second figure: + Adam step (BASELINE config 3)
    with_adam = None
    if args.mode == "native" and not use_dist:
        pnames = ("means3D", "scales", "rotations", "colors_precomp", "opacities")
        gnames = ("means3D", "scales", "rotations", "colors", "opacity")
        # the op's inputs are activated values (not the trainer's log-/logit-space parameters): keep the
        # updates negligible so that the workload (R, splat sizes) stays the one being measured
        lrs = (1e-9, 1e-10, 1e-9, 1e-9, 1e-9)
        kw0 = packed[0][1]
        plist = [kw0[n] for n in pnames]
        if args.impl == "mine":
            from gaussianhaircut_b200.optim import FusedAdam
            opt = FusedAdam([{"params": [p], "lr": lr} for p, lr in zip(plist, lrs)], eps=1e-15)

            def adam_step(i):
                step(0)
                opt.step(grads=[last["views"][g].reshape(p.shape) for g, p in zip(gnames, plist)])
        else:
            for p in plist:
                p.requires_grad_(True)
            opt = torch.optim.Adam([{"params": [p], "lr": lr} for p, lr in zip(plist, lrs)], lr=0.0, eps=1e-15)
            gidx = {"means3D": 3, "scales": 7, "rotations": 8, "colors": 1, "opacity": 2}   # positions in the 9-tuple

            def adam_step(i):
                step(0)
                g9 = last["grads"]
                for gname, p in zip(gnames, plist):
                    p.grad = g9[gidx[gname]].reshape(p.shape)
                # the reference trainer's NaN guard: one blocking .isnan().any() per parameter (train_gaussians.py:175-178)
                for p in plist:
                    if p.grad is not None and p.grad.isnan().any():
                        opt.zero_grad(set_to_none=True)
                opt.step()
                opt.zero_grad(set_to_none=True)
        with torch.no_grad():
            saved = [p.detach().clone() for p in plist]
            for i in range(3):
                adam_step(i)
            ms_adam = timed(args.steps, adam_step)
            for p, q in zip(plist, saved):
                p.copy_(q)                                   # restore the scene for the following sections
        with_adam = {"ms_per_step": ms_adam / args.steps, "value": args.steps * P / (ms_adam * 1e-3), "unit": UNIT,
                     "optimizer": "gh_adam_step (fused, device-side NaN guard)" if args.impl == "mine"
                                  else "torch.optim.Adam + per-parameter isnan().any() host syncs (reference trainer)",
                     "parameters": list(pnames)}
        log(f"[bench] +Adam: {with_adam['ms_per_step']:.3f} ms/step -> {with_adam['value'] / 1e6:.1f} M Gaussians/s")

    # ---------------------------------------------------------------- third figure: the training iteration built so far
    # forward -> image-space losses (dL/dout) -> backward -> Adam: the op plus its two neighbours
    # ('next' rows 4 and 2).  Reference arm: the reference CUDA rasterizer + the PyTorch loss the reference
    # trainer runs (oracle/loss_oracle.py, a restatement of src/utils/loss_utils.py) through autograd +
    # torch.optim.Adam with the trainer's NaN host syncs.
    train_iter = None
    if args.mode == "native" and not use_dist and with_adam is not None:
        gen = torch.Generator(device="cpu").manual_seed(11)
        gt_image = torch.rand(3, H, W, generator=gen).to(device)
        gt_mask = ((torch.rand(2, H, W, generator=gen) > 0.3).float() * (0.5 + 0.5 * torch.rand(2, H, W, generator=gen))).to(device)
        gt_angle = torch.rand(1, H, W, generator=gen).to(device)
        gt_conf = torch.rand(1, H, W, generator=gen).to(device)
        lambdas = (0.8, 0.2, 0.1, 0.1)      # lambda_dl1, lambda_dssim, lambda_dmask, lambda_dorient
        fw0, kw0, s0, e0, g0 = packed[0]

        def bw_args(radii, geom, R, binning, img, dLt):
            return (s0["bg"], kw0["means3D"], radii, g0("colors_precomp"), g0("scales"), g0("rotations"), s0["scale_modifier"],
                    g0("cov3D_precomp"), g0("conic_precomp"), s0["viewmatrix"], s0["projmatrix"], s0["tanfovx"], s0["tanfovy"],
                    dLt, e0, s0["sh_degree"], s0["campos"], geom, R, binning, img, False)

        if args.impl == "mine":
            from gaussianhaircut_b200 import losses as ghl
            ws = torch.empty(ghl.workspace_elems(W, H), dtype=torch.float64, device=device)

            def loss_only(i):
                last["loss"] = ghl.image_loss_forward_backward(last["color"], gt_image, gt_mask, gt_angle, gt_conf, *lambdas, workspace=ws)

            def iteration(i):
                R, color, radii, geom, binning, img = native.rasterize_gaussians(*fw0)
                losses, dLt = ghl.image_loss_forward_backward(color, gt_image, gt_mask, gt_angle, gt_conf, *lambdas, workspace=ws)
                flat, grads, _ = native.rasterize_gaussians_backward_arena(*bw_args(radii, geom, R, binning, img, dLt))
                opt.step(grads=[grads[g].reshape(p.shape) for g, p in zip(gnames, plist)])
                last["loss"] = losses
        else:
            import loss_oracle

            def loss_only(i):
                c = last["color"].detach().requires_grad_(True)
                with torch.enable_grad():
                    l, _ = loss_oracle.training_loss(c, gt_image, gt_mask, gt_angle, gt_conf, *lambdas)
                    l.backward()
                last["loss"] = l

            def iteration(i):
                R, color, radii, geom, binning, img = native.rasterize_gaussians(*fw0)
                c = color.detach().requires_grad_(True)
                with torch.enable_grad():
                    l, _ = loss_oracle.training_loss(c, gt_image, gt_mask, gt_angle, gt_conf, *lambdas)
                    l.backward()
                g9 = native.rasterize_gaussians_backward(*bw_args(radii, geom, R, binning, img, c.grad))
                for gname, p in zip(gnames, plist):
                    p.grad = g9[gidx[gname]].reshape(p.shape)
                for p in plist:
                    if p.grad is not None and p.grad.isnan().any():
                        opt.zero_grad(set_to_none=True)
                opt.step()
                opt.zero_grad(set_to_none=True)
                last["loss"] = l
        with torch.no_grad():
            last["color"] = native.rasterize_gaussians(*fw0)[1]
            for i in range(3):
                loss_only(i)
            ms_loss = timed(args.steps, loss_only) / args.steps
            saved = [p.detach().clone() for p in plist]
            for i in range(3):
                iteration(i)
            ms_iter = timed(args.steps, iteration) / args.steps
            for p, q in zip(plist, saved):
                p.copy_(q)
        loss_bytes = 100 * W * H      # read render 8 ch + 10 supervision channels... = 60 B/px, write dL 40 B/px
        train_iter = {"ms_per_step": ms_iter, "value": P / (ms_iter * 1e-3), "unit": UNIT,
                      "stages": "rasterizer forward -> image losses (L1 + SSIM + mask + orientation, fwd+bwd) -> rasterizer backward -> Adam",
                      "image_loss_ms": ms_loss,
                      "image_loss_alg_bytes": loss_bytes,
                      "image_loss_frac_of_hbm_peak": (loss_bytes / (ms_loss * 1e-3) / 1e9) / measured_peak_gbs()[0],
                      "image_loss_impl": "gh_image_loss (4 launches)" if args.impl == "mine"
                                         else "PyTorch restatement of the reference's loss_utils + autograd (oracle/loss_oracle.py)"}
        log(f"[bench] iteration (fwd + losses + bwd + Adam): {ms_iter:.3f} ms/step; image losses alone {ms_loss:.3f} ms")

    # ---------------------------------------------------------------- fourth figure: a train_gaussians.py iteration from RAW model parameters
    # What src/train_gaussians.py:96-181 runs per iteration: render(cam, gaussians) -- i.e. the model-side projection
    # preamble (SURVEY.md 8f row 1, a24) + the rasterizer -- then the image losses, backward and the optimizer step over
    # the model's 8 parameter tensors.  mine: renderer.render_raw (fused projection + rasterizer, one autograd node) ->
    # losses.hair_image_loss -> backward -> FusedAdam.  reference: the reference's OWN render() imported unmodified
    # (oracle/ref_python.py) on its own rasterizer build -> the PyTorch losses of its trainer -> torch.optim.Adam with the
    # trainer's per-parameter NaN host syncs.
    train_full = None
    if args.mode == "native" and (rank == 0 or use_dist):          # at N > 1 every rank takes part (one view per rank)
        import types
        import ref_python
        gen = torch.Generator(device="cpu").manual_seed(11)
        gt_image = torch.rand(3, H, W, generator=gen).to(device)
        gt_mask = ((torch.rand(2, H, W, generator=gen) > 0.3).float() * (0.5 + 0.5 * torch.rand(2, H, W, generator=gen))).to(device)
        gt_angle = torch.rand(1, H, W, generator=gen).to(device)
        gt_conf = torch.rand(1, H, W, generator=gen).to(device)
        lambdas = (0.8, 0.2, 0.1, 0.1)
        raw = synth.raw_params_from_scene(scene, "gaussian_model")
        cam_d = synth.make_camera((rank * 8) % 64, W, H)             # rank r renders its own camera
        cam_ns = ref_python.make_camera(cam_d, device)
        bg_t = torch.tensor(synth.BG_DEFAULT, device=device)
        pnames = ("_xyz", "_features_dc", "_features_rest", "_opacity", "_label", "_scaling", "_rotation", "_orient_conf")
        keys = ("xyz", "f_dc", "f_rest", "opacity", "label", "scaling", "rotation", "conf")
        lrs8 = (1e-9,) * 8          # negligible updates: the workload (R, splat sizes) stays the one being measured
        how = None
        if args.impl == "mine":
            from gaussianhaircut_b200 import renderer, losses as ghl
            from gaussianhaircut_b200.optim import FusedAdam
            pc = types.SimpleNamespace(active_sh_degree=3, max_sh_degree=3)
            for n, k in zip(pnames, keys):
                setattr(pc, n, torch.nn.Parameter(raw[k].to(device).contiguous()))
            opt8 = FusedAdam([{"params": [getattr(pc, n)], "lr": lr, "name": n} for n, lr in zip(pnames, lrs8)], eps=1e-15)
            pipe_ns = types.SimpleNamespace(debug=False)

            ws_l = torch.empty(ghl.workspace_elems(W, H), dtype=torch.float64, device=device)
            nan_flag = torch.zeros(1, dtype=torch.int32, device=device)
            par_m = None
            if use_dist:
                # data parallel: the projection backward writes the model gradients (61 floats per Gaussian) into ONE
                # symmetric-memory arena, reduced by ONE gh_allreduce_p2p; its NaN verdict and error flag gate the optimizer
                from gaussianhaircut_b200 import projection
                par_m = ghdist.PeerAllReduce(projection.grad_arena_floats(P_total), device,
                                             use_multicast={"auto": None, "peer-mc": True, "peer-nomc": False, "nccl": None}[args.collective])
                projection.set_gradient_arena(par_m.buffer)
                order8 = ("xyz", "f_dc", "f_rest", "opacity", "label", "scaling", "rotation", "conf")
            else:
                renderer.set_nan_flag(nan_flag)      # single GPU: the NaN guard rides on the projection backward

            def full_iter(i):
                renders, radii, viewspace = renderer.render_raw(cam_ns, pc, pipe_ns, bg_t)
                # loss value + dL/d(render) in one native call; the gradient goes straight into the render's backward
                losses8, dLr = ghl.image_loss_forward_backward(renders.detach(), gt_image, gt_mask, gt_angle, gt_conf, *lambdas, workspace=ws_l)
                renders.backward(dLr)
                if par_m is not None:
                    par_m.all_reduce(n_floats=projection.grad_arena_floats(P_total))
                    a8 = projection.carve_grad_arena(par_m.buffer, P_total)
                    opt8.step(grads=[a8[k] for k in order8], skip_flags=(par_m.error_flag,), nan_flag_in=par_m.nan_flag)
                else:
                    opt8.step(nan_flag_in=nan_flag)
                opt8.zero_grad(set_to_none=True)
                last["loss"] = losses8[0]
            how = "renderer.render_raw (gh_project_forward/backward + rasterizer) -> gh_image_loss -> " + \
                  ("one gh_allreduce_p2p over the model-gradient arena (61 floats per Gaussian) -> " if use_dist else "") + "FusedAdam (8 tensors)"
        elif ref_python.available():
            gr = ref_python.load_renderer("ref")
            import utils.loss_utils as loss_oracle        # the reference's own loss functions (src/utils/loss_utils.py), unmodified
            pc = ref_python.make_gaussian_model(scene, device)
            plist8 = [getattr(pc, n) for n in pnames]
            opt8 = torch.optim.Adam([{"params": [p], "lr": lr, "name": n} for p, n, lr in zip(plist8, pnames, lrs8)], lr=0.0, eps=1e-15)
            pipe_ns = ref_python.pipe()

            def full_iter(i):
                pkg = gr.render(cam_ns, pc, pipe_ns, bg_t)
                # the trainer's loss (train_gaussians.py:126-140) on the maps render() returns
                Ll1 = loss_oracle.l1_loss(pkg["render"], gt_image, mask=gt_mask[1:].detach())
                Lssim = 1.0 - loss_oracle.ssim(pkg["render"] * gt_mask[1:], gt_image * gt_mask[1:])
                Lmask = loss_oracle.l1_loss(pkg["mask"], gt_mask)
                Lor = loss_oracle.or_loss(pkg["orient_angle"], gt_angle, pkg["orient_conf"], weight=torch.ones_like(gt_mask[:1]) * gt_conf, mask=gt_mask[:1])
                if torch.isnan(Lor).any():
                    Lor = torch.zeros_like(Ll1)
                loss = Ll1 * lambdas[0] + Lssim * lambdas[1] + Lmask * lambdas[2] + Lor * lambdas[3]
                loss.backward()
                with torch.no_grad():
                    for p8 in plist8[:7]:
                        if p8.grad is not None and p8.grad.isnan().any():
                            opt8.zero_grad(set_to_none=True)
                    opt8.step()
                    opt8.zero_grad(set_to_none=True)
                last["loss"] = loss
            how = ("the reference's own render() (src/gaussian_renderer/__init__.py:23, imported unmodified) on its own rasterizer build -> "
                   "PyTorch losses of its trainer -> torch.optim.Adam + NaN host syncs")
        if how is not None:
            for i in range(3):
                full_iter(i)
            ms_full = timed(max(5, args.steps // 2), full_iter) / max(5, args.steps // 2)
            if args.impl == "mine":
                renderer.set_nan_flag(None)
                if use_dist:
                    projection.set_gradient_arena(None)
                    if not par_m.ok():
                        raise SystemExit("[bench] gh_allreduce_p2p reported a missing peer during the training-iteration figure")
            train_full = {"ms_per_step": ms_full, "value": n_eff * P_total / (ms_full * 1e-3), "unit": UNIT, "how": how,
                          "parameters": list(pnames), "loss": float(last["loss"].detach())}
            log(f"[bench] train_gaussians.py iteration from raw parameters: {ms_full:.3f} ms/step (loss {train_full['loss']:.5f})")

    if args.impl == "reference":
        cpu_baseline = {"value": value, "unit": UNIT, "cores": sm_count, "kind": "reference",
                        "sample": f"{args.steps} steps of the same workload; the reference's own CUDA extension "
                                  f"(no CPU rasterizer exists), {sm_count} SMs"}

    if rank == 0:
        path_gbs = path_bytes / (ms_per_step * 1e-3) / 1e9
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": N, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "ms_per_step_repeats": [w / args.steps for w in windows], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"strands({args.strands}) = {P_total} Gaussians, {W}x{H}, fwd+bwd, mode={args.mode}",
                       "gaussians_per_view": P, "num_rendered": int(last["R"]), "views_cycled": args.views,
                       "parallelism": f"views sharded one per GPU (dp{N}), one all-reduce of the gradient arena per step: {collective}" if N > 1 else "single GPU",
                       "l2": "per-step footprint ~0.3 GB (83 MB image + 83 MB upstream grad + 68 MB grads + inputs/workspaces) > 126 MB L2; views cycled"},
            "clocks": clocks,
            "e2e": e2e,
            "gpu_launches": gpu_launches,
            "allreduce_check": allreduce_check,
            "roofline": roofline,
            "path_roofline": {"alg_bytes": int(path_bytes), "achieved": path_gbs, "peak": peak, "unit": "GB/s",
                              "frac": path_gbs / peak, "formula": "400P+52R+96WH+24T (344P if conic supplied)"},
            "stages": stages,
            "call_shapes": call_shapes,
            "with_adam": with_adam,
            "train_iteration": train_iter,
            "train_iteration_full": train_full,
            "cpu_baseline": cpu_baseline,
        }
        if args.impl == "reference":
            line["impl"] = "reference"
            line["e2e"] = e2e if e2e is not None else {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
            line["gpu_launches"] = None
        print(json.dumps(line), flush=True)
    if use_dist:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
