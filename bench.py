#!/usr/bin/env python
"""bench.py -- forward+backward views/sec of the Gaussian-splat rasterizer hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Metric (BASELINE.json): forward+backward views/sec @ 3M Gaussians, 1920x1080, SH degree 3,
plus achieved HBM GB/s of the dominant kernel vs the measured peak.  One "step" = one view
rendered forward and backward on each GPU (weak scaling: every rank renders its own view of the
replicated cloud; for N>1 the per-Gaussian gradients are summed over the ranks inside the op's backward,
over peer memory or NCCL -- sugar_b200/parallel.py, --exchange).

Prints ONE JSON line (rank 0).  Keys are documented in DESIGN.md section "Measurement".
  value        views/s, inputs resident in HBM, CUDA-event timed, max over ranks
  e2e          views/s through the public drop-in API with per-step host->device copies of the
               view's camera + upstream image gradient (pinned) and a device->host loss read
  roofline     dominant kernel: algorithmic bytes / CUDA-event duration vs MEASURED_PEAKS.json
  cpu_baseline the CPU oracle (scalar C port of the reference) on a bounded sample
--impl reference runs the UNMODIFIED reference CUDA build (oracle/_ref) through its own
GaussianRasterizer on the same tensors and protocol (the reference has no CPU rasterizer; its
CUDA build is the baseline BASELINE.md section 2 names), falling back to the CPU oracle port
when oracle/_ref is absent.
--dump-outputs DIR writes what the last timed step computed -- the rendered image, radii and every gradient a
caller of the rasterizer receives -- as DIR/<name>.npy (float32; see dump_outputs), so that two builds run with
the same arguments (hence the same seeded inputs) can be compared output for output.
"""
import argparse
import functools
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "forward+backward views/sec @3M Gaussians 1920x1080"


def load_scenes():
    """sugar_b200/scenes.py by path (numpy only).  `import sugar_b200` would map libsugar_b200.so into the
    process, which the reference arm must not do."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("sgr_scenes", os.path.join(ROOT, "sugar_b200", "scenes.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="raster", choices=["raster", "c5", "coarse_sdf_step", "refine_step"],
                    help="raster: the headline (one view per GPU per step, fwd+bwd); c5: BASELINE config 5, a batch of "
                         "8 views of 6M Gaussians at 3840x2160 sharded over the GPUs (strong scaling); the others: "
                         "bench_workloads.py")
    ap.add_argument("--views-per-step", type=int, default=None,
                    help="views in one step's batch, sharded round-robin over the ranks (default: one per GPU)")
    ap.add_argument("--gaussians", type=int, default=None)
    ap.add_argument("--width", type=int, default=None)
    ap.add_argument("--height", type=int, default=None)
    ap.add_argument("--sh-degree", type=int, default=3)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-sh-factors", action="store_true",
                    help="N>1: all-reduce the full dL_dsh instead of all-gathering the SH factors")
    ap.add_argument("--chunks", type=int, default=4,
                    help="N>1: Gaussian ranges of the per-Gaussian backward pass; each range's all-reduce overlaps the next")
    ap.add_argument("--side-stream", action="store_true",
                    help="N>1: finalize each range on a second stream as soon as its collective is done (parallel.ViewParallel)")
    ap.add_argument("--exchange", default="auto", choices=["auto", "peer", "nccl"],
                    help="N>1: how the ranks' gradients meet inside the backward.  peer: the peer-memory kernels "
                         "(csrc/sgr_peer.cu: CUDA IPC mappings, flags, TMA loads / stores over NVLink); nccl: all-gather + "
                         "chunked all-reduce; auto (default): peer on the world sizes it was measured faster on "
                         "(sugar_b200.parallel.PEER_AUTO_WORLDS), else nccl")
    ap.add_argument("--peer", action="store_true", help="same as --exchange peer")
    ap.add_argument("--no-taper", action="store_true",
                    help="N>1, peer exchange: equal chunks instead of halving ones")
    ap.add_argument("--force-exchange", action="store_true",
                    help="diagnostic, N=1: run the exchange path's kernels (factor-mode backward + finalize) without NCCL")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="raster / c5: write the last timed step's image, radii and gradients to DIR/<name>.npy "
                         f"(float32, at most {DUMP_BYTES >> 20} MB in all: larger arrays are sampled, the same elements "
                         "in every run)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.workload not in ("raster", "c5"):
        ap.error("--dump-outputs: only the raster and c5 workloads")
    if args.peer:
        args.exchange = "peer"
    return args


# ---------------------------------------------------------------------------------------------
# algorithmic bytes per kernel launch (DESIGN.md "Algorithmic bytes"; SURVEY.md section 8d)
# P Gaussians, V visible, R instances, T tiles, M stored / D active SH, W x H pixels
# ---------------------------------------------------------------------------------------------
# which resource bounds each kernel (DESIGN.md section 3): the blend kernels do ~256 pair evaluations
# per 40 bytes and are bound by FP32 instruction issue, not by HBM
KERNEL_BOUND = {"preprocess": "hbm", "preprocess_backward": "hbm", "scatter": "l2-atomics", "tile_scan": "latency",
                "tile_sort_smem": "shared-memory", "tile_sort_global": "l2", "blend_forward": "fp32-issue",
                "blend_backward": "fp32-issue", "field_forward": "hbm", "field_backward": "l2-atomics"}


def load_ncu_facts():
    """Per-kernel facts from the committed ncu capture (profiles/ncu_kernels.json, written by
    scripts/summarize_ncu.py): DRAM bytes and warp-instructions per launch at the headline workload."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_kernels.json")) as f:
            return json.load(f)
    except Exception:
        return {}


def algorithmic_bytes(P, V, R, W, H, M, D, sh_written=True):
    """`sh_written`: False in SH factor mode (N > 1), where the per-Gaussian backward does not write dL_dsh."""
    T = ((W + 15) // 16) * ((H + 15) // 16)
    sh = 12 * (D + 1) ** 2
    return {
        "preprocess": P * (44 + sh) + P * 12 + V * 56 + R * 4,
        "tile_scan": T * 12,
        "scatter": P * 8 + V * 4 + R * 12,
        "tile_sort_smem": R * 12,
        "tile_sort_global": R * 12,
        "blend_forward": R * 40 + W * H * 20,
        "blend_backward": R * 40 + W * H * 20 + V * 36 * 2,
        "preprocess_backward": V * (36 + 44 + sh) + P * (92 + (12 * M if sh_written else 0)),
    }


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(index)], stdout=subprocess.PIPE, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def stop(self, load=None, timed=None):
        """`load` = (t0, t1) of the window in which the GPU ran the benchmark's steps back to back (pre-roll +
        timed region + post-roll); only rows stamped inside it count.  `timed` = the timed region itself."""
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons, inside = [], [], set(), 0
        for stamp, r in self.rows:
            if load is not None and not (load[0] + 0.05 <= stamp <= load[1]):
                continue
            if timed is not None and timed[0] <= stamp <= timed[1]:
                inside += 1
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "samples_in_timed_region": inside,
                "window": "steps run back to back from pre-roll through the timed region to post-roll"}


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


DUMP_BYTES = 64 << 20


def dump_outputs(outdir, arrays):
    """Write each tensor of `arrays` as float32 <outdir>/<name>.npy within DUMP_BYTES in all, shared equally.  A tensor
    over its share is replaced by a sample of its flattened elements, drawn by numpy's PCG64 from seed 0 and sorted:
    the same elements in every run with the same arguments."""
    import torch
    os.makedirs(outdir, exist_ok=True)
    share = (DUMP_BYTES // len(arrays) - 4096) // 4   # float32 elements per file; 4 KB for the .npy header
    for name, x in arrays.items():
        a = x.detach()
        if a.numel() > share:
            idx = np.sort(np.random.default_rng(0).choice(a.numel(), share, replace=False))
            a = a.reshape(-1)[torch.from_numpy(idx).to(a.device)]
        np.save(os.path.join(outdir, name + ".npy"), a.float().cpu().numpy())


def _cpu_sample(job):
    """One worker of cpu_baseline(): forward+backward of the C oracle on one 1/64-area sample."""
    seed, P, W, H, D = job
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import helpers as h
    scenes = load_scenes()
    sc = scenes.make_scene(P, W, H, seed=seed)
    dL = scenes.upstream_grad(W, H)
    t0 = time.perf_counter()
    h.run_oracle(sc, np.zeros(3, np.float32), dL, use_sh=True, sh_degree=D)
    return time.perf_counter() - t0


def cpu_baseline(args):
    """The C oracle (port of the reference algorithm; the reference has no CPU rasterizer) on a bounded
    sample, on all host cores: the view is cut into 64 pieces of 1/64 of its area with the same splat
    density (P/64 Gaussians at W/8 x H/8 each); min(cores, 64) of them run concurrently, one per core,
    forward+backward.  views/s = pieces done / 64 / wall time."""
    import concurrent.futures as cf
    import multiprocessing as mp
    f = 8
    P, W, H = args.gaussians // (f * f), args.width // f, args.height // f
    cores = os.cpu_count() or 1
    n = max(1, min(cores, f * f))
    jobs = [(s, P, W, H, args.sh_degree) for s in range(n)]
    with cf.ProcessPoolExecutor(max_workers=n, mp_context=mp.get_context("spawn")) as ex:
        list(ex.map(_cpu_sample, jobs[:n]))  # start the workers / load the library
        t0 = time.perf_counter()
        per = list(ex.map(_cpu_sample, jobs))
        dt = time.perf_counter() - t0
    return {"value": n / (f * f) / dt, "unit": "views/s", "cores": n, "kind": "port",
            "sample": f"{n} of the 64 1/64-area pieces of the workload ({P} Gaussians @ {W}x{H} each, same splat "
                      f"density), one per core, fwd+bwd; {dt:.2f} s wall, {sum(per):.1f} core-seconds",
            "host_cores": cores}


def cpu_baseline_density(args):
    """north_star: the reference's pure-PyTorch density / SDF path (oracle/field_oracle.py restates
    sugar_model.py:730-750, 1247-1316 op for op) timed on the box's host cores, bounded sample."""
    import torch
    from oracle import field_oracle as fo
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    from scipy.spatial import cKDTree
    Pg, N, K = 200_000, 100_000, 16
    g = torch.Generator().manual_seed(0)
    points = torch.randn(Pg, 3, generator=g)
    scaling = torch.exp(torch.randn(Pg, 3, generator=g) * 0.5 - 3.5)
    quats = torch.nn.functional.normalize(torch.randn(Pg, 4, generator=g), dim=-1)
    strengths = torch.sigmoid(torch.randn(Pg, generator=g) * 2.0)
    knn = torch.from_numpy(cKDTree(points.numpy()).query(points.numpy(), k=K, workers=-1)[1].astype(np.int64))
    gi = torch.randint(0, Pg, (N,), generator=g)
    x = points[gi] + fo.quaternion_apply(quats[gi], 1.5 * scaling[gi] * torch.randn(N, 3, generator=g))
    f = lambda a: np.ascontiguousarray(a.numpy())
    case = dict(x=f(x), nbr_idx=f(knn[gi]), gaussian_idx=f(gi), points=f(points), scaling=f(scaling),
                quaternions=f(quats), strengths=f(strengths), density_factor=1.0 / 16.0, density_threshold=1.0)
    fo.field_values(**case)  # warm-up (thread pool, allocator)
    t0 = time.perf_counter()
    reps = 3
    for _ in range(reps):
        fo.field_values(**case)
    dt = (time.perf_counter() - t0) / reps
    return {"value": N / dt, "unit": "samples/s", "cores": cores, "kind": "port",
            "sample": f"density+SDF forward of {N} samples, K={K} neighbours, {Pg} Gaussians, PyTorch CPU "
                      f"({cores} threads), {dt*1e3:.0f} ms per call"}


def verify_exchange(torch, dist, mod, parallel, scenes, dev, rank, world, D, sh_factors, chunks, side_stream=False,
                    peer="auto"):
    """N > 1, before any timing: on a small scene every rank renders its own view twice -- once with the
    exchange inside the backward, once plainly followed by an ordinary all-reduce of each gradient -- and the
    two sets of summed gradients must agree.  Returns the largest |a-b|_inf / |b|_inf over tensors and ranks."""
    P, W, H = 200_000, 640, 360
    sc = scenes.make_scene(P, W, H, seed=3)
    sc = scenes.with_camera_offset(sc, 0.04 * rank, (0.05 * rank, 0.0, 0.0))
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    names = ("means3D", "scales", "rotations", "opacities", "shs")
    dL = t(scenes.upstream_grad(W, H, seed=2 + rank))
    st = mod.GaussianRasterizationSettings(image_height=H, image_width=W, tanfovx=sc.tanfovx, tanfovy=sc.tanfovy,
                                           bg=torch.zeros(3, device=dev), scale_modifier=1.0, viewmatrix=t(sc.viewmatrix),
                                           projmatrix=t(sc.projmatrix), sh_degree=D, campos=t(sc.campos),
                                           prefiltered=False, debug=False)

    def run():
        ps = {k: t(getattr(sc, k)).requires_grad_(True) for k in names}
        m2 = torch.zeros_like(ps["means3D"], requires_grad=True)
        color, _ = mod.GaussianRasterizer(st)(means3D=ps["means3D"], means2D=m2, opacities=ps["opacities"],
                                              shs=ps["shs"], scales=ps["scales"], rotations=ps["rotations"])
        torch.autograd.backward(color, dL)
        return ps
    plain = run()
    for k in names:
        dist.all_reduce(plain[k].grad)
    vp = parallel.ViewParallel(sh_factors=sh_factors, chunks=chunks, side_stream=side_stream, peer=peer)
    worst = 0.0
    with vp.context():
        for _ in range(3):   # three backwards: the peer exchange alternates its factor blocks by step parity
            ex = run()
            for k in names:
                a, b = ex[k].grad, plain[k].grad
                worst = max(worst, float((a - b).abs().max() / b.abs().max().clamp_min(1e-30)))
    w = torch.tensor([worst], device=dev)
    dist.all_reduce(w, op=dist.ReduceOp.MAX)
    worst = float(w.item())
    if not worst <= 1e-4:
        raise RuntimeError(f"view-parallel exchange disagrees with a plain all-reduce: rel err {worst:.3e}")
    used_peer = bool(vp.peer) and any(v is not None for v in vp._peer_states.values())
    out = {"max_rel_err": worst, "tolerance": 1e-4, "scene": f"{P} Gaussians {W}x{H}, one view per rank, 3 backwards",
           "nccl_collectives_per_backward": vp.stats["collectives"] // 3, "peer_memory": used_peer,
           "peer_fallback_reason": vp.peer_error}
    vp.close()
    return out


def main():
    args = parse()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.workload == "c5":   # BASELINE.json configs[4]; SURVEY 8(d): strong scaling of a fixed 8-view batch
        args.gaussians, args.width, args.height = args.gaussians or 6_000_000, args.width or 3840, args.height or 2160
        args.views_per_step = args.views_per_step or 8
    elif args.workload != "raster":
        if rank != 0:
            return 0  # single-GPU workloads: rank 0 alone runs them
        import bench_workloads
        return bench_workloads.run(args, load_scenes(), load_peaks, ClockSampler, cpu_baseline_density)
    args.gaussians = args.gaussians or 3_000_000
    args.width = args.width or 1920
    args.height = args.height or 1080
    import torch
    dist = None
    if world > 1:
        if args.impl == "reference" and rank != 0:
            return 0  # the reference is single-GPU: rank 0 alone runs it
        if args.impl != "reference":
            import torch.distributed as dist
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    P, W, H, D = args.gaussians, args.width, args.height, args.sh_degree

    scenes = load_scenes()
    use_ref = False
    if args.impl == "reference":
        import helpers as h
        if h.have_ref():
            mod = h.load_ref_module()
            use_ref = True
        elif args.dump_outputs:
            raise SystemExit("--dump-outputs: no reference CUDA build (oracle/_ref) to run")
        else:
            # no reference CUDA build on this box: the CPU oracle port is the reference arm
            cb = cpu_baseline(args)
            print(json.dumps({"metric": METRIC, "value": cb["value"], "unit": "views/s", "n_gpus": 1,
                              "steps": 1, "warmup": 0, "ms_per_step": 1000.0 / cb["value"], "higher_is_better": True,
                              "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                              "impl": "reference",
                              "config": {"workload": f"{P} Gaussians (SH deg {D}, M=16) {W}x{H}, 1 view per GPU per step, "
                                                     "fwd+bwd"},
                              "cpu_baseline": cb, "gpu_launches": 0,
                              "e2e": {"value": cb["value"], "unit": "views/s", "h2d_bytes_per_step": 0,
                                      "d2h_bytes_per_step": 0}}))
            return 0
    else:
        from sugar_b200 import diff_gaussian_rasterization as mod
        from sugar_b200 import _lib

    # ---- workload: the same cloud on every rank, one camera per rank (seeded) ----------------
    sc = scenes.make_scene(P, W, H, seed=0)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    params = {k: t(getattr(sc, k)).requires_grad_(True) for k in ("means3D", "scales", "rotations", "opacities", "shs")}
    means2D = torch.zeros_like(params["means3D"], requires_grad=True)
    # every view of the batch looks at the cloud from its own (seeded) pose: rotated about the view axis.  The
    # batch's views are dealt round-robin to the ranks (parallel.shard_views); loss = mean over the batch: the
    # 1/views factor is folded into the upstream gradients.
    views_total = args.views_per_step or max(world, 1)
    my_views = list(range(rank, views_total, max(world, 1))) if not use_ref else [0]
    Pm = scenes.projection_matrix(0.01, 100.0, sc.tanfovx, sc.tanfovy)

    def make_view(v):
        ang = 0.05 * v
        Rz = np.eye(4, dtype=np.float64)
        Rz[0, 0] = Rz[1, 1] = math.cos(ang); Rz[0, 1] = -math.sin(ang); Rz[1, 0] = math.sin(ang)
        host = (torch.from_numpy(Rz.T.astype(np.float32)).pin_memory(),
                torch.from_numpy((Rz.T @ Pm.T).astype(np.float32)).pin_memory(), torch.zeros(3).pin_memory(),
                torch.zeros(3).pin_memory(),
                torch.from_numpy(scenes.upstream_grad(W, H, seed=1 + v) / (views_total if not use_ref else 1)).pin_memory())
        return {"host": host, "dev": tuple(x.to(dev) for x in host)}
    views = [make_view(v) for v in my_views]
    dL_h = views[0]["host"][4]
    viewmatrix, projmatrix, campos, bg, dL = views[0]["dev"]

    def settings(vm, pm, cp, b):
        return mod.GaussianRasterizationSettings(image_height=H, image_width=W, tanfovx=sc.tanfovx, tanfovy=sc.tanfovy,
                                                 bg=b, scale_modifier=1.0, viewmatrix=vm, projmatrix=pm, sh_degree=D,
                                                 campos=cp, prefiltered=False, debug=False)

    exchange_check = None
    if dist is not None or (args.force_exchange and not use_ref):
        # view-parallel exchange inside the op's backward (sugar_b200/parallel.py): SH factors all-gathered,
        # the other 44 B/Gaussian all-reduced chunk by chunk underneath the per-Gaussian pass
        import contextlib
        from sugar_b200 import parallel
        vp = parallel.ViewParallel(sh_factors=not args.no_sh_factors, chunks=args.chunks, side_stream=args.side_stream,
                                   force=args.force_exchange, peer={"auto": "auto", "peer": True, "nccl": False}[args.exchange],
                                   taper=not args.no_taper)
        if dist is not None:
            exchange_check = verify_exchange(torch, dist, mod, parallel, scenes, dev, rank, world, D,
                                             sh_factors=not args.no_sh_factors, chunks=args.chunks,
                                             side_stream=args.side_stream,
                                             peer={"auto": "auto", "peer": True, "nccl": False}[args.exchange])
        stack = contextlib.ExitStack()
        stack.enter_context(vp.context())  # the autograd node keeps the context for the backward thread

    def zero_grads():
        for p in params.values():
            p.grad = None
        means2D.grad = None

    def step_device(keep=None):
        """`keep`: a dict that receives what a caller of the rasterizer gets back from this step."""
        for v, view in zip(my_views, views):   # this rank's views of the batch: each backward runs its own exchange
            vm, pm, cp, b, g = view["dev"]
            rast = mod.GaussianRasterizer(settings(vm, pm, cp, b))
            color, radii = rast(means3D=params["means3D"], means2D=means2D, opacities=params["opacities"],
                                shs=params["shs"], scales=params["scales"], rotations=params["rotations"])
            torch.autograd.backward(color, g)
            if keep is not None:
                sfx = "" if len(views) == 1 else f"_view{v}"
                keep["color" + sfx], keep["radii" + sfx] = color.detach(), radii
        if keep is not None:
            keep.update({"grad_" + k: p.grad for k, p in params.items()}, grad_means2D=means2D.grad)
        zero_grads()
        return radii

    # e2e: every step copies ITS view's camera + upstream image gradient from pinned host memory
    # and reads the scalar loss back.  Like any input pipeline, the copy of step k+1 is issued on
    # a side stream while step k computes (double buffered); it is still one H2D per step inside
    # the timed region.  The loss of every step is copied device -> host into pinned memory on the
    # compute stream (asynchronously, like a training loop that logs without stalling); all reads
    # complete before the timed region closes and are checked afterwards.
    copy_stream = torch.cuda.Stream(device=dev)
    slots = [None, None]
    slot_ready = [torch.cuda.Event(), torch.cuda.Event()]
    e2e_state = {"i": 0}
    loss_ring = torch.full((4096,), float("nan")).pin_memory()

    def prefetch(k, view):
        with torch.cuda.stream(copy_stream):
            slots[k] = tuple(x.to(dev, non_blocking=True) for x in view["host"])
            slot_ready[k].record(copy_stream)

    def step_e2e():
        for n, view in enumerate(views):
            k = e2e_state["i"] & 1
            e2e_state["i"] += 1
            if slots[k] is None:
                prefetch(k, view)
            cur = torch.cuda.current_stream(dev)
            cur.wait_event(slot_ready[k])
            vm, pm, cp, b, g = slots[k]
            for x in slots[k]:
                x.record_stream(cur)  # allocated on the copy stream, consumed on this one
            prefetch(k ^ 1, views[(n + 1) % len(views)])  # the next view's inputs (fresh tensors)
            rast = mod.GaussianRasterizer(settings(vm, pm, cp, b))
            color, radii = rast(means3D=params["means3D"], means2D=means2D, opacities=params["opacities"],
                                shs=params["shs"], scales=params["scales"], rotations=params["rotations"])
            loss = (color * g).sum()
            loss.backward()
            # device -> host read of the view's result
            loss_ring[(e2e_state["i"] - 1) % loss_ring.numel()].copy_(loss.detach(), non_blocking=True)
        zero_grads()

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, last=None):
        """ms per step of `steps` calls of fn; `last`, if given, is called instead of fn for the final step."""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            (last if last is not None and i == steps - 1 else fn)()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1) / steps
        if dist is not None:
            tms = torch.tensor([ms], device=dev)
            dist.all_reduce(tms, op=dist.ReduceOp.MAX)
            ms = float(tms.item())
        return ms

    for _ in range(max(args.warmup, 3)):
        radii = step_device()
    torch.cuda.synchronize()
    V_vis = int((radii > 0).sum())
    # nvidia-smi needs up to a second to deliver its first row and the timed region is short: run the
    # same step back to back before (pre-roll, ~1.2 s) and after (post-roll, ~0.3 s) the timed region, the
    # same number of times on every rank, and keep the clock samples of that whole loaded window.
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5):
        step_device()
    e1.record()
    torch.cuda.synchronize()
    probe_ms = max(e0.elapsed_time(e1) / 5, 0.05)
    rolls = torch.tensor([min(max(int(1200.0 / probe_ms), 50), 2000), min(max(int(300.0 / probe_ms), 10), 500)],
                         device=dev)
    if dist is not None:
        dist.broadcast(rolls, src=0)  # collectives inside the step: every rank must run the same count
    PRE_ROLL, POST_ROLL = (int(v) for v in rolls.tolist())
    clocks = ClockSampler(local)
    t_load0 = time.perf_counter()
    for _ in range(PRE_ROLL):
        step_device()

    # per-kernel durations: every launch bracketed by CUDA events on its own stream.  One GPU: inside the timed region
    # itself (a dozen launches per step).  N > 1: the exchange adds dozens of microsecond-sized launches on side
    # streams whose bracketing would distort the step, so the timed region runs plain and the SAME steps are repeated
    # right after it with the bracketing on (same count on every rank: the steps contain collectives / peer flags).
    profile_in_timed = not use_ref and dist is None
    if profile_in_timed:
        _lib.profile(True)   # allocates the event pool
        step_device()
        torch.cuda.synchronize()
        _lib.profile_read()
    launches0 = 0 if use_ref else _lib.lib.sgr_launch_count()
    t_timed0 = time.perf_counter()
    dumped = {}
    ms = timed(step_device, args.steps, last=functools.partial(step_device, keep=dumped) if args.dump_outputs else None)
    t_timed1 = time.perf_counter()
    launches = 0 if use_ref else int(_lib.lib.sgr_launch_count() - launches0)
    prof = {}
    if profile_in_timed:
        prof = _lib.profile_read()
        _lib.profile(False)
    elif not use_ref:
        _lib.profile(True)
        step_device()
        torch.cuda.synchronize()
        _lib.profile_read()
        for _ in range(args.steps):
            step_device()
        torch.cuda.synchronize()
        prof = _lib.profile_read()
        _lib.profile(False)
    for _ in range(POST_ROLL):
        step_device()
    torch.cuda.synchronize()
    clk = clocks.stop(load=(t_load0, time.perf_counter()), timed=(t_timed0, t_timed1))

    for _ in range(3):
        step_e2e()
    e2e_first = e2e_state["i"]
    ms_e2e = timed(step_e2e, args.steps)
    e2e_losses = loss_ring[[(e2e_first + k) % loss_ring.numel() for k in range(args.steps * len(views))]]
    if not bool(torch.isfinite(e2e_losses).all()):
        raise RuntimeError("e2e: a step's loss did not reach the host")

    # `config` is identical in both arms (the driver compares them); arm-specific facts live elsewhere
    strong = args.views_per_step is not None
    metric = METRIC if args.workload == "raster" and args.gaussians == 3_000_000 and (W, H) == (1920, 1080) else \
        f"forward+backward views/sec @{P} Gaussians {W}x{H}"
    out = {"metric": metric, "value": views_total / (ms * 1e-3) if not use_ref else 1.0 / (ms * 1e-3), "unit": "views/s",
           "n_gpus": 1 if use_ref else world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms,
           "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None, "dtype": "f32",
           "data": "synthetic",
           "config": {"workload": (f"{P} Gaussians (SH deg {D}, M=16) {W}x{H}, " +
                                   (f"a batch of {views_total} views per step sharded over the GPUs" if strong else
                                    "1 view per GPU per step") + ", fwd+bwd"),
                      "visible": V_vis, "l2_policy": "inputs (708 MB of Gaussian parameters) larger than L2; no flush"},
           "parallelism": {"mode": f"view-dp{world}" if world > 1 else "single",
                           "side_stream_finalize": bool(args.side_stream), "forced_exchange": bool(args.force_exchange),
                           "exchange": ("none" if world == 1 else "all-reduce 236 B/Gaussian" if args.no_sh_factors else
                                        f"inside the backward, NCCL: all-gather 12 B/Gaussian/view SH factors under the "
                                        f"per-Gaussian pass + all-reduce 44 B/Gaussian in {args.chunks} overlapped chunks"
                                        if not (exchange_check or {}).get("peer_memory") else
                                        f"inside the backward, over peer memory (CUDA IPC, no NCCL call): the finalize "
                                        f"kernel loads every view's 12 B/Gaussian SH factors from its owner GPU; the "
                                        f"44 B/Gaussian records are reduced by a two-shot P2P kernel in {args.chunks} "
                                        f"chunks under the per-Gaussian pass; flags in peer memory order the ranks"),
                           "exchange_check": exchange_check},
           "clocks": clk}
    if not use_ref:
        out["stage_timing"] = ("CUDA events around every launch inside the timed region" if profile_in_timed else
                               "CUDA events around every launch in a repeat of the timed steps right after the timed region")
    n_e2e = 1 if use_ref else views_total
    out["e2e"] = {"value": n_e2e / (ms_e2e * 1e-3), "unit": "views/s",
                  "h2d_bytes_per_step": int((dL_h.numel() * 4 + (16 + 16 + 3 + 3) * 4) * len(views)),
                  "d2h_bytes_per_step": 4 * len(views),
                  "ms_per_step": ms_e2e,
                  "resident": "the Gaussian parameters (708 MB: the trainer's nn.Parameters) stay device-resident in "
                              "both arms, as in the reference's training loop; per-step H2D = this view's camera "
                              "(38 floats) + upstream image gradient (24.9 MB, pinned, prefetched one step ahead)",
                  "d2h": "the step's loss, copied asynchronously into pinned host memory every step; all reads "
                         "complete inside the timed region (checked finite afterwards)"}
    out["gpu_launches"] = launches
    if use_ref:
        out["impl"] = "reference"
        out["impl_note"] = "unmodified diff-gaussian-rasterization CUDA sources compiled for sm_100a (oracle/_ref)"
        out["gpu_launches"] = 0
    if rank == 0 and not use_ref:
        # R of this view for the byte model
        with torch.no_grad():
            from sugar_b200 import _C
            R = _C.rasterize_gaussians(bg, params["means3D"], torch.Tensor([]), params["opacities"], params["scales"],
                                       params["rotations"], 1.0, torch.Tensor([]), viewmatrix, projmatrix, sc.tanfovx,
                                       sc.tanfovy, H, W, params["shs"], D, campos, False, False)[0]
        # the per-Gaussian pass writes dL_dsh itself on one GPU, with --no-sh-factors, and in the peer-memory exchange
        # (there summed over all views); only the NCCL factor exchange leaves it to the epilogue
        used_peer = bool((exchange_check or {}).get("peer_memory")) or (args.force_exchange and args.exchange != "nccl")
        alg = algorithmic_bytes(P, V_vis, R, W, H, 16, D, sh_written=(world == 1 or args.no_sh_factors or used_peer))
        peak, peak_src = load_peaks()
        ncu = load_ncu_facts()
        sm_clock = (clk.get("sm_mhz") or 1965.0) * 1e6
        issue_peak = 148 * 4 * sm_clock  # warp-instructions / s the chip can issue at the measured clock
        stages = {}
        for name, (tot, cnt) in prof.items():
            avg_ms = tot / cnt
            # a view's pass of this kernel may be split into several launches (the per-Gaussian backward runs in
            # Gaussian-range chunks under the view-parallel exchange): rates are per VIEW PASS, i.e. the byte /
            # instruction model of one view over the summed duration of that view's launches
            pass_ms = tot / (args.steps * len(views))
            b = alg.get(name)
            st = {"ms": round(avg_ms, 4), "launches_per_step": cnt / args.steps, "ms_per_view_pass": round(pass_ms, 4),
                  "gbs": round(b / (pass_ms * 1e-3) / 1e9, 1) if b else None,
                  "hbm_frac": round(b / (pass_ms * 1e-3) / 1e9 / peak, 4) if b else None,
                  "bound": KERNEL_BOUND.get(name, "latency")}
            inst = (ncu.get(name) or {}).get("warp_instructions")
            if inst:
                st["issue_frac"] = round(inst / (pass_ms * 1e-3) / issue_peak, 4)
            stages[name] = st
        dom = max(stages, key=lambda k: stages[k]["ms"] * stages[k]["launches_per_step"]) if stages else None
        if dom:
            facts = ncu.get(dom) or {}
            out["roofline"] = {"kernel": dom, "bound": KERNEL_BOUND.get(dom, "hbm"), "achieved": stages[dom]["gbs"],
                               "peak": peak, "unit": "GB/s",
                               "frac": stages[dom]["hbm_frac"], "traffic": facts.get("dram_bytes"),
                               "peak_source": peak_src, "algorithmic_bytes": alg.get(dom)}
            if facts.get("warp_instructions"):
                # the blend kernels are FP32-issue bound (~256 pair evaluations per 40 bytes): their roofline
                # is the issue rate, warp-instructions (ncu smsp__inst_executed.sum) / duration vs SMs x 4 x clock
                out["roofline"]["issue"] = {
                    "achieved": round(facts["warp_instructions"] / (stages[dom]["ms_per_view_pass"] * 1e-3) / 1e9, 1),
                    "peak": round(issue_peak / 1e9, 1), "unit": "G warp-inst/s", "frac": stages[dom].get("issue_frac"),
                    "warp_instructions": facts["warp_instructions"], "source": facts.get("source")}
            # the HBM-bound stages BASELINE.md holds to >= 60 % of peak
            out["roofline"]["hbm_stages"] = {k: v["hbm_frac"] for k, v in stages.items()
                                             if v["bound"] == "hbm" and v["hbm_frac"] is not None}
        out["stages"] = stages
        out["workload_stats"] = {"num_rendered": R, "visible": V_vis}
        total_alg = sum(alg[k] for k in alg if k in stages)
        out["hbm_gbs_whole_step"] = round(total_alg / (ms * 1e-3) / 1e9, 1)
        if not args.no_cpu_baseline:
            try:
                out["cpu_baseline"] = cpu_baseline(args)
            except Exception as ex:  # the oracle is a checker; never let it break the bench line
                out["cpu_baseline"] = {"error": repr(ex)}
            try:
                out["cpu_baseline_density"] = cpu_baseline_density(args)
            except Exception as ex:
                out["cpu_baseline_density"] = {"error": repr(ex)}
    if use_ref:
        out["cpu_baseline"] = {"value": out["value"], "unit": "views/s", "cores": 0, "kind": "reference",
                               "sample": "full workload on the GPU: the reference path has no CPU implementation"}
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, dumped)
    if rank == 0:
        print(json.dumps(out))
    if dist is not None:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
