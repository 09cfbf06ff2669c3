#!/usr/bin/env python
"""bench.py -- forward+backward views/s of the render hot path on the BASELINE.json workload.

    python bench.py --gpus 1 --steps K --warmup W                 (ours, N=1)
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W                    (ours, N GPUs of one node, NCCL)
    python bench.py --impl reference ...                          (the CPU restatement of the reference path)

Workload (BASELINE.json configs[1], BASELINE.md "Synthetic inputs"): 1M random Gaussians (seed 0), 1920x1080,
sh_degree 3, cameras on the radius-3 Fibonacci sphere.  A step = `views_per_rank` views per rank, each one
render_view forward + ``(img*w).sum()`` backward down to the six parameter gradients, accumulated into the
dense per-Gaussian gradient buffer; with N>1 ranks the buffer is all-reduced once per step (weak scaling:
per-GPU work fixed).  `value` = views of all ranks / max-over-ranks device time, inputs resident in HBM.
`e2e` = same through the public API with the per-view host inputs (camera matrices + uint8 target image in
pinned memory) copied H2D and the loss read back D2H inside the timed region.

Inputs are larger than L2 (236 MB of parameters are streamed by every view), so no explicit L2 flush is needed.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "forward+backward views/sec @1080p 1M Gaussians"
UNIT = "views/s"
PARAM_KEYS = ("xyz", "scale", "rot", "sh_0", "sh_rest", "opacity")


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed steps (at least 1)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--gaussians", type=int, default=1_000_000)
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--height", type=int, default=1080)
    ap.add_argument("--tile", default="8x16", help="8x16 (reference default) | 12x16 | 16x16 | 8x8")
    ap.add_argument("--sh-degree", type=int, default=3)
    ap.add_argument("--views-per-rank", type=int, default=8)
    ap.add_argument("--n-views", type=int, default=64, help="size of the camera lattice the step's views are drawn from")
    ap.add_argument("--cpu-views", type=int, default=2, help="views of the CPU baseline sample (N=1 only)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--level", default="B", choices=["A", "B"], help="B = fused render_view (default), A = op-by-op surface")
    ap.add_argument("--staging", default=None, choices=[None, "bulk", "cpasync"])
    ap.add_argument("--streams", type=int, default=4, help="CUDA streams the views of a step alternate over (1 = serial)")
    ap.add_argument("--config", default="c2", choices=["c2", "c4"],
                    help="c2 = BASELINE.json configs[1] (1M Gaussians, 1080p: the configuration the metric is quoted on; default); "
                         "c4 = configs[3] (5M Gaussians, 3840x2160, log-scales shifted by -0.5: tile-overflow / sort-bound stress)")
    ap.add_argument("--allreduce", default="sync", choices=["sync", "overlap"],
                    help="N>1: sync = the step's all-reduce completes before the next step starts (what synchronous training needs; "
                         "headline); overlap = it hides behind the next step's rendering (gradients one step late)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned (per-view losses, accumulated gradients at a fixed "
                         "sample of Gaussians) as DIR/<name>.npy, to compare the outputs of two builds on identical inputs")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    a.log_scale_range = (0.002, 0.02)
    if a.config == "c4":
        a.gaussians, a.width, a.height = 5_000_000, 3840, 2160
        a.log_scale_range = (0.002 * math.exp(-0.5), 0.02 * math.exp(-0.5))
    return a


# ---------------------------------------------------------------------------------------------------
# helpers
# ---------------------------------------------------------------------------------------------------

class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed region (B200_PROFILING.md recipe).

    nvidia-smi needs a few hundred ms to print its first line, longer than a short timed region, so the sampler is started before
    the warm-up steps (the same workload) and every line carries nvidia-smi's own timestamp; stop() keeps the samples whose
    timestamp falls between mark_begin() and mark_end() (host clock, taken right after the synchronising barriers that bracket
    the timed region).  If none falls inside (very short runs) the samples taken under the warm-up load are reported and
    ``window`` says so."""
    Q = ("timestamp,index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx, self.proc, self.path = gpu_index, None, None
        self.t_begin = self.t_end = None

    def start(self):
        try:
            f = tempfile.NamedTemporaryFile(prefix="clocks_", suffix=".csv", delete=False)
            self.path = f.name
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50",
                                          "-i", str(self.idx)], stdout=f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def mark_begin(self):
        self.t_begin = time.time()

    def mark_end(self):
        self.t_end = time.time()

    @staticmethod
    def _stamp(text):
        """nvidia-smi prints local time as 'YYYY/MM/DD HH:MM:SS.mmm'."""
        import datetime
        try:
            return datetime.datetime.strptime(text.strip(), "%Y/%m/%d %H:%M:%S.%f").timestamp()
        except Exception:
            return None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        try:
            self.proc.terminate()
            self.proc.wait(timeout=5)
        except Exception:
            try:                                        # never leave a polling nvidia-smi behind this process
                self.proc.kill()
                self.proc.wait(timeout=5)
            except Exception:
                pass
        try:
            rows = []                                   # (timestamp or None, sm, max, reasons)
            for line in open(self.path):
                c = [x.strip() for x in line.split(",")]
                if len(c) < 10:
                    continue
                try:
                    sm_, mx_ = float(c[2]), float(c[3])
                except ValueError:
                    continue
                rs = {name for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[6:10])
                      if v.lower().startswith("active")}
                rows.append((self._stamp(c[0]), sm_, mx_, rs))
            inside = [r for r in rows if r[0] is not None and self.t_begin is not None and self.t_end is not None
                      and self.t_begin <= r[0] <= self.t_end]
            window = "timed region"
            if not inside:
                # nothing stamped inside the region: everything sampled since the sampler started (warm-up + timed region, same load)
                inside, window = rows, "warm-up + timed region (no sample stamped inside the timed region)"
            if inside:
                reasons = set()
                for r in inside:
                    reasons |= r[3]
                out = {"sm_mhz": float(np.median([r[1] for r in inside])), "sm_max_mhz": float(max(r[2] for r in inside)),
                       "reasons": sorted(reasons), "samples": len(inside), "window": window, "samples_total": len(rows)}
            os.unlink(self.path)
        except Exception:
            pass
        return out


class StageTimer:
    """CUDA events around each C-ABI call (on the stream the kernels are launched on), to attribute the step
    time to stages and to give the roofline its per-launch duration."""

    def __init__(self):
        self.enabled = False
        self.rec = {}
        self.sort_kernels = 0          # kernels launched by our own radix sort (3 per pass: histogram, row scan, scatter)

    def install(self):
        import torch
        from litegs_b200 import _lib
        orig = _lib.call
        timer = self

        def call(name, *a):
            if not timer.enabled:
                return orig(name, *a)
            e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
            e0.record()
            orig(name, *a)
            e1.record()
            timer.rec.setdefault(name, []).append((e0, e1))
            if os.environ.get("LGS_SORT", "lgs") != "cub":
                if name in ("lgs_sort_pairs_u16", "lgs_sort_pairs_u32"):
                    if not (int(a[6]) - int(a[5]) > 14 and int(a[4]) > (8 << 20)):      # (that case runs the library's onesweep: not ours)
                        timer.sort_kernels += 3 * ((int(a[6]) - int(a[5]) + 7) // 8)
                elif name == "lgs_sort_pairs_u32_rebased":
                    timer.sort_kernels += 3 * ((int(a[6]) + 7) // 8)
                elif name == "lgs_sort_pairs_u32_dev":
                    timer.sort_kernels += 3 * ((int(a[7]) + 7) // 8)
                elif name in ("lgs_sort_pairs_u16_dev", "lgs_sort_pairs_u32k_dev"):
                    timer.sort_kernels += 3 * ((int(a[7]) - int(a[6]) + 7) // 8)
        _lib.call = call

    def summary(self):
        """name -> (total ms, launches)."""
        out = {}
        for name, evs in self.rec.items():
            out[name] = (sum(a.elapsed_time(b) for a, b in evs), len(evs))
        return out


def _list_lengths(ranges, n_pairs):
    """Per-tile list lengths from the range table i32[tiles+2]: entry t (1-based tile id) = first pair of tile t or -1,
    entry tiles+1 = number of pairs; a list ends where the next entry >= 0 begins (an empty tile right after a populated one
    carries that end marker and gets length 0)."""
    import torch
    r = ranges.to(torch.int64)
    ntile = r.shape[0] - 2
    big = torch.full_like(r, n_pairs)
    rr = torch.where(r >= 0, r, big)
    nxt = torch.flip(torch.cummin(torch.flip(rr, [0]), 0).values, [0])       # nxt[t] = smallest entry at or after t
    start = r[1:ntile + 1]
    ln = torch.where(start >= 0, nxt[2:ntile + 2] - start, torch.zeros_like(start))
    return ln.clamp_(min=0)


def load_scene(args):
    from litegs_b200 import scene
    return scene.make_scene(args.gaussians, sh_degree=3, seed=0, log_scale_range=args.log_scale_range)


def camera_np(i, args):
    from litegs_b200 import scene
    return scene.make_camera(i % args.n_views, args.n_views, args.width, args.height)


DUMP_SAMPLE = 65536          # Gaussians whose gradients --dump-outputs writes (59 floats each at sh_degree 3: 15.5 MB)


def dump_outputs(out_dir, losses, grads):
    """--dump-outputs: what a step of render_views hands back to its caller -- the per-view losses it returns and the gradients
    it accumulated into the dense buffer ("_touched" = the per-chunk marks) -- as float32 DIR/<name>.npy.  The per-Gaussian
    gradients are written at DUMP_SAMPLE Gaussian slots drawn with a fixed seed (all of them when there are fewer), in
    ascending slot order, so that every file stays small at any workload size and two runs write the same elements."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    out = {"losses": torch.stack([l_.reshape(()) for l_ in losses]), "touched": grads["_touched"]}
    n = grads["xyz"].shape[-2] * grads["xyz"].shape[-1]
    idx = np.sort(np.random.default_rng(0).choice(n, min(n, DUMP_SAMPLE), replace=False))
    idx_t = torch.from_numpy(idx).to(grads["xyz"].device)
    for k in PARAM_KEYS:
        g = grads[k]
        out[f"grad_{k}"] = g.reshape(*g.shape[:-2], n).index_select(-1, idx_t)
    for name, t in out.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), t.detach().float().cpu().numpy())


def stage_bytes(stats, S, K):
    """Algorithmic bytes per view and stage (DESIGN.md section 5)."""
    Nv, Nmax, D, P, Nvis = stats["Nv"], stats["Nmax"], stats["D"], stats["P"], stats["N_visible"]
    # Gaussians whose record gradient is non-zero: project_backward reads every live slot's 48-byte record gradient but does the
    # parameter work (geometry re-read, read-modify-write of the dense gradient rows) only for these
    Ng = stats.get("N_grad", Nv)
    par = 4 * (3 + 3 + 4 + 3 * K + 1)
    bits_passes = stats["tile_sort_passes"]
    return {
        "lgs_frustum_culling_aabb": 28 * (Nmax // S),
        "lgs_project_forward": par * Nv + 60 * Nmax,
        "lgs_sort_pairs_u32(depth)": (4 + 4 * 16) * Nv,
        "lgs_scan_gathered": 12 * Nv,
        "lgs_emit_pairs": 60 * Nv + 8 * D,
        "lgs_emit_pairs_u16": 60 * Nv + 6 * D,
        "lgs_sort_pairs_u32(tile)": (4 + bits_passes * 16) * D,
        "lgs_sort_pairs_u16(tile)": (2 + bits_passes * 12) * D,
        "lgs_tile_range": 4 * D,
        "lgs_tile_range_u16": 2 * D,
        "lgs_rasterize_forward_packed": 4 * D + 48 * Nvis + 18 * P,
        "lgs_rasterize_backward": 48 * Nmax + 4 * D + 48 * Nvis + 30 * P + 36 * Nvis,
        "lgs_project_backward": 48 * Nv + (44 + 2 * par) * Ng,
        "lgs_sparse_chunk_op": 3 * par * Nv,
    }


# ---------------------------------------------------------------------------------------------------
# CPU arm (oracle): used for cpu_baseline inside the "ours" line and as the whole `--impl reference` run
# ---------------------------------------------------------------------------------------------------

def cpu_views_per_s(args, scene_np, n_views, weights_seed=1):
    import oracle
    # all host threads (torchrun exports OMP_NUM_THREADS=1 to its workers, which would make this a 1-core run)
    oracle.set_num_threads(len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1))
    P = {k: scene_np[k] for k in PARAM_KEYS}
    aabb = (scene_np["cluster_origin"], scene_np["cluster_extend"])
    th, tw = [int(x) for x in args.tile.split("x")]
    H, W = args.height, args.width
    w = np.random.default_rng(weights_seed).standard_normal((1, 3, H, W), dtype=np.float32)
    t0 = time.perf_counter()
    for i in range(n_views):
        cam = camera_np(i, args)
        oracle.render_forward_backward(P, aabb, cam, (H, W), (th, tw), args.sh_degree, lambda img: w)
    dt = time.perf_counter() - t0
    return n_views / dt, dt, oracle.num_threads()


def run_reference(args, rank):
    """The reference has no CPU implementation of this path (SURVEY fact 1); its CPU arm is the oracle port
    (oracle/, C + OpenMP on all host threads), one full-size view per step."""
    if rank != 0:
        return
    scene_np = load_scene(args)
    import oracle
    for _ in range(min(args.warmup, 1)):
        cpu_views_per_s(args, scene_np, 1)
    t0 = time.perf_counter()
    vps, dt, threads = cpu_views_per_s(args, scene_np, max(1, args.steps))
    line = {
        "impl": "reference", "metric": METRIC, "value": vps, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1000.0 * dt / max(1, args.steps), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{args.gaussians} Gaussians, {args.width}x{args.height}, sh_degree {args.sh_degree}, tile {args.tile}",
                   "views_per_step": 1},
        "cpu_baseline": {"value": vps, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": f"{max(1, args.steps)} full-size views, one per step (oracle/, C + OpenMP)"},
        "e2e": {"value": vps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    # informational: the reference's own CUDA kernels (sm_100a build in oracle/_ref) under the same op-level
    # orchestration, when a GPU and the prebuilt module are available.
    try:
        line["ref_cuda"] = ref_cuda_views_per_s(args, scene_np)
    except Exception as e:  # pragma: no cover
        line["ref_cuda"] = {"unavailable": str(e)[:200]}
    emit_line(line)


def ref_cuda_views_per_s(args, scene_np, iters=24):
    """The GPU-side comparison target (informational keys of the reference line): the reference's OWN CUDA kernels (unmodified
    sources built for sm_100a, oracle/_ref) against ours under identical orchestration, in two harnesses:

      *_cold  : litegs_b200.render Level A (op by op), feedback buffers None -- the reference's first-epoch mode with one blocking
                size read-back per view (GR/compact.cu:527-549, GR/binning.cu:137-163);
      *_warm  : the reference's own, unmodified Python (litegs.render.render_preprocess + render from the staged package,
                baseline/_ref) with its pinned feedback buffers filled by a previous pass over the same cameras -- the
                reference's steady-state (best) mode.  `ours_under_reference_python_warm` swaps only the native module."""
    import torch
    if not torch.cuda.is_available():
        raise RuntimeError("no GPU")
    from oracle import build_ref
    mod = build_ref.load()
    if mod is None:
        raise RuntimeError("oracle/_ref not built")
    from litegs_b200 import render, wrapper
    from litegs_b200.arguments import PipelineParams
    ours_mod = __import__("litegs_b200.fused", fromlist=["x"])
    dev = torch.device("cuda:0")
    th, tw = [int(x) for x in args.tile.split("x")]
    pp = PipelineParams(tile_size=(th, tw))
    out = {}
    n_cams = 8
    w = torch.randn((1, 3, args.height, args.width), device=dev)
    cams = [{k: torch.from_numpy(v).to(dev) for k, v in camera_np(i, args).items()} for i in range(n_cams)]
    A = [torch.from_numpy(scene_np[k]).to(dev) for k in ("cluster_origin", "cluster_extend")]

    def timed(one, warm):
        for i in range(warm):
            one(i)
        torch.cuda.synchronize()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(iters):
            one(i)
        e1.record(); torch.cuda.synchronize()
        return {"value": iters / (e0.elapsed_time(e1) / 1000.0), "unit": UNIT}

    for name, backend in (("reference_kernels_cold", mod), ("ours_level_a_cold", ours_mod)):
        wrapper.set_backend(backend)
        try:
            P = {k: torch.from_numpy(scene_np[k]).to(dev).requires_grad_(True) for k in PARAM_KEYS}

            def one(i):
                c = cams[i % n_cams]
                ids, num, cx, cs, cr, col, cop = render.render_preprocess(A[0], A[1], c["frustumplane"], c["view"], P["xyz"], P["scale"],
                                                                          P["rot"], P["sh_0"], P["sh_rest"], P["opacity"], None, None, pp,
                                                                          args.sh_degree)
                img = render.render(c["view"], c["proj"], cx, cs, cr, col, cop, num * pp.cluster_size, None, None, args.sh_degree,
                                    (args.height, args.width), pp)[0]
                (img * w).sum().backward()
                for k in PARAM_KEYS:
                    P[k].grad = None
            out[name] = timed(one, 3)
        finally:
            wrapper.set_backend(ours_mod)
    # the reference's own Python, warm feedback buffers
    try:
        path = build_ref.reference_python_path()
        if path is None:
            raise RuntimeError("reference Python package not staged (baseline/_ref)")
        from litegs_b200 import shims
        shims.install()
        if path not in sys.path:
            sys.path.insert(1, path)
        import litegs
        import litegs.config
        import litegs_fused as ours_pybind_shaped
        W = litegs.utils.wrapper
        lp, op, rpp, dp = litegs.config.get_default_arg()
        rpp.tile_size = (th, tw)
        for name, backend in (("reference_python_warm", mod), ("ours_under_reference_python_warm", ours_pybind_shaped)):
            keep = W.litegs_fused
            W.litegs_fused = backend
            try:
                P = {k: torch.from_numpy(scene_np[k]).to(dev).requires_grad_(True) for k in PARAM_KEYS}
                fb_chunks = torch.zeros(n_cams, dtype=torch.int32).pin_memory()
                fb_alloc = torch.zeros(n_cams, dtype=torch.int32).pin_memory()
                idxs = [torch.tensor([i]) for i in range(n_cams)]

                def one(i):
                    c = cams[i % n_cams]; idx = idxs[i % n_cams]
                    ids, num, cx, cs, cr, col, cop = litegs.render.render_preprocess(A[0], A[1], c["frustumplane"], c["view"], P["xyz"],
                                                                                     P["scale"], P["rot"], P["sh_0"], P["sh_rest"], P["opacity"],
                                                                                     fb_chunks, idx, rpp, args.sh_degree)
                    img = litegs.render.render(c["view"], c["proj"], cx, cs, cr, col, cop, num * rpp.cluster_size, fb_alloc, idx,
                                               args.sh_degree, (args.height, args.width), rpp)[0]
                    (img * w).sum().backward()
                    for k in PARAM_KEYS:
                        P[k].grad = None
                out[name] = timed(one, 2 * n_cams)            # two passes over the cameras: the feedback values are warm
            finally:
                W.litegs_fused = keep
    except Exception as e:  # pragma: no cover
        out["reference_python_warm"] = {"unavailable": str(e)[:300]}
    out["note"] = ("views/s of one GPU, forward + backward of one view at a time, single stream; *_cold = litegs_b200.render (Level A) "
                   "without feedback buffers, *_warm = the reference's unmodified litegs.render with warm pinned feedback buffers; "
                   "reference kernels blend in fp16, ours in fp32")
    return out


# ---------------------------------------------------------------------------------------------------
# ours
# ---------------------------------------------------------------------------------------------------

# instructions the dominant kernels issue per unit of work, calibrated ONCE per kernel version from an ncu capture
# (profiles/ncu_raster_r2a_v2_8x16.txt: smsp__inst_executed.sum / work units of that launch) -- the work units themselves are
# counted in-run, so the issue roofline follows the workload and the clocks of THIS run
ISSUE_MODEL = {
    # kernel: (warp instructions per (tile, splat) iteration, description of the unit)
    "lgs_rasterize_backward": {"8x16": 135.7, "unit": "(tile, splat) iterations = sum over tiles of the deepest consumed list position",
                               "source": "profiles/ncu_all_kernels_r2g_c2.txt launch 23: 225.07 M warp instructions / 1.659 M iterations"},
}


def run_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from litegs_b200 import _lib, dist as lgs_dist, pipeline, render
    from litegs_b200.arguments import PipelineParams

    dev = torch.device(f"cuda:{local_rank}")
    torch.cuda.set_device(dev)
    _lib.load()
    if args.staging:
        _lib.call("lgs_set_staging", 1 if args.staging == "bulk" else 0)
    th, tw = [int(x) for x in args.tile.split("x")]
    H, W = args.height, args.width
    pp = PipelineParams(tile_size=(th, tw), sparse_grad=True)

    scene_np = load_scene(args)
    P = {k: torch.from_numpy(scene_np[k]).to(dev).requires_grad_(True) for k in PARAM_KEYS}
    A = [torch.from_numpy(scene_np[k]).to(dev) for k in ("cluster_origin", "cluster_extend")]
    C_chunks, S = P["xyz"].shape[-2:]
    K = (args.sh_degree + 1) ** 2
    vpr = args.views_per_rank
    my_views = [rank + world * j for j in range(vpr)]
    cams_np = [camera_np(v, args) for v in my_views]
    cams = [{k: torch.from_numpy(v).to(dev) for k, v in c.items()} for c in cams_np]
    g = torch.Generator(device="cpu").manual_seed(1)
    w_host = torch.randn((1, 3, H, W), generator=g)
    w = w_host.to(dev)
    # sync (headline): one gradient buffer, the step's all-reduce is enqueued on the compute stream and the next step starts
    # after it -- the dependency synchronous training has (next forward <- optimizer <- reduced gradients).
    # overlap (reported beside it): two buffers, step k's all-reduce runs on a side stream behind step k+1's rendering, which
    # corresponds to applying gradients one step late.
    overlap = world > 1 and args.allreduce == "overlap" and args.level == "B"
    accs = [lgs_dist.GradAccumulator(P), lgs_dist.GradAccumulator(P)] if overlap else [lgs_dist.GradAccumulator(P)]
    acc = accs[0]
    step_no = {"k": 0}
    timer = StageTimer(); timer.install()
    comm_events = []

    acc_views_all = [a.grads() for a in accs]
    n_streams = max(1, args.streams) if args.level == "B" else 1

    def render_one_level_a(cam, weight):
        ids, num, cx, cs, cr, col, cop = render.render_preprocess(A[0], A[1], cam["frustumplane"], cam["view"], P["xyz"], P["scale"],
                                                                  P["rot"], P["sh_0"], P["sh_rest"], P["opacity"], None, None, pp,
                                                                  args.sh_degree)
        img = render.render(cam["view"], cam["proj"], cx, cs, cr, col, cop, num * pp.cluster_size, None, None, args.sh_degree,
                            (H, W), pp)[0]
        loss = (img * weight).sum()
        loss.backward()
        ids_ = P["xyz"].grad.chunk_ids
        cnt = torch.full((1,), ids_.shape[0], dtype=torch.int32, device=dev)
        acc.add_view({k: P[k].grad.compacted_values for k in PARAM_KEYS}, ids_, cnt)
        for k in PARAM_KEYS:
            P[k].grad = None
        return loss.detach()

    def run_views(camera_fn, loss_fn, serial=False):
        """One step's views through the public API: litegs_b200.render.render_views (fused level B: views pipelined over
        CUDA streams, gradients accumulated into the dense buffer by the backward kernel) or the op-by-op level A."""
        if args.level == "B":
            return render.render_views(vpr, camera_fn, loss_fn, A[0], A[1], P["xyz"], P["scale"], P["rot"], P["sh_0"], P["sh_rest"],
                                       P["opacity"], args.sh_degree, (H, W), pp, acc_views_all[step_no["k"] % len(accs)],
                                       n_streams=n_streams)
        return [render_one_level_a(camera_fn(j), loss_fn(j, None)) for j in range(vpr)]

    def reduce_step(a, record):
        """The step's only exchange: one all-reduce of the dense gradient buffer (+ chunk marks)."""
        if world == 1:
            return
        if overlap:
            a.all_reduce(async_op=True)
            return
        if record:
            c0 = torch.cuda.Event(enable_timing=True); c1 = torch.cuda.Event(enable_timing=True)
            c0.record()
            a.all_reduce(async_op=False)          # enqueued in stream order on the compute stream: the next step starts after it
            c1.record()
            comm_events.append((c0, c1))
        else:
            a.all_reduce(async_op=False)

    last_losses = []

    def step(serial=False, record=False):
        a = accs[step_no["k"] % len(accs)]
        a.wait()                      # overlap mode: this buffer's previous all-reduce (two steps ago) must have landed
        a.zero_()
        if args.level == "B":
            last_losses[:] = run_views(lambda j: cams[j], lambda j, img: (img * w).sum(), serial)
        else:
            last_losses[:] = run_views(lambda j: cams[j], lambda j, img: w, serial)
        reduce_step(a, record)
        step_no["k"] += 1

    def barrier():
        for a in accs:
            a.wait()                  # every step's all-reduce is inside the timed region
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---- value: inputs resident ------------------------------------------------------------------
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()                   # before the warm-up: nvidia-smi's first line takes longer than a short timed region
    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    barrier()
    sampler.mark_begin()
    e0.record()
    for _ in range(args.steps):
        step(record=True)
    for a in accs:
        a.wait()
    e1.record()
    barrier()
    sampler.mark_end()
    clocks = sampler.stop() if rank == 0 else None
    ms = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last_losses, accs[(step_no["k"] - 1) % len(accs)].grads())
    comm_ms = sum(a_.elapsed_time(b_) for a_, b_ in comm_events) / max(1, len(comm_events)) if comm_events else 0.0
    # stage attribution / roofline durations: the same steps once more on ONE stream with CUDA events around every
    # C-ABI call (with overlapping streams a kernel's event-to-event time includes the other stream's work).
    # (CUDA graphs off and one view at a time on ONE stream for this pass: the C-ABI calls have to be visible one by one)
    timer.enabled = True
    graphs_keep, n_streams_keep = pipeline.GRAPHS_ENABLED, n_streams
    pipeline.GRAPHS_ENABLED, n_streams = False, 1
    s0 = torch.cuda.Event(enable_timing=True); s1 = torch.cuda.Event(enable_timing=True)
    s0.record()
    for _ in range(args.steps):
        step(serial=True)
    s1.record()
    barrier()
    timer.enabled = False
    pipeline.GRAPHS_ENABLED, n_streams = graphs_keep, n_streams_keep
    ms_serial = s0.elapsed_time(s1)
    # max over ranks of the step time; per-rank render time and all-reduce time gathered for the imbalance / limiter report
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    per_rank = torch.tensor([ms, comm_ms * args.steps], dtype=torch.float64, device=dev)
    gathered = [torch.zeros_like(per_rank) for _ in range(world)] if world > 1 else [per_rank]
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_gather(gathered, per_rank)
    ms = float(t.item())
    total_views = vpr * world * args.steps
    value = total_views / (ms / 1000.0)

    # ---- N > 1: the other all-reduce schedule, reported beside the headline -------------------------------
    other = None
    if world > 1 and args.level == "B":
        alt = "overlap" if not overlap else "sync"
        accs2 = [lgs_dist.GradAccumulator(P), lgs_dist.GradAccumulator(P)] if alt == "overlap" else [accs[0]]
        views2 = [a.grads() for a in accs2]
        k2 = {"k": 0}

        def step2():
            a = accs2[k2["k"] % len(accs2)]
            a.wait(); a.zero_()
            render.render_views(vpr, lambda j: cams[j], lambda j, img: (img * w).sum(), A[0], A[1], P["xyz"], P["scale"], P["rot"],
                                P["sh_0"], P["sh_rest"], P["opacity"], args.sh_degree, (H, W), pp, views2[k2["k"] % len(accs2)],
                                n_streams=n_streams)
            a.all_reduce(async_op=(alt == "overlap"))
            k2["k"] += 1
        for _ in range(3):
            step2()
        for a in accs2:
            a.wait()
        barrier()
        o0 = torch.cuda.Event(enable_timing=True); o1 = torch.cuda.Event(enable_timing=True)
        o0.record()
        for _ in range(args.steps):
            step2()
        for a in accs2:
            a.wait()
        o1.record()
        barrier()
        t3 = torch.tensor([o0.elapsed_time(o1)], dtype=torch.float64, device=dev)
        dist.all_reduce(t3, op=dist.ReduceOp.MAX)
        other = {"allreduce": alt, "value": total_views / (float(t3.item()) / 1000.0), "unit": UNIT,
                 "note": ("all-reduce of step k hidden behind the rendering of step k+1 (two buffers): gradients are applied one step "
                          "late; NOT the headline") if alt == "overlap" else "all-reduce completes before the next step starts"}
        del accs2, views2

    # per-view workload statistics (for the roofline arithmetic), from one extra un-timed view
    with torch.no_grad():
        params = {k: P[k].detach() for k in PARAM_KEYS}
        _, st, _ = pipeline.render_view_forward(params, A[0], A[1], cams[0]["frustumplane"], cams[0]["view"], cams[0]["proj"],
                                                args.sh_degree, (H, W), (th, tw))
        gx, gy = (W + tw - 1) // tw, (H + th - 1) // th
        lens = _list_lengths(st.ranges[0], st.n_pairs)
        kmax_t = st.last[0, 0].view(torch.uint16).to(torch.int32).reshape(gy, th, gx, tw).amax(dim=(1, 3))   # per-tile backward trip count
        stats = {"Nv": st.n_chunks_visible * S, "Nmax": C_chunks * S, "D": st.n_pairs, "P": gx * tw * gy * th,
                 "N_visible": int((st.tile_count[: st.n_chunks_visible * S] > 0).sum().item()),
                 "tiles": gx * gy, "tile_sort_passes": math.ceil((gx * gy).bit_length() / 8),
                 "mean_contributors_per_pixel": float(st.last.view(torch.uint16).float().mean().item()),
                 "max_list_len": int(lens.max().item()), "mean_list_len": float(lens.float().mean().item()),
                 "backward_tile_splat_iterations": int(kmax_t.sum().item())}
        try:
            # how many Gaussians receive a gradient from this view (the others are behind saturated pixels): one un-timed backward
            # with the bench's loss weights, count the non-zero 48-byte record gradients
            d_pad = torch.zeros((1, 3, gy * th, gx * tw), dtype=torch.float32, device=dev)
            d_pad[..., :H, :W] = w
            _, pg = pipeline.render_view_backward(params, st, d_pad, accumulate_into=None)
            stats["N_grad"] = int((pg[0, : st.n_chunks_visible * S] != 0).any(dim=1).sum().item())
            del d_pad, pg
        except Exception as e:                                   # statistics only: never fail the run over it
            print(f"[bench] N_grad not measured ({e}); project_backward bytes use N_v", file=sys.stderr)

    # ---- e2e: host inputs, H2D + D2H inside the timed region ------------------------------------------
    e2e = None
    if not args.no_e2e:
        gt_host = [(torch.rand((1, 3, H, W), generator=g) * 255).to(torch.uint8).pin_memory() for _ in range(2)]
        cam_host = [{k: torch.from_numpy(v).pin_memory() for k, v in c.items()} for c in cams_np]
        h2d = sum(v.numel() * v.element_size() for v in cam_host[0].values()) + gt_host[0].numel()
        losses = []

        # the step's losses are read on the host one step late (double-buffered pinned target + event), so that the host
        # can enqueue step k+1 while the device still runs step k; every step's result is still read inside the timed region
        loss_hosts = [torch.zeros(vpr, dtype=torch.float32).pin_memory() for _ in range(2)]
        loss_ev = [torch.cuda.Event(), torch.cuda.Event()]
        pending = {"k": None}

        # target images: a fixed device buffer per view of the step, filled from pinned memory on a copy stream BEFORE the view's
        # forward is enqueued (no allocation inside the loop, the copy overlaps the view's own kernels)
        copy_stream = torch.cuda.Stream(device=dev)
        gt_dev = [torch.empty((1, 3, H, W), dtype=torch.uint8, device=dev) for _ in range(vpr)]
        gt_ready = [None] * vpr
        gt_consumed = [None] * vpr

        e2e_mode = os.environ.get("LGS_E2E_MODE", "C")     # experiment switch: A autograd loss, B fused loss on the view stream, C + copy stream

        def e2e_camera(j):          # H2D of the view's camera on the view's stream; the target image is prefetched on the copy stream
            cam = {k: v.to(dev, non_blocking=True) for k, v in cam_host[j].items()}
            if e2e_mode != "C":
                return cam
            if gt_consumed[j] is not None:
                copy_stream.wait_event(gt_consumed[j])       # last step's loss of this slot has read the buffer
            with torch.cuda.stream(copy_stream):
                gt_dev[j].copy_(gt_host[j % 2], non_blocking=True)
                ev = torch.cuda.Event(); ev.record(copy_stream)
            gt_ready[j] = ev
            return cam

        def e2e_loss(j, img):       # (H2D of the uint8 target was started before the view's forward), loss, D2H of the result
            cur = torch.cuda.current_stream(dev)
            if e2e_mode == "A":
                gt = gt_host[j % 2].to(dev, non_blocking=True)
                weight = torch.sub(gt, 127.5)
                if img is None:
                    return weight * (1.0 / 255.0)
                loss = (img * weight).sum() * (1.0 / 255.0)
                loss_hosts[step_no["k"] % 2][j:j + 1].copy_(loss.detach().reshape(1), non_blocking=True)
                return loss
            if e2e_mode == "B":
                gt_dev[j].copy_(gt_host[j % 2], non_blocking=True)
            else:
                cur.wait_event(gt_ready[j])
            gt = gt_dev[j]
            # loss = sum(img * (gt/255 - 0.5)) and its gradient (gt - 127.5)/255, handed to the rasterizer directly
            # (render_views' loss-and-gradient form): two elementwise kernels and one dot product per view
            d_img = torch.sub(gt, 127.5).mul_(1.0 / 255.0)
            ev = torch.cuda.Event(); ev.record(cur)
            gt_consumed[j] = ev
            if img is None:
                return d_img
            with torch.no_grad():          # img may be an autograd leaf (render_views' loss_fn form): the gradient is returned explicitly,
                loss = torch.dot(img.reshape(-1), d_img.reshape(-1))    # and a graph hanging off the pinned result buffer would keep every d_img alive
            loss_hosts[step_no["k"] % 2][j:j + 1].copy_(loss.detach().reshape(1), non_blocking=True)
            return loss, d_img

        def read_losses(k):         # D2H results of step k: wait for its event, then read the pinned buffer
            loss_ev[k % 2].synchronize()
            losses.append(float(loss_hosts[k % 2].detach().sum()))

        trace = [] if os.environ.get("LGS_E2E_TRACE") == "1" else None     # diagnostic: per-step host enqueue / wait times + device step ends

        def e2e_step():
            t_a = time.perf_counter()
            a = accs[step_no["k"] % len(accs)]
            a.wait()
            a.zero_()
            out = run_views(e2e_camera, e2e_loss)
            reduce_step(a, False)                                      # same schedule as the resident-input loop
            k = step_no["k"]
            if args.level == "A":
                loss_hosts[k % 2].copy_(torch.stack(out).detach().reshape(-1), non_blocking=True)
            loss_ev[k % 2].record(torch.cuda.current_stream(dev))     # render_views has joined the view streams into this one
            step_no["k"] += 1
            t_b = time.perf_counter()
            if pending["k"] is not None:
                read_losses(pending["k"])                             # previous step's result, now that this one is enqueued
            pending["k"] = k
            if trace is not None:
                ev = torch.cuda.Event(enable_timing=True); ev.record(torch.cuda.current_stream(dev))
                trace.append((t_b - t_a, time.perf_counter() - t_b, ev))

        def e2e_drain():
            if pending["k"] is not None:
                read_losses(pending["k"])
                pending["k"] = None
        for _ in range(3):
            e2e_step()
        e2e_drain()
        barrier()
        # the end-to-end loop is host-sensitive (one stall of the launching thread is a visible fraction of a 20-step region):
        # the timed region of K steps is repeated five times and the MEDIAN is reported, all five are listed
        n_e2e = max(1, args.steps)
        reps = []
        for _rep in range(5):
            f0 = torch.cuda.Event(enable_timing=True); f1 = torch.cuda.Event(enable_timing=True)
            f0.record()
            for _ in range(n_e2e):
                e2e_step()
            e2e_drain()                    # the last step's losses are read inside the timed region too
            for a in accs:
                a.wait()                   # the last steps' all-reduces end inside the timed region
            f1.record()
            barrier()
            t2 = torch.tensor([f0.elapsed_time(f1)], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(t2, op=dist.ReduceOp.MAX)
            reps.append(vpr * world * n_e2e / (float(t2.item()) / 1000.0))
        if trace:
            torch.cuda.synchronize(dev)
            enq = sorted(((t[0] * 1e3, i) for i, t in enumerate(trace)), reverse=True)[:8]
            waits = sorted(((t[1] * 1e3, i) for i, t in enumerate(trace)), reverse=True)[:8]
            gaps = sorted(((trace[i][2].elapsed_time(trace[i + 1][2]), i + 1) for i in range(len(trace) - 1)), reverse=True)[:8]
            med = lambda xs: sorted(xs)[len(xs) // 2]
            print(f"[e2e trace rank {rank}] steps {len(trace)}  median enqueue {med([t[0] for t in trace]) * 1e3:.2f} ms  median wait "
                  f"{med([t[1] for t in trace]) * 1e3:.2f} ms\n  longest host enqueue (ms, step): {[(round(a_, 1), i) for a_, i in enq]}\n"
                  f"  longest host wait for step k-1 (ms, step): {[(round(a_, 1), i) for a_, i in waits]}\n"
                  f"  longest device step-to-step gaps (ms, step): {[(round(a_, 1), i) for a_, i in gaps]}", file=sys.stderr)
        e2e = {"value": sorted(reps)[2], "unit": UNIT,
               "h2d_bytes_per_step": int(h2d * vpr), "d2h_bytes_per_step": int(4 * vpr), "steps": n_e2e, "repetitions": reps,
               "note": "median of five timed regions of K steps; per view: pinned camera H2D on the view's stream, uint8 target H2D on a copy "
                       "stream started before the view's forward, loss + dL/dimg from the target (render_views' loss-and-gradient form), loss "
                       "D2H into pinned memory; the host reads each step's losses after enqueuing the next step (every step's result is "
                       "read inside the timed region)"}

    if rank != 0:
        return
    # ---- stage attribution + roofline -------------------------------------------------------------------
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak_gbs = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    summ = timer.summary()
    n_views_rank = vpr * args.steps
    bytes_per = stage_bytes(stats, S, K)
    stages = {}
    for name, (tot, n) in summ.items():
        stages[name] = {"ms_per_view": tot / n_views_rank, "launches_per_view": n / n_views_rank}
    for old, new in (("lgs_sort_pairs_u32_rebased", "lgs_sort_pairs_u32(depth)"), ("lgs_sort_pairs_u32", "lgs_sort_pairs_u32(tile)"),
                     ("lgs_sort_pairs_u16", "lgs_sort_pairs_u16(tile)"), ("lgs_sort_pairs_u32_dev", "lgs_sort_pairs_u32(depth)"),
                     ("lgs_sort_pairs_u16_dev", "lgs_sort_pairs_u16(tile)"), ("lgs_sort_pairs_u32k_dev", "lgs_sort_pairs_u32(tile)"),
                     ("lgs_scan_gathered_dev", "lgs_scan_gathered"), ("lgs_tile_range_u16_dev", "lgs_tile_range_u16"),
                     ("lgs_tile_range_dev", "lgs_tile_range")):
        if old in stages:                       # the GPU-driven (device-side count) entry points are the same kernels
            stages[new] = stages.pop(old)
    if "lgs_emit_pairs_dev" in stages:
        stages["lgs_emit_pairs_u16" if (stats["tiles"] + 1) < 65536 else "lgs_emit_pairs"] = stages.pop("lgs_emit_pairs_dev")
    for name, s_ in stages.items():
        b = bytes_per.get(name)
        if b is not None and s_["ms_per_view"] > 0:
            s_["alg_bytes"] = int(b)
            s_["gbs"] = b / (s_["ms_per_view"] / 1000.0) / 1e9
    dom = max(stages.items(), key=lambda kv: kv[1]["ms_per_view"])[0] if stages else None
    roofline, roofline_issue = None, None
    if dom is not None and "gbs" in stages[dom]:
        traffic, traffic_src = None, None
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json"))).get(dom)
            if tj and tj.get("tile") == args.tile and tj.get("config", "c2") == args.config:
                traffic, traffic_src = tj["bytes"], tj.get("source")
        except Exception:
            pass
        # the contract's roofline entry: algorithmic bytes of the dominant kernel over its measured duration against the HBM
        # peak.  For the raster kernels this fraction is small BY CONSTRUCTION (they are bound by instruction issue: DRAM
        # throughput 3 % of peak under ncu); `roofline_issue` below is the ceiling that actually bounds them.
        roofline = {"kernel": dom, "bound": "hbm", "achieved": stages[dom]["gbs"], "peak": peak_gbs, "unit": "GB/s",
                    "frac": stages[dom]["gbs"] / peak_gbs, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                    "alg_bytes_per_launch": stages[dom]["alg_bytes"], "ms_per_launch": stages[dom]["ms_per_view"],
                    "limiter": "instruction issue, not HBM: see roofline_issue" if dom in ISSUE_MODEL else None}
        im = ISSUE_MODEL.get(dom)
        if im is not None and args.tile in im and clocks and clocks.get("sm_mhz"):
            work = stats["backward_tile_splat_iterations"]
            inst = im[args.tile] * work
            sms = torch.cuda.get_device_properties(dev).multi_processor_count
            peak_ips = sms * 4 * clocks["sm_mhz"] * 1e6                 # one warp instruction per scheduler per cycle, 4 per SM
            ach = inst / (stages[dom]["ms_per_view"] / 1000.0)
            roofline_issue = {"kernel": dom, "bound": "sm_issue", "achieved": ach / 1e12, "peak": peak_ips / 1e12,
                              "unit": "T warp-inst/s", "frac": ach / peak_ips, "work_units_per_launch": work, "unit_of_work": im["unit"],
                              "warp_inst_per_unit": im[args.tile], "calibration": im["source"], "sm_count": sms,
                              "sm_mhz_in_run": clocks["sm_mhz"], "ms_per_launch": stages[dom]["ms_per_view"]}
    # whole path = the stages this run actually launched (bytes_per also lists the variants that were not: 32-bit tile keys,
    # the compacted-gradient scatter of level A)
    path_bytes = sum(s_["alg_bytes"] for s_ in stages.values() if "alg_bytes" in s_)
    survey_bytes = 748 * stats["Nv"] + 172 * stats["D"] + 48 * stats["P"]
    ms_view = ms / (vpr * args.steps)
    ms_view_serial = ms_serial / (vpr * args.steps)
    path = {"alg_bytes_per_view": int(path_bytes), "gbs": path_bytes / (ms_view / 1000.0) / 1e9,
            "frac": path_bytes / (ms_view / 1000.0) / 1e9 / peak_gbs,
            "survey_formula_bytes": int(survey_bytes), "survey_formula_frac": survey_bytes / (ms_view / 1000.0) / 1e9 / peak_gbs,
            "ms_per_view": ms_view, "ms_per_view_single_stream": ms_view_serial}
    hand_written = ("lgs_frustum_culling_aabb", "lgs_project_forward", "lgs_emit_pairs", "lgs_emit_pairs_u16", "lgs_tile_range",
                    "lgs_tile_range_u16", "lgs_rasterize_forward_packed", "lgs_rasterize_backward", "lgs_project_backward",
                    "lgs_sparse_chunk_op", "lgs_pack_params", "lgs_tile_order", "lgs_emit_pairs_dev", "lgs_tile_range_u16_dev",
                    "lgs_tile_range_dev", "lgs_view_params")
    gpu_launches = 0
    for name, (tot, n) in summ.items():
        if name in hand_written:
            gpu_launches += n
    gpu_launches += timer.sort_kernels
    comm = None
    if world > 1:
        pr = [[float(x) for x in gthr.tolist()] for gthr in gathered]
        comm = {"allreduce": args.allreduce if args.level == "B" else "sync", "bytes_per_step": int(accs[0].flat.numel() * 4),
                "allreduce_impl": ("own NVLS kernel over the buffer's NVSwitch multicast address (multimem.ld_reduce / multimem.st, csrc/nvls.cu)"
                                   if accs[0]._nvls is not None else "ncclAllReduce"),
                "allreduce_ms_per_step_rank0": comm_ms,
                "allreduce_ms_per_step_by_rank": [r_[1] / args.steps for r_ in pr],
                "step_ms_by_rank": [r_[0] / args.steps for r_ in pr],
                "note": "all-reduce time = CUDA events around the collective on the stream it is enqueued on (includes waiting for the "
                        "slowest rank to arrive, i.e. the render-time imbalance between ranks); step_ms_by_rank = each rank's own "
                        "timed region / steps",
                "other_schedule": other}
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": f"{args.config.upper()}: {args.gaussians} Gaussians (seed 0), {W}x{H}, sh_degree {args.sh_degree}, tile {args.tile}, "
                               f"{vpr} views/rank/step (render_views) + dense grad accumulate"
                               + ((" + NCCL all-reduce of the step's gradient buffer, " + ("completed before the next step starts" if not overlap else
                                   "overlapped with the next step (2 buffers, gradients one step late)")) if world > 1 else ""),
                   "parallelism": f"dp{world} (views sharded, parameters replicated)", "level": args.level,
                   "l2": "inputs exceed L2 (236 MB of parameters streamed per view); no explicit flush",
                   "staging": args.staging or os.environ.get("LGS_STAGING", "default"), "streams": n_streams,
                   "backward_kernel": os.environ.get("LGS_BWD", "v2"), "tile_order": os.environ.get("LGS_TILE_ORDER", "1") != "0",
                   "gpu_driven_sizing": bool(pipeline.SYNC_FREE and args.level == "B"), "cuda_graphs": bool(pipeline.GRAPHS_ENABLED and pipeline.SYNC_FREE and args.level == "B" and n_streams > 1),
                   "stage_timing": "serialized pass of the same steps on one stream (CUDA events around every C-ABI call)"},
        "clocks": clocks, "e2e": e2e, "gpu_launches": int(gpu_launches),
        "roofline": roofline, "roofline_issue": roofline_issue, "path_roofline": path, "workload_stats": stats, "stages": stages,
    }
    if comm is not None:
        line["comm"] = comm
    if world == 1 and not args.no_cpu_baseline:
        try:
            vps, dt, threads = cpu_views_per_s(args, scene_np, args.cpu_views)
            line["cpu_baseline"] = {"value": vps, "unit": UNIT, "cores": threads, "kind": "port",
                                    "sample": f"{args.cpu_views} full-size views of the same workload (oracle/, C + OpenMP), {dt:.1f} s"}
        except Exception as e:
            line["cpu_baseline"] = {"unavailable": str(e)[:200]}
    emit_line(line)


_REAL_STDOUT = None


def emit_line(obj):
    """The one JSON line of this run, on the real stdout."""
    data = (json.dumps(obj) + "\n").encode()
    if _REAL_STDOUT is not None:
        os.write(_REAL_STDOUT, data)
    else:
        sys.stdout.write(data.decode()); sys.stdout.flush()


def main():
    global _REAL_STDOUT
    args = parse()
    # stdout carries exactly one JSON line: everything else (NCCL's version banner, library chatter) goes to stderr
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if args.gpus > 1 and world == 1:
        sys.exit("bench.py --gpus N>1 must be launched with: python -m torch.distributed.run --nnodes=1 --nproc-per-node N "
                 "--master-addr 127.0.0.1 --master-port P bench.py --gpus N ...")
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench.py needs a CUDA device: litegs_b200 has no CPU path")
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local_rank}"))
    try:
        run_ours(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
