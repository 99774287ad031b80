#!/usr/bin/env python
"""bench.py -- projections/sec on the headline scene (100k Gaussians, 512x512 cone-beam, 50 views).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one forward X-ray projection of the synthetic scene (views cycle through the 50 angles).

ours arm
  value     projections/s with every input resident in HBM: K steps through the asynchronous C ABI
            (r2x_raster_forward_async, no host synchronisation), each step bracketed by its own pair of CUDA
            events with L2 flushed (256 MiB memset) between steps; value = K / sum(step durations); for N > 1
            the Gaussians are sharded across ranks and each step includes the exchange of the detector image
            (--reduce p2p: one kernel over NVLink peer memory, r2x_peer_allreduce_sum; --reduce nccl:
            dist.all_reduce); the per-rank sums are max-reduced over ranks.
  e2e       the same metric with HOST buffers through the public API (engine.HostProjector.project): every step
            copies the Gaussian parameters + view matrices host->device from pinned memory, runs the 4 kernels
            and reads the image back device->host, one request at a time; wall clock around the K steps.
            pipelined_value = the same requests through HostProjector.submit()/wait() (copies of neighbouring
            requests overlap the kernels); autograd_module_value = through GaussianRasterizer, the reference's
            Python surface (used for N > 1, where the per-rank images are summed on the device first).
  roofline  the dominant kernel (raster_render_kernel) re-run alone on the forward's state
            (r2x_raster_render_only), CUDA events, L2 flushed; achieved = (32 R + 4 N) bytes / duration
            against the measured HBM copy peak (MEASURED_PEAKS.json).  The kernel is FP32/MUFU-bound, not
            HBM-bound (DESIGN.md section 5), so the fraction is small by construction; the FP32-issue fraction is
            reported beside it.
  cpu_baseline  the CPU oracle port (oracle/r2_oracle.c, OpenMP) on the host cores, 2 projections of the
            same scene; cpu_baseline_torch = the pure-PyTorch CPU additive projector of SURVEY 8(d)
            (oracle/torch_projector.py), 3 projections.

reference arm (--impl reference)
  The reference has no CPU implementation of this path: its "own implementation" IS a CUDA rasterizer.  The
  arm therefore times the UNMODIFIED reference CUDA sources compiled for sm_100a into oracle/_ref/libr2ref.so
  (oracle/build_ref.sh) on the GPU with the identical per-step event / L2-flush protocol; if that library is
  absent it falls back to the CPU oracle port.  Rank 0 only.

--dump-outputs DIR
  After the timed steps, writes what the last timed step returned to its caller as DIR/image.npy (the [1,H,W]
  detector image) and, on one GPU, DIR/radii.npy (per-Gaussian screen radii), both float32.  Both GPU arms write the
  same names.  The scene and the views are seeded, so the same arguments give the same inputs in every run and two
  builds can be compared output for output.  An array over its share of 64 MiB is replaced by a fixed, seeded
  sample of its elements (the same positions in every run).
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "projections_per_sec"
UNIT = "projections/s"


_T0 = time.time()


def trace(msg: str) -> None:
    """Stage markers on stderr when R2X_BENCH_TRACE is set (stdout carries the one JSON line only)."""
    if os.environ.get("R2X_BENCH_TRACE"):
        print(f"[bench +{time.time() - _T0:7.1f}s] {msg}", file=sys.stderr, flush=True)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--gaussians", type=int, default=100_000)
    ap.add_argument("--detector", type=int, default=512)
    ap.add_argument("--views", type=int, default=50)
    ap.add_argument("--cloud", default="init", choices=["init", "trained"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the `secondary` block (other BASELINE configs)")
    ap.add_argument("--no-parity", action="store_true", help="skip the `parity` block (timed views vs the reference's kernels)")
    ap.add_argument("--cpu-baseline-child", default=None, choices=["port", "torch"], help=argparse.SUPPRESS)
    ap.add_argument("--reduce", default="p2p", choices=["p2p", "nccl"],
                    help="N > 1: how the per-rank partial images are summed (NVLink peer-memory kernel | NCCL)")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write the outputs of the last timed step as DIR/<name>.npy (float32)")
    return ap.parse_args()


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200", "-i", str(self.gpu)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def __exit__(self, *a):
        if self.proc is not None:
            time.sleep(0.25)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self) -> dict:
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}


def load_peaks() -> tuple[float, str]:
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def load_traffic() -> float | None:
    """dram bytes per launch of the render kernel from the committed ncu --set full capture."""
    p = os.path.join(ROOT, "profiles", "render_traffic.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["raster_render_kernel"]["dram_bytes_per_launch"])
        except Exception:
            return None
    return None


# ------------------------------------------------------------------------------------------------
def build_scene(args):
    from r2_gaussian_b200 import scene

    sc = scene.cone_beam_scanner(args.detector, 256)
    views = scene.make_views(sc, args.views)
    cloud = scene.make_cloud(args.gaussians, kind=args.cloud, seed=0)
    return sc, views, cloud


def device_views(views, dev):
    import torch

    return [dict(view=torch.tensor(v.viewmatrix, device=dev), proj=torch.tensor(v.projmatrix, device=dev),
                 campos=torch.tensor(v.campos, device=dev), tx=v.tanfovx, ty=v.tanfovy, mode=v.mode) for v in views]


def timed_steps(step_fn, steps, warmup, flush_buf, stream_sync):
    """Per-step CUDA-event timing with an L2 flush between steps.  Returns list of ms."""
    import torch

    for i in range(warmup):
        flush_buf.zero_()
        step_fn(i)
    stream_sync()
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    stops = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    for i in range(steps):
        flush_buf.zero_()
        starts[i].record()
        step_fn(warmup + i)
        stops[i].record()
    stream_sync()
    return [s.elapsed_time(e) for s, e in zip(starts, stops)]


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(path: str, arrays: dict) -> None:
    """arrays: name -> numpy array, written as float32 DIR/<name>.npy; an array over its share of DUMP_LIMIT_BYTES
    is replaced by a sample of its flattened elements at positions drawn from a fixed seed."""
    os.makedirs(path, exist_ok=True)
    share = DUMP_LIMIT_BYTES // len(arrays) - 4096           # room for the .npy header
    for name, a in arrays.items():
        a = np.ascontiguousarray(a, dtype=np.float32)
        if a.nbytes > share:
            idx = np.random.default_rng(0).choice(a.size, share // a.itemsize, replace=False)
            a = a.reshape(-1)[np.sort(idx)]
        np.save(os.path.join(path, name + ".npy"), a)


def usable_cores() -> int:
    """Host threads this process may really use: the affinity mask, capped by the cgroup CPU quota (a container limited
    to a few cores still reports every core of the box in os.cpu_count(); OpenMP / torch threads beyond the quota spin)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except (OSError, ValueError):
        pass
    return max(1, n)


def guarded_cpu_baseline(args, kind: str, limit_s: int = 150) -> dict:
    """cpu_baseline / cpu_baseline_torch in a child process with a time limit: a slow or oversubscribed host can cost
    the bench line its CPU baseline, never the line itself."""
    cmd = [sys.executable, os.path.abspath(__file__), "--cpu-baseline-child", kind, "--gaussians", str(args.gaussians),
           "--detector", str(args.detector), "--views", str(args.views), "--cloud", args.cloud]
    env = dict(os.environ, OMP_WAIT_POLICY="passive", CUDA_VISIBLE_DEVICES="")
    try:
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=limit_s, env=env, cwd=ROOT)
        for line in reversed(r.stdout.strip().splitlines()):
            if line.startswith("{"):
                return json.loads(line)
        return {"unavailable": f"child exited {r.returncode}: {r.stderr.strip()[-300:]}", "kind": kind}
    except subprocess.TimeoutExpired:
        return {"unavailable": f"timed out after {limit_s} s on this host ({usable_cores()} usable cores)", "kind": kind}


def cpu_baseline(cloud, views, n_proj=2):
    from oracle import r2_oracle as orc

    orc.lib()
    orc.set_num_threads(usable_cores())
    t0 = time.perf_counter()
    for i in range(n_proj):
        v = views[i % len(views)]
        orc.raster_forward(cloud.means, cloud.scales, cloud.rotations, cloud.density, v.viewmatrix, v.projmatrix,
                           v.image_width, v.image_height, v.tanfovx, v.tanfovy, v.mode)
    dt = time.perf_counter() - t0
    return {"value": n_proj / dt, "unit": UNIT, "cores": orc.num_threads(), "kind": "port",
            "sample": f"{n_proj} full projections of the same scene ({cloud.P} Gaussians, "
                      f"{views[0].image_width}x{views[0].image_height}), oracle/r2_oracle.c with OpenMP"}


def cpu_baseline_torch(cloud, views, n_proj=3):
    """SURVEY 8(d)'s CPU baseline: the pure-PyTorch additive projector (oracle/torch_projector.py) on all host cores."""
    import torch

    from oracle import torch_projector as tp
    cores = usable_cores()
    torch.set_num_threads(cores)
    v = views[0]
    tp.project(cloud.means, cloud.density, cloud.scales, cloud.rotations, v.viewmatrix, v.projmatrix, v.image_width,
               v.image_height, v.tanfovx, v.tanfovy, v.mode)            # warm-up (thread pool, allocator)
    t0 = time.perf_counter()
    for i in range(n_proj):
        v = views[(i + 1) % len(views)]
        tp.project(cloud.means, cloud.density, cloud.scales, cloud.rotations, v.viewmatrix, v.projmatrix,
                   v.image_width, v.image_height, v.tanfovx, v.tanfovy, v.mode)
    dt = time.perf_counter() - t0
    return {"value": n_proj / dt, "unit": UNIT, "cores": cores, "kind": "pure-PyTorch CPU additive projector",
            "sample": f"{n_proj} full projections of the same scene after one warm-up projection"}


def parity_vs_reference(render_view, cloud, views, dev, W, H, which=(0, 17, 34)):
    """The image (and radii, when `render_view` returns them for the whole cloud) of three of the timed views against
    the UNMODIFIED reference CUDA rasterizer (oracle/_ref/libr2ref.so) run on the same inputs on this GPU.
    render_view(i) -> (image [1,H,W] device tensor, radii int32[P] device tensor or None)."""
    import torch

    ref_path = os.path.join(ROOT, "oracle", "_ref", "libr2ref.so")
    if not os.path.exists(ref_path):
        return {"unavailable": "oracle/_ref/libr2ref.so not present"}
    lib = C.CDLL(ref_path)
    lib.ref_raster_forward.restype = C.c_int
    P = cloud.P
    means = torch.tensor(cloud.means, device=dev); scales = torch.tensor(cloud.scales, device=dev)
    rots = torch.tensor(cloud.rotations, device=dev); dens = torch.tensor(cloud.density, device=dev)
    dv = device_views(views, dev)
    vp = lambda t: C.c_void_p(t.data_ptr())
    f = C.c_float
    res = {"views": [], "max_abs": 0.0, "max_rel_to_max": 0.0, "radii_equal": True, "num_rendered_equal": None,
           "bar": "|ours - ref| <= 1e-5 * max|ref| + 1e-7; radii bit-exact",
           "reference": "oracle/_ref/libr2ref.so (the reference's RAS/*.cu, unmodified) on the same GPU"}
    rel_all = []
    for i in which:
        i = i % len(dv)
        v = dv[i]
        out = torch.zeros((1, H, W), device=dev); radii = torch.zeros(P, dtype=torch.int32, device=dev)
        torch.cuda.synchronize(dev)
        lib.ref_raster_forward(P, W, H, vp(means), vp(dens), vp(scales), f(1.0), vp(rots), None, vp(v["view"]),
                               vp(v["proj"]), vp(v["campos"]), f(v["tx"]), f(v["ty"]), int(v["mode"]), vp(out), vp(radii))
        torch.cuda.synchronize(dev)
        img, my_radii = render_view(i)
        torch.cuda.synchronize(dev)
        diff = (img.double() - out.double()).abs()
        scale = float(out.abs().max())
        res["views"].append(int(i))
        res["max_abs"] = max(res["max_abs"], float(diff.max()))
        res["max_rel_to_max"] = max(res["max_rel_to_max"], float(diff.max()) / max(scale, 1e-30))
        if my_radii is not None:
            res["radii_equal"] = bool(res["radii_equal"] and torch.equal(my_radii, radii))
        nz = out.abs() > 1e-3 * scale            # per-pixel relative error where the signal is not negligible
        rel_all.append((diff[nz] / out.double().abs()[nz]).flatten())
    rel = torch.cat(rel_all)
    if rel.numel():
        q = torch.quantile(rel[:: max(1, rel.numel() // 1_000_000)], torch.tensor([0.5, 0.99, 0.9999], dtype=rel.dtype, device=rel.device))
        res["per_pixel_rel_err"] = {"median": float(q[0]), "p99": float(q[1]), "p99.99": float(q[2]), "max": float(rel.max()),
                                    "over": "pixels with |ref| > 1e-3 max|ref|"}
    res["pass"] = bool(res["max_rel_to_max"] <= 1e-5 + 1e-7 / max(scale, 1e-30) and res["radii_equal"])
    return res


# ------------------------------------------------------------------------------------------------
def run_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist

    from r2_gaussian_b200 import scene
    from r2_gaussian_b200.engine import RasterEngine
    from r2_gaussian_b200.rasterization import GaussianRasterizationSettings, GaussianRasterizer
    from r2_gaussian_b200.sharded import shard_bounds

    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    sc, views, cloud = build_scene(args)
    W = H = args.detector
    lo, hi = shard_bounds(cloud.P, rank, world)
    shard = scene.Cloud(cloud.means[lo:hi], cloud.scales[lo:hi], cloud.rotations[lo:hi], cloud.density[lo:hi])
    P = shard.P
    means = torch.tensor(shard.means, device=dev); scales = torch.tensor(shard.scales, device=dev)
    rots = torch.tensor(shard.rotations, device=dev); dens = torch.tensor(shard.density, device=dev)
    dv = device_views(views, dev)
    eng = RasterEngine(P, W, H, dev)

    def fwd(i, out=None):
        v = dv[i % len(dv)]
        return eng.forward(means, dens, scales, rots, v["view"], v["proj"], v["campos"], v["tx"], v["ty"], v["mode"], out=out)

    # provision the instance capacity from the views themselves (one pass, synchronising), 25 % headroom
    Rs = []
    for i in range(len(dv)):
        while True:
            fwd(i)
            if eng.check():
                break
        Rs.append(eng.num_rendered())
    eng._reserve(int(max(Rs) * 1.25) + 4096)
    R_mean = float(np.mean(Rs))

    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def sync():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    # N > 1: the exchange step.  Default = one-shot sum over NVLink peer memory (r2x_peer_allreduce_sum: every
    # rank renders into an IPC-shared partial image, one kernel adds the partials in rank order); --reduce nccl
    # uses dist.all_reduce instead.
    reducer = None
    if world > 1 and args.reduce == "p2p":
        from r2_gaussian_b200.peer import PeerReducer
        try:
            reducer = PeerReducer(W * H, dev)
            ok = 1
        except Exception as e:  # e.g. no peer access between these GPUs: agree on NCCL, loudly
            print(f"[bench] rank {rank}: peer-memory exchange unavailable ({e}); using NCCL", file=sys.stderr, flush=True)
            ok = 0
        flag = torch.tensor([ok], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if int(flag.item()) == 0:
            reducer, args.reduce = None, "nccl"
    final = torch.empty((1, H, W), dtype=torch.float32, device=dev)
    last = {}

    def step(i):
        if reducer is not None:
            fwd(i, out=reducer.partial().view(1, H, W))
            last["image"] = reducer.reduce(final)
            return
        out = fwd(i)
        if world > 1:
            dist.all_reduce(out, op=dist.ReduceOp.SUM)
        last["image"] = out

    sampler = ClockSampler(local_rank)
    sync()
    with sampler:
        ms = timed_steps(step, args.steps, args.warmup, flush, sync)
    total_ms = float(sum(ms))
    if args.dump_outputs and rank == 0:     # before the buffers are reused below
        outputs = {"image": last["image"].cpu().numpy()}
        if world == 1:
            outputs["radii"] = eng.radii.cpu().numpy()
        dump_outputs(args.dump_outputs, outputs)
    # back-to-back (warm L2, launches pipelined) for information; with N > 1 the all-reduce of step i runs on a
    # side stream and overlaps the render of step i+1 (ring of output buffers)
    sync()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if world > 1 and reducer is not None:
        e0.record()
        for i in range(args.steps):
            step(i)
        e1.record()
    elif world > 1:
        ring = [torch.empty((1, H, W), dtype=torch.float32, device=dev) for _ in range(4)]
        comm = torch.cuda.Stream(device=dev)
        done = [None] * 4
        e0.record()
        for i in range(args.steps):
            k = i % 4
            if done[k] is not None:
                torch.cuda.current_stream(dev).wait_event(done[k])   # buffer k free again
            fwd(i, out=ring[k])
            ready = torch.cuda.Event(); ready.record()
            with torch.cuda.stream(comm):
                comm.wait_event(ready)
                dist.all_reduce(ring[k], op=dist.ReduceOp.SUM)
                done[k] = torch.cuda.Event(); done[k].record(comm)
        torch.cuda.current_stream(dev).wait_stream(comm)
        e1.record()
    else:
        e0.record()
        for i in range(args.steps):
            step(i)
        e1.record()
    sync()
    warm_ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([total_ms, warm_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms, warm_ms = float(t[0]), float(t[1])
    # overflow check for the timed region (status of the last forward; capacity is per scene)
    assert eng.check(), "instance capacity overflowed during the timed region"
    if reducer is not None:
        assert reducer.ok(), "a peer never arrived in r2x_peer_allreduce_sum"

    # ---- roofline of the dominant kernel (rank 0's shard) ----
    fwd(0)
    sync()
    R0 = eng.num_rendered()
    ms_r = timed_steps(lambda i: eng.render_only(), 50, 5, flush, lambda: torch.cuda.synchronize(dev))
    t_render = float(np.mean(ms_r)) * 1e-3
    N = W * H
    alg_bytes = 32.0 * R0 + 4.0 * N
    peak, peak_src = load_peaks()
    achieved = alg_bytes / t_render / 1e9
    pairs = 256.0 * R0
    roofline = {"bound": "hbm", "kernel": "raster_render_kernel", "achieved": achieved, "peak": peak,
                "unit": "GB/s", "frac": achieved / peak, "traffic": load_traffic(),
                "algorithmic_bytes_per_launch": alg_bytes, "kernel_ms": t_render * 1e3, "peak_source": peak_src,
                "pair_evals_per_launch": pairs, "pair_evals_per_s": pairs / t_render,
                "timed": "r2x_raster_render_only = two small memsets (queue head, arrival counters) + the render kernel, CUDA events, L2 flushed",
                "note": "kernel is FP32-issue-bound (multiplicative forward differences: ~5 issue slots and 0.5 "
                        "MUFU.EX2 per pixel-Gaussian pair), not HBM-bound; see DESIGN.md section 5"}
    try:   # the bounds that do apply (both measured on this part, scripts/micro/): MUFU.EX2 rate and the FP32 issue rate
        props = torch.cuda.get_device_properties(dev)
        mhz = float(sampler.summary().get("sm_mhz") or 0.0) or 1965.0
        sms = props.multi_processor_count
        ex2_peak = 15.85 * sms * mhz * 1e6
        roofline["mufu"] = {"achieved": 0.5 * pairs / t_render, "peak": ex2_peak, "unit": "ex2/s",
                            "frac": 0.5 * pairs / t_render / ex2_peak, "ex2_per_pair": 0.5,
                            "peak_source": f"15.85 ex2/clk/SM (measured, mufu_rate.cu) x {sms} SMs x {mhz:.0f} MHz"}
        loop_peak = 19.9 * sms * mhz * 1e6
        roofline["issue"] = {"achieved": pairs / t_render, "peak": loop_peak, "unit": "pairs/s", "frac": pairs / t_render / loop_peak,
                             "peak_source": f"19.9 pairs/clk/SM: the kernel's inner loop (f32x2 multiplicative differences) alone, "
                                            f"all operands in registers (measured, render_loop4.cu; profiles/r02_micro_render_loop4.txt) "
                                            f"x {sms} SMs x {mhz:.0f} MHz"}
    except Exception as e:   # informational only
        roofline["mufu"] = {"error": str(e)}

    # ---- parity of the timed path against the reference's own kernels (rank 0; N > 1: the summed image) ----
    parity = None
    if not args.no_parity:
        which = (0, 17, 34)
        if world == 1:
            parity = parity_vs_reference(lambda i: (fwd(i).clone(), eng.radii.clone()), cloud, views, dev, W, H, which)
        else:
            imgs = []
            for i in which:                 # every rank takes part in the exchange
                if reducer is not None:
                    step(i)
                    imgs.append(final.clone())
                else:
                    o = fwd(i)
                    dist.all_reduce(o, op=dist.ReduceOp.SUM)
                    imgs.append(o.clone())
            sync()
            if rank == 0:
                it = iter(imgs)
                parity = parity_vs_reference(lambda i: (next(it), None), cloud, views, dev, W, H, which)
            sync()

    result = {
        "metric": METRIC, "value": args.steps / (total_ms * 1e-3), "unit": UNIT, "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": total_ms / args.steps,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{args.gaussians} Gaussians ({args.cloud}-like, seed 0), {W}x{H} cone-beam "
                               f"(DSD 7, DSO 5), {args.views} views cycled; forward projection",
                   "gaussians": args.gaussians, "detector": [H, W], "views": args.views,
                   "parallelism": f"gaussian-shard x{world}" + ((" + one-shot NVLink peer-memory sum of the image (r2x_peer_allreduce_sum)"
                                                                   if args.reduce == "p2p" else " + NCCL all-reduce of the image") if world > 1 else ""),
                   "l2": "flushed between steps (256 MiB memset outside the timed events)",
                   "num_rendered_mean": R_mean * 1.0, "api": "r2x_raster_forward_async (C ABI, no host sync)"},
        "value_warm_l2_back_to_back": args.steps / (warm_ms * 1e-3),  # N > 1: all-reduce overlapped with the next render
        # preprocess(+tile histogram), direct_scan, direct_fill, render (+ the peer-memory sum when N > 1)
        "gpu_launches": args.steps * (5 if (world > 1 and args.reduce == "p2p") else 4),
        "roofline": roofline,
        "clocks": sampler.summary(),
    }
    if parity is not None:
        result["parity"] = parity

    # ---- e2e: host buffers in, host image out, through the public API ----
    if not args.no_e2e:
        from r2_gaussian_b200.engine import HostProjector
        pin = lambda a: torch.tensor(a).pin_memory()
        h_means, h_scales, h_rots, h_dens = pin(shard.means), pin(shard.scales), pin(shard.rotations), pin(shard.density)
        h_views = [(pin(v.viewmatrix), pin(v.projmatrix), pin(v.campos), v) for v in views]
        h_outs = [torch.empty((1, H, W), dtype=torch.float32).pin_memory() for _ in range(4)]
        h2d = sum(t.numel() * 4 for t in (h_means, h_scales, h_rots, h_dens)) + (16 + 16 + 3) * 4
        d2h = H * W * 4
        hp = HostProjector(P, W, H, dev, depth=3, capacity=eng.capacity)

        def request(i):
            hv, hpj, hc, v = h_views[i % len(h_views)]
            return (h_means, h_dens, h_scales, h_rots, hv, hpj, hc, v.tanfovx, v.tanfovy, v.mode, h_outs[i % 4])

        def e2e_serial(i):      # strict: upload -> kernels -> download -> wait, one request at a time
            hp.project(*request(i))

        def e2e_autograd(i):    # the reference-facing module (allocates its state per call, one host sync inside)
            hv, hpj, hc, v = h_views[i % len(h_views)]
            m = h_means.to(dev, non_blocking=True); s_ = h_scales.to(dev, non_blocking=True)
            r = h_rots.to(dev, non_blocking=True); d = h_dens.to(dev, non_blocking=True)
            settings = GaussianRasterizationSettings(
                image_height=H, image_width=W, tanfovx=v.tanfovx, tanfovy=v.tanfovy, scale_modifier=1.0,
                viewmatrix=hv.to(dev, non_blocking=True), projmatrix=hpj.to(dev, non_blocking=True),
                campos=hc.to(dev, non_blocking=True), prefiltered=False, mode=v.mode, debug=False)
            with torch.no_grad():
                img, _radii = GaussianRasterizer(settings)(means3D=m, means2D=None, opacities=d, scales=s_, rotations=r)
            if reducer is not None:
                reducer.partial().view_as(img).copy_(img)
                img = reducer.reduce(final)
            elif world > 1:
                dist.all_reduce(img, op=dist.ReduceOp.SUM)
            h_outs[0].copy_(img, non_blocking=True)
            torch.cuda.current_stream(dev).synchronize()

        def wall(fn, finish=None):
            for i in range(min(args.warmup, 10)):
                fn(i)
            if finish:
                finish()
            sync()
            t0 = time.perf_counter()
            for i in range(args.steps):
                fn(i)
            if finish:
                finish()
            sync()
            dt = time.perf_counter() - t0
            if world > 1:
                t = torch.tensor([dt], device=dev, dtype=torch.float64)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                dt = float(t[0])
            return args.steps / dt

        e2e = {"unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h)}
        e2e["autograd_module_value"] = wall(e2e_autograd)
        if world == 1:
            e2e["value"] = wall(e2e_serial)
            e2e["pipelined_value"] = wall(lambda i: hp.submit(*request(i)), hp.drain)
            e2e["api"] = ("engine.HostProjector.project(pinned host parameters, pinned host image): upload, 4 kernels, "
                          "download, wait -- one request at a time; pipelined_value = HostProjector.submit()/wait(), "
                          "uploads / kernels / downloads of consecutive requests overlapped on three streams; "
                          "autograd_module_value = GaussianRasterizer(settings)(...) with the same copies")
        else:
            e2e["value"] = e2e["autograd_module_value"]
            e2e["api"] = ("GaussianRasterizer(settings)(means3D, means2D, opacities, scales, rotations) per rank, image "
                          "summed over ranks on the device, pinned host inputs, image read back each step")
        result["e2e"] = e2e

    trace("headline measured")
    if rank == 0 and world == 1 and not args.no_secondary:
        sys.path.insert(0, os.path.join(ROOT, "scripts"))
        import secondary
        del eng
        torch.cuda.empty_cache()
        result["secondary"] = secondary.measure(dev, peak, trace=trace)
        trace("secondary done")
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        result["cpu_baseline"] = guarded_cpu_baseline(args, "port")
        trace("cpu baseline (oracle port)")
        result["cpu_baseline_torch"] = guarded_cpu_baseline(args, "torch")
        trace("cpu baseline (torch projector)")
    return result


# ------------------------------------------------------------------------------------------------
def run_reference(args):
    """The reference's own CUDA rasterizer (oracle/_ref) on cuda:0, same protocol; else the CPU oracle."""
    sc, views, cloud = build_scene(args)
    W = H = args.detector
    ref_path = os.path.join(ROOT, "oracle", "_ref", "libr2ref.so")
    base = {
        "impl": "reference", "metric": METRIC, "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{args.gaussians} Gaussians ({args.cloud}-like, seed 0), {W}x{H} cone-beam "
                               f"(DSD 7, DSO 5), {args.views} views cycled; forward projection",
                   "gaussians": args.gaussians, "detector": [H, W], "views": args.views,
                   "parallelism": "single GPU (the reference has no multi-GPU path)",
                   "l2": "flushed between steps (256 MiB memset outside the timed events)"},
    }
    have_gpu = False
    try:
        import torch
        have_gpu = torch.cuda.is_available() and os.path.exists(ref_path)
    except Exception:
        have_gpu = False
    if not have_gpu:
        cb = cpu_baseline(cloud, views, 2)
        base.update(value=cb["value"], ms_per_step=1e3 / cb["value"], cpu_baseline=cb,
                    e2e={"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                    reference_kind="CPU oracle port (oracle/_ref/libr2ref.so not available)")
        return base

    import torch

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    lib = C.CDLL(ref_path)
    lib.ref_raster_forward.restype = C.c_int
    P = cloud.P
    means = torch.tensor(cloud.means, device=dev); scales = torch.tensor(cloud.scales, device=dev)
    rots = torch.tensor(cloud.rotations, device=dev); dens = torch.tensor(cloud.density, device=dev)
    dv = device_views(views, dev)
    out = torch.zeros((1, H, W), device=dev); radii = torch.zeros(P, dtype=torch.int32, device=dev)
    vp = lambda t: C.c_void_p(t.data_ptr())
    f = C.c_float
    Rs = []

    def step(i):
        v = dv[i % len(dv)]
        # the binding zero-fills the image and radii every call (SUB/rasterize_points.cu:55-56)
        out.zero_(); radii.zero_()
        R = lib.ref_raster_forward(P, W, H, vp(means), vp(dens), vp(scales), f(1.0), vp(rots), None, vp(v["view"]),
                                   vp(v["proj"]), vp(v["campos"]), f(v["tx"]), f(v["ty"]), int(v["mode"]), vp(out),
                                   vp(radii))
        Rs.append(R)

    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    sampler = ClockSampler(0)
    sync = lambda: torch.cuda.synchronize(dev)
    with sampler:
        ms = timed_steps(step, args.steps, args.warmup, flush, sync)
    total_ms = float(sum(ms))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"image": out.cpu().numpy(), "radii": radii.cpu().numpy()})
    value = args.steps / (total_ms * 1e-3)
    # back-to-back, warm L2
    sync()
    t0 = time.perf_counter()
    for i in range(args.steps):
        step(i)
    sync()
    warm = args.steps / (time.perf_counter() - t0)
    # end-to-end for the reference arm, same protocol as ours: pinned host parameters and matrices copied to the
    # device every step, image read back every step, wall clock.  (The generic contract puts 0 bytes here
    # because it assumes a CPU reference; this reference runs on the GPU, so it gets the same copies we pay.)
    pin = lambda a: torch.tensor(a).pin_memory()
    h = [pin(cloud.means), pin(cloud.scales), pin(cloud.rotations), pin(cloud.density)]
    hv = [(pin(v.viewmatrix), pin(v.projmatrix), pin(v.campos), v) for v in views]
    h_out = torch.empty((1, H, W), dtype=torch.float32).pin_memory()
    h2d = sum(t.numel() * 4 for t in h) + (16 + 16 + 3) * 4
    d2h = H * W * 4

    def e2e_step(i):
        a, b, c, v = hv[i % len(hv)]
        dm, ds, dr, dd = (t.to(dev, non_blocking=True) for t in h)
        va, vb, vc = a.to(dev, non_blocking=True), b.to(dev, non_blocking=True), c.to(dev, non_blocking=True)
        o = torch.zeros((1, H, W), device=dev); rr = torch.zeros(P, dtype=torch.int32, device=dev)
        lib.ref_raster_forward(P, W, H, vp(dm), vp(dd), vp(ds), f(1.0), vp(dr), None, vp(va), vp(vb), vp(vc),
                               f(v.tanfovx), f(v.tanfovy), int(v.mode), vp(o), vp(rr))
        h_out.copy_(o, non_blocking=True)
        torch.cuda.current_stream(dev).synchronize()

    for i in range(min(args.warmup, 10)):
        e2e_step(i)
    sync()
    t0 = time.perf_counter()
    for i in range(args.steps):
        e2e_step(i)
    sync()
    e2e_value = args.steps / (time.perf_counter() - t0)
    base.update(value=value, ms_per_step=total_ms / args.steps, value_warm_l2_back_to_back=warm,
                clocks=sampler.summary(), gpu_launches=0,
                reference_kind="the reference's own CUDA rasterizer (RAS/*.cu, unmodified) compiled for sm_100a into "
                               "oracle/_ref/libr2ref.so with a GLM stand-in; called through its C++ API "
                               "CudaRasterizer::Rasterizer::forward with persistent scratch buffers (cheaper than its "
                               "torch binding, which re-allocates them every call)",
                e2e={"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                     "note": "GPU reference: same pinned-host -> device copies and image read-back per step as the "
                             "'ours' arm (the generic contract's 0 bytes assumes a CPU reference)"})
    base["config"]["num_rendered_mean"] = float(np.mean(Rs[-args.steps:]))
    if not args.no_cpu_baseline:
        base["cpu_baseline"] = guarded_cpu_baseline(args, "port")
    return base


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.cpu_baseline_child:
        _sc, views, cloud = build_scene(args)
        fn = cpu_baseline if args.cpu_baseline_child == "port" else cpu_baseline_torch
        print(json.dumps(fn(cloud, views)), flush=True)
        return 0
    if args.impl == "reference":
        if rank != 0:
            return 0
        print(json.dumps(run_reference(args)), flush=True)
        return 0

    import torch

    if not torch.cuda.is_available():
        print(json.dumps({"metric": METRIC, "error": "no CUDA device: the B200 path has no CPU fallback"}), flush=True)
        return 1
    if world > 1:
        import torch.distributed as dist

        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        res = run_ours(args, rank, world, local_rank)
        if rank == 0:
            print(json.dumps(res), flush=True)
    finally:
        if world > 1:
            import torch.distributed as dist

            dist.barrier()
            dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
