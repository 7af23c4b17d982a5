#!/usr/bin/env python
"""bench.py -- BASELINE.json metric on B200: tile-pairs/sec of FFT phase correlation on
512^3 uint16 overlap crops (configs[1]: 112 pairs, 1 B200), plus the fused Mvoxels/sec of
SparkAffineFusion's config (64 tiles -> 2048^3 float32) as the `fusion` sub-object.

    python bench.py --gpus N --steps K --warmup W          (N>1: launched under torchrun)
    python bench.py --impl reference ...                    (CPU arm: the oracle port on host cores)
    python bench.py ... --dump-outputs DIR                  (also write rank 0's outputs as DIR/<name>.npy)

A "step" is one pass of the hot path over the whole batch (112 pairs).  `value` is measured
with the crops resident in HBM; `e2e` goes through the same C-ABI call with pinned HOST
buffers (H2D inside the timed region).  Every timed section runs K steps.  One JSON line is
printed by rank 0.

--dump-outputs writes what the last timed step of each GPU section returned: the phase-correlation
results (pcm_*, pcm_e2e_*), a fixed seeded sample of the fused volume (fusion_sample*) and the DoG
detections (dog_*).  All inputs are seeded, so two builds can be compared output for output.
"""
from __future__ import annotations

import argparse
import dataclasses
import json
import multiprocessing as mp
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "tile-pairs/sec (phase-corr, 512^3 uint16 overlaps)"
UNIT = "pairs/s"
DUMP_SAMPLE = 1 << 21      # voxels of the fused volume that --dump-outputs keeps (24 MB with their indices)


# ------------------------------------------------------------------------------------------ utils
def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200", "-i", str(self.index)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def ncu_traffic(tag):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full`
    capture (profiles/ncu_traffic_r1.json; bench.py cannot run ncu itself), or None."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic_r1.json")
    try:
        return int(json.load(open(p))["bytes_per_launch"][tag])
    except Exception:
        return None


def dump(dirname, name, values):
    """--dump-outputs: one output array as ``dirname/name.npy``; float32 stays float32, everything else becomes float64."""
    if dirname is None:
        return
    os.makedirs(dirname, exist_ok=True)
    a = np.asarray(values)
    np.save(os.path.join(dirname, name + ".npy"), a if a.dtype == np.float32 else a.astype(np.float64))


def dump_pcm(dirname, prefix, results):
    """one array per PcmResult field, one row per pair"""
    for f in dataclasses.fields(results[0]):
        dump(dirname, f"{prefix}_{f.name}", [getattr(r, f.name) for r in results])


def pcm_bytes_per_pair(n, P, K_px):
    """SURVEY.md 8(d): B_pair = 4n + 12 S + 2 R + 4 * (Pearson voxels)."""
    S = P[2] * P[1] * (P[0] // 2 + 1) * 8
    R = P[0] * P[1] * P[2] * 4
    return 4 * n + 12 * S + 2 * R + 4 * K_px


def pcm_kernel_bytes(n, P, pearson_px):
    S = P[2] * P[1] * (P[0] // 2 + 1) * 8
    R = P[0] * P[1] * P[2] * 4
    return {"fft_x_r2c": 4 * n + 2 * S, "fft_y": 4 * S, "fft_z_xpower": 3 * S, "fft_y_inv": 2 * S,
            "fft_x_c2r": S + R, "peaks": R, "pearson": 4 * pearson_px}


# ------------------------------------------------------------------------------------------ CPU arm
_CPU = {}


def _cpu_pcm_worker(threads):
    from oracle import pcm_oracle as po
    r = po.pcm_shift(_CPU["a"], _CPU["b"], workers=threads)
    return r.shift_int


def _cpu_fuse_worker(job):
    from oracle import fusion_oracle as fo
    views, bmin, bsz = _CPU["views"], job[0], job[1]
    out = fo.fuse_block(views, bmin, bsz, fo.AVG_BLEND)
    return float(out.sum())


def cpu_pcm_sample(n, procs, threads, repeats=1, pairs=None):
    """CPU arm of the phase-correlation metric.  Preferred: the C / OpenMP restatement of the oracle
    (oracle/c/pcm_oracle.c: own batched FFT, all host threads on one pair at a time -- ~10x the numpy oracle), on
    ``pairs`` distinct seeded pairs; fallback: the numpy/scipy oracle as `procs` concurrent single-pair workers (the
    shape of the reference's Spark local[N], J/SparkPairwiseStitching.java:210).  Returns (pairs/s, [seconds per step])."""
    from tests import synth
    try:
        from oracle import c_pcm
        c_pcm.load()
        pairs = pairs or 2
        key = ("c", n, pairs)
        if _CPU.get("key") != key:
            _CPU["pairs"] = [synth.shifted_pair((n, n, n), (7 - i, -5 + i, 3), seed=99 + i, margin=12, sigma=2.0) for i in range(pairs)]
            _CPU["key"] = key
            # thread count: every logical CPU or one per physical core, whichever runs a pair faster on this box (the
            # FFT passes are memory-bound, so SMT siblings usually lose) -- calibrated once on the first pair
            logical = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
            best = None
            for nt in sorted({logical, c_pcm.physical_cores()}, reverse=True):
                c_pcm.set_num_threads(nt)
                t0 = time.perf_counter()
                c_pcm.pcm_shift(*_CPU["pairs"][0])
                dt = time.perf_counter() - t0
                if best is None or dt < best[0]:
                    best = (dt, nt)
            c_pcm.set_num_threads(best[1])
            _CPU["threads"] = best[1]
        times = []
        for _ in range(repeats):
            t0 = time.perf_counter()
            for a, b in _CPU["pairs"]:
                r = c_pcm.pcm_shift(a, b)
                assert r.found
            times.append(time.perf_counter() - t0)
        _CPU["impl"] = f"oracle/c/pcm_oracle.c, {c_pcm.num_threads()} OpenMP threads, {pairs} pairs per step one after the other"
        _CPU["cores"] = c_pcm.num_threads()
        _CPU["pairs_per_step"] = pairs
        return pairs / min(times), times
    except Exception:
        pass
    if _CPU.get("n") != n:   # generate the sample pair once per process
        _CPU["a"], _CPU["b"] = synth.shifted_pair((n, n, n), (7, -5, 3), seed=99, margin=12, sigma=2.0)
        _CPU["n"] = n
    ctxm = mp.get_context("fork")
    times = []
    with ctxm.Pool(procs) as pool:
        for _ in range(repeats):
            t0 = time.perf_counter()
            pool.map(_cpu_pcm_worker, [threads] * procs)
            times.append(time.perf_counter() - t0)
    _CPU["impl"] = f"oracle/pcm_oracle.py (numpy + scipy pocketfft), {procs} concurrent pairs x {threads} FFT threads"
    _CPU["cores"] = procs * threads
    _CPU["pairs_per_step"] = procs
    return procs / min(times), times


def cpu_fusion_sample(procs, blocks_per_proc=2, tile=160, bs=96):
    """CPU arm of the fusion metric.  Preferred: the C / OpenMP restatement of the oracle
    (oracle/c/fusion_oracle.c, all host threads) on a 2x2x2 grid of 320^3 tiles, fusing one
    512x512x128 region; fallback: the numpy oracle over a process pool.  Returns
    (Mvoxels/s, seconds, cores, sample description)."""
    from oracle import fusion_oracle as fo
    from tests import synth
    rng = np.random.default_rng(7)
    try:
        from oracle import c_fusion
        c_fusion.set_num_threads(_CPU.get("threads") or c_fusion.physical_cores())   # the count the PCM arm calibrated
        nthreads = c_fusion.num_threads()
        t = 320
        stride = int(t * 491 / 576)
        vol = synth.tile_from(synth.field((t,) * 3, seed=5, sigma=2.0), (0, 0, 0), (t,) * 3, 5)
        views = []
        for k in range(2):
            for j in range(2):
                for i in range(2):
                    M = synth.translation(stride * np.array([i, j, k]) + rng.uniform(-2, 2, 3))
                    border, rngb = fo.adjust_blending(M)
                    views.append(fo.View(vol, M, border, rngb))
        size = (512, 512, 128)
        bmin = (20, 20, stride - 64)
        c_fusion.fuse_block(views, bmin, (64, 64, 16), fo.AVG_BLEND)   # warm-up (thread pool, page faults)
        reps, t0 = 0, time.perf_counter()
        while reps < 1 or (time.perf_counter() - t0 < 8.0 and reps < 64):   # bounded sample: ~8 s of CPU work
            c_fusion.fuse_block(views, bmin, size, fo.AVG_BLEND)
            reps += 1
        dt = time.perf_counter() - t0
        return (reps * size[0] * size[1] * size[2] / dt / 1e6, dt, nthreads,
                f"{reps} x one 512x512x128 block over a 2x2x2 grid of 320^3 uint16 tiles, AVG_BLEND, {dt:.1f} s, "
                f"C/OpenMP restatement of the oracle (oracle/c/fusion_oracle.c)")
    except Exception:
        pass
    stride = int(tile * 491 / 576)
    views = []
    vol = synth.tile_from(synth.field((tile,) * 3, seed=5, sigma=2.0), (0, 0, 0), (tile,) * 3, 5)
    for k in range(2):
        for j in range(2):
            for i in range(2):
                M = synth.translation(stride * np.array([i, j, k]) + rng.uniform(-2, 2, 3))
                border, rngb = fo.adjust_blending(M)
                views.append(fo.View(vol, M, border, rngb))
    _CPU["views"] = views
    jobs = []
    for q in range(procs * blocks_per_proc):
        o = (stride - bs // 2 + (q % 3) * 7, stride - bs // 2 + (q % 5) * 3, stride - bs // 2)
        jobs.append((o, (bs, bs, bs)))
    ctxm = mp.get_context("fork")
    with ctxm.Pool(procs) as pool:
        t0 = time.perf_counter()
        pool.map(_cpu_fuse_worker, jobs)
        dt = time.perf_counter() - t0
    return (len(jobs) * bs ** 3 / dt / 1e6, dt, procs,
            f"{len(jobs)} blocks of {bs}^3, 8 views, AVG_BLEND, {dt:.1f} s (oracle/fusion_oracle.py, numpy)")


def cpu_dog_sample():
    """CPU arm of the DoG row: the numpy / scipy oracle (oracle/dog_oracle.py: scipy's multi-pass separable correlation,
    one thread) on one 256x256x64 bead block.  Returns (Mvoxels/s, seconds, description) or None."""
    try:
        from oracle import dog_oracle as do
        rng = np.random.default_rng(5)
        shape = (64, 256, 256)
        img = rng.normal(200.0, 8.0, shape)
        zz, yy, xx = np.mgrid[0:9, 0:9, 0:9] - 4
        bead = 3000.0 * np.exp(-(zz ** 2 + yy ** 2 + xx ** 2) / (2 * 1.8 ** 2))
        for _ in range(40):
            z, y, x = (int(rng.integers(4, s - 5)) for s in shape)
            img[z - 4:z + 5, y - 4:y + 5, x - 4:x + 5] += bead
        img = np.clip(np.rint(img), 0, 65535).astype(np.uint16)
        t0 = time.perf_counter()
        pts = do.detect(img, (0, 0, 0), shape[::-1], sigma=1.8, threshold=0.008, min_intensity=0.0, max_intensity=4000.0)
        dt = time.perf_counter() - t0
        return img.size / dt / 1e6, dt, f"oracle/dog_oracle.py (numpy + scipy, 1 thread) on one 256x256x64 bead block, {len(pts)} detections, {dt:.1f} s"
    except Exception:
        return None


def cpu_layout():
    """All host threads: ncores/4 concurrent single-pair workers (capped at 32: ~6 GB each) x 4 FFT
    threads -- the shape of the reference's Spark local[N] (one task per slot)."""
    ncores = os.cpu_count() or 1
    procs = max(1, min(32, ncores // 4))
    threads = max(1, min(4, ncores // procs))
    return ncores, procs, threads


def run_reference(args, rank):
    """--impl reference: the reference's CPU implementation of the path is not runnable here
    (no JVM, arithmetic in un-vendored Maven artefacts -- SURVEY.md 8c), so this arm times the
    oracle port (oracle/c/pcm_oracle.c, C / OpenMP, thread count calibrated per box) on the box's host cores.  Rank 0 only."""
    if rank != 0:
        return
    ncores, procs, threads = cpu_layout()
    n = args.size
    t_all = time.perf_counter()
    v0, t0 = cpu_pcm_sample(n, procs, threads)          # warm-up step (also sizes the time box)
    # every step is a bounded sample (`procs` pairs); the whole run is time-boxed to a few minutes
    budget_s = 170.0
    nsteps = args.steps if args.ref_full else max(1, min(args.steps, int(budget_s / max(t0[0], 1e-3))))
    vals, step_times = [], []
    for _ in range(nsteps):
        v, tt = cpu_pcm_sample(n, procs, threads)
        vals.append(v)
        step_times.append(tt)
    value = float(np.median(vals))     # host boxes differ a lot between leases: the median of the steps, all listed below
    sample = f"{n}^3 uint16 pairs, {_CPU.get('impl', '?')}"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": nsteps, "steps_requested": args.steps, "warmup": 1, "ms_per_step": 1000.0 * _CPU.get("pairs_per_step", procs) / value,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD_PCM if n == 512 else f"phase-correlation: {n}^3 uint16 overlap crops",
                   "sampling": f"every step is a bounded sample of that workload ({_CPU.get('impl', '?')})",
                   "note": "Java reference not runnable in this image (no JVM; arithmetic in un-vendored Maven "
                           "artefacts); CPU arm = the oracle port on all host cores"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": _CPU.get("cores", procs * threads), "host_cores": ncores,
                         "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "step_values": [round(v, 4) for v in vals],
        "wall_s": time.perf_counter() - t_all,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------ GPU arm
WORKLOAD_PCM = ("phase-correlation: 112 overlapping pairs of 512^3 uint16 overlap crops (BASELINE configs[1], 4x4x2 tile "
                "grid), 5-smooth pad 540^3, peaks=5, subpixel, minOverlap 0.25")


def ncu_traffic_r2(tag):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the committed `ncu --set full` capture of the
    CURRENT kernels (profiles/ncu_traffic_r2.json; bench.py cannot run ncu itself), or None."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic_r2.json")
    try:
        return json.load(open(p))[tag]
    except Exception:
        return None


def run_gpu(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    import bsgpu
    from bsgpu import synthetic

    # ---- CPU baseline first (rank 0, N=1): forks worker processes, so it runs before CUDA is touched
    cpu = cpu_fusion = cpu_dog = None
    if rank == 0 and world == 1 and not args.skip_cpu:
        ncores, procs, threads = cpu_layout()
        v, times = cpu_pcm_sample(args.size, procs, threads)
        cpu = {"value": v, "unit": UNIT, "cores": _CPU.get("cores", procs * threads), "host_cores": ncores, "kind": "port",
               "sample": f"{args.size}^3 uint16 pairs, {_CPU.get('impl', '?')}, {times[0]:.1f} s "
                         f"(Java reference not runnable here)"}
        if not args.skip_fusion:
            fv, fdt, fcores, fsample = cpu_fusion_sample(procs)
            cpu_fusion = {"value": fv, "unit": "Mvoxels/s", "cores": fcores, "kind": "port", "sample": fsample}
        if not args.skip_dog:
            cd = cpu_dog_sample()
            if cd is not None:
                cpu_dog = {"value": cd[0], "unit": "Mvoxels/s", "cores": 1, "kind": "port", "sample": cd[2]}

    torch.cuda.set_device(local_rank)
    from bsgpu import parallel as bpar
    numa_node = bpar.bind_to_gpu_numa_node(local_rank)     # before any pinned buffer exists (first touch)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    stream = torch.cuda.Stream(device=dev)
    ctx = bsgpu.Context(local_rank, stream=stream.cuda_stream)
    peak_gbs, peak_src = measured_peaks()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    timed_calls = [0]

    def timed(fn, steps):
        """K steps between barrier + synchronize on both sides, device time by CUDA events on the launching stream, max
        over ranks; ``timed.last`` is what the last step returned.  A step that raises still completes this call's
        collectives (then re-raises), so the other ranks are never left alone inside a barrier."""
        timed_calls[0] += 1
        barrier()
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        w0 = time.perf_counter()
        e0.record(stream)
        err = None
        try:
            for _ in range(steps):
                timed.last = fn()
        except Exception as exc:
            err = exc
        e1.record(stream)
        e1.synchronize()
        barrier()
        wall = (time.perf_counter() - w0) * 1000.0
        ms = max_over_ranks(e0.elapsed_time(e1))
        if err is not None:
            raise err
        return ms, wall

    def optional(fn, n_timed):
        """Run an optional section that makes ``n_timed`` timed() calls.  If it fails on this rank, the remaining timed()
        calls are made with an empty step so that every rank goes through the same sequence of collectives."""
        start = timed_calls[0]
        try:
            return fn(), None
        except Exception as exc:
            if world > 1:
                while timed_calls[0] - start < n_timed:
                    try:
                        timed(lambda: None, 1)
                    except Exception:
                        break
            return None, exc
    timed.optional = optional

    # ---------------------------------------------------------------- phase correlation
    n = args.size
    npairs = args.pairs
    imgs1, imgs2, shifts = synthetic.make_pcm_workload(npairs, n=n, device=dev, seed=42 + rank, n_fields=args.fields)
    torch.cuda.synchronize()
    params = ctx.pcm_params(peaks_to_check=5, do_subpixel=True, min_overlap_frac=0.25, extension=(10, 10, 10))
    dims = [(n, n, n)] * npairs

    def step_resident():
        return ctx.pcm_batch(imgs1, imgs2, params, dims, bsgpu.native.DTYPE_U16)

    res = None
    for _ in range(max(args.warmup, 3)):
        res = step_resident()
    # planted real-valued shifts (half of the pairs carry a Fourier-domain sub-pixel part)
    recovered = sum(1 for r, s in zip(res, shifts) if r.found and max(abs(a - b) for a, b in zip(r.shift_sub, s)) < 0.5)
    sub_err = [max(abs(a - b) for a, b in zip(r.shift_sub, s)) for r, s in zip(res, shifts) if r.found]
    P = res[0].pad
    pearson_px_mean = float(np.mean([r.pearson_px for r in res]))
    ncand_mean = float(np.mean([r.n_candidates for r in res]))

    # ---- parity spot check against the oracle, outside the timed region (rank 0, N = 1): one integer-shift pair
    # and one sub-pixel pair of the benchmarked workload
    oracle_check = None
    if rank == 0 and world == 1 and not args.skip_oracle:
        from oracle import pcm_oracle as po
        ok = []
        for i in (0, 1)[:min(2, npairs)]:
            a = imgs1[i].cpu().numpy().view(np.uint16)
            b = imgs2[i].cpu().numpy().view(np.uint16)
            o = po.pcm_shift(a, b, workers=-1)
            g = res[i]
            ok.append(bool(g.found == o.found and g.shift_int == o.shift_int and g.peak_index == o.peak_index and
                           abs(g.r - o.r) < 1e-9 and max(abs(x - y) for x, y in zip(g.shift_sub, o.shift_sub)) < 1e-3))
        oracle_check = f"{sum(ok)}/{len(ok)} pairs identical to oracle/pcm_oracle.py (index, shift, r 1e-9, sub-pixel 1e-3)"

    sampler = ClockSampler(local_rank)
    sampler.start()
    l0 = ctx.launch_count()
    ms, wall_ms = timed(step_resident, args.steps)
    launches = ctx.launch_count() - l0
    clocks = sampler.stop()
    dump_pcm(args.dump_outputs, "pcm", timed.last)
    ms_per_step = ms / args.steps
    value = world * npairs / (ms_per_step / 1000.0)

    # ---- per-kernel device timing (CUDA events on the launching stream, separate pass)
    kern = {}
    if rank == 0:
        ctx.profile_reset()
        ctx.profile_enable(True)
        nprof = min(16, npairs)
        rp = ctx.pcm_batch(imgs1[:nprof], imgs2[:nprof], params, dims[:nprof], bsgpu.native.DTYPE_U16)
        ctx.profile_enable(False)
        ppx = float(np.mean([r.pearson_px for r in rp]))
        kb = pcm_kernel_bytes(n ** 3, P, ppx)
        for tag, b in kb.items():
            tms, cnt = ctx.profile_get(tag)
            if cnt:
                avg = tms / cnt
                kern[tag] = {"ms": round(avg, 4), "alg_bytes": int(b), "gbs": round(b / avg / 1e6, 1),
                             "frac": round(b / avg / 1e6 / peak_gbs, 4)}
    del imgs1, imgs2
    torch.cuda.empty_cache()

    # ---- e2e: the `stitching` command's shape.  The 32 tiles of the 4x4x2 grid are uploaded ONCE per step from
    # pinned host memory (async, on the copy stream) and the 112 pairs are phase-correlated on the resident tiles
    # (crops cut on the device; here the overlap crop is the whole 512^3 tile, the unit north_star names)
    def pcm_e2e():
        ntile = 32
        tiles, offs = synthetic.make_pcm_grid_workload(n=n, device=dev, seed=43 + rank, n_tiles=ntile)
        host_tiles = [t.cpu().pin_memory() for t in tiles]
        host_np = [h.numpy().view(np.uint16) for h in host_tiles]
        del tiles
        torch.cuda.empty_cache()
        gpairs = synthetic.grid_pairs_4x4x2()
        gpairs = sorted(gpairs, key=lambda p: max(p))          # pairs become runnable as their tiles arrive
        if npairs < len(gpairs):
            gpairs = gpairs[:npairs]
        used = sorted({t for p in gpairs for t in p})

        def step_host():
            hs = {t: ctx.volume_upload_async(host_np[t]) for t in used}
            jobs = [(hs[a], hs[b], (0, 0, 0), (0, 0, 0), (n, n, n)) for a, b in gpairs]
            out = ctx.pcm_volumes_batch(jobs, params)
            for h in hs.values():
                ctx.volume_free(h)
            return out

        rh = step_host()
        good = 0
        for (a, b), r in zip(gpairs, rh):
            want = tuple(offs[b][d] - offs[a][d] for d in range(3))     # img2(p) = img1(p + s), s = s_b - s_a
            good += int(r.found and tuple(r.shift_int) == want)
        step_host()
        e2e_ms, _ = timed(step_host, args.steps)
        dump_pcm(args.dump_outputs, "pcm_e2e", timed.last)
        e2e_value = world * len(gpairs) / (e2e_ms / args.steps / 1000.0)
        return {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": len(used) * n ** 3 * 2,
               "d2h_bytes_per_step": len(gpairs) * 2400, "ms_per_step": e2e_ms / args.steps,
               "what": f"{len(used)} tiles of {n}^3 uint16 uploaded once per step from pinned host memory "
                       f"(bs_volume_upload_async), {len(gpairs)} pairs on the resident tiles (bs_pcm_volumes_batch), "
                       f"one result block read back per pair",
               "recovered_planted_shifts": f"{good}/{len(gpairs)}"}

    e2e = None
    if not args.skip_pcm_e2e:
        e2e, exc = optional(pcm_e2e, 1)   # an optional section must never take the headline line down (or hang a rank)
        if exc is not None:
            e2e = {"value": None, "unit": UNIT, "error": f"{type(exc).__name__}: {exc}"}
        torch.cuda.empty_cache()

    # ---------------------------------------------------------------- affine fusion (config 3)
    fusion_obj = None
    if not args.skip_fusion:
        torch.cuda.empty_cache()
        fusion_obj = bench_fusion(args, ctx, stream, dev, rank, world, timed, peak_gbs, peak_src)
    if fusion_obj is not None and cpu_fusion is not None:
        fusion_obj["cpu_baseline"] = cpu_fusion

    # ---------------------------------------------------------------- DoG interest points (BASELINE configs[3], stretch row)
    dog_obj = None
    if not args.skip_dog:
        torch.cuda.empty_cache()
        dog_obj, exc = optional(lambda: bench_dog(args, ctx, stream, dev, rank, world, timed, peak_gbs), 1)
        if exc is not None:
            dog_obj = {"value": None, "error": f"{type(exc).__name__}: {exc}"}
        elif cpu_dog is not None:
            dog_obj["cpu_baseline"] = cpu_dog

    if rank == 0:
        bpp = pcm_bytes_per_pair(n ** 3, P, pearson_px_mean)
        dom = max(kern, key=lambda k: kern[k]["ms"]) if kern else None
        roof = None
        if dom:
            tr = ncu_traffic_r2("pcm") or {}
            roof = {"bound": "hbm", "kernel": dom, "achieved": kern[dom]["gbs"], "peak": peak_gbs, "unit": "GB/s",
                    "frac": kern[dom]["frac"],
                    "traffic": tr.get(dom) if (n, tuple(P)) == (512, (540, 540, 540)) else None,
                    "traffic_source": "profiles/ncu_traffic_r2.json (ncu --set full capture of this round's kernels, 512^3 pair)",
                    "peak_source": peak_src,
                    "alg_bytes_per_launch": kern[dom]["alg_bytes"], "ms_per_launch": kern[dom]["ms"],
                    "kernels": kern,
                    "pipeline": {"alg_bytes_per_pair": int(bpp), "pad": list(P),
                                 "gbs": round(value / world * bpp / 1e9, 1),
                                 "frac": round(value / world * bpp / 1e9 / peak_gbs, 4)}}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD_PCM if (npairs, n) == (112, 512) else
                       f"phase-correlation: {npairs} pairs/GPU of {n}^3 uint16 overlap crops, pad {P[0]}x{P[1]}x{P[2]}",
                       "pairs_per_gpu": npairs, "l2": "inputs larger than L2 (no flush needed)",
                       "distinct_fields": args.fields,
                       "planted_shifts": "integer in [-20,20]^3, every second pair + Fourier-domain sub-pixel part in [-0.5,0.5)^3",
                       "recovered_planted_shifts": f"{recovered}/{npairs} within 0.5 px (the three-point quadratic fit of the reference is not exact for band-limited shifts)",
                       "max_subpixel_error_px": round(float(max(sub_err)), 4) if sub_err else None,
                       "oracle_check": oracle_check,
                       "mean_pearson_candidates": ncand_mean,
                       "numa_node_of_rank0": numa_node},
            "e2e": e2e,
            "gpu_launches": int(launches), "wall_ms_timed": wall_ms, "clocks": clocks,
            "roofline": roof, "cpu_baseline": cpu, "fusion": fusion_obj, "dog": dog_obj,
        }
        print(json.dumps(line), flush=True)
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


def bench_dog(args, ctx, stream, dev, rank, world, timed, peak_gbs):
    """SparkInterestPointDetection's DoG (sigma 1.8, threshold 0.008, quadratic localisation) on one synthetic bead tile
    per rank, processed in the reference's 512x512x128 blocks (+1 px halo inside the image, J/SparkInterestPointDetection.java:
    397-424).  Mvoxels/s of tile voxels; algorithmic bytes per voxel = 2 (uint16 read) -- everything else is scratch."""
    import torch
    import bsgpu
    from bsgpu import fusion as bf
    n = args.dog_size
    g = torch.Generator(device=dev)
    g.manual_seed(77 + rank)
    vol = torch.rand((n // 4 if n >= 512 else n, n, n), generator=g, device=dev) * 60 + 180     # [z, y, x] background
    nz = vol.shape[0]
    nb = 400
    cz = torch.randint(4, nz - 4, (nb,), generator=g, device=dev)
    cy = torch.randint(4, n - 4, (nb,), generator=g, device=dev)
    cx = torch.randint(4, n - 4, (nb,), generator=g, device=dev)
    r = torch.arange(-4, 5, device=dev, dtype=torch.float32)
    bead = 3000.0 * torch.exp(-(r[:, None, None] ** 2 + r[None, :, None] ** 2 + r[None, None, :] ** 2) / (2 * 1.8 ** 2))
    for i in range(nb):
        z, y, x = int(cz[i]), int(cy[i]), int(cx[i])
        vol[z - 4:z + 5, y - 4:y + 5, x - 4:x + 5] += bead
    tile = torch.clamp(torch.round(vol), 0, 32767).to(torch.int16).contiguous()
    del vol
    torch.cuda.synchronize()
    h = ctx.volume_wrap(tile, (n, n, nz), bsgpu.native.DTYPE_U16)
    blocks = []
    for (off, size, _) in bf.grid_create((n, n, nz), (512, 512, 128)):
        lo = [max(0, off[d] - 1) for d in range(3)]
        hi = [min((n, n, nz)[d] - 1, off[d] + size[d]) for d in range(3)]
        blocks.append((lo, [hi[d] - lo[d] + 1 for d in range(3)]))
    found = []

    def step():
        found.clear()
        for lo, sz in blocks:
            found.extend(ctx.dog_detect(h, lo, sz, sigma=1.8, threshold=0.008, min_intensity=0.0, max_intensity=4000.0))
    step()
    nfound = len({p[2] for p in found})
    ms, _ = timed(step, args.steps)
    ms /= args.steps
    if args.dump_outputs:
        for i, name in enumerate(("loc", "value", "voxel", "is_max")):
            dump(args.dump_outputs, "dog_" + name, [p[i] for p in found])
    nvox = n * n * nz
    ctx.volume_free(h)
    return {"metric": "DoG interest points, Mvoxels/sec", "value": world * nvox / (ms / 1000.0) / 1e6, "unit": "Mvoxels/s", "ms_per_step": ms,
            "config": {"workload": f"one {n}x{n}x{nz} uint16 bead tile per GPU, {len(blocks)} blocks of 512x512x128 (+1 px), sigma 1.8, "
                                   f"threshold 0.008, MAX, quadratic localisation", "planted_beads": nb, "detections": nfound},
            "frac_of_hbm_peak": round(2.0 * nvox / (ms / 1000.0) / 1e9 / peak_gbs, 4)}


def bench_fusion(args, ctx, stream, dev, rank, world, timed, peak_gbs, peak_src):
    """SparkAffineFusion config: 4x4x4 grid of 576^3 uint16 tiles -> 2048^3 float32, AVG_BLEND,
    super-blocks 256x256x128 (blockSize 128^3, blockScale 2,2,1); z-slab per rank (strong scaling)."""
    import torch
    import bsgpu
    from bsgpu import fusion as bf
    from bsgpu import synthetic
    nat = bsgpu.native

    g, tile, stride, out_n = args.fusion_grid, args.fusion_tile, args.fusion_stride, args.fusion_size
    tiles, models, tdims = synthetic.make_fusion_workload((g, g, g), tile, stride, dev, n_distinct=args.fusion_distinct)
    torch.cuda.synchronize()
    nviews = len(tiles)
    regs = {i: models[i] for i in range(nviews)}
    vdims = {i: tdims for i in range(nviews)}
    zs = out_n // world
    z_lo, z_hi = rank * zs, (rank + 1) * zs if rank < world - 1 else out_n
    mine = bf.find_overlapping_views(vdims, regs, (0, 0, z_lo), (out_n - 1, out_n - 1, z_hi - 1))
    handles = {i: ctx.volume_wrap(tiles[i], tdims, nat.DTYPE_U16) for i in mine}
    blending = {i: bf.adjust_blending(models[i]) for i in mine}
    grid = [b for b in bf.grid_create((out_n, out_n, out_n), (256, 256, 128), (128, 128, 128))
            if z_lo <= b[0][2] < z_hi]
    grid.sort(key=lambda b: (b[0][2], b[0][1], b[0][0]))
    nvox_rank = sum(int(np.prod(b[1])) for b in grid)
    nvox_total = out_n ** 3
    out = torch.empty(nvox_rank, dtype=torch.float32, device=dev)
    CH = args.fusion_blocks_per_call

    def build_calls(view_dicts, out_ptr, esize):
        """one bs_fuse_blocks call per CH super-blocks (the work-queue form of the reference's per-block tasks)"""
        calls, off = [], 0
        for c0 in range(0, len(grid), CH):
            chunk = grid[c0:c0 + CH]
            lo = tuple(min(b[0][d] for b in chunk) for d in range(3))
            hi = tuple(max(b[0][d] + b[1][d] - 1 for b in chunk) for d in range(3))
            vregs = {v: view_dicts[v]["src_to_world"] for v in mine}      # the variant's own registrations
            vids = bf.find_overlapping_views(vdims, vregs, lo, hi, mine)
            views = ctx.make_views(view_dicts[v] for v in vids)
            ptrs = []
            for (_, sz, _g) in chunk:
                ptrs.append(out_ptr + esize * off)
                off += int(np.prod(sz))
            calls.append((views, [b[0] for b in chunk], [b[1] for b in chunk], ptrs, vids))
        return calls

    def view_dict(v, handle):
        return dict(src_to_world=models[v], vol_handle=handle, blend_border=blending[v][0], blend_range=blending[v][1])

    def run_variant(fusion_type, view_dicts, steps):
        p = ctx.fuse_params(fusion_type, 1, nat.DTYPE_F32)
        calls = build_calls(view_dicts, out.data_ptr(), 4)

        def step():
            for views, mins, sizes, ptrs, _ in calls:
                ctx.fuse_blocks(views, mins, sizes, p, outs=ptrs)
        for _ in range(3):
            step()
        l0 = ctx.launch_count()
        ms, _ = timed(step, steps)
        return ms / steps, ctx.launch_count() - l0, step

    vd = {v: view_dict(v, handles[v]) for v in mine}
    ms_step, launches, step_resident = run_variant("AVG_BLEND", vd, args.steps)
    launches //= args.steps
    value = nvox_total / (ms_step / 1000.0) / 1e6
    if args.dump_outputs:   # before the variants below overwrite `out`
        idx = np.sort(np.random.default_rng(0).choice(nvox_rank, min(DUMP_SAMPLE, nvox_rank), replace=False))
        dump(args.dump_outputs, "fusion_sample_index", idx)
        dump(args.dump_outputs, "fusion_sample", out[torch.from_numpy(idx).to(dev)].cpu().numpy())

    # ---- parity spot check against the C oracle, outside the timed region: one super-block at a 8-tile junction
    oracle_check = None
    if rank == 0 and world == 1 and not args.skip_oracle and (g, tile, stride) == (4, 576, 491):
        try:
            from oracle import c_fusion, fusion_oracle as fo
            bmin, bsz = (384, 384, 384), (256, 256, 128)
            vids = bf.find_overlapping_views(vdims, regs, bmin, tuple(bmin[d] + bsz[d] - 1 for d in range(3)), mine)
            ov = [fo.View(tiles[v].cpu().numpy().view(np.uint16), models[v], blending[v][0], blending[v][1], None) for v in vids]
            want = c_fusion.fuse_block(ov, bmin, bsz, fo.AVG_BLEND)
            got = ctx.fuse_block(ctx.make_views(vd[v] for v in vids), bmin, bsz, ctx.fuse_params("AVG_BLEND", 1, nat.DTYPE_F32))
            err = np.abs(got - want) / np.maximum(np.abs(want), 250.0)
            oracle_check = (f"super-block {bmin}+{bsz}, {len(vids)} views: max rel err {float(err.max()):.2e}, "
                            f"{int((err > 1e-4).sum())} of {err.size} voxels beyond 1e-4 (oracle/c/fusion_oracle.c)")
            del ov, want, got
        except Exception as e:  # the check must never take the bench down
            oracle_check = f"failed: {e}"

    # ---- per-kernel timing pass + roofline of the fusion kernel
    roof = None
    if rank == 0:
        ctx.profile_reset()
        ctx.profile_enable(True)
        step_resident()
        ctx.profile_enable(False)
        tms, cnt = ctx.profile_get("fuse")
        pms, pcnt = ctx.profile_get("fuse_plan")
        src_vox = 0
        for i in mine:
            bmin, bmax = bf.transformed_bounding_box(tdims, models[i])
            lo = np.maximum(bmin, (0, 0, z_lo))
            hi = np.minimum(bmax, (out_n - 1, out_n - 1, z_hi - 1))
            src_vox += int(np.prod(np.maximum(hi - lo + 1, 0)))
        alg = nvox_rank * 4 + src_vox * 2
        if cnt:
            tr = ncu_traffic_r2("fusion") or {}
            traffic = None
            if tr.get("bytes_per_voxel"):
                traffic = int(tr["bytes_per_voxel"] * nvox_rank / cnt)
            roof = {"bound": "hbm", "kernel": "fuse_tma_kernel<translation>", "achieved": round(alg / tms / 1e6, 1),
                    "peak": peak_gbs, "unit": "GB/s", "frac": round(alg / tms / 1e6 / peak_gbs, 4), "traffic": traffic,
                    "traffic_source": "profiles/ncu_traffic_r2.json: dram read+write bytes per output voxel of the ncu --set full "
                                      "capture (64 super-blocks, 2.1 GB output + 1.8 GB input: larger than L2), scaled to this launch",
                    "peak_source": peak_src, "alg_bytes_per_step": int(alg), "alg_bytes_per_launch": int(alg / cnt),
                    "ms_per_launch": round(tms / cnt, 4), "launches_per_step": int(cnt),
                    "plan_kernel_ms_per_step": round(pms, 4),
                    "bytes_per_voxel": round(alg / nvox_rank, 3), "kernel_only_mvox_s": round(nvox_rank / tms / 1e3, 1)}

    # ---- named variants (resident): 0.5 degree rotation (general affine kernel), content-based blending
    def run_variants(variants):
        t2, m2, _ = synthetic.make_fusion_workload((g, g, g), tile, stride, dev, n_distinct=args.fusion_distinct, rot_deg=0.5)
        del t2
        models_rot = m2
        vd_rot = {v: dict(src_to_world=models_rot[v], vol_handle=handles[v], blend_border=bf.adjust_blending(models_rot[v])[0],
                          blend_range=bf.adjust_blending(models_rot[v])[1]) for v in mine}
        ms_r, _, _ = run_variant("AVG_BLEND", vd_rot, args.steps)
        variants["rotated_0.5deg_z"] = {"value": nvox_total / (ms_r / 1000.0) / 1e6, "unit": "Mvoxels/s", "ms_per_step": ms_r,
                                        "kernel": "fuse_tma_kernel<general> (xy-affine z-marching tiles for <= 2 views, per-voxel tiles otherwise)"}
        # a rotation about an oblique axis has no exploitable structure: every voxel samples 8 taps
        ax = np.array([1.0, 1.0, 1.0]) / np.sqrt(3.0)
        th = np.deg2rad(0.5)
        K = np.array([[0, -ax[2], ax[1]], [ax[2], 0, -ax[0]], [-ax[1], ax[0], 0]])
        Rg = np.eye(3) + np.sin(th) * K + (1 - np.cos(th)) * (K @ K)
        models_obl = []
        for v in range(nviews):
            t = np.asarray(models[v])[:, 3]
            c = np.array([tile / 2, tile / 2, tile / 2])
            models_obl.append(np.hstack([Rg, (t + c - Rg @ c)[:, None]]))
        vd_obl = {v: dict(src_to_world=models_obl[v], vol_handle=handles[v], blend_border=bf.adjust_blending(models_obl[v])[0],
                          blend_range=bf.adjust_blending(models_obl[v])[1]) for v in mine}
        ms_o, _, _ = run_variant("AVG_BLEND", vd_obl, args.steps)
        variants["rotated_0.5deg_oblique"] = {"value": nvox_total / (ms_o / 1000.0) / 1e6, "unit": "Mvoxels/s", "ms_per_step": ms_o,
                                              "kernel": "fuse_tma_kernel<general> (per-voxel 8-tap tiles)"}
        if not args.skip_fusion_content:
            # content-based weights G_s2 * (I - G_s1 * I)^2 (sigma 20 / 40) are precomputed per DISTINCT tile volume
            t0 = time.perf_counter()
            chandle = {}
            for v in mine:
                key = tiles[v].data_ptr()
                if key not in chandle:
                    chandle[key] = ctx.content_weights(handles[v], 20.0, 40.0)
            ctx.synchronize()
            pre_s = time.perf_counter() - t0
            vd_c = {v: dict(vd[v], content_handle=chandle[tiles[v].data_ptr()]) for v in mine}
            ms_c, _, _ = run_variant("AVG_BLEND_CONTENT", vd_c, args.steps)
            variants["content_based"] = {"value": nvox_total / (ms_c / 1000.0) / 1e6, "unit": "Mvoxels/s", "ms_per_step": ms_c,
                                         "fusion_type": "AVG_BLEND_CONTENT", "sigma": [20.0, 40.0],
                                         "alg_bytes_per_voxel": 12.54, "kernel": "fuse_tma_kernel<translation, content> (content taps from global memory)",
                                         "frac_of_hbm_peak": round(12.54 * nvox_rank / (ms_c / 1000.0) / 1e9 / peak_gbs, 4),
                                         "content_precompute_s": round(pre_s, 3),
                                         "content_volumes": len(chandle)}
            for h in chandle.values():
                ctx.volume_free(h)

    variants = {}
    if not args.skip_fusion_variants:
        _, exc = timed.optional(lambda: run_variants(variants), 2 if args.skip_fusion_content else 3)
        if exc is not None:
            variants["error"] = f"{type(exc).__name__}: {exc}"

    # ---- e2e: the `affine-fusion` command's shape.  Every step uploads the z-range of each tile that the rank's
    # slab needs from pinned host memory (windowed views, async on the copy stream), fuses CH super-blocks per call
    # and streams the blocks back to pinned host buffers on the D2H stream while the next group is fused.
    def fusion_e2e():
        hosts = {}
        for i in mine:
            key = tiles[i].data_ptr()
            if key not in hosts:
                hosts[key] = tiles[i].cpu().pin_memory()
        host_np = {i: hosts[tiles[i].data_ptr()].numpy().view(np.uint16) for i in mine}
        # block-wise source staging (the reference's OverlappingBlocks idea): per call (CH super-blocks = one z-layer of
        # the block grid) every overlapping tile contributes only the z-range that layer can sample, as a windowed view
        plan = []
        for c0 in range(0, len(grid), CH):
            chunk = grid[c0:c0 + CH]
            lo = tuple(min(b[0][d] for b in chunk) for d in range(3))
            hi = tuple(max(b[0][d] + b[1][d] - 1 for b in chunk) for d in range(3))
            vids = bf.find_overlapping_views(vdims, regs, lo, hi, mine)
            wins = {}
            for v in vids:
                w0 = int(max(0, np.floor(lo[2] - models[v][2][3]) - 3))
                w1 = int(min(tdims[2] - 1, np.ceil(hi[2] - models[v][2][3]) + 3))
                if w1 >= w0:
                    wins[v] = (w0, w1)
            plan.append((chunk, [v for v in vids if v in wins], wins, [b[0] for b in chunk], [b[1] for b in chunk]))
        ring_n = min(len(grid), 2 * CH)
        h2d = sum((w1 - w0 + 1) * tdims[0] * tdims[1] * 2 for (_, _, wins, _, _) in plan for (w0, w1) in wins.values())

        def make_step(out_dtype, ring):
            p = ctx.fuse_params("AVG_BLEND", 1, out_dtype, 0, 0.0, 65535.0)
            ring_np = ring.numpy()
            outs_of, slot = [], 0
            for (chunk, _, _, _, _) in plan:
                o = []
                for (_, sz, _g) in chunk:
                    o.append(ring_np[slot % ring_n][:int(np.prod(sz))].reshape(sz[2], sz[1], sz[0]))
                    slot += 1
                outs_of.append(o)

            def step_host():
                # every window of the step is queued on the copy stream up front, in the order the calls need them
                handles_of = []
                for (_, vids, wins, _, _) in plan:
                    handles_of.append({v: ctx.volume_upload_async(host_np[v][wins[v][0]:wins[v][1] + 1]) for v in vids})
                for (chunk, vids, wins, mins, sizes), hs, outs in zip(plan, handles_of, outs_of):
                    views = ctx.make_views(dict(vd[v], vol_handle=hs[v], full_dims=tdims, window_min=(0, 0, wins[v][0])) for v in vids)
                    ctx.fuse_blocks(views, mins, sizes, p, outs=outs)
                    for h in hs.values():
                        ctx.volume_free(h)
            return step_host

        nst = args.steps
        ring_f32 = torch.empty((ring_n, 256 * 256 * 128), dtype=torch.float32).pin_memory()
        step_host = make_step(nat.DTYPE_F32, ring_f32)
        step_host()
        e2e_ms, _ = timed(step_host, nst)
        e2e = {"value": nvox_total / (e2e_ms / nst / 1000.0) / 1e6, "unit": "Mvoxels/s", "h2d_bytes_per_step": int(h2d),
               "d2h_bytes_per_step": int(nvox_rank * 4), "ms_per_step": e2e_ms / nst,
               "what": f"per bs_fuse_blocks call ({CH} super-blocks = one z-layer of the grid) the z-range of every overlapping tile is "
                       "uploaded from pinned host memory as a windowed view (async, copy stream); float32 blocks stream to pinned "
                       "host buffers on the D2H stream while the next group is fused"}
        del ring_f32, step_host
        ring_u16 = torch.empty((ring_n, 256 * 256 * 128), dtype=torch.int16).pin_memory()
        step_host16 = make_step(nat.DTYPE_U16, ring_u16)
        step_host16()
        e2e16_ms, _ = timed(step_host16, nst)
        e2e_u16 = {"value": nvox_total / (e2e16_ms / nst / 1000.0) / 1e6, "unit": "Mvoxels/s", "h2d_bytes_per_step": int(h2d),
                   "d2h_bytes_per_step": int(nvox_rank * 2), "ms_per_step": e2e16_ms / nst,
                   "what": "same with uint16 output (the reference's usual -d UINT16, min 0 / max 65535)"}
        return e2e, e2e_u16

    e2e = e2e_u16 = None
    if not args.skip_fusion_e2e:
        res, exc = timed.optional(fusion_e2e, 2)
        if exc is not None:
            e2e = {"value": None, "unit": "Mvoxels/s", "error": f"{type(exc).__name__}: {exc}"}
        else:
            e2e, e2e_u16 = res

    # ---- view-sharded mode (N > 1): the ONE exchange step of the path -- every rank accumulates its share of the views
    # of one 8-tile-junction super-block, one grouped NCCL all-reduce of [sum wI, sum w] behind the C ABI
    # (bs_fuse_accumulate -> bs_fuse_allreduce -> bs_fuse_finish, all on the context's stream, no host sync between)
    view_sharded = None
    if world > 1:
        import torch.distributed as dist
        from bsgpu import parallel as bpar

        def all_ranks_ok(ok):
            """collective agreement BEFORE a section with its own collectives: one failing rank must not leave the
            others waiting inside an all-reduce"""
            t = torch.tensor([1 if ok else 0], device=dev, dtype=torch.int32)
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            return bool(t.item())

        hs, err = {}, None
        try:   # ---- per-rank preparation, no collectives
            bmin, bsz = (384, 384, 384), (256, 256, 128)
            vids = bf.find_overlapping_views(vdims, regs, bmin, tuple(bmin[d] + bsz[d] - 1 for d in range(3)), list(range(nviews)))
            my = bpar.partition_views(vids, rank, world)
            hs = {v: ctx.volume_wrap(tiles[v], tdims, nat.DTYPE_U16) for v in my}
            myviews = ctx.make_views(dict(src_to_world=models[v], vol_handle=hs[v], blend_border=bf.adjust_blending(models[v])[0],
                                          blend_range=bf.adjust_blending(models[v])[1]) for v in my)
            nb = int(np.prod(bsz))
            with torch.cuda.stream(stream):
                swi = torch.zeros(nb, dtype=torch.float32, device=dev)
                sw = torch.zeros(nb, dtype=torch.float32, device=dev)
                outd = torch.empty(nb, dtype=torch.float32, device=dev)
            pvs = ctx.fuse_params("AVG_BLEND", 1, nat.DTYPE_F32)
        except Exception as exc:
            err = exc
        if not all_ranks_ok(err is None):
            view_sharded = {"value": None, "error": f"{type(err).__name__}: {err}" if err else "another rank failed to prepare"}
        else:
            bpar.comm_init_from_torch(ctx)

            def step_vs():
                with torch.cuda.stream(stream):
                    swi.zero_()
                    sw.zero_()
                ctx.fuse_accumulate(myviews, bmin, bsz, pvs, swi, sw)
                ctx.fuse_allreduce(swi, sw, nb)
                ctx.fuse_finish(swi, sw, nb, pvs, outd)
            for _ in range(3):
                step_vs()
            ms_vs, _ = timed(step_vs, args.steps)
            ms_vs /= args.steps
            view_sharded = {"value": nb / (ms_vs / 1000.0) / 1e6, "unit": "Mvoxels/s", "ms_per_block": ms_vs,
                            "block": list(bsz), "views_total": len(vids), "views_on_rank0": len(my),
                            "allreduce_bytes_per_block": 2 * nb * 4,
                            "what": "one 256x256x128 super-block at an 8-tile junction, views partitioned over the ranks, one grouped "
                                    "NCCL all-reduce of the two float32 partial-sum buffers on the context's stream, result on every rank"}
            ctx.comm_destroy()
        for h in hs.values():
            ctx.volume_free(h)

    for h in handles.values():
        ctx.volume_free(h)
    return {"metric": "fused Mvoxels/sec (affine fusion, AVG_BLEND, float32 out)", "value": value, "unit": "Mvoxels/s",
            "scaling": "strong", "ms_per_step": ms_step, "gpu_launches": int(launches),
            "config": {"workload": f"{g}x{g}x{g} grid of {tile}^3 uint16 tiles (stride {stride}, jitter +-2 px) -> "
                                   f"{out_n}^3 float32, super-blocks 256x256x128, z-slab per GPU",
                       "distinct_tile_volumes": args.fusion_distinct, "views_on_rank0": len(mine),
                       "blocks_per_call": CH, "oracle_check": oracle_check,
                       "l2": "output 34 GB + inputs larger than L2"},
            "e2e": e2e, "e2e_uint16": e2e_u16, "variants": variants, "view_sharded": view_sharded,
            "roofline": roof}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--pairs", type=int, default=112)
    ap.add_argument("--size", type=int, default=512)
    ap.add_argument("--fields", type=int, default=4)
    ap.add_argument("--skip-fusion", action="store_true")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--skip-fusion-e2e", action="store_true")
    ap.add_argument("--skip-pcm-e2e", action="store_true")
    ap.add_argument("--skip-oracle", action="store_true", help="skip the oracle spot checks outside the timed region")
    ap.add_argument("--skip-fusion-variants", action="store_true")
    ap.add_argument("--skip-fusion-content", action="store_true")
    ap.add_argument("--skip-dog", action="store_true")
    ap.add_argument("--dog-size", type=int, default=1024)
    ap.add_argument("--fusion-blocks-per-call", type=int, default=64)
    ap.add_argument("--skip-pcm", action="store_true", help="debug: tiny PCM workload")
    ap.add_argument("--ref-full", action="store_true", help="reference arm: run all warm-up steps too")
    ap.add_argument("--fusion-grid", type=int, default=4)
    ap.add_argument("--fusion-tile", type=int, default=576)
    ap.add_argument("--fusion-stride", type=int, default=491)
    ap.add_argument("--fusion-size", type=int, default=2048)
    ap.add_argument("--fusion-distinct", type=int, default=64)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write rank 0's outputs of the last timed steps as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if rank != 0:
        args.dump_outputs = None
    wd = int(os.environ.get("BS_BENCH_WATCHDOG", "0"))
    if wd > 0:      # debugging aid for multi-rank runs: every `wd` seconds each rank dumps where it is
        import faulthandler
        faulthandler.dump_traceback_later(wd, repeat=True, file=sys.stderr)
    if args.impl == "reference":
        run_reference(args, rank)
        return
    run_gpu(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
