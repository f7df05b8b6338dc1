#!/usr/bin/env python
"""Benchmark of the alignment hot path (BASELINE.json: audio-hours aligned per second).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--pairs B] [--impl ours|reference] [--dump-outputs DIR]

A step = one pass of the hot path over one batch of B synthetic pairs per GPU of the C2 shape (22-min
video audio vs 27-min description, 202 s start offset, injected skips; SURVEY.md 8d): features of both
tracks, device stage A (describealign.py:596-700) and device stage B (:895-993).  The host-side
rate-change fit between the two device stages (:702-893) is outside the timed regions, as BASELINE.json
prescribes; it is solved once per distinct pair and reused for as long as stage A returns the identical
pass-1 path.  The pairs go through the library's batch engine (include/describealign_b200.h, dab_engine_*):
W slots per GPU, every device stage enqueued in one go by one scheduler thread, one Python thread serving
the event queue.  The configuration (W, B, distinct pairs per GPU) is the same at every N.

value   device-resident: PCM already in HBM when the timed region starts; one CUDA-event bracket around
        the whole step.
e2e     the same passes from pinned HOST buffers: H2D of the PCM and D2H of the results inside the region.
One rank per GPU (torchrun for N > 1); ranks process disjoint pairs (weak scaling), no data-path
collective; timings are max over ranks.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

# one CUDA stream per pair in flight: ask for the maximum number of hardware queues before CUDA starts
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")
# the benchmark may run from a read-only tree: it writes nothing there, bytecode caches included
sys.dont_write_bytecode = True

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "audio_hours_aligned_per_second"
UNIT = "audio-hours/s"
WORKLOADS = {
    "C2": "C2: synthetic 22-min video audio vs 27-min description, 202 s offset, 10 inserted skips, mono 44.1 kHz s16",
    "C3": "C3: the C2 pair in stereo (--stretch_audio feature semantics: features from 2 channels), 44.1 kHz s16",
    "C4": "C4: batch mode, 64 distinct synthetic 45-min episode/description pairs (offset 10-90 s, 4-8 skips) sharded over the GPUs, mono 44.1 kHz s16",
    "C5": "C5: long-form, ONE synthetic 2.5-h film vs 3-h description (300 s offset, ~12 skips), match stage and corridor scoring split over the GPUs by audio rows, mono 44.1 kHz s16",
}
WORKLOAD = WORKLOADS["C2"]      # the configuration BASELINE.json's metric is quoted on (the default)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--pairs", type=int, default=0, help="pairs per GPU per step (default: 8 x slots)")
    ap.add_argument("--workers", type=int, default=0, help="engine slots = pairs on the device at once per GPU (default 32, at every N)")
    ap.add_argument("--distinct", type=int, default=0,
                    help="distinct synthetic pairs per GPU, a step cycles over them (default 4 at every N: 1 GB of PCM, 8x the L2)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="C2", choices=sorted(WORKLOADS),
                    help="C2 (default, the metric's configuration), C3 (stereo), C4 (64 x 45-min pairs over all GPUs: strong scaling), "
                         "C5 (one long pair split over all GPUs: strong scaling)")
    ap.add_argument("--scale", type=float, default=1.0, help="shrink the C2 durations (debugging only)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-numa-bind", action="store_true", help="do not pin the rank to the CPUs of its GPU's NUMA node")
    ap.add_argument("--no-long-pair", action="store_true", help="N > 1: skip the long-pair (C5) check that runs on all ranks after the timed steps")
    ap.add_argument("--long-scale", type=float, default=0.1, help="scale of the C5 pair used for the N > 1 long-pair check")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last device-resident step computed as DIR/<name>.npy: pass-1 path, "
                         "features and final path rows of its first %d distinct pairs, copied inside that step (C5: the nodes "
                         "and path of the pair); a seeded sample of rows where that exceeds 64 MB" % DUMP_PAIRS)
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs --impl ours: the reference arm keeps no outputs")
    return args


DUMP_PAIRS = 4
DUMP_BYTES = 60 << 20       # the arrays; with the .npy headers the files stay under 64 MB


def dump_outputs(out_dir, arrays, seed=0):
    """arrays: name -> float32 / float64 array, written as out_dir/<name>.npy.  When they hold more than DUMP_BYTES,
    every array over 1 MB keeps the same fraction of its rows, chosen with a fixed seed and kept in order, and
    out_dir/<name>_rows.npy lists which rows those are."""
    os.makedirs(out_dir, exist_ok=True)
    large = [name for name, a in arrays.items() if a.nbytes > 1 << 20]
    budget = DUMP_BYTES - sum(a.nbytes for name, a in arrays.items() if name not in large)
    frac = 1.0
    if sum(arrays[name].nbytes for name in large) > budget:
        frac = budget / sum(arrays[name].nbytes + 8 * len(arrays[name]) for name in large)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        if name in large and frac < 1.0:
            rows = np.sort(np.random.default_rng(seed).choice(len(a), size=int(frac * len(a)), replace=False))
            a = a[rows]
            np.save(os.path.join(out_dir, name + "_rows.npy"), rows.astype(np.float64))
        np.save(os.path.join(out_dir, name + ".npy"), a)


def pair_arrays(x, y, video_features, audio_features):
    """What the batch engine hands a caller at the end of stage A, copied out of its slot buffers."""
    out = {"path1": np.stack([x, y], axis=1).astype(np.float64)}
    for track, feats in (("video", video_features), ("audio", audio_features)):
        for f, arr in enumerate(feats):
            out[f"{track}_feature{f}"] = np.array(arr, dtype=np.float32)
    return out


def make_pairs(n, first_seed, scale, world=1, config="C2"):
    """n pairs of a named configuration with distinct seeds, generated in parallel worker processes (the
    host's cores are shared by the `world` ranks of the node)."""
    from concurrent.futures import ProcessPoolExecutor
    from describealign_b200 import synth
    seeds = [first_seed + k for k in range(n)]
    if n == 1:
        return [synth.config_pair(config, seeds[0], scale)]
    with ProcessPoolExecutor(max_workers=max(1, min(n, (os.cpu_count() or 1) // max(1, world)))) as ex:
        return list(ex.map(_make_one, [(s, scale, config) for s in seeds]))


def _make_one(arg):
    from describealign_b200 import synth
    return synth.config_pair(arg[2], arg[0], arg[1])


def audio_hours(pairs):
    return sum(v.shape[0] + a.shape[0] for v, a in pairs) / 44100.0 / 3600.0


def visible_gpu_ids(world):
    """What `nvidia-smi -i` must be given to see the GPU of local rank 0 .. world-1: the rank itself, or the rank's
    entry of CUDA_VISIBLE_DEVICES (index or UUID) when the launcher restricted the devices."""
    vis = [t.strip() for t in os.environ.get("CUDA_VISIBLE_DEVICES", "").split(",") if t.strip()]
    return [vis[r] if r < len(vis) else str(r) for r in range(world)]


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region.  ONE process (rank 0's) watches the GPUs
    of all local ranks - `ids`, one nvidia-smi identifier (index or UUID) per rank - so that the other ranks' host
    cores are left alone."""
    Q = "index,uuid,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, ids, period_ms=200):
        self.ids = [str(i) for i in (ids if isinstance(ids, (list, tuple)) else [ids])]
        self.period_ms = int(period_ms)
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", ",".join(self.ids), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", str(self.period_ms)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def _rank_of(self, index, uuid):
        for r, ident in enumerate(self.ids):
            if ident == index or (not ident.isdigit() and uuid.startswith(ident)):
                return r
        return None

    def stop(self):
        """Summary over all watched GPUs (lowest median clock, every reason seen) + "per_gpu": {local rank: summary}."""
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "per_gpu": {}}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        per = {}
        mx = None
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                clk = float(f[2]); mx = float(f[3])
            except ValueError:
                continue
            r = self._rank_of(f[0], f[1])
            if r is None:
                continue
            g = per.setdefault(r, {"sm": [], "reasons": set()})
            g["sm"].append(clk)
            for k, nm in enumerate(names):
                if f[5 + k].lower().startswith("active"):
                    g["reasons"].add(nm)
        per_gpu = {r: {"sm_mhz": float(np.median(g["sm"])) if g["sm"] else None, "reasons": sorted(g["reasons"]),
                       "samples": len(g["sm"])} for r, g in per.items()}
        meds = [g["sm_mhz"] for g in per_gpu.values() if g["sm_mhz"] is not None]
        return {"sm_mhz": min(meds) if meds else None, "sm_max_mhz": mx,
                "reasons": sorted({r for g in per_gpu.values() for r in g["reasons"]}),
                "samples": sum(g["samples"] for g in per_gpu.values()), "gpus_sampled": len(per_gpu), "per_gpu": per_gpu}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        with open(p) as f:
            return json.load(f), "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------
# CPU arm (oracle port; the reference is Python and not present on the GPU box)
# ------------------------------------------------------------------------------------------------

def cpu_pass(pair, keep=False):
    """One pass of the hot path on the CPU through the oracle port.  Returns (times, outputs): times has
    hot_path_s = features + align() minus scipy.optimize.linprog (BASELINE.md section 3), linprog_s, and
    device_stages_s = only what the GPU arm times (features, stage A, stage B)."""
    import scipy.optimize
    from describealign_b200 import host_fit
    from oracle import align_oracle as ao, features as of
    v, a = pair
    lp = [0.0]

    def timed_linprog(*args, **kw):
        t = time.perf_counter()
        try:
            return scipy.optimize.linprog(*args, **kw)
        finally:
            lp[0] += time.perf_counter() - t

    t0 = time.perf_counter()
    V, A = of.all_features(v), of.all_features(a)
    sa = ao.stage_a(V, A, V[0], A[0])
    t1 = time.perf_counter()
    x, y = sa["path_x"], sa["path_y"]
    kp = host_fit.continuity_error(x, y) < 3
    kx, ky = x[kp], y[kp]
    a_s, v_s = host_fit.scale_features(V, A, kx, ky)
    fx, fy = host_fit.compress_path(kx, ky)
    fit = host_fit.rate_change_fit(fx, fy, linprog=timed_linprog)
    clusters = host_fit.line_clusters(fit)
    plans = ao.plan_corridors(clusters, a_s, v_s)
    t2 = time.perf_counter()
    sb = ao.stage_b(plans, len(clusters), a_s, v_s)
    path = sb["path"]
    nx, ny, sim = host_fit.build_nodes(path, len(A[0]), len(V[0]), len(a_s), len(v_s))
    t3 = time.perf_counter()
    times = {"hot_path_s": (t3 - t0) - lp[0], "linprog_s": lp[0], "device_stages_s": (t1 - t0) + (t3 - t2),
             "total_s": t3 - t0}
    out = len(path)
    if keep:
        out = {"V": V, "A": A, "path1": (x, y), "path": path, "nodes": (nx, ny), "similarity": sim}
    return times, out


def _cpu_worker(pair):
    os.environ.setdefault("OMP_NUM_THREADS", "1")
    return cpu_pass(pair)


def real_reference_pass(pair):
    """The UNMODIFIED reference (describealign.py installed under baseline/_ref by tools/install_reference.sh,
    loaded with stubs for its GUI / ffmpeg imports) on one pair in this process: its own get_energy /
    get_zero_crossings / get_freq_bands on the float16 (ch, S) arrays of describealign.py:156, then its own
    align().  Returns {"hot_path_s": seconds minus scipy.optimize.linprog (BASELINE.md section 3),
    "linprog_s": ...}, or None where the reference is not installed."""
    try:
        from oracle import ref_loader
        da = ref_loader.load()
    except Exception:
        return None
    if da is None:
        return None
    import contextlib
    import scipy.optimize
    v, a = pair
    lp = [0.0]
    orig = scipy.optimize.linprog

    def timed(*args, **kw):
        t = time.perf_counter()
        try:
            return orig(*args, **kw)
        finally:
            lp[0] += time.perf_counter() - t

    va = np.ascontiguousarray(v.T).astype(np.float16) if v.ndim == 2 else v.astype(np.float16)[None, :]
    aa = np.ascontiguousarray(a.T).astype(np.float16) if a.ndim == 2 else a.astype(np.float16)[None, :]
    scipy.optimize.linprog = timed
    try:
        with contextlib.redirect_stdout(sys.stderr):
            t0 = time.perf_counter()
            vf = [da.get_energy(va), da.get_zero_crossings(va)] + list(da.get_freq_bands(va))
            af = [da.get_energy(aa), da.get_zero_crossings(aa)] + list(da.get_freq_bands(aa))
            da.align(vf, af, vf[0], af[0])
            t1 = time.perf_counter()
    finally:
        scipy.optimize.linprog = orig
    return {"hot_path_s": (t1 - t0) - lp[0], "linprog_s": lp[0]}


def _ref_worker(pair):
    os.environ.setdefault("OMP_NUM_THREADS", "1")
    return real_reference_pass(pair)


def reference_installed():
    try:
        from oracle import ref_loader
        return any(os.path.isfile(p) for p in ref_loader.INSTALLED_CANDIDATES)
    except Exception:
        return False


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU path on all host cores, one pair per process (the reference is
    single-threaded and loops over a batch sequentially, describealign.py:1077; one process per core is the
    harness-side extension BASELINE.md section 3 allows).

    Where the unmodified describealign.py is installed under baseline/_ref (tools/install_reference.sh; it
    travels to the GPU box with the snapshot) THAT is what every step times - its own feature functions and
    align() through its own module-level API - and the oracle port (C features, C match + DPs, numpy/scipy
    host stage; ~6x faster per core) is timed once beside it.  Without an installed reference the port is
    the timed arm ("kind": "port")."""
    if rank != 0:
        return
    import oracle
    oracle.build()
    from concurrent.futures import ProcessPoolExecutor
    real = reference_installed()
    # bounded sample: one pair per host core (at most 16), whatever --pairs / --gpus say
    pairs = make_pairs(max(1, min(16, os.cpu_count() or 1)), 0, args.scale, 1, args.workload)
    hours = audio_hours(pairs)
    cores = min(len(pairs), os.cpu_count() or 1)
    worker = _ref_worker if real else _cpu_worker
    times, times_dev = [], []
    port_once = None
    with ProcessPoolExecutor(max_workers=cores) as ex:
        for step in range(args.warmup + args.steps):
            res = list(ex.map(worker, pairs))
            res = [r if real else r[0] for r in res]
            # each worker times its own pass (linprog subtracted, BASELINE.md section 3); with one process per
            # pair running concurrently the step takes as long as the slowest one
            hot = [r["hot_path_s"] for r in res]
            devs = [r.get("device_stages_s", r["hot_path_s"]) for r in res]
            if step >= args.warmup:
                times.append(max(max(hot) if cores >= len(pairs) else sum(hot) / cores, 1e-9))
                times_dev.append(max(max(devs) if cores >= len(pairs) else sum(devs) / cores, 1e-9))
        if real:
            # the port on the same pairs, one step, for the record
            res = [r[0] for r in ex.map(_cpu_worker, pairs)]
            port_once = {"value": hours / max(r["hot_path_s"] for r in res), "unit": UNIT, "cores": cores, "kind": "port",
                         "value_device_stages_only": hours / max(r["device_stages_s"] for r in res),
                         "sample": f"{len(pairs)} full {args.workload} pairs, one oracle-port process per pair, one step"}
    ms = 1e3 * float(np.mean(times))
    value = hours / (ms / 1e3)
    what = "the unmodified describealign.py (baseline/_ref)" if real else "the oracle port"
    cpu = {"value": value, "unit": UNIT, "cores": cores, "kind": "reference" if real else "port",
           "sample": f"{len(pairs)} full {args.workload} pairs per step, one process of {what} per pair",
           "host_cpu": _cpu_model(), "host_cores": os.cpu_count()}
    if real:
        cpu["oracle_port_beside_it"] = port_once
    else:
        cpu["value_device_stages_only"] = hours / float(np.mean(times_dev))
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32+f64", "data": "synthetic", "impl": "reference",
            "config": {"workload": WORKLOADS[args.workload], "pairs_per_step": len(pairs), "audio_hours_per_step": hours,
                       "scale": args.scale,
                       "timed": "features + align() minus scipy.optimize.linprog (BASELINE.md section 3), per pair, one process per pair"},
            "cpu_baseline": cpu,
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------

def d2h_probe(pinned, seconds=1.0):
    """GB/s this rank reaches copying device buffers of the size of its PCM back into its pinned buffers' twins,
    back to back for about `seconds` (all ranks at once): the ceiling of the result copies under contention."""
    import torch
    src = [torch.empty_like(t, device="cuda") for pair in pinned for t in pair]
    dst = [torch.empty(t.shape, dtype=t.dtype).pin_memory() for t in src[:2]]      # host twins of the first pair's tracks
    stream = torch.cuda.Stream()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    nbytes, t_end = 0, time.perf_counter() + seconds
    with torch.cuda.stream(stream):
        e0.record()
        while time.perf_counter() < t_end:
            for k, s_ in enumerate(src):
                d, sv = dst[k % 2].view(-1), s_.view(-1)
                m = min(d.numel(), sv.numel())
                d[:m].copy_(sv[:m], non_blocking=True)
                nbytes += m * sv.element_size()
            stream.synchronize()
        e1.record()
    e1.synchronize()
    return nbytes / (e0.elapsed_time(e1) * 1e-3) / 1e9


def h2d_probe(pinned, seconds=1.0):
    """GB/s this rank's pinned PCM buffers reach when copied back to back for about `seconds` (all ranks
    do this at the same time: the ceiling of the end-to-end number under the box's real contention)."""
    import torch
    bufs = [t for pair in pinned for t in pair]
    dst = [torch.empty_like(t, device="cuda") for t in bufs]
    stream = torch.cuda.Stream()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    nbytes, t_end = 0, time.perf_counter() + seconds
    with torch.cuda.stream(stream):
        e0.record()
        while time.perf_counter() < t_end:
            for d, s_ in zip(dst, bufs):
                d.copy_(s_, non_blocking=True)
                nbytes += s_.numel() * s_.element_size()
            stream.synchronize()
        e1.record()
    e1.synchronize()
    del dst
    return nbytes / (e0.elapsed_time(e1) * 1e-3) / 1e9


def long_pair_pcm(rank, scale, barrier):
    """The C5 pair, generated once (rank 0, segments in worker processes) and shared through /dev/shm."""
    from describealign_b200 import synth
    base = f"/dev/shm/dab_c5_{os.getuid()}_{scale:g}"
    if rank == 0:
        v, a = synth.long_pair(0, scale, workers=max(1, min(10, os.cpu_count() or 1)))
        np.save(base + "_v.npy", v)
        np.save(base + "_a.npy", a)
    barrier()
    if rank != 0:
        v, a = np.load(base + "_v.npy"), np.load(base + "_a.npy")
    barrier()
    if rank == 0:
        for suffix in ("_v.npy", "_a.npy"):
            try:
                os.remove(base + suffix)
            except OSError:
                pass
    return v, a


def run_long(args, rank, world, local_rank):
    """--workload C5: one long pair per step on ALL ranks (batch.align_long_pair).  Strong scaling: the match
    stage and the corridor scoring are sharded by audio rows (two all-gathers), both DPs run on rank 0.  The
    timed figure is device time - CUDA events on each rank around every phase, max over ranks - without the
    host rate-change fit (solved during warm-up, looked up afterwards: BASELINE.json excludes it)."""
    import torch
    import torch.distributed as dist
    from describealign_b200 import api, batch, build
    build.build()
    api.set_device(local_rank)
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    lv, la = long_pair_pcm(rank, args.scale, barrier)
    hours = audio_hours([(lv, la)])
    numa = batch.bind_to_gpu_numa_node(local_rank) if not args.no_numa_bind else {"bound": False, "disabled": True}
    # end-to-end arm: the PCM starts in pinned host memory (the H2D copy is inside align_long_pair's first phase);
    # device-resident arm: the PCM is handed over as device pointers
    pv, pa = torch.from_numpy(lv).pin_memory(), torch.from_numpy(la).pin_memory()
    dv, da_ = pv.cuda(), pa.cuda()
    dev_in = ((dv.data_ptr(), dv.shape[0], dv.shape[1]), (da_.data_ptr(), da_.shape[0], da_.shape[1]))
    cache = {}

    def cached_host_stage(job):
        c = cache.get("fit")
        if c is not None and np.array_equal(c["x"], job.x) and np.array_equal(c["y"], job.y):
            for name in c["keep"]:
                setattr(job, name, c["keep"][name])
            return
        job.host_stage()
        cache["fit"] = {"x": job.x.copy(), "y": job.y.copy(),
                        "keep": {name: getattr(job, name) for name in
                                 ("kept_x", "kept_y", "gains", "n_audio_scaled", "n_video_scaled", "fit", "clusters", "lines")}}

    def one_step(host_input):
        det = {}
        out = batch.align_long_pair(pv.numpy() if host_input else dev_in[0], pa.numpy() if host_input else dev_in[1],
                                    details=det, host_stage=cached_host_stage)
        ph = det["phases_ms"]
        dev_ms = sum(v for k, v in ph.items() if k not in batch.HOST_PHASES)
        return dev_ms, det, out

    def run_steps(host_input):
        for _ in range(args.warmup):
            one_step(host_input)
        barrier()
        tot, det, out = 0.0, None, None
        phases = {}
        for _ in range(args.steps):
            ms, det, out = one_step(host_input)
            t = torch.tensor([ms], device="cuda", dtype=torch.float64)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            tot += float(t[0])
            for k, v in det["phases_ms"].items():
                phases[k] = phases.get(k, 0.0) + v / args.steps
        barrier()
        return tot / args.steps, phases, det, out

    ctx = api.context()
    sampler = ClockSampler(visible_gpu_ids(world))    # rank 0 watches every local rank's GPU (one node)
    if rank == 0:
        sampler.start()
    l0 = ctx.launches()
    ms_dev, ph_dev, det, out = run_steps(False)
    launches = (ctx.launches() - l0) * args.steps // (args.steps + args.warmup)
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0 and args.dump_outputs:
        nx, ny, sim, path, med = out
        dump_outputs(args.dump_outputs, {"nodes_x": np.asarray(nx, np.float64), "nodes_y": np.asarray(ny, np.float64),
                                         "path2": np.asarray(path, np.float64), "similarity": np.array([sim], np.float64),
                                         "median_slope": np.array([med], np.float64)})
    ms_e2e, ph_e2e, _, _ = run_steps(True)
    lt = torch.tensor([float(launches)], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(lt, op=dist.ReduceOp.SUM)

    single = cpu = None
    if rank == 0:
        import contextlib
        with contextlib.redirect_stdout(sys.stderr):
            t1 = time.perf_counter()
            ref = api.align_pcm(lv, la)
            t_single = time.perf_counter() - t1
        single = {"identical_to_single_gpu_path": bool(np.array_equal(out[3], ref[3]) and np.array_equal(out[0], ref[0]) and
                                                       np.array_equal(out[1], ref[1])),
                  "wall_s_single_gpu_incl_host_fit": t_single}
        if not args.no_cpu_baseline:
            import oracle
            oracle.build()
            cpu_t, o = cpu_pass((lv, la), keep=True)
            cpu = {"value": hours / cpu_t["hot_path_s"], "unit": UNIT, "cores": 1, "kind": "port",
                   "sample": "the same long pair once through the oracle port; timed as BASELINE.md section 3 (minus linprog)",
                   "seconds": cpu_t["hot_path_s"], "seconds_linprog_subtracted": cpu_t["linprog_s"],
                   "host_cpu": _cpu_model(), "host_cores": os.cpu_count()}
            single["identical_to_oracle_path"] = bool(out[3].shape == o["path"].shape and np.array_equal(out[3][:, 1], o["path"][:, 1]) and
                                                      np.array_equal(out[3][:, 2], o["path"][:, 2]))
        peaks, peak_src = measured_peaks()
        sh = det.get("shards", {})
        pcm_b = lv.nbytes + la.nbytes
        feat_ms = ph_dev.get("features", 0.0)
        line = {"metric": METRIC, "value": hours / (ms_dev * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_dev, "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "f32+f64 (u32 packed codes)", "data": "synthetic",
                "config": {"workload": WORKLOADS["C5"], "scale": args.scale,
                           "pair_minutes": [len(lv) / 44100 / 60, len(la) / 44100 / 60], "audio_hours_per_step": hours,
                           "l2_policy": "inputs larger than L2 (%d MB of PCM per step; 126 MB L2)" % int(pcm_b / 1e6),
                           "timed": "per step ONE long pair on all ranks: features (every rank, the PCM once), match stage sharded by audio rows, all-gather of the match points, DP1 + traceback on rank 0, [host rate-change fit on rank 0: solved in warm-up, looked up inside the region, untimed by BASELINE.json], corridor scoring sharded by audio rows, all-gather of the quals, DP2 + traceback on rank 0, final path to the host; [similarity and node list in Python on rank 0, describealign.py:993-1026: untimed like in the C2 arm]; CUDA events per phase on every rank, summed without the two host phases, max over ranks"},
                "phases_ms_rank0": ph_dev,
                "e2e": {"value": hours / (ms_e2e * 1e-3), "unit": UNIT, "ms_per_step": ms_e2e,
                        "h2d_bytes_per_step": float(pcm_b * world), "d2h_bytes_per_step": float(40 * len(out[3])),
                        "phases_ms_rank0": ph_e2e,
                        "note": "every rank uploads the whole PCM from pinned host memory inside the region (features are computed redundantly per rank)"},
                "gpu_launches": int(lt[0]),
                "collectives": {"all_gather_points": {"elements": sh.get("shard_a", (0, 0, 0, 0))[3], "bytes": 16 * sh.get("shard_a", (0, 0, 0, 0))[3],
                                                     "ms_rank0": ph_dev.get("all_gather_points")},
                                "all_gather_quals": {"elements": sh.get("shard_b", (0, 0, 0, 0))[3], "bytes": 8 * sh.get("shard_b", (0, 0, 0, 0))[3],
                                                    "ms_rank0": ph_dev.get("all_gather_quals")}},
                "roofline": {"bound": "hbm", "kernel": "features_kernel", "achieved": (pcm_b + 24 * (len(lv) + len(la)) // 210) / (feat_ms * 1e-3) / 1e9 if feat_ms else None,
                             "peak": peaks["hbm_gbs"], "unit": "GB/s",
                             "frac": ((pcm_b + 24 * (len(lv) + len(la)) // 210) / (feat_ms * 1e-3) / 1e9 / peaks["hbm_gbs"]) if feat_ms else None,
                             "peak_source": peak_src, "traffic": None,
                             "note": "features phase of rank 0 (both tracks, incl. the device-to-device hand-over); the step is bounded by the two single-CTA DPs on rank 0 (latency), see phases_ms_rank0"},
                "host_fit_s_first_solve": det.get("host_fit_s"),
                "parity": single, "cpu_baseline": cpu, "clocks": clocks,
                "host_side": {"numa_binding_rank0": numa}}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def run_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from describealign_b200 import api, batch, build
    from describealign_b200 import _cabi
    build.build()
    api.set_device(local_rank)
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # The same configuration at every N: W slots (pairs on the device at once), B pairs per step cycling
    # over `distinct` synthetic pairs per GPU (generating one takes ~35 s of CPU).
    W = args.workers if args.workers > 0 else 32
    c4_total = c4_mine = None
    if args.workload == "C4":
        # batch mode (describealign.py:1077): 64 distinct episodes in all, handed to batch.align_batch, which
        # assigns them to the ranks; a step is one align_batch call over the whole batch
        c4_total = args.distinct if args.distinct > 0 else 64
        c4_mine = batch.assign_pairs([1.0] * c4_total, world)[rank]
        distinct = B = len(c4_mine)
        from concurrent.futures import ProcessPoolExecutor
        with ProcessPoolExecutor(max_workers=max(1, min(len(c4_mine), (os.cpu_count() or 1) // max(1, world)))) as ex:
            base_pairs = list(ex.map(_make_one, [(int(k), args.scale, "C4") for k in c4_mine]))
    else:
        B = args.pairs if args.pairs > 0 else 8 * W
        distinct = max(1, min(B, args.distinct if args.distinct > 0 else 4))
        base_pairs = make_pairs(distinct, rank * distinct, args.scale, world, args.workload)
    # before any page-locked buffer or engine thread exists (and after the generator's worker processes have
    # used all cores): run on, and allocate from, the GPU's own NUMA node
    numa = batch.bind_to_gpu_numa_node(local_rank) if not args.no_numa_bind else {"bound": False, "disabled": True}
    pairs = [base_pairs[k % distinct] for k in range(B)]
    hours_rank = audio_hours(pairs)

    # device-resident copies (int16 interleaved) and pinned host copies of the distinct pairs
    dev = [(torch.from_numpy(np.ascontiguousarray(v)).cuda(), torch.from_numpy(np.ascontiguousarray(a)).cuda())
           for v, a in base_pairs]
    pinned = [(torch.from_numpy(np.ascontiguousarray(v)).pin_memory(), torch.from_numpy(np.ascontiguousarray(a)).pin_memory())
              for v, a in base_pairs]
    pinned_np = [(v.numpy(), a.numpy()) for v, a in pinned]
    # what the host-to-device link gives: one large pinned copy on an idle box, and every rank copying at once
    h2d_single = h2d_all_ranks = d2h_all_ranks = None
    try:
        src = pinned[0][1]
        dst = torch.empty_like(src, device="cuda")
        best = 0.0
        for _ in range(4):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); dst.copy_(src, non_blocking=True); e1.record(); e1.synchronize()
            best = max(best, src.numel() * src.element_size() / (e0.elapsed_time(e1) * 1e-3) / 1e9)
        h2d_single = best
        del dst
        barrier()
        h2d_all_ranks = h2d_probe(pinned)
        barrier()
        d2h_all_ranks = d2h_probe(pinned)
        barrier()
    except Exception:
        pass
    ctx = api.context()
    eng = batch.engine(W)
    host_cache = {}

    def stage_b_struct_for(k, evt):
        """The rate-change fit is outside the metric (BASELINE.json); its result only depends on the pass-1
        path, so it is solved once per distinct pair (during warm-up) and reused for as long as stage A keeps
        returning that same path: inside the timed region it is a comparison of the path and a lookup."""
        x, y = eng.path1(evt)
        c = host_cache.get(k % distinct)
        if c is not None and np.array_equal(c["x"], x) and np.array_equal(c["y"], y):
            return c["struct"]
        job = api.AlignJob(detached=True)
        job.video_features = [f.copy() for f in eng.features(evt, _cabi.VIDEO)]
        job.audio_features = [f.copy() for f in eng.features(evt, _cabi.AUDIO)]
        job.check_path1_length(int(evt.n_path1))
        job.x, job.y = x.astype(np.int64), y.astype(np.int64)
        job.host_stage()
        st = eng.stage_b_struct(**job.stage_b_input())
        host_cache[k % distinct] = {"x": x.copy(), "y": y.copy(), "struct": st, "job": job}
        return st

    def c4_host_stage(job):
        c = host_cache.get(("c4", job.tag))
        if c is not None and np.array_equal(c["x"], job.x) and np.array_equal(c["y"], job.y):
            for name in ("kept_x", "kept_y", "gains", "n_audio_scaled", "n_video_scaled", "fit", "clusters", "lines"):
                setattr(job, name, c[name])
            return
        job.host_stage()
        host_cache[("c4", job.tag)] = {"x": job.x, "y": job.y, **{name: getattr(job, name) for name in
                                       ("kept_x", "kept_y", "gains", "n_audio_scaled", "n_video_scaled", "fit", "clusters", "lines")}}

    def c4_step(host_input: bool, keep=None):
        """One batch.align_batch call over the 64 episodes (every rank passes the same list; a rank only
        touches the pairs align_batch assigns to it).  keep: dict that receives the outputs of this rank's
        first DUMP_PAIRS episodes."""
        lst = [None] * c4_total
        for pos, k in enumerate(c4_mine):
            if host_input:
                lst[k] = pinned_np[pos]
            else:
                v, a = dev[pos]
                lst[k] = ((v.data_ptr(), v.shape[0], v.shape[1]), (a.data_ptr(), a.shape[0], a.shape[1]))
        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        out = batch.align_batch(lst, durations=[1.0] * c4_total, in_flight=W, gather=False,
                                host_stage=c4_host_stage, finish=False, host_workers=1)
        stop.record()
        stop.synchronize()
        results = []
        for k, job in out:
            if isinstance(job, Exception):
                raise job
            if keep is not None and len(keep) < DUMP_PAIRS:
                keep[k] = {**pair_arrays(job.x, job.y, job.video_features, job.audio_features), "path2": job.path}
            results.append({"kernel_ms": job.timings, "work": job.stats, "n_path1": len(job.x), "n_path2": len(job.path), "t_done": 0.0})
        return start.elapsed_time(stop), results

    def one_step(host_input: bool, n_pairs=None, first=0, keep=None):
        if c4_total is not None and n_pairs is None:
            return c4_step(host_input, keep)
        """n_pairs pairs through stage A -> (cached) host fit -> stage B, W on the device at a time, all
        driven by this one thread through the engine's event queue.  Returns the device time between an
        event recorded before the first submit and one recorded after the last result reached the host.
        keep: dict that receives the outputs of the first DUMP_PAIRS pairs (one per distinct input)."""
        n_pairs = B if n_pairs is None else n_pairs
        n_keep = 0 if keep is None else min(DUMP_PAIRS, distinct, n_pairs)
        results = [None] * n_pairs
        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        start.record()
        for k in range(first, first + n_pairs):
            if host_input:
                hv, ha = pinned_np[k % distinct]
                eng.submit(k, hv, ha)
            else:
                v, a = dev[k % distinct]
                eng.submit(k, (v.data_ptr(), v.shape[0], v.shape[1]), (a.data_ptr(), a.shape[0], a.shape[1]))
        done = 0
        while done < n_pairs:
            evt = eng.next(1000)
            if evt is None:
                continue
            if evt.status != 0:
                raise RuntimeError(f"pair {evt.tag} failed on the device: {eng.error(evt)}")
            k = int(evt.tag)
            if evt.kind == _cabi.EVENT_STAGE_A:
                if k - first < n_keep:
                    keep[k] = pair_arrays(*eng.path1(evt), eng.features(evt, _cabi.VIDEO), eng.features(evt, _cabi.AUDIO))
                eng.submit_b(evt.slot, struct=stage_b_struct_for(k, evt))
            else:
                if k - first < n_keep:
                    keep[k]["path2"] = eng.rows(evt).copy()
                results[k - first] = {"kernel_ms": eng.timings(evt), "work": evt.stats.as_dict(), "n_path1": int(evt.n_path1),
                                      "n_path2": int(evt.n_path2), "t_done": time.perf_counter() - t0}
                eng.release(evt.slot)
                done += 1
        stop.record()
        stop.synchronize()
        return start.elapsed_time(stop), results

    alloc0 = {}

    def run_steps(host_input, keep=None):
        for _ in range(args.warmup):
            one_step(host_input)
        barrier()
        l0 = ctx.launches()
        alloc0.update(_cabi.alloc_stats())
        total, res = 0.0, None
        for s in range(args.steps):
            ms, res = one_step(host_input, keep=keep if s == args.steps - 1 else None)
            total += ms
        barrier()
        return total / args.steps, ctx.launches() - l0, res

    # rank 0 samples the clocks of EVERY rank's GPU during the device-resident steps (one nvidia-smi process for the
    # node): the step time is the maximum over ranks, so one power-capped GPU of the box would set it
    sampler = ClockSampler(visible_gpu_ids(world))
    if rank == 0:
        sampler.start()
    cpu0, wall0 = os.times(), time.perf_counter()
    kept = {} if rank == 0 and args.dump_outputs else None
    ms_dev, launches, res_dev = run_steps(False, kept)
    cpu1, wall1 = os.times(), time.perf_counter()
    cpu_cores_busy = ((cpu1.user - cpu0.user) + (cpu1.system - cpu0.system)) / max(wall1 - wall0, 1e-9)
    alloc1 = _cabi.alloc_stats()
    alloc_before = dict(alloc0)     # the e2e steps below update the dict run_steps writes to
    clocks = sampler.stop() if rank == 0 else None
    if kept is not None:
        dump_outputs(args.dump_outputs, {f"pair{k}_{name}": arr for k in sorted(kept) for name, arr in kept[k].items()})
    sched0 = eng.counters()
    ms_e2e, _, res_e2e = run_steps(True)
    per_rank = [{"rank": rank, "ms_per_step": ms_dev, "ms_per_step_e2e": ms_e2e, "host_cores_busy": cpu_cores_busy,
                 "scheduler_ms_per_pair": float(np.mean([r["kernel_ms"]["host_in_set_pcm"] for r in res_dev]))}]
    if world > 1:
        gathered = [None] * world
        dist.all_gather_object(gathered, per_rank[0])
        per_rank = gathered
    if rank == 0:
        per_gpu = clocks.pop("per_gpu", {})
        for p_ in per_rank:
            g = per_gpu.get(p_["rank"]) or {}          # local rank = GPU index on the one node the bench runs on
            p_["sm_mhz"], p_["reasons"] = g.get("sm_mhz"), g.get("reasons")
    # bytes that crossed the link per pair in the end-to-end arm (counted from the arrays copied)
    def bytes_of(k, r):
        v, a = pinned_np[k % distinct]
        feat = sum(4 * (x.shape[0] // 210 + 1) * 3 for x in (v, a))
        return v.nbytes + a.nbytes + 16 * 32, 8 * r["n_path1"] + feat + 40 * r["n_path2"] + 2 * 128
    h2d = sum(bytes_of(k, r)[0] for k, r in enumerate(res_e2e))
    d2h = sum(bytes_of(k, r)[1] for k, r in enumerate(res_e2e))

    # one pair alone on the GPU (device-resident PCM, three passes, the last one is kept): BASELINE.json's
    # second figure, "ms per 22-min pair"
    solo = None
    if rank == 0:
        for _ in range(3):
            _, r1 = one_step(False, n_pairs=1)
        solo = r1[0]

    # parity inside the run: rank 0 checks its first pair against the oracle
    parity = None
    cpu = None
    if rank == 0 and not args.no_cpu_baseline:
        import oracle
        oracle.build()
        cpu_t, o = cpu_pass(pairs[0], keep=True)
        det = {}
        import contextlib
        with contextlib.redirect_stdout(sys.stderr):     # progress labels (describealign.py:604,635,726,860) stay off the JSON line
            nx, ny, sim, path, med = api.align_pcm(pairs[0][0], pairs[0][1], details=det)
        # the same pair through the batch engine must give the same thing as the synchronous API
        eres = batch.run_engine([pairs[0]], in_flight=W)[0]
        ox, oy = o["nodes"]
        opath = o["path"]
        same_shape = path.shape == opath.shape
        parity = {
            "features_f32_identical": bool(all(np.array_equal(det["video_features"][k], o["V"][k]) and
                                               np.array_equal(det["audio_features"][k], o["A"][k]) for k in range(4))),
            "path1_identical": bool(np.array_equal(det["path1"][0], o["path1"][0]) and np.array_equal(det["path1"][1], o["path1"][1])),
            "path2_rows": int(len(path)),
            "path2_int_identical": bool(same_shape and np.array_equal(path[:, 1], opath[:, 1]) and
                                        np.array_equal(path[:, 2], opath[:, 2]) and
                                        np.allclose(path[:, 0], opath[:, 0], rtol=0, atol=1e-9)),
            "nodes_max_abs_diff_s": float(max(np.max(np.abs(nx - ox)), np.max(np.abs(ny - oy)))) if len(nx) == len(ox) else None,
            "similarity_diff": float(abs(sim - o["similarity"])),
            "engine_equals_sync_api": bool(not isinstance(eres, Exception) and np.array_equal(eres[3], path) and
                                           np.array_equal(eres[0], nx) and np.array_equal(eres[1], ny)),
            "bench_loop_path1_is_this_path1": bool(np.array_equal(host_cache[0]["x"], det["path1"][0]) and
                                                   np.array_equal(host_cache[0]["y"], det["path1"][1])),
        }
        h1 = audio_hours(pairs[:1])
        cpu = {"value": h1 / cpu_t["hot_path_s"], "unit": UNIT, "cores": 1, "kind": "port",
               "sample": "1 full " + args.workload + " pair through the oracle port (C features, C match + DPs, numpy host stage and corridors); "
                         "timed as BASELINE.md section 3: features + align() minus scipy.optimize.linprog",
               "seconds": cpu_t["hot_path_s"], "seconds_linprog_subtracted": cpu_t["linprog_s"],
               "seconds_device_stages_only": cpu_t["device_stages_s"],
               "value_device_stages_only": h1 / cpu_t["device_stages_s"],
               "host_cpu": _cpu_model(), "host_cores": os.cpu_count()}

    # N > 1: one long pair on all ranks (match stage and corridor scoring sharded by audio rows, all-gathers
    # over NCCL, DPs and host fit on rank 0), checked against the single-GPU path on the same PCM
    long_pair = None
    if world > 1 and not args.no_long_pair:
        from describealign_b200 import synth
        lv, la = synth.config_pair("C5", 0, args.long_scale)
        barrier()
        ldet = {}
        t0 = time.perf_counter()
        lout = batch.align_long_pair(lv, la, details=ldet)
        torch.cuda.synchronize()
        t_long = time.perf_counter() - t0
        same = None
        if rank == 0:
            import contextlib
            with contextlib.redirect_stdout(sys.stderr):
                t1 = time.perf_counter()
                lref = api.align_pcm(lv, la)
                t_single = time.perf_counter() - t1
            same = bool(np.array_equal(lout[3], lref[3]) and np.array_equal(lout[0], lref[0]) and np.array_equal(lout[1], lref[1]))
            sh = ldet.get("shards", {})
            long_pair = {"workload": "C5 (2.5 h film vs 3 h description) at scale %g: %.1f + %.1f min, mono 44.1 kHz" % (
                             args.long_scale, len(lv) / 44100 / 60, len(la) / 44100 / 60),
                         "ranks": world, "identical_to_single_gpu_path": same,
                         "wall_s_all_ranks_incl_host_fit": t_long, "wall_s_single_gpu_incl_host_fit": t_single,
                         "match_points_all_gathered": sh.get("shard_a", (0, 0, 0, 0))[3],
                         "all_gather_bytes_stage_a": 16 * sh.get("shard_a", (0, 0, 0, 0))[3],
                         "quals_all_gathered": sh.get("shard_b", (0, 0, 0, 0))[3],
                         "all_gather_bytes_stage_b": 8 * sh.get("shard_b", (0, 0, 0, 0))[3],
                         "note": "the frontier DPs and the host fit do not shard (SURVEY.md 8e: replicas only); they run on rank 0"}
        barrier()

    # max over ranks
    t = torch.tensor([ms_dev, ms_e2e], device="cuda", dtype=torch.float64)
    tot = torch.tensor([hours_rank, float(launches), float(h2d), float(d2h)], device="cuda", dtype=torch.float64)
    probe = torch.tensor([h2d_all_ranks or 0.0, d2h_all_ranks or 0.0], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
        dist.all_reduce(probe, op=dist.ReduceOp.SUM)
    ms_dev, ms_e2e = float(t[0]), float(t[1])
    hours, launches_all, h2d_all, d2h_all = (float(x) for x in tot)
    h2d_probe_sum, d2h_probe_sum = float(probe[0]), float(probe[1])

    if rank == 0:
        peaks, peak_src = measured_peaks()
        timings = [r["kernel_ms"] for r in res_dev]
        stats = [r["work"] for r in res_dev]
        agg = {k: sum(tm[k] for tm in timings) for k in timings[0] if not k.startswith("host_in_")}
        sched = {"scheduler_ms_per_pair": float(np.mean([tm["host_in_set_pcm"] for tm in timings])),
                 "submit_to_stage_a_results_ms": float(np.mean([tm["host_in_stage_a"] for tm in timings])),
                 "stage_b_input_to_path_ms": float(np.mean([tm["host_in_stage_b"] for tm in timings]))}
        solo_ms = {k: v for k, v in solo["kernel_ms"].items() if not k.startswith("host_in_")}
        solo_work = solo["work"]
        clk_hz = 1e6 * float(peaks.get("sm_max_mhz", 1965.0))

        def pcm_bytes(pair_list):
            return sum(2 * (v.shape[0] * v.shape[1] + a.shape[0] * a.shape[1]) + 24 * (v.shape[0] // 210 + a.shape[0] // 210)
                       for v, a in pair_list)

        def rooflines(kernel_ms, work, pair_list):
            feat_ms = kernel_ms["features_video"] + kernel_ms["features_audio"]
            # feature kernel: algorithmic bytes = PCM read once + 24 B per output frame (SURVEY.md 8d)
            feat_bytes = pcm_bytes(pair_list)
            out = {"features": {"bound": "hbm", "achieved": feat_bytes / (feat_ms * 1e-3) / 1e9 if feat_ms > 0 else None,
                                "peak": peaks["hbm_gbs"], "unit": "GB/s", "ms": feat_ms, "launches": 2 * len(pair_list),
                                "algorithmic_bytes": feat_bytes}}
            # DP kernels: 24 B per point (i, v, qual in; back pointer out), SURVEY.md 8(d).  They are bound by
            # latency, not bandwidth: the reference point is one dependent f64 add + select per point (52 SM
            # cycles on this chip, profiles/r1_v18_dp2_block_hot_loops.txt); the scan formulation of DP 2 is not
            # held to that chain any more, so its fraction can exceed 1
            for key, npts in (("dp1_trace", work["n_points1"]), ("dp2_trace", work["n_points2"])):
                ms = kernel_ms[key]
                out[key] = {"bound": "latency", "achieved": 24 * npts / (ms * 1e-3) / 1e9 if ms > 0 else None,
                            "peak": peaks["hbm_gbs"], "unit": "GB/s", "ms": ms, "launches": len(pair_list), "points": npts,
                            "points_per_s": npts / (ms * 1e-3) if ms > 0 else None,
                            "serial_chain_ms": 1e3 * 52.0 * npts / clk_hz,
                            "speedup_over_serial_chain": (1e3 * 52.0 * npts / clk_hz) / ms if ms > 0 else None}
            for v in out.values():
                v["frac"] = v["achieved"] / v["peak"] if v.get("achieved") is not None else None
            return out

        work_all = {k: sum(st[k] for st in stats) for k in stats[0]}
        roof_load = rooflines(agg, work_all, pairs)
        roof = rooflines(solo_ms, solo_work, pairs[:1])
        # the dominant kernel of the STEP: the one with the largest share of full-GPU time.  The DPs run on one
        # CTA per pair beside everything else, so the kernel that bounds device-resident throughput is the
        # feature kernel (ncu launch list under profiles/); its roofline is the headline, the step-level
        # figure (all algorithmic bytes of a step over the step time) sits beside it.
        main_roof = dict(roof["features"])
        ncu_traffic = (116.477696e6 + 19.665920e6 + 142.943232e6 + 22.880000e6) / 2     # profiles/r2_v21_features_gate_full.txt
        step_bytes = pcm_bytes(pairs) + 24 * (work_all["n_points1"] + work_all["n_points2"])
        main_roof.update({"kernel": "features_kernel", "peak_source": peak_src,
                          "measured": "CUDA events on the pair's stream, one pair alone on the GPU right after the timed steps",
                          "traffic": ncu_traffic if args.scale == 1.0 else None,
                          "traffic_note": "bytes per launch (dram read + write), ncu --set full of one C2 pair (mono), see profiles/",
                          "step": {"bound": "hbm", "algorithmic_bytes": step_bytes, "ms": ms_dev,
                                   "achieved": step_bytes / (ms_dev * 1e-3) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                                   "frac": step_bytes / (ms_dev * 1e-3) / 1e9 / peaks["hbm_gbs"]}})
        e2e_gbs = h2d_all / world / (ms_e2e * 1e-3) / 1e9
        line = {
            "metric": METRIC, "value": hours / (ms_dev * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_dev, "higher_is_better": True,
            "scaling": "strong" if args.workload == "C4" else "weak",
            "vs_baseline": None, "dtype": "f32+f64 (u32 packed codes)", "data": "synthetic",
            "config": {"workload": WORKLOADS[args.workload], "pairs_per_gpu_per_step": B, "pairs_in_flight_per_gpu": W,
                       "distinct_pairs_per_gpu": distinct, "audio_hours_per_step": hours,
                       "l2_policy": "inputs larger than L2 (each pair streams %d MB of PCM, %d distinct pairs per GPU; 126 MB L2)" % (
                           int(sum(v.nbytes + a.nbytes for v, a in base_pairs[:1]) / 1e6), distinct),
                       "timed": "one region per step: every pair through device stage A (features, prep, tables, gate, score, DP1, traceback) and device stage B (feature scaling, corridors, DP2, traceback) incl. the result copies to the host, W pairs on the device at a time, driven by the library's scheduler thread; the host rate-change fit between the stages (describealign.py:702-893 and the corridor planning :895-930) is solved during warm-up and is a path comparison + lookup inside the region (untimed by BASELINE.json)",
                       "scale": args.scale},
            "ms_per_pair": ms_dev / B,
            "pairs_in_flight": W,
            "e2e": {"value": hours / (ms_e2e * 1e-3), "unit": UNIT, "ms_per_step": ms_e2e,
                    "h2d_bytes_per_step": h2d_all, "d2h_bytes_per_step": d2h_all,
                    "h2d_gbs_achieved_per_gpu": e2e_gbs,
                    "h2d_gbs_single_copy_idle_box": h2d_single,
                    "h2d_gbs_probe_all_ranks_at_once_per_gpu": h2d_probe_sum / world if h2d_probe_sum else None,
                    "frac_of_h2d_probe": e2e_gbs / (h2d_probe_sum / world) if h2d_probe_sum else None,
                    "d2h_gbs_probe_all_ranks_at_once_per_gpu": d2h_probe_sum / world if d2h_probe_sum else None,
                    "d2h_gbs_needed_per_gpu_device_resident": d2h_all / world / (ms_dev * 1e-3) / 1e9,
                    "note": "PCM is 2 bytes per sample per channel; the end-to-end rate is bounded by the host-to-device link (probe: every rank copying its pinned PCM back to back at the same time)"},
            "gpu_launches": int(launches_all),
            "roofline": main_roof,
            "roofline_by_kernel": roof,
            "roofline_by_kernel_under_load": roof_load,
            "kernel_ms_one_pair_alone": solo_ms,
            "ms_per_pair_alone": {"submit_to_final_path_on_host_excl_host_fit": solo["kernel_ms"]["host_in_stage_a"] + solo["kernel_ms"]["host_in_stage_b"],
                                  "kernels_only": sum(v for k, v in solo_ms.items() if k != "dp2"),
                                  "cpu_port_same_pair": 1e3 * cpu["seconds_device_stages_only"] if cpu else None,
                                  "note": "one C2 pair (22-min video, 27-min description) alone on the GPU, PCM device-resident; wall time from submit to the stage-A results on the host plus stage-B input to the final path on the host"},
            "kernel_ms_last_step": agg,
            "host_side": {"numa_binding_rank0": numa, **sched, **{k: eng.counters()[k] - sched0[k] for k in sched0},
                          "python_threads": 1, "scheduler_threads": 1, "host_cores_busy_rank0": cpu_cores_busy,
                          "host_cores_per_rank": (os.cpu_count() or 1) / world},
            "allocator_activity_in_timed_steps": {k: alloc1[k] - alloc_before[k] for k in alloc1},
            "work": work_all,
            "clocks": clocks,
            "per_rank": per_rank,
            "cpu_baseline": cpu,
            "parity": parity,
            "long_pair": long_pair,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def _cpu_model():
    try:
        with open("/proc/cpuinfo") as f:
            for ln in f:
                if ln.startswith("model name"):
                    return ln.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    elif args.workload == "C5":
        run_long(args, rank, world, local_rank)
    else:
        run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
