#!/usr/bin/env python
"""Time the cross-match of a batch (describealign_b200.pairing.cross_match) on one GPU.

    python tools/bench_pairing.py [--sizes 16,64] [--minutes 45] [--repeats 3] [--out FILE]

N videos x N descriptions of C4 shape (a 45-min episode and its description, synth.config_pair("C4") with
distinct seeds), so the diagonal matches and every other cell is a mismatch - the common case of a batch.  The
tracks are generated on the host's cores, moved to the GPU as they arrive and handed to cross_match as
device-resident PCM, so the timed region holds no synthesis and no host -> device copy.  Per run: total seconds,
ms per cell, and the split between the index phase (features + index build, per video) and the cell phase
(description features + stage A against the indices).  SM clocks are sampled during the runs (bench.py's
sampler); the GPU's name and power limit are recorded next to the numbers.  Prints one JSON object.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _make(arg):
    seed, minutes = arg
    from describealign_b200 import synth
    return synth.config_pair("C4", seed, minutes / 45.0)


class DeviceTrack:
    """Mono int16 samples in HBM, in the shape cross_match takes device PCM (decode.DevicePcm's)."""
    features = None

    def __init__(self, pcm):
        import torch
        self.t = torch.from_numpy(np.ascontiguousarray(pcm[:, 0])).cuda()

    def device(self):
        return (self.t.data_ptr(), self.t.numel(), 1)


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    try:
        r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits"], capture_output=True,
                           text=True, timeout=30)
        name, power, clk = [x.strip() for x in r.stdout.strip().splitlines()[0].split(",")]
        return {"name": name, "power_limit_w": float(power), "sm_max_mhz": float(clk)}
    except Exception as exc:
        return {"error": str(exc)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="16,64")
    ap.add_argument("--minutes", type=float, default=45.0)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--in-flight", type=int, default=32)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    sizes = [int(s) for s in args.sizes.split(",")]
    import torch
    from concurrent.futures import ProcessPoolExecutor
    from bench import ClockSampler, visible_gpu_ids
    from describealign_b200 import build, pairing
    build.build()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this benchmark only runs on the GPU")
    n = max(sizes)
    t0 = time.perf_counter()
    videos, descriptions = [], []
    with ProcessPoolExecutor(max_workers=max(1, min(n, os.cpu_count() or 1))) as ex:
        for v, a in ex.map(_make, [(1000 + k, args.minutes) for k in range(n)]):
            videos.append(DeviceTrack(v))
            descriptions.append(DeviceTrack(a))
    torch.cuda.synchronize()
    t_gen = time.perf_counter() - t0
    out = {"workload": f"C4-shaped pairs ({args.minutes:g}-min video, its description), N x N, diagonal matching",
           "gpu": gpu_info(), "host_cores": os.cpu_count(), "generate_s": round(t_gen, 1),
           "in_flight": args.in_flight, "runs": {}}
    # warm-up: module load, allocator pools, pinned staging
    pairing.cross_match(videos[:2], descriptions[:2], in_flight=2)
    sampler = ClockSampler(visible_gpu_ids(1))
    sampler.start()
    for size in sizes:
        runs = []
        for _ in range(args.repeats):
            t = time.perf_counter()
            res = pairing.cross_match(videos[:size], descriptions[:size], in_flight=args.in_flight)
            total = time.perf_counter() - t
            pick = pairing.assign(res)
            runs.append({"total_s": total, "index_s": res.seconds["index"], "cells_s": res.seconds["cells"],
                         "ms_per_cell": 1e3 * total / size ** 2,
                         "index_ms_per_video": 1e3 * res.seconds["index"] / size,
                         "cells_ms_per_cell": 1e3 * res.seconds["cells"] / size ** 2,
                         "errors": int(sum(e is not None for e in res.errors.ravel())),
                         "passing_cells": int(res.passes.sum()),
                         "diagonal_recovered": pick.pairs == [(k, k) for k in range(size)]})
        med = {k: float(np.median([r[k] for r in runs])) for k in runs[0] if k.endswith("_s") or "ms" in k}
        spread = {k: [round(min(r[k] for r in runs), 4), round(max(r[k] for r in runs), 4)] for k in med}
        out["runs"][f"{size}x{size}"] = {"median": med, "min_max": spread, "per_run": runs}
    out["clocks"] = sampler.stop()
    out["clocks"].pop("per_gpu", None)
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
