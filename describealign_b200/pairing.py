"""Cross-match a batch: which description belongs to which video.

The reference pairs a video directory with a description directory by sorted file name (`combine()`,
describealign.py:1033-1046); a wrong pairing ("Ep 10" sorting before "Ep 2", a missing episode, a director's cut
next to the theatrical cut) shows only after a full alignment, as "Alignment failed, are the input files
mismatched?".  Its own first accept/reject test is stage A: the pass-1 path must be at least
`min_path_length` long (:698-699).  Here that test runs for every (video, description) combination:

* features are computed once per track;
* the video side of stage A (prep, codes, hashed-frame list, hash tables) is built once per video into a
  read-only index (dab_index_build), shared by every description;
* each combination then costs the description's prep, the gate, the scoring, DP 1 and the traceback
  (dab_pair_stage_a_against), with only the 128-byte counts coming back;
* `in_flight` pairs, each on its own stream and host thread, run at once.

`assign` turns the matrix into a one-to-one pairing that maximises the total pass-1 path length over passing
cells, and says where it disagrees with the name order.  `python -m describealign_b200.pairing VIDEOS
DESCRIPTIONS` does both for two directories (or files) of media.
"""
from __future__ import annotations

import math
import os
import sys
import threading
import time
from concurrent.futures import ThreadPoolExecutor
from dataclasses import dataclass, field

import numpy as np

from . import _cabi, api, host_fit
from ._cabi import AUDIO, VIDEO

# what a track's cells report instead of failing the batch: a track too short for stage A, a failed decode
_TRACK_ERRORS = (_cabi.DabError, ValueError, TypeError, ChildProcessError)


@dataclass
class CrossMatch:
    """Stage-A counts of every (video v, description d) combination; -1 where the cell has an error."""
    points: np.ndarray         # (V, D) pass-1 match points
    path1: np.ndarray          # (V, D) pass-1 path length
    min_len: np.ndarray        # (V, D) shortest accepted path, rounded up (host_fit.min_path_length)
    candidates: np.ndarray     # (V, D) gate candidates
    passes: np.ndarray         # (V, D) bool: path1 >= min_len, the reference's stage-A rule
    errors: np.ndarray         # (V, D) object: None, or why the cell has no result
    seconds: dict = field(default_factory=dict)   # wall time: "index" (features + index build), "cells"


def _load(pair, track: int, pcm):
    """PCM in any form the API takes: int16 (S, ch), the reference's float16 (ch, S), or a decode.DevicePcm."""
    if hasattr(pcm, "device") and hasattr(pcm, "features"):
        pair.set_pcm_device(track, *pcm.device())
    else:
        pair.set_pcm(track, api.host_pcm(pcm))
    return pair.feature_lens(track)[0]      # energy length (min_path_length)


def cross_match(videos, descriptions, in_flight: int = 32) -> CrossMatch:
    """Stage A of every combination of `videos` x `descriptions` on this process's GPU."""
    nv, nd = len(videos), len(descriptions)
    if in_flight < 1:
        raise ValueError("in_flight must be >= 1")
    out = CrossMatch(points=np.full((nv, nd), -1, np.int64), path1=np.full((nv, nd), -1, np.int64),
                     min_len=np.full((nv, nd), -1, np.int64), candidates=np.full((nv, nd), -1, np.int64),
                     passes=np.zeros((nv, nd), bool), errors=np.full((nv, nd), None, object))
    tls = threading.local()
    made = []
    lock = threading.Lock()

    def worker_pair():
        pair = getattr(tls, "pair", None)
        if pair is None:
            pair = tls.pair = _cabi.Pair(api.context())
            with lock:
                made.append(pair)
        return pair

    indices = [None] * nv
    v_len = [0] * nv

    def build(v):
        pair = worker_pair()
        try:
            v_len[v] = _load(pair, VIDEO, videos[v])
            indices[v] = _cabi.Index(pair)
        except _TRACK_ERRORS as exc:
            out.errors[v, :] = f"video {v}: {exc}"

    def column(d):
        pair = worker_pair()
        try:
            a_len = _load(pair, AUDIO, descriptions[d])
        except _TRACK_ERRORS as exc:
            for v in range(nv):
                if indices[v] is not None:
                    out.errors[v, d] = f"description {d}: {exc}"
            return
        for v in range(nv):
            if indices[v] is None:
                continue
            try:
                n_points, n_path = pair.stage_a_against(indices[v])
            except _cabi.DabError as exc:
                out.errors[v, d] = f"description {d}: {exc}"
                continue
            out.points[v, d], out.path1[v, d] = n_points, n_path
            out.candidates[v, d] = pair.stats()["n_candidates"]
            out.min_len[v, d] = math.ceil(host_fit.min_path_length(v_len[v], a_len))
            out.passes[v, d] = n_path >= out.min_len[v, d]

    try:
        with ThreadPoolExecutor(max_workers=in_flight) as ex:
            t0 = time.perf_counter()
            list(ex.map(build, range(nv)))
            t1 = time.perf_counter()
            list(ex.map(column, range(nd)))
            t2 = time.perf_counter()
        out.seconds = {"index": t1 - t0, "cells": t2 - t1}
    finally:
        for ix in indices:
            if ix is not None:
                ix.free()
        for pair in made:
            pair.close()
    return out


@dataclass
class Assignment:
    pairs: list                     # [(video, description)] one-to-one, every cell passing
    unmatched_videos: list
    unmatched_descriptions: list
    disagreements: list             # [(k, suggested description of video k or None)] where name order pairs k with k


def assign(result: CrossMatch) -> Assignment:
    """The one-to-one pairing that maximises the total pass-1 path length over passing cells
    (scipy.optimize.linear_sum_assignment), and where it differs from the name order (video k with
    description k, as the reference pairs sorted file names)."""
    from scipy.optimize import linear_sum_assignment
    passes = np.asarray(result.passes, bool)
    nv, nd = passes.shape
    weight = np.where(passes, np.asarray(result.path1, np.int64), 0)
    rows, cols = linear_sum_assignment(weight, maximize=True)
    pairs = sorted((int(v), int(d)) for v, d in zip(rows, cols) if passes[v, d])
    of_video = dict(pairs)
    matched_d = {d for _, d in pairs}
    disagreements = [(k, of_video.get(k)) for k in range(min(nv, nd)) if of_video.get(k) != k]
    disagreements += [(v, d) for v, d in pairs if v >= nd]
    return Assignment(pairs=pairs, unmatched_videos=[v for v in range(nv) if v not in of_video],
                      unmatched_descriptions=[d for d in range(nd) if d not in matched_d],
                      disagreements=disagreements)


# ---------------------------------------------------------------------------------------------
# command line
# ---------------------------------------------------------------------------------------------
def list_files(path: str):
    """A directory gives its files, a file gives itself, in natural order (natsort) where available.
    Returns (files, used_natsort)."""
    files = [os.path.join(path, f) for f in os.listdir(path)] if os.path.isdir(path) else [path]
    files = [f for f in files if os.path.isfile(f)]
    try:
        from natsort import natsorted
    except ImportError:
        return sorted(files), False
    return natsorted(files), True


def format_report(videos, descriptions, result: CrossMatch, pick: Assignment) -> str:
    name = os.path.basename
    lines = ["pass-1 path length / minimum (* passes)"]
    width = max(12, *(len(name(d)) for d in descriptions)) if descriptions else 12
    lines.append(" " * 4 + "".join(f"  d{d:<{width - 1}}" for d in range(len(descriptions))))
    for v in range(len(videos)):
        cells = []
        for d in range(len(descriptions)):
            if result.errors[v, d] is not None:
                cells.append("error")
            else:
                cells.append(f"{result.path1[v, d]}/{result.min_len[v, d]}{'*' if result.passes[v, d] else ''}")
        lines.append(f"v{v:<3}" + "".join(f"  {c:<{width}}" for c in cells))
    lines.append("")
    for k, f in enumerate(videos):
        lines.append(f"v{k}: {f}")
    for k, f in enumerate(descriptions):
        lines.append(f"d{k}: {f}")
    errs = sorted({e for e in result.errors.ravel() if e is not None})
    if errs:
        lines.append("")
        lines += [f"error: {e}" for e in errs]
    lines.append("")
    lines.append("suggested pairs:")
    lines += [f"  {name(videos[v])}  <->  {name(descriptions[d])}  (path {result.path1[v, d]})" for v, d in pick.pairs]
    lines += [f"  {name(videos[v])}  <->  (no description passes)" for v in pick.unmatched_videos]
    lines += [f"  (no video)  <->  {name(descriptions[d])}" for d in pick.unmatched_descriptions]
    lines.append("")
    if not pick.disagreements:
        lines.append("the name order agrees with the suggested pairs")
    else:
        lines.append("the name order disagrees:")
        for k, d in pick.disagreements:
            by_name = name(descriptions[k]) if k < len(descriptions) else "(none)"
            lines.append(f"  {name(videos[k])}: by name {by_name}, by audio "
                         f"{name(descriptions[d]) if d is not None else '(none)'}")
    return "\n".join(lines)


def main(argv=None) -> int:
    import argparse
    ap = argparse.ArgumentParser(prog="python -m describealign_b200.pairing",
                                 description="Cross-match videos and audio descriptions by stage A on the GPU.")
    ap.add_argument("videos", help="a video file or a directory of them")
    ap.add_argument("descriptions", help="an audio description file or a directory of them")
    ap.add_argument("--in-flight", type=int, default=32)
    ap.add_argument("--ffmpeg", default="ffmpeg")
    args = ap.parse_args(argv)
    videos, nat_v = list_files(args.videos)
    descriptions, nat_d = list_files(args.descriptions)
    if not (nat_v and nat_d):
        print("natsort is not installed: files are in sorted() order, not natural order ('Ep 10' before 'Ep 2')")
    if not videos or not descriptions:
        print("no files found")
        return 1
    from . import decode
    # mono, as the reference's default mode decodes (num_channels=1)
    v_pcm = [decode.parse_audio_from_file(f, 1, args.ffmpeg) for f in videos]
    d_pcm = [decode.parse_audio_from_file(f, 1, args.ffmpeg) for f in descriptions]
    try:
        result = cross_match(v_pcm, d_pcm, in_flight=args.in_flight)
    finally:
        for p in v_pcm + d_pcm:
            p.close()
    print(format_report(videos, descriptions, result, assign(result)))
    return 0


if __name__ == "__main__":
    sys.exit(main())
