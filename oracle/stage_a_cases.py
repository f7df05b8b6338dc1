"""TEST INFRASTRUCTURE ONLY - deterministic stage-A inputs at the edges where the match stage and DP 1 go wrong.

Match-stage inputs (repeated material: every repeat matches every other one)
  m1_periodic     features of period 6 frames: 128 expanded entries for most hashed video frames, all match
                  points at qual 50 (mass ties for DP 1)
  m2_tone         a sample-exact 1050 Hz tone at the head of both tracks: every tone frame is bit-identical
  m3_loop         a 6 s noise segment repeated sample-exactly in the video, carried by the description at an
                  offset under narration

DP 1 point sets (i, v, q), sorted by (i, v), v = 4 * rank (the hashed frames of a video whose energy is 1.0
everywhere), quals in [0.046, 50]
  f1_*            one chain summed by the speculative run sum, one by tree queries, bit-equal sums
  f2_rounding     every add of a stretch of the chain is an exact rounding tie; runs straddle warp batches
  f3_tree         more than 32^3 ranks; predecessors found at each level of the 32-ary tree
  f4_*            sizes around 32, paths of 255 to 513 points, a path that leaves the top's chain, one large set
  f5_limit        the largest video the DP tree takes (2^20 hashed-frame slots), and one frame more
  f6_*            paths placed on the traceback's chunks of 1024 point ids: predecessors across chunk
                  boundaries, skipped chunks, an end alone in the last chunk, a late first point, one point

Each F builder returns a dict with i, v, q (int32, int32, float64), Le (video length in frames whose hashed
frames are 4 * arange), Lv (bound on v for ao.dp1) and what the tests check about it.
"""
from __future__ import annotations

import numpy as np

SR = 44100
FRAME = 210
DP_TREE_SLOTS = 1 << 20          # 32^4 leaves of the 4-level DP tree


def stage_a_caps(video_energy_len: int, audio_energy_len: int):
    """First capacity guess of the match stage for these track lengths: (table entries, candidates)."""
    vsel_ub = (video_energy_len - 41 + 3) // 4 + 1
    return 80 * vsel_ub + 4096, 2 * (audio_energy_len - 41) + 4096


def vsel_ub(video_energy_len: int) -> int:
    """Upper bound on the hashed video frames that sizes the DP tree (from the energy length, not the count)."""
    return (video_energy_len - 41 + 3) // 4 + 1


def expanded_entries(v_flags, v_sel) -> int:
    """Entries of the five video hash tables: 2^(flagged digits) per hashed frame and table."""
    return int(sum(np.sum(1 << np.unpackbits(np.asarray(fl)[v_sel][:, None], axis=1).sum(axis=1)) for fl in v_flags))


# ------------------------------------------------------------------------------------------
# match-stage inputs
# ------------------------------------------------------------------------------------------

M1_PATTERN = np.array([0.19, -0.32, -0.22, 0.78, -0.55, 0.25])


def m1_periodic(n: int = 600):
    """Features of both tracks (identical): all five features repeat every 6 frames, so the 7 digit positions
    t + 2 + 6k of a frame see one value.  With this pattern nearly every hashed video frame has all 7 digits
    flagged (128 expanded entries per table), every audio frame finds its phase in every hashed frame, and
    every candidate scores qual 50.  Energy is 1 +- 0.16, above the 0.5 gate."""
    f = np.tile(M1_PATTERN, n // 6 + 2)
    feats = [(1.0 + 0.2 * f[:n + 1]).astype(np.float32)] + [f[:n].astype(np.float32)] * 3 + [f[:n].astype(np.float64)]
    return feats, [x.copy() for x in feats]


def tone(n: int) -> np.ndarray:
    """round(3000 sin(2 pi n / 42)): period 42 samples, so every 210-sample frame is bit-identical."""
    return np.round(3000.0 * np.sin(2.0 * np.pi * np.arange(n) / 42.0)).astype(np.int16)


def m2_tone(tone_s: float, video_s: float = 100.0, offset_s: float = 5.0, seed: int = 7):
    """synth.make_pair(video_s, offset_s, seed) with the tone written over the first tone_s seconds of both tracks
    (sample-exact, from sample 0 of each)."""
    from describealign_b200 import synth
    v, a = synth.make_pair(video_s, offset_s, seed=seed)
    n = int(round(tone_s * SR))
    v, a = v.copy(), a.copy()
    v[:n, 0] = tone(n)
    a[:n, 0] = tone(n)
    return v, a


def m2a_tone():
    """15 s tone: about 49 times the first candidate guess (fits after six doublings)."""
    return m2_tone(15.0)


def m2b_tone():
    """30 s tone: about 200 times the first candidate guess, more than doubling reaches in 8 runs."""
    return m2_tone(30.0)


def m3_loop(video_s: float = 95.0, offset_s: float = 5.0, loop_at: float = 2.0, loop_s: float = 6.0, reps: int = 15,
            seed: int = 31):
    """Video: synth programme audio with a 6 s noise segment repeated `reps` times sample-exactly from loop_at.
    Description: an independent intro of offset_s, then the video audio, with synth's gated narration over it."""
    from describealign_b200 import synth
    v, d = synth.make_pair(video_s, offset_s, seed=seed, narration_frac=0)
    rng = np.random.default_rng(np.random.PCG64(seed + 1))
    seg = synth._to_int16(synth._programme(rng, int(round(loop_s * SR))))
    s0, n = int(round(loop_at * SR)), len(seg)
    assert s0 + reps * n <= len(v)
    v = v.copy()
    for r in range(reps):
        v[s0 + r * n:s0 + (r + 1) * n, 0] = seg
    off = int(round(offset_s * SR))
    body = np.concatenate([d[:off, 0].astype(np.float64), v[:, 0].astype(np.float64)])
    gate = np.clip((synth._smooth_unit_noise(rng, len(body), 44100, 3) - 0.5244) * 4.0, 0.0, 1.0)
    voice = synth._programme(rng, len(body)) * 1.6
    a = synth._to_int16(body + gate * voice)[:, None]
    return v, a


# ------------------------------------------------------------------------------------------
# DP 1 point sets
# ------------------------------------------------------------------------------------------

def _case(i, r, q, n_ranks, **extra):
    i = np.asarray(i, np.int64); r = np.asarray(r, np.int64); q = np.asarray(q, np.float64)
    order = np.lexsort((r, i))
    i, r, q = i[order], r[order], q[order]
    assert len(i) == 0 or np.all((np.diff(i) > 0) | ((np.diff(i) == 0) & (np.diff(r) > 0))), "(i, rank) not unique"
    assert np.all((q >= 0.046) & (q <= 50.0))
    assert len(r) == 0 or (r.min() >= 0 and r.max() < n_ranks)
    Le = 4 * n_ranks + 41
    out = dict(i=i.astype(np.int32), v=(4 * r).astype(np.int32), q=q, Le=Le, Lv=4 * n_ranks + 4)
    out.update(extra)
    return out


def _dyadic_quals(rng, n):
    """Quals that are multiples of 2^-10: every float64 add of them is exact, so the speculative run sum of
    dp1_kernel passes its check and is used."""
    return np.round(rng.uniform(0.05, 50.0, n) * 1024.0) / 1024.0


def f1_fast_vs_tree(m: int = 300, seed: int = 1):
    """Chain A: rows 0..m-1, ranks RA + k, one run (summed by the warp prefix sum after its first batch).
    Chain B: rows m..2m-1, ranks RB + k < RA, each point left of the top (A's end), so every cum is one tree
    query and one add.  Same quals, so cum(A end) == cum(B end) bit for bit.  B's end ties with the top and
    takes it (smaller rank); the final point right of both extends the top: path = B + final."""
    rng = np.random.default_rng(seed)
    q = _dyadic_quals(rng, m)
    RA, RB = 2000, 1000
    i = list(range(m)) + list(range(m, 2 * m)) + [2 * m]
    r = [RA + k for k in range(m)] + [RB + k for k in range(m)] + [RA + m + 5]
    qq = list(q) + list(q) + [1.0]
    return _case(i, r, qq, 4096, chain_a=np.arange(m), chain_b=np.arange(m, 2 * m), final=2 * m,
                 want_path_ranks=[RB + k for k in range(m)] + [RA + m + 5])


def f1_mirror(m: int = 300, seed: int = 2):
    """f1_fast_vs_tree with the tie decided by the warp arg-max instead of the top update: a far-right point D
    (rows after both chains) becomes the top, then the final point lies between the chains' ends and D, so its
    predecessor is a tree query that sees A's end (a level-1 node) and B's end (a level-2 node, another lane)
    with equal cums: it must take B's (smaller rank)."""
    rng = np.random.default_rng(seed)
    q = _dyadic_quals(rng, m)
    RA, RB = 2000, 1000
    i = list(range(m)) + list(range(m, 2 * m)) + [2 * m, 2 * m + 1]
    r = [RA + k for k in range(m)] + [RB + k for k in range(m)] + [RA + m + 400, RA + m + 10]
    qq = list(q) + list(q) + [0.5, 2.0]
    return _case(i, r, qq, 4096, chain_a=np.arange(m), chain_b=np.arange(m, 2 * m), final=2 * m + 1,
                 want_path_ranks=[RB + k for k in range(m)] + [RA + m + 10])


F2_RUN_STARTS = (30, 31, 0, 1)


def f2_rounding(competitor: str = "tie", n_batches: int = 24, seed: int = 3):
    """Chain A from the seed (its first run starts at top_cum == 0) with quals 40 + (2j + 1) 2^-39 and
    40 + (4j + 1) 2^-40 in turn.  Below 2^13 every add is exact.  While the cum is in [2^13, 2^14) its unit u is
    2^-39: the first kind of add is exact and leaves an odd multiple of u, the second is an exact halfway case that
    round-to-even then resolves upwards, while the qual rounded to u alone (what the speculative run sum adds up)
    rounds downwards: the speculative sum falls one u short per pair, so dp1_kernel must take the serial sum.
    (Halfway adds alone do not show this: after one of them the sum is an even multiple of u, and rounding the
    qual alone then agrees with the serial add.)  The chain crosses 2^14 inside a run.  One noise point per warp batch of 32 points (a tree query: left of the top) ends
    A's run, so that the next run starts at offsets 30, 31, 0, 1 mod 32 in turn.
    The path only shows a cum that is off by an ulp when a tie depends on it: chain B (rows after A, ranks below
    everything, tree queries, serial adds) ends on A's exact serial sum ("tie": B wins on its smaller rank) or one
    ulp below it ("below": A wins), and a final point right of both extends the winner."""
    rng = np.random.default_rng(seed)
    pts = []                          # (rank, qual, is_chain)
    noise_rank, chain_rank = 50000, 100000
    total = 32 * n_batches
    noise_at = set()
    for b in range(n_batches):
        start = F2_RUN_STARTS[b % 4]
        noise_at.add(32 * b + start - 1 if start > 0 else 32 * b - 1)
    noise_at.discard(-1)
    for p in range(total):
        if p in noise_at:
            pts.append((noise_rank, float(rng.uniform(0.046, 1.0)), False))
            noise_rank += 1
        else:
            # alternately an exact add that leaves the sum an odd multiple of 2^-39, and a halfway add
            # (odd = 1 mod 4, so that round-to-even of the sum rounds up where rounding the qual alone rounds down)
            j = int(rng.integers(0, 1 << 28))
            half = (chain_rank - 100000) % 2 == 1
            pts.append((chain_rank, 40.0 + ((4 * j + 1) * 2.0 ** -40 if half else (2 * j + 1) * 2.0 ** -39), True))
            chain_rank += 1
    i = list(range(total))
    r = [p[0] for p in pts]
    q = [p[1] for p in pts]
    chain = np.array([k for k, p in enumerate(pts) if p[2]])
    qa = [q[k] for k in chain]
    qb = list(qa)
    if competitor == "below":
        c = 0.0
        for x in qa[:-1]:
            c = c + x
        s = c + qa[-1]
        qb[-1] = float(np.nextafter(s, 0.0)) - c            # exact: both are multiples of the unit of [2^14, 2^15)
        assert c + qb[-1] == np.nextafter(s, 0.0)
    m = len(qa)
    i += list(range(total, total + m)) + [total + m]
    r += [1000 + k for k in range(m)] + [chain_rank + 5]
    q += qb + [1.0]
    chain_b = np.arange(total, total + m)
    return _case(i, r, q, chain_rank + 32, chain=chain, chain_b=chain_b, final=total + m,
                 noise_at=np.array(sorted(noise_at)), competitor=competitor)


def f3_tree(n_random: int = 4000, seed: int = 4):
    """Over 32^3 ranks (40 000 hashed frames).  In order:
    E2 (rank 34000) then E1 (rank 700): equal cums in different level-3 blocks;
    chain C (ranks 36000.., qual 50): the top, far above everything that follows;
    QE (rank 35900): its tree query sees E1 at level 3 (lane 0) and E2 at level 2 (lane 1), equal cums;
    X3 / J3: J3's predecessor is X3 in a level-3 block to the left; X2 / J2 and X1 / J1 the same at levels 2 and 1;
    S, S': the same rank in consecutive rows (tree queries);
    L: left of the top inside the top's own level-0 block;
    then C continues (runs), then random points over all ranks."""
    rng = np.random.default_rng(seed)
    i, r, q = [], [], []

    def add(row, rank, qual):
        i.append(row); r.append(rank); q.append(qual)
        return len(i) - 1
    row = 0
    e2 = add(row, 34000, 7.0); row += 1
    e1 = add(row, 700, 7.0); row += 1
    for k in range(100):
        add(row, 36000 + k, 50.0); row += 1
    qe = add(row, 35900, 1.0); row += 1
    x3 = add(row, 100, 20.0); row += 1
    j3 = add(row, 32800, 1.0); row += 1
    x2 = add(row, 33000, 20.0); row += 1
    j2 = add(row, 34200, 1.0); row += 1
    x1 = add(row, 34300, 20.0); row += 1
    j1 = add(row, 34400, 1.0); row += 1
    s1 = add(row, 20000, 0.5); row += 1
    s2 = add(row, 20000, 0.5); row += 1
    lt = add(row, 36097, 0.25); row += 1
    for k in range(100, 400):
        add(row, 36000 + k, float(rng.choice([0.25, 1.0, 50.0]))); row += 1
    rows = row + np.sort(rng.integers(0, n_random // 3, n_random))
    ranks = rng.integers(0, 40000, n_random)
    quals = rng.choice([0.25, 0.5, 1.0, 2.0, 50.0], n_random)
    seen = set(zip(i, r))
    for a, b, c in zip(rows.tolist(), ranks.tolist(), quals.tolist()):
        if (a, b) not in seen:
            seen.add((a, b)); add(a, b, c)
    marks = dict(e1=e1, e2=e2, qe=qe, x3=x3, j3=j3, x2=x2, j2=j2, x1=x1, j1=j1, s1=s1, s2=s2, lt=lt)
    return _case(i, r, q, 40000, marks=marks)


def f4_small(n: int, seed: int = 5):
    """n points over 64 rows and 200 ranks, quals mixed from a few values and a uniform draw."""
    rng = np.random.default_rng(seed + n)
    cells = rng.choice(64 * 200, size=n, replace=False)
    i, r = cells // 200, cells % 200
    q = np.where(rng.uniform(size=n) < 0.5, rng.choice([0.25, 1.0, 50.0], n), rng.uniform(0.046, 50.0, n))
    return _case(i, r, q, 256)


F4_SIZES = (0, 1, 31, 32, 33, 63, 64, 65)
F4_PATHS = (255, 256, 257, 511, 512, 513)


def f4_path(length: int, seed: int = 6):
    """A chain of exactly `length` points (rows 0.., ranks 100.., qual 1), with low-rank noise points in later
    rows whose cums stay below the chain's: the path is the chain."""
    rng = np.random.default_rng(seed + length)
    i = list(range(length)); r = [100 + k for k in range(length)]; q = [1.0] * length
    n_noise = length // 3
    nrows = np.sort(rng.choice(np.arange(1, length), size=n_noise, replace=False))
    for k, row in enumerate(nrows.tolist()):
        i.append(row); r.append(k % 90); q.append(0.05)
    return _case(i, r, q, 100 + length + 32, want_len=length)


def f4_superseded(seed: int = 7):
    """Chain M (rows 0..599, ranks 1000 + 2k, qual 1) is the top for 600 points; then branch B (rows 600..1199,
    ranks 1201.., qual 2) leaves M at its point 100 and overtakes it.  The path is M[0..100] + B: the back records
    of M's points 101..599 stay written but are no longer on the path."""
    i = list(range(600)) + list(range(600, 1200))
    r = [1000 + 2 * k for k in range(600)] + [1201 + k for k in range(600)]
    q = [1.0] * 600 + [2.0] * 600
    return _case(i, r, q, 2300, want_len=101 + 600)


def f4_large(n: int = 2_000_000, n_ranks: int = 150_000, seed: int = 8):
    """2e6 points over 150 000 ranks: a noisy diagonal (the true alignment, with gaps and backward jumps) in a
    field of false matches; quals mixed from {0.25, 0.5, 1, 2, 50} and a uniform draw."""
    rng = np.random.default_rng(seed)
    n_rows = 600_000
    n_diag = n // 4
    di = np.sort(rng.choice(n_rows, size=n_diag, replace=False))
    dr = np.clip((di * (n_ranks / n_rows) + rng.normal(0, 3, n_diag)).astype(np.int64), 0, n_ranks - 1)
    fi = rng.integers(0, n_rows, int(n * 0.8))
    fr = rng.integers(0, n_ranks, int(n * 0.8))
    i = np.concatenate([di, fi]); r = np.concatenate([dr, fr])
    key = np.unique(i * n_ranks + r)[:n]
    i, r = key // n_ranks, key % n_ranks
    m = len(i)
    q = np.where(rng.uniform(size=m) < 0.5, rng.choice([0.25, 0.5, 1.0, 2.0, 50.0], m), rng.uniform(0.046, 50.0, m))
    return _case(i, r, q, n_ranks)


def f5_limit(over: bool = False, seed: int = 9):
    """The largest video length Le with vsel_ub(Le) <= 2^20 (the DP tree's leaves), or one frame more.  At the
    limit the hashed frames are ceil((Le - 41) / 4) = 2^20 - 1, so the top rank is 2^20 - 2: points sit on it,
    on ranks at the ends of level-3 blocks, and on a chain that climbs to the top rank."""
    rng = np.random.default_rng(seed)
    Le = 4 * DP_TREE_SLOTS + 37          # (Le - 38) // 4 + 1 == 2^20
    if over:
        Le += 1
    n_sel = (Le - 41 + 3) // 4
    top = n_sel - 1
    i, r, q = [], [], []
    ranks = sorted(set([0, 31, 32, 1023, 1024, 32767, 32768] + [(b << 15) - 1 for b in range(1, 32)] +
                       rng.integers(0, top, 200).tolist()))
    for k, rk in enumerate(rng.permutation(ranks).tolist()):
        i.append(k); r.append(rk); q.append(float(rng.choice([0.25, 1.0, 50.0])))
    base = len(ranks)
    for k in range(300):
        i.append(base + k); r.append(top - 299 + k); q.append(2.0)
    i.append(base + 300); r.append(top); q.append(50.0)
    i.append(base + 301); r.append(top); q.append(1.0)
    out = _case(i, r, q, n_sel, top_rank=top)
    out["Le"] = Le
    out["Lv"] = 4 * n_sel + 4
    return out


TB_CHUNK = 1024                  # point ids per chunk of the traceback


def f6_chunks(path_ids, n: int):
    """n points, one per row, so a point's id is its row.  The points at path_ids (ascending) form the path: ranks
    R, R + 1, ..., qual 1.  Every other point has qual 0.05 and cannot be a predecessor of a path point: before the
    first path point the ranks lie above the path's, after it below, and both kinds fall with the id, so each noise
    point chains from the seed (cum 0.05) and the path's cums 1, 2, ... win every comparison."""
    path_ids = sorted(path_ids)
    assert path_ids and path_ids[-1] < n
    on_path = set(path_ids)
    n_high = sum(1 for p in range(path_ids[0]) if p not in on_path)
    n_low = n - len(path_ids) - n_high
    R, L = n_low, len(path_ids)
    high, low = iter(range(R + L + n_high - 1, R + L - 1, -1)), iter(range(R - 1, -1, -1))
    r, q, k = [], [], 0
    for p in range(n):
        if p in on_path:
            r.append(R + k); q.append(1.0); k += 1
        else:
            r.append(next(high) if p < path_ids[0] else next(low)); q.append(0.05)
    return _case(np.arange(n), r, q, R + L + n_high, path_ids=np.array(path_ids))


F6_CASES = {
    "f6_across": lambda: f6_chunks([5, 700, 1023, 1024, 1500, 2047, 2048, 2600], 3000),   # preds 1023 -> 1024, 2047 -> 2048
    "f6_skip": lambda: f6_chunks([10, 500, 4200, 4201, 6000], 6200),                    # chunks 1-3 and 6 not visited
    "f6_end_alone": lambda: f6_chunks([3, 1030, 2000, 2048], 2049),                      # the last chunk is the end point
    "f6_late_start": lambda: f6_chunks([1024, 1025, 2100, 3000], 3100),                  # nothing on chunk 0
    "f6_single": lambda: f6_chunks([1700], 2500),
}


def literal_small(case) -> bool:
    """Small enough for the pure-Python literal_dp1."""
    return len(case["i"]) <= 20000
