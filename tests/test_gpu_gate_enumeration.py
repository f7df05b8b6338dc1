"""Stage A's gate when a pair's queries visit more than 2^31 bucket entries in all (csrc/stage_a.cu, count pass).

gate_plan_kernel gives every audio query the entry count of its two cheapest buckets, a 64-bit exclusive scan of
those counts places every entry, and gate_entries_kernel walks the entries in tiles of GE_TILE.  The cases below
drive the total past 2^31 and 2^32 with almost no candidates, from features set directly (no PCM) and a gate energy
that keeps every frame not quiet:

  video   three groups of G frames: group A has feature 0 flat, group B feature 1, group C feature 3, every other
          feature white noise; then a noise segment of D frames (all features)
  audio   Q queries with features 0, 1 and 3 flat and noise in 2 and 4; then a copy of the video's noise segment

A flat stretch mean-subtracts to zero and its norm clips at 1e-3, so every flat frame has the code 3333333 (base 7).
Each valid bucket pair of a flat query ({3,4} or two of {0,1,2}) then holds one whole group: the query visits about
G / 4 hashed frames, and matches them in one feature only.  The copied segment gives the true matches and the path.

  control   just under 2^31 entries
  L1        more than 2^31
  L2        more than 2^32: the high word of the total is used

The CPU restates the bucket choice over the oracle's codes and flags: the exact entry count of every query, the rows
where the prefix crosses 2^31 and 2^32, and row shards that each stay under 2^31 with boundaries on those rows.  It
also shows that a 32-bit prefix (what the gate used before) wraps there.  The GPU compares the one-shot stage A, the
row shards, the oracle on row ranges around each crossing, the oracle's DP 1 and a shared index.
"""
import os
import re

import numpy as np
import pytest

NCODE = 7 ** 7
FLAT_CODE = 3 * (NCODE - 1) // 6          # seven digits 3
GE_TILE = 2048                            # entries per tile of gate_entries_kernel (GE_THREADS x GE_PER)
G = 60000                                 # frames per flat group (G / 4 hashed)
D = 20000                                 # frames of the copied noise segment
QUERIES = {"control": 140000, "L1": 200000, "L2": 300000}

_CASES = {}


def _video():
    rng = np.random.default_rng(21)
    n = 3 * G + D
    V = [rng.standard_normal(n + (1 if f == 0 else 0)) for f in range(5)]
    for g, f in enumerate((0, 1, 3)):
        V[f][g * G:(g + 1) * G] = 0.0
    return _as_features(V)


def _audio(V, q):
    rng = np.random.default_rng(22)
    A = []
    for f in range(5):
        x = rng.standard_normal(q) if f in (2, 4) else np.zeros(q)
        A.append(np.concatenate([x, V[f][3 * G:3 * G + D + (1 if f == 0 else 0)]]))
    return _as_features(A)


def _as_features(F):
    return [F[0].astype(np.float32)] + [x.astype(np.float32) for x in F[1:4]] + [F[4].astype(np.float64)]


def _bucket_counts(V):
    """Entries per slot of each of the five video tables: a hashed frame is stored under 2^flags codes."""
    from oracle import align_oracle as ao
    _, _, code, flags = ao.prep_track(V, True)
    sel = ao.not_quiet(np.ones(len(V[0])))[::4]
    p7 = 7 ** np.arange(7)
    out = []
    for f in range(5):
        c = code[f][sel].astype(np.int64)
        fl = flags[f][sel].astype(np.int64)
        slots = [c[(fl & sub) == sub] + int(sum(p7[k] for k in range(7) if sub >> k & 1)) for sub in range(128)]
        out.append(np.bincount(np.concatenate(slots), minlength=NCODE))
    return out, code


def _entries_per_query(cnt, A):
    """gate_plan_kernel's bucket choice: the joint length of the cheapest valid bucket pair, ties to the first."""
    from oracle import align_oracle as ao
    _, _, a_code, _ = ao.prep_track(A, False)
    q = ao.not_quiet(np.ones(len(A[0])))
    nb = [cnt[f][a_code[f][q]].astype(np.int64) for f in range(5)]
    best = nb[0] + nb[1]
    for s in (nb[0] + nb[2], nb[1] + nb[2], nb[3] + nb[4]):
        best = np.where(s < best, s, best)
    return best, a_code


def _crossing(P, x):
    """The query row that owns entry x: P[r] <= x < P[r + 1]."""
    return int(np.searchsorted(P, x, side="right") - 1)


def _case(name):
    if "video" not in _CASES:
        V = _video()
        _CASES["video"] = (V, *_bucket_counts(V))
    if name not in _CASES:
        V, cnt, v_code = _CASES["video"]
        q = QUERIES[name]
        A = _audio(V, q)
        best, a_code = _entries_per_query(cnt, A)
        P = np.concatenate([[0], np.cumsum(best)])
        cross = [_crossing(P, x) for x in (1 << 31, 1 << 32) if x < P[-1]]
        # shards: every crossing row starts a shard, and shards are split until each is under 2^31 / 2
        bounds = sorted({0, len(best), *cross})
        while True:
            wide = [k for k in range(len(bounds) - 1) if P[bounds[k + 1]] - P[bounds[k]] >= 1 << 30]
            if not wide:
                break
            k = wide[0]
            bounds.insert(k + 1, _crossing(P, (P[bounds[k]] + P[bounds[k + 1]]) // 2))
        _CASES[name] = dict(V=V, A=A, q=q, best=best, P=P, total=int(P[-1]), cross=cross, bounds=bounds,
                            v_code=v_code, a_code=a_code)
    return _CASES[name]


def _shard_rows(w):
    b = w["bounds"]
    return [(b[k], b[k + 1] if k + 2 < len(b) else 2 ** 62) for k in range(len(b) - 1)]


# ---------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------
def test_model_matches_the_source():
    """The tile size and the bucket rule of the model are those of stage_a.cu; the prefix the gate reads is 64-bit."""
    src = open(os.path.join(os.path.dirname(__file__), "..", "describealign_b200", "csrc", "stage_a.cu")).read()
    m = re.search(r"constexpr int GE_THREADS = (\d+), GE_PER = (\d+), GE_TILE = GE_THREADS \* GE_PER;", src)
    assert int(m.group(1)) * int(m.group(2)) == GE_TILE
    plan = src[src.index("__global__ void gate_plan_kernel"):src.index("constexpr int GE_THREADS")]
    assert re.search(r"int fa = 0, fb = 1, best = nb\[0\] \+ nb\[1\];\s*"
                     r"if \(nb\[0\] \+ nb\[2\] < best\) \{ best = nb\[0\] \+ nb\[2\]; fa = 0; fb = 2; \}\s*"
                     r"if \(nb\[1\] \+ nb\[2\] < best\) \{ best = nb\[1\] \+ nb\[2\]; fa = 1; fb = 2; \}\s*"
                     r"if \(nb\[3\] \+ nb\[4\] < best\) \{ best = nb\[3\] \+ nb\[4\]; fa = 3; fb = 4; \}", plan)
    assert "nb[f] = g.start[slot + 1] - st[f];" in plan
    assert re.search(r"gate_entries_kernel\(GateArgs g, const GateQ \*rec, const int64_t \*P\)", src)
    assert re.search(r"dab_exclusive_scan\(pr, g_best, g_P, q_ub, nullptr, dc \+ DC_ENUM_LO\)", src)
    assert "int64_t *g_P" in src


def test_cases_reach_their_edges(oracle_lib):
    """Totals past 2^31 and 2^32, shards under 2^31 that start on the crossing rows, and the wrap of a 32-bit prefix."""
    V, cnt, v_code = _case("control")["V"], *_CASES["video"][1:]
    # every flat frame inside a group has the code 3333333, and the group's bucket holds about G / 4 hashed frames
    for g, f in enumerate((0, 1, 3)):
        assert np.all(v_code[f][g * G + 20:(g + 1) * G - 60] == FLAT_CODE)
        assert G // 4 - 30 <= cnt[f][FLAT_CODE] <= G // 4 + 100, (f, cnt[f][FLAT_CODE])
    for name, (lo, hi) in {"control": (1 << 30, (1 << 31) - 1), "L1": ((1 << 31) + 1, 1 << 32),
                           "L2": ((1 << 32) + 1, 1 << 33)}.items():
        w = _case(name)
        for f in (0, 1, 3):
            assert np.all(w["a_code"][f][20:w["q"] - 60] == FLAT_CODE)
        assert lo <= w["total"] <= hi, (name, w["total"])
        assert w["best"].max() < 1 << 31
        assert len(w["cross"]) == {"control": 0, "L1": 1, "L2": 2}[name]
        P, b = w["P"], w["bounds"]
        # the int32 prefix the gate used to read: it falls at the row that crosses 2^31 (int32) and again at the row
        # that crosses 2^32 (its 32 bits), so the owner search in it no longer holds
        u32 = P.astype(np.uint64).astype(np.uint32)
        for r, x, p32 in zip(w["cross"], (1 << 31, 1 << 32), (u32.view(np.int32), u32)):
            assert P[r] <= x < P[r + 1] and r in b
            assert p32[r + 1] < p32[r], name
        if name == "control":
            assert np.all(np.diff(u32.view(np.int32).astype(np.int64)) >= 0)
        for k in range(len(b) - 1):
            assert 0 < P[b[k + 1]] - P[b[k]] < 1 << 31, (name, k)
    # the old gate read its total as one int32 word: L1 reads negative (nothing visited), L2 reads the low word only
    low = {n: int(np.array([_case(n)["total"]], np.int64).astype(np.uint32).view(np.int32)[0]) for n in ("L1", "L2")}
    assert low["L1"] < 0
    assert low["L2"] == _case("L2")["total"] - (1 << 32)


# ---------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------
def _pair(ctx, w):
    from describealign_b200 import _cabi
    pair = _cabi.Pair(ctx)
    for t, F in ((_cabi.VIDEO, w["V"]), (_cabi.AUDIO, w["A"])):
        pair.set_features(t, F)
        pair.set_gate_energy(t, np.ones(len(F[0]), np.float32))
    return pair


def _oracle_rows(w, rows):
    from oracle import align_oracle as ao
    V, A = w["V"], w["A"]
    pi, pv, pq, _, _ = ao.match_points(V, A, np.ones(len(V[0])), np.ones(len(A[0])), rows=rows)
    return pi, pv, pq


def _rows_of(points, rows):
    i, v, q = points
    m = (i >= rows[0]) & (i < rows[1])
    return i[m], v[m], q[m]


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(QUERIES))
def test_one_shot_equals_shards_and_oracle(gpu_ctx, name):
    """stage_a(): the exact entry count; its points are the row shards' (each under 2^31 entries) and the oracle's on
    rows around every crossing and on the copied segment; its path is the oracle's DP 1 over those points."""
    from oracle import align_oracle as ao
    w = _case(name)
    pair = _pair(gpu_ctx, w)
    try:
        pair.stage_a()
        st = pair.stats()
        assert st["n_enumerated"] == w["total"]
        full = pair.points1()
        path = pair.path1()
        assert len(full[0]) > 1000 and len(path[0]) > 1000
        shards, n_cand = [], 0
        for lo, hi in _shard_rows(w):
            pair.stage_a_match(lo, hi)
            sst = pair.stats()
            assert sst["n_enumerated"] == w["P"][min(hi, len(w["best"]))] - w["P"][lo], (lo, hi)
            n_cand += sst["n_candidates"]
            shards.append(pair.points1())
    finally:
        pair.close()
    assert n_cand == st["n_candidates"]
    for k in range(3):
        assert np.array_equal(np.concatenate([s[k] for s in shards]), full[k]), k
    ranges = [(0, 300), (w["q"] - 200, w["q"] + D)] + [(r - 200, r + 200) for r in w["cross"]]
    for rows in ranges:
        pi, pv, pq = _oracle_rows(w, rows)
        gi, gv, gq = _rows_of(full, rows)
        assert np.array_equal(gi, pi) and np.array_equal(gv, pv), rows
        np.testing.assert_allclose(gq, pq, rtol=1e-12, atol=0, err_msg=str(rows))
    Lv = len(w["V"][0]) - 40
    px, py, _, _ = ao.dp1(full[0], full[1], full[2], Lv)
    assert np.array_equal(path[0], px) and np.array_equal(path[1], py)


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(QUERIES))
def test_index_gives_the_same_counts_and_path(gpu_ctx, name):
    """The same pair against a shared index of its video (the cross-match cell): entries, candidates, points, path."""
    from describealign_b200 import _cabi
    w = _case(name)
    pair = _pair(gpu_ctx, w)
    try:
        want_counts = pair.stage_a()
        want_st, want_path = pair.stats(), pair.path1()
        ix = _cabi.Index(pair)
        try:
            assert pair.stage_a_against(ix) == want_counts
            st = pair.stats()
            assert st["n_enumerated"] == w["total"]
            assert st["n_candidates"] == want_st["n_candidates"]
            x, y = pair.path1()
            assert np.array_equal(x, want_path[0]) and np.array_equal(y, want_path[1])
        finally:
            ix.free()
    finally:
        pair.close()


@pytest.mark.gpu
def test_engine_event_carries_the_enumeration_count(gpu_ctx):
    """An engine slot's stage-A event carries n_enumerated and the path of the synchronous API on the same PCM."""
    from describealign_b200 import _cabi, synth
    v, a = synth.make_pair(60.0, 4.0, seed=5)
    pair = _cabi.Pair(gpu_ctx)
    try:
        pair.set_pcm(_cabi.VIDEO, v)
        pair.set_pcm(_cabi.AUDIO, a)
        pair.stage_a()
        want_st, want_path = pair.stats(), pair.path1()
    finally:
        pair.close()
    assert want_st["n_enumerated"] > 0 and len(want_path[0]) > 0
    eng = _cabi.Engine(gpu_ctx, slots=1)
    try:
        eng.submit(0, v, a)
        evt = eng.next(60000)
        assert evt is not None and evt.kind == _cabi.EVENT_STAGE_A and evt.status == 0, eng.error(evt) if evt else None
        assert evt.stats.as_dict()["n_enumerated"] == want_st["n_enumerated"]
        x, y = _cabi.Engine.path1(evt)
        assert np.array_equal(x, want_path[0]) and np.array_equal(y, want_path[1])
        eng.release(evt.slot)
    finally:
        eng.close()
