"""Stage A's hash tables (two-level counting sort, csrc/stage_a.cu table_*_kernel) at their edges, against the oracle.

The slots are f * 7^7 + code over the five tables, cut into super-buckets of 4096; every super-bucket is sorted by
one CTA in chunks of 2048 entries.  Constructed features reach:
  mixed       random features 0-3 and a spike train of period 6 in feature 4: a super-bucket of more than 100 sort
              chunks, entries on both sides of super-bucket boundaries (local slots 4095 and 0), slot 5 * 7^7 - 1
              (all seven digits 6, in the partial last super-bucket, also looked up by the audio), and more entries
              than the first capacity guess (an entries overflow, then a retry)
  no_hashed   a quiet video: no hashed frames, empty tables
  one_hashed  one not-quiet video frame: one hashed frame
The CPU computes each case's slots from the oracle's codes and flags and asserts the case is reached; the GPU
runs it through Pair.stage_a and a shared index, with the bars of test_gpu_stage_a_edges._check.
"""
import numpy as np
import pytest

NCODE = 7 ** 7
NSLOTS = 5 * NCODE
SB = 4096
SORT_CHUNK = 2048           # entries a super-bucket's CTA takes per step (TS_THREADS x TS_UNROLL)

_CASES = {}


def _mixed():
    rng = np.random.default_rng(11)
    n = 40000
    V = [rng.uniform(0.6, 1.4, n + 1).astype(np.float32)] + [rng.standard_normal(n).astype(np.float32) for _ in range(3)]
    b2 = np.zeros(n)
    b2[2::6] = 1.0          # hashed frames t = 0 mod 6 sample seven spikes: ms / nrm > 0.3375, every digit 6
    V.append(b2)
    lo, hi = 5000, 15000
    A = [V[0][lo:hi + 1].copy()] + [x[lo:hi].copy() for x in V[1:]]
    return V, A


def _quiet(seed):
    rng = np.random.default_rng(seed)
    m = 3000
    V = [np.full(m + 1, 0.3, np.float32)] + [rng.standard_normal(m).astype(np.float32) for _ in range(3)] + [rng.standard_normal(m)]
    return V, rng


def _no_hashed():
    V, rng = _quiet(12)
    A = [rng.uniform(0.6, 1.4, 1001).astype(np.float32)] + [rng.standard_normal(1000).astype(np.float32) for _ in range(3)]
    A.append(rng.standard_normal(1000))
    return V, A


def _one_hashed():
    V, _ = _quiet(13)
    V[0][1000] = 1.0
    return V, [x.copy() for x in V]


BUILDERS = {"mixed": _mixed, "no_hashed": _no_hashed, "one_hashed": _one_hashed}


def _slots(V):
    """Every expanded entry's slot f * 7^7 + code (2^flags per hashed frame and table), and the hashed frames."""
    from oracle import align_oracle as ao
    _, _, code, flags = ao.prep_track(V, True)
    sel = ao.not_quiet(V[0])[::4]
    p7 = 7 ** np.arange(7)
    out = [np.zeros(0, np.int64)]
    for f in range(5):
        c = code[f][sel].astype(np.int64)
        fl = flags[f][sel].astype(np.int64)
        for sub in range(128):
            has = (fl & sub) == sub
            out.append(f * NCODE + c[has] + int(sum(p7[k] for k in range(7) if sub >> k & 1)))
    return np.concatenate(out), sel


def _case(name):
    from oracle import align_oracle as ao, stage_a_cases as sc
    if name not in _CASES:
        V, A = BUILDERS[name]()
        slots, sel = _slots(V)
        pi, pv, pq, Lv, dbg = ao.match_points(V, A, V[0], A[0])
        px, py, _, _ = ao.dp1(pi, pv, pq, Lv)
        _, _, a_code, _ = ao.prep_track(A, False)
        a_nq = ao.not_quiet(A[0])
        _CASES[name] = dict(V=V, A=A, slots=slots, n_sel=len(sel), entries=sc.expanded_entries(ao.prep_track(V, True)[3], sel),
                            cap=sc.stage_a_caps(len(V[0]), len(A[0]))[0], a_code4=a_code[4][a_nq],
                            pi=pi, pv=pv, pq=pq, px=px, py=py, scored=dbg["scored"])
    return _CASES[name]


def test_cases_reach_their_edges(oracle_lib):
    """CPU: the slots of each case, from the oracle's codes and flags."""
    w = _case("mixed")
    s = w["slots"]
    assert len(s) == w["entries"]
    per_sb = np.bincount(s // SB, minlength=(NSLOTS + SB - 1) // SB)
    assert per_sb.max() >= 100 * SORT_CHUNK, per_sb.max()
    occ = np.zeros(NSLOTS + 1, bool)
    occ[s] = True
    last_of_sb = np.arange(SB - 1, NSLOTS - 1, SB)
    assert np.sum(occ[last_of_sb] & occ[last_of_sb + 1]) >= 10          # local slots 4095 and 0 side by side
    assert occ[NSLOTS - 1] and (NSLOTS - 1) // SB == len(per_sb) - 1 and NSLOTS % SB != 0
    assert np.any(w["a_code4"] == NCODE - 1)                             # the gate reads start[5 * 7^7]
    assert w["entries"] > w["cap"]                                       # overflows the first guess
    assert len(w["px"]) > 1000

    w = _case("no_hashed")
    assert w["n_sel"] == 0 and len(w["slots"]) == 0 and len(w["pi"]) == 0
    w = _case("one_hashed")
    assert w["n_sel"] == 1 and w["entries"] == len(w["slots"]) > 0 and len(w["px"]) == 1


def _check(pair, w, what):
    pi, pv, pq = pair.points1()
    assert np.array_equal(pi, w["pi"]) and np.array_equal(pv, w["pv"]), what
    np.testing.assert_allclose(pq, w["pq"], rtol=1e-12, atol=0, err_msg=what)
    x, y = pair.path1()
    assert np.array_equal(x, w["px"]) and np.array_equal(y, w["py"]), what
    assert pair.stats()["n_candidates"] == w["scored"], what
    assert pair.stats()["n_table_entries"] == w["entries"], what


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(BUILDERS))
def test_tables_vs_oracle(gpu_ctx, name):
    """A fresh pair, then a rerun on the same pair: points, path, candidates and entries of the oracle.  The
    mixed case overflows the entries' first guess: its first call is two runs (launches of the first call over
    those of the rerun), the others one."""
    from describealign_b200 import _cabi
    w = _case(name)
    pair = _cabi.Pair(gpu_ctx)
    try:
        pair.set_features(_cabi.VIDEO, w["V"])
        pair.set_features(_cabi.AUDIO, w["A"])
        l0 = gpu_ctx.launches()
        pair.stage_a()
        l1 = gpu_ctx.launches()
        _check(pair, w, f"{name} first")
        l2 = gpu_ctx.launches()
        pair.stage_a()
        l3 = gpu_ctx.launches()
        _check(pair, w, f"{name} rerun")
    finally:
        pair.close()
    first, per_run = l1 - l0, l3 - l2
    assert per_run > 0 and first % per_run == 0, (first, per_run)
    assert first // per_run == (2 if w["entries"] > w["cap"] else 1), (first, per_run)


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(BUILDERS))
def test_index_tables_vs_oracle(gpu_ctx, name):
    """The cross-match index builds the same tables (its own grow-and-retry loop): entries, path and counts."""
    from describealign_b200 import _cabi
    w = _case(name)
    pair = _cabi.Pair(gpu_ctx)
    try:
        pair.set_features(_cabi.VIDEO, w["V"])
        pair.set_features(_cabi.AUDIO, w["A"])
        ix = _cabi.Index(pair)
        try:
            assert ix.info()["n_table_entries"] == w["entries"]
            assert ix.info()["n_video_selected"] == w["n_sel"]
            assert pair.stage_a_against(ix) == (len(w["pi"]), len(w["px"]))
            x, y = pair.path1()
            assert np.array_equal(x, w["px"]) and np.array_equal(y, w["py"])
            assert pair.stats()["n_candidates"] == w["scored"]
        finally:
            ix.free()
    finally:
        pair.close()
