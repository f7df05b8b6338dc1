"""Stage A on repeated material and on tie-heavy DP 1 point sets, against the oracle (oracle/stage_a_cases.py).

Match-stage cases M1 (periodic features), M2a / M2b (a sample-exact tone at the head of both tracks, 15 s and
30 s) and M3 (a looped noise bed) overflow the first capacity guess of the match stage, so every path that owns
a grow-and-retry loop is run on them: a fresh pair, a reused pair, the row-sharded match stage, the batch engine
and the public API.  Bars of test_stage_a_golden: (i, v) identical, quals rel 1e-12, pass-1 path identical, and
the gate's candidate count equal to the oracle's.

DP 1 sets F1-F6 are imported into a pair whose video has energy 1.0 everywhere (hashed frames 4 * arange):
the pass-1 path must equal the oracle's.
"""
import numpy as np
import pytest

from conftest import golden_pair_pcm

pytestmark = pytest.mark.gpu

_ORACLE = {}


def _inputs(name):
    """(features V, A, PCM pair or None) of a match-stage case."""
    from oracle import features as of, stage_a_cases as sc
    if name == "m1":
        V, A = sc.m1_periodic()
        return V, A, None
    v, a = {"m2a": sc.m2a_tone, "m2b": sc.m2b_tone, "m3": sc.m3_loop}[name]()
    return of.all_features(v), of.all_features(a), (v, a)


def _want(name):
    from oracle import align_oracle as ao
    if name not in _ORACLE:
        V, A, pcm = _inputs(name)
        pi, pv, pq, Lv, dbg = ao.match_points(V, A, V[0], A[0])
        px, py, _, _ = ao.dp1(pi, pv, pq, Lv)
        _ORACLE[name] = dict(V=V, A=A, pcm=pcm, pi=pi, pv=pv, pq=pq, px=px, py=py, scored=dbg["scored"])
    return _ORACLE[name]


def _golden_a(golden_align):
    from oracle import align_oracle as ao, features as of
    if "pair_a" not in _ORACLE:
        data, meta = golden_align
        v, a = golden_pair_pcm(meta, "pair_a")
        V, A = of.all_features(v), of.all_features(a)
        g = data["pair_a"]
        _, _, _, _, dbg = ao.match_points(V, A, V[0], A[0])
        _ORACLE["pair_a"] = dict(V=V, A=A, pcm=(v, a), pi=g["points1_i"], pv=g["points1_v"], pq=g["points1_q"],
                                 px=g["path1_x"], py=g["path1_y"], scored=dbg["scored"])
    return _ORACLE["pair_a"]


def _load(pair, w):
    from describealign_b200 import _cabi
    pair.set_features(_cabi.VIDEO, w["V"])
    pair.set_features(_cabi.AUDIO, w["A"])


def _check(pair, w, what):
    pi, pv, pq = pair.points1()
    assert np.array_equal(pi, w["pi"]) and np.array_equal(pv, w["pv"]), what
    np.testing.assert_allclose(pq, w["pq"], rtol=1e-12, atol=0, err_msg=what)
    x, y = pair.path1()
    assert np.array_equal(x, w["px"]) and np.array_equal(y, w["py"]), what
    assert pair.stats()["n_candidates"] == w["scored"], what


M_CASES = ["m1", "m2a", "m2b", "m3"]


@pytest.mark.parametrize("name", M_CASES)
def test_fresh_pair_retries_and_matches_oracle(gpu_ctx, name):
    """A fresh pair overflows, grows and reruns: runs = launches of the first call / launches of an immediate
    rerun (one attempt; launches per attempt are fixed for fixed lengths).  Every case needs a second run;
    sizing a rerun from the totals of the run that overflowed bounds it at three (an entries overflow hides
    the candidate total for one run)."""
    from describealign_b200 import _cabi
    w = _want(name)
    pair = _cabi.Pair(gpu_ctx)
    try:
        _load(pair, w)
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
    runs = first // per_run
    assert 2 <= runs <= 3, runs


@pytest.mark.parametrize("name", M_CASES)
def test_reused_pair_keeps_no_state_between_inputs(gpu_ctx, golden_align, name):
    """M, then the golden pair_a, then M again on one pair: capacities only grow, nothing of an earlier
    run leaks into the next."""
    from describealign_b200 import _cabi
    w, g = _want(name), _golden_a(golden_align)
    pair = _cabi.Pair(gpu_ctx)
    try:
        for k, x in enumerate((w, g, w)):
            _load(pair, x)
            pair.stage_a()
            _check(pair, x, f"{name} step {k}")
    finally:
        pair.close()


@pytest.mark.parametrize("name", M_CASES)
def test_row_shards_retry_on_their_own(gpu_ctx, name):
    """stage_a_match over three row shards (each shard overflows and retries by itself), then the points
    imported back and DP 1: the oracle's points and path; the shards' candidates add up to the oracle's."""
    from describealign_b200 import _cabi, batch
    w = _want(name)
    pair = _cabi.Pair(gpu_ctx)
    try:
        _load(pair, w)
        parts, n_cand = [], 0
        for lo, hi in batch.row_shards(len(w["A"][0]), 3):
            n = pair.stage_a_match(lo, hi)
            pi, pv, pq = pair.points1()
            assert len(pi) == n and (n == 0 or (pi.min() >= lo and pi.max() < hi))
            parts.append((pi, pv, pq))
            n_cand += pair.stats()["n_candidates"]
        pi, pv, pq = (np.concatenate([p[k] for p in parts]) for k in range(3))
        assert np.array_equal(pi, w["pi"]) and np.array_equal(pv, w["pv"])
        np.testing.assert_allclose(pq, w["pq"], rtol=1e-12, atol=0)
        assert n_cand == w["scored"]
        pair.import_points1(pi, pv, pq)
        pair.dp1()
        x, y = pair.path1()
        assert np.array_equal(x, w["px"]) and np.array_equal(y, w["py"])
    finally:
        pair.close()


def _same_result(got, want, what):
    if isinstance(want, Exception):
        assert type(got) is type(want) and str(got) == str(want), (what, got, want)
        return
    assert not isinstance(got, Exception), (what, got)
    for k in (0, 1, 3):
        np.testing.assert_array_equal(got[k], want[k], err_msg=what)
    assert got[2] == want[2] and got[4] == want[4], what


def _align_or_exc(v, a):
    from describealign_b200 import api
    try:
        return api.align_pcm(v, a)
    except Exception as e:       # the engine reports a failing pair as its exception
        return e


@pytest.mark.parametrize("name", ["m2a", "m2b", "m3"])
def test_engine_slots_retry_and_match_the_api(gpu_ctx, golden_align, name):
    """The batch engine's own retry loop, with slots reused (in_flight 1) and two pairs in flight: [M, pair_a, M]
    gives what api.align_pcm gives for each pair, or the same exception."""
    from describealign_b200 import batch, _cabi
    w, g = _want(name), _golden_a(golden_align)
    pairs = [w["pcm"], g["pcm"], w["pcm"]]
    want = [_align_or_exc(*p) for p in pairs]
    for in_flight in (1, 2):
        got = batch.run_engine(pairs, in_flight=in_flight)
        for k, (x, y) in enumerate(zip(got, want)):
            if isinstance(y, _cabi.DabError) and isinstance(x, _cabi.DabError):
                # the engine's message carries the same error text after its own prefix
                assert str(y).split(": ", 1)[-1] in str(x), (x, y)
                continue
            _same_result(x, y, f"{name} in_flight={in_flight} pair {k}")


@pytest.mark.parametrize("name", ["m2a", "m3"])
def test_end_to_end_vs_oracle_on_repeated_audio(gpu_ctx, name):
    """api.align_pcm against ao.align with the bars of test_end_to_end_vs_oracle, or the same exception."""
    from describealign_b200 import api, host_fit
    from oracle import align_oracle as ao
    w = _want(name)
    v, a = w["pcm"]
    V, A = w["V"], w["A"]
    try:
        want = ao.align(V, A, V[0], A[0], host_fit)
    except Exception as e:
        with pytest.raises(type(e)) as got:
            api.align_pcm(v, a)
        assert str(got.value) == str(e)
        return
    nx, ny, sim, path, med = api.align_pcm(v, a)
    ox, oy, osim, opath, omed = want
    assert path.shape == opath.shape
    assert np.array_equal(path[:, 1], opath[:, 1]) and np.array_equal(path[:, 2], opath[:, 2])
    np.testing.assert_allclose(path[:, 0], opath[:, 0], rtol=0, atol=1e-9)
    np.testing.assert_allclose(path[:, 3:], opath[:, 3:], rtol=0, atol=1e-8)
    np.testing.assert_allclose(nx, ox, rtol=0, atol=1e-9)
    np.testing.assert_allclose(ny, oy, rtol=0, atol=1e-9)
    assert abs(sim - osim) < 1e-9 and med == omed


# ------------------------------------------------------------------------------------------
# DP 1 point sets
# ------------------------------------------------------------------------------------------

def _f_pair(ctx, Le):
    """A pair whose video has Le frames of energy 1.0 (hashed frames 4 * arange) and zero elsewhere, with the
    hashed-frame list built by a match stage over no audio rows."""
    from describealign_b200 import _cabi
    z = np.zeros(Le, np.float32)
    V = [np.ones(Le, np.float32), z, z, z, np.zeros(Le, np.float64)]
    za = np.zeros(200, np.float32)
    A = [np.ones(200, np.float32), za, za, za, np.zeros(200, np.float64)]
    pair = _cabi.Pair(ctx)
    pair.set_features(_cabi.VIDEO, V)
    pair.set_features(_cabi.AUDIO, A)
    pair.stage_a_match(0, 0)
    return pair


def _f_run(pair, case):
    pair.import_points1(case["i"], case["v"], case["q"])
    pair.dp1()
    return pair.path1()


def _f_cases():
    from oracle import stage_a_cases as sc
    out = [("f1", sc.f1_fast_vs_tree), ("f1_mirror", sc.f1_mirror), ("f2", lambda: sc.f2_rounding("tie")), ("f2_below", lambda: sc.f2_rounding("below")), ("f3", sc.f3_tree),
           ("f4_superseded", sc.f4_superseded), ("f4_large", sc.f4_large), ("f5_limit", sc.f5_limit)]
    out += [(f"f4_n{n}", (lambda n=n: sc.f4_small(n))) for n in sc.F4_SIZES]
    out += [(f"f4_path{n}", (lambda n=n: sc.f4_path(n))) for n in sc.F4_PATHS]
    out += list(sc.F6_CASES.items())
    return out


def test_dp1_point_sets_vs_oracle(gpu_ctx):
    """Every F set through import_points1 + dp1 + path1: the oracle's path.  Sets of one video length share a pair."""
    from oracle import align_oracle as ao
    pairs = {}
    try:
        for name, build in _f_cases():
            case = build()
            if case["Le"] not in pairs:
                pairs[case["Le"]] = _f_pair(gpu_ctx, case["Le"])
            x, y = _f_run(pairs[case["Le"]], case)
            px, pv, _, _ = ao.dp1(case["i"], case["v"], case["q"], case["Lv"])
            assert np.array_equal(x, px) and np.array_equal(y, pv), (name, len(x), len(px))
    finally:
        for p in pairs.values():
            p.close()


def test_dp1_tree_limit_one_frame_over(gpu_ctx):
    """One video frame past the DP tree's 2^20 slots: a clean error, not a crash or a wrong path."""
    from describealign_b200 import _cabi
    from oracle import stage_a_cases as sc
    case = sc.f5_limit(over=True)
    pair = _f_pair(gpu_ctx, case["Le"])
    try:
        pair.import_points1(case["i"], case["v"], case["q"])
        with pytest.raises(_cabi.DabError, match="too many hashed video frames for the DP tree"):
            pair.dp1()
    finally:
        pair.close()
