"""Cross-matching a batch (describealign_b200.pairing): one shared video index per video, every description run
against it by dab_pair_stage_a_against.

Every cell must equal a fresh pair's stage_a() on that combination alone (match points, pass-1 path length,
gate candidates), and on these small cases the oracle's match_points + dp1; the matrix must not depend on how
many pairs run at once or on the input order.
"""
import threading
import time

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

SR = 44100


@pytest.fixture(scope="module")
def ctx():
    from describealign_b200 import _cabi, build
    build.build()
    return _cabi.Context(-1)


@pytest.fixture(scope="module")
def tracks():
    """3 videos x 4 descriptions: v0, v1, and v0 again without its first 7 s; d0 describes v0, d1 v1, d2 v0 with
    a longer intro (so it also describes v2), d3 a video that is not in the set."""
    from describealign_b200 import synth
    v0, d0 = synth.make_pair(45.0, 3.0, seed=101)
    v1, d1 = synth.make_pair(45.0, 4.0, seed=102)
    _, d2 = synth.make_pair(45.0, 9.0, seed=101)
    _, d3 = synth.make_pair(45.0, 3.0, seed=103)
    v2 = np.ascontiguousarray(v0[7 * SR:])
    return [v0, v1, v2], [d0, d1, d2, d3]


def _fresh(ctx, v, d):
    from describealign_b200 import _cabi
    pair = _cabi.Pair(ctx)
    try:
        pair.set_pcm(_cabi.VIDEO, v)
        pair.set_pcm(_cabi.AUDIO, d)
        n_points, n_path = pair.stage_a()
        return n_points, n_path, pair.stats()["n_candidates"]
    finally:
        pair.close()


def _check_fresh(ctx, videos, descriptions, res):
    assert all(e is None for e in res.errors.ravel()), res.errors
    for v in range(len(videos)):
        for d in range(len(descriptions)):
            want = _fresh(ctx, videos[v], descriptions[d])
            got = (res.points[v, d], res.path1[v, d], res.candidates[v, d])
            assert got == want, (v, d, got, want)


@pytest.fixture(scope="module")
def matrix(ctx, tracks):
    from describealign_b200 import pairing
    return pairing.cross_match(*tracks, in_flight=4)


def test_cells_equal_fresh_stage_a(ctx, tracks, matrix):
    _check_fresh(ctx, *tracks, matrix)
    # the pairs that belong together pass, the stranger passes nowhere
    assert matrix.passes[0, 0] and matrix.passes[1, 1] and matrix.passes[0, 2] and matrix.passes[2, 0]
    assert not matrix.passes[:, 3].any()
    assert not matrix.passes[1, 0] and not matrix.passes[0, 1]


def test_cells_equal_oracle(tracks, matrix):
    from describealign_b200 import host_fit
    from oracle import align_oracle as ao, features as of
    videos, descriptions = tracks
    F_v = [of.all_features(v) for v in videos]
    F_d = [of.all_features(d) for d in descriptions]
    for v, V in enumerate(F_v):
        for d, A in enumerate(F_d):
            pi, pv, pq, Lv, dbg = ao.match_points(V, A, V[0], A[0])
            px, _, _, _ = ao.dp1(pi, pv, pq, Lv)
            assert (matrix.points[v, d], matrix.path1[v, d], matrix.candidates[v, d]) == (len(pi), len(px), dbg["scored"]), (v, d)
            min_len = host_fit.min_path_length(len(V[0]), len(A[0]))
            assert matrix.passes[v, d] == (len(px) >= min_len), (v, d)


@pytest.mark.parametrize("in_flight", [1, 2, 32])
def test_in_flight_does_not_change_the_matrix(tracks, matrix, in_flight):
    from describealign_b200 import pairing
    res = pairing.cross_match(*tracks, in_flight=in_flight)
    for name in ("points", "path1", "min_len", "candidates", "passes"):
        assert np.array_equal(getattr(res, name), getattr(matrix, name)), name


def test_permuted_inputs_permute_the_matrix(tracks, matrix):
    from describealign_b200 import pairing
    videos, descriptions = tracks
    pv, pd = [2, 0, 1], [3, 1, 0, 2]
    res = pairing.cross_match([videos[k] for k in pv], [descriptions[k] for k in pd], in_flight=3)
    for name in ("points", "path1", "min_len", "candidates", "passes"):
        assert np.array_equal(getattr(res, name), getattr(matrix, name)[np.ix_(pv, pd)]), name


def test_reference_layouts_give_the_same_matrix(tracks, matrix):
    """The reference's float16 (ch, S) arrays are accepted as well as int16 (S, ch)."""
    from describealign_b200 import pairing, synth
    videos, descriptions = tracks
    res = pairing.cross_match([synth.as_reference_input(v) for v in videos], descriptions, in_flight=4)
    assert np.array_equal(res.path1, matrix.path1) and np.array_equal(res.points, matrix.points)


def test_one_index_serves_four_concurrent_pairs(ctx, tracks):
    from describealign_b200 import _cabi
    videos, descriptions = tracks
    src = _cabi.Pair(ctx)
    src.set_pcm(_cabi.VIDEO, videos[0])
    ix = _cabi.Index(src)
    src.close()                 # the index keeps nothing of the pair it was built from
    want = [_fresh(ctx, videos[0], d)[:2] for d in descriptions]
    got = [[] for _ in descriptions]
    start = threading.Barrier(len(descriptions))

    def run(d):
        pair = _cabi.Pair(_cabi.Context(-1))
        try:
            pair.set_pcm(_cabi.AUDIO, descriptions[d])
            start.wait()
            for _ in range(3):
                got[d].append(pair.stage_a_against(ix))
            x, y = pair.path1()
            got[d].append(len(x))
            with pytest.raises(_cabi.DabError, match="index"):
                pair.points1()
        finally:
            pair.close()

    threads = [threading.Thread(target=run, args=(d,)) for d in range(len(descriptions))]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    for d in range(len(descriptions)):
        assert got[d][:3] == [want[d]] * 3, (d, got[d])
        assert got[d][3] == want[d][1]
    assert ix.info()["users"] == 0
    ix.free()


@pytest.mark.parametrize("names", [("m2a", "m3")])
def test_overflowing_descriptions_retry_like_stage_a(ctx, tracks, names):
    """M2a (a sample-exact tone) and M3 (a looped bed) overflow the first capacity guesses; run as descriptions
    against their own videos and others, every cell equals stage_a()."""
    from oracle import stage_a_cases as sc
    cases = {"m2a": sc.m2a_tone, "m3": sc.m3_loop}
    pcm = [cases[n]() for n in names]
    videos = [v for v, _ in pcm] + [tracks[0][0]]
    descriptions = [a for _, a in pcm]
    from describealign_b200 import pairing
    res = pairing.cross_match(videos, descriptions, in_flight=2)
    _check_fresh(ctx, videos, descriptions, res)


def test_short_track_errors_only_its_cells(ctx, tracks):
    from describealign_b200 import pairing
    videos, descriptions = tracks
    short = np.ascontiguousarray(videos[0][:60 * 210])      # 60 frames < 82
    res = pairing.cross_match([videos[0], short], [descriptions[0], short], in_flight=2)
    assert res.errors[0, 0] is None and res.passes[0, 0]
    for v, d in ((0, 1), (1, 0), (1, 1)):
        assert "shorter than 82 frames" in res.errors[v, d], res.errors[v, d]
        assert res.path1[v, d] == -1 and not res.passes[v, d]


def test_free_is_refused_while_a_pair_runs_against_the_index(ctx, tracks):
    """The pair's stream is held up by a sleeping kernel, so its stage_a_against call stays inside the library
    until the sleep ends; freeing the index meanwhile is refused and frees nothing."""
    import torch
    from describealign_b200 import _cabi
    videos, descriptions = tracks
    src = _cabi.Pair(ctx)
    src.set_pcm(_cabi.VIDEO, videos[0])
    ix = _cabi.Index(src)
    src.close()
    pair = _cabi.Pair(ctx)
    pair.set_pcm(_cabi.AUDIO, descriptions[0])
    pair.sync()
    result = []
    try:
        with torch.cuda.stream(torch.cuda.ExternalStream(pair.stream)):
            torch.cuda._sleep(int(3e9))           # about 1.5 s
        t = threading.Thread(target=lambda: result.append(pair.stage_a_against(ix)))
        t.start()
        t0 = time.time()
        while ix.info()["users"] == 0 and time.time() - t0 < 10:
            time.sleep(0.001)
        assert ix.info()["users"] == 1
        with pytest.raises(_cabi.DabError, match="still running"):
            ix.free()
        t.join()
        assert result == [_fresh(ctx, videos[0], descriptions[0])[:2]]
        ix.free()
        assert ix.handle is None
    finally:
        pair.close()


def test_one_pair_switches_between_an_index_and_its_own_video_side(ctx, tracks):
    """One pair with the features of a video and a description runs stage_a_against an index of that video,
    stage_a, stage_a_against again, then stage_a_match over two row shards + import_points1 + dp1.  Every step
    gives a fresh pair's stage_a() counts and path.  After stage_a_against the points are ranks into the index, so
    points1, import_points1 and dp1 are refused (DAB_E_STATE); after the pair's own stage A they work again."""
    from describealign_b200 import _cabi, batch
    videos, descriptions = tracks
    fresh = _cabi.Pair(ctx)
    try:
        fresh.set_pcm(_cabi.VIDEO, videos[0])
        fresh.set_pcm(_cabi.AUDIO, descriptions[0])
        want = fresh.stage_a() + (fresh.stats()["n_candidates"],)
        want_points, want_path = fresh.points1(), fresh.path1()
        features = [fresh.get_features(t) for t in (_cabi.VIDEO, _cabi.AUDIO)]
    finally:
        fresh.close()
    assert want[1] > 0

    pair = _cabi.Pair(ctx)
    try:
        for t in (_cabi.VIDEO, _cabi.AUDIO):
            pair.set_features(t, features[t])
        ix = _cabi.Index(pair)

        def check_path():
            x, y = pair.path1()
            assert np.array_equal(x, want_path[0]) and np.array_equal(y, want_path[1])

        def check_refused():
            for call in (pair.points1, lambda: pair.import_points1(*want_points), pair.dp1):
                with pytest.raises(_cabi.DabError, match="error 3:"):
                    call()

        def check_own_points():
            got = pair.points1()
            for g, w in zip(got, want_points):
                assert np.array_equal(g, w)
            pair.import_points1(*want_points)
            assert pair.dp1() == want[1]
            check_path()

        for step in ("against", "own", "against"):
            got = pair.stage_a_against(ix) if step == "against" else pair.stage_a()
            assert got + (pair.stats()["n_candidates"],) == want, (step, got)
            check_path()
            if step == "against":
                check_refused()
            else:
                check_own_points()

        parts, n_cand = [], 0
        for lo, hi in batch.row_shards(pair.feature_lens(_cabi.AUDIO)[0], 2):
            pair.stage_a_match(lo, hi)
            parts.append(pair.points1())
            n_cand += pair.stats()["n_candidates"]
        points = [np.concatenate([p[k] for p in parts]) for k in range(3)]
        assert (len(points[0]), n_cand) == (want[0], want[2])
        pair.import_points1(*points)
        assert pair.dp1() == want[1]
        check_path()
        ix.free()
    finally:
        pair.close()


def test_assign_recovers_pairs_and_flags_the_name_order(tracks):
    from describealign_b200 import pairing
    videos, descriptions = tracks
    # names in the wrong order: description k is not the one of video k
    shuffled = [descriptions[1], descriptions[3], descriptions[0]]
    res = pairing.cross_match(videos[:2], shuffled, in_flight=3)
    pick = pairing.assign(res)
    assert pick.pairs == [(0, 2), (1, 0)]
    assert pick.unmatched_descriptions == [1] and pick.unmatched_videos == []
    assert (0, 2) in pick.disagreements and (1, 0) in pick.disagreements
    report = pairing.format_report(["v0.mkv", "v1.mkv"], ["a.wav", "b.wav", "c.wav"], res, pick)
    assert "disagrees" in report
