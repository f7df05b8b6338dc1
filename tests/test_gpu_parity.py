"""GPU parity tests: the CUDA path, called through the C ABI, against the oracle and the
golden fixtures made from the reference (tests/golden/, tools/make_golden.py).

Bars: float32 features bit-exact; band 2 (float64) within 4 ulp; integer outputs (match
points, pass-1 path, pass-2 (i, int(j), cluster)) identical; float64 quals rel 1e-12 (pow /
log10 are the device's libm, not glibc's); node times within 1e-9 s.
"""
import numpy as np
import pytest

from conftest import golden_pair_pcm

pytestmark = pytest.mark.gpu


def _features_gpu(ctx, pcm):
    from describealign_b200 import _cabi
    pair = _cabi.Pair(ctx)
    pair.set_pcm(_cabi.VIDEO, pcm)
    f = pair.get_features(_cabi.VIDEO)
    pair.close()
    return f


def _check_features(got, want, what):
    names = ["energy", "zero_crossings", "band0", "band1", "band2"]
    for k in range(5):
        assert got[k].shape == want[k].shape, f"{what}: {names[k]} length {got[k].shape} != {want[k].shape}"
    for k in range(4):
        bad = np.flatnonzero(got[k] != want[k])
        assert bad.size == 0, f"{what}: {names[k]} differs at {bad[:5]} ({bad.size} of {got[k].size})"
    err = np.abs(got[4] - want[4])
    assert np.all(err <= 4 * np.spacing(np.abs(want[4]))), f"{what}: band2 max err {err.max()}"


def test_features_golden(gpu_ctx, golden_features):
    """CUDA features == the reference's own outputs (portable mode) on the golden clips."""
    from describealign_b200 import synth
    data, meta = golden_features
    for case in meta["cases"]:
        pcm, _ = synth.make_pair(case["seconds"], 0.5, seed=case["seed"], ch=case["ch"], narration_frac=0)
        got = _features_gpu(gpu_ctx, pcm)
        want = [data[f"{case['name']}.{k}"] for k in ("energy", "zc", "b0", "b1", "b2")]
        _check_features(got, want, case["name"])


def test_features_extremes(gpu_ctx, golden_features):
    data, _ = golden_features
    S = 210 * 60 + 17
    ext = {"silence": np.zeros((S, 1), np.int16),
           "square": (np.where((np.arange(S) // 3) % 2 == 0, 32767, -32768).astype(np.int16))[:, None],
           "impulse": np.zeros((S, 1), np.int16)}
    ext["impulse"][S // 2, 0] = 12345
    for name, pcm in ext.items():
        got = _features_gpu(gpu_ctx, pcm)
        want = [data[f"{name}.{k}"] for k in ("energy", "zc", "b0", "b1", "b2")]
        _check_features(got, want, name)


@pytest.mark.parametrize("ch,seconds,seed", [(1, 33.37, 101), (2, 21.013, 102), (1, 1.0, 103), (2, 0.5, 104)])
def test_features_vs_oracle(gpu_ctx, ch, seconds, seed):
    from describealign_b200 import synth
    from oracle import features as of
    pcm, _ = synth.make_pair(seconds, 0.2, seed=seed, ch=ch, narration_frac=0)
    _check_features(_features_gpu(gpu_ctx, pcm), of.all_features(pcm), f"ch{ch}")
    # float16 input (the reference's own array type) gives the same result as int16 input
    f16 = np.ascontiguousarray(pcm).astype(np.float16)
    _check_features(_features_gpu(gpu_ctx, f16), of.all_features(pcm), f"ch{ch} f16")


def test_features_tiny_and_empty(gpu_ctx):
    from oracle import features as of
    rng = np.random.default_rng(5)
    for S in (0, 1, 104, 105, 209, 210, 211, 419, 420, 1000):
        pcm = rng.integers(-3000, 3000, size=(S, 1)).astype(np.int16)
        got = _features_gpu(gpu_ctx, pcm)
        want = of.all_features(pcm)
        _check_features(got, want, f"S={S}")


def _stage_a_gpu(ctx, V, A):
    from describealign_b200 import _cabi
    pair = _cabi.Pair(ctx)
    pair.set_features(_cabi.VIDEO, V)
    pair.set_features(_cabi.AUDIO, A)
    pair.stage_a()
    return pair


def test_stage_a_golden(gpu_ctx, golden_align):
    """Match points and the pass-1 path equal the reference's on the golden pairs."""
    from oracle import features as of
    data, meta = golden_align
    for name in meta["cases"]:
        g = data[name]
        v, a = golden_pair_pcm(meta, name)
        V, A = of.all_features(v), of.all_features(a)
        pair = _stage_a_gpu(gpu_ctx, V, A)
        pi, pv, pq = pair.points1()
        assert np.array_equal(pi, g["points1_i"]) and np.array_equal(pv, g["points1_v"]), name
        np.testing.assert_allclose(pq, g["points1_q"], rtol=1e-12, atol=0)
        x, y = pair.path1()
        assert np.array_equal(x, g["path1_x"]) and np.array_equal(y, g["path1_y"]), name
        pair.close()


def test_end_to_end_golden(gpu_ctx, golden_align):
    """PCM in -> nodes out through the public API equals the reference's result."""
    from describealign_b200 import api
    data, meta = golden_align
    for name in meta["cases"]:
        g = data[name]
        v, a = golden_pair_pcm(meta, name)
        det = {}
        nx, ny, sim, path, med = api.align_pcm(v, a, details=det)
        gp = g["path2"]
        assert path.shape == gp.shape, name
        assert np.array_equal(path[:, 1] * 210, gp[:, 1]) or np.allclose(path[:, 1] * 210, gp[:, 1], atol=1e-6)
        assert np.array_equal(path[:, 2], gp[:, 2]), name
        np.testing.assert_allclose(path[:, 0] * 210, gp[:, 0], rtol=0, atol=1e-7)
        np.testing.assert_allclose(path[:, 3], gp[:, 3], rtol=0, atol=1e-9)
        np.testing.assert_allclose(nx, g["nodes_x"], rtol=0, atol=1e-9)
        np.testing.assert_allclose(ny, g["nodes_y"], rtol=0, atol=1e-9)
        assert abs(sim - float(g["similarity"])) < 1e-9


def test_end_to_end_vs_oracle(gpu_ctx):
    """A pair that is not in the fixtures: CUDA path vs oracle on identical PCM."""
    from describealign_b200 import api, host_fit, synth
    from oracle import align_oracle as ao, features as of
    v, a = synth.make_pair(140.0, 9.0, skips=[(50.0, 2.0), (90.0, -3.0)], seed=77, ch=2)
    det = {}
    nx, ny, sim, path, med = api.align_pcm(v, a, details=det)
    V, A = of.all_features(v), of.all_features(a)
    odet = {}
    ox, oy, osim, opath, omed = ao.align(V, A, V[0], A[0], host_fit, details=odet)
    assert path.shape == opath.shape
    assert np.array_equal(path[:, 1], opath[:, 1]) and np.array_equal(path[:, 2], opath[:, 2])
    np.testing.assert_allclose(path[:, 0], opath[:, 0], rtol=0, atol=1e-9)
    np.testing.assert_allclose(path[:, 3:], opath[:, 3:], rtol=0, atol=1e-8)
    np.testing.assert_allclose(nx, ox, rtol=0, atol=1e-9)
    np.testing.assert_allclose(ny, oy, rtol=0, atol=1e-9)
    assert abs(sim - osim) < 1e-9 and med == omed


def test_mismatched_inputs_fail_like_the_reference(gpu_ctx):
    from describealign_b200 import api, synth
    v, _ = synth.make_pair(60.0, 1.0, seed=201)
    _, a = synth.make_pair(60.0, 1.0, seed=202)
    with pytest.raises(RuntimeError, match="Alignment failed, are the input files mismatched"):
        api.align_pcm(v, a)


def _random_stage_b_case(seed, n_a=9000, n_v=9000, n_cor=6, crossing=True, slopes=(0.7, 1.25)):
    """Synthetic pass-2 input: smooth random scaled features and hand-made corridors (different
    slopes so that lines cross and share cells, one line duplicated a quarter cell away so that
    the 'first cluster to claim (i, int(j)) wins' rule fires).  The audio is made to follow a
    different corridor in each stretch of ~600 rows, with short corrupted runs inside, so that
    the best path uses global jumps, same-cluster jumps and cross-cluster local steps."""
    rng = np.random.default_rng(seed)

    def feats(n):
        x = rng.standard_normal((n + 40, 3)).cumsum(axis=0)
        x = x[40:] - x[:-40]
        return np.ascontiguousarray((x / 6.0).astype(np.float32))
    audio, video = feats(n_a), feats(n_v)
    plans = []
    for k in range(n_cor):
        slope = float(rng.uniform(*slopes)) if crossing else 1.0
        offset = float(rng.uniform(4.0, 0.15 * n_v)) + (0.0 if crossing else 40.0 * k)
        if k == 2:                       # same line as corridor 1, shifted by a fraction of a cell
            slope, offset = plans[1][3], plans[1][4] + 0.25
        lo = int(rng.integers(0, n_a // 8))
        hi = int(rng.integers(7 * n_a // 8, n_a))
        lo = max(lo, int(np.ceil((4 - offset) / slope)), 0)
        hi = min(hi, int(np.floor((n_v - 4 - offset) / slope)))
        plans.append((k, lo, hi, slope, offset))
    seg = 600
    for s0 in range(0, n_a, seg):
        idx, lo, hi, slope, offset = plans[int(rng.integers(0, n_cor))]
        a0, a1 = max(s0, lo), min(s0 + seg, hi)
        if a1 - a0 < 50:
            continue
        rows = np.arange(a0, a1)
        y = slope * rows + offset
        f = np.floor(y).astype(np.int64)
        t = (y - f)[:, None]
        good = video[f] * (1 - t) + video[f + 1] * t + 0.01 * rng.standard_normal((a1 - a0, 3))
        b0 = int(rng.integers(0, a1 - a0 - 40))
        good[b0:b0 + 30] += rng.standard_normal((30, 3))          # a corrupted run: cluster jump
        audio[a0:a1] = good.astype(np.float32)
    # energy column: keep most frames within 2.5 of the maximum so that the gates stay open
    audio[:, 0] = np.clip(audio[:, 0], -1.0, 1.0)
    video[:, 0] = np.clip(video[:, 0], -1.0, 1.0)
    return audio, video, plans, n_cor


@pytest.mark.parametrize("seed,crossing", [(1, True), (2, True), (3, False), (4, True), (5, True)])
@pytest.mark.parametrize("impl", [0, 2])
def test_stage_b_adversarial_vs_oracle(gpu_ctx, seed, crossing, impl):
    """Corridor scoring + DP #2 + traceback on inputs built to hit the rare branches (crossing
    lines, shared cells, dropped duplicates, negative quals, cluster jumps), for the
    corridor-state DP and for the generic tree DP; both must equal the oracle bit for bit in the
    integer columns and to 1e-9 in the float ones.  impl 0 = scan kernel (product path),
    2 = generic tree DP."""
    from describealign_b200 import _cabi
    from oracle import align_oracle as ao
    audio, video, plans, n_clusters = _random_stage_b_case(seed, crossing=crossing)
    want = ao.stage_b(plans, n_clusters, audio, video)
    gpu_ctx.set_option("dp2_impl", impl)
    try:
        pair = _cabi.Pair(gpu_ctx)
        pair.stage_b(audio, video, plans, n_clusters)
        i, j, c, q = pair.points2()
        path = pair.path2()
        stats = pair.stats()
        pair.close()
    finally:
        gpu_ctx.set_option("dp2_impl", 0)
    assert np.array_equal(i, want["points_i"]) and np.array_equal(c, want["points_c"])
    np.testing.assert_array_equal(j, want["points_j"])
    np.testing.assert_allclose(q, want["points_q"], rtol=0, atol=1e-9)
    wp = want["path"]
    assert path.shape == wp.shape, (path.shape, wp.shape)
    np.testing.assert_array_equal(path[:, :3], wp[:, :3])
    np.testing.assert_allclose(path[:, 3:], wp[:, 3:], rtol=0, atol=1e-8)
    if impl != 2 and crossing:
        assert stats["n_dp2_neighbour"] > 0, "the test is meant to exercise the shared-cell branch"


@pytest.mark.parametrize("seed,slopes,n_v", [(11, (0.3, 0.6), 6000), (12, (1.8, 3.0), 30000), (13, (0.95, 1.05), 9000)])
@pytest.mark.parametrize("impl", [0, 2])
def test_stage_b_slopes_vs_oracle(gpu_ctx, seed, slopes, n_v, impl):
    """Shallow lines (several rows per prev_cache cell), steep lines (cells more than two apart,
    so no local step is possible) and near-parallel lines, against the oracle."""
    from describealign_b200 import _cabi
    from oracle import align_oracle as ao
    audio, video, plans, n_clusters = _random_stage_b_case(seed, n_v=n_v, slopes=slopes)
    want = ao.stage_b(plans, n_clusters, audio, video)
    gpu_ctx.set_option("dp2_impl", impl)
    try:
        pair = _cabi.Pair(gpu_ctx)
        pair.stage_b(audio, video, plans, n_clusters)
        i, j, c, q = pair.points2()
        path = pair.path2()
        pair.close()
    finally:
        gpu_ctx.set_option("dp2_impl", 0)
    assert np.array_equal(i, want["points_i"]) and np.array_equal(c, want["points_c"])
    np.testing.assert_array_equal(j, want["points_j"])
    wp = want["path"]
    assert path.shape == wp.shape, (path.shape, wp.shape)
    np.testing.assert_array_equal(path[:, :3], wp[:, :3])
    np.testing.assert_allclose(path[:, 3:], wp[:, 3:], rtol=0, atol=1e-8)


@pytest.mark.parametrize("seed,n_cor", [(21, 9), (22, 12), (23, 5)])
def test_stage_b_block_dp_many_corridors(gpu_ctx, seed, n_cor):
    """The block DP on a longer input where the audio follows a different corridor every ~600 rows:
    corridors overtake one another (leaders become followers and back), queried points see entries
    of the same block, and checks fail so that only a prefix of a block commits.  Against the
    oracle, and the counters show that most points went through blocks."""
    from describealign_b200 import _cabi
    from oracle import align_oracle as ao
    audio, video, plans, n_clusters = _random_stage_b_case(seed, n_a=30000, n_v=30000, n_cor=n_cor, crossing=False)
    want = ao.stage_b(plans, n_clusters, audio, video)
    pair = _cabi.Pair(gpu_ctx)
    pair.stage_b(audio, video, plans, n_clusters)
    path = pair.path2()
    stats = pair.stats()
    pair.close()
    wp = want["path"]
    assert path.shape == wp.shape, (path.shape, wp.shape)
    np.testing.assert_array_equal(path[:, :3], wp[:, :3])
    np.testing.assert_allclose(path[:, 3:], wp[:, 3:], rtol=0, atol=1e-8)
    # (corridor 2 duplicates corridor 1 a quarter cell away: their points are NEAR and stay on the one-point path)
    assert stats["n_dp2_run_points"] > 0.05 * stats["n_points2"], stats


def test_stage_b_scaling_on_device_equals_uploaded_arrays(gpu_ctx, golden_align):
    """The product's stage B (scaled features rebuilt on the device from 6 scalars, describealign.py:737-741)
    against dab_pair_stage_b with the host's numpy arrays and the corridors the product planned, on the same
    pair: both take the energy maxima on the device, so any difference would come from the scaling.
    Identical points, quals and path, with far fewer bytes uploaded."""
    from describealign_b200 import api, host_fit
    _, meta = golden_align
    v, a = golden_pair_pcm(meta, "pair_warp")
    job = api.AlignJob()
    try:
        job.load_pcm(v, a)
        job.device_stage_a()
        job.host_stage()
        job.device_stage_b()
        points_dev, path_dev = job.pair.points2(), job.path.copy()
        audio_scaled, video_scaled = host_fit.scale_features(job.video_features, job.audio_features, job.kept_x, job.kept_y)
        job.pair.stage_b(audio_scaled, video_scaled, job.pair.corridors(), len(job.clusters))
        points_host, path_host = job.pair.points2(), job.pair.path2()
    finally:
        job.close()
    for x, y in zip(points_dev, points_host):
        np.testing.assert_array_equal(x, y)
    np.testing.assert_array_equal(path_dev, path_host)
    assert 24 + 40 * len(job.lines) < audio_scaled.nbytes + video_scaled.nbytes


@pytest.mark.parametrize("case", ["pair_a", "pair_warp", "synthetic"])
def test_device_corridor_planning_vs_oracle(gpu_ctx, golden_align, case):
    """Corridor planning on the device (csrc/refine.cuh: row limits, sub-frame offset refinement, +-30 s
    extension, energy maxima; describealign.py:895-932) against the oracle's numpy / np.linalg.lstsq
    planning on the same clusters: identical row ranges and clusters, refined offsets within 1e-9 (the
    device divides float64 sums instead of calling LAPACK), identical integer path columns."""
    from describealign_b200 import api, host_fit, synth
    from oracle import align_oracle as ao
    if case == "synthetic":
        v, a = synth.make_pair(200.0, 11.0, skips=[(60.0, 3.0), (130.0, -2.0)], seed=88)
    else:
        _, meta = golden_align
        v, a = golden_pair_pcm(meta, case)
    job = api.AlignJob()
    try:
        job.load_pcm(v, a)
        job.device_stage_a()
        job.host_stage()
        job.device_stage_b()
        cor_dev, path_dev = job.pair.corridors(), job.path.copy()
        audio_scaled, video_scaled = host_fit.scale_features(job.video_features, job.audio_features, job.kept_x, job.kept_y)
        want = [p for p in ao.plan_corridors(job.clusters, audio_scaled, video_scaled) if p[2] > p[1]]
        offsets0 = [c[1] for c in job.clusters]
        job.pair.stage_b(audio_scaled, video_scaled, want, len(job.clusters))
        path_host = job.pair.path2()
    finally:
        job.close()
    assert len(cor_dev) == len(want)
    refined = 0
    for got, w in zip(cor_dev, want):
        assert got[0] == w[0] and got[1] == w[1] and got[2] == w[2], (got, w)
        assert got[3] == w[3]
        assert abs(got[4] - w[4]) <= 1e-9 * max(1.0, abs(w[4])), (got, w)
        refined += int(w[4] != offsets0[w[0]])
    assert path_dev.shape == path_host.shape
    np.testing.assert_array_equal(path_dev[:, 1:3], path_host[:, 1:3])
    np.testing.assert_allclose(path_dev[:, 0], path_host[:, 0], rtol=0, atol=1e-8)
    np.testing.assert_allclose(path_dev[:, 3:], path_host[:, 3:], rtol=0, atol=1e-6)
    if case == "synthetic":
        assert refined >= 0     # (whether the refinement fires depends on the pair; the offsets agree either way)


def test_end_to_end_dp2_variants_agree(gpu_ctx, golden_align):
    """Same pair through both pass-2 DPs: identical paths (the scan DP is the product path;
    the tree DP is the generic fallback)."""
    from describealign_b200 import api
    _, meta = golden_align
    v, a = golden_pair_pcm(meta, "pair_warp")
    out = []
    for impl in (0, 2):
        api.context().set_option("dp2_impl", impl)
        try:
            out.append(api.align_pcm(v, a))
        finally:
            api.context().set_option("dp2_impl", 0)
    for other in out[1:]:
        np.testing.assert_array_equal(out[0][3], other[3])
        np.testing.assert_array_equal(out[0][0], other[0])
        np.testing.assert_array_equal(out[0][1], other[1])


def test_stage_a_row_shards_reassemble(gpu_ctx, golden_align):
    """Row-sharded match stage (the long-pair protocol, SURVEY.md 8e): the shards' match points,
    concatenated in row order and imported back, give the reference's pass-1 path."""
    from describealign_b200 import _cabi, batch
    from oracle import features as of
    data, meta = golden_align
    g = data["pair_a"]
    v, a = golden_pair_pcm(meta, "pair_a")
    V, A = of.all_features(v), of.all_features(a)
    pair = _cabi.Pair(gpu_ctx)
    pair.set_features(_cabi.VIDEO, V)
    pair.set_features(_cabi.AUDIO, A)
    parts = []
    for lo, hi in batch.row_shards(len(A[0]), 3):
        n = pair.stage_a_match(lo, hi)
        pi, pv, pq = pair.points1()
        assert len(pi) == n and (n == 0 or (pi.min() >= lo and pi.max() < hi))
        parts.append((pi, pv, pq))
    pi = np.concatenate([p[0] for p in parts]); pv = np.concatenate([p[1] for p in parts])
    pq = np.concatenate([p[2] for p in parts])
    assert np.array_equal(pi, g["points1_i"]) and np.array_equal(pv, g["points1_v"])
    np.testing.assert_allclose(pq, g["points1_q"], rtol=1e-12, atol=0)
    pair.import_points1(pi, pv, pq)
    pair.dp1()
    x, y = pair.path1()
    assert np.array_equal(x, g["path1_x"]) and np.array_equal(y, g["path1_y"])
    # a frame that is not a hashed video frame is rejected, not silently mapped
    bad = pv.copy(); bad[0] = bad[0] + 1 if bad[0] + 1 not in set(pv[:50].tolist()) else bad[0] + 2
    with pytest.raises(_cabi.DabError):
        pair.import_points1(pi, bad, pq)
    pair.close()


def test_stage_b_row_shards_reassemble(gpu_ctx, golden_align):
    """Row-sharded corridor scoring (the long-pair protocol, SURVEY.md 8e): two pairs holding the same
    features score disjoint audio-row ranges; their qual slices, concatenated in row order and imported
    into one of them, give the path of the unsharded stage B."""
    from describealign_b200 import api
    _, meta = golden_align
    v, a = golden_pair_pcm(meta, "pair_warp")
    jobs = [api.AlignJob(), api.AlignJob()]
    try:
        for job in jobs:
            job.load_pcm(v, a)
            job.device_stage_a()
        jobs[0].host_stage()
        b = jobs[0].stage_b_input()
        want_path = jobs[0].device_stage_b().copy()
        want_q = jobs[0].pair.points2()[3]
        mid = b["n_audio"] // 2 + 17
        parts, total = [], None
        for job, (lo, hi) in zip(jobs, ((0, mid), (mid, b["n_audio"]))):
            n2, first, mine = job.pair.stage_b_score(b["gains"], b["audio_stds"], b["n_audio"], b["n_video"], b["lines"], lo, hi)
            assert total is None or total == n2
            total = n2
            parts.append((first, job.pair.export_quals2(first, mine)))
        assert parts[0][0] == 0 and parts[1][0] == len(parts[0][1]) and len(parts[0][1]) + len(parts[1][1]) == total
        assert len(parts[0][1]) > 0 and len(parts[1][1]) > 0
        q_all = np.concatenate([p[1] for p in parts])
        np.testing.assert_array_equal(q_all, want_q)
        # before the import, the second pair's own quals are zero outside its rows
        assert np.all(jobs[1].pair.points2()[3][:parts[1][0]] == 0.0)
        jobs[1].pair.import_quals2(q_all)
        jobs[1].pair.dp2()
        np.testing.assert_array_equal(jobs[1].pair.path2(), want_path)
    finally:
        for job in jobs:
            job.close()


def test_long_pair_two_gpus():
    """align_long_pair under torchrun with NCCL (needs 2 GPUs; the 1-GPU box skips it)."""
    import subprocess, sys, os
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    res = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                          "--master-addr", "127.0.0.1", "--master-port", "29533",
                          os.path.join(root, "tools", "run_long_pair.py"), "--seconds", "240", "--check"],
                         capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-2000:]
    assert "long pair ok" in res.stdout


@pytest.mark.parametrize("name,scale", [("C1", 1.0), ("C3", 0.12), ("C4", 0.05)])
def test_baseline_config_shapes_vs_oracle(gpu_ctx, name, scale):
    """BASELINE.json's other configurations (trimmed-media stand-in at full size; the stereo
    --stretch_audio shape and a batch episode at reduced length) through the public API against
    the oracle on identical PCM."""
    from describealign_b200 import api, host_fit, synth
    from oracle import align_oracle as ao, features as of
    v, a = synth.config_pair(name, 3, scale)
    nx, ny, sim, path, med = api.align_pcm(v, a)
    V, A = of.all_features(v), of.all_features(a)
    ox, oy, osim, opath, omed = ao.align(V, A, V[0], A[0], host_fit)
    assert path.shape == opath.shape
    assert np.array_equal(path[:, 1], opath[:, 1]) and np.array_equal(path[:, 2], opath[:, 2])
    np.testing.assert_allclose(path[:, 0], opath[:, 0], rtol=0, atol=1e-9)
    np.testing.assert_allclose(nx, ox, rtol=0, atol=1e-9)
    np.testing.assert_allclose(ny, oy, rtol=0, atol=1e-9)
    assert abs(sim - osim) < 1e-9 and med == omed
    # start offset as the reference's report prints it (describealign.py:211-214)
    assert round(float(ny[0] - nx[0]), 4) == round(float(oy[0] - ox[0]), 4)


def test_full_size_pair_properties_and_concurrency(gpu_ctx):
    """BASELINE.json's headline shape (C2, 22-min video / 27-min description) at full size: size-independent
    properties of the result (the oracle takes too long here; bench.py compares one such pair with it in every
    run) and 12 copies of the pair in flight at once - own streams, polling host waits, mapped count
    read-backs - returning bit-identical results."""
    from describealign_b200 import api, batch, synth
    v, a = synth.config_pair("C2", 5, 1.0)
    nx, ny, sim, path, med = api.align_pcm(v, a)
    n_a, n_v = a.shape[0] // 210, v.shape[0] // 210
    assert len(path) >= max(min(n_a, n_v) / 500, 1050)                    # describealign.py:991-992
    assert np.all(np.diff(path[:, 1]) >= 0) and np.all(np.diff(path[:, 0]) >= 0)   # the chain never goes back
    assert path[:, 1].min() >= 0 and path[:, 1].max() * 210 < n_a and path[:, 0].max() * 210 < n_v
    assert np.all(np.diff(nx) >= 0) and 0 < sim <= 100
    assert abs((ny[0] - nx[0]) + 202.0) < 1.0                             # the 202 s start offset of the shape
    again = api.align_pcm(v, a)                                           # idempotent, buffers reused
    for x, y in zip((nx, ny, path), (again[0], again[1], again[3])):
        np.testing.assert_array_equal(x, y)
    res = batch.run_local([(v, a)] * 12, in_flight=12)
    for r in res:
        assert not isinstance(r, Exception), r
        np.testing.assert_array_equal(r[0], nx); np.testing.assert_array_equal(r[1], ny)
        np.testing.assert_array_equal(r[3], path)
        assert r[2] == sim and r[4] == med


def test_batch_run_local_matches_sequential(gpu_ctx):
    """Several pairs in flight on one GPU (batch.run_local, one CUDA stream per pair) give the
    results of running them one after the other; a mismatched pair yields its exception."""
    from describealign_b200 import api, batch, synth
    specs = [(45.0, 4.0, [(20.0, 1.5)], 11), (75.0, 6.0, [(30.0, 2.0)], 7), (40.0, 3.0, [], 12), (60.0, 2.0, [(25.0, -1.0)], 14)]
    pairs = [synth.make_pair(vs, off, skips=sk, seed=sd) for vs, off, sk, sd in specs]
    bad_v, _ = synth.make_pair(60.0, 1.0, seed=201)
    _, bad_a = synth.make_pair(60.0, 1.0, seed=202)
    pairs.append((bad_v, bad_a))
    got = batch.run_local(pairs, in_flight=4)
    assert isinstance(got[-1], RuntimeError) and "Alignment failed" in str(got[-1])
    for pair, res in zip(pairs[:-1], got[:-1]):
        assert not isinstance(res, Exception), res
        want = api.align_pcm(*pair)
        np.testing.assert_array_equal(res[0], want[0])
        np.testing.assert_array_equal(res[1], want[1])
        np.testing.assert_array_equal(res[3], want[3])
        assert res[2] == want[2] and res[4] == want[4]
    assert batch.align_batch(pairs[:2], in_flight=2)[1][2] == got[1][2]     # world size 1: no process group needed
