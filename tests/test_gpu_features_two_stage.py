"""Edges of the 210 Hz feature kernel against the oracle.

Feature extraction runs as two kernels (csrc/features.cu).  `features_kernel` writes the per-frame intermediates of
frames [0, L) to a scratch buffer: 42 + 6 residual band energies, the band-2 frame energy, the zero-crossing count and
the two block energies of frames [0, Le).  `bands_kernel` is a plain grid of one CTA per FR output frames; a thread
takes one of the 48 phases for a run of TC frames, and its 15-tap window reaches 7 frames to each side, so an output
near a CTA edge reads frames that other CTAs own and an output near a track edge reads frames outside the scratch,
which must read as zero.

CPU part: the bands_kernel geometry, held to the source by regex, and checks that every GPU case reaches its edge.
GPU part: every case against oracle.features.all_features, int16 and float16 input, mono and stereo, with the bars of
test_gpu_parity.py (energy, zero crossings, bands 0 and 1 bit-identical; band 2 within 4 ulp).
"""
import re

import numpy as np
import pytest

from test_gpu_feature_edges import B200_SMS, FEATURES_CU, _check_all, lengths, noise_segments

FR = 32           # output frames per bands_kernel CTA
TC = 8            # frames per phase run
CTAS_PER_SM = 6   # __launch_bounds__ minimum: one wave is CTAS_PER_SM * sms CTAs
REACH = 7         # window frames each side of an output (15 taps)


def n_ctas(S):
    L, _, Le = lengths(S)
    return -(-max(L, Le) // FR)


def wave(sms):
    return CTAS_PER_SM * sms


def boundary_len():
    """S of a track over 6 CTAs plus 10 frames, with the trailing energy frame (S mod 210 = 150)."""
    return 210 * (6 * FR + 10) + 150


def boundary_edges(S):
    """Sample edges at every CTA's first frame, shifted by -1, 0, +1 frames in turn."""
    L = lengths(S)[0]
    edges = []
    for c in range(1, n_ctas(S)):
        f = c * FR + (c % 3 - 1)
        if 0 < f < L:
            edges.append(210 * f)
    return edges


SHORT_L = (0, 1, 7, 14, 15, 16)
SHORT_R = (0, 104, 105, 209)


def short_cases():
    """(name, S): L = 0, 1, 7, 14, 15, 16 with S mod 210 in {0, 104, 105, 209} (Le = L or L + 1)."""
    return [(f"L={L} S%210={r}", 210 * L + r) for L in SHORT_L for r in SHORT_R if 210 * L + r > 0]


def trailing_cases():
    """(name, S): Le = L + 1 with L a multiple of FR, so the last energy frame is frame 0 of a CTA of its own."""
    return [(f"L={k}FR S%210={r}", 210 * k * FR + r) for k in (1, 3) for r in (105, 150)]


def long_len(sms):
    """S of a track over two waves of bands_kernel CTAs and then some."""
    return 210 * ((2 * wave(sms) + 3) * FR + 5) + 60


# ---- CPU ----------------------------------------------------------------------------------------------------------
def test_bands_geometry_matches_features_cu():
    with open(FEATURES_CU) as f:
        src = f.read()
    assert int(re.search(r"constexpr int FR = (\d+);", src).group(1)) == FR
    assert int(re.search(r"constexpr int TC = (\d+);", src).group(1)) == TC
    assert re.search(r"constexpr int THREADS2 = 48 \* FR / TC;", src)
    assert int(re.search(r"__launch_bounds__\(THREADS2, (\d+)\) bands_kernel", src).group(1)) == CTAS_PER_SM
    assert re.search(r"bands_kernel<CH><<<\(unsigned\)cdiv\(frames, FR\), THREADS2, 0, pr->stream>>>", src)
    # the window: output t0 + tb + t reads frames t0 + tb + t - 7 .. + 7
    assert re.search(r"const int64_t fw = t0 \+ tb - 7;", src)
    assert FR % TC == 0 and FR % 32 == 0           # S4: one role per warp


def test_boundary_case_reaches_cta_edges():
    for ch in (1, 2):
        S = boundary_len()
        L, _, Le = lengths(S)
        assert n_ctas(S) == 7 and Le == L + 1
        shifts = {(e // 210) - round(e / 210 / FR) * FR for e in boundary_edges(S)}
        assert shifts == {-1, 0, 1}
        # every CTA edge is within one window's reach of a segment edge
        for c in range(1, n_ctas(S)):
            assert any(abs(e // 210 - c * FR) <= 1 for e in boundary_edges(S))


def test_short_cases_reach_track_edges():
    cases = dict(short_cases())
    Ls = {lengths(S)[0] for S in cases.values()}
    assert Ls == set(SHORT_L)
    # every short track sits in one CTA, and its outputs' windows reach past both ends of the track
    for S in cases.values():
        L, _, Le = lengths(S)
        assert n_ctas(S) <= 1 and L < 2 * REACH + 3
    assert {n for n, S in cases.items() if lengths(S)[2] == lengths(S)[0] + 1} == \
        {f"L={L} S%210={r}" for L in SHORT_L for r in (105, 209)}
    assert "L=0 S%210=0" not in cases and lengths(cases["L=0 S%210=105"]) == (0, 1, 1)


def test_trailing_cases_put_last_energy_frame_on_cta_edge():
    for name, S in trailing_cases():
        L, _, Le = lengths(S)
        assert Le == L + 1 and L % FR == 0 and n_ctas(S) == L // FR + 1


def test_long_case_exceeds_one_wave():
    S = long_len(B200_SMS)
    assert n_ctas(S) > 2 * wave(B200_SMS)


# ---- GPU ----------------------------------------------------------------------------------------------------------
def _run(ctx, pcm):
    from describealign_b200 import _cabi
    pair = _cabi.Pair(ctx)
    try:
        pair.set_pcm(_cabi.VIDEO, pcm)
        return pair.get_features(_cabi.VIDEO)
    finally:
        pair.close()


def _both_formats(ctx, name, pcm, res):
    from oracle import features as of
    want = of.all_features(pcm)
    res.append((f"{name} int16", _run(ctx, pcm), want))
    res.append((f"{name} float16", _run(ctx, pcm.astype(np.float16)), want))


@pytest.mark.gpu
@pytest.mark.parametrize("ch", [1, 2])
def test_cta_boundaries(gpu_ctx, ch):
    S = boundary_len()
    res = []
    _both_formats(gpu_ctx, f"ch{ch} CTA edges", noise_segments(S, ch, boundary_edges(S), seed=40 + ch), res)
    _check_all(res)


@pytest.mark.gpu
@pytest.mark.parametrize("ch", [1, 2])
def test_short_tracks(gpu_ctx, ch):
    res = []
    for i, (name, S) in enumerate(short_cases()):
        _both_formats(gpu_ctx, f"ch{ch} {name}", noise_segments(S, ch, [], seed=50 + 10 * ch + i), res)
    _check_all(res)


@pytest.mark.gpu
@pytest.mark.parametrize("ch", [1, 2])
def test_trailing_energy_frame(gpu_ctx, ch):
    res = []
    for i, (name, S) in enumerate(trailing_cases()):
        edges = [210 * f for f in range(FR, lengths(S)[0], FR)]
        _both_formats(gpu_ctx, f"ch{ch} {name}", noise_segments(S, ch, edges, seed=70 + 10 * ch + i), res)
    _check_all(res)


@pytest.mark.gpu
def test_longer_than_one_wave(gpu_ctx):
    import torch
    sms = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
    S = long_len(sms)
    assert n_ctas(S) > 2 * wave(sms)
    res = []
    for ch in (1, 2):
        _both_formats(gpu_ctx, f"ch{ch} two waves", noise_segments(S, ch, boundary_edges(S), seed=90 + ch), res)
    _check_all(res)
