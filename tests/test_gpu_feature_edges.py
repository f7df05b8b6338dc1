"""Edges of the feature kernel against the oracle: the persistent tile loop, unaligned device PCM, the trailing
energy-only tile and extreme sample values.

`features_kernel` (csrc/features.cu) is persistent: min(tiles, 2 * sm_count) CTAs take tiles of FT output frames
from an atomic ticket.  A tile is staged by a bulk copy (mono interior tiles of 16-byte aligned PCM, issued during
the previous tile and completed on an mbarrier), by 16-byte thread loads, or element by element (edge tiles and
unaligned PCM).  The feature tests of test_gpu_parity.py use tracks short enough that no CTA takes a second tile.

CPU part: a model of the tile geometry, stated once from `Tile<CH>` and held to the source by regex, and checks
that every GPU case reaches the branch it is named for.  If the tiling changes, these fail instead of the case
table quietly drifting off the edges.

GPU part: every case against oracle.features.all_features on the same int16 PCM, with the bars of
test_gpu_parity.py: equal lengths; energy, zero crossings, band 0 and band 1 bit-identical; band 2 within 4 ulp.
(test_gpu_fullsize.py compares only the first four features; the long tracks here cover band 2 as well.)
"""
import functools
import os
import re

import numpy as np
import pytest

FEATURES_CU = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                           "describealign_b200", "csrc", "features.cu")
B200_SMS = 148

# ---- tile geometry of features_kernel (Tile<CH>, FH, PADS, bulk_ok, launch) -------------------------------------
FH = 8          # halo frames each side
PADS = 40       # halo samples each side


def tile_consts(ch):
    """(FT, NF, NS): output frames per tile, frames staged, samples staged."""
    ft = 100 if ch == 1 else 48
    nf = ft + 2 * FH
    return ft, nf, nf * 210 + 2 * PADS


def lengths(S):
    """(L, nb, Le): band / zero-crossing frames, 105-sample blocks, energy frames."""
    L, nb = S // 210, S // 105
    return L, nb, (nb + 1) // 2


def n_tiles(S, ch):
    L, _, Le = lengths(S)
    return -(-max(L, Le) // tile_consts(ch)[0])


def grid(S, ch, sms):
    return min(n_tiles(S, ch), 2 * sms)


def window(tile, ch):
    """[s, e): the samples tile `tile` stages (may reach below 0 and past the band signal)."""
    ft, _, ns = tile_consts(ch)
    s = (tile * ft - FH) * 210 - PADS
    return s, s + ns


def bulk_ok(tile, S, ch, aligned=True):
    """The tile is fetched by the bulk copy: mono, 16-byte aligned PCM, window inside [0, L * 210)."""
    if ch != 1 or not aligned or tile >= n_tiles(S, ch):
        return False
    s, e = window(tile, ch)
    return s >= 0 and e <= 210 * lengths(S)[0]


def bulk_tiles(S, ch):
    return [t for t in range(n_tiles(S, ch)) if bulk_ok(t, S, ch)]


def hbm_block_tiles(S, ch):
    """Tiles that read block 2L (the block past the band signal when S mod 210 >= 105) straight from the PCM."""
    L, nb, _ = lengths(S)
    if nb == 2 * L:
        return []
    ft, nf, _ = tile_consts(ch)
    return [t for t in range(n_tiles(S, ch)) if t * ft - FH <= L < t * ft - FH + nf]


def energy_only_tile(S, ch):
    """The index of the tile whose only output is the last energy value (Le = L + 1, L % FT == 0), or None."""
    L, _, Le = lengths(S)
    ft = tile_consts(ch)[0]
    return L // ft if Le == L + 1 and L % ft == 0 else None


def vector_group_straddles(S, tile, ch):
    """The 8-sample staging group of `tile` that holds sample L * 210 - 1 also holds samples past the band signal
    (so it is staged element by element)."""
    Sb = 210 * lengths(S)[0]
    return (Sb - window(tile, ch)[0]) % 8 != 0


def zc_chunk_starts(ch):
    """First sample of each of the four zero-crossing chunks of a frame (105 mono words of two samples, 210 stereo
    words of one (l, r) sample)."""
    nw = 105 if ch == 1 else 210
    return [(nw * c) // 4 * (2 if ch == 1 else 1) for c in range(4)]


# ---- case tables --------------------------------------------------------------------------------------------------
AMPS = (0, 3000, 32768)       # silence, +-3000, full scale


def persistent_len(ch, sms):
    """S of the persistent-loop track: 2 * (2 * sms) + 3 tiles, a half-full last tile and the trailing HBM block."""
    ft = tile_consts(ch)[0]
    return 210 * ((4 * sms + 3) * ft - ft // 2) + 150


def persistent_edges(ch, sms):
    """Segment edges: each tile boundary and each window start, shifted by -1, 0, +1 in turn."""
    ft = tile_consts(ch)[0]
    edges = []
    for t in range(1, n_tiles(persistent_len(ch, sms), ch)):
        d = t % 3 - 1
        edges += [t * ft * 210 + d, window(t, ch)[0] + d]
    return sorted(edges)


def noise_segments(S, ch, edges, seed, amps=AMPS):
    """Seeded noise whose amplitude changes at every edge (the next amplitude always differs from the last)."""
    rng = np.random.default_rng(seed)
    bounds = np.concatenate([[0], np.asarray(edges, np.int64), [S]])
    level = np.cumsum(rng.integers(1, len(amps), bounds.size - 1)) % len(amps)
    amp = np.repeat(np.asarray(amps, np.int64)[level], np.diff(bounds))
    x = rng.integers(-32768, 32768, (S, ch), dtype=np.int64)
    return np.clip((x * amp[:, None]) >> 15, -32768, 32767).astype(np.int16)


def length_table(ch, sms):
    """(name, S) for every L in {FT-1, FT, FT+1, 2FT, 2 sms FT, 2 sms FT + FT} and S mod 210 in {0, 1, 104, 105, 106,
    209}, the geometry-model lengths, and (stereo) S < 210."""
    ft = tile_consts(ch)[0]
    cases = []
    for lname, L in (("FT-1", ft - 1), ("FT", ft), ("FT+1", ft + 1), ("2FT", 2 * ft), ("2smFT", 2 * sms * ft),
                     ("2smFT+FT", 2 * sms * ft + ft)):
        for r in (0, 1, 104, 105, 106, 209):
            cases.append((f"ch{ch} L={lname} S%210={r}", 210 * L + r))
    cases += [(f"ch{ch} {name}", S) for name, S in model_lengths(ch).items()]
    if ch == 2:
        cases += [(f"ch2 S={S}", S) for S in (0, 1, 105, 209)]
    return cases


def model_lengths(ch):
    """Two lengths per channel count at the end of the staged data, with 209 samples behind the band signal that
    must not be staged.  A bulk window ends at 40 (mod 210), so it can never end exactly at L * 210: the tightest
    fit ends 170 samples before it (L = 3 FT + 9), and a frame less pushes that tile's window 40 samples past it,
    onto thread staging.  Stereo has no bulk copy: there the last 16-byte staging group ends exactly at L * 210
    (L = 3 FT + 8) or, a frame shorter, straddles it."""
    ft = tile_consts(ch)[0]
    if ch == 1:
        return {"bulk window tightest fit": 210 * (3 * ft + 9) + 209, "bulk window a frame shorter": 210 * (3 * ft + 8) + 209}
    return {"vector group ends at L*210": 210 * (3 * ft + 8) + 209, "vector group a frame shorter": 210 * (3 * ft + 7) + 209}


UNALIGNED_OFFSETS = (0, 1, 2, 3, 4, 7, 8)      # int16 / float16 elements past a 16-byte aligned allocation


def unaligned_len(ch):
    ft = tile_consts(ch)[0]
    return 210 * (4 * ft + 37) + 150


def all_int16_track(seed=11):
    """Mono: seeded permutations of all 65 536 int16 values, back to back, over 8 tiles: bulk tiles 1-6, edge
    tiles 0 and 7, and the trailing HBM block."""
    rng = np.random.default_rng(seed)
    S = 210 * 750 + 150
    every = np.arange(-32768, 32768, dtype=np.int64)
    x = np.concatenate([rng.permutation(every) for _ in range(-(-S // every.size))])[:S]
    return x.astype(np.int16)[:, None]


def f16_tie(x):
    """x (float32) lies exactly halfway between two neighbouring float16 values."""
    x = np.asarray(x, np.float32)
    h = x.astype(np.float16)
    other = np.nextafter(h, np.where(x > h.astype(np.float32), np.float16(np.inf), np.float16(-np.inf)))
    return (h.astype(np.float32) != x) & (np.abs(x - h.astype(np.float32)) == np.abs(other.astype(np.float32) - x))


def stereo_tie_track(seed=12):
    """Stereo: every (l, r) has a float16 mean (float32 (l + r) / 2 rounded to float16) on a rounding tie, from
    the binades above 2048 of both signs, and near +-32767 (where int16 -> float16 rounds to 32768)."""
    rng = np.random.default_rng(seed)
    S = 210 * (5 * 48 + 13) + 120
    out = []
    for lo, hi in ((2048, 4096), (4096, 8192), (8192, 16384), (16384, 32768), (32000, 32768)):
        m = rng.integers(lo, hi + 1, 4 * S)
        sign = rng.choice([-1, 1], m.size)
        l = np.clip(sign * m, -32768, 32767)
        r = np.clip(sign * np.clip(m + rng.integers(-64, 65, m.size), lo, hi), -32768, 32767)
        lf, rf = (c.astype(np.int16).astype(np.float16).astype(np.float32) for c in (l, r))
        keep = f16_tie((lf + rf) / np.float32(2))
        out.append(np.stack([l[keep], r[keep]], 1))
    pairs = np.concatenate(out)
    return pairs[rng.permutation(pairs.shape[0])[:S]].astype(np.int16)


def square_track(S, ch, period):
    x = np.where((np.arange(S) // period) % 2 == 0, 32767, -32768).astype(np.int16)
    return np.repeat(x[:, None], ch, 1)


def antiphase_track(S, seed=13):
    """Stereo l = -r at full scale (-(-32768) saturates to 32767): the mid signal is 0 whatever the energy."""
    l = np.random.default_rng(seed).integers(-32768, 32768, S)
    return np.stack([l, np.clip(-l, -32768, 32767)], 1).astype(np.int16)


def zero_run_track(ch, seed=14):
    """Negative noise with +0 runs that start and end on the first sample of a frame, on the zero-crossing chunk
    edges of a frame and on sample 0 of a tile: every sign change sits on one of those edges, except the end of
    a one-sample run that starts a tile."""
    rng = np.random.default_rng(seed)
    ft = tile_consts(ch)[0]
    L = 4 * ft + 21
    S = 210 * L + 150
    cand = [f * 210 + o for f in range(L) for o in zc_chunk_starts(ch)]
    toggles = set(rng.choice(cand, len(cand) // 3, replace=False).tolist())
    toggles |= {t * ft * 210 for t in range(1, n_tiles(S, ch))}
    toggles |= {t * ft * 210 + 1 for t in (2,)}                     # a one-sample run at a tile start
    bounds = np.array(sorted(toggles) + [S])
    zero = np.zeros(S, bool)
    for k in range(0, bounds.size - 1, 2):
        zero[bounds[k]:bounds[k + 1]] = True
    x = -rng.integers(1, 3001, (S, ch))
    x[zero] = 0
    return x.astype(np.int16)


def value_cases():
    """(name, int16 PCM) of the sample-value cases."""
    S1, S2 = 210 * (3 * 100 + 37) + 150, 210 * (3 * 48 + 37) + 150
    return [("all int16 values", all_int16_track()),
            ("stereo float16-mean ties", stereo_tie_track()),
            ("stereo full-scale square", square_track(S2, 2, 7)),
            ("stereo l = -r", antiphase_track(S2)),
            ("mono sign alternates every sample", square_track(S1, 1, 1)),
            ("stereo sign alternates every sample", square_track(S2, 2, 1)),
            ("mono zero runs", zero_run_track(1)),
            ("stereo zero runs", zero_run_track(2))]


# ---- CPU: the model agrees with features.cu ---------------------------------------------------------------------
def _source():
    with open(FEATURES_CU) as f:
        return f.read()


def test_geometry_model_matches_features_cu():
    src = _source()
    assert int(re.search(r"constexpr int FH = (\d+);", src).group(1)) == FH
    assert int(re.search(r"constexpr int PADS = (\d+);", src).group(1)) == PADS
    ft = re.search(r"static constexpr int FT = CH == 1 \? (\d+) : (\d+);", src)
    assert (int(ft.group(1)), int(ft.group(2))) == (tile_consts(1)[0], tile_consts(2)[0])
    assert re.search(r"static constexpr int NF = FT \+ 2 \* FH;", src)
    assert re.search(r"static constexpr int NS = NF \* 210 \+ 2 \* PADS;", src)
    # bulk_ok: mono, aligned, tile < tiles, window [s, s + NS) inside [0, Sb) with Sb = L * 210
    assert re.search(r"if \(CH != 1 \|\| !a\.vec_ok \|\| tile >= a\.tiles\) return false;\s*"
                     r"const int64_t s = \(tile \* FT - FH\) \* 210 - PADS;\s*return s >= 0 && s \+ NS <= Sb;", src)
    assert re.search(r"const int64_t Sb = a\.L \* 210;", src)
    # the launch: tiles cover max(L, Le) frames; the grid is min(tiles, 2 * sm_count)
    assert re.search(r"const int64_t L = tk\.S / 210, nb = tk\.S / 105, Le = \(nb \+ 1\) / 2;", src)
    assert re.search(r"const int64_t frames = Le > L \? Le : L;", src)
    assert re.search(r"const int64_t tiles = cdiv\(frames, Tile<CH>::FT\);", src)
    assert re.search(r"grid = tiles < 2 \* \(int64_t\)ctx->sm_count \? tiles : 2 \* \(int64_t\)ctx->sm_count;", src)
    # the block past the band signal is read from the PCM; zero-crossing chunks are (NW * c) / 4 words
    assert re.search(r"if \(\(b \+ 1\) \* 105 <= Sb\)", src)
    assert re.search(r"constexpr int NW = CH == 1 \? 105 : 210;", src)
    assert re.search(r"const int wlo = \(NW \* c\) / 4", src)


def test_geometry_model_facts():
    for ch in (1, 2):
        ft, nf, ns = tile_consts(ch)
        assert ns % 8 == 0
        # a bulk window always ends at 40 (mod 210): it can never end exactly at L * 210
        assert all(window(t, ch)[1] % 210 == PADS for t in range(50))
    assert lengths(210 * 1000 + 150) == (1000, 2001, 1001)
    assert n_tiles(210 * 1000 + 104, 1) == 10 and n_tiles(210 * 1000 + 105, 1) == 11
    assert energy_only_tile(210 * 1000 + 105, 1) == 10 and energy_only_tile(210 * 1000 + 104, 1) is None
    assert bulk_tiles(210 * 1000, 2) == [] and bulk_tiles(210 * 1000, 1) == list(range(1, 9))
    assert zc_chunk_starts(1) == [0, 52, 104, 156] and zc_chunk_starts(2) == [0, 52, 105, 157]


@pytest.mark.parametrize("ch", [1, 2])
def test_persistent_case_reaches_second_tiles(ch):
    S = persistent_len(ch, B200_SMS)
    tiles, ft = n_tiles(S, ch), tile_consts(ch)[0]
    assert tiles == 2 * (2 * B200_SMS) + 3 and tiles > 2 * grid(S, ch, B200_SMS)     # every CTA takes two tiles, some three
    L, _, Le = lengths(S)
    assert Le == L + 1 and L % ft != 0 and hbm_block_tiles(S, ch) == [tiles - 1]
    edges = persistent_edges(ch, B200_SMS)
    assert edges == sorted(set(edges)) and 0 < edges[0] and edges[-1] < S
    # every tile boundary and every window start, with -1, 0 and +1 each
    ts = 210 * ft
    near = lambda e, at: (e - at + ts // 2) % ts - ts // 2           # signed distance to the nearest at + k * ts
    assert {-1, 0, 1} <= {near(e, 0) for e in edges} and {-1, 0, 1} <= {near(e, window(0, ch)[0]) for e in edges}
    if ch == 1:
        # the window edges are those of bulk-copied tiles, and all tiles but the first and the last are bulk-copied
        bulk = bulk_tiles(S, 1)
        assert len(bulk) == tiles - 2
        on_bulk = {e - window(t, 1)[0] for e in edges for t in (round((e - window(0, 1)[0]) / ts),) if t in bulk}
        assert {-1, 0, 1} <= on_bulk
    pcm = noise_segments(S, ch, edges, seed=1)
    amp = np.abs(pcm.astype(np.int64)).max(1)
    bounds = np.concatenate([[0], edges, [S]])
    peaks = [amp[a:b].max() for a, b in zip(bounds[:-1], bounds[1:])]
    assert 0 in peaks and max(peaks) == 32768 and any(2000 < p <= 3000 for p in peaks)


@pytest.mark.parametrize("ch", [1, 2])
def test_length_table_reaches_branches(ch):
    ft = tile_consts(ch)[0]
    cases = dict(length_table(ch, B200_SMS))
    assert len(cases) == 36 + 2 + (4 if ch == 2 else 0)
    trailing = [n for n, S in cases.items() if energy_only_tile(S, ch) is not None]
    # the trailing energy-only tile: exactly the L % FT == 0 rows with S mod 210 >= 105 (and L = 0, S >= 105)
    assert sorted(trailing) == sorted([f"ch{ch} L={l} S%210={r}" for l in ("FT", "2FT", "2smFT", "2smFT+FT")
                                       for r in (105, 106, 209)] + (["ch2 S=105", "ch2 S=209"] if ch == 2 else []))
    for n in trailing:
        S = cases[n]
        L, _, Le = lengths(S)
        assert Le == L + 1 and L % ft == 0 and n_tiles(S, ch) == L // ft + 1
        assert n_tiles(S, ch) - 1 in hbm_block_tiles(S, ch)
    # at L = 2 sms FT the energy-only tile is the one tile a CTA takes second
    S = cases[f"ch{ch} L=2smFT S%210=105"]
    assert n_tiles(S, ch) == 2 * B200_SMS + 1 == grid(S, ch, B200_SMS) + 1
    assert n_tiles(cases[f"ch{ch} L=2smFT+FT S%210=105"], ch) == grid(S, ch, B200_SMS) + 2
    model = model_lengths(ch)
    if ch == 1:
        S, Sp = model["bulk window tightest fit"], model["bulk window a frame shorter"]
        t = max(bulk_tiles(S, 1))
        assert 210 * lengths(S)[0] - window(t, 1)[1] == 210 - PADS          # the least gap a window end can have
        assert lengths(Sp)[0] == lengths(S)[0] - 1 and not bulk_ok(t, Sp, 1) and t < n_tiles(Sp, 1)
        assert window(t, 1)[1] - 210 * lengths(Sp)[0] == PADS
        assert max(bulk_tiles(Sp, 1)) == t - 1
    else:
        S, Sp = model["vector group ends at L*210"], model["vector group a frame shorter"]
        last = n_tiles(S, 2) - 1
        assert not vector_group_straddles(S, last, 2) and vector_group_straddles(Sp, n_tiles(Sp, 2) - 1, 2)
        assert lengths(Sp)[0] == lengths(S)[0] - 1
        assert all(n_tiles(cases[f"ch2 S={s}"], 2) <= 1 for s in (0, 1, 105, 209))
    for S in model.values():
        assert S % 210 == 209 and n_tiles(S, ch) >= 4


@pytest.mark.parametrize("ch", [1, 2])
def test_unaligned_cases(ch):
    assert [k for k in UNALIGNED_OFFSETS if (2 * k) % 16 == 0] == [0, 8]
    S = unaligned_len(ch)
    assert n_tiles(S, ch) >= 5 and lengths(S)[2] == lengths(S)[0] + 1 and hbm_block_tiles(S, ch)
    if ch == 1:
        assert len(bulk_tiles(S, 1)) >= 2 and not any(bulk_ok(t, S, 1, aligned=False) for t in range(n_tiles(S, 1)))
    # the long case of the same test gives each CTA more than one tile
    assert n_tiles(persistent_len(ch, B200_SMS), ch) > 2 * grid(persistent_len(ch, B200_SMS), ch, B200_SMS)


def test_sample_value_cases():
    cases = dict(value_cases())
    x = cases["all int16 values"][:, 0]
    S = x.size
    assert np.unique(x).size == 65536 and S % 210 >= 105
    bulk = bulk_tiles(S, 1)
    assert len(bulk) >= 3 and hbm_block_tiles(S, 1) and n_tiles(S, 1) - 1 not in bulk and 0 not in bulk
    lo, hi = window(bulk[0], 1)[0], window(bulk[-1], 1)[1]
    assert np.unique(x[lo:hi]).size == 65536                      # every value through the bulk copy's conversion

    t = cases["stereo float16-mean ties"].astype(np.int16)
    lf, rf = (t[:, c].astype(np.float16).astype(np.float32) for c in (0, 1))
    mean = (lf + rf) / np.float32(2)
    assert f16_tie(mean).all()
    up = np.abs(mean.astype(np.float16).astype(np.float32)) > np.abs(mean)
    assert 0.2 < up.mean() < 0.8                                  # ties to even round both ways
    assert (np.abs(mean) > 2048).all() and (mean > 32700).any() and (mean < -32700).any()
    assert (t == 32767).any() and (t == -32768).any()
    assert n_tiles(t.shape[0], 2) >= 5

    a = cases["stereo l = -r"].astype(np.int64)
    assert (np.clip(-a[:, 0], -32768, 32767) == a[:, 1]).all() and (a[:, 0] == -32768).any()
    for name in ("mono sign alternates every sample", "stereo sign alternates every sample"):
        s = cases[name]
        assert ((s[1:] < 0) != (s[:-1] < 0)).all()

    for ch in (1, 2):
        z = cases[f"{'mono' if ch == 1 else 'stereo'} zero runs"]
        ft = tile_consts(ch)[0]
        assert (z <= 0).all() and ((z[:, 0] < 0) == (z[:, -1] < 0)).all()
        flips = np.flatnonzero((z[1:, 0] < 0) != (z[:-1, 0] < 0)) + 1       # first sample after each sign change
        starts = flips[z[flips, 0] == 0]
        ends = flips[z[flips, 0] < 0]
        for pos in (starts, ends):
            assert set(zc_chunk_starts(ch)) <= set((pos % 210).tolist())
            assert any(p % (210 * ft) == 0 for p in pos)                 # a run starts / ends on sample 0 of a tile
        assert lengths(z.shape[0])[2] == lengths(z.shape[0])[0] + 1


# ---- GPU ----------------------------------------------------------------------------------------------------------
NAMES = ("energy", "zero_crossings", "band0", "band1", "band2")


def _check_features(got, want, what):
    for k in range(5):
        assert got[k].shape == want[k].shape, f"{what}: {NAMES[k]} length {got[k].shape} != {want[k].shape}"
    for k in range(4):
        bad = np.flatnonzero(got[k] != want[k])
        assert bad.size == 0, (f"{what}: {NAMES[k]} differs at frames {bad[:8].tolist()} ({bad.size} of {got[k].size}): "
                               f"got {got[k][bad[:3]].tolist()}, want {want[k][bad[:3]].tolist()}")
    err = np.abs(got[4] - want[4])
    bad = np.flatnonzero(err > 4 * np.spacing(np.abs(want[4])))
    assert bad.size == 0, (f"{what}: band2 beyond 4 ulp at frames {bad[:8].tolist()} ({bad.size} of {got[4].size}), "
                           f"max err {err.max()}")


def _check_all(results):
    """results: (what, got, want); every case is checked before the first failure is reported."""
    fails = []
    for what, got, want in results:
        try:
            _check_features(got, want, what)
        except AssertionError as e:
            fails.append(str(e).split("\n")[0])
    assert not fails, f"{len(fails)} of {len(results)} cases differ from the oracle:\n" + "\n".join(fails)


@functools.lru_cache(maxsize=None)
def _sms():
    import torch
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


@functools.lru_cache(maxsize=None)
def _persistent(ch):
    S = persistent_len(ch, _sms())
    pcm = noise_segments(S, ch, persistent_edges(ch, _sms()), seed=ch)
    from oracle import features as of
    return pcm, of.all_features(pcm)


def _features(pair, track, pcm):
    pair.set_pcm(track, pcm)
    return pair.get_features(track)


def _fresh(ctx, pcm):
    from describealign_b200 import _cabi
    pair = _cabi.Pair(ctx)
    try:
        return _features(pair, _cabi.VIDEO, pcm)
    finally:
        pair.close()


@pytest.mark.gpu
@pytest.mark.parametrize("ch", [1, 2])
def test_persistent_loop(gpu_ctx, ch):
    """Every CTA takes two or three tiles: the bulk prefetch of the next tile, the mbarrier parity, the handover
    without a barrier after S4 and the reset of the zero-crossing counts of a reused CTA."""
    from describealign_b200 import _cabi
    from oracle import features as of
    pcm, want = _persistent(ch)
    assert n_tiles(pcm.shape[0], ch) > 2 * grid(pcm.shape[0], ch, _sms())
    rev = np.ascontiguousarray(pcm[::-1])
    want_rev = of.all_features(rev)
    f16 = pcm.astype(np.float16)
    res = []
    pair = _cabi.Pair(gpu_ctx)
    try:
        # one pair, four runs: the ticket and every output are rewritten by each
        res.append((f"ch{ch} int16", _features(pair, _cabi.VIDEO, pcm), want))
        res.append((f"ch{ch} float16", _features(pair, _cabi.VIDEO, f16), want))
        res.append((f"ch{ch} reversed", _features(pair, _cabi.VIDEO, rev), want_rev))
        res.append((f"ch{ch} int16 again", _features(pair, _cabi.VIDEO, pcm), want))
    finally:
        pair.close()
    # the audio track of a pair whose video track is shorter and has the other channel count
    short = noise_segments(unaligned_len(3 - ch), 3 - ch, [], seed=5)
    pair = _cabi.Pair(gpu_ctx)
    try:
        pair.set_pcm(_cabi.VIDEO, short)
        pair.set_pcm(_cabi.AUDIO, pcm)
        res.append((f"ch{ch} as audio", pair.get_features(_cabi.AUDIO), want))
        res.append((f"ch{ch} its video", pair.get_features(_cabi.VIDEO), of.all_features(short)))
    finally:
        pair.close()
    _check_all(res)


@pytest.mark.gpu
@pytest.mark.parametrize("ch", [1, 2])
def test_unaligned_device_pcm(gpu_ctx, ch):
    """The same samples at element offsets 0-8 of a device allocation, int16 and float16: offsets 0 and 8 take the
    16-byte and bulk paths, the others the element path; all equal the oracle."""
    import torch
    from describealign_b200 import _cabi
    from oracle import features as of
    S = unaligned_len(ch)
    pcm = noise_segments(S, ch, [210 * tile_consts(ch)[0] * t for t in range(1, n_tiles(S, ch))], seed=20 + ch)
    tracks = [(f"ch{ch} S={S}", pcm, of.all_features(pcm), UNALIGNED_OFFSETS)]
    big, big_want = _persistent(ch)
    tracks.append((f"ch{ch} persistent S={big.shape[0]}", big, big_want, (3, 8)))
    res = []
    for name, x, want, offsets in tracks:
        for fmt, dtype, host in ((_cabi.PCM_S16, torch.int16, x), (_cabi.PCM_F16, torch.float16, x.astype(np.float16))):
            flat = torch.from_numpy(np.ascontiguousarray(host).reshape(-1))
            buf = torch.empty(flat.numel() + 16, dtype=dtype, device="cuda")
            assert buf.data_ptr() % 16 == 0
            for k in offsets:
                buf.zero_()
                buf[k:k + flat.numel()].copy_(flat)
                torch.cuda.synchronize()          # the pair's stream reads the tensor
                pair = _cabi.Pair(gpu_ctx)
                try:
                    pair.set_pcm_device(_cabi.VIDEO, buf.data_ptr() + 2 * k, x.shape[0], ch, fmt)
                    res.append((f"{name} {dtype} offset {k}", pair.get_features(_cabi.VIDEO), want))
                finally:
                    pair.close()
    _check_all(res)


@pytest.mark.gpu
@pytest.mark.parametrize("ch", [1, 2])
def test_length_table(gpu_ctx, ch):
    """Around one and two tiles, one tile per CTA, and the trailing energy-only tile (L % FT == 0, S mod 210 >= 105)."""
    from oracle import features as of
    ft = tile_consts(ch)[0]
    res = []
    for i, (name, S) in enumerate(length_table(ch, _sms())):
        edges = [210 * ft * t for t in range(1, n_tiles(S, ch))]
        pcm = noise_segments(S, ch, edges, seed=100 * ch + i, amps=AMPS[1:])
        res.append((name, _fresh(gpu_ctx, pcm), of.all_features(pcm)))
    _check_all(res)


@pytest.mark.gpu
def test_sample_values(gpu_ctx):
    """Every int16 value, stereo means on float16 rounding ties, full scale, l = -r, a sign change on every sample
    and +0 runs on frame, chunk and tile edges; int16 and float16 input."""
    from oracle import features as of
    res = []
    for name, pcm in value_cases():
        want = of.all_features(pcm)
        res.append((f"{name} int16", _fresh(gpu_ctx, pcm), want))
        res.append((f"{name} float16", _fresh(gpu_ctx, pcm.astype(np.float16)), want))
    _check_all(res)
