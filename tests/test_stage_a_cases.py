"""The stage-A edge inputs of oracle/stage_a_cases.py have the properties the GPU tests rely on (CPU only).

DP 1 point sets: the oracle's prefix-max DP equals the literal frontier-list DP on them, and each set has the
rank / qual structure its builder claims.  Match-stage inputs: the oracle's candidate and table-entry counts are
above the first capacity guess of the match stage, so the GPU tests do reach its grow-and-retry path.
"""
from fractions import Fraction

import numpy as np
import pytest

from oracle import align_oracle as ao, features as of, stage_a_cases as sc


def _dp1(case):
    return ao.dp1(case["i"], case["v"], case["q"], case["Lv"])


def _small_cases():
    out = {"f1": sc.f1_fast_vs_tree(), "f1_mirror": sc.f1_mirror(), "f2": sc.f2_rounding("tie"),
           "f2_below": sc.f2_rounding("below"), "f3": sc.f3_tree(),
           "f4_superseded": sc.f4_superseded(), "f5_limit": sc.f5_limit()}
    for n in sc.F4_SIZES:
        out[f"f4_n{n}"] = sc.f4_small(n)
    for n in sc.F4_PATHS:
        out[f"f4_path{n}"] = sc.f4_path(n)
    out.update((name, build()) for name, build in sc.F6_CASES.items())
    return out


SMALL = _small_cases()


@pytest.mark.parametrize("name", sorted(SMALL))
def test_oracle_dp1_equals_literal_on_f_sets(oracle_lib, name):
    case = SMALL[name]
    assert sc.literal_small(case)
    px, pv, _, _ = _dp1(case)
    lit = ao.literal_dp1(zip(case["i"].tolist(), case["v"].tolist(), case["q"].tolist()))
    assert [(int(v), int(i)) for i, v in zip(px, pv)] == lit


def _serial(q):
    c = 0.0
    out = []
    for x in q.tolist():
        c = c + x
        out.append(c)
    return np.array(out)


def _tops_before(case, cum):
    """Rank of the frontier's top (largest cum, ties to the smallest rank) before each point."""
    r = case["v"] // 4
    tops, bc, br = [], 0.0, -1
    for k in range(len(r)):
        tops.append(br)
        if cum[k] > bc or (cum[k] == bc and r[k] < br):
            bc, br = cum[k], int(r[k])
    return np.array(tops)


@pytest.mark.parametrize("name", ["f1", "f1_mirror"])
def test_f1_chains_have_bit_equal_serial_sums(oracle_lib, name):
    case = SMALL[name]
    qa, qb = case["q"][case["chain_a"]], case["q"][case["chain_b"]]
    sa, sb = _serial(qa), _serial(qb)
    assert sa[-1].tobytes() == sb[-1].tobytes()
    r = case["v"] // 4
    assert r[case["chain_b"]].max() < r[case["chain_a"]].min()          # B left of A: B never chains from A
    _, _, cum, back = _dp1(case)
    np.testing.assert_array_equal(cum[case["chain_a"]], sa)
    np.testing.assert_array_equal(cum[case["chain_b"]], sb)
    tops = _tops_before(case, cum)
    assert np.all(r[case["chain_b"]] < tops[case["chain_b"]])           # every B point is a tree query
    assert np.all(r[case["chain_a"][1:]] >= tops[case["chain_a"][1:]])  # every A point extends the top
    px, pv, _, _ = _dp1(case)
    assert (pv // 4).tolist() == case["want_path_ranks"]
    if name == "f1_mirror":
        assert r[case["final"]] < tops[case["final"]]                   # the final point is a tree query


def i_of(case, idx):
    return case["i"][idx].tolist()


@pytest.mark.parametrize("name", ["f2", "f2_below"])
def test_f2_adds_in_the_binade_are_rounding_ties(oracle_lib, name):
    case = SMALL[name]
    chain = case["chain"]
    q = case["q"][chain]
    _, _, cum, back = _dp1(case)
    np.testing.assert_array_equal(cum[chain], _serial(q))
    assert np.array_equal(back[chain[1:]], chain[:-1]) and back[chain[0]] == -1
    prev = np.concatenate([[0.0], cum[chain][:-1]])
    u = Fraction(2) ** -39                      # the unit of [2^13, 2^14)
    ties, after_exact = 0, False
    for c0, qq, c1 in zip(prev.tolist(), q.tolist(), cum[chain].tolist()):
        c0, qq, c1 = Fraction(c0), Fraction(qq), Fraction(c1)
        assert qq.denominator in (2 ** 39, 2 ** 40)
        if 2 ** 13 <= c0 and c1 < 2 ** 14:
            if qq.denominator == 2 ** 39:       # exact, leaves an odd multiple of u
                assert c0 + qq == c1 and (c1 / u) % 2 == 1
            else:                               # halfway: the sum rounds to even, the qual alone to even
                assert abs(c1 - (c0 + qq)) == u / 2 and (qq / u - Fraction(1, 2)) % 2 == 0
                if after_exact:                 # from an odd multiple of u: the sum rounds up, the qual down
                    assert c1 - (c0 + qq) == u / 2
                    ties += 1
            after_exact = qq.denominator == 2 ** 39
        elif c1 < 2 ** 13:
            assert c0 + qq == c1
    assert ties > 75
    # the chain crosses 2^14 between two consecutive chain points (inside a run)
    k = int(np.argmax(cum[chain] >= 2.0 ** 14))
    assert chain[k] == chain[k - 1] + 1
    # runs start after each noise point, at offsets 30, 31, 0 and 1 of a warp batch; the first from the seed
    starts = {(int(n) + 1) % 32 for n in case["noise_at"]}
    assert starts == {30, 31, 0, 1}
    assert chain[0] == 0
    tops = _tops_before(case, cum)
    r = case["v"] // 4
    assert np.all(r[case["noise_at"]] < tops[case["noise_at"]])
    # chain B: tree queries, ending on A's serial sum (tie, B wins) or one ulp below it (A wins)
    b = case["chain_b"]
    assert np.all(r[b] < tops[b]) and back[b[0]] == -1
    a_end, b_end = cum[chain[-1]], cum[b[-1]]
    px, _, _, _ = _dp1(case)
    if name == "f2":
        assert b_end == a_end and px[:-1].tolist() == i_of(case, b)
    else:
        assert b_end == np.nextafter(a_end, 0.0) and px[:-1].tolist() == i_of(case, chain)


def test_f3_tree_structure(oracle_lib):
    case = SMALL["f3"]
    m = case["marks"]
    r = case["v"] // 4
    i = case["i"]
    _, _, cum, back = _dp1(case)
    tops = _tops_before(case, cum)
    assert r.max() >= 32 ** 3
    # predecessors in a block to the left at level 3, 2 and 1 (and in the same block one level up)
    for lvl, (x, j) in {3: ("x3", "j3"), 2: ("x2", "j2"), 1: ("x1", "j1")}.items():
        rx, rj = r[m[x]], r[m[j]]
        assert back[m[j]] == m[x], (lvl, back[m[j]])
        assert (rx >> (5 * lvl)) < (rj >> (5 * lvl)) and (rx >> (5 * lvl + 5)) == (rj >> (5 * lvl + 5))
        assert rj < tops[m[j]]
    # equal cums in different level-3 blocks, both seen by one tree query that takes the smaller rank
    assert cum[m["e1"]] == cum[m["e2"]] and (r[m["e1"]] >> 15) != (r[m["e2"]] >> 15)
    assert back[m["qe"]] == m["e1"] and r[m["qe"]] < tops[m["qe"]]
    # the same rank in consecutive rows
    assert r[m["s1"]] == r[m["s2"]] and i[m["s2"]] == i[m["s1"]] + 1 and back[m["s2"]] == m["s1"]
    # left of the top inside the top's own level-0 block
    lt = m["lt"]
    assert r[lt] < tops[lt] and (r[lt] >> 5) == (tops[lt] >> 5)


def test_f4_sizes_and_paths(oracle_lib):
    for n in sc.F4_SIZES:
        assert len(SMALL[f"f4_n{n}"]["i"]) == n
    for n in sc.F4_PATHS:
        px, _, _, _ = _dp1(SMALL[f"f4_path{n}"])
        assert len(px) == n
    case = SMALL["f4_superseded"]
    px, pv, _, _ = _dp1(case)
    assert len(px) == case["want_len"] and px[100] == 100 and px[101] == 600


def test_f6_paths_on_traceback_chunks(oracle_lib):
    """The oracle's path is each case's path_ids (a point's id is its row), placed on the chunks as named."""
    paths = {}
    for name in sc.F6_CASES:
        case = SMALL[name]
        assert np.array_equal(case["i"], np.arange(len(case["i"])))
        px, _, _, back = _dp1(case)
        assert px.tolist() == case["path_ids"].tolist(), name
        assert back[px[0]] == -1 and back[px[1:]].tolist() == px[:-1].tolist(), name
        paths[name] = px.tolist()
    c = sc.TB_CHUNK
    p = paths["f6_across"]
    for k in (c, 2 * c):
        assert k in p and p[p.index(k) - 1] == k - 1
    chunks = {x // c for x in paths["f6_skip"]}
    assert {1, 2, 3} & chunks == set() and min(chunks) == 0 and max(chunks) > 3
    assert (len(SMALL["f6_skip"]["i"]) - 1) // c not in chunks
    p, n = paths["f6_end_alone"], len(SMALL["f6_end_alone"]["i"])
    assert p[-1] == n - 1 and (n - 1) % c == 0 and p[-2] // c < p[-1] // c
    assert paths["f6_late_start"][0] >= c
    assert len(paths["f6_single"]) == 1


def test_f4_large_shape(oracle_lib):
    case = sc.f4_large()
    assert 1_900_000 <= len(case["i"]) <= 2_000_000
    assert (case["v"] // 4).max() < 150_000
    px, _, _, _ = _dp1(case)
    assert len(px) > 1000


def test_f5_tree_limit():
    at, over = sc.f5_limit(), sc.f5_limit(over=True)
    assert sc.vsel_ub(at["Le"]) == sc.DP_TREE_SLOTS and sc.vsel_ub(over["Le"]) == sc.DP_TREE_SLOTS + 1
    assert over["Le"] == at["Le"] + 1
    assert (at["v"] // 4).max() == at["top_rank"] == sc.DP_TREE_SLOTS - 2
    assert (over["v"] // 4).max() == over["top_rank"] == sc.DP_TREE_SLOTS - 1


def _match(V, A):
    pi, pv, pq, Lv, dbg = ao.match_points(V, A, V[0], A[0])
    e0, c0 = sc.stage_a_caps(len(V[0]), len(A[0]))
    return dbg, e0, c0


def test_m1_overflows_entries_and_candidates(oracle_lib):
    V, A = sc.m1_periodic()
    dbg, e0, c0 = _match(V, A)
    assert sc.expanded_entries(dbg["v_flags"], dbg["v_sel"]) > e0
    assert dbg["scored"] > c0
    full = np.mean([np.mean(fl[dbg["v_sel"]] == 127) for fl in dbg["v_flags"]])
    assert full >= 1 / 6


@pytest.mark.parametrize("name,factor", [("m2a", 1), ("m2b", 128), ("m3", 1)])
def test_pcm_cases_overflow_candidates(oracle_lib, name, factor):
    v, a = {"m2a": sc.m2a_tone, "m2b": sc.m2b_tone, "m3": sc.m3_loop}[name]()
    dbg, e0, c0 = _match(of.all_features(v), of.all_features(a))
    assert dbg["scored"] > factor * c0
