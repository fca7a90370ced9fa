"""The read-support oracle (oracle/support_oracle.py) on hand-worked cases, and its numpy form against the literal
per-read loop.  Codes: A0 C1 G2 T3 N4 -5 _6; a read (r, c) has c[t] at site r+t+1."""
import numpy as np
import pytest

from gretel_b200 import synth
from oracle import support_oracle as so

A, C, G, T, N, DEL, GAP = range(7)
Q = 1 << 32


def run(haps, reads, max_mismatch=-1):
    """haps: lists of codes for sites 1..N; reads: (rank, [codes]).  Both oracles, checked equal."""
    haps = np.array([[GAP] + list(h) for h in haps], dtype=np.uint8)
    rank = np.array([r for r, _ in reads], dtype=np.int32)
    off = np.concatenate([[0], np.cumsum([len(c) for _, c in reads])]).astype(np.int64)
    codes = np.array([x for _, c in reads for x in c], dtype=np.uint8)
    got = so.assign(haps, rank, off, codes, max_mismatch)
    loop = so.assign_loop(haps, rank, off, codes, max_mismatch)
    for k in got:
        assert np.array_equal(np.asarray(got[k]), np.asarray(loop[k])), k
    return got


def check(res, unique, shared, share_q32, totals, best_mm, n_best, first_best):
    assert res["unique"].tolist() == unique
    assert res["shared"].tolist() == shared
    assert res["share_q32"].tolist() == share_q32
    assert (res["assigned"], res["uninformative"], res["over_limit"]) == totals
    assert res["best_mm"].tolist() == best_mm
    assert res["n_best"].tolist() == n_best
    assert res["first_best"].tolist() == first_best


def test_unique_best():
    res = run([[A, C, G, T], [A, C, G, A]], [(0, [A, C, G, T])])
    check(res, [1, 0], [0, 0], [Q, 0], (1, 0, 0), [0], [1], [0])


def test_two_way_tie():
    # the read ends before site 4, the only site where the haplotypes differ
    res = run([[A, C, G, T], [A, C, G, A]], [(0, [A, C])])
    check(res, [0, 0], [1, 1], [Q // 2, Q // 2], (1, 0, 0), [0], [2], [0])


def test_three_way_tie():
    haps = [[A, C, G, T], [T, C, G, T], [A, C, G, T], [A, C, G, T]]
    # haplotype 1 differs at site 1: B = {0, 2, 3}
    res = run(haps, [(0, [A, C])])
    assert Q // 3 == 1431655765
    check(res, [0, 0, 0, 0], [1, 0, 1, 1], [Q // 3, 0, Q // 3, Q // 3], (1, 0, 0), [0], [3], [0])
    # a read that starts after site 1 ties all four, each at one mismatch (site 3 is G, the read says A)
    res = run(haps, [(1, [C, A, T])])
    check(res, [0, 0, 0, 0], [1, 1, 1, 1], [Q // 4] * 4, (1, 0, 0), [1], [4], [0])


def test_uninformative_read():
    res = run([[A, C, G, T], [A, C, G, A]], [(0, [N, GAP, N]), (3, [])])
    check(res, [0, 0], [0, 0], [0, 0], (0, 2, 0), [-1, -1], [0, 0], [-1, -1])


def test_deletion_matches_deletion():
    res = run([[A, DEL, G, T], [A, C, G, T]], [(0, [A, DEL])])
    check(res, [1, 0], [0, 0], [Q, 0], (1, 0, 0), [0], [1], [0])


def test_haplotype_n_mismatches_informative_code():
    res = run([[N, C, G, T], [A, C, G, T]], [(0, [A]), (0, [N, C])])
    # read 0: N != A on haplotype 0; read 1: its N is not informative, C matches both
    check(res, [0, 1], [1, 1], [Q // 2, Q + Q // 2], (2, 0, 0), [0, 0], [1, 2], [1, 0])


@pytest.mark.parametrize("max_mismatch,totals,first", [(0, (0, 0, 1), -1), (1, (1, 0, 0), 0)])
def test_max_mismatch_boundary(max_mismatch, totals, first):
    res = run([[A, C, G, T], [G, G, G, G]], [(0, [C, C, G, T])], max_mismatch)
    assigned = totals[0]
    check(res, [assigned, 0], [0, 0], [Q * assigned, 0], totals, [1], [1], [first])


@pytest.mark.parametrize("seed", range(12))
def test_numpy_oracle_matches_loop(seed):
    rng = np.random.default_rng(seed)
    N = int(rng.integers(1, 90))
    H = int(rng.integers(1, 7))
    rank, off, codes = synth.random_packed(rng, N, int(rng.integers(0, 300)), min(40, N), p_special=0.3,
                                           sort=bool(seed % 2))
    haps = rng.integers(0, 7, size=(H, N + 1)).astype(np.uint8)
    if seed % 3 == 0:                      # few alleles: many ties
        haps = rng.integers(0, 2, size=(H, N + 1)).astype(np.uint8)
    mm = [-1, 0, 1, 3][seed % 4]
    a = so.assign(haps, rank, off, codes, mm)
    b = so.assign_loop(haps, rank, off, codes, mm)
    for k in a:
        assert np.array_equal(np.asarray(a[k]), np.asarray(b[k])), k
    assert a["assigned"] + a["uninformative"] + a["over_limit"] == len(rank)


def test_oracle_rejects_invalid_input():
    haps = np.array([[GAP, A, C]], dtype=np.uint8)
    with pytest.raises(ValueError):
        so.assign(haps, np.array([1], np.int32), np.array([0, 2]), np.array([A, C], np.uint8))
    with pytest.raises(ValueError):
        so.assign(haps, np.array([0], np.int32), np.array([0, 1]), np.array([7], np.uint8))
    with pytest.raises(ValueError):
        so.assign(np.array([[GAP, 7, C]], np.uint8), np.array([0], np.int32), np.array([0, 1]), np.array([A], np.uint8))
