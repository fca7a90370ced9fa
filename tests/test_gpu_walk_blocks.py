"""The parallel-in-time walk (recover.cu: k_walk_pick, k_walk_q<NIT>, k_walk_fix<NIT>) against the C oracle.

From N = 1024 sites on, the fixed-point walk (1 <= L <= 32, L <= W) cuts the region into blocks that are walked at the
same time from guessed histories: the majority allele `warm` sites before the block, and up to five earlier haplotypes.
k_walk_fix accepts a block whose guessed history equals the final path on the L sites before it, and walks any other
block again from the final path until it falls in step with a speculative walk on L consecutive sites.  Every case here
asserts that it really runs in block mode, compares the haplotypes, their statistics and the reweighted band with the
oracle loop of gretel/cmd.py:148-161, and checks the redo counter against what the speculation must have done: the oracle
knows the true path, so which speculative starts failed can be worked out on the host (_speculation)."""
import ctypes as C
import json
import os
import subprocess
import sys
import textwrap

import numpy as np
import pytest

from gretel_b200 import synth
from tests.test_gpu_recover_switches import same_stats

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MAX_K = 40                       # SNPs per read: the band is 39 wide, so every L <= 32 takes the fixed-point walk
N_CAND = 5                       # earlier haplotypes a block may start from (HX_WALK_CAND - 1)


# ---- cases ---------------------------------------------------------------------------------------------------------
def case(band, N, W, L, v_site="from", skip_unsym=True):
    return dict(band=band, N=N, W=W, L=L, v_site=v_site, skip_unsym=skip_unsym)


def thin_band(c_oracle, seed, N, n_reads, p_special=0.05):
    """Random reads of up to MAX_K SNPs, any code: thin evidence, so exact ties between candidates are frequent.  Two
    reads of random alleles at each end of the region keep its first and last sites covered."""
    rng = np.random.default_rng(seed)
    rank, off, codes = synth.random_packed(rng, N, n_reads, MAX_K, p_special=p_special)
    rank = np.concatenate([rank, np.array([0, 0, N - MAX_K, N - MAX_K], np.int32)])
    off = np.concatenate([off, off[-1] + MAX_K * np.arange(1, 5)])
    codes = np.concatenate([codes, rng.integers(0, 4, 4 * MAX_K).astype(np.uint8)])
    band, _ = c_oracle.ingest(rank, off, codes, N, MAX_K - 1)
    return band.astype(np.float32)


def make_strains(rng, N, n_strains, shared=()):
    """[n_strains][N] alleles of sites 1..N, different for every strain at every site except in the `shared`
    stretches (first, last site), where all strains carry the alleles of strain 0."""
    strains = np.stack([rng.permutation(4)[:n_strains] for _ in range(N)], axis=1).astype(np.uint8)
    for a, b in shared:
        strains[:, a - 1:b] = strains[0, a - 1:b]
    return strains


def strain_reads(rng, strains, n_reads):
    """Error-free reads of 2..MAX_K SNPs from strains of equal abundance (full linkage), plus one read of every strain
    at each end of the region.  -> rank, off, codes."""
    S, N = strains.shape
    ks = rng.integers(2, MAX_K + 1, size=n_reads)
    ranks = np.array([rng.integers(0, N - k + 1) for k in ks])
    who = rng.integers(0, S, size=n_reads)
    ends = [(s, 0, MAX_K) for s in range(S)] + [(s, N - MAX_K, MAX_K) for s in range(S)]
    reads = sorted([(int(r), int(s), int(k)) for s, r, k in zip(who, ranks, ks)] + [(r, s, k) for s, r, k in ends])
    rank = np.array([r for r, _, _ in reads], np.int32)
    off = np.zeros(len(reads) + 1, np.int64)
    off[1:] = np.cumsum([k for _, _, k in reads])
    codes = np.concatenate([strains[s, r:r + k] for r, s, k in reads]).astype(np.uint8)
    return rank, off, codes


def strain_band(c_oracle, seed, N, n_strains, n_reads, shared=()):
    rng = np.random.default_rng(seed)
    strains = make_strains(rng, N, n_strains, shared)
    rank, off, codes = strain_reads(rng, strains, n_reads)
    band, _ = c_oracle.ingest(rank, off, codes, N, MAX_K - 1)
    return band.astype(np.float32), strains


# ---- block geometry (launch_generate) -----------------------------------------------------------------------------
def geometry(N, L, blocks=24):
    """How launch_generate cuts the region; HX_WALK_BLOCKS=`blocks` (default 24; 1 = the sequential walk)."""
    warm = max(4 * L, 64)
    blk_len = max(-(-N // blocks), 2 * warm)
    return dict(N=N, L=L, nit=(L + 2) // 4, warm=warm, blk_len=blk_len, n_blocks=-(-N // blk_len))


def block_mode(N, W, L, blocks=24):
    return 1 <= L <= 32 and L <= W and N >= 1024 and blocks != 1


def blocks_of(geo):
    """(start, end) of the blocks b >= 1: the speculative ones."""
    N, blk = geo["N"], geo["blk_len"]
    return [(1 + b * blk, min(N, (b + 1) * blk)) for b in range(1, geo["n_blocks"])]


# ---- the oracle loop, and what the speculation must have done --------------------------------------------------------
def _pick(mask, w):
    """gretel.py:166-174: the first maximum among the candidates."""
    best = -1
    for s in range(7):
        if mask >> s & 1 and (best < 0 or w[s] > w[best]):
            best = s
    return best


def _speculation(c_oracle, cur, c, geo, path, earlier):
    """Which blocks b >= 1 no speculative walk started from the right history, for the walk of `path` over the band
    `cur`.  The majority-allele start walks the `warm` sites before the block from the per-site majority allele; an
    earlier haplotype is a start if it is among the N_CAND most recent distinct ones on the L sites before the block.
    -> (blocks whose majority start failed, blocks none of whose starts matched, whether distinct-filtering dropped a
    coinciding earlier haplotype somewhere)."""
    N, W, L = c["N"], c["W"], c["L"]
    counts = c_oracle.counts_all(cur, N, W)
    cand = counts[:, :7] > 0
    if c["skip_unsym"]:
        cand[:, [4, 6]] = False
    guess = np.argmax(np.where(cand, counts[:, :7], -1.0), axis=1).astype(np.uint8)
    guess[0] = 6
    c0_failed, failed, deduped = [], [], False
    for start, end in blocks_of(geo):
        s0, need = max(1, start - geo["warm"]), min(L, start - 1)
        hist = guess.copy()
        for snp in range(s0, start):
            mask, w, _ = c_oracle.edge_weights_at(cur, N, W, L, snp, hist, c["v_site"], c["skip_unsym"])
            assert mask, "a hole on a complete path"
            hist[snp] = _pick(mask, w)
        picked = []
        for p in earlier[::-1]:
            if len(picked) == N_CAND:
                break
            h = bytes(p[start - need:start])
            if h in picked:
                deduped = True
            else:
                picked.append(h)
        if np.array_equal(hist[start - need:start], path[start - need:start]):
            continue
        c0_failed.append((start, end))
        if bytes(path[start - need:start]) not in picked:
            failed.append((start, end))
    return c0_failed, failed, deduped


def oracle_loop(c_oracle, c, n, geo=None, keep=()):
    """The loop hx_recover keeps on the device, on the C oracle: generate_path, ratio = max(min marginal, 0.01),
    reweight_path, stop at a hole.  -> (haplotypes, hole site or None, {k: band after k haplotypes for k in keep})."""
    N, W, L = c["N"], c["W"], c["L"]
    cur, orig = c["band"].copy(), c["band"].copy()
    its, bands, hole = [], {}, None
    for it in range(n):
        if it in keep:
            bands[it] = cur.copy()
        pc, res = c_oracle.generate_path(cur, orig, N, W, L, c["v_site"], c["skip_unsym"])
        if pc is None:
            hole = res
            break
        spec = None
        if geo is not None:
            spec = _speculation(c_oracle, cur, c, geo, pc, [i["path"] for i in its])
        ratio = max(res[2], 0.01)
        removed = c_oracle.reweight_path(cur, N, W, pc, ratio)
        its.append(dict(path=pc, stats=(res[0], res[1], res[2], ratio, removed), spec=spec))
    bands[len(its)] = cur
    return its, hole, bands


def redo_bounds(c, its, resident):
    """Sites k_walk_fix must walk again for these haplotypes: every failed block is walked again until the walk agrees
    with a speculative one on L sites (or to its end), never a block that a speculative walk continues."""
    lo = hi = 0
    for i in its:
        for start, end in i["spec"][1 if resident else 0]:
            lo += min(c["L"], end - start + 1)
            hi += end - start + 1
    return lo, hi


# ---- the device -----------------------------------------------------------------------------------------------------
def device_matrix(c):
    from gretel_b200.hansel import Hansel, REF_SYMBOLS, REF_UNSYMBOLS
    h = Hansel.init_matrix(REF_SYMBOLS, REF_UNSYMBOLS, c["N"], band_w=c["W"])
    h.load_band(c["band"])
    h.L, h.v_site, h.candidates_skip_unsymbols = c["L"], c["v_site"], c["skip_unsym"]
    return h


def redone(h):
    """hx_debug_walk_redone: sites walked again by k_walk_fix, summed over every walk of the handle so far."""
    from gretel_b200 import _lib
    fn = C.CFUNCTYPE(C.c_int, C.c_void_p, C.POINTER(C.c_int))(("hx_debug_walk_redone", _lib.load()))
    n = C.c_int()
    _lib.check(fn(h._h, C.byref(n)))
    return n.value


def check_case(c_oracle, c, n_res=6, n_gen=2, blocks=24, hole=None):
    """Both device entry points against the oracle loop: recover_codes (resident, earlier haplotypes as starts) for
    n_res haplotypes and generate_path_codes + reweight_path_codes (no earlier haplotypes) for n_gen.  `hole`: the
    site where the oracle must stop after the haplotypes it found, or None for no hole.
    -> summary: geometry, haplotypes, redone sites per entry point and their bounds."""
    N, W, L = c["N"], c["W"], c["L"]
    geo = geometry(N, L, blocks)
    mode = block_mode(N, W, L, blocks)
    n = max(n_res, n_gen)
    its, o_hole, bands = oracle_loop(c_oracle, c, n, geo if mode else None, keep=(n_res, n_gen))
    assert o_hole == hole, "the oracle stops at %r, the case expects %r" % (o_hole, hole)

    h = device_matrix(c)
    orig = h.copy()
    r0 = redone(h)
    paths, stats = h.recover_codes(orig, n_res, 0.01)
    r_res = redone(h) - r0
    want = its[:n_res]
    assert len(paths) == len(want), "recover_codes found %d haplotypes, the oracle %d" % (len(paths), len(want))
    for k, (p, s, e) in enumerate(zip(paths, stats, want)):
        bad = np.flatnonzero(p != e["path"])
        assert bad.size == 0, "resident haplotype %d differs from site %d on (%d sites)" % (k, bad[0], bad.size)
        same_stats(s, e["stats"], N, W, "resident haplotype %d" % k)
    assert np.array_equal(h.band(), bands[len(want)]), "band after recover_codes"
    h.close()

    h = device_matrix(c)
    orig = h.copy()
    r_gen = []
    for k in range(n_gen):
        r0 = redone(h)
        got = h.generate_path_codes(orig)
        r_gen.append(redone(h) - r0)
        if k == len(its):
            assert got[0] is None and got[1] == o_hole, "generate_path_codes %r, the oracle's hole is at %r" % (
                got[:2], o_hole)
            assert r_gen[-1] == 0
            break
        assert got[0] is not None, "generate_path_codes reports a hole at %d, the oracle none" % got[1]
        bad = np.flatnonzero(got[0] != its[k]["path"])
        assert bad.size == 0, "haplotype %d differs from site %d on (%d sites)" % (k, bad[0], bad.size)
        ratio = max(got[3], 0.01)
        removed = h.reweight_path_codes(got[0], ratio)
        same_stats(got[1:] + (ratio, removed), its[k]["stats"], N, W, "haplotype %d" % k)
    assert np.array_equal(h.band(), bands[min(n_gen, len(its))]), "band after generate_path_codes"
    h.close()

    out = dict(geo, block_mode=mode, found=len(its), redone_resident=r_res, redone_single=sum(r_gen), its=its)
    if not mode:
        assert r_res == 0 and sum(r_gen) == 0
        return out
    done = its[:min(n_gen, len(its))]
    for k, (i, r) in enumerate(zip(done, r_gen)):
        lo, hi = redo_bounds(c, [i], resident=False)
        assert lo <= r <= hi, "haplotype %d: %d sites walked again, the speculation asks for %d..%d" % (k, r, lo, hi)
    lo, hi = redo_bounds(c, want, resident=True)
    assert lo <= r_res <= hi, "recover_codes: %d sites walked again, the speculation asks for %d..%d" % (r_res, lo, hi)
    out.update(bounds_single=redo_bounds(c, done, resident=False), bounds_resident=(lo, hi))
    return out


def report(name, s):
    print("WALK %s" % json.dumps(dict(case=name, **{k: v for k, v in s.items() if k != "its"})))


# ---- 1. every NIT and warm-up length in block mode ------------------------------------------------------------------
@pytest.mark.parametrize("L", range(1, 33))
def test_every_lookback_in_block_mode(c_oracle, L):
    """L = 1..32 covers k_walk_q / k_walk_fix for NIT 0..8 and warm = 64..128, on 8-20 blocks of 128-256 sites."""
    N = 2000 + 29 * L
    c = case(thin_band(c_oracle, 5100 + L, N, 6 * N), N, MAX_K - 1, L, v_site="to" if L % 2 else "from")
    geo = geometry(N, L)
    assert block_mode(N, c["W"], L) and 8 <= geo["n_blocks"] <= 24 and 128 <= geo["blk_len"] <= 256
    s = check_case(c_oracle, c, n_res=6, n_gen=2)
    assert s["found"] == 6
    report("L%d" % L, s)


# ---- 2. geometry edges ----------------------------------------------------------------------------------------------
def _edge_sizes():
    out = []
    for L, k in ((1, 10), (8, 9), (17, 9), (32, 5)):
        blk = 2 * max(4 * L, 64)
        for N in (1023, 1024, 1025, k * blk, k * blk + 1):
            out.append((L, N))
    return out + [(1, 3600)]                    # above 24 * 2 * warm: blocks of ceil(N / 24) sites


@pytest.mark.parametrize("L,N", _edge_sizes())
def test_block_geometry_edges(c_oracle, L, N):
    """The gate (N = 1023 walks sequentially, 1024 does not), a last block of one site, a last block that ends exactly
    at N, the 2 * warm floor of the block length and a block length above it."""
    geo = geometry(N, L)
    assert block_mode(N, MAX_K - 1, L) == (N >= 1024)
    if N >= 1024:
        assert geo["n_blocks"] > 1
        assert geo["blk_len"] == (2 * geo["warm"] if N <= 48 * geo["warm"] else -(-N // 24))
    c = case(thin_band(c_oracle, 7000 + N + L, N, 6 * N), N, MAX_K - 1, L, v_site="to" if L % 2 else "from")
    s = check_case(c_oracle, c, n_res=3, n_gen=2)
    assert s["found"] == 3
    report("L%d_N%d" % (L, N), s)


def test_geometry_edges_are_reached():
    """The sizes above include every edge they are meant to."""
    sizes = _edge_sizes()
    ends = {(N - 1) % geometry(N, L)["blk_len"] for L, N in sizes if N >= 1024}
    assert 0 in ends                                           # last block of one site
    assert any(N % geometry(N, L)["blk_len"] == 0 for L, N in sizes)
    assert any(not block_mode(N, MAX_K - 1, L) for L, N in sizes)
    assert any(geometry(N, L)["blk_len"] > 2 * geometry(N, L)["warm"] for L, N in sizes)


# ---- 3. speculation fails: redo and join ----------------------------------------------------------------------------
def _strain_case(c_oracle, L, seed, n_strains=2, join=True):
    """Strains of equal abundance that differ at every site: the walk keeps to the strain it is on, and a block whose
    majority-allele start settled on another strain than the path fails.  With `join`, every odd block has a stretch
    of L + 4 sites, shortly after its start, where all strains agree: a walk that is redone there falls in step with
    the speculative walks after it."""
    N = 2400
    geo = geometry(N, L)
    shared = [(s + 10, s + 13 + L) for s, _ in blocks_of(geo)[::2]] if join else []
    for a, b in shared:
        assert b < a - 10 + geo["warm"]                       # the next block's warm-up is not in the stretch
    band, strains = strain_band(c_oracle, seed, N, n_strains, 3 * N, shared)
    return case(band, N, MAX_K - 1, L), shared


@pytest.mark.parametrize("L,n_strains", [(1, 2), (6, 3), (20, 2)])
def test_failed_speculation_is_redone_and_joined(c_oracle, L, n_strains):
    c, shared = _strain_case(c_oracle, L, 300 + L, n_strains)
    s = check_case(c_oracle, c, n_res=6, n_gen=3)
    assert s["found"] == 6
    lo, hi = s["bounds_single"]
    assert hi > 0, "the majority-allele start never failed: the data does not test the redo"
    assert s["redone_single"] > 0 and s["redone_resident"] > 0
    # a failed block with a shared stretch is walked again only up to a join
    failed = [b for i in s["its"][:3] for b in i["spec"][0]]
    assert any(a <= st <= b for a, b in failed for st, _ in shared)
    assert s["redone_single"] < hi, "no redo was cut short by a join"
    report("strains_L%d" % L, s)


def test_failed_speculation_without_join(c_oracle):
    """No shared stretch: a block whose starts all failed is walked again to its end."""
    c, _ = _strain_case(c_oracle, 17, 411, 2, join=False)
    s = check_case(c_oracle, c, n_res=4, n_gen=2)
    assert s["bounds_single"][1] > 0 and s["redone_single"] == s["bounds_single"][1]
    report("strains_nojoin_L17", s)


@pytest.mark.parametrize("L", [8, 20])
def test_histories_that_differ_only_at_lookback_L(c_oracle, L):
    """Two strains that agree on the L - 1 sites before every block start, and on the L - 1 sites before the first
    point where a redone walk may join (max(L, 48) sites into the block), but not on the L-th site before either.  A
    speculative walk on the other strain then looks right on L - 1 sites and goes on along its own strain: only a
    check of all L sites tells it from the path."""
    N = 2400
    geo = geometry(N, L)
    first_join = max(L, 48) - 1
    shared = [r for s, _ in blocks_of(geo) for r in ((s - L + 1, s - 1), (s + first_join - L + 2, s + first_join))]
    band, _ = strain_band(c_oracle, 600 + L, N, 2, 3 * N, shared)
    s = check_case(c_oracle, case(band, N, MAX_K - 1, L), n_res=4, n_gen=2)
    assert s["found"] == 4
    failed = [b for i in s["its"][:2] for b in i["spec"][0]]
    assert failed and s["redone_single"] == s["bounds_single"][1]
    report("near_miss_L%d" % L, s)


# ---- 4. earlier haplotypes as starts --------------------------------------------------------------------------------
@pytest.mark.parametrize("L,n_strains", [(4, 3), (15, 4)])
def test_earlier_haplotypes_as_starts(c_oracle, L, n_strains):
    """12 haplotypes of 3-4 strains: from the sixth on k_walk_pick has more earlier haplotypes than starts, several
    of which agree before a block; blocks whose majority start failed are continued from an earlier haplotype."""
    N = 2300
    band, _ = strain_band(c_oracle, 500 + L, N, n_strains, 3 * N)
    c = case(band, N, MAX_K - 1, L)
    s = check_case(c_oracle, c, n_res=12, n_gen=2)
    assert s["found"] == 12
    its = s["its"]
    rescued = sum(len(i["spec"][0]) - len(i["spec"][1]) for i in its)
    assert rescued > 0, "no block was continued from an earlier haplotype"
    assert any(i["spec"][2] for i in its[N_CAND + 1:]), "no coinciding earlier haplotypes were filtered"
    report("earlier_L%d" % L, s)


# ---- 5. holes in block mode -----------------------------------------------------------------------------------------
def _hole_sites(geo):
    N, blk, warm = geo["N"], geo["blk_len"], geo["warm"]
    b = 3
    start = 1 + b * blk
    return [[1], [blk // 2], [start], [start + blk - 1], [start + 2 * blk - warm // 2], [N],
            [start + blk // 3, start + 3 * blk + 5], [blk // 3, start + 2 * blk]]


HOLE_L, HOLE_N = 12, 2000


@pytest.mark.parametrize("sites", _hole_sites(geometry(HOLE_N, HOLE_L)),
                         ids=["site1", "in_block0", "block_first", "block_last", "next_warmup", "siteN", "two",
                              "two_block0"])
def test_hole_in_block_mode(c_oracle, sites):
    """A site without candidates (its d = 1 cell zeroed): both entry points report the first one, and recover_codes
    leaves the band untouched."""
    N, L = HOLE_N, HOLE_L
    band = thin_band(c_oracle, 909, N, 6 * N)
    assert c_oracle.generate_path(band.copy(), band, N, MAX_K - 1, L)[0] is not None
    for p in sites:
        band[p + 1, 0] = 0.0                                  # cell (p, p+1): the counts of site p
    c = case(band, N, MAX_K - 1, L)
    s = check_case(c_oracle, c, n_res=3, n_gen=1, hole=min(sites))
    assert s["found"] == 0 and s["redone_single"] == 0
    report("hole_%s" % "_".join(map(str, sites)), s)


def test_hole_after_reweighting(c_oracle):
    """One strain, and below site P a two-SNP read per site that pairs the strain's allele with another allele at the
    next site.  Every site has one candidate, so the first haplotype has the minimum marginal 1, the ratio 1, and its
    reweighting empties every cell on it: from site P on no site keeps evidence, and the second haplotype stops at P,
    in block 5."""
    N, L, P = 1500, 8, 700
    rng = np.random.default_rng(17)
    x = make_strains(rng, N, 2)
    rank, off, codes = strain_reads(rng, x[:1], 2 * N)
    deco = np.array([[x[0, q - 1], x[1, q]] for q in range(1, P)], np.uint8)      # sites q, q+1 for q < P
    rank = np.concatenate([rank, np.arange(P - 1, dtype=np.int32)])
    off = np.concatenate([off, off[-1] + 2 * np.arange(1, P, dtype=np.int64)])
    codes = np.concatenate([codes, deco.ravel()])
    band, _ = c_oracle.ingest(rank, off, codes, N, MAX_K - 1)
    c = case(band.astype(np.float32), N, MAX_K - 1, L)
    geo = geometry(N, L)
    assert geo["n_blocks"] > 1 and (P - 1) // geo["blk_len"] == 5
    s = check_case(c_oracle, c, n_res=4, n_gen=2, hole=P)
    assert s["found"] == 1 and s["its"][0]["stats"][3] == 1.0
    report("hole_after_reweight", s)


# ---- 6. fixed-point range -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("L", [6, 20])
def test_block_walk_leaves_fixed_point_range(c_oracle, L):
    """Counts so large that a log10 term does not fit the fixed-point tables: every walk, speculative ones included,
    decides each site from the float64 terms."""
    N = 2100
    band = thin_band(c_oracle, 77 + L, N, 6 * N)
    band[band > 0] *= np.float32(1e17)
    band[10:N:97] *= np.float32(1e3)
    assert np.log10(band.max()) > 15
    s = check_case(c_oracle, case(band, N, MAX_K - 1, L), n_res=3, n_gen=2)
    assert s["found"] == 3
    report("fixed_point_L%d" % L, s)


# ---- 7. unsymbols as candidates -------------------------------------------------------------------------------------
def test_block_walk_keeps_unsymbols(c_oracle):
    N, L = 2200, 10
    band = thin_band(c_oracle, 4242, N, 6 * N, p_special=0.5)
    c = case(band, N, MAX_K - 1, L, skip_unsym=False)
    s = check_case(c_oracle, c, n_res=4, n_gen=2)
    assert s["found"] == 4
    assert any(np.isin(i["path"][1:], (4, 6)).any() for i in s["its"]), "no 'N' or '_' was chosen"
    report("keep_unsymbols_L%d" % L, s)


# ---- 8. forced block counts ------------------------------------------------------------------------------------------
def forced_cases(c_oracle):
    """A thin case and a strain case large enough that 2, 24, 64 and 1000 requested blocks give different cuts."""
    N = 9000
    yield "thin", case(thin_band(c_oracle, 8080, N, 6 * N), N, MAX_K - 1, 4, v_site="to")
    yield "strains", case(strain_band(c_oracle, 8081, N, 2, 3 * N)[0], N, MAX_K - 1, 5)


_FORCED = textwrap.dedent("""
    import hashlib, json, os, sys
    import numpy as np
    from oracle import c_oracle
    from tests import test_gpu_walk_blocks as t
    blocks = int(os.environ["HX_WALK_BLOCKS"])
    for name, c in t.forced_cases(c_oracle):
        try:
            s = t.check_case(c_oracle, c, n_res=4, n_gen=2, blocks=blocks)
        except AssertionError as e:
            print("FAIL %s: %s" % (name, str(e).splitlines()[0]))
            continue
        digest = hashlib.sha256(b"".join(i["path"].tobytes() for i in s.pop("its", []))).hexdigest()
        print("CASE " + json.dumps(dict(s, case=name, blocks=blocks, paths=digest)))
""")


def test_forced_block_counts(c_oracle):
    """HX_WALK_BLOCKS is read once per process, so each count runs in a fresh one.  Every count matches the oracle (and
    so every other count); with one block nothing is walked again."""
    runs = {}
    for blocks in (1, 2, 64, 1000):
        env = dict(os.environ, HX_WALK_BLOCKS=str(blocks), PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""))
        out = subprocess.run([sys.executable, "-c", _FORCED], capture_output=True, text=True, timeout=280, cwd=ROOT,
                             env=env)
        assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
        fails = [ln for ln in out.stdout.splitlines() if ln.startswith("FAIL")]
        assert not fails, "HX_WALK_BLOCKS=%d: %s" % (blocks, fails)
        for ln in out.stdout.splitlines():
            if ln.startswith("CASE "):
                s = json.loads(ln[5:])
                runs[(s["case"], blocks)] = s
                print("WALK " + ln[5:])
    for name in ("thin", "strains"):
        r = {b: runs[(name, b)] for b in (1, 2, 64, 1000)}
        assert len({s["paths"] for s in r.values()}) == 1
        assert not r[1]["block_mode"] and r[1]["redone_resident"] == r[1]["redone_single"] == 0
        assert [r[b]["n_blocks"] for b in (2, 64, 1000)] == [2, 64, 71]
