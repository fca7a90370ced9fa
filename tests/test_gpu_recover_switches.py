"""Recovery (recover.cu: k_walk_q, k_walk_q + k_walk_fix, k_walk_tables, k_walk_wide) under both arithmetic switches,
v_site ("from" / "to": HX_F_VSITE_TO) and candidates_skip_unsymbols (HX_F_KEEP_UNSYMBOLS), against the loop of
gretel/cmd.py:148-161 on the C oracle.

Every haplotype is compared in full: the path exactly; hp_current, hp_original, min_marginal and ratio bit for bit (both
sides take the same glibc log10 of the same marginals in the same site order); the removed mass within the rounding of
two summation orders of the same non-negative terms (`same_stats`); the band after the last reweighting bit for bit.
The resident loop (recover_codes, hx_recover) and the host loop (generate_path_codes + reweight_path_codes) are both
run, and agree with each other bit for bit.

Cases that need no GPU show that each case reaches what it is meant to: that its switches change the oracle's walk on
its data, that N or '_' is chosen where unsymbols are candidates, that every candidate's 10**x underflows at some site,
and that a weight overflows to inf (and normalising gives NaN) on the path."""
import ctypes as C
import functools

import numpy as np
import pytest

from gretel_b200 import synth
from oracle import hansel_oracle as o

FLAGS = {"from": ("from", True), "to": ("to", True), "from_keep": ("from", False), "to_keep": ("to", False)}
HX_MAX_L = 4095                 # HX_RING - 1: the deepest lookback the walk's history ring holds
SYM_N, SYM_GAP = 4, 6


# ---- bands ----------------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def _reads_band(seed, N, max_k, unsym, per_site=6, mono=0.0):
    """Random reads of up to max_k SNPs, any code, per_site * N of them, plus two reads at each end of the region; the band is
    max_k - 1 wide.  With `unsym`, evidence whose first symbol is N or '_' (which ingestion never writes) is added as a
    caller of add_observation could: at 40% of the sites a count up to half the site's total, so that N and '_' are
    candidates that can win, and in 15% of the lookback cells a few counts, so that a history holding them matters."""
    from oracle import c_oracle
    rng = np.random.default_rng(seed)
    k = min(max_k, N)
    rank, off, codes = synth.random_packed(rng, N, per_site * N, max_k, p_special=0.1)
    rank = np.concatenate([rank, np.array([0, 0, N - k, N - k], np.int32)])
    off = np.concatenate([off, off[-1] + k * np.arange(1, 5)])
    codes = np.concatenate([codes, rng.integers(0, 4, 4 * k).astype(np.uint8)])
    if mono:
        # a fraction `mono` of the sites carries A in every read: one valid symbol there (V = 1, log10(1 / V) = 0)
        site = np.repeat(rank.astype(np.int64), np.diff(off)) + np.arange(len(codes)) - np.repeat(off[:-1], np.diff(off))
        codes[(rng.random(N) < mono)[site]] = 0
    W = max_k - 1
    band = c_oracle.ingest(rank, off, codes, N, W)[0].astype(np.float32)
    if unsym:
        for p in np.flatnonzero(rng.random(N + 1) < 0.4):
            if p == 0:
                continue
            tot = float(band[p + 1, 0].sum())
            band[p + 1, 0, rng.choice((SYM_N, SYM_GAP)), rng.integers(0, 7)] += 1 + np.floor(rng.random() * tot / 2)
        for pj, d0 in zip(*np.nonzero(rng.random((N + 1, W)) < 0.15)):
            if d0 >= 1 and pj - d0 - 1 >= 0:
                band[pj, d0, rng.choice((SYM_N, SYM_GAP)), rng.integers(0, 7)] += rng.integers(1, 6)
    band.setflags(write=False)
    return band


def laplace_band(N, W, R, sigma, seed, s_star=3):
    """A run of R sites from N // 2 whose evidence is only N (V = 0 there), and the cells pairing each run site with
    every later site in the band given a support of `sigma` in column s_star alone.  Under v_site="from" each such
    lookback term of s_star is log10((1 + obs) / sigma); the other columns have a Laplace denominator of 0 and drop the
    term.  -> (band, first site after the run)."""
    band = _reads_band(seed, N, W + 1, False).copy()
    P = N // 2
    for p in range(P, P + R):
        for snp in range(p + 1, min(p + W, N) + 1):
            cell = band[snp, snp - p - 1]
            cell[:] = 0.0
            cell[SYM_N, s_star] = sigma
        band[p + 1, 0, SYM_N, SYM_N] = 10.0                        # the counts of site p: N only
    return band, P + R


def case(band, N, W, L, flags="from"):
    v_site, skip = FLAGS[flags]
    return dict(band=band, N=N, W=W, L=L, v_site=v_site, skip_unsym=skip)


# name -> (N, max_k, seed); the band of every matrix case carries unsymbol evidence
GEOMETRY = {"q_seq": (300, 40, 11), "q_blocks": (2100, 40, 12), "tables_in": (300, 61, 13), "narrow": (300, 6, 14),
            "narrow_long": (1100, 6, 15), "wide": (400, 170, 16), "wide_beyond": (800, 170, 77)}
MATRIX = [("q_seq", L) for L in (1, 4, 5, 17, 32)] + [("q_blocks", L) for L in (3, 16, 29)] + \
         [("tables_in", L) for L in (33, 47)] + [("narrow", L) for L in (6, 8, 17, 32, 40)] + \
         [("narrow_long", 17), ("q_seq", 0), ("wide", "W"), ("wide_beyond", 700)]


def matrix_case(name, L, flags):
    """wide_beyond: beyond the band a lookback term log10(1 / V) is the same for every candidate, so it can only
    change the walk by taking every candidate's 10**x below the smallest double.  Its band is thin, has one allele
    (V = 1, a term of 0) at half the sites and counts scaled by 1e30 (a pair never seen together gives a term of about
    -31), so that whether the in-band and the up to 530 beyond-band terms sum below -323 varies from site to site and
    depends on which site's V each beyond-band term takes."""
    N, max_k, seed = GEOMETRY[name]
    W = max_k - 1
    L = W if L == "W" else L
    if name != "wide_beyond":
        return case(_reads_band(seed, N, max_k, True), N, W, L, flags)
    band = _reads_band(seed, N, max_k, True, 1, 0.5).copy()
    band[band > 0] *= np.float32(1e30)
    return case(band, N, W, L, flags)


def walk_kernel(N, W, L):
    """Which walk launch_generate runs (recover.cu)."""
    if 1 <= L <= 32 and L <= W:
        return "q_blocks" if N >= 1024 else "q_seq"
    Lw = min(max(L, 1), W)
    return "wide" if (200 * 1024) // (3 * (Lw * 448 + 64)) < 1 else "tables"


# ---- the oracle loop and the comparison -----------------------------------------------------------------------------
def oracle_loop(c_oracle, c, n, min_remove=0.01, keep=()):
    """gretel/cmd.py:148-161 on the C oracle: generate_path, ratio = max(min marginal, min_remove), reweight_path, stop
    at a hole.  -> (haplotypes [(path, stats)], hole site or None, {k: band after k haplotypes} for k in keep that
    were reached and for the last one)."""
    N, W, L = c["N"], c["W"], c["L"]
    cur, orig = c["band"].copy(), c["band"]
    its, hole, bands = [], None, {}
    for k in range(n):
        if k in keep:
            bands[k] = cur.copy()
        pc, res = c_oracle.generate_path(cur, orig, N, W, L, c["v_site"], c["skip_unsym"])
        if pc is None:
            hole = res
            break
        ratio = max(res[2], min_remove)
        removed = c_oracle.reweight_path(cur, N, W, pc, ratio)
        its.append((pc, (res[0], res[1], res[2], ratio, removed)))
    bands[len(its)] = cur
    return its, hole, bands


def _bits(x):
    return np.asarray(x, dtype=np.float64).view(np.uint64)


def same_stats(got, exp, N, W, what=""):
    """hp_current, hp_original, min_marginal and ratio bit for bit (-inf included).  removed: both sides add the same
    non-negative per-cell terms, at most n = (N + 1) * (W + 1) of them, the oracle in call order and the device in a
    tree; each sum is within (n - 1) * 2^-53 of the exact one, relative, so they differ by at most 2 n 2^-53 removed."""
    names = ("hp_current", "hp_original", "min_marginal", "ratio")
    for k in range(4):
        assert _bits(got[k]) == _bits(exp[k]), "%s %s: %r != %r" % (what, names[k], got[k], exp[k])
    n = (N + 1) * (W + 1)
    assert abs(got[4] - exp[4]) <= 2 * n * 2.0 ** -53 * exp[4], "%s removed: %r != %r" % (what, got[4], exp[4])


def same_band(got, exp, what):
    assert np.array_equal(got.view(np.uint32), exp.view(np.uint32)), what


def device_matrix(c):
    from gretel_b200.hansel import Hansel, REF_SYMBOLS, REF_UNSYMBOLS
    h = Hansel.init_matrix(REF_SYMBOLS, REF_UNSYMBOLS, c["N"], band_w=c["W"])
    h.load_band(c["band"])
    h.L, h.v_site, h.candidates_skip_unsymbols = c["L"], c["v_site"], c["skip_unsym"]
    return h


def check(c_oracle, c, n_res=4, n_gen=2, min_remove=0.01, make=device_matrix):
    """Both device entry points against the oracle loop: recover_codes for n_res haplotypes, generate_path_codes +
    reweight_path_codes for n_gen; the stats and band after each; the two against each other.
    -> (oracle haplotypes, oracle hole, recover_codes' stats, recover_codes' band)."""
    N, W = c["N"], c["W"]
    its, hole, bands = oracle_loop(c_oracle, c, max(n_res, n_gen), min_remove, keep=(n_res, n_gen))
    h = make(c)
    orig = h.copy()
    paths, stats = h.recover_codes(orig, n_res, min_remove)
    want = its[:n_res]
    assert len(paths) == len(want), "recover_codes found %d haplotypes, the oracle %d" % (len(paths), len(want))
    for k, (p, s, (ep, es)) in enumerate(zip(paths, stats, want)):
        bad = np.flatnonzero(p != ep)
        assert bad.size == 0, "resident haplotype %d differs from site %d on (%d sites)" % (k, bad[0], bad.size)
        same_stats(s, es, N, W, "resident haplotype %d" % k)
    res_band = h.band()
    same_band(res_band, bands[len(want)], "band after recover_codes")
    h.close()
    orig.close()

    h = make(c)
    orig = h.copy()
    removed = []
    for k in range(n_gen):
        got = h.generate_path_codes(orig)
        if k == len(its):
            assert got[0] is None and got[1] == hole, "generate_path_codes %r, the oracle's hole is at %r" % (
                got[:2], hole)
            break
        assert got[0] is not None, "generate_path_codes reports a hole at %d, the oracle none" % got[1]
        bad = np.flatnonzero(got[0] != its[k][0])
        assert bad.size == 0, "haplotype %d differs from site %d on (%d sites)" % (k, bad[0], bad.size)
        ratio = max(got[3], min_remove)
        removed.append(h.reweight_path_codes(got[0], ratio))
        same_stats(got[1:] + (ratio, removed[-1]), its[k][1], N, W, "haplotype %d" % k)
    gen_band = h.band()
    same_band(gen_band, bands[min(n_gen, len(its))], "band after generate_path_codes")
    h.close()
    orig.close()
    for k, r in enumerate(removed[:len(stats)]):
        assert _bits(stats[k][4]) == _bits(r), "haplotype %d: the entry points remove %r and %r" % (k, stats[k][4], r)
    if len(removed) == len(stats):
        same_band(gen_band, res_band, "the two entry points leave different bands")
    return its, hole, stats, res_band


def _summary(its, hole):
    return [(p.tobytes(), _bits(s[:4]).tobytes()) for p, s in its] + [hole]


def assert_switch_matters(c_oracle, c, n):
    """The case's switches change the oracle loop on its data; with unsymbols kept, some path chooses N or '_'."""
    its, hole, _ = oracle_loop(c_oracle, c, n)
    base, base_hole, _ = oracle_loop(c_oracle, dict(c, v_site="from", skip_unsym=True), n)
    assert _summary(its, hole) != _summary(base, base_hole), "the switches change nothing on this case"
    if not c["skip_unsym"]:
        assert any(np.isin(p[1:], (SYM_N, SYM_GAP)).any() for p, _ in its), "no N or '_' was chosen"
    return its


# ---- 1. kernel x switch matrix --------------------------------------------------------------------------------------
def _matrix_params(with_default):
    out = []
    for name, L in MATRIX:
        for f in FLAGS:
            if with_default or f != "from":
                out.append(pytest.param(name, L, f, id="%s-L%s-%s" % (name, L, f)))
    return out


@pytest.mark.parametrize("name,L,flags", _matrix_params(False))
def test_matrix_case_reaches_its_switch(c_oracle, name, L, flags):
    c = matrix_case(name, L, flags)
    kernel = {"tables_in": "tables", "narrow": "tables", "narrow_long": "tables", "wide_beyond": "wide"}.get(name, name)
    assert walk_kernel(c["N"], c["W"], c["L"]) == (kernel if L != 0 else "tables")
    assert (c["L"] > c["W"]) == (name.startswith("narrow") or name == "wide_beyond")
    if L == 0:
        # no lookback terms: v_site cannot matter, only which symbols are candidates
        other = oracle_loop(c_oracle, dict(c, v_site="to" if c["v_site"] == "from" else "from"), 4)
        assert _summary(*oracle_loop(c_oracle, c, 4)[:2]) == _summary(*other[:2])
        if c["skip_unsym"]:
            return
    assert_switch_matters(c_oracle, c, 4)


@pytest.mark.parametrize("flags", list(FLAGS))
def test_wide_case_depends_on_the_terms_beyond_the_band(c_oracle, flags):
    """k_walk_wide's striped sum beyond the band decides whether a site is re-evaluated exactly: on this case the
    oracle loop at L = 700 differs from the one on the same band at L = W, under either V rule."""
    c = matrix_case("wide_beyond", 700, flags)
    its, hole, _ = oracle_loop(c_oracle, c, 4)
    at_w, hole_w, _ = oracle_loop(c_oracle, dict(c, L=c["W"]), 4)
    assert _summary(its, hole) != _summary(at_w, hole_w)


@pytest.mark.gpu
@pytest.mark.parametrize("name,L,flags", _matrix_params(True))
def test_walk_kernel_under_switches(c_oracle, name, L, flags):
    c = matrix_case(name, L, flags)
    its, hole, _, _ = check(c_oracle, c, n_res=4, n_gen=2)
    assert len(its) == 4 and hole is None


@pytest.mark.gpu
def test_narrow_band_above_the_block_size_walks_sequentially(c_oracle):
    """W < L <= 32 at N >= 1024 takes k_walk_tables, not the block walk: no block is picked, fixed or walked again, so
    one walk launches exactly as many kernels as on a short narrow region."""
    from tests.test_gpu_walk_blocks import redone

    def launches(name):
        h = device_matrix(matrix_case(name, 17, "from_keep"))
        orig = h.copy()
        n0, r0 = h.launch_count(), redone(h)
        assert h.generate_path_codes(orig)[0] is not None
        return h.launch_count() - n0, redone(h) - r0

    assert launches("narrow_long") == launches("narrow")
    assert launches("narrow_long")[1] == 0


# ---- 2. value extremes ----------------------------------------------------------------------------------------------
# name -> (N, max_k, L, reads per site, share of single-allele sites): thin enough that many pairs are unseen.
# narrow: up to 995 terms log10(1 / V) beyond the band; with V = 1 at half the sites, whether they sum below -323
# depends on which site's V each term takes (v_site)
UNDERFLOW = {"q_seq": (300, 40, 32, 2, 0.0), "tables": (300, 61, 47, 2, 0.0), "narrow": (1100, 6, 1000, 6, 0.5),
             "wide": (400, 170, 169, 1, 0.0)}


def underflow_case(name, flags):
    """Counts scaled by 1e30: a pair never seen together gives a lookback term of about -31."""
    N, max_k, L, per_site, mono = UNDERFLOW[name]
    band = _reads_band(40 + max_k, N, max_k, False, per_site, mono).copy()
    band[band > 0] *= np.float32(1e30)
    return case(band, N, max_k - 1, L, flags)


@pytest.mark.parametrize("name", list(UNDERFLOW))
@pytest.mark.parametrize("flags", list(FLAGS))
def test_underflow_case_reaches_zero_total(c_oracle, name, flags):
    """At some site of the path every candidate's 10**x is 0, and the first candidate in symbol order wins there."""
    c = underflow_case(name, flags)
    assert walk_kernel(c["N"], c["W"], c["L"]) == {"narrow": "tables"}.get(name, name)
    its, _, _ = oracle_loop(c_oracle, c, 1)
    path = its[0][0]
    hits = 0
    for snp in range(1, c["N"] + 1):
        mask, w, tw = c_oracle.edge_weights_at(c["band"], c["N"], c["W"], c["L"], snp, path, c["v_site"],
                                               c["skip_unsym"])
        if mask and tw == 0.0:
            hits += 1
            assert path[snp] == (mask & -mask).bit_length() - 1
    assert hits > 0, "no site where every candidate underflows"


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(UNDERFLOW))
@pytest.mark.parametrize("flags", list(FLAGS))
def test_walk_where_every_candidate_underflows(c_oracle, name, flags):
    check(c_oracle, underflow_case(name, flags), n_res=2, n_gen=2)


# (N, W, L): the fixed-point walk sequential and in blocks, k_walk_tables and k_walk_wide
OVERFLOW_GEOMETRY = {"q_seq": (300, 39, 32), "q_blocks": (1100, 39, 32), "tables": (300, 60, 47),
                     "wide": (400, 169, 169)}
# run sites and support: 12 terms of +35, and up to 40 terms of +14 (each below the fixed-point walk's range limit of 15)
OVERFLOW_RUNS = {"deep": (12, 1e-35), "long": (40, 1e-14)}


def overflow_case(kernel, run):
    N, W, L = OVERFLOW_GEOMETRY[kernel]
    R, sigma = OVERFLOW_RUNS[run]
    R = min(R, L - 4)
    band, after = laplace_band(N, W, R, np.float32(sigma), 20 + W)
    return case(band, N, W, L, "from_keep"), after


@pytest.mark.parametrize("run", list(OVERFLOW_RUNS))
@pytest.mark.parametrize("kernel", list(OVERFLOW_GEOMETRY))
def test_overflow_case_reaches_infinite_total(c_oracle, kernel, run):
    """After the run of V = 0 sites, candidate T's weight is 10**(> 308) = inf: the total is inf, normalising gives
    T inf / inf = NaN and the others 0, and the first-max rule keeps the first candidate in symbol order, not T."""
    c, after = overflow_case(kernel, run)
    assert walk_kernel(c["N"], c["W"], c["L"]) == kernel
    its, _, _ = oracle_loop(c_oracle, c, 1)
    path = its[0][0]
    mask, w, tw = c_oracle.edge_weights_at(c["band"], c["N"], c["W"], c["L"], after, path, "from", False)
    assert tw == np.inf and np.isnan(w[3]) and mask & 1 << 3
    first = (mask & -mask).bit_length() - 1
    assert first != 3 and path[after] == first
    if kernel.startswith("q_"):
        # "long": every term fits the fixed-point range, so the quantised walk takes its fast path at the overflowing
        # sites and only its test of the best log weight against +300 sends them to the exact evaluation (without it
        # the long cases fail).  "deep": a term of +35 is out of range and forces the exact evaluation everywhere.
        assert (fixed_point_max_term(c) < 15) == (run == "long")


def fixed_point_max_term(c):
    """The largest |lookback term| of the fixed-point walk's tables (k_walk_terms: l <= L <= W, every history
    symbol a and candidate s; a term whose Laplace denominator is 0 is dropped).  At 15 or more the walk decides every
    site by the exact evaluation."""
    from oracle import c_oracle
    band, N, L = c["band"], c["N"], c["L"]
    cnt = c_oracle.counts_all(band, N, c["W"])
    vseen = (cnt[:, [0, 1, 2, 3, 5]] > 0).sum(axis=1)
    worst = 0.0
    for snp in range(1, N + 1):
        for l in range(1, min(L, snp) + 1):
            cell = band[snp, l - 1].astype(np.float64)                    # cell (snp - l, snp): [a][s]
            v = vseen[snp] if c["v_site"] == "to" else vseen[snp - l]
            den = v + cell.sum(axis=0)
            t = np.log10((1.0 + cell[:, den != 0]) / den[den != 0])
            worst = max(worst, float(np.abs(t).max(initial=0.0)))
    return worst


@pytest.mark.gpu
@pytest.mark.parametrize("run", list(OVERFLOW_RUNS))
@pytest.mark.parametrize("kernel", list(OVERFLOW_GEOMETRY))
def test_walk_where_a_weight_overflows(c_oracle, kernel, run):
    c, _ = overflow_case(kernel, run)
    check(c_oracle, c, n_res=2, n_gen=2)


@pytest.mark.parametrize("flags", list(FLAGS))
@pytest.mark.parametrize("name,L", [("narrow", 400), ("q_seq", 301)])
def test_lookback_longer_than_the_region(c_oracle, name, L, flags):
    c = matrix_case(name, L, flags)
    assert c["L"] > c["N"] and walk_kernel(c["N"], c["W"], c["L"]) == "tables"
    if flags != "from":
        assert_switch_matters(c_oracle, c, 3)


@pytest.mark.gpu
@pytest.mark.parametrize("flags", list(FLAGS))
@pytest.mark.parametrize("name,L", [("narrow", 400), ("q_seq", 301)])
def test_walk_with_lookback_longer_than_the_region(c_oracle, name, L, flags):
    check(c_oracle, matrix_case(name, L, flags), n_res=3, n_gen=2)


@pytest.mark.gpu
def test_deepest_lookback(c_oracle):
    """L = HX_MAX_L on a band 5 wide: up to 4090 terms log10(1 / V) beyond the band at every site."""
    N = 1500
    c = case(_reads_band(17, N, 6, False), N, 5, HX_MAX_L, "from")
    check(c_oracle, c, n_res=2, n_gen=2)


@pytest.mark.gpu
def test_lookback_beyond_the_limit_is_refused():
    from gretel_b200 import _lib
    c = matrix_case("narrow", HX_MAX_L + 1, "from")
    h = device_matrix(c)
    orig = h.copy()
    for call in (lambda: h.generate_path_codes(orig), lambda: h.recover_codes(orig, 2)):
        with pytest.raises(_lib.HanselxError) as e:
            call()
        assert e.value.code == _lib.HX_E_ARG
        same_band(h.band(), c["band"], "a refused walk changed the band")


# ---- 3. driver loop -------------------------------------------------------------------------------------------------
def strain_case(c_oracle, L=8):
    """Two strains of equal abundance that differ at every site, N = 300, reads of up to 40 SNPs."""
    from tests.test_gpu_walk_blocks import MAX_K, make_strains, strain_reads
    rng = np.random.default_rng(4711)
    N = 300
    rank, off, codes = strain_reads(rng, make_strains(rng, N, 2), 3 * N)
    band = c_oracle.ingest(rank, off, codes, N, MAX_K - 1)[0].astype(np.float32)
    return case(band, N, MAX_K - 1, L)


def touched_cells(path, N, W):
    """Index arrays into the band of the cells reweight_path scales (gretel.py:79-98, hansel_oracle.c)."""
    idx = []
    for i in range(N):
        for j in range(max(0, i - W), i):
            idx.append((i, i - j - 1, path[j], path[i]))
        idx.append((i + 1, 0, path[i], path[i + 1]))
    idx.append((N + 1, 0, path[N], path[0]))
    return tuple(np.array(idx).T)


@pytest.mark.gpu
@pytest.mark.parametrize("min_remove", [0.0, 0.01, 0.3, 1.0])
def test_driver_loop_clamps_the_ratio(c_oracle, min_remove):
    """ratio = max(min marginal, min_remove) (cmd.py:157-160), exactly; more haplotypes asked for than the evidence
    holds returns the oracle's count; with min_remove = 1 every haplotype empties its cells."""
    c = strain_case(c_oracle)
    its, hole, stats, band = check(c_oracle, c, n_res=12, n_gen=3, min_remove=min_remove)
    assert len(stats) == len(its) >= 1
    assert np.array_equal(_bits(stats[:, 3]), _bits(np.maximum(stats[:, 2], min_remove)))
    if min_remove == 1.0:
        assert hole is not None and len(its) < 12
        for p, _ in its:
            assert not band[touched_cells(p, c["N"], c["W"])].any()
    if min_remove == 0.3:
        assert (stats[:, 2] < 0.3).any() and (stats[:, 2] > 0.3).any()


def test_strain_case_reaches_both_sides_of_the_clamp(c_oracle):
    """min marginals on both sides of 0.3 and a hole within 12 haplotypes at min_remove = 1."""
    c = strain_case(c_oracle)
    its, _, _ = oracle_loop(c_oracle, c, 12, 0.3)
    m = np.array([s[2] for _, s in its])
    assert (m < 0.3).any() and (m > 0.3).any()
    its, hole, _ = oracle_loop(c_oracle, c, 12, 1.0)
    assert hole is not None and 1 <= len(its) < 12


@pytest.mark.gpu
def test_zero_paths_do_nothing(c_oracle):
    c = strain_case(c_oracle)
    h = device_matrix(c)
    orig = h.copy()
    n0 = h.launch_count()
    paths, stats = h.recover_codes(orig, 0)
    assert paths.shape == (0, c["N"] + 1) and stats.shape == (0, 5)
    assert h.launch_count() == n0
    same_band(h.band(), c["band"], "recover_codes(0) changed the band")


# ---- 4. the matrix surface recovery reads ---------------------------------------------------------------------------
def _small_packed(seed, N, max_k):
    rng = np.random.default_rng(seed)
    return synth.random_packed(rng, N, 8 * N, max_k, p_special=0.1)


@pytest.mark.gpu
@pytest.mark.parametrize("ratio", [0.3, 1.0 / 3.0, 0.99])
def test_reweight_matrix_then_recover(c_oracle, ratio):
    """reweight_matrix equals OracleHansel.reweight_matrix bit for bit, in the band and in the spill of cells outside
    it; recovery on the reweighted matrix equals the oracle's."""
    from gretel_b200 import util
    N, W = 40, 8
    rank, off, codes = _small_packed(31, N, W + 1)
    ho = o.load_from_packed(rank, off, codes, N)

    def make(c):
        h = util.load_from_packed(rank, off, codes, N, band_w=W)
        for a, b, i, j in (("A", "C", 2, 30), ("A", "C", 2, 30), ("T", "G", 0, N + 1), ("N", "_", 5, 5 + W + 1)):
            h.add_observation(a, b, i, j)
        h.reweight_matrix(ratio)
        h.L, h.v_site, h.candidates_skip_unsymbols = c["L"], c["v_site"], c["skip_unsym"]
        return h

    for a, b, i, j in (("A", "C", 2, 30), ("A", "C", 2, 30), ("T", "G", 0, N + 1), ("N", "_", 5, 5 + W + 1)):
        ho.add_observation(a, b, i, j)
    ho.reweight_matrix(ratio)
    c = case(o.band_of(ho, W), N, W, 5)
    h = make(c)
    assert np.array_equal(h.to_dense().view(np.uint32), ho.m.view(np.uint32))
    h.close()
    check(c_oracle, c, n_res=3, n_gen=2, make=make)


@pytest.mark.gpu
def test_reweight_observation_against_oracle():
    """Random in-band cells, (0,1), (N,N+1) and cells d = W: the removed mass and the stored cell equal the oracle's;
    a cell outside the band is reweighted in the spill."""
    from gretel_b200 import util
    N, W = 40, 8
    rank, off, codes = _small_packed(32, N, W + 1)
    ho = o.load_from_packed(rank, off, codes, N)
    h = util.load_from_packed(rank, off, codes, N, band_w=W)
    h.add_observation("G", "T", 3, 3 + W + 4)
    ho.add_observation("G", "T", 3, 3 + W + 4)
    rng = np.random.default_rng(33)
    S = o.SYMBOLS
    cells = [("_", "A", 0, 1), ("_", "C", 0, 1), ("A", "_", N, N + 1), ("T", "_", N, N + 1)]
    cells += [(S[rng.integers(0, 7)], S[rng.integers(0, 7)], i, i + W) for i in rng.integers(0, N + 2 - W, 6)]
    nz = np.argwhere(ho.m > 0)
    nz = nz[(nz[:, 3] - nz[:, 2] >= 1) & (nz[:, 3] - nz[:, 2] <= W)]
    cells += [(S[a], S[b], int(i), int(j)) for a, b, i, j in nz[rng.choice(len(nz), 30, replace=False)]]
    cells += [("G", "T", 3, 3 + W + 4)] * 2
    for a, b, i, j in cells:
        ratio = float(rng.random())
        got, exp = h.reweight_observation(a, b, i, j, ratio), ho.reweight_observation(a, b, i, j, ratio)
        assert _bits(got) == _bits(exp), (a, b, i, j)
        assert np.float32(h.get_observation(a, b, i, j)).view(np.uint32) == \
            np.float32(ho.get_observation(a, b, i, j)).view(np.uint32), (a, b, i, j)
    assert h._spill == {(2, 3, 3, 3 + W + 4): np.float32(ho.m[2, 3, 3, 3 + W + 4])}
    assert np.array_equal(h.to_dense().view(np.uint32), ho.m.view(np.uint32))


@pytest.mark.gpu
def test_every_mutation_refreshes_the_site_counts(c_oracle):
    """counts_all, get_marginal_of_at and the device's own hx_counts_all / hx_marginal_of_at equal the oracle's counts
    bit for bit after ingestion and after each call that changes the band: the cached counts (the device's
    counts_dirty flag, Hansel._counts_cache) are read before every call, so a cache the call leaves stale is seen."""
    from gretel_b200 import _lib, util
    w = synth.scaled(synth.WORKLOADS["metagenome"], 200_000)
    d = synth.generate(w)
    N, W = w.n_snps, d["max_k"] - 1
    cur = c_oracle.ingest(d["rank"], d["off"], d["codes"], N, W)[0].astype(np.float32)
    h = util.load_from_packed(d["rank"], d["off"], d["codes"], N, band_w=W)
    h.L = 4
    lib = _lib.load()
    rng = np.random.default_rng(99)

    def same_counts(what):
        exp = c_oracle.counts_all(cur, N, W)
        dev = np.zeros((N + 1, 8), dtype=np.float64)
        _lib.check(lib.hx_counts_all(h._h, dev.ctypes.data))
        assert np.array_equal(_bits(dev), _bits(exp)), "hx_counts_all after %s" % what
        assert np.array_equal(_bits(h._counts_all()), _bits(exp)), "Hansel counts after %s" % what
        for pos in rng.integers(0, N + 1, 8):
            s = int(np.argmax(exp[pos, :7]))
            m = exp[pos, s] / exp[pos, 7] if exp[pos, 7] != 0 else 0.0
            assert _bits(h.get_marginal_of_at(h.symbols[s], int(pos))) == _bits(m), "marginal after %s" % what
            out = C.c_double()
            _lib.check(lib.hx_marginal_of_at(h._h, s, int(pos), C.byref(out)))
            assert _bits(out.value) == _bits(m), "hx_marginal_of_at after %s" % what

    same_counts("ingestion")
    orig, h_orig = cur.copy(), h.copy()                    # the matrix at ingestion, on both sides
    pc, res = c_oracle.generate_path(cur, orig, N, W, 4)
    assert pc is not None
    got = h.generate_path_codes(h_orig)
    assert np.array_equal(got[0], pc)
    removed = c_oracle.reweight_path(cur, N, W, pc, 0.4)
    same_stats(got[1:] + (0.4, h.reweight_path_codes(got[0], 0.4)), res + (0.4, removed), N, W, "first haplotype")
    same_counts("reweight_path_codes")

    paths, stats = h.recover_codes(h_orig, 2)
    assert len(paths) == 2
    for k, (p, st) in enumerate(zip(paths, stats)):
        q, res = c_oracle.generate_path(cur, orig, N, W, 4)
        assert np.array_equal(p, q)
        ratio = max(res[2], 0.01)
        same_stats(st, res + (ratio, c_oracle.reweight_path(cur, N, W, q, ratio)), N, W, "resident haplotype %d" % k)
    same_counts("recover_codes")

    h.reweight_matrix(0.25)
    c64 = cur.astype(np.float64)
    cur[...] = c64 - 0.25 * c64
    same_counts("reweight_matrix")

    for p in rng.integers(1, N, 4):
        s = int(np.argmax(cur[p + 1, 0].sum(axis=1)))
        b = int(np.argmax(cur[p + 1, 0, s]))
        old = float(cur[p + 1, 0, s, b])
        cur[p + 1, 0, s, b] = old - 0.5 * old
        h.reweight_observation(h.symbols[s], h.symbols[b], int(p), int(p) + 1, 0.5)
        same_counts("reweight_observation at %d" % p)

    cur[2:N:3] = cur[2:N:3] * np.float32(3)
    h.load_band(cur)
    same_counts("load_band")

    for p in rng.integers(1, N, 4):
        cur[p + 1, 0, 5, 1] += np.float32(1)
        h.add_observation("-", "C", int(p), int(p) + 1)
        same_counts("add_observation at %d" % p)
