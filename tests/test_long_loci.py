"""Multi-megabase loci.  A locus longer than one tile is stored as overlapping tiles, and the f3 kernels and the traceback
find row i's owner tile with a reciprocal multiply (tile_of_row in mirfold_internal.cuh).  The multiply alone is off by
one for some rows of loci of several Mb, so these tests pin the exact form on the host for every tile step and fold
loci well past the first row the multiply alone gets wrong, against the CPU oracle.

Loci of 8-10 Mb at spans 9 and 20 are compared whole.  At wider spans the oracle is too slow for a whole locus, so only
a suffix of about 23 kb is folded on the CPU and compared by suffix locality (test_suffix_locality)."""
import numpy as np
import pytest

import mir_prefer_b200 as mp
from mir_prefer_b200.fastaindex import FastaIndex
from mir_prefer_b200.fold import plan_fill_units

MIN_STEP, MAX_STEP = 64, 864   # MF_TILE_MIN_STEP .. MF_TILE_LEN_BIG: every tile step the engine can plan
MAX_ROW = 1 << 30              # rows i - 1 < 2^30 (loci up to 2^30 - 1 nt, validate_offsets)
M32 = np.uint64(0xFFFFFFFF)


def _rcp(S):
    """LocusDesc::tile_rcp of tile step S (shape_locus in host.cu)."""
    return ((1 << 32) + S - 1) // S


def owner_tile(x, S):
    """Mirror of tile_of_row() in mirfold_internal.cuh before its clamp to tile_last: x = i - 1 (uint32), 32-bit products."""
    x = np.asarray(x, np.uint64)
    t = (x * np.uint64(_rcp(S))) >> np.uint64(32)                 # __umulhi(x, tile_rcp)
    return t - (((t * np.uint64(S)) & M32) > x).astype(np.uint64)  # t -= (t * tile_step > x)


def owner_tile_estimate(x, S):
    """The reciprocal multiply alone (the owner-tile expression before the correction)."""
    return (np.asarray(x, np.uint64) * np.uint64(_rcp(S))) >> np.uint64(32)


def first_wrong_row(S):
    """Smallest x = i - 1 at which owner_tile_estimate differs from x // S.  With e = tile_rcp*S - 2^32, the estimate is
    floor(x/S + x*e/(S*2^32)): it is one too high iff x*e >= (S - x mod S) * 2^32, first for x mod S = S - 1."""
    e = _rcp(S) * S - (1 << 32)
    if e == 0:
        return None
    x0 = -(-(1 << 32) // e)
    return x0 + (S - 1 - x0) % S


def wrong_rows(S, n):
    """How many rows of an n-nt locus the estimate alone puts in the wrong tile."""
    x = np.arange(max(0, first_wrong_row(S) - S), n, dtype=np.uint64)
    return int((owner_tile_estimate(x, S) != x // np.uint64(S)).sum())


def tile_step(L):
    return plan_fill_units(1 << 29, L)["tile_step"]


# ---------------------------------------------------------------------------------------------------- CPU: the mapping
def test_owner_tile_is_exact():
    """tile_of_row() equals (i-1) // S for every step S in [64, 864] and every i - 1 < 2^30.  Within one residue class
    mod S the estimate's error x*e/(S*2^32) only grows with x, so the largest x < 2^30 of each class is its worst case."""
    checked = 0
    for S in range(MIN_STEP, MAX_STEP + 1):
        r = np.arange(S, dtype=np.uint64)
        x = r + ((np.uint64(MAX_ROW - 1) - r) // np.uint64(S)) * np.uint64(S)   # largest x < 2^30 with x mod S == r
        assert (x < MAX_ROW).all() and (x + np.uint64(S) >= MAX_ROW).all()
        assert (owner_tile(x, S) == x // np.uint64(S)).all(), S
        small = np.arange(4 * S, dtype=np.uint64)                                # and the first rows, where e*x is tiny
        assert (owner_tile(small, S) == small // np.uint64(S)).all(), S
        checked += len(x)
    assert checked == sum(range(MIN_STEP, MAX_STEP + 1))


def test_owner_tile_estimate_alone_is_wrong_on_long_loci():
    """The harness sees the bug the correction fixes: the plain reciprocal multiply puts row x = 10 035 251 of an L = 300
    locus (864-nt tiles, step 564) into tile 17 793 instead of 17 792, and goes wrong at the first rows tabulated here."""
    assert int(owner_tile_estimate(10_035_251, 564)) == 17_793 and 10_035_251 // 564 == 17_792
    assert int(owner_tile(10_035_251, 564)) == 17_792
    want = {604: 7_158_607, 599: 9_061_671, 588: 8_590_091, 508: 8_729_979, 309: 30_034_799, 564: 10_035_251,
            558: 7_752_851, 364: 39_768_455}
    for S, fw in want.items():
        assert first_wrong_row(S) == fw
    wrong_below_limit = 0
    for S in range(MIN_STEP, MAX_STEP + 1):
        fw = first_wrong_row(S)
        if fw is None:                 # S a power of two: the reciprocal is exact
            assert S & (S - 1) == 0
            continue
        # fw is wrong and the whole period before it is right, so (the error growing with x in every residue class) it is
        # the first wrong row
        window = np.arange(fw - S, fw + 1, dtype=np.uint64)
        bad = owner_tile_estimate(window, S) != window // np.uint64(S)
        assert bad[-1] and not bad[:-1].any(), S
        wrong_below_limit += fw < MAX_ROW
    assert wrong_below_limit == 779    # of the 801 steps; 4 are powers of two, 18 first go wrong beyond 2^30
    assert min((first_wrong_row(S) or MAX_ROW, S) for S in range(MIN_STEP, MAX_STEP + 1)) == (5_089_479, 860)
    assert min((first_wrong_row(S) or MAX_ROW, S) for S in range(MIN_STEP, 605)) == (7_158_607, 604)


def test_planned_tile_steps_are_in_the_checked_range_or_untiled():
    """Every span the engine accepts up to the 864-nt bucket tiles a 2^30 - 1 nt locus with a step test_owner_tile_is_exact
    covers, or does not tile it; the step and rcp pairing is the one the mirror assumes.  A span that does not tile (L > 800)
    plans longer loci as one generic unit, and a 2^30 - 1 nt locus is then rejected: its unit would hold more than 2^31
    band cells, beyond the kernels' 32-bit band offsets (tests/test_wide_spans.py)."""
    steps = set()
    untiled = []
    for L in range(5, MAX_STEP + 1):
        try:
            p = plan_fill_units(MAX_ROW - 1, L)
        except mp.MirfoldError as e:
            assert e.code == -3, L
            g = plan_fill_units(MAX_STEP + 1, L)
            assert g["kernel"] == 0 and g["n_units"] == 1, (L, g)
            untiled.append(L)
            continue
        if p["n_units"] > 1:
            assert MIN_STEP <= p["tile_step"] <= MAX_STEP, (L, p)
            assert p["tile_step"] == p["tile_len"] - p["dmax"]
            steps.add(p["tile_step"])
        else:
            assert p["kernel"] == 0, (L, p)   # a span too wide to tile: the generic kernel, untiled
    assert untiled == list(range(801, MAX_STEP + 1))
    # spans 5..800 give 540 distinct steps; the first row any of them gets wrong without the correction is x = 7 615 399
    assert len(steps) == 540
    assert min(first_wrong_row(S) for S in steps if first_wrong_row(S)) == 7_615_399


# ----------------------------------------------------------------------------------------------- loci and the oracle rule
_COMP = bytes.maketrans(b"GC", b"CG")


def _locus(seed, n, L, tail=40_000):
    """Seeded ACGU locus with planted perfect GC stem-loops (stems up to the span), densely in the last `tail` nt, and
    N runs: one in the middle, one in the tail."""
    rng = np.random.default_rng(seed)
    s = np.frombuffer(b"ACGU", np.uint8)[rng.integers(0, 4, n)].copy()
    stem = max(2, min(12, (L - 4) // 2))
    at = np.concatenate([rng.integers(0, n - 64, 200), rng.integers(max(0, n - tail), n - 64, 60)])
    for a in at.tolist():
        arm = np.frombuffer(b"GC", np.uint8)[rng.integers(0, 2, stem)].tobytes()
        hp = arm + b"UUCG" + arm.translate(_COMP)[::-1]
        s[a:a + len(hp)] = np.frombuffer(hp, np.uint8)
    for a in (n // 2, n - tail // 2):
        s[a:a + int(rng.integers(50, 400))] = ord("N")
    return s.tobytes().decode()


def assert_suffix_local(whole, suffix):
    """Suffix locality.  Row i's c, fML and f3, and RNALfold's emission state machine down to row i, depend only on
    s[i..n]; so the hits of fold(s) with start > i0 are the first hits of fold(s[i0-1:]) shifted by i0 - 1 with start
    > i0.  The suffix fold may have one more, its last: the pending structure it flushes at its row 1, which the whole
    fold prints or drops by a traceback below i0.  Hits starting at i0 itself are left out: there the whole fold traces
    (i0, L+1) back from row i0 - 1 where the suffix takes its final (1, L).
    whole: [(ss, e, start)] of fold(s) with start > i0; suffix: the suffix fold's, shifted, with start > i0."""
    assert suffix[:len(whole)] == whole
    assert len(suffix) - len(whole) in (0, 1), (len(suffix), len(whole))


def _shifted(hits, i0):
    return [(ss, e, st + i0 - 1) for ss, e, st in hits if st + i0 - 1 > i0]


def test_suffix_locality(oracle):
    """The premise of the wide-span GPU checks, pinned on the oracle: seeded loci with planted helices and N runs, random
    cut points and cuts at, before and after hit starts."""
    rng = np.random.default_rng(20261020)
    compared = 0
    for L, n, ncut in ((9, 8000, 5), (20, 8000, 5), (40, 6000, 4), (60, 5000, 4), (150, 4000, 3), (300, 3000, 3)):
        s = _locus(1000 + L, n, L, tail=n // 2)
        hits = oracle.fold(s, L)["hits"]
        starts = sorted({h[2] for h in hits if n // 4 < h[2] < 3 * n // 4})
        cuts = [int(c) for c in rng.integers(n // 4, 3 * n // 4, ncut)]
        cuts += [starts[len(starts) // 3], starts[len(starts) // 3] - 1, starts[2 * len(starts) // 3] + 1]
        for i0 in cuts:
            whole = [h for h in hits if h[2] > i0]
            assert_suffix_local(whole, _shifted(oracle.fold(s[i0 - 1:], L)["hits"], i0))
            compared += len(whole)
    assert compared > 5000


# ------------------------------------------------------------------------------------------------------- GPU: long loci
def _hits_above(res, r, i0):
    """res.hits(r) restricted to start > i0 (a prefix: hits are in RNALfold's order, descending start)."""
    b, k = int(res.hit_begin[r]), int(res.hit_count[r])
    tab = res.hit_table[b:b + k]
    st = tab["start"]
    assert (np.diff(st) < 0).all()
    m = int((st > i0).sum())
    arena = res.arena
    return [(arena[int(o):int(o) + int(ln)].tobytes().decode("ascii"), int(e), int(s))
            for o, ln, e, s in zip(tab["ss_off"][:m], tab["len"][:m], tab["mfe_dcal"][:m], st[:m])]


def _past_first_wrong(L, margin):
    """Locus length for span L that runs `margin` rows past the first row the estimate alone gets wrong."""
    S = tile_step(L)
    n = first_wrong_row(S) + margin
    assert plan_fill_units(n, L)["n_units"] > 1 and wrong_rows(S, n - 4) >= 20
    return n


@pytest.mark.gpu
def test_l9_locus_matches_oracle_whole(mf, oracle):
    """9.07 Mb at L = 9 (608-nt tiles, step 599): every hit, the total and the RNALfold text, whose start columns are
    wider than %4d, equal the oracle's."""
    L = 9
    n = _past_first_wrong(L, 12_000)
    s = _locus(9, n, L)
    o = oracle.fold(s, L)
    with mf.fold([s], L) as res:
        assert res.total(0) == o["total"]
        assert res.hits(0) == o["hits"]
    text = ">chr_l9 a whole chromosome\n%s\n" % s
    assert mf.fold_text(text, L) == oracle.fold_text(text, L)


@pytest.mark.gpu
def test_l20_locus_matches_oracle_whole_with_matrices(mf, oracle):
    """8.6 Mb at L = 20 (step 588): hits and total, and the whole f3 vector with c / fML cell for cell."""
    L = 20
    n = _past_first_wrong(L, 12_000)
    s = _locus(20, n, L)
    o = oracle.fold(s, L, matrices=True)
    with mf.fold([s], L) as res:
        assert res.total(0) == o["total"]
        assert res.hits(0) == o["hits"]
    c, m, f3 = mf.debug_matrices(s, L)
    assert (o["f3"][:n + 3] == f3[:n + 3]).all()
    assert (o["c"] == c).all()
    assert (np.minimum(o["m"], 1000000) == np.minimum(m, 1000000)).all()


def _device_bytes(n, L):
    """Device bytes the library budgets for one locus (locus_bytes() in host.cu): 13 B per band cell, one DML ring per
    tile, sequence-sized arrays and traceback scratch for about one traceback per 8 nt."""
    p = plan_fill_units(n, L)
    ls = min(L, n)
    per_tb = ((ls + 8) & ~3) + (ls // 4 + 16) * 8 + 64
    return 13 * p["band_cells"] + 64 * p["stride"] * p["n_units"] + 16 * n + (n // 8 + 2) * per_tb


def _free_device_bytes():
    import torch
    return torch.cuda.mem_get_info()[0]


@pytest.mark.gpu
@pytest.mark.parametrize("L", [300, 306, 100], ids=["L300-864tiles", "L306-earliest864", "L100-608tiles"])
def test_wide_span_locus_suffix_matches_oracle(oracle, L):
    """L = 300 (the default span, 864-nt tiles, step 564), L = 306 (the earliest first wrong row of the 864-nt tiles at
    these spans) and L = 100 (608-nt tiles): the whole locus on the GPU, a suffix that starts 5 000 rows before the first
    wrong row on the oracle, compared by suffix locality.  The locus is folded in a context of its own, closed after."""
    n = _past_first_wrong(L, 18_000)
    i0 = first_wrong_row(tile_step(L)) - 5_000
    need, free = _device_bytes(n, L), _free_device_bytes()
    if free < need + (need >> 3) + (2 << 30):
        pytest.skip("L=%d locus of %d nt needs about %d device bytes, %d free" % (L, n, need, free))
    s = _locus(L, n, L)
    with mp.MirFold() as ctx, ctx.fold([s], L) as res:
        whole = _hits_above(res, 0, i0)
        assert res.stats["n_chunks"] == 1
    suffix = _shifted(oracle.fold(s[i0 - 1:], L)["hits"], i0)
    assert len(whole) > 100
    assert_suffix_local(whole, suffix)


@pytest.mark.gpu
def test_minus_strand_genome_region_equals_string_path(mf, tmp_path):
    """A 9.1 Mb minus-strand region of a device-resident genome at L = 9: k_prepare reads it backwards and complements it;
    hits and total equal those of the string path on the host's reverse complement."""
    L = 9
    n = _past_first_wrong(L, 40_000)
    fa = tmp_path / "chr.fa"
    s = _locus(91, n, L).replace("U", "T")
    with open(fa, "w") as f:
        f.write(">chr1\n")
        for k in range(0, n, 80):
            f.write(s[k:k + 80] + "\n")
    idx = FastaIndex(str(fa))
    with mf.upload_genome(idx) as g:
        rc = g.sequence(0, 1, n + 1, "-")
        assert len(rc) == n
        with g.fold_regions([(0, 1, n + 1, ord("-"))], L) as got, mf.fold([rc], L) as want:
            assert got.total(0) == want.total(0)
            assert got.hits(0) == want.hits(0)
