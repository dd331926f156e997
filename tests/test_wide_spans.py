"""Spans 801-4096 (RNALfold -L up to the hairpin table's 4096; the reference allows PRECURSOR_LEN up to 3000).

At these spans a locus longer than 864 nt is not tiled: it is one unit of k_fill_generic (one CTA, global-memory Cm ring,
stride about n).  Spans above MF16_MAX_SPAN (1000) force the 32-bit kernels for every bucket unit.  The traceback windows,
k_f3_cta and the hairpin table up to size 4094 only see spans in the thousands here, and the fused candidate pass only
sees hairpins longer than 800 chars.  A generic unit whose scratch does not fit shared memory (more than about 34 100 nt)
keeps it in global memory, and a unit of 2^31 band cells or more is rejected on the host.

The oracle folds are the slow part (about 2-3 ns x n x L*^2 of one core).  They are submitted to a thread pool, longest
first, when the first GPU test asks for them, so that the CPU work overlaps the GPU tests; oracle.fold is a ctypes call
and releases the GIL."""
import os
import re
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest
from conftest import ROOT
from test_long_loci import _hits_above, _locus, _shifted, assert_suffix_local
from test_shuffle_significance import _fold_totals

import mir_prefer_b200 as mp
from mir_prefer_b200.fold import SHUFFLE_STAT_DTYPE, plan_fill_units

ERR_ARG = -3
INF = 1000000
BUCKETS = (160, 352, 608, 864)
SMEM_EDGE = 34116          # the longest generic unit whose scratch fits the 200 KB of shared memory
WIDE_SPANS = (801, 1000, 1001, 2048, 3000, 4096)


def _consts():
    src = open(os.path.join(ROOT, "mir_prefer_b200", "csrc", "mirfold_internal.cuh")).read()
    return {k: int(v) for k, v in re.findall(r"#define (MF16M?_\w+|MF_MAX_SPAN) \(?(-?\d+)\)?", src)}


# ------------------------------------------------------------------------------------------------------------ records
_COMP = str.maketrans("ACGU", "UGCA")


def _plain(seed, n):
    rng = np.random.default_rng(seed)
    gc = float(rng.uniform(0.25, 0.75))
    p = [(1 - gc) / 2, gc / 2, gc / 2, (1 - gc) / 2]
    return np.frombuffer(b"ACGU", np.uint8)[rng.choice(4, size=n, p=p)].tobytes().decode()


def _helix(seed, n, arm=60):
    """A planted perfect GC helix of `arm` pairs (deep energies, long stacks) in a random record."""
    rng = np.random.default_rng(seed + 7)
    s = _plain(seed, n)
    a = "".join(rng.choice(list("GC"), size=arm))
    hp = a + "UUCG" + a[::-1].translate(_COMP)
    at = n // 3
    return s[:at] + hp + s[at + len(hp):]


def _iupac(seed, n):
    rng = np.random.default_rng(seed)
    return "".join(rng.choice(list("ACGUTacgutNnKXIRYkxi"), size=n))


# n per span; the longest record carries a planted helix, the first of at least 160 nt is IUPAC / lower-case
SPAN_LENGTHS = {
    801: [5, 160, 161, 608, 609, 864, 865, 1200, 2500],
    1000: [864, 865, 999, 1000, 1001, 1500],
    1001: [864, 865, 999, 1000, 1001, 1500],
    2048: [160, 352, 608, 864, 865, 2047, 2048, 2049],
    3000: [1200, 2999, 3001],
    4096: [864, 4096],
}


def span_records(L):
    lens = SPAN_LENGTHS[L]
    seed = 1000 if L in (1000, 1001) else L            # the same records on either side of the 16-bit / wide switch
    iu = next(k for k, n in enumerate(lens) if n >= 160)
    out = []
    for k, n in enumerate(lens):
        if n == max(lens):
            out.append(_helix(seed * 100 + k, n))
        elif k == iu:
            out.append(_iupac(seed * 100 + k, n))
        else:
            out.append(_plain(seed * 100 + k, n))
    return out


ADVERSARIAL = ["U" + "C" * 862 + "A", "G" + "A" * 862 + "C"]   # one closing pair across a whole 864-nt unit
MATRIX_CASES = [("gen1001", _plain(71, 1001), 1001), ("b608L2000", _helix(72, 600, 40), 2000),
                ("gen2049", _plain(73, 2049), 2048)]
TEXT_RECORDS = [_plain(80 + k, n) if k % 3 else _iupac(80 + k, n)
                for k, n in enumerate((1200, 40, 777, 1199, 5, 960, 310, 1024))]
TEXT = "".join(">wide%d some header\n%s\n" % (k, s) for k, s in enumerate(TEXT_RECORDS))
EDGE_LOCI = {n: _locus(n, n, 801, tail=n // 2) for n in (SMEM_EDGE, SMEM_EDGE + 1)}


def _oracle_jobs():
    """key -> (cost estimate, callable args) of every oracle fold the GPU tests compare with."""
    jobs = {}
    for L in SPAN_LENGTHS:
        for k, s in enumerate(span_records(L)):
            jobs[("span", L, k)] = (len(s) * min(L, len(s)) ** 2, (s, L, False))
    for name, s, L in MATRIX_CASES:
        jobs[("mat", name)] = (len(s) * min(L, len(s)) ** 2, (s, L, True))
    for n, s in EDGE_LOCI.items():
        jobs[("edge", n)] = (n * 801 ** 2, (s, 801, False))
    jobs[("text",)] = (sum(len(s) ** 3 for s in TEXT_RECORDS), None)
    return jobs


@pytest.fixture(scope="module")
def ojobs(oracle):
    """Every oracle job of the GPU tests, submitted at once, longest first; tests take results with ojobs(key)."""
    oracle.fold("GGGGAAACCCC", 5)     # the first call initialises the oracle's static parameter table
    jobs = _oracle_jobs()
    ex = ThreadPoolExecutor(max_workers=max(2, os.cpu_count() or 2))
    fut = {}
    for key in sorted(jobs, key=lambda k: -jobs[k][0]):
        args = jobs[key][1]
        fut[key] = ex.submit(oracle.fold_text, TEXT, 3000) if key == ("text",) else ex.submit(oracle.fold, *args[:2], matrices=args[2])
    yield lambda key: fut[key].result()
    ex.shutdown(wait=True, cancel_futures=True)


def _assert_same_span(mf, ojobs, L):
    seqs = span_records(L)
    with mf.fold(seqs, L) as res:
        for r, s in enumerate(seqs):
            o = ojobs(("span", L, r))
            assert res.hits(r) == o["hits"], (r, len(s), L)
            assert res.total(r) == o["total"], (r, len(s), L)
        return res.stats


def _assert_matrices(mf, o, s, L, flags=0):
    c, m, f3 = mf.debug_matrices(s, L, flags=flags)
    n = len(s)
    assert (o["c"] == c).all()
    assert (np.minimum(o["m"], INF) == np.minimum(m, INF)).all()
    assert (o["f3"][:n + 3] == f3[:n + 3]).all()


# ------------------------------------------------------------------------------------------------ CPU: routing, limits
def _band_limit_n(L):
    """First locus length whose generic unit holds 2^31 band cells or more: (dmax - 3) * stride >= 2^31, dmax = L."""
    stride = -(-(1 << 31) // (L - 3))
    stride = (stride + 31) & ~31
    return stride - 31


def test_wide_span_routing():
    """Which kernel, stride and band each (n, L) gets at spans 801-4096: buckets up to 864 nt (never tiled), the generic
    kernel beyond, with a stride that is a multiple of 32 and never a bucket stride."""
    for L in WIDE_SPANS:
        for n in sorted({5, 159, 160, 161, 352, 353, 608, 609, 863, 864, 865, 866, 896, 897, L - 1, L, L + 1,
                         SMEM_EDGE, SMEM_EDGE + 1, _band_limit_n(L) - 1}):
            p = plan_fill_units(n, L)
            dmax = min(L, n - 1)
            assert p["dmax"] == dmax and p["n_units"] == 1 and p["tile_len"] == p["tile_step"] == n, (n, L, p)
            if n <= 864:
                want = next(b for b in BUCKETS if n <= b)
                assert p["kernel"] == p["stride"] == want, (n, L, p)
            else:
                assert p["kernel"] == 0 and p["stride"] % 32 == 0 and p["stride"] not in BUCKETS, (n, L, p)
                assert p["stride"] == (n + 31) & ~31, (n, L, p)
            assert p["band_cells"] == (dmax - 3) * p["stride"], (n, L, p)


def test_band_limit_rejected_on_the_host():
    """An untiled unit is addressed with 32-bit offsets (d-4)*stride + i-1: mirfold_plan_fill_units rejects the first n
    whose unit holds 2^31 band cells or more (MIRFOLD_ERR_ARG) and accepts the one below it.  Tiled loci are unaffected."""
    for L in WIDE_SPANS:
        n0 = _band_limit_n(L)
        p = plan_fill_units(n0 - 1, L)
        assert p["kernel"] == 0 and p["band_cells"] < (1 << 31) <= (L - 3) * (p["stride"] + 32), (L, p)
        with pytest.raises(mp.MirfoldError) as e:
            plan_fill_units(n0, L)
        assert e.value.code == ERR_ARG
    assert _band_limit_n(801) == 2_691_073 and _band_limit_n(4096) == 524_673
    assert plan_fill_units(2_691_072, 801)["band_cells"] == 2_147_475_456
    for L in (9, 300, 800):                       # tiled: any length up to 2^30 - 1
        p = plan_fill_units((1 << 30) - 1, L)
        assert p["n_units"] > 1 and p["kernel"] in (608, 864)


def test_fml16_headroom_at_the_last_16bit_span(oracle):
    """MF16_MAX_SPAN = 1000 relies on fML < MF16M_VALID / 2 = 1350 for every finite fML of a 16-bit strip.  The worst case is
    a single possible closing pair across a whole 864-nt unit (the largest hairpin of the bucket plus the AU penalty and
    MLintern); an INF operand plus the most negative fML the guard keeps must still read as INF."""
    k = _consts()
    assert k["MF16_MAX_SPAN"] == 1000 and k["MF16M_VALID"] == 2700
    worst = []
    for s in ADVERSARIAL:
        m = oracle.fold(s, k["MF16_MAX_SPAN"], matrices=True)["m"]
        fin = m[m < INF]
        assert fin.size >= 1
        worst.append(int(fin.max()))
    assert max(worst) < k["MF16M_VALID"] // 2, worst
    assert worst == [1211, 1061]
    assert k["MF16M_INF"] + (k["MF16M_GUARD"] + 1) > k["MF16M_VALID"]


def test_suffix_locality_at_a_wide_span(oracle):
    """The premise of the 40 kb GPU checks below, on the oracle at L = 1001: the hits of fold(s) that start after i0 are
    those of fold(s[i0-1:]), shifted, plus at most one at its end."""
    L, n = 1001, 6000
    s = _locus(4242, n, L, tail=n // 2)
    oracle.fold("GGGGAAACCCC", 5)
    cuts = (2001, 3333, 4100)
    with ThreadPoolExecutor(max_workers=4) as ex:
        whole = ex.submit(oracle.fold, s, L)
        parts = [ex.submit(oracle.fold, s[i0 - 1:], L) for i0 in cuts]
        hits = whole.result()["hits"]
        compared = 0
        for i0, f in zip(cuts, parts):
            w = [h for h in hits if h[2] > i0]
            assert_suffix_local(w, _shifted(f.result()["hits"], i0))
            compared += len(w)
    assert compared > 200


# ------------------------------------------------------------------------------------------------ GPU: against the oracle
@pytest.mark.gpu
def test_matrices_16bit_bucket_at_span_1000(mf, oracle):
    """c, fML and f3 cell for cell on the 864-nt 16-bit bucket at L = 1000 (the switching DYNW instantiation), for the
    sequences that put fML at the top of its 16-bit range."""
    for s in ADVERSARIAL:
        assert plan_fill_units(len(s), 1000)["kernel"] == 864
        _assert_matrices(mf, oracle.fold(s, 1000, matrices=True), s, 1000)


@pytest.mark.gpu
@pytest.mark.parametrize("name,kernel", [("gen1001", 0), ("b608L2000", 608), ("gen2049", 0)])
def test_matrices_wide_spans(mf, ojobs, name, kernel):
    """(1001, L = 1001): generic, forced wide; (600, L = 2000): k_fill_smem<608>, forced wide, L > n; (2049, L = 2048):
    generic, n > L."""
    _, s, L = next(c for c in MATRIX_CASES if c[0] == name)
    assert plan_fill_units(len(s), L)["kernel"] == kernel
    _assert_matrices(mf, ojobs(("mat", name)), s, L)


@pytest.mark.gpu
@pytest.mark.parametrize("L", [801, 1000, 1001, 2048, 3000])
def test_hits_and_totals_against_oracle(mf, ojobs, L):
    st = _assert_same_span(mf, ojobs, L)
    assert st["fill_units"] == sum(1 for n in SPAN_LENGTHS[L] if n >= 5)


@pytest.mark.gpu
def test_fold_text_at_span_3000(mf, ojobs):
    assert mf.fold_text(TEXT, 3000) == ojobs(("text",))


@pytest.mark.gpu
def test_span_bounds(mf):
    """4096 is the widest span (the hairpin table's length); 4097 is MIRFOLD_ERR_ARG for mirfold_fold and mirfold_fold_text."""
    s = _plain(5, 300)
    with mf.fold([s], 4096) as a, mf.fold([s], 300) as b:
        assert a.total(0) == b.total(0) and a.hits(0) == b.hits(0)
    assert mf.fold_text(">x\n%s\n" % s, 4096) == mf.fold_text(">x\n%s\n" % s, 300)
    for call in (lambda: mf.fold([s], 4097), lambda: mf.fold_text(">x\n%s\n" % s, 4097)):
        with pytest.raises(mp.MirfoldError) as e:
            call()
        assert e.value.code == ERR_ARG


def _candidate_records(seed, L, n_rec, arm_min):
    """Records of 1.2-3 kb, most with a planted perfect hairpin of at least 2 * arm_min + 4 nt that fits the span, and
    matures anywhere on the record."""
    rng = np.random.default_rng(seed)
    seqs, regions, matures, moff = [], [], [], [0]
    for k in range(n_rec):
        n = int(rng.integers(1200, 3001))
        s = _plain(seed * 10 + k, n)
        if k % 4 != 3:
            arm_len = int(rng.integers(arm_min, min(L, n) // 2 - 10))
            arm = _plain(seed * 10 + k + 5000, arm_len)
            hp = arm + "GAAA" + arm[::-1].translate(_COMP)
            at = int(rng.integers(0, n - len(hp)))
            s = s[:at] + hp + s[at + len(hp):]
        rs = int(rng.integers(1, 50000))
        regions.append([rs, rs + n])
        for _ in range(int(rng.integers(1, 5))):
            mlen = int(rng.choice([18, 20, 21, 22, 24, 25]))
            m0 = rs + int(rng.integers(0, n - mlen))
            matures.append((m0, m0 + mlen, "+-"[int(rng.integers(2))], int(rng.integers(1, 99))))
        moff.append(len(matures))
        seqs.append(s)
    return seqs, regions, matures, moff


@pytest.mark.gpu
@pytest.mark.parametrize("L,longer_than", [(1000, 804), (3000, 1000)])
def test_fused_candidates_equal_separate_stages_at_wide_spans(mf, L, longer_than):
    """mirfold_fold_candidates == mirfold_fold + mirfold_classify + mirfold_duplex, with candidate structures longer than
    804 chars (L = 1000: a hit spans at most L + 1 chars) and longer than 1000 chars (L = 3000)."""
    seqs, regions, matures, moff = _candidate_records(L, L, 24, longer_than // 2)
    buf, off = mf.pack(seqs)
    with mf.fold_packed(buf, off, L) as res:
        per_rec = res.classify(55)
    queries, keys = [], []
    for r, structs in enumerate(per_rec):
        for k, (_e, fs, ss, _t) in enumerate(structs):
            for m in matures[moff[r]:moff[r + 1]]:
                if 18 <= m[1] - m[0] <= 24:
                    queries.append((ss, (m[0], m[1]), fs, regions[r][0], regions[r][1], m[2]))
                    keys.append((r, k, m))
    want = dict(zip(keys, mf.duplex(queries)))
    cand = mf.fold_candidates(buf, off, L, regions, matures, np.array(moff, np.uint64))
    got = {}
    longest = max(len(x[2]) for p in per_rec for x in p)
    for r in range(len(seqs)):
        assert cand.structures(r) == per_rec[r], r
        for k, m, v in cand.verdicts_of(r):
            got[(r, k, m)] = v
    assert got == want and len(want) > 20
    assert sum(len(x[2]) > longer_than for p in per_rec for x in p) >= 3, longest


@pytest.mark.gpu
def test_global_shuffle_test_on_long_records(mf):
    """shuffle_test(span = 0) on records of 1001-4096 nt folds each at L = n: natives equal mirfold_fold's totals at span
    n, and the tally equals the exported shuffles folded at span n."""
    seqs = [_plain(90, 1001), _iupac(91, 1500), _helix(92, 2600), _plain(93, 4096)]
    K, seed = 2, 77
    tab = mf.shuffle_test(seqs, K, seed=seed, mode="di", span=0)
    fold = _fold_totals(mf, 0)
    want = np.zeros(len(seqs), SHUFFLE_STAT_DTYPE)
    want["native_dcal"] = fold(seqs)
    for k in range(K):
        t = np.array(fold(mf.shuffle_sequences(seqs, k, seed=seed, mode="di")), np.int64)
        want["n_le"] += t <= want["native_dcal"]
        want["sum_dcal"] += t
        want["sumsq_dcal"] += t * t
    for f in SHUFFLE_STAT_DTYPE.names:
        assert tab[f].tolist() == want[f].tolist(), f


# ------------------------------------------------------------------------ GPU: loci past the generic kernel's shared memory
@pytest.mark.gpu
@pytest.mark.parametrize("n", [SMEM_EDGE, SMEM_EDGE + 1], ids=["34116-shared", "34117-global"])
def test_generic_unit_at_the_shared_memory_edge(mf, ojobs, n):
    """34 116 nt is the longest generic unit whose scratch fits shared memory; from 34 117 nt on it lives in global memory.
    Whole-locus hits and total at L = 801 against the oracle."""
    s = EDGE_LOCI[n]
    assert plan_fill_units(n, 801)["kernel"] == 0
    with mf.fold([s], 801) as res:
        o = ojobs(("edge", n))
        assert res.total(0) == o["total"]
        assert res.hits(0) == o["hits"]


@pytest.mark.gpu
@pytest.mark.parametrize("L", [1001, 3000])
def test_40kb_locus_suffix_equals_shared_memory_fold(mf, L):
    """A 40 kb locus (scratch in global memory) and its last 20 000 nt (scratch in shared memory), both on the GPU,
    compared by suffix locality."""
    n = 40_000
    i0 = n - 19_999
    s = _locus(L + 40, n, L, tail=n // 2)
    with mf.fold([s], L) as res:
        whole = _hits_above(res, 0, i0)
    with mf.fold([s[i0 - 1:]], L) as res:
        suffix = _shifted(_hits_above(res, 0, 1), i0)
    assert len(whole) > 100
    assert_suffix_local(whole, suffix)


@pytest.mark.gpu
def test_band_limit_rejected_before_folding(mf):
    """A batch with one locus at the 2^31 band limit is MIRFOLD_ERR_ARG as a whole, before anything is allocated or folded,
    and the context keeps working."""
    small = _plain(6, 400)
    for L in (4096, 801):
        n0 = _band_limit_n(L)
        big = "A" * n0
        for call in (lambda: mf.fold([small, big], L), lambda: mf.fold_text(">a\n%s\n>b\n%s\n" % (small, big), L)):
            with pytest.raises(mp.MirfoldError) as e:
                call()
            assert e.value.code == ERR_ARG and "2^31" in str(e.value)
    with mf.fold([small], 801) as res:
        assert res.nhits > 0


@pytest.mark.gpu
def test_hits_and_totals_against_oracle_span_4096(mf, ojobs):
    """L = 4096: the longest oracle job (a 4096-nt record folded globally), so this test comes last."""
    _assert_same_span(mf, ojobs, 4096)
