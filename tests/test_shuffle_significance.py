"""MFE significance against shuffled sequences (mirfold_shuffle_test, mirfold_shuffle_sequences; MirFold.shuffle_test,
records.hairpin_significance).  The CPU tests pin a Python mirror of csrc/shuffle_rng.cuh + csrc/shuffle.cu (test
infrastructure, like oracle/); the GPU tests hold the device kernel to that mirror byte for byte and the device tally to a
host tally of the exported shuffles folded by mirfold_fold and by the CPU oracle."""
import collections
import ctypes as C
import itertools
import json
import os

import numpy as np
import pytest
from conftest import GOLDEN

import mir_prefer_b200 as mp
from mir_prefer_b200 import _lib
from mir_prefer_b200 import records as R
from mir_prefer_b200.corpus import synth_loci
from mir_prefer_b200.fold import FLAG_SERIAL, SHUFFLE_DTYPE, SHUFFLE_STAT_DTYPE, shuffle_fields

ERR_ARG = -3
M64 = (1 << 64) - 1
GAMMA = 0x9E3779B97F4A7C15


# ------------------------------------------------------------------------------------ Python mirror of the device shuffles
def _mix64(z):
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M64
    return z ^ (z >> 31)


class _Rng:
    """splitmix64 seeded from (seed, r, k); below(m) = high word of draw * m (shuffle_rng.cuh)."""

    def __init__(self, seed, r, k):
        self.s = _mix64(_mix64((seed + GAMMA) & M64) ^ ((r << 32) | k))

    def below(self, m):
        self.s = (self.s + GAMMA) & M64
        return (_mix64(self.s) * m) >> 64


def _convert(seq):
    b = seq.encode("latin-1") if isinstance(seq, str) else bytes(seq)
    return b.upper().replace(b"T", b"U")


def mirror_mono(seq, seed, r, k):
    a = bytearray(_convert(seq))
    g = _Rng(seed, r, k)
    for i in range(len(a) - 1, 0, -1):
        j = g.below(i + 1)
        a[i], a[j] = a[j], a[i]
    return a.decode("latin-1")


def mirror_di(seq, seed, r, k):
    s = _convert(seq)
    n = len(s)
    sym, idx = [], []
    for c in s:
        if c not in sym:
            sym.append(c)
        idx.append(sym.index(c))
    assert len(sym) <= 16
    if n <= 2:
        return s.decode("latin-1")
    ns = len(sym)
    edges = [[] for _ in range(ns)]
    for t in range(n - 1):
        edges[idx[t]].append(idx[t + 1])
    first, last = idx[0], idx[-1]
    g = _Rng(seed, r, k)
    tree, nxt = [False] * ns, [0] * ns
    tree[last] = True
    for u in range(ns):
        x = u
        while not tree[x]:
            nxt[x] = g.below(len(edges[x]))
            x = edges[x][nxt[x]]
        x = u
        while not tree[x]:
            tree[x] = True
            x = edges[x][nxt[x]]
    for u in range(ns):
        e = edges[u]
        m = len(e)
        if u != last:
            e[nxt[u]], e[m - 1] = e[m - 1], e[nxt[u]]
            m -= 1
        for i in range(m - 1, 0, -1):
            j = g.below(i + 1)
            e[i], e[j] = e[j], e[i]
    pos = [0] * ns
    out, cur = [sym[first]], first
    for _ in range(n - 1):
        v = edges[cur][pos[cur]]
        pos[cur] += 1
        out.append(sym[v])
        cur = v
    return bytes(out).decode("latin-1")


MIRROR = {"mono": mirror_mono, "di": mirror_di}


def _dinucs(s):
    return collections.Counter(s[t:t + 2] for t in range(len(s) - 1))


def _host_tally(seqs, totals_of, n_shuffles, seed, mode):
    """SHUFFLE_STAT_DTYPE rows from totals_of(list of str) over the natives and the mirror's shuffles."""
    out = np.zeros(len(seqs), SHUFFLE_STAT_DTYPE)
    out["native_dcal"] = totals_of([_convert(s).decode("latin-1") for s in seqs])
    for k in range(n_shuffles):
        t = totals_of([MIRROR[mode](s, seed, r, k) for r, s in enumerate(seqs)])
        for r, x in enumerate(t):
            out[r]["n_le"] += x <= out[r]["native_dcal"]
            out[r]["sum_dcal"] += x
            out[r]["sumsq_dcal"] += x * x
    return out


def _mixed_seqs(seed, n_long=(300, 1000)):
    """Lengths 0-7 and 20-1000; lower case, T and U, N runs, IUPAC letters."""
    rng = np.random.default_rng(seed)
    out = ["", "a", "Gt", "acg", "NNNN", "ACGUa", "tttttt", "GcAuTgN"]
    for n in (20, 64, 150) + tuple(n_long):
        s = list("".join(synth_loci(int(rng.integers(1 << 30)), 1, (n, n), plain=False))[:n].ljust(n, "A"))
        for q in rng.integers(0, n, size=max(1, n // 25)):
            s[int(q)] = "NRYKMSWnrykt"[int(rng.integers(12))]
        for q in rng.integers(0, n, size=n // 10):
            s[int(q)] = s[int(q)].lower()
        out.append("".join(s))
    return out


# ------------------------------------------------------------------------------------ CPU
def test_abi_layout():
    assert C.sizeof(_lib.ShuffleStat) == 24 and SHUFFLE_STAT_DTYPE.itemsize == 24
    assert [getattr(_lib.ShuffleStat, f).offset for f in SHUFFLE_STAT_DTYPE.names] == [SHUFFLE_STAT_DTYPE.fields[f][1] for f in SHUFFLE_STAT_DTYPE.names]
    assert {"mirfold_shuffle_test", "mirfold_shuffle_sequences"} <= set(_lib.EXPORTS)


def test_mono_keeps_multiset():
    for r, s in enumerate(_mixed_seqs(1)):
        for k in range(5):
            got = mirror_mono(s, 7, r, k)
            assert sorted(got) == sorted(_convert(s).decode("latin-1")), (r, k)


def test_di_keeps_dinucleotides_and_ends():
    seqs = _mixed_seqs(2) + ["acgTTgca" * 3, "UUUU", "ACGU", "aAa", "RYKMSWBDHVNacgtu" * 2]
    for r, s in enumerate(seqs):
        c = _convert(s).decode("latin-1")
        for k in range(6):
            got = mirror_di(s, 11, r, k)
            assert len(got) == len(c) and _dinucs(got) == _dinucs(c), (r, k)
            assert got[:1] == c[:1] and got[-1:] == c[-1:], (r, k)
            assert sorted(got) == sorted(c)


def test_determinism_and_seeds():
    s = _mixed_seqs(3)[-2]
    for mode, f in MIRROR.items():
        a = f(s, 5, 2, 9)
        assert f(s, 5, 2, 9) == a
        assert f(s, 6, 2, 9) != a and f(s, 5, 3, 9) != a and f(s, 5, 2, 10) != a, mode
        assert f(s, (1 << 64) - 1, 2, 9) != a


def _eulerian_sequences(s):
    """Every sequence with the dinucleotide counts and the ends of s (brute force over the distinct permutations)."""
    want = _dinucs(s)
    out = set()
    for p in set(itertools.permutations(s)):
        q = "".join(p)
        if q[0] == s[0] and q[-1] == s[-1] and _dinucs(q) == want:
            out.add(q)
    return sorted(out)


def test_di_uniform_over_eulerian_paths():
    """A short sequence with few Eulerian paths: every path is drawn, with frequencies a chi-square test accepts."""
    from scipy.stats import chisquare
    s = "AGACAGCAGA"
    paths = _eulerian_sequences(s)
    assert 10 <= len(paths) <= 200
    draws = 300 * len(paths)
    cnt = collections.Counter(mirror_di(s, 2026, 0, k) for k in range(draws))
    assert set(cnt) == set(paths)
    assert chisquare([cnt[p] for p in paths]).pvalue > 1e-3


def test_mono_uniform_over_permutations():
    from scipy.stats import chisquare
    s = "AACGU"
    perms = sorted(set("".join(p) for p in itertools.permutations(s)))
    cnt = collections.Counter(mirror_mono(s, 99, 4, k) for k in range(200 * len(perms)))
    assert set(cnt) == set(perms)
    assert chisquare([cnt[p] for p in perms]).pvalue > 1e-3


def _oracle_totals(oracle, span):
    return lambda seqs: [oracle.fold(x, span if span else max(len(x), 5))["total"] for x in seqs]


def test_scoring_with_mirror_and_oracle(oracle):
    """mirror + oracle.fold totals -> the statistics; the derived fields equal numpy's over the list of totals."""
    seqs = ["GGGGAAACCCCAUAUGGGGAAACCCC", synth_loci(8, 1, (70, 70))[0], "ACGUN"]
    K = 12
    stat = _host_tally(seqs, _oracle_totals(oracle, 0), K, 3, "di")
    tab = shuffle_fields(stat, K)
    for r, s in enumerate(seqs):
        tot = np.array([oracle.fold(mirror_di(s, 3, r, k), max(len(s), 5))["total"] for k in range(K)], np.int64)
        native = oracle.fold(_convert(s).decode(), max(len(s), 5))["total"]
        assert tab[r]["native_dcal"] == native and tab[r]["n_le"] == int((tot <= native).sum())
        assert tab[r]["sum_dcal"] == tot.sum() and tab[r]["sumsq_dcal"] == (tot * tot).sum()
        assert tab[r]["p_value"] == (int((tot <= native).sum()) + 1) / (K + 1)
        assert np.isclose(tab[r]["mean"], tot.mean()) and np.isclose(tab[r]["sd"], tot.std())
        if tot.std() > 0:
            assert np.isclose(tab[r]["z"], (native - tot.mean()) / tot.std())
        else:
            assert np.isnan(tab[r]["z"])
    assert tab[0]["native_dcal"] < 0 and tab[0]["p_value"] < 0.5


def test_shuffle_fields_ties_and_zero():
    stat = np.zeros(2, SHUFFLE_STAT_DTYPE)
    stat[0] = (-500, 4, -2000, 1000000)       # four shuffles all at -500
    stat[1] = (0, 4, 0, 0)
    t = shuffle_fields(stat, 4)
    assert t.dtype == SHUFFLE_DTYPE and list(t["sd"]) == [0.0, 0.0] and np.isnan(t["z"]).all()
    assert list(t["p_value"]) == [1.0, 1.0] and list(t["mean"]) == [-500.0, 0.0]


# ------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def mixed():
    return _mixed_seqs(5)


def _fold_totals(mf, span):
    def f(seqs):
        if span:
            with mf.fold(seqs, span) as res:
                return [res.total(r) for r in range(len(seqs))]
        out = [0] * len(seqs)
        for n in sorted({len(s) for s in seqs if len(s) >= 5}):   # global: every length at span n
            idx = [r for r, s in enumerate(seqs) if len(s) == n]
            with mf.fold([seqs[r] for r in idx], n) as res:
                for j, r in enumerate(idx):
                    out[r] = res.total(j)
        return out
    return f


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["di", "mono"])
def test_device_shuffles_equal_mirror(mf, mixed, mode):
    """Several thousand (record, replicate) pairs, records of 0-1000 nt with IUPAC, N and lower-case letters."""
    seqs = mixed * 2
    pairs = 0
    for k in list(range(60)) + [1000, 65535, 4000000000]:
        got = mf.shuffle_sequences(seqs, k, seed=77, mode=mode)
        assert got == [MIRROR[mode](s, 77, r, k) for r, s in enumerate(seqs)], k
        pairs += len(seqs)
    assert pairs >= 1500
    assert mf.shuffle_sequences(seqs, 3, seed=78, mode=mode) != mf.shuffle_sequences(seqs, 3, seed=77, mode=mode)


@pytest.mark.gpu
@pytest.mark.parametrize("span", [150, 0])
def test_native_equals_fold_total(mf, mixed, span):
    tab = mf.shuffle_test(mixed, 2, seed=1, span=span)
    assert tab["native_dcal"].tolist() == _fold_totals(mf, span)(mixed)
    short = np.array([len(s) < 5 for s in mixed])
    assert (tab["n_le"][short] == 2).all() and (tab["sum_dcal"][short] == 0).all() and (tab["native_dcal"][short] == 0).all()


@pytest.mark.gpu
@pytest.mark.parametrize("mode,span", [("di", 150), ("di", 0), ("mono", 300)])
def test_tally_equals_exported_shuffles_folded(mf, mixed, mode, span):
    """shuffle_test == a host tally of mirfold_fold over the device's own exported shuffles; the stats count natives too."""
    K, seed = 6, 2024
    tab, st = mf.shuffle_test(mixed, K, seed=seed, mode=mode, span=span, with_stats=True)
    fold = _fold_totals(mf, span)
    want = np.zeros(len(mixed), SHUFFLE_STAT_DTYPE)
    want["native_dcal"] = fold(mixed)
    for k in range(K):
        t = np.array(fold(mf.shuffle_sequences(mixed, k, seed=seed, mode=mode)), np.int64)
        want["n_le"] += t <= want["native_dcal"]
        want["sum_dcal"] += t
        want["sumsq_dcal"] += t * t
    for f in SHUFFLE_STAT_DTYPE.names:
        assert tab[f].tolist() == want[f].tolist(), f
    assert st["nt"] == sum(len(s) for s in mixed) + K * sum(len(s) for s in mixed if len(s) >= 5)
    assert st["tracebacks"] == 0


@pytest.mark.gpu
def test_against_cpu_oracle(mf, oracle):
    seqs = ["GGGGAAACCCCAUAUGGGGAAACCCC"] + synth_loci(8, 3, (60, 130))
    for mode in ("di", "mono"):
        tab = mf.shuffle_test(seqs, 10, seed=3, mode=mode)
        want = _host_tally(seqs, _oracle_totals(oracle, 0), 10, 3, mode)
        for f in SHUFFLE_STAT_DTYPE.names:
            assert tab[f].tolist() == want[f].tolist(), (mode, f)


@pytest.mark.gpu
def test_independent_of_devices_rounds_and_lanes(mf):
    """devices [0] vs [0, 0] (two pipelines), a forced small round size and MIRFOLD_FLAG_SERIAL give identical results."""
    seqs = synth_loci(31, 120, (40, 420)) + ["ACGU", "acgunnnACGU"]
    ref, st1 = mf.shuffle_test(seqs, 40, seed=9, span=200, with_stats=True)
    with mp.MirFold(devices=[0, 0]) as m2:
        two, st2 = m2.shuffle_test(seqs, 40, seed=9, span=200, with_stats=True)
    assert st2["n_devices"] == 2 and st2["cells"] == st1["cells"]
    os.environ["MIRFOLD_SHUFFLE_ROUND_NT"] = "5000"
    try:
        small, st3 = mf.shuffle_test(seqs, 40, seed=9, span=200, with_stats=True)
    finally:
        del os.environ["MIRFOLD_SHUFFLE_ROUND_NT"]
    assert st3["n_chunks"] > st1["n_chunks"] + 100
    serial = mf.shuffle_test(seqs, 40, seed=9, span=200, flags=FLAG_SERIAL)
    for other in (two, small, serial):
        assert other.tobytes() == ref.tobytes()
    assert mf.shuffle_test(seqs, 40, seed=10, span=200).tobytes() != ref.tobytes()


@pytest.fixture(scope="module")
def e2e_case(tmp_path_factory):
    """The first case of the end-to-end fixture (tests/golden/e2e_mirna.json) as test_genome_regions lays it out on a genome:
    one contig per record, 'N' padding, then the record's plus-strand bases at its region."""
    from test_genome_regions import _write_fasta
    d = json.load(open(os.path.join(GOLDEN, "e2e_mirna.json")))
    case = d["cases"][0]
    recs = [R.LocusRecord(x[0], tuple(x[1]), x[2], tuple(x[3]), x[4], [tuple(p) for p in x[5]], [tuple(m) for m in x[6]], x[7])
            for x in case["records"]]
    contigs = [("rec%d" % k, "N" * (r.region[0] - 1) + r.seq) for k, r in enumerate(recs)]
    idx = _write_fasta(tmp_path_factory.mktemp("shuffle_e2e") / "e2e.fa", contigs)
    coord = [r._replace(seqid="rec%d" % k, seq=None) for k, r in enumerate(recs)]
    return d["span"], idx, recs, coord


@pytest.mark.gpu
def test_hairpin_significance_string_and_genome_paths(mf, e2e_case):
    span, idx, recs, coord = e2e_case
    _, _, cand = R.candidates_of_records(mf, recs, span)
    with mf.upload_genome(idx) as g:
        _, _, cand_g = R.candidates_of_records(mf, coord, span, genome=g)
        got_g = R.hairpin_significance(mf, cand_g, coord, 15, seed=5, genome=g)
        every_g = R.hairpin_significance(mf, cand_g, coord, 3, seed=5, genome=g, only_passing=False)
    got = R.hairpin_significance(mf, cand, recs, 15, seed=5)
    every = R.hairpin_significance(mf, cand, recs, 3, seed=5, only_passing=False)
    assert len(got) == cand.nstructs == cand_g.nstructs
    assert got.tobytes() == got_g.tobytes() and every.tobytes() == every_g.tobytes()
    assert every["scored"].all()
    sc = got[got["scored"]]
    assert 5 <= len(sc) < len(got)
    assert ((sc["p_value"] > 0) & (sc["p_value"] <= 1)).all() and np.isnan(got["p_value"][~got["scored"]]).all()
    passing = [bool((cand.verdicts["code"][int(cand.verdict_begin[k]):int(cand.verdict_begin[k]) + int(cand.verdict_count[k])] == 0).any())
               for k in range(cand.nstructs)]
    assert got["scored"].tolist() == passing
    # the scored rows are shuffle_test of the distinct precursors, in order of first appearance by (record, structure)
    sc = sc[np.lexsort((sc["struct"], sc["rec"]))]
    seq_of = [R.fold_sequence(r) for r in recs]
    pre = [seq_of[int(x["rec"])][int(x["fold_start"]) - 1:int(x["fold_start"]) - 1 + int(x["len"])] for x in sc]
    uniq = list(dict.fromkeys(pre))
    direct = mf.shuffle_test(uniq, 15, seed=5)
    for f in SHUFFLE_DTYPE.names:
        assert np.array_equal(sc[f], direct[f][[uniq.index(p) for p in pre]], equal_nan=True), f


@pytest.mark.gpu
def test_argument_errors_leave_no_output(mf):
    lib = mf._lib
    seqs = ["ACGUACGUAGCUAGCUAGCAUCGA", "GGGGAAACCCC"]
    buf, off = mf.pack(seqs)
    sentinel = np.full(2, -12345, SHUFFLE_STAT_DTYPE)

    def call(ctx, b, o, span, mode, k, out=None):
        out = sentinel.copy() if out is None else out
        rc = lib.mirfold_shuffle_test(ctx, b.ctypes.data_as(C.c_void_p), o.ctypes.data_as(C.POINTER(C.c_uint64)), len(o) - 1, span, 0,
                                      mode, k, 1, out.ctypes.data_as(C.c_void_p), None)
        return rc, out

    assert call(mf._ctx, buf, off, 0, 2, 3)[0] == 0
    for span, mode, k in ((0, 2, 0), (0, 0, 3), (0, 3, 3), (4, 2, 3), (4097, 2, 3), (-1, 1, 3)):
        rc, out = call(mf._ctx, buf, off, span, mode, k)
        assert rc == ERR_ARG and out.tobytes() == sentinel.tobytes(), (span, mode, k)
    b17, o17 = mf.pack(["ACGUNRYKMSWBDHVXZ", "ACGU"])          # 17 symbols: dinucleotide mode refuses, mono takes it
    assert call(mf._ctx, b17, o17, 0, 2, 3)[0] == ERR_ARG and call(mf._ctx, b17, o17, 0, 1, 3)[0] == 0
    big, ob = mf.pack(["ACGU" * 1100])
    assert call(mf._ctx, big, ob, 0, 2, 1)[0] == ERR_ARG
    out = np.zeros(len(b17), np.uint8)
    rc = lib.mirfold_shuffle_sequences(mf._ctx, b17.ctypes.data_as(C.c_void_p), o17.ctypes.data_as(C.POINTER(C.c_uint64)), 2, 2, 1, 0,
                                       out.ctypes.data_as(C.c_void_p))
    assert rc == ERR_ARG
    with pytest.raises(mp.MirfoldError):
        mf.shuffle_test(seqs, 3, mode="tri")
    m = mp.MirFold()
    live = m.fold(seqs, 100)          # a live result keeps the closed context's bookkeeping (and its handle) valid
    ctx = m._ctx
    m.close()
    rc, out = call(ctx, buf, off, 0, 2, 3)
    assert rc == ERR_ARG and out.tobytes() == sentinel.tobytes()
    out = np.zeros(len(buf), np.uint8)
    assert lib.mirfold_shuffle_sequences(ctx, buf.ctypes.data_as(C.c_void_p), off.ctypes.data_as(C.POINTER(C.c_uint64)), 2, 2, 1, 0,
                                         out.ctypes.data_as(C.c_void_p)) == ERR_ARG
    live.close()
