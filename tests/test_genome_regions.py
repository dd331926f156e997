"""Folding records given as coordinates against a genome resident in HBM (mirfold_genome_upload, mirfold_fold_regions,
mirfold_fold_regions_stream, mirfold_fold_candidates_regions; MirFold.upload_genome): every result must equal, byte for
byte, what the text entry points give on the host-extracted sequences (FastaIndex.extend_region_sequence +
records.fold_sequence), and through them the reference's own fixtures."""
import ctypes as C
import json
import os
import re
import sys

import numpy as np
import pytest

from conftest import GOLDEN

import mir_prefer_b200 as mp
from mir_prefer_b200 import _lib
from mir_prefer_b200 import records as R
from mir_prefer_b200.corpus import synth_loci
from mir_prefer_b200.fastaindex import FastaIndex
from mir_prefer_b200.fold import GENOME_REGION_DTYPE, Genome, _mature_array

ERR_ARG, ERR_CALLBACK = -3, -7


def _write_fasta(path, contigs, width=60):
    with open(path, "w") as f:
        for name, seq in contigs:
            f.write(">%s some description\n" % name)
            for k in range(0, len(seq), width):
                f.write(seq[k:k + width] + "\n")
    return FastaIndex(str(path))


def _clip(names, bases, off, contig, start, end):
    """The device's region rule restated on the packed upload: samtools faidx of seqid:start-(end-1)."""
    if contig < 0:
        return b""
    clen = int(off[contig + 1] - off[contig])
    s, e = max(start, 1), min(end - 1, clen)
    return bases[int(off[contig]) + s - 1:int(off[contig]) + e] if s <= e else b""


def _seeded_genome(seed=11):
    """3 contigs: synthetic loci (hairpins) with lower-case masks, N runs, IUPAC letters, U/u next to T/t; contig 0 also
    holds a poly-A stretch and a long N gap (hairpin-free regions)."""
    rng = np.random.default_rng(seed)
    contigs = []
    for c, n in enumerate((26, 10, 6)):
        s = list("".join(synth_loci(seed + c, n, (300, 700), plain=False)))
        L = len(s)
        for _ in range(max(2, L // 1500)):                       # masked stretches
            a = int(rng.integers(0, L - 200)); b = a + int(rng.integers(20, 200))
            s[a:b] = [x.lower() for x in s[a:b]]
        for _ in range(max(1, L // 3000)):                       # N runs
            a = int(rng.integers(0, L - 60)); k = int(rng.integers(1, 60))
            s[a:a + k] = ["N"] * k
        for k in rng.integers(0, L, size=L // 100):                # IUPAC letters, upper and lower case
            s[int(k)] = "RYKMSWBDHVNrykn"[int(rng.integers(0, 15))]
        for k in rng.integers(0, L, size=L // 40):                 # RNA letters among DNA ones
            s[int(k)] = {"T": "U", "t": "u"}.get(s[int(k)], s[int(k)])
        contigs.append(("ctg%d" % c, "".join(s)))
    name, s0 = contigs[0]
    contigs[0] = (name, s0[:5000] + "A" * 1500 + "N" * 800 + s0[5000:])
    return contigs


POLY_A = (5001, 6501)      # [start, end) of contig 0's poly-A stretch
N_GAP = (6501, 7301)


def _seeded_regions(lengths, seed=5, n_mid=2200, n_long=90):
    """About 3 000 regions: both strands, 0-4 / 5-600 / 900-3000 nt, and every clipping case; with 0-3 matures each."""
    rng = np.random.default_rng(seed)
    rows = []
    nc = len(lengths)

    def add(c, a, b, strand):
        rows.append((c, a, b, strand))

    for _ in range(n_mid):
        c = int(rng.integers(0, nc)); n = int(rng.integers(5, 601)); a = int(rng.integers(1, max(2, lengths[c] - n)))
        add(c, a, a + n, "+-"[int(rng.integers(2))])
    for _ in range(150):
        c = int(rng.integers(0, nc)); n = int(rng.integers(0, 5)); a = int(rng.integers(1, lengths[c]))
        add(c, a, a + n, "+-"[int(rng.integers(2))])
    for _ in range(n_long):
        c = int(rng.integers(0, nc)); n = int(rng.integers(900, 3001)); a = int(rng.integers(1, max(2, lengths[c] - n)))
        add(c, a, a + n, "+-"[int(rng.integers(2))])
    for c in range(nc):
        Lc = lengths[c]
        for strand in "+-":
            for a, b in ((-50, 200), (0, 300), (1, 2), (Lc - 100, Lc + 500), (Lc - 4, Lc + 1), (Lc, Lc + 100), (500, 500),
                         (600, 400), (Lc + 10, Lc + 300), (Lc + 1, Lc + 2), (-300, -10), (1, min(Lc + 1, 3001))):
                add(c, a, b, strand)
    for strand in "+-":
        add(-1, 100, 400, strand)
        add(-1, -5, 5, strand)
    order = rng.permutation(len(rows))
    rows = [rows[k] for k in order]
    matures, moff = [], [0]
    for c, a, b, strand in rows:
        for _ in range(int(rng.integers(0, 4))):
            mlen = int(rng.choice([16, 20, 21, 22, 24, 25]))
            m0 = a + int(rng.integers(0, max(1, b - a - mlen)))
            matures.append((m0, m0 + mlen, "+-"[int(rng.integers(2))], int(rng.integers(1, 500))))
        moff.append(len(matures))
    return rows, matures, np.array(moff, np.uint64)


def _table(rows):
    reg = np.zeros(len(rows), GENOME_REGION_DTYPE)
    if rows:
        a = np.array([(c, s, e, ord(t)) for c, s, e, t in rows], np.int64)
        for k, name in enumerate(GENOME_REGION_DTYPE.names):
            reg[name] = a[:, k]
    return reg


def _host_seqs(index, names, rows):
    out = []
    for c, a, b, strand in rows:
        s = index.extend_region_sequence(names[c], (a, b)) if c >= 0 else ""
        out.append(R.get_reverse_complement(s) if strand == "-" else s)
    return out


def _folds(res):
    return [(res.hits(r), res.total(r)) for r in range(res.nseq)]


def _cands(cand):
    return [(cand.structures(r), cand.verdicts_of(r)) for r in range(cand.nseq)]


# ------------------------------------------------------------------------------------ CPU
def test_genome_region_layout_matches_header():
    assert C.sizeof(_lib.GenomeRegion) == 16
    assert [getattr(_lib.GenomeRegion, f).offset for f in ("contig", "start", "end", "strand")] == [0, 4, 8, 12]
    assert GENOME_REGION_DTYPE.itemsize == 16
    assert [GENOME_REGION_DTYPE.fields[f][1] for f in GENOME_REGION_DTYPE.names] == [0, 4, 8, 12]
    assert all(s in _lib.EXPORTS for s in ("mirfold_genome_upload", "mirfold_genome_free", "mirfold_fold_regions",
                                           "mirfold_fold_regions_stream", "mirfold_fold_candidates_regions"))


def test_packed_fasta_reproduces_fetch_and_samtools(tmp_path):
    """The upload format + the region rule == FastaIndex.fetch, and == samtools 0.1.18's own output (faidx.json)."""
    contigs = _seeded_genome(3)
    idx = _write_fasta(tmp_path / "g.fa", contigs)
    names, bases, off = idx.packed()
    assert names == [n for n, _ in contigs] and off.dtype == np.uint64 and int(off[-1]) == len(bases)
    lengths = [len(s) for _, s in contigs]
    rows, _, _ = _seeded_regions(lengths, seed=7, n_mid=400, n_long=20)
    for c, a, b, _strand in rows:
        want = idx.extend_region_sequence(names[c], (a, b)) if c >= 0 else idx.extend_region_sequence("no_such_contig", (a, b))
        assert _clip(names, bases, off, c, a, b).decode("ascii") == want, (c, a, b)
    pinned = 0
    for case in json.load(open(os.path.join(GOLDEN, "faidx.json")))["cases"]:
        fa = tmp_path / "pin.fa"
        fa.write_text(case["fasta"])
        idx = FastaIndex(str(fa))
        names, bases, off = idx.packed()
        for q in case["queries"]:
            m = re.match(r"^(\S+):(\d+)-(\d+)$", q["region"])
            if not m or q["rc"] != 0:
                continue
            c = names.index(m.group(1)) if m.group(1) in names else -1
            got = _clip(names, bases, off, c, int(m.group(2)), int(m.group(3)) + 1)
            assert got.decode("ascii") == "".join(q["stdout"].split("\n")[1:]), q["region"]
            pinned += 1
    assert pinned >= 10


def test_region_table_from_records():
    """records.region_table: seqids to contig indices (-1 when unknown), strands to '+' / '-' codes (0 otherwise)."""
    g = Genome.__new__(Genome)
    g.names, g.contig_ids = ["a", "b"], {"a": 0, "b": 1}
    recs = [R.LocusRecord("b", (5, 90), "-", (1, 2), "0", [], [], None), R.LocusRecord("zz", (-3, 4), "+", (1, 2), "L", [], [], None),
            R.LocusRecord("a", (1, 1), "?", (1, 2), "R", [], [], None)]
    t = R.region_table(g, recs)
    assert t.dtype == GENOME_REGION_DTYPE
    assert t.tolist() == [(1, 5, 90, 45), (-1, -3, 4, 43), (0, 1, 1, 0)]


# ------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def seeded(tmp_path_factory):
    contigs = _seeded_genome()
    idx = _write_fasta(tmp_path_factory.mktemp("genome") / "g.fa", contigs)
    names, _, _ = idx.packed()
    rows, matures, moff = _seeded_regions([len(s) for _, s in contigs])
    return idx, names, rows, matures, moff


@pytest.mark.gpu
@pytest.mark.parametrize("span", [150, 300, 500])
def test_regions_equal_host_path(mf, seeded, span):
    """fold_regions == fold of the host-extracted strings, and fold_candidates_regions == fold_candidates on the packed host
    buffer, per record, over all clipping cases, both strands, short / bucket / tiled lengths."""
    idx, names, rows, matures, moff = seeded
    seqs = _host_seqs(idx, names, rows)
    reg = _table(rows)
    with mf.upload_genome(idx) as g:
        with mf.fold(seqs, span) as want, g.fold_regions(reg, span) as got:
            assert got.nseq == len(rows) and got.nhits == want.nhits > 1000
            assert _folds(got) == _folds(want)
            assert got.stats["nt"] == want.stats["nt"] and got.stats["cells"] == want.stats["cells"]
        buf, off = mf.pack(seqs)
        want_c = mf.fold_candidates(buf, off, span, [[a, b] for _, a, b, _ in rows], matures, moff)
        got_c = g.fold_candidates(reg, span, matures, moff)
        assert got_c.nstructs == want_c.nstructs > 50 and got_c.nverdicts == want_c.nverdicts
        assert _cands(got_c) == _cands(want_c)


@pytest.mark.gpu
def test_hairpin_free_call(mf, seeded):
    """A call of only hairpin-free records (poly-A, poly-U on the minus strand, N, empty): RNALfold prints one unpaired '.'
    line per locus of at least 5 nt, the candidate pass finds no structure, and both equal the host path."""
    idx, names, _, _, _ = seeded
    rows = []
    for k in range(40):
        a = POLY_A[0] + 7 * k
        rows.append((0, a, min(a + 30 + 11 * k, POLY_A[1]), "+-"[k % 2]))
        b = N_GAP[0] + 5 * k
        rows.append((0, b, min(b + 20 + 13 * k, N_GAP[1]), "-+"[k % 2]))
        rows.append((k % 3, 100 + k, 100 + k, "+"))
        rows.append((-1, 1, 400, "-"))
    matures = [(r[1] + 2, r[1] + 23, "+", 5) for r in rows]
    moff = np.arange(len(rows) + 1, dtype=np.uint64)
    seqs = _host_seqs(idx, names, rows)
    assert all(set(s) <= set("AUN") for s in seqs)
    reg = _table(rows)
    buf, off = mf.pack(seqs)
    with mf.upload_genome(idx) as g:
        cand = g.fold_candidates(reg, 300, matures, moff)
        want_c = mf.fold_candidates(buf, off, 300, [[a, b] for _, a, b, _ in rows], matures, moff)
        assert cand.nstructs == 0 and cand.nverdicts == 0 and _cands(cand) == _cands(want_c)
        with g.fold_regions(reg, 300) as got, mf.fold(seqs, 300) as want:
            assert _folds(got) == _folds(want)
            assert {h for hits, _t in _folds(got) for h in hits} == {(".", 0, 1)}
            assert got.nhits == sum(len(s) >= 5 for s in seqs) > 60


@pytest.mark.gpu
def test_two_pipelines_equal_one(mf, seeded):
    """A context that lists the same ordinal twice (two pipelines, small memory budget: several chunks each) == one device."""
    idx, names, rows, matures, moff = seeded
    reg = _table(rows)
    with mf.upload_genome(idx) as g, g.fold_regions(reg, 300) as one:
        want, want_c = _folds(one), _cands(g.fold_candidates(reg, 300, matures, moff))
    os.environ["MIRFOLD_MEM_BUDGET_MB"] = "64"
    try:
        with mp.MirFold(devices=[0, 0]) as m2, m2.upload_genome(idx) as g2:
            with g2.fold_regions(reg, 300) as two:
                assert two.stats["n_devices"] == 2 and two.stats["n_chunks"] >= 4
                assert _folds(two) == want
            cand = g2.fold_candidates(reg, 300, matures, moff)
            assert cand.stats["n_chunks"] >= 4 and _cands(cand) == want_c
    finally:
        del os.environ["MIRFOLD_MEM_BUDGET_MB"]


@pytest.mark.gpu
def test_stream_reassembles_and_aborts(mf, seeded):
    idx, _, rows, _, _ = seeded
    reg = _table(rows)
    got = {}

    def sink(ch):
        for k, r in enumerate(ch.records.tolist()):
            assert r not in got
            got[r] = (ch.hits(k), int(ch.total_mfe_dcal[k]))

    with mf.upload_genome(idx) as g:
        with g.fold_regions(reg, 300) as whole:
            st = g.fold_regions_stream(reg, 300, sink)
            assert sorted(got) == list(range(len(rows)))
            assert [got[r] for r in range(len(rows))] == _folds(whole)
            assert st["nt"] == whole.stats["nt"]
        lib = mf._lib
        rc = lib.mirfold_fold_regions_stream(mf._ctx, g._ptr, reg.ctypes.data_as(C.c_void_p), len(reg), 300, 0,
                                             _lib.CHUNK_FN(lambda _u, _c: 1), None, None)
        assert rc == ERR_CALLBACK


@pytest.mark.gpu
def test_regions_against_cpu_oracle(mf, seeded, oracle):
    """Independent of the device's text path: 64 regions (both strands, masked / IUPAC / RNA letters) == the CPU oracle."""
    idx, names, rows, _, _ = seeded
    pick = [r for r in rows if r[0] >= 0 and 40 <= r[2] - r[1] <= 700][:64]
    assert len(pick) == 64 and {r[3] for r in pick} == {"+", "-"}
    seqs = _host_seqs(idx, names, pick)
    with mf.upload_genome(idx) as g, g.fold_regions(_table(pick), 300) as res:
        for r, s in enumerate(seqs):
            o = oracle.fold(s, 300)
            assert res.hits(r) == o["hits"], r
            assert res.total(r) == o["total"], r


@pytest.mark.gpu
def test_lifetime_and_argument_errors(mf, seeded):
    idx, _, rows, matures, moff = seeded
    reg = _table(rows[:50])
    m1 = mp.MirFold()
    g1 = m1.upload_genome(idx)
    g1.close()                      # free, then close
    m1.close()
    m2 = mp.MirFold()
    g2 = m2.upload_genome(idx)
    with g2.fold_regions(reg, 300) as r2:
        want = _folds(r2)
    m2.close()                      # close, then free: the genome keeps the context's bookkeeping alive
    with pytest.raises(mp.MirfoldError) as e:
        g2.fold_regions(reg, 300)
    assert e.value.code == ERR_ARG
    g2.close()

    lib = mf._lib
    with mf.upload_genome(idx) as g, mp.MirFold() as other, other.upload_genome(idx) as g_other:
        with g.fold_regions(reg, 300) as r:
            assert _folds(r) == want
        res = C.POINTER(_lib.Result)()
        rc = lib.mirfold_fold_regions(mf._ctx, g_other._ptr, reg.ctypes.data_as(C.c_void_p), len(reg), 300, 0, C.byref(res))
        assert rc == ERR_ARG and not res
        cand = C.POINTER(_lib.Candidates)()
        mat = _mature_array(matures)
        rc = lib.mirfold_fold_candidates_regions(mf._ctx, g_other._ptr, reg.ctypes.data_as(C.c_void_p), len(reg), 300, 0,
                                                 mat.ctypes.data_as(C.c_void_p), moff.ctypes.data_as(C.POINTER(C.c_uint64)),
                                                 55, 3, 18, 24, C.byref(cand))
        assert rc == ERR_ARG and not cand
        rc = lib.mirfold_fold_regions_stream(mf._ctx, g_other._ptr, reg.ctypes.data_as(C.c_void_p), len(reg), 300, 0,
                                             _lib.CHUNK_FN(lambda _u, _c: 0), None, None)
        assert rc == ERR_ARG
        for field, value in (("contig", len(g.names)), ("contig", -2), ("strand", ord(".")), ("strand", 0)):
            bad = reg.copy()
            bad[field][17] = value
            with pytest.raises(mp.MirfoldError) as e:
                g.fold_regions(bad, 300)
            assert e.value.code == ERR_ARG, (field, value)
            with pytest.raises(mp.MirfoldError) as e:
                g.fold_candidates(bad, 300, matures[:int(moff[50])], moff[:51])
            assert e.value.code == ERR_ARG, (field, value)
            with pytest.raises(mp.MirfoldError) as e:
                g.fold_regions_stream(bad, 300, lambda ch: None)
            assert e.value.code == ERR_ARG, (field, value)


@pytest.mark.gpu
def test_upload_bytes(mf, seeded):
    """Per call only descriptors go up: the sequence bytes of the host path are gone from h2d_bytes."""
    idx, names, rows, matures, moff = seeded
    packed = idx.packed()
    keep = [k for k, r in enumerate(rows) if not 0 < len(_clip(*packed, r[0], r[1], r[2])) < 5]
    rows = [rows[k] for k in keep]
    seqs = _host_seqs(idx, names, rows)
    nt = sum(len(s) for s in seqs)
    reg = _table(rows)
    with mf.upload_genome(idx) as g, g.fold_regions(reg, 300) as got, mf.fold(seqs, 300) as want:
        assert got.stats["nt"] == nt
        assert got.stats["h2d_bytes"] <= want.stats["h2d_bytes"] - nt


@pytest.mark.gpu
def test_record_level_genome_path(mf, seeded):
    """fold_records / candidates_of_records with genome=g on records without sequences == the same calls on records whose
    seq is the host-extracted plus-strand sequence (duplicated records included)."""
    idx, names, rows, _, _ = seeded
    rng = np.random.default_rng(2)
    recs_seq, recs_none = [], []
    for k, (c, a, b, strand) in enumerate(rows[:400] + rows[:20]):
        seqid = names[c] if c >= 0 else "not_in_fasta"
        m = [(a + 5, a + 27, strand, 9), (a + 40, a + 61, "+-"[k % 2], 3)][:int(rng.integers(0, 3))]
        plus = idx.extend_region_sequence(seqid, (a, b))
        rec = R.LocusRecord(seqid, (a, b), strand, (a + 5, a + 27), "0LR"[k % 3], [(a + 5, a + 27, strand)], m, plus)
        recs_seq.append(rec)
        recs_none.append(rec._replace(seq=None))
    with mf.upload_genome(idx) as g:
        with R.fold_records(mf, recs_seq, 300) as want, R.fold_records(mf, recs_none, 300, genome=g) as got:
            assert list(got.structures(55)) == list(want.structures(55))
            assert got.rnalfold_text() == want.rnalfold_text()
        ss_w, tab_w, cand_w = R.candidates_of_records(mf, recs_seq, 300)
        ss_g, tab_g, cand_g = R.candidates_of_records(mf, recs_none, 300, genome=g)
        assert ss_g == ss_w and tab_g._table == tab_w._table and cand_g.nverdicts == cand_w.nverdicts > 20


# ------------------------------------------------------------------------------------ reference pin (GPU)
def _run_ours(aln, ssrecs, allow_no_star, details, maturestar):
    sys.path.insert(0, GOLDEN)
    import predict_stub as PS
    from mir_prefer_b200 import predict as P
    return [PS.canon(x) for x in P.filter_next_loci(
        aln, ssrecs, PS.mapinfo_stub, PS.SAMPLES, True, allow_no_star, details, 18, 24, 20, maturestar, PS.check_expression_stub)]


@pytest.mark.gpu
def test_end_to_end_mirna_list_from_genome(mf, tmp_path):
    """The composed end-to-end fixture (tests/golden/e2e_mirna.json: the reference's binary + parser + filter_next_loci)
    through the genome path: one contig per record ('N' padding, then the plus-strand bases at the region), records without
    sequences, candidates_of_records(genome=g) and the consumer with the records' original seqids."""
    d = json.load(open(os.path.join(GOLDEN, "e2e_mirna.json")))
    for case in d["cases"]:
        recs = [R.LocusRecord(x[0], tuple(x[1]), x[2], tuple(x[3]), x[4], [tuple(p) for p in x[5]], [tuple(m) for m in x[6]], x[7])
                for x in case["records"]]
        assert sum(r.strand == "-" for r in recs) >= 60 and sum(r.seq != r.seq.upper() for r in recs) >= 10
        contigs = [("rec%d" % k, "N" * (r.region[0] - 1) + r.seq) for k, r in enumerate(recs)]
        idx = _write_fasta(tmp_path / ("e2e_%d.fa" % case["seed"]), contigs)
        coord = [r._replace(seqid="rec%d" % k, seq=None) for k, r in enumerate(recs)]
        with mf.upload_genome(idx) as g:
            ssrecs, table, cand = R.candidates_of_records(mf, coord, d["span"], genome=g)
        assert cand.nverdicts > 100 and cand.nstructs > 100
        aln = [[[r.seqid, r.region, r.strand], r.tag, {}, list(r.matures)] for r in recs]
        for key in ("11", "10", "01", "00"):
            got = _run_ours(aln, ssrecs, key[0] == "1", key[1] == "1", table)
            assert got == case["expected"][key], (case["seed"], key)
