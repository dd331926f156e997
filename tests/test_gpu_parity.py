"""GPU (-m gpu): libmirfold through the C ABI vs the oracle / golden RNALfold text, bit-exact."""
import hashlib
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN, golden_cases
from mir_prefer_b200.corpus import lcg_records, records_to_fasta, synth_loci

pytestmark = pytest.mark.gpu


def assert_same(mf, oracle, seqs, L):
    with mf.fold(seqs, L) as res:
        assert res.nseq == len(seqs)
        for r, s in enumerate(seqs):
            o = oracle.fold(s, L)
            assert res.hits(r) == o["hits"], (r, len(s), L)
            assert res.total(r) == o["total"], (r, len(s), L)
        return res.stats


@pytest.mark.parametrize("name,L", golden_cases())
def test_fold_text_matches_reference_golden(mf, name, L):
    """RNALfold CLI contract: byte-identical text to the reference binary's committed output."""
    text = open(os.path.join(GOLDEN, name + ".in")).read()
    want = open(os.path.join(GOLDEN, "%s.L%d.out" % (name, L))).read()
    assert mf.fold_text(text, L) == want


@pytest.mark.parametrize("seed", [3, 1, 2])
def test_sha256_pins(mf, seed):
    p = next(x for x in json.load(open(os.path.join(GOLDEN, "pins.json")))["pins"] if x["seed"] == seed)
    text = records_to_fasta(lcg_records(p["seed"], p["nrec"], p["lo"], p["span"]))
    out = mf.fold_text(text, p["L"])
    assert len(out) == p["stdout_bytes"]
    assert hashlib.sha256(out.encode()).hexdigest() == p["sha256_stdout"]


def test_matrices_cell_for_cell(mf, oracle):
    """c / fML / f3 against the oracle's intermediate matrices (which RNALfold cannot expose)."""
    for s, L in ((synth_loci(5, 1, (60, 60))[0], 30), (synth_loci(6, 1, (320, 320))[0], 300),
                 (synth_loci(7, 1, (400, 400))[0], 150), ("GC" * 40, 300)):
        o = oracle.fold(s, L, matrices=True)
        c, m, f3 = mf.debug_matrices(s, L)
        n = len(s)
        assert (o["c"] == c).all()
        assert (np.minimum(o["m"], 1000000) == np.minimum(m, 1000000)).all()
        assert (o["f3"][:n + 3] == f3[:n + 3]).all()


def test_wide_kernel_flag_gives_identical_results(mf, oracle):
    """MIRFOLD_FLAG_WIDE forces the 32-bit fill kernel for every locus; both kernels are bit-exact."""
    from mir_prefer_b200.fold import FLAG_WIDE
    seqs = synth_loci(21, 48, "parity") + synth_loci(22, 24, (20, 200)) + synth_loci(23, 8, (610, 900))
    with mf.fold(seqs, 300) as a, mf.fold(seqs, 300, flags=FLAG_WIDE) as b:
        for r, s in enumerate(seqs):
            assert a.hits(r) == b.hits(r) and a.total(r) == b.total(r)
            if r % 8 == 0:
                o = oracle.fold(s, 300)
                assert a.hits(r) == o["hits"] and a.total(r) == o["total"]
    s = synth_loci(6, 1, (320, 320))[0]
    for fl in (0, FLAG_WIDE):
        o = oracle.fold(s, 300, matrices=True)
        c, m, f3 = mf.debug_matrices(s, 300, flags=fl)
        assert (o["c"] == c).all() and (np.minimum(o["m"], 1000000) == np.minimum(m, 1000000)).all()
        assert (o["f3"][:len(s) + 3] == f3[:len(s) + 3]).all()


def test_energies_below_16bit_range_fall_back_to_wide_kernel(mf, oracle):
    """Windows below -320 kcal/mol (perfect GC helices) leave the 16-bit ring's range: the locus is
    flagged on the device and redone by the 32-bit kernel, transparently."""
    seqs = ["GC" * 150, "G" * 148 + "AAAA" + "C" * 148, "GC" * 100 + "A" * 7 + "GC" * 100,
            "G" * 100 + "UUCG" + "C" * 100, "GGGGCCCC" * 60, synth_loci(5, 1, (300, 300))[0]]
    for L in (300, 150):
        assert_same(mf, oracle, seqs, L)
    o = oracle.fold(seqs[0], 300, matrices=True)
    assert o["c"].min() < -32000          # the case really is out of range
    c, m, f3 = mf.debug_matrices(seqs[0], 300)
    assert (o["c"] == c).all() and (np.minimum(o["m"], 1000000) == np.minimum(m, 1000000)).all()


def test_edge_lengths_and_empty(mf, oracle):
    seqs = ["", "A", "ACG", "ACGU", "GCGCA", "GGGAAACCC", "GGGGAAAACCCC", "A" * 21, "ACGUNNNACGU", "N" * 50,
            "GGGGGTTTTCCCCCAAAAGGGGGTTTTCCCCC"]
    for L in (5, 6, 10, 30, 300):
        assert_same(mf, oracle, seqs, L)
    with mf.fold([], 300) as res:
        assert res.nseq == 0 and res.nhits == 0


def test_alphabet_iupac_lowercase(mf, oracle):
    rng = np.random.default_rng(3)
    seqs = ["".join(rng.choice(list("ACGUTacgutNnKXIRYkxi"), size=int(rng.integers(5, 200)))) for _ in range(60)]
    assert_same(mf, oracle, seqs, 40)
    assert_same(mf, oracle, seqs, 300)


def test_sequence_families(mf, oracle):
    rng = np.random.default_rng(4)
    seqs = []
    for k in range(30):
        n = int(rng.integers(40, 420))
        alpha, p = [("GC", None), ("AU", None), ("ACGU", [.15, .35, .35, .15]), ("ACGU", None)][k % 4]
        seqs.append("".join(rng.choice(list(alpha), size=n, p=p)))
    assert_same(mf, oracle, seqs, 300)
    assert_same(mf, oracle, seqs, 61)


def test_parity_config_sample(mf, oracle):
    """cfg-2 shape (300-600 nt, L=300): seeded sample small enough for the oracle."""
    assert_same(mf, oracle, synth_loci(1001, 48, "parity"), 300)


def test_arabidopsis_length_law(mf, oracle):
    assert_same(mf, oracle, synth_loci(1002, 48, "arabidopsis"), 300)


def test_span_sweep(mf, oracle):
    seqs = synth_loci(1004, 24, "sweep")
    for L in (150, 300, 500):
        assert_same(mf, oracle, seqs, L)


def test_long_loci(mf, oracle):
    assert_same(mf, oracle, synth_loci(1003, 2, "long") + synth_loci(12, 4, (1000, 2000)), 300)


def test_tiled_long_loci_edges(mf, oracle):
    """Loci longer than 608 nt are filled as overlapping tiles (LocusDesc::tile_*): 608-nt tiles at spans < 300 (step
    608-L), 864-nt tiles from L=300 on (step 864-L; more in test_big_tile_bucket_edges).  Lengths around every tile-count
    boundary of both at L=299 (step 309) and L=300 (step 564), and other spans, cell for cell and hit for hit."""
    from mir_prefer_b200.fold import plan_fill_units
    lens = [609, 610, 864, 865, 917, 918, 1226, 1227, 1428, 1429, 2500]
    seqs = [synth_loci(400 + n, 1, (n, n))[0] for n in lens]
    st = assert_same(mf, oracle, seqs, 300)
    assert [plan_fill_units(n, 300)["n_units"] for n in lens] == [1, 1, 1, 2, 2, 2, 2, 2, 2, 3, 4]
    assert st["fill_units"] == 22
    st = assert_same(mf, oracle, seqs, 299)
    assert [plan_fill_units(n, 299)["n_units"] for n in lens] == [2, 2, 2, 2, 2, 3, 3, 4, 4, 4, 8]
    assert st["fill_units"] == 36
    assert_same(mf, oracle, seqs[:6], 150)
    assert_same(mf, oracle, seqs[:4], 500)
    assert_same(mf, oracle, seqs[3:6], 544)    # 864-nt tiles (the last span a 608-nt tile could hold)
    assert_same(mf, oracle, seqs[:2], 545)
    for L in (5, 9, 31, 40):                   # f3 CTA kernel windows at tiny spans
        assert_same(mf, oracle, seqs[:2], L)
    for s, L in ((seqs[3], 300), (seqs[5], 150), (seqs[1], 500), (seqs[6], 299)):
        o = oracle.fold(s, L, matrices=True)
        c, m, f3 = mf.debug_matrices(s, L)
        assert (o["c"] == c).all()
        assert (np.minimum(o["m"], 1000000) == np.minimum(m, 1000000)).all()
        assert (o["f3"][:len(s) + 3] == f3[:len(s) + 3]).all()
    # a long GC helix leaves the 16-bit range inside some tiles only: those tiles are redone wide
    s = synth_loci(77, 1, (400, 400))[0] + "GC" * 160 + synth_loci(78, 1, (500, 500))[0]
    assert_same(mf, oracle, [s], 300)


def test_big_tile_bucket_edges(mf, oracle):
    """Spans >= 300 put loci longer than 608 nt into the stride-864 bucket (one 1024-thread CTA per unit): a single unit up
    to 864 nt, overlapping 864-nt tiles beyond (step 864-L).  Lengths around every tile-count boundary for L=500 (step 364),
    the last tiled span (L=800: 64 owned rows per tile), the first span at which longer loci use the generic kernel again
    (L=801, while loci <= 864 nt stay in the bucket with diagonals up to n-1), cell for cell and hit for hit."""
    from mir_prefer_b200.fold import plan_fill_units
    lens = [864, 865, 1228, 1229, 1593]
    seqs = [synth_loci(900 + n, 1, (n, n))[0] for n in lens]
    st = assert_same(mf, oracle, seqs, 500)
    plans = [plan_fill_units(n, 500) for n in lens]
    assert [p["n_units"] for p in plans] == [1, 2, 2, 3, 4] and all(p["kernel"] == 864 for p in plans)
    assert st["fill_units"] == 12
    assert_same(mf, oracle, [seqs[1], seqs[3]], 800)
    assert plan_fill_units(1229, 800)["n_units"] == 7
    assert_same(mf, oracle, [seqs[0], seqs[1] + "A"], 801)
    assert plan_fill_units(864, 801)["kernel"] == 864 and plan_fill_units(866, 801)["kernel"] == 0
    for s, L in ((seqs[3], 500), (seqs[0], 801)):
        o = oracle.fold(s, L, matrices=True)
        c, m, f3 = mf.debug_matrices(s, L)
        assert (o["c"] == c).all()
        assert (np.minimum(o["m"], 1000000) == np.minimum(m, 1000000)).all()
        assert (o["f3"][:len(s) + 3] == f3[:len(s) + 3]).all()
    # a long GC helix leaves the 16-bit range inside one 864-nt tile only: that tile is redone by the 32-bit kernel
    s = synth_loci(77, 1, (500, 500))[0] + "GC" * 170 + synth_loci(78, 1, (600, 600))[0]
    assert_same(mf, oracle, [s], 500)


def test_randomized_lengths_and_spans(mf, oracle):
    """Seeded fuzz over (n, L): bucket boundaries (160/161, 352/353, 608/609), spans that are odd, tiny,
    equal to n, larger than n, and GC contents from 0.2 to 0.8 -- every record bit-exact vs the oracle."""
    rng = np.random.default_rng(20261017)
    edge_n = [5, 6, 9, 31, 32, 33, 159, 160, 161, 351, 352, 353, 607, 608, 609, 640]
    for L in (7, 37, 99, 161, 300, 353, 401):
        seqs = []
        for k in range(14):
            n = int(edge_n[(k + L) % len(edge_n)]) if k % 2 == 0 else int(rng.integers(5, 700))
            gc = float(rng.uniform(0.2, 0.8))
            p = [(1 - gc) / 2, gc / 2, gc / 2, (1 - gc) / 2]
            s = "".join(rng.choice(list("ACGT"), size=n, p=p))
            if k % 5 == 0 and n > 60:      # a planted perfect helix: deep energies, long stacks
                a = "".join(rng.choice(list("GC"), size=int(rng.integers(8, 25))))
                rc = a[::-1].translate(str.maketrans("GC", "CG"))
                s = s[:10] + a + "TTCG" + rc + s[10 + 2 * len(a) + 4:]
            seqs.append(s)
        assert_same(mf, oracle, seqs, L)


@pytest.mark.parametrize("pin", json.load(open(os.path.join(GOLDEN, "bulk_pins.json")))["pins"],
                         ids=lambda p: "%s-%d-L%d" % (p["law"], p["nloci"], p["span"]))
def test_full_size_configs_match_rnalfold_sha256(mf, pin):
    """Whole BASELINE configs at (or near) full size: the complete RNALfold-format text has the sha256 of the
    text the reference's own RNALfold binary produced on the same input (tools/bulk_parity.py, run once on a
    GPU box with oracle/_ref/RNALfold on all host cores; byte-identical there)."""
    seqs = synth_loci(pin["seed"], pin["nloci"], pin["law"])
    text = "".join(">locus%d:%d-%d + 1-22 0 1,22,+\n%s\n" % (k, 1, len(s) + 1, s) for k, s in enumerate(seqs))
    out = mf.fold_text(text, pin["span"])
    if "bytes" in pin:
        assert len(out) == pin["bytes"]
    assert hashlib.sha256(out.encode()).hexdigest() == pin["sha256"]


def test_native_text_path_equals_python_path(mf):
    """mirfold_fold_text (parse + fold + format natively) == the Python parser + mirfold_format_records, byte for byte, on the
    golden inputs and on awkward text: no final newline, '@' terminator, tabs / CR / blank-only lines, '*' lines, raw bytes."""
    for name in ("edge", "alphabet", "synth8"):
        text = open(os.path.join(GOLDEN, name + ".in")).read()
        for L in (30, 300):
            assert mf.fold_text_bytes(text, L) == mf.fold_text_bytes_py(text, L), (name, L)
    odd = ">h1 x\r\nGGGGAAAACCCC extra tokens\n\n   \n\tacgtacgtac\r\n*note\n>caf\u00e9\nACGUNNNACGU\n@\n>never\nGGGG\n"
    assert mf.fold_text_bytes(odd, 300) == mf.fold_text_bytes_py(odd, 300)
    assert b">never" not in mf.fold_text_bytes(odd, 300)
    tail = ">a\nGGGGGTTTTCCCCC"                           # no newline at the end
    assert mf.fold_text_bytes(tail, 300) == mf.fold_text_bytes_py(tail, 300)
    assert mf.fold_text_bytes(b"", 300) == b"" and mf.fold_text_bytes(b"\n", 300) == b"\n"
    raw = b">x\xff\xfe\nACGTACGTAA\n"
    assert mf.fold_text_bytes(raw, 300).startswith(b">x\xff\xfe\n")


def test_native_formatter_equals_python_formatter(mf):
    """mirfold_format_records() (C, multi-threaded) vs the Python format_record() on every record, including
    empty / tiny records, lower case and IUPAC letters, and more than 256 records (threaded path)."""
    from mir_prefer_b200 import format_record
    seqs = synth_loci(55, 300, (5, 420)) + ["", "acgu", "ACGTNNRYacgtn" * 9, "G" * 30 + "TTCG" + "C" * 30]
    with mf.fold(seqs, 300) as res:
        data, offs = res.record_blocks()
        assert len(offs) == len(seqs) + 1 and int(offs[-1]) == len(data)
        for r, s in enumerate(seqs):
            assert data[int(offs[r]):int(offs[r + 1])].decode() == format_record(s, res.hits(r), res.total(r)), r


def test_against_reference_binary_live(mf, oracle):
    """When the reference's own RNALfold travelled to this box (oracle/_ref), compare against it."""
    if not oracle.have_rlf():
        pytest.skip("oracle/_ref/RNALfold not staged")
    text = records_to_fasta([("s%d" % k, s) for k, s in enumerate(synth_loci(88, 24, "parity"))])
    assert mf.fold_text(text, 300) == oracle.fold_text(text, 300, binary=oracle.RLF)


def test_chunking_is_invisible(oracle):
    """Forcing many memory chunks must not change results (batch-composition independence)."""
    import mir_prefer_b200 as mp
    seqs = synth_loci(21, 40, (80, 400))
    os.environ["MIRFOLD_MEM_BUDGET_MB"] = "2"
    try:
        with mp.MirFold() as small, small.fold(seqs, 300) as a:
            assert a.stats["n_chunks"] > 3
            got = [(a.hits(r), a.total(r)) for r in range(len(seqs))]
    finally:
        del os.environ["MIRFOLD_MEM_BUDGET_MB"]
    assert got == [(o["hits"], o["total"]) for o in (oracle.fold(s, 300) for s in seqs)]


def _check_structure_properties(res, lens, L):
    hb, hc = res.hit_begin.astype(np.int64), res.hit_count.astype(np.int64)
    tab = res.hit_table
    # the per-record runs tile the hit table exactly once
    order = np.argsort(hb, kind="stable")
    nz = order[hc[order] > 0]
    assert hc.sum() == res.nhits and (hb[nz][1:] == (hb[nz] + hc[nz])[:-1]).all() and (len(nz) == 0 or hb[nz][0] == 0)
    assert (tab["len"] >= 1).all() and (tab["len"] <= L + 3).all()   # window touching the 3' end: up to L*+3 chars
    assert (tab["start"] >= 1).all()
    arena = res.arena
    # balanced brackets over the whole arena: every string is NUL-terminated, so a running depth
    # that returns to 0 at each NUL proves each structure is balanced
    depth = np.cumsum((arena == ord("(")).astype(np.int64) - (arena == ord(")")).astype(np.int64))
    nul = np.flatnonzero(arena == 0)
    assert (depth[nul] == 0).all()
    assert set(np.unique(arena).tolist()) <= {0, ord("("), ord(")"), ord(".")}
    rec_of_hit = np.empty(res.nhits, np.int64)
    rec_of_hit[np.repeat(hb, hc) + (np.arange(res.nhits) - np.repeat(np.cumsum(hc) - hc, hc))] = np.repeat(np.arange(res.nseq), hc)
    assert (tab["start"] + tab["len"] - 1 <= lens[rec_of_hit]).all()
    # every record with n >= 5 prints at least the final backtrack; total MFE <= every hit energy
    assert (hc[lens >= 5] >= 1).all()
    assert (res.total_mfe_dcal[rec_of_hit] <= tab["mfe_dcal"]).all()
    assert (res.total_mfe_dcal <= 0).all()


def test_full_size_properties_and_determinism(mf, oracle):
    """BASELINE configs[1] at full size (10k loci, 300-600 nt, L=300): size-independent properties,
    permutation invariance (checksum of per-record checksums) and oracle parity on a seeded sample."""
    seqs = synth_loci(1001, 10000, "parity")
    lens = np.array([len(s) for s in seqs])

    def digest(res, order):
        out = [None] * len(order)
        for k, r in enumerate(order):
            b = int(res.hit_begin[k])
            e = b + int(res.hit_count[k])
            h = hashlib.sha256()
            t = res.hit_table[b:e]   # explicit columns: a multi-field view would drag ss_off along in tobytes()
            h.update(np.stack([t["start"], t["len"], t["mfe_dcal"]]).astype("<i4").tobytes())
            if e > b:
                o0 = int(res.hit_table[b]["ss_off"])
                o1 = int(res.hit_table[e - 1]["ss_off"]) + int(res.hit_table[e - 1]["len"])
                h.update(res.arena[o0:o1].tobytes())
            h.update(int(res.total_mfe_dcal[k]).to_bytes(4, "little", signed=True))
            out[r] = h.digest()
        return hashlib.sha256(b"".join(out)).hexdigest()

    with mf.fold(seqs, 300) as res:
        _check_structure_properties(res, lens, 300)
        d1 = digest(res, list(range(len(seqs))))
        rng = np.random.default_rng(0)
        for r in rng.choice(len(seqs), size=12, replace=False):
            o = oracle.fold(seqs[r], 300)
            assert res.hits(int(r)) == o["hits"] and res.total(int(r)) == o["total"]
    perm = np.random.default_rng(1).permutation(len(seqs))
    with mf.fold([seqs[k] for k in perm], 300) as res2:
        assert digest(res2, perm.tolist()) == d1


def test_device_resident_entry_counts_match(mf):
    import torch
    seqs = synth_loci(31, 200, "arabidopsis")
    buf, off = mf.pack(seqs)
    with mf.fold_packed(buf, off, 300) as host:
        nh, nb = host.nhits, host.ss_bytes
    d = torch.from_numpy(buf.copy()).cuda()
    torch.cuda.synchronize()
    with mf.fold_device(d.data_ptr(), off, 300, stream=torch.cuda.current_stream().cuda_stream) as dev:
        assert dev.nhits == nh and dev.ss_bytes == nb and not dev.downloaded


def _records(res, n):
    return [(res.hits(r), res.total(r)) for r in range(n)]


def test_multi_device_sharding_matches_single(mf):
    """One context over several devices (LPT shards, one host thread per device, downloads straight into the shared
    result buffers) == the single-device result.  On a 1-GPU box the same ordinal is opened twice: two independent
    pipelines on one GPU run exactly the multi-device host path."""
    import torch
    import mir_prefer_b200 as mp
    ng = torch.cuda.device_count()
    devices = list(range(ng)) if ng >= 2 else [0, 0]
    seqs = synth_loci(41, 300, "parity") + ["", "ACG", "GGGAAACCC"] + synth_loci(42, 6, (700, 1500))
    with mf.fold(seqs, 300) as a:
        want = _records(a, len(seqs))
    with mp.MirFold(devices=devices) as m2, m2.fold(seqs, 300) as b:
        assert b.stats["n_devices"] == len(devices) and b.nhits == sum(len(h) for h, _ in want)
        assert _records(b, len(seqs)) == want
        _check_structure_properties(b, np.array([len(s) for s in seqs]), 300)
    # several chunks per device and both lanes in flight on every device
    os.environ["MIRFOLD_MEM_BUDGET_MB"] = "24"
    try:
        with mp.MirFold(devices=devices + [0]) as m3, m3.fold(seqs, 300) as c:
            assert c.stats["n_devices"] == len(devices) + 1 and c.stats["n_chunks"] >= 2 * len(devices)
            assert _records(c, len(seqs)) == want
    finally:
        del os.environ["MIRFOLD_MEM_BUDGET_MB"]


def test_result_buffer_overflow_path(mf):
    """The shared result buffers are sized from an estimate; chunks that do not fit take the overflow path and the
    result is rebuilt once at exact size.  MIRFOLD_RESULT_CAP_SCALE shrinks the estimate to force it.  The 12 kb locus
    is larger than the 16 MB budget and is folded in segments, so a segmented record takes the overflow path too."""
    import mir_prefer_b200 as mp
    from mir_prefer_b200.fold import plan_segments
    seqs = synth_loci(43, 120, (200, 420)) + synth_loci(47, 1, (12_000, 12_000))
    assert len(plan_segments(12_000, 300, (16 << 20) // 2)) > 1   # one lane's share of the budget
    with mf.fold(seqs, 300) as a:
        want = _records(a, len(seqs))
    os.environ["MIRFOLD_MEM_BUDGET_MB"] = "16"
    try:
        for scale in ("0.0", "0.3"):     # nothing fits / the first chunks fit, the rest overflows
            os.environ["MIRFOLD_RESULT_CAP_SCALE"] = scale
            with mp.MirFold(devices=[0, 0]) as m2, m2.fold(seqs, 300) as b:
                assert b.stats["n_chunks"] >= 4
                assert _records(b, len(seqs)) == want
                _check_structure_properties(b, np.array([len(s) for s in seqs]), 300)
    finally:
        del os.environ["MIRFOLD_MEM_BUDGET_MB"]
        os.environ.pop("MIRFOLD_RESULT_CAP_SCALE", None)


def test_serial_flag_and_lanes_give_identical_results(mf):
    from mir_prefer_b200.fold import FLAG_SERIAL
    import mir_prefer_b200 as mp
    seqs = synth_loci(44, 200, "arabidopsis")
    os.environ["MIRFOLD_MEM_BUDGET_MB"] = "64"
    try:
        with mp.MirFold() as m, m.fold(seqs, 300) as a, m.fold(seqs, 300, flags=FLAG_SERIAL) as b:
            assert a.stats["n_chunks"] >= 3 and b.stats["n_chunks"] >= 2
            assert _records(a, len(seqs)) == _records(b, len(seqs))
    finally:
        del os.environ["MIRFOLD_MEM_BUDGET_MB"]


def test_streamed_chunks_equal_whole_result(mf, oracle):
    """mirfold_fold_stream: every input record arrives in exactly one chunk, with the hits mirfold_fold returns;
    records shorter than 5 nt arrive in the final hit-less chunk; an exception in the callback aborts the fold."""
    import mir_prefer_b200 as mp
    seqs = synth_loci(45, 150, (60, 420)) + ["", "ACGU", "GGGGAAAACCCC"] + synth_loci(46, 3, (800, 1200))
    buf, off = mf.pack(seqs)
    with mf.fold_packed(buf, off, 300) as a:
        want = _records(a, len(seqs))
    os.environ["MIRFOLD_MEM_BUDGET_MB"] = "16"
    try:
        with mp.MirFold(devices=[0, 0]) as m2:
            got, devices = {}, set()

            def on_chunk(ch):
                devices.add(ch.device)
                for k, r in enumerate(ch.records.tolist()):
                    assert r not in got
                    got[r] = (ch.hits(k), int(ch.total_mfe_dcal[k]))

            st = m2.fold_stream(buf, off, 300, on_chunk)
            assert st["n_chunks"] >= 4 and -1 in devices
            assert [got[r] for r in range(len(seqs))] == want
            o = oracle.fold(seqs[7], 300)
            assert got[7] == (o["hits"], o["total"])

            def boom(ch):
                raise ValueError("stop")

            with pytest.raises(ValueError):
                m2.fold_stream(buf, off, 300, boom)
            with m2.fold_packed(buf, off, 300) as again:          # the context is still usable afterwards
                assert _records(again, len(seqs)) == want
    finally:
        del os.environ["MIRFOLD_MEM_BUDGET_MB"]


def test_resident_batch_matches_host_path(mf):
    """mirfold_batch_upload / mirfold_batch_fold: sequences resident in HBM on every device of the context."""
    import mir_prefer_b200 as mp
    seqs = synth_loci(47, 160, "arabidopsis") + ["", "ACG"]
    buf, off = mf.pack(seqs)
    with mf.fold_packed(buf, off, 300) as a:
        want = _records(a, len(seqs))
        nh, nb = a.nhits, a.ss_bytes
    with mp.MirFold(devices=[0, 0]) as m2, m2.upload(buf, off, 300) as batch:
        with batch.fold(download=False) as dev:
            assert dev.nhits == nh and dev.ss_bytes == nb and not dev.downloaded and dev.stats["n_devices"] == 2
        with batch.fold(download=True) as host:
            assert _records(host, len(seqs)) == want


def test_result_may_outlive_its_context():
    """mirfold_close() with live results defers the context's deletion (ADVICE r1: use-after-free)."""
    import gc
    import mir_prefer_b200 as mp
    seqs = synth_loci(48, 20, (100, 300))
    m = mp.MirFold()
    r1, r2 = m.fold(seqs, 300), m.fold(seqs[:5], 300)
    want = _records(r1, len(seqs))
    m.close()
    assert _records(r1, len(seqs)) == want       # the pinned buffers belong to the result
    r1.close()
    del r2
    gc.collect()
    with pytest.raises(mp.MirfoldError):
        m.fold(seqs, 300)


def test_bad_offsets_are_rejected(mf):
    import mir_prefer_b200 as mp
    buf = np.frombuffer(b"ACGUACGUACGU", np.uint8)
    with pytest.raises(mp.MirfoldError):
        mf.fold_packed(buf, np.array([0, 8, 4, 12], np.uint64), 300)


def test_fold_fasta_files_matches_golden_and_leaves_no_partial_file(mf, tmp_path, monkeypatch):
    """fold_use_RNALfold() replacement (MP:3047-3119): one output file per shard, byte-identical to RNALfold's, folded
    in line batches; CRLF / non-ASCII header bytes are echoed unchanged; a failing shard leaves neither the output nor
    a .tmp file behind (the reference only renames a completed shard, MP:3098)."""
    import mir_prefer_b200 as mp
    names = [("synth8", 300), ("edge", 300)]
    fas, outs = [], []
    for k, (name, L) in enumerate(names):
        fas.append(os.path.join(GOLDEN, name + ".in"))
        outs.append(str(tmp_path / ("x_rnalfoldoutput_%d" % k)))
    assert mf.fold_fasta_files(fas, outs, 300, batch_lines=5) == outs
    for (name, L), out in zip(names, outs):
        assert open(out, "rb").read() == open(os.path.join(GOLDEN, "%s.L%d.out" % (name, L)), "rb").read()
    assert sorted(os.listdir(tmp_path)) == ["x_rnalfoldoutput_0", "x_rnalfoldoutput_1"]
    # raw bytes in header lines
    odd = tmp_path / "odd.fa"
    odd.write_bytes(b">loc\xe9 1\r\nGGGGAAAACCCC\n>b\rc\nACGUACGUAC\n")
    mf.fold_fasta_files([str(odd)], [str(tmp_path / "odd.out")], 300)
    got = (tmp_path / "odd.out").read_bytes()
    assert got.startswith(b">loc\xe9 1\r\n") and b">b\rc\n" in got
    # failure in the second batch of the second shard
    calls = {"n": 0}
    real = mp.MirFold.fold_text_bytes

    def flaky(self, text, span, encoding=None):
        calls["n"] += 1
        if calls["n"] == 3:
            raise mp.MirfoldError(-2, "injected")
        return real(self, text, span, encoding)

    monkeypatch.setattr(mp.MirFold, "fold_text_bytes", flaky)
    outs2 = [str(tmp_path / "y_0"), str(tmp_path / "y_1")]
    with pytest.raises(mp.MirfoldError):
        mf.fold_fasta_files(fas, outs2, 300, batch_lines=10)
    left = sorted(f for f in os.listdir(tmp_path) if f.startswith("y_"))
    assert left in ([], ["y_0"]) and not any(f.endswith(".tmp") for f in os.listdir(tmp_path))
