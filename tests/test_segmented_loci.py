"""Segmented folds of long tiled loci (mirfold_plan_segments; fold_segmented in host.cu).  A tiled locus larger than its
device entry's memory budget is folded as segments of owned tiles plus halo tiles, from the 3' end; the result must be
byte-identical to the fold of the whole band.

CPU: the exported planner -- order, partition, halo reach, bytes.  GPU: forced segmentation through a small
MIRFOLD_MEM_BUDGET_MB in a context of its own, against the same library's unsegmented fold and the CPU oracle, planted cases
at segment edges, every fold entry point on batches that mix segmented and ordinary records, and loci beyond HBM."""
import contextlib
import os

import numpy as np
import pytest

import mir_prefer_b200 as mp
from mir_prefer_b200.fold import plan_fill_units, plan_segments
from test_genome_regions import _cands, _folds, _table, _write_fasta
from test_long_loci import _hits_above, _locus, _shifted, assert_suffix_local

SPANS = [5, 9, 20, 28, 100, 150, 299, 300, 306, 500, 544, 545, 799, 800]
MAX_N = (1 << 30) - 1
FLAG_SERIAL = 2


def _check_plan(n, L, budget):
    """Every property the engine relies on, for one (n, L, budget)."""
    f = plan_fill_units(n, L)
    p = plan_segments(n, L, budget)
    whole = plan_segments(n, L, 1 << 62)
    assert len(whole) == 1 and whole["halo_tiles"][0] == 0
    if f["n_units"] <= 1 or int(whole["device_bytes"][0]) <= budget:   # fits, or one unit: today's path
        assert len(p) == 1 and (p["tile_first"][0], p["tile_last"][0]) == (0, max(f["n_units"] - 1, 0))
        assert (p["row_first"][0], p["row_last"][0]) == (1, n)
        return p
    S, last, Ls = f["tile_step"], f["n_units"] - 1, min(L, n)
    # 3' end first; owned tiles partition [0, tile_last] exactly once; owned rows are the tiles' rows
    assert p["tile_last"][0] == last and p["tile_first"][-1] == 0
    assert (p["tile_first"] <= p["tile_last"]).all()
    assert (p["tile_last"][1:] == p["tile_first"][:-1] - 1).all()
    assert (p["row_first"] == p["tile_first"].astype(np.int64) * S + 1).all()
    hi = np.where(p["tile_last"] == last, n, (p["tile_last"].astype(np.int64) + 1) * S)
    assert (p["row_last"] == hi).all()
    # the worst row of every segment, its last owned row (the clamped last tile's too): every row up to min(n, i + L* + 1)
    # is owned or in the halo (owner tile of a row: min((i - 1) // S, tile_last))
    reach = np.minimum(n, hi + Ls + 1)
    owner = np.minimum((reach - 1) // S, last)
    assert (owner == p["tile_last"].astype(np.int64) + p["halo_tiles"]).all()
    assert (p["tile_last"].astype(np.int64) + p["halo_tiles"] <= last).all()
    # bytes within the budget, except a segment of one owned tile (the smallest there is)
    one = p["tile_first"] == p["tile_last"]
    assert ((p["device_bytes"] <= budget) | one).all()
    return p


@pytest.mark.parametrize("L", SPANS)
def test_plan_segments_partition_and_halo(L):
    tl = plan_fill_units(1 << 20, L)["tile_len"]
    checked = 0
    for n in (tl + 1, tl + 2, 3 * tl, 20_000, 300_001, 9_999_991, MAX_N):
        p1 = plan_fill_units(n, L)
        whole = int(plan_segments(n, L, 1 << 62)["device_bytes"][0])
        seq_bytes = 16 * n
        budgets = {whole, whole + 1, whole - 1, whole // 2, whole // 7, seq_bytes + whole // max(p1["n_units"], 1) * 3, 1 << 20, 0}
        if n == MAX_N:   # millions of segments: keep to the extremes
            budgets = {whole, whole - 1, whole // 3, 0}
        for b in sorted(budgets):
            p = _check_plan(n, L, b)
            checked += len(p)
            if b >= whole:
                assert len(p) == 1
            elif p1["n_units"] > 1:
                assert len(p) > 1
    assert checked > 100


def test_plan_segments_halo_sizes_and_errors():
    """Halo tiles: 1 at spans up to 300, 2 at 500 (864-nt tiles, step 364), 13 at 800 (step 64); untiled spans are one unit."""
    for L, halo in ((9, 1), (150, 1), (300, 1), (500, 2), (800, 13)):
        p = plan_segments(300_000, L, 1 << 20)
        assert len(p) > 10 and p["halo_tiles"][0] == 0 and p["halo_tiles"].max() == halo and (p["halo_tiles"][-5:] == halo).all(), L
    assert len(plan_segments(2_000_000, 801, 1 << 20)) == 1          # one generic unit: out of scope, never segmented
    assert len(plan_segments(500, 300, 0)) == 1
    with pytest.raises(mp.MirfoldError):
        plan_segments(1 << 30, 300, 1 << 30)
    with pytest.raises(mp.MirfoldError):
        plan_segments(1000, 4, 1 << 30)


def test_plan_segments_maize_chr1_at_default_span():
    """What the engine runs for a 308 Mb contig at L = 300 with a 48 GB lane: ~1.9 TB by locus_bytes, folded in segments of
    at most the lane's bytes, each refilling one halo tile."""
    n, L, lane = 308_000_000, 300, 48 << 30
    p = _check_plan(n, L, lane)
    whole = int(plan_segments(n, L, 1 << 62)["device_bytes"][0])
    assert whole > 1.8e12 and 30 <= len(p) <= 60 and (p["device_bytes"] <= lane).all()
    owned = int((p["tile_last"] - p["tile_first"] + 1).sum())
    assert int(p["halo_tiles"].sum()) / owned < 1e-4


# ------------------------------------------------------------------------------------------------------------------ GPU
@contextlib.contextmanager
def budget_ctx(mb, devices=None):
    """A fresh context whose device entries each have a budget of `mb` MiB (segments get half of it: one lane's share)."""
    old = os.environ.get("MIRFOLD_MEM_BUDGET_MB")
    os.environ["MIRFOLD_MEM_BUDGET_MB"] = str(int(mb))
    try:
        ctx = mp.MirFold(devices=devices)
    finally:
        if old is None:
            del os.environ["MIRFOLD_MEM_BUDGET_MB"]
        else:
            os.environ["MIRFOLD_MEM_BUDGET_MB"] = old
    with ctx:
        yield ctx


def _whole_bytes(n, L):
    return int(plan_segments(n, L, 1 << 62)["device_bytes"][0])


def _seg_plan(n, L, mb, serial=False):
    return plan_segments(n, L, (mb << 20) // (1 if serial else 2))


def _edge_evidence(hits, plan):
    """Edges (a segment's first row r: rows below r belong to the segments after it) that a printed hit spans, and
    segments whose own traceback starts (rows row_first+1 .. row_last+1) include a printed hit."""
    starts = np.array([h[2] for h in hits])
    ends = np.array([h[2] + len(h[0]) - 1 for h in hits])
    crossed = sum(bool(((starts < r) & (ends >= r)).any()) for r in plan["row_first"][:-1].tolist())
    with_hit = sum(bool(((starts > a) & (starts <= b + 1)).any()) for a, b in zip(plan["row_first"].tolist(), plan["row_last"].tolist()))
    return crossed, with_hit


CASES = [(9, 40_000, True), (20, 30_000, True), (100, 50_000, True), (150, 120_000, False), (299, 45_000, True),
         (300, 300_000, False), (306, 50_000, True), (500, 200_000, False), (800, 60_000, False)]


@pytest.mark.gpu
@pytest.mark.parametrize("L,n,with_oracle", CASES, ids=["L%d-%dk" % (c[0], c[1] // 1000) for c in CASES])
def test_segmented_equals_unsegmented(mf, oracle, L, n, with_oracle):
    """Hits and total equal the unsegmented fold (and the oracle up to 50 kb) at several budgets per locus, from segments of
    one owned tile to a few segments; printed hits span segment edges and every segment's decisions cross into the next."""
    s = _locus(7000 + L, n, L, tail=n // 3)
    with mf.fold([s], L) as res:
        want = (res.hits(0), res.total(0))
        assert res.stats["n_chunks"] == 1
    if with_oracle:
        o = oracle.fold(s, L)
        assert want == (o["hits"], o["total"])
    whole = _whole_bytes(n, L)
    crossed = 0
    for frac in (3, 11, 40, 1000):
        mb = max(1, whole // frac >> 20)
        plan = _seg_plan(n, L, mb)
        if len(plan) > 400:   # L = 800 at tiny budgets: 13 halo tiles per owned tile; one-tile segments on a shorter locus below
            continue
        assert len(plan) > 1
        with budget_ctx(mb) as ctx, ctx.fold([s], L) as res:
            assert res.stats["n_chunks"] == 1 and res.stats["fill_units"] >= plan_fill_units(n, L)["n_units"]
            assert (res.hits(0), res.total(0)) == want, mb
        c, w = _edge_evidence(want[0], plan)
        crossed += c
        assert w >= len(plan) - 1
    assert crossed > 0
    # segments of one owned tile (at L = 800 each with a 13-tile halo: on the locus' 3' 20 kb)
    if len(plan_segments(n, L, 1)) > 400:
        s = s[-20_000:]
        with mf.fold([s], L) as res:
            want = (res.hits(0), res.total(0))
    p1 = _seg_plan(len(s), L, 1)
    assert len(p1) <= 400 and (p1["tile_first"] == p1["tile_last"]).all()
    with budget_ctx(1) as ctx, ctx.fold([s], L) as res:
        assert (res.hits(0), res.total(0)) == want


def _traceback_starts(f3, n):
    """k_plan on the whole f3 vector: RNALfold's traceback starts in print order (descending)."""
    f3 = [int(x) for x in f3[:n + 3]]
    out, do_bt, have_prev, fnext = [], False, False, f3[n - 3]
    for i in range(n - 4, 0, -1):
        if f3[i] != fnext:
            do_bt = True
        elif do_bt:
            out.append(i + 1)
            have_prev, do_bt = True, False
        if i == 1 and (do_bt or not have_prev):
            out.append(1)
        fnext = f3[i]
    return out


def _carried_decisions(starts, hits, plan):
    """The last traceback of every segment but the last is decided against the first one of the segment below (k_emit_seg,
    entry 0).  Returns (suppressed, compared): carried tracebacks RNALfold dropped, and carried tracebacks printed after the
    structure compare (the one below reaches at least as far, so its slot was compared with the carried slot).  A
    traceback is printed iff a hit has its start."""
    st = np.array(starts)
    length = {h[2]: len(h[0]) for h in hits}
    sup = cmp = 0
    for a, b in zip(plan["row_first"][:-1].tolist(), plan["row_last"][:-1].tolist()):
        own = st[(st > a) & (st <= b + 1)]
        below = st[st <= a]
        if len(own) and len(below):
            x, y = int(own.min()), int(below.max())
            if x not in length:
                sup += 1
            elif y in length and y + length[y] >= x + length[x]:
                cmp += 1
    return sup, cmp


def _plant_at(base, pos, motif):
    return base[:pos - 1] + motif + base[pos - 1 + len(motif):]


@pytest.mark.gpu
@pytest.mark.parametrize("L", [100, 300])
def test_planted_cases_at_segment_edges(mf, oracle, L):
    """Planted at a segment edge r (a segment's lowest owned row): hairpins shifted across r so that printed hits start at
    r (traced by the segment below from its halo) and at r + 1 (traced from the lowest plan row of the segment above), the
    structures RNALfold drops because the next (lower) traceback contains them, on either side of r -- the tracebacks are
    recomputed from the fold's f3 to show that carried entries were decided by comparing their slot with the first
    structure of the segment below; and a
    poly-A f3 plateau longer than a segment spanning edges, so that a segment has no traceback of its own and the carried
    one passes through it."""
    n, mb = 24_000, 1
    rng = np.random.default_rng(L)
    base = "".join(np.array(list("ACGU"))[rng.integers(0, 4, n)].tolist())
    plan = _seg_plan(n, L, mb)
    assert len(plan) > 5
    r = int(plan["row_first"][len(plan) // 2])
    hp = "GGGCGCAGUUCGCUGCGCCC"
    starts_seen = set()
    compared = 0
    with budget_ctx(mb) as ctx:
        for shift in range(-6, 5):
            s = _plant_at(base, r + shift, "AAAA" + hp + "AAAA")
            with mf.fold([s], L) as a, ctx.fold([s], L) as b:
                want = (a.hits(0), a.total(0))
                assert (b.hits(0), b.total(0)) == want, shift
                starts_seen |= {h[2] for h in want[0]}
            sup, cmp = _carried_decisions(_traceback_starts(mf.debug_matrices(s, L)[2], n), want[0], plan)
            compared += sup + cmp
        assert {r, r + 1} <= starts_seen
        assert compared > 0
        # plateau: poly-A over three segments around the middle one
        lo, hi = int(plan["row_first"][len(plan) // 2 + 1]) - 50, int(plan["row_last"][len(plan) // 2 - 1]) + 50
        s = base[:lo - 1] + "A" * (hi - lo + 1) + base[hi:]
        with mf.fold([s], L) as a, ctx.fold([s], L) as b:
            assert (b.hits(0), b.total(0)) == (a.hits(0), a.total(0))
            assert not any(lo + 4 < h[2] < hi - L - 4 for h in a.hits(0))
        o = oracle.fold(s, L)
        with ctx.fold([s], L) as b:
            assert (b.hits(0), b.total(0)) == (o["hits"], o["total"])


# ------------------------------------------------------------------------------------------ every entry point, mixed batch
L_MIX, MB_MIX = 300, 48


def _mixed(seed=3):
    rng = np.random.default_rng(seed)
    seqs = [_locus(seed, 90_000, L_MIX, tail=30_000)]
    for k in range(30):
        m = int(rng.integers(3, 2500))
        seqs.append("".join(np.array(list("ACGT"))[rng.integers(0, 4, m)].tolist()))
    seqs.insert(7, _locus(seed + 1, 70_000, L_MIX, tail=20_000))
    return seqs


@pytest.mark.gpu
def test_mixed_batch_every_entry_point(mf, tmp_path):
    seqs = _mixed()
    assert _whole_bytes(90_000, L_MIX) > MB_MIX << 20 and _whole_bytes(2500, L_MIX) < MB_MIX << 19
    buf, off = mf.pack(seqs)
    with mf.fold(seqs, L_MIX) as w:
        want = _folds(w)
    names = ["c%d" % k for k in range(len(seqs))]
    idx = _write_fasta(tmp_path / "g.fa", list(zip(names, seqs)))
    rows = [(k, 1, len(s) + 1, "+-"[k % 2]) for k, s in enumerate(seqs)]
    regions = [[a, b] for _, a, b, _ in rows]
    matures = [(a + 40, a + 61, "+", 5) for _, a, _, _ in rows]
    moff = np.arange(len(rows) + 1, dtype=np.uint64)
    text = "".join(">r%d\n%s\n" % (k, s) for k, s in enumerate(seqs))
    with mf.upload_genome(idx) as g, g.fold_regions(_table(rows), L_MIX) as wr:
        want_r = _folds(wr)
        want_c = _cands(mf.fold_candidates(buf, off, L_MIX, regions, matures, moff))
        want_cr = _cands(g.fold_candidates(_table(rows), L_MIX, matures, moff))
    want_text = mf.fold_text(text, L_MIX)
    want_shuf = mf.shuffle_test(seqs[:9], 3, seed=5, span=L_MIX)
    for devices, flags in ((None, 0), ([0, 0], 0), (None, FLAG_SERIAL)):
        with budget_ctx(MB_MIX, devices) as ctx:
            with ctx.fold(seqs, L_MIX, flags) as got:
                assert _folds(got) == want, (devices, flags)
                assert got.stats["n_chunks"] >= 2
            chunks = {}

            def sink(ch):
                for k, r in enumerate(ch.records.tolist()):
                    assert r not in chunks
                    chunks[r] = (ch.hits(k), int(ch.total_mfe_dcal[k]))

            ctx.fold_stream(buf, off, L_MIX, sink, flags)
            assert [chunks[r] for r in range(len(seqs))] == want
            with ctx.upload(buf, off, L_MIX) as batch, batch.fold(download=True, flags=flags) as got:
                assert _folds(got) == want
            assert _cands(ctx.fold_candidates(buf, off, L_MIX, regions, matures, moff, flags=flags)) == want_c
            with ctx.upload_genome(idx) as g:
                with g.fold_regions(_table(rows), L_MIX, flags) as got:
                    assert _folds(got) == want_r
                chunks.clear()
                g.fold_regions_stream(_table(rows), L_MIX, sink, flags)
                assert [chunks[r] for r in range(len(seqs))] == want_r
                assert _cands(g.fold_candidates(_table(rows), L_MIX, matures, moff, flags=flags)) == want_cr
            if devices is None and flags == 0:
                assert ctx.fold_text(text, L_MIX) == want_text
                assert ctx.shuffle_test(seqs[:9], 3, seed=5, span=L_MIX).tolist() == want_shuf.tolist()


@pytest.mark.gpu
def test_fold_device_mixed_batch(mf):
    """mirfold_fold_device leaves the results in HBM and returns counts only: hits and tracebacks must match (a count
    check; the hits themselves are compared through the other entry points above)."""
    import torch
    seqs = _mixed(9)
    buf, off = mf.pack(seqs)
    d = torch.from_numpy(buf).cuda()
    torch.cuda.synchronize()
    with mf.fold_device(d.data_ptr(), off, L_MIX) as want:
        wn, wt = want.nhits, want.stats["tracebacks"]
    with budget_ctx(MB_MIX) as ctx, ctx.fold_device(d.data_ptr(), off, L_MIX) as got:
        assert got.nhits == wn > 1000 and got.stats["tracebacks"] == wt


# ---------------------------------------------------------------------------------------------------------- beyond HBM
def _free_device_bytes():
    import torch
    return torch.cuda.mem_get_info()[0]


@pytest.mark.gpu
def test_contig_beyond_device_memory_from_resident_genome(oracle, tmp_path):
    """A 40 Mb seeded contig at L = 300 (about 247 GB by locus_bytes, more than the B200's 180 GB) folded from a resident
    genome in the default context.  Before segmented folds the whole band was allocated at once and the call returned
    MIRFOLD_ERR_NOMEM.  Its 3'-most ~20 kb of hits match the oracle by suffix locality; the total is at most every hit's
    energy."""
    n, L = 40_000_000, 300
    whole = _whole_bytes(n, L)
    need, free = 16 * n + (3 << 30), _free_device_bytes()
    assert whole > 240e9
    if free < need:
        pytest.skip("the 40 Mb locus needs about %d device bytes beyond its band segments, %d free" % (need, free))
    s = _locus(40, n, L, tail=30_000)
    idx = _write_fasta(tmp_path / "chr.fa", [("chr1", s.replace("U", "T"))], width=80)
    i0 = n - 20_000
    with mp.MirFold() as ctx, ctx.upload_genome(idx) as g, g.fold_regions(_table([(0, 1, n + 1, "+")]), L) as res:
        assert res.stats["n_chunks"] == 1
        whole_hits = _hits_above(res, 0, i0)
        total = res.total(0)
        assert total <= int(res.hit_table["mfe_dcal"][int(res.hit_begin[0]):int(res.hit_begin[0]) + int(res.hit_count[0])].min())
    assert len(whole_hits) > 100
    assert_suffix_local(whole_hits, _shifted(oracle.fold(s[i0 - 1:], L)["hits"], i0))


@pytest.mark.gpu
def test_12mb_locus_segmented_equals_unsegmented():
    """A ~12 Mb locus at L = 300 (about 74 GB): whole band in the default context, segments in a 16 GB one; hits and total
    byte-identical."""
    n, L = 12_000_000, 300
    whole = _whole_bytes(n, L)
    free = _free_device_bytes()
    if whole > 0.6 * free or whole > (96 << 30):   # the default context's budget: min(60 % of free, 96 GB)
        pytest.skip("the unsegmented 12 Mb fold needs about %d device bytes, %d free" % (whole, free))
    s = _locus(12, n, L)
    with mp.MirFold() as ctx, ctx.fold([s], L) as a:
        want = (a.hits(0), a.total(0))
    assert len(_seg_plan(n, L, 16 << 10)) > 5
    with budget_ctx(16 << 10) as ctx, ctx.fold([s], L) as b:
        assert (b.hits(0), b.total(0)) == want
