"""Every loop-energy term of every fill kernel, on designed loci that oracle mutants prove decisive.

The band fill restates each two-loop energy in four forms: the 16-bit word-term schedule of k_fill_s16 (params.cu:
build_s16_schedule, a 17-slot ring rotating every 34 diagonals), the 32-bit skew schedule of k_fill_smem (gen_c / gen_us,
a 33-slot ring), the ilc pairing of k_fill_generic (a 64-slot global ring) and tb_loop_energy of the traceback.  A wrong
term goes unnoticed unless it is the unique minimiser of some cell of a tested fold.

A term class K is decisive on a design if the oracle with K raised by 1 dcal (oracle.fold(..., perturb=K)) gives a
different c matrix: K is then the unique minimiser of some cell, and a kernel whose K term is off by any non-zero amount
must differ from the oracle in that cell.  K is printed-decisive if the mutant also changes the printed hits.  Classes:
  shape  (n1, n2, parity of j-i): all 496 two-loop shapes (stacks, bulges, interior loops) at both parities
  ring   (s, d): two-loops of size s = n1 + n2 = 0..30 on 64 consecutive diagonals d (every slot of the 34-diagonal
         16-bit rotation, the 33-slot and the 64-slot rings)
  stack, int11, int21 (both orientations), int22, mismatchI entries of the six canonical pair types
  hairpin sizes 3..300 on designs (longer ones by the printed energy of long hairpins at L = 4096), every mismatchH and
         tetraloop entry, triloops of every closing pair
Designs come from deterministic templates (designs()): an outer GC helix, loop bases that cannot pair inside the loop
(A, or the table entry's own bases), an inner GC helix and an A hairpin whose length moves d.  tools/loop_corpus.py
searches seeds (other helix lengths, inner hairpins and GC helices around the same loop) for every design whose template
is not decisive and writes tests/golden/loop_corpus.json: those seeds, the sha256 of the expanded corpus and the
per-class counts, which the CPU tests pin.  Table entries that stay undecisive have loop bases that can pair across the
loop, or C / G loop bases that can pair with the helices: a stacked or slipped helix beats the loop in every seed tried.

c(i,j) depends only on bases i..j, so a design's cells are the same in any locus that contains it.  The GPU tests join the
designs into loci that select each fill kernel (plan_fill_units), compare c cell for cell in every design's block with
the design's own oracle fold, and compare one whole locus per kernel (c, fML, f3, hits, total) with the oracle.  Hairpins
longer than 300 nt are checked at sampled sizes only."""
import hashlib
import json
import os
from concurrent.futures import ThreadPoolExecutor
from multiprocessing import get_context

import numpy as np
import pytest

from conftest import GOLDEN
from mir_prefer_b200.fold import FLAG_WIDE

CORPUS_FILE = os.path.join(GOLDEN, "loop_corpus.json")
INF = 1000000
MAXLOOP = 30
PAIR = {1: "CG", 2: "GC", 3: "GU", 4: "UG", 5: "AU", 6: "UA"}
RTYPE = (0, 2, 1, 4, 3, 6, 5, 7)
BASES = "ACGU"                                   # codes 1..4
TETRALOOPS = ("GGGGAC GGUGAC CGAAAG GGAGAC CGCAAG GGAAAC CGGAAG CUUCGG CGUGAG CGAAGG CUACGG GGCAAC CGCGAG UGAGAG CGAGAG "
              "AGAAAU CGUAAG CUAACG UGAAAG GGAAGC GGGAAC UGAAAA AGCAAU AGUAAU CGGGAG AGUGAU GGCGAC GGGAGC GUGAAC UGGAAA").split()
RING_DIAGONALS = 64
HAIRPIN_MAX = 300                                # hairpin sizes checked on designs; longer ones by LONG_HAIRPINS
_COMP = str.maketrans("ACGU", "UGCA")


def _comp(s):
    return s[::-1].translate(_COMP)


def _gc(rng, n):
    return "".join(rng.choice(["G", "C"], size=n).tolist())


# ------------------------------------------------------------------------------------------------------------ designs
def _two_loop(rng, t, t2, left, right, hin, hl, hout=4):
    """A design in which the pair (i, j) of type t closes a two-loop with loop strands `left` (i+1..p-1) and `right`
    (q+1..j-1) around the pair (p, q) of type rtype[t2]; GC helices of `hout` pairs outside and `hin` pairs inside, an A
    hairpin loop of `hl` nt."""
    ho, hi = _gc(rng, hout), _gc(rng, hin)
    bi, bj = PAIR[t]
    bp, bq = PAIR[RTYPE[t2]]
    s = "AA" + ho + bi + left + bp + hi + "A" * hl + _comp(hi) + bq + right + bj + _comp(ho) + "AA"
    return s


def _hairpin(rng, t, loop, hout=4):
    ho = _gc(rng, hout)
    return "AA" + ho + PAIR[t][0] + loop + PAIR[t][1] + _comp(ho) + "AA"


def loop_design(n1, n2, d, seed=0):
    """A two-loop of n1 x n2 A's closed by a GC pair on diagonal d = j - i (d >= n1 + n2 + 14); seeds above 0 also
    lengthen the outer helix to 4-7 pairs."""
    rng = np.random.default_rng([1, n1, n2, d, seed])
    hl = d - (n1 + n2) - 11
    assert hl >= 3
    t, t2 = int(rng.integers(1, 3)), int(rng.integers(1, 3))
    return _two_loop(rng, t, t2, "A" * n1, "A" * n2, 4, hl, 4 + seed % 4)


def loop_keys():
    """(n1, n2, d) of the loop designs: for each s, 64 consecutive diagonals; the shape cycles through n1 = 0..s every two
    diagonals, so every shape of size s is met at both parities (2 (s + 1) <= 64)."""
    out = []
    for s in range(MAXLOOP + 1):
        for k in range(RING_DIAGONALS):
            u = (k // 2) % (s + 1)
            out.append((u, s - u, s + 14 + k))
    return out


def _shape_of(seed):
    """(outer helix pairs, inner helix pairs, inner hairpin loop) of a table design: the template at seed 0, 4-7 / 3-6 /
    4-7 at seeds above 0."""
    return (4, 3, 4) if seed == 0 else (4 + seed % 4, 3 + (seed // 4) % 4, 4 + (seed // 16) % 4)


def table_design(table, key, seed=0):
    """The design whose closing two-loop reads table[key]: (t, t2) closing pairs, loop bases as the entry's indices;
    seeds above 0 change the helix lengths, the inner hairpin and the GC helices."""
    rng = np.random.default_rng([2, len(table)] + list(key) + ([seed] if seed else []))
    b = lambda x: BASES[x - 1]                    # noqa: E731
    if table == "stack":
        t, t2 = key
        left = right = ""
    elif table == "int11":
        t, t2, x, y = key
        left, right = b(x), b(y)
    elif table == "int21":                        # (n1, t, t2, x, y, z): int21[t][t2][x][y][z] as read with that n1
        o, T, T2, x, y, z = key
        if o == 1:                                # x = i+1, y = q+1, z = j-1
            t, t2, left, right = T, T2, b(x), b(y) + b(z)
        else:                                     # int21[t2][t]: x = q+1, y = i+1, z = p-1
            t, t2, left, right = T2, T, b(y) + b(z), b(x)
    elif table == "int22":                        # a = i+1, b = p-1, c = q+1, d = j-1
        t, t2, a1, b1, c1, d1 = key
        left, right = b(a1) + b(b1), b(c1) + b(d1)
    elif table == "mismatchI":                    # a 2x3 loop whose outer mismatch is (x, y)
        t, x, y = key
        t2, left, right = 2, b(x) + "A", "AA" + b(y)
    else:
        raise KeyError(table)
    hout, hin, hl = _shape_of(seed)
    return _two_loop(rng, t, t2, left, right, hin, hl, hout)


def table_keys(table):
    ts = range(1, 7)
    xs = range(1, 5)
    if table == "stack":
        return [(t, t2) for t in ts for t2 in ts]
    if table == "int11":
        return [(t, t2, x, y) for t in ts for t2 in ts for x in xs for y in xs]
    if table == "int21":
        return [(o, t, t2, x, y, z) for o in (1, 2) for t in ts for t2 in ts for x in xs for y in xs for z in xs]
    if table == "int22":
        return [(t, t2, a, b, c, d) for t in ts for t2 in ts for a in xs for b in xs for c in xs for d in xs]
    if table == "mismatchI":
        return [(t, x, y) for t in ts for x in xs for y in xs]
    raise KeyError(table)


TABLES = ("stack", "int11", "int21", "int22", "mismatchI")


def hairpin_design(kind, key, seed=0):
    """Seeds above 0 change the outer helix (4-7 GC pairs) of the size, mismatchH and triloop designs."""
    rng = np.random.default_rng([3, len(kind)] + list(key) + ([seed] if seed else []))
    hout = _shape_of(seed)[0]
    if kind == "size":                            # (s,): an A loop of s nt closed by a GC pair
        return _hairpin(rng, int(rng.integers(1, 3)), "A" * key[0], hout)
    if kind == "mismatchH":                       # (t, x, y): loop x AAA y
        t, x, y = key
        return _hairpin(rng, t, BASES[x - 1] + "AAA" + BASES[y - 1], hout)
    if kind == "tetra":                           # (k,): the k-th tetraloop with its own closing pair
        six = TETRALOOPS[key[0]]
        ho = _gc(rng, 4)
        return "AA" + ho + six + _comp(ho) + "AA"
    if kind == "triloop":                         # (t,): AAA closed by a pair of type t (AU / GU closures pay TerminalAU)
        return _hairpin(rng, key[0], "AAA", hout)
    raise KeyError(kind)


def hairpin_keys(kind):
    if kind == "size":
        return [(s,) for s in range(3, HAIRPIN_MAX + 1)]
    if kind == "mismatchH":
        return [(t, x, y) for t in range(1, 7) for x in range(1, 5) for y in range(1, 5)]
    if kind == "tetra":
        return [(k,) for k in range(len(TETRALOOPS))]
    if kind == "triloop":
        return [(t,) for t in range(1, 7)]
    raise KeyError(kind)


HAIRPINS = ("size", "mismatchH", "tetra", "triloop")


def _perturbs(family, key):
    """The oracle perturbations (oracle.PERTURB) whose classes a design exists for."""
    if family == "loop":
        n1, n2, d = key
        return [("shape", n1, n2, d % 2), ("ring", n1 + n2, d)]
    if family in TABLES:
        return [(family,) + tuple(key)]
    kind = family[3:]
    if kind == "size":
        return [("hairpin_size", key[0])]
    if kind == "mismatchH":
        return [("mismatchH",) + tuple(key)]
    if kind == "tetra":
        return [("tetra", key[0])]
    return [("hairpin", 3)]


def seed_key(family, key):
    return "%s:%s" % (family, ",".join(map(str, key)))


def design(family, key, seed=0):
    if family == "loop":
        return loop_design(*key, seed=seed)
    if family in TABLES:
        return table_design(family, key, seed)
    return hairpin_design(family[3:], key, seed)


def design_keys():
    """[(family, key)] of the whole corpus, in a fixed order."""
    out = [("loop", k) for k in loop_keys()]
    out += [(tab, k) for tab in TABLES for k in table_keys(tab)]
    out += [("hp_" + kind, k) for kind in HAIRPINS for k in hairpin_keys(kind)]
    return out


def designs(seeds=None):
    """[(family, key, sequence)] of the whole corpus; seeds: {seed_key(family, key): seed} of the designs whose template
    (seed 0) is not decisive (the committed list by default)."""
    if seeds is None:
        seeds = json.load(open(CORPUS_FILE))["seeds"]
    return [(f, k, design(f, k, seeds.get(seed_key(f, k), 0))) for f, k in design_keys()]


def corpus_sha(ds):
    return hashlib.sha256("".join("%s %s %s\n" % (f, ",".join(map(str, k)), s) for f, k, s in ds).encode()).hexdigest()


# -------------------------------------------------------------------------------------------------------------- audit
def audit_one(item):
    """(family, key, [(perturbation, decisive, printed-decisive, smallest decisive diagonal or None, mutant's (hits,
    total))], (hits, total)) of one design, folded at a span of its own length."""
    import oracle as O
    fam, key, s = item
    n = len(s)
    base = O.fold(s, n, matrices=True)
    printed = base["hits"], base["total"]
    out = []
    for p in _perturbs(fam, key):
        mut = O.fold(s, n, matrices=True, perturb=p)
        diff = np.nonzero(base["c"] != mut["c"])
        dmin = int(diff[1].min()) if diff[1].size else None
        out.append((p, dmin is not None, (mut["hits"], mut["total"]) != printed, dmin, (mut["hits"], mut["total"])))
    return fam, key, out, printed


def audit(items, jobs=None):
    with get_context("forkserver").Pool(jobs or os.cpu_count()) as pool:
        return pool.map(audit_one, items, chunksize=64)


def class_counts(results):
    """{class family: [decisive, printed-decisive, total]} with shape / ring classes counted once per class."""
    shape, ring, counts = {}, {}, {}
    for fam, key, rows, _ in results:
        for p, dec, prn, _, _ in rows:
            if p[0] in ("shape", "ring"):
                a = (shape if p[0] == "shape" else ring).setdefault(p[1:], [False, False])
                a[0] |= dec
                a[1] |= prn
            else:
                name = "int21_n1=%d" % key[0] if fam == "int21" else fam
                c = counts.setdefault(name, [0, 0, 0])
                c[0] += dec
                c[1] += prn
                c[2] += 1
    counts["shape"] = [sum(a[0] for a in shape.values()), sum(a[1] for a in shape.values()), len(shape)]
    counts["ring"] = [sum(a[0] for a in ring.values()), sum(a[1] for a in ring.values()), len(ring)]
    return counts, shape, ring


_AUDIT = {}


@pytest.fixture(scope="module")
def audited(oracle):
    if not _AUDIT:
        ds = designs()
        _AUDIT["designs"] = ds
        _AUDIT["results"] = audit([(f, k, s) for f, k, s in ds])
    return _AUDIT


# ------------------------------------------------------------------------------------------------------------- CPU
def test_perturbation_at_delta_zero_is_the_oracle(oracle):
    """Every perturbation kind with delta = 0 gives the unmodified fold (hits, total, c, fML, f3), and delta = 1 on a
    random record changes c for the classes it surely contains."""
    rng = np.random.default_rng(11)
    s = "".join(rng.choice(list("ACGU"), size=400).tolist())
    base = oracle.fold(s, 150, matrices=True)
    kinds = [("shape", 0, 0, 1), ("shape", 3, 7, 0), ("ring", 0, 40), ("ring", 30, 77), ("hairpin_size", 5),
             ("stack", 2, 1), ("bulge", 3), ("internal_loop", 6), ("int11", 1, 2, 1, 1), ("int21", 1, 1, 2, 1, 1, 1),
             ("int21", 2, 1, 2, 1, 1, 1), ("int22", 1, 2, 3, 1, 1, 4), ("mismatchI", 1, 1, 1), ("mismatchH", 2, 1, 1),
             ("hairpin", 4), ("tetra", 7), ("hairpin_size", 40)]
    assert {k[0] for k in kinds} == set(oracle.PERTURB)
    for p in kinds:
        o = oracle.fold(s, 150, matrices=True, perturb=p, delta=0)
        assert (o["hits"], o["total"]) == (base["hits"], base["total"]), p
        for m in ("c", "m", "f3"):
            assert (o[m] == base[m]).all(), (p, m)
    for p in (("shape", 0, 0, 0), ("stack", 1, 2), ("hairpin_size", 5)):
        assert (oracle.fold(s, 150, matrices=True, perturb=p)["c"] != base["c"]).any(), p
    for bad in (("shape", 31, 0, 0), ("stack", 8, 1), ("int21", 3, 1, 1, 1, 1, 1), ("tetra", 30)):
        with pytest.raises(ValueError):
            oracle.fold(s, 150, perturb=bad)


def test_hairpin_energy_export(oracle):
    """lfold_oracle_hairpin_energy equals the c of a lone hairpin's closing pair (nothing else can pair in G A^s C) and
    extends the lxc * log extrapolation to 4094."""
    for s in (3, 4, 5, 29, 30, 31, 100, 250):
        seq = "G" + "A" * s + "C"
        assert oracle.hairpin_energy(seq, 1, s + 2) == oracle.fold(seq, s + 2, matrices=True)["c"][1, s + 1], s
    e30 = oracle.hairpin_energy("G" + "A" * 30 + "C", 1, 32)
    for s in (500, 4094):
        assert oracle.hairpin_energy("G" + "A" * s + "C", 1, s + 2) == e30 + int(107.856 * np.log(s / 30.)), s
    assert oracle.hairpin_energy("AAAAAAA", 1, 7) == INF


def test_tetraloop_list_matches_the_tables():
    from conftest import ROOT
    src = open(os.path.join(ROOT, "mir_prefer_b200", "csrc", "turner99_v185_tables.inc")).read()
    line = next(ln for ln in src.splitlines() if "T99_Tetraloops[]" in ln)
    assert line.split('"')[1].split() == TETRALOOPS
    assert len(set(TETRALOOPS)) == len(TETRALOOPS)   # no duplicates: "first listed wins" never decides here


def test_corpus_is_pinned():
    ds = designs()
    pin = json.load(open(CORPUS_FILE))
    assert corpus_sha(ds) == pin["sha256"] and len(ds) == pin["designs"]
    assert max(len(s) for f, _, s in ds if not f.startswith("hp_")) < 150


def test_every_class_is_decisive(audited):
    """Each class raised by 1 dcal changes c on its design.  Every shape x parity and ring class is decisive (and every
    shape is printed-decisive at least once); the table counts (decisive / printed / total) are pinned exactly."""
    counts, shape, ring = class_counts(audited["results"])
    pin = json.load(open(CORPUS_FILE))["counts"]
    for name in sorted(counts):
        print("%-16s decisive %5d  printed %5d  of %5d" % (name, *counts[name]))
    assert len(shape) == 992 and len(ring) == (MAXLOOP + 1) * RING_DIAGONALS
    missing = sorted(k for k, a in shape.items() if not a[0]) + sorted(k for k, a in ring.items() if not a[0])
    assert not missing, missing
    unprinted = sorted({k[:2] for k, a in shape.items() if a[1]} ^ {k[:2] for k in shape})
    assert not unprinted, unprinted
    assert counts == {k: list(v) for k, v in pin.items()}


def test_decisive_cells_lie_inside_each_design(audited):
    """Each decisive class changes c on a diagonal below 150 (the span of the 16-bit loci) except long hairpins."""
    for fam, key, rows, _ in audited["results"]:
        for p, dec, _, dmin, _ in rows:
            if dec and fam != "hp_size":
                assert dmin < 150, (fam, key, p, dmin)


# --------------------------------------------------------------------------------------------------------- GPU loci
# Sequences put at the 5' end of every locus of a config: a perfect GC helix below -320 kcal/mol, whose fill unit the
# 16-bit kernel flags and k_fill_smem redoes (the redone unit then holds designs too).
PREFIX = {None: "", "helix300": "GC" * 160, "helix500": "GC" * 170}

# (name, span, flags, locus length range, expected plan kernel, tiled, prefix)
CONFIGS = [
    ("s16_160", 150, 0, (100, 160), 160, False, None),
    ("s16_352", 150, 0, (161, 352), 352, False, None),
    ("s16_608", 150, 0, (353, 608), 608, False, None),
    ("s16_tile608", 150, 0, (2000, 5000), 608, True, None),
    ("s16_864", 300, 0, (609, 864), 864, False, None),
    ("s16_tile864", 300, 0, (2000, 5000), 864, True, None),
    ("dynw_608", 400, 0, (353, 608), 608, False, None),
    ("dynw_864", 400, 0, (609, 864), 864, False, None),
    ("dynw_tile864", 500, 0, (2000, 5000), 864, True, None),
    ("smem_160", 150, FLAG_WIDE, (100, 160), 160, False, None),
    ("smem_352", 150, FLAG_WIDE, (161, 352), 352, False, None),
    ("smem_tile608", 150, FLAG_WIDE, (2000, 5000), 608, True, None),
    ("smem_608", 300, FLAG_WIDE, (353, 608), 608, False, None),
    ("smem_tile864", 500, FLAG_WIDE, (2000, 5000), 864, True, None),
    ("smem_864_L1001", 1001, 0, (609, 864), 864, False, None),
    ("redo_tile864_L300", 300, 0, (2000, 5000), 864, True, "helix300"),
    ("redo_864_L500", 500, 0, (609, 864), 864, False, "helix500"),
    ("generic_L801", 801, 0, (1000, 1200), 0, False, None),
    ("generic_L2000", 2000, 0, (1000, 1200), 0, False, None),
]


def loci(ds, lo, hi, prefix=""):
    """The designs joined in corpus order after `prefix` into loci of lo..hi nt (the last padded with A's):
    [(locus, [(offset, index)])].  Designs longer than hi - len(prefix) are left out."""
    out, cur, parts = [], prefix, []
    for k, (_, _, s) in enumerate(ds):
        if len(prefix) + len(s) > hi:
            continue
        if len(cur) + len(s) > hi:
            out.append((cur + "A" * max(0, lo - len(cur)), parts))
            cur, parts = prefix, []
        parts.append((len(cur), k))
        cur += s
    if parts:
        out.append((cur + "A" * max(0, lo - len(cur)), parts))
    return out


def _config_loci(ds, cfg):
    return loci(ds, *cfg[3], PREFIX[cfg[6]])


def _design_c(s):
    import oracle as O
    return O.fold(s, len(s), matrices=True)["c"]


_DESIGN_C = {}


@pytest.fixture(scope="module")
def ref(oracle, audited):
    """(designs, {index: c of the design's own fold}, name -> oracle fold of the config's first locus); the locus folds
    run in a thread pool while the tests go on."""
    oracle.fold("GGGGAAACCCC", 5)
    ds = designs()
    if not _DESIGN_C:
        with get_context("forkserver").Pool(os.cpu_count()) as pool:
            _DESIGN_C.update(enumerate(pool.map(_design_c, [s for _, _, s in ds], chunksize=64)))
    ex = ThreadPoolExecutor(max_workers=max(2, os.cpu_count() or 2))
    whole = {cfg[0]: ex.submit(oracle.fold, _config_loci(ds, cfg)[0][0], cfg[1], True) for cfg in CONFIGS}
    yield ds, _DESIGN_C, lambda name: whole[name].result()
    ex.shutdown(wait=True, cancel_futures=True)


def _assert_blocks(c, L, n, parts, ds, dc):
    """Each design's c block of the locus equals the design's own fold, shifted, on every diagonal below min(L, n)."""
    dl = min(L, n)
    for off, k in parts:
        m = len(ds[k][2])
        want = dc[k]
        w = min(m, dl)
        got = c[off + 1:off + m + 1, :w]
        exp = want[1:m + 1, :w]
        ii, dd = np.meshgrid(np.arange(1, m + 1), np.arange(w), indexing="ij")
        inside = ii + dd <= m
        bad = np.nonzero((got != exp) & inside)
        assert bad[0].size == 0, (ds[k][0], ds[k][1], [(int(i) + 1, int(d)) for i, d in zip(*bad)][:5])


def test_loci_hold_the_design_blocks(ref):
    """The locality the GPU tests rely on, on the oracle: in the first locus of every config, each design's c block equals
    the design's own fold, shifted, on every diagonal below the span.  (The GPU test compares every block of every locus
    with the design's fold, so a locus where this failed would fail there.)  The loci reach the paths they are named for:
    c below -320 kcal/mol in the helix-prefixed loci (the unit is flagged and redone), and in the first DYNW loci fML below
    MF16M_GUARD (-136 kcal/mol) with every c inside the 16-bit range (the DML strips switch to int32, nothing is redone)."""
    ds, dc, whole = ref
    for cfg in CONFIGS:
        s, parts = _config_loci(ds, cfg)[0]
        o = whole(cfg[0])
        _assert_blocks(o["c"], cfg[1], len(s), parts, ds, dc)
        if cfg[6] in ("helix300", "helix500"):
            assert o["c"].min() < -32000, cfg[0]
        if cfg[0] in ("dynw_608", "dynw_864"):
            assert o["m"].min() < -13600 and o["c"].min() > -32000, (cfg[0], o["m"].min(), o["c"].min())


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", CONFIGS, ids=[c[0] for c in CONFIGS])
def test_kernel_cells_equal_design_folds(mf, ref, cfg):
    """Every design joined into loci that select one fill kernel: c cell for cell in every design block against the
    design's oracle fold, and the first locus whole (c, fML, f3, hits, total) against the oracle."""
    from mir_prefer_b200.fold import plan_fill_units
    name, L, flags, (lo, hi), kernel, tiled, prefix = cfg
    ds, dc, whole = ref
    ls = _config_loci(ds, cfg)
    placed = sum(len(p) for _, p in ls)
    assert placed == len([1 for _, _, s in ds if len(s) + len(PREFIX[prefix]) <= hi])
    for r, (s, parts) in enumerate(ls):
        plan = plan_fill_units(len(s), L)
        assert plan["kernel"] == kernel and (plan["n_units"] > 1) == tiled, (name, len(s), plan)
        c, m, f3 = mf.debug_matrices(s, L, flags=flags)
        _assert_blocks(c, L, len(s), parts, ds, dc)
        if r == 0:
            o = whole(name)
            n = len(s)
            assert (o["c"] == c).all(), name
            assert (np.minimum(o["m"], INF) == np.minimum(m, INF)).all(), name
            assert (o["f3"][:n + 3] == f3[:n + 3]).all(), name
            with mf.fold([s], L, flags) as res:
                assert (res.hits(0), res.total(0)) == (o["hits"], o["total"]), name
    print("%s: %d designs in %d loci" % (name, placed, len(ls)))


@pytest.mark.gpu
@pytest.mark.parametrize("flags", [0, FLAG_WIDE], ids=["fill16", "wide"])
def test_printed_decisive_classes_reach_the_traceback(mf, audited, flags):
    """Every design folded on its own at L = 150 prints the oracle's hits, and differs from the +1 mutant of each of its
    printed-decisive classes: tb_loop_energy resolved the class, not just the fill."""
    ds, res = audited["designs"], audited["results"]
    idx = [k for k, (_, _, s) in enumerate(ds) if len(s) <= 150]
    with mf.fold([ds[k][2] for k in idx], 150, flags) as out:
        got = {k: (out.hits(r), out.total(r)) for r, k in enumerate(idx)}
    checked = 0
    for k in idx:
        _, _, rows, printed = res[k]
        assert got[k] == printed, ds[k][:2]
        for p, _, prn, _, mut in rows:
            if prn:
                assert got[k] != mut, (ds[k][:2], p)
                checked += 1
    assert checked > 10000


LONG_HAIRPINS = sorted(set(range(HAIRPIN_MAX + 1, 4081, 97)) | {600, 601, 864, 865, 999, 1000, 1001, 2048, 3000, 4080})


@pytest.mark.gpu
def test_long_hairpins_at_span_4096(mf, oracle):
    """G^8 A^s C^8 at L = 4096 for hairpin sizes past the designs: one printed hairpin whose energy is 7 G-C stacks plus
    the oracle's hairpin energy of size s (the stacks measured on the oracle's fold of s = 40)."""
    def rec(s):
        return "G" * 8 + "A" * s + "C" * 8
    o = oracle.fold(rec(40), 4096)
    stacks = o["total"] - oracle.hairpin_energy(rec(40), 8, 49)
    seqs = [rec(s) for s in LONG_HAIRPINS]
    with mf.fold(seqs, 4096) as res:
        for r, s in enumerate(LONG_HAIRPINS):
            want = stacks + oracle.hairpin_energy(seqs[r], 8, s + 9)
            hits = res.hits(r)
            assert len(hits) == 1 and hits[0][1] == want == res.total(r), (s, hits, want)
