"""The traceback's tie-breaking, rule by rule.  RNALfold prints the first of several equal-energy structures that each scan
of its backtrack() meets; k_traceback (trace.cu) restates every such scan as lane-parallel ballots, skips runs 32 positions
at a time and speculates along helices.  Random loci rarely contain the ties that each rule has to break, so a traceback
that broke one the other way could still match the oracle on them.

The oracle's tie-break mutants (oracle.TIEBREAK: one bit flips one first-match rule) show which ties a corpus contains.
The corpus here is built from seeded design families, and tests/golden/tie_corpus.json (written by tools/tie_corpus.py)
lists the (family, seed, span) records on which the flipped rules change the printed output:
  twins  3- and 4-way junctions with a branch that can form at either of two places with equal energy, at the end of a
         multiloop segment or between two strong branches (fML peel order, split k, pair order; multiloop split k)
  micro  microsatellites with point interruptions (two-loop scan, exterior scan)
  slip   a C-run / G-run hairpin that can slip by one base, at the 5' end of a short locus (the traceback from base 1
         meets (1,k) and (2,k) with the 5' dangle of base 1 at the same energy and k: exterior scan order) or as a
         multiloop branch (pair (i,j) against (i+1,j) with the 5' dangle of i: fML pair priority)
  long   multibranch designs with A/C linkers and exterior spacers of 0-5, 30-34 and 62-66 nt (the 32-wide run steps,
         the j == n push of the exterior scan)
  helix  helix runs of 30-33 and 62-65 stacked pairs with a small loop at pair 30-33 / 62-64, interior loops of
         u+v = 29 / 30 nt, a 30-nt bulge, large loops just above a hairpin (K = d-6 < 30)

CPU: every mutant bit changes at least 3 records; the oracle's structures contain the shapes the families promise.
GPU: every record, the records as RNALfold text, and the records joined into 5-20 kb loci (tile edges, the generic kernel,
a segmented fold) equal the unmodified oracle; a few records cell for cell."""
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN
from mir_prefer_b200.fold import FLAG_WIDE

CORPUS_FILE = os.path.join(GOLDEN, "tie_corpus.json")
MIN_CAUGHT = 3
_COMP = str.maketrans("ACGU", "UGCA")


def _comp(s):
    return s[::-1].translate(_COMP)


def _rand(rng, n, alphabet="ACGU"):
    return "".join(rng.choice(list(alphabet), size=int(n)).tolist())


def _stem(rng, n):
    """A helix arm of mixed composition (about half G/C): its complement pairs it, and c stays far above -320 kcal/mol."""
    return _rand(rng, n)


def _hairpin(rng, stem, loop=None):
    a = _stem(rng, stem)
    return a + _rand(rng, loop if loop is not None else int(rng.integers(4, 7))) + _comp(a)


def _ac(rng, n):
    """Unpaired linker or spacer: A and C never pair with each other."""
    return _rand(rng, n, "AC")


# --------------------------------------------------------------------------------------------------------- families
def _twin(rng):
    """Two equal-energy hairpins of which only one can form: a AAA ~a AAA a folds as a AAA ~a or as ~a AAA a -- the same
    duplex turned around, closed by C-G into a triloop (no mismatch term) and opened by G-C next to an A either way."""
    a = "G" + _rand(rng, rng.integers(1, 4)) + "C"
    x = "A" if rng.random() < 0.7 else ""
    return x + a + "AAA" + _comp(a) + "AAA" + a + x


# where the twin sits among the strong branches Y: at either end of the junction, between two strong branches of one
# multiloop segment, or twice
TWIN_LAYOUTS = ("TY", "YT", "YTY", "YYTY", "YYT", "TYT")


def twins(seed):
    """A 3- or 4-way junction with a twin branch (one hairpin that can form at either of two places with the same energy)
    at the end of a multiloop segment or between two strong hairpins, with A/C linkers of 0-5 nt around every branch."""
    rng = np.random.default_rng(1_000_000 + seed)
    layout = TWIN_LAYOUTS[seed % len(TWIN_LAYOUTS)]
    branches = [_twin(rng) if ch == "T" else _hairpin(rng, int(rng.integers(4, 9))) for ch in layout]
    inner = "".join(_ac(rng, rng.integers(0, 6)) + b for b in branches) + _ac(rng, rng.integers(0, 6))
    outer = _stem(rng, int(rng.integers(5, 9)))
    return _rand(rng, rng.integers(3, 20)) + outer + inner + _comp(outer) + _rand(rng, rng.integers(3, 20))


MICRO_REPEATS = ("CUG", "CAG", "CCG", "AU", "GGAUCC")


def micro(seed):
    """(CUG)n, (CAG)n, (CCG)n, (AU)n or (GGAUCC)n of 90-300 nt with 0-3 point interruptions."""
    rng = np.random.default_rng(2_000_000 + seed)
    rep = MICRO_REPEATS[seed % len(MICRO_REPEATS)]
    n = int(rng.integers(90, 301))
    s = list((rep * (n // len(rep) + 1))[:n])
    for _ in range(int(rng.integers(0, 4))):
        s[int(rng.integers(0, n))] = "ACGU"[int(rng.integers(4))]
    return "".join(s)


def _slipped(rng):
    """C^(m+1..m+2) L G^m, m = 3-5, L a 3-6 nt loop: the G-run pairs with the first or the second C at the same cost
    where one more loop base is worth the second C's 5' dangle on the first C."""
    m = int(rng.integers(3, 6))
    return "C" * (m + int(rng.integers(1, 3))) + _rand(rng, rng.integers(3, 7)) + "G" * m


def slip(seed):
    """Even seeds: a slipped C-run / G-run hairpin at the 5' end of a 25-85 nt locus, where base 1 has no 5' neighbour
    that could dangle on (1,k) instead (the exterior scan's (i,k) / (i+1,k) order).  Odd seeds: the slipped hairpin as a
    branch of a 3-way junction between strong hairpins, with A/C linkers of 0-5 nt (the fML segment's pair priority)."""
    rng = np.random.default_rng(5_000_000 + seed)
    if seed % 2 == 0:
        return _slipped(rng) + _rand(rng, rng.integers(5, 60))
    branches = [_hairpin(rng, int(rng.integers(4, 8))), _slipped(rng), _hairpin(rng, int(rng.integers(4, 8)))]
    inner = "".join(_ac(rng, rng.integers(0, 6)) + b for b in branches) + _ac(rng, rng.integers(0, 6))
    outer = _stem(rng, int(rng.integers(5, 9)))
    return _rand(rng, rng.integers(3, 15)) + outer + inner + _comp(outer) + _rand(rng, rng.integers(3, 15))


LINKER_CLASSES = ((0, 5), (30, 34), (62, 66))


def _linker_len(rng, cls):
    lo, hi = LINKER_CLASSES[cls]
    return int(rng.integers(lo, hi + 1))


def long_linkers(seed):
    """A multibranch design (2-4 branches) whose A/C linkers are 0-5 nt except one or two of 30-34 or 62-66 nt, with A/C
    exterior spacers of the same classes on both sides; every third design's 3' spacer runs to the last base."""
    rng = np.random.default_rng(3_000_000 + seed)
    nb = int(rng.integers(2, 5))
    big = 1 + seed % 2
    cls = [0] * (nb + 1)
    for k in rng.choice(nb + 1, size=big, replace=False).tolist():
        cls[k] = 1 + (seed // 2) % 2
    parts = [_ac(rng, _linker_len(rng, c)) for c in cls]
    branches = [_hairpin(rng, int(rng.integers(5, 9))) for _ in range(nb)]
    inner = "".join(parts[k] + branches[k] for k in range(nb)) + parts[nb]
    outer = _stem(rng, int(rng.integers(6, 10)))
    design = outer + inner + _comp(outer)
    sp5 = _ac(rng, _linker_len(rng, int(rng.integers(0, 3))))
    sp3 = _ac(rng, _linker_len(rng, int(rng.integers(1, 3))))
    tail = "" if seed % 3 == 0 else _rand(rng, rng.integers(5, 30))
    return _rand(rng, rng.integers(5, 30)) + sp5 + design + sp3 + tail


def helix(seed):
    """A helix run of 30-33 or 62-65 stacked pairs of mixed composition, one defect in it (a 1-nt bulge, or a 1x1, 1x2 or
    2x2 loop at pair 30-33 / 62-64; an interior loop of u+v = 29 or 30; a 30-nt bulge; or a 12-20 nt loop around a 3-pair
    hairpin, so that the scan window K = d-6 is below 30)."""
    rng = np.random.default_rng(4_000_000 + seed)
    kind = seed % 4
    run = int(rng.integers(30, 34)) if seed % 8 < 4 else int(rng.integers(62, 66))
    a, loop = _stem(rng, run + 8), _rand(rng, rng.integers(4, 9))
    if kind == 0:      # small loop at pair 30-33 / 62-64
        at = int(rng.integers(30, 34)) if run < 62 else int(rng.integers(62, 65))
        u, v = ((1, 0), (0, 1), (1, 1), (1, 2), (2, 1), (2, 2))[int(rng.integers(0, 6))]
    elif kind == 1:    # u + v = 29 or 30
        at = run
        u = int(rng.integers(1, 29))
        v = int(rng.integers(29, 31)) - u
    elif kind == 2:    # 30-nt bulge
        at = run
        u, v = (30, 0) if rng.random() < 0.5 else (0, 30)
    else:              # loop near the window edge: a 3-pair inner hairpin inside a 12-20 nt loop (d < 36)
        at = run
        u = int(rng.integers(6, 11))
        v = int(rng.integers(6, 11))
    s5, s3 = a[:at], a[at:] if kind != 3 else a[at:at + 3]
    inner = s3 + loop + _comp(s3)
    core = s5 + _ac(rng, u) + inner + _ac(rng, v) + _comp(s5)
    return _rand(rng, rng.integers(3, 25)) + core + _rand(rng, rng.integers(3, 25))


FAMILIES = {"twins": twins, "micro": micro, "slip": slip, "long": long_linkers, "helix": helix}
SPANS = {"twins": (150, 300), "micro": (150, 300), "slip": (25, 40, 150), "long": (300,), "helix": (300,)}


def corpus():
    """[(family, seed, span, sequence)] of the committed list."""
    entries = json.load(open(CORPUS_FILE))["records"]
    return [(e["family"], e["seed"], e["span"], FAMILIES[e["family"]](e["seed"])) for e in entries]


def outcome(oracle, seq, span, tiebreak=0):
    """(hits, total), or None where the (mutant) traceback fails -- which counts as a difference."""
    try:
        o = oracle.fold(seq, span, tiebreak=tiebreak)
    except RuntimeError:
        return None
    return o["hits"], o["total"]


_RUNS = {}


@pytest.fixture(scope="module")
def runs(oracle):
    """{tiebreak mask: [outcome per corpus record]} for 0 and every single bit (computed once per session)."""
    if not _RUNS:
        recs = corpus()
        for mask in [0] + sorted(oracle.TIEBREAK.values()):
            _RUNS[mask] = [outcome(oracle, s, L, mask) for _, _, L, s in recs]
    return _RUNS


# ------------------------------------------------------------------------------------------------ structure shapes
def pair_table(ss):
    pt, st = [-1] * len(ss), []
    for k, ch in enumerate(ss):
        if ch == "(":
            st.append(k)
        elif ch == ")":
            i = st.pop()
            pt[i], pt[k] = k, i
    return pt


def _gaps(pt, i, j):
    """Unpaired runs between the branches of the loop spanning i..j-1 (runs before the first and after the last included)."""
    gaps, gap, k = [], 0, i
    while k < j:
        if pt[k] > k:
            gaps.append(gap)
            gap, k = 0, pt[k] + 1
        else:
            gap, k = gap + 1, k + 1
    return gaps + [gap]


def shapes(ss):
    """(helix runs: (stacked pairs, (u, v) of the loop below or None), multiloop linkers, exterior spacers) of a structure.
    A multiloop's linkers are listed 5' to 3', each list ending with None: the traceback splits a multiloop at the first
    k, so every linker but the last is peeled from the 5' side of a segment, the last one from the 3' side."""
    pt = pair_table(ss)
    helices, ml = [], []
    for i, j in enumerate(pt):
        if j <= i or (i > 0 and pt[i - 1] == j + 1):
            continue
        run = 1
        while pt[i + run] == j - run:
            run += 1
        p, q = i + run - 1, j - run + 1
        g = _gaps(pt, p + 1, q)
        if len(g) == 2:       # one pair inside: the run ends in an interior loop or bulge
            a = p + 1 + g[0]
            helices.append((run, (g[0], q - 1 - pt[a])))
        else:
            helices.append((run, None))
            if len(g) > 2:
                ml.extend(g + [None])
    return helices, ml, _gaps(pt, 0, len(ss))[1:-1]


# ------------------------------------------------------------------------------------------------------------- CPU

def test_corpus_file_lists_every_family():
    recs = corpus()
    assert {f for f, _, _, _ in recs} == set(FAMILIES) and all(L in SPANS[f] for f, _, L, _ in recs)
    assert len({(f, s, L) for f, s, L, _ in recs}) == len(recs)


def test_every_tiebreak_rule_changes_corpus_records(oracle, runs):
    """Flip one first-match rule of the oracle's traceback at a time: each flip changes the printed output (or fails the
    backtrack) on at least MIN_CAUGHT records, so a GPU traceback that broke that tie the other way would be caught."""
    recs = corpus()
    assert all(b is not None for b in runs[0])
    caught = {}
    for name, bit in oracle.TIEBREAK.items():
        diff = [r for r, (a, b) in enumerate(zip(runs[0], runs[bit])) if a != b]
        caught[name] = len(diff)
        print("%-15s changes %3d of %d records (%s)" % (name, len(diff), len(recs), ", ".join(sorted({recs[r][0] for r in diff}))))
    assert all(v >= MIN_CAUGHT for v in caught.values()), caught


def _linker_sides(ml):
    """Multiloop linkers of shapes() -> (peeled from the 5' side, peeled from the 3' side)."""
    five, three = [], []
    for g, nxt in zip(ml, ml[1:] + [None]):
        if g is not None:
            (three if nxt is None else five).append(g)
    return five, three


def test_oracle_structures_have_the_promised_shapes(runs):
    """The shapes the long-linker and helix families exist for are in the oracle's printed structures, so that an edit to
    a generator cannot silently lose them.  A run step of 32 (trace.cu: eq == FULL, go == FULL) needs 32 equal cells after
    the at most one base a dangle takes on either side, hence 34+ below: multiloop linkers of 30-34 and 62-66 unpaired
    bases, a 34+ linker peeled from the 5' side of its segment and one peeled from the 3' side, exterior spacers of 34+
    between printed branches, a 3' spacer of 34+ running to the last base of a locus whose last window was traced (the
    j == n push), helix runs of 32+ and 62+ stacked pairs, a small loop right after 30-33 and after 62-64 stacked pairs,
    an interior loop of u+v = 29 or 30, a 30-nt bulge, and a 12+ nt loop closed by a pair of span d < 36 (K = d-6 < 30)."""
    five, three, ext, to_end, runs_, small, big, edge = [], [], [], 0, [], set(), set(), 0
    for (fam, _, L, s), res in zip(corpus(), runs[0]):
        n = len(s)
        for ss, _, start in res[0]:
            hel, ml, ex = shapes(ss)
            if fam == "long":
                f5, f3 = _linker_sides(ml)
                five += f5
                three += f3
                ext += ex
                end = start + len(ss) - 1
                to_end += start + L >= n and n - end >= 34 and set(s[end:]) <= set("AC")
            if fam == "helix":
                for run, loop in hel:
                    runs_.append(run)
                    if loop is None:
                        continue
                    u, v = loop
                    if 0 < u + v <= 4 and (30 <= run <= 33 or 62 <= run <= 64):
                        small.add(run >= 62)
                    if u + v in (29, 30):
                        big.add((min(u, v) == 0, u + v))
                pt = pair_table(ss)
                for i, j in enumerate(pt):
                    if i < j and j - i < 36:
                        g = _gaps(pt, i + 1, j)
                        edge += len(g) == 2 and sum(g) >= 12
    link = five + three
    assert any(30 <= g <= 34 for g in link) and any(62 <= g <= 66 for g in link), sorted(link)[-8:]
    assert max(five) >= 34 and max(three) >= 34, (sorted(five)[-4:], sorted(three)[-4:])
    assert max(ext) >= 34, sorted(ext)[-8:]
    assert to_end >= 1
    assert max(runs_) >= 62 and any(32 <= r < 62 for r in runs_), sorted(runs_)[-8:]
    assert small == {False, True}, small
    assert (True, 30) in big and any(not bulge for bulge, _ in big), big
    assert edge >= 1


# ------------------------------------------------------------------------------------------------------------- GPU


def _fold_all(mf, recs, flags=0):
    """[(hits, total)] of every record, one batch per span."""
    out = [None] * len(recs)
    for L in sorted({r[2] for r in recs}):
        idx = [k for k, r in enumerate(recs) if r[2] == L]
        with mf.fold([recs[k][3] for k in idx], L, flags) as res:
            for r, k in enumerate(idx):
                out[k] = (res.hits(r), res.total(r))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("flags", [0, FLAG_WIDE], ids=["fill16", "wide"])
def test_corpus_equals_oracle(mf, oracle, runs, flags):
    """Every record at its span equals the unmodified oracle -- with the 16-bit fill's traceback hint and with the wide
    kernels, which set every hint byte so that the two-loop scan always runs -- and differs from every mutant where the
    mutant differs from the oracle: a traceback that broke any of these ties the other way would fail here."""
    recs = corpus()
    got = _fold_all(mf, recs, flags)
    bad = [(recs[k][:3]) for k in range(len(recs)) if got[k] != runs[0][k]]
    assert not bad, bad
    for name, bit in oracle.TIEBREAK.items():
        assert sum(g != m for g, m in zip(got, runs[bit])) >= MIN_CAUGHT, name


@pytest.mark.gpu
def test_corpus_text_equals_oracle_cli(mf, oracle):
    recs = corpus()
    for L in sorted({r[2] for r in recs}):
        text = "".join(">%s_%d\n%s\n" % (f, s, q) for f, s, span, q in recs if span == L)
        assert mf.fold_text(text, L) == oracle.fold_text(text, L), L


def joined(n_min, seed):
    """Corpus records joined by A/C spacers of 0-40 nt into one locus of at least n_min nt (designs straddle tile edges)."""
    rng = np.random.default_rng(seed)
    recs = corpus()
    parts, n = [], 0
    while n < n_min:
        s = recs[int(rng.integers(len(recs)))][3] + _ac(rng, rng.integers(0, 41))
        parts.append(s)
        n += len(s)
    return "".join(parts)


JOINED = [(150, 20_000), (500, 10_000), (1000, 5_000)]
_JOINED_ORACLE = {}


def _joined_oracle(oracle, L, n):
    """(locus, (hits, total) of the oracle), folded once per session."""
    if (L, n) not in _JOINED_ORACLE:
        s = joined(n, L)
        o = oracle.fold(s, L)
        _JOINED_ORACLE[L, n] = s, (o["hits"], o["total"])
    return _JOINED_ORACLE[L, n]


@pytest.mark.gpu
@pytest.mark.parametrize("L,n", JOINED, ids=["L%d" % L for L, _ in JOINED])
def test_joined_loci_equal_oracle(mf, oracle, L, n):
    """The records joined into long loci: 608-nt tiles at L=150, 864-nt tiles at L=500, the generic kernel at L=1000."""
    from mir_prefer_b200.fold import plan_fill_units
    s, want = _joined_oracle(oracle, L, n)
    assert L == 1000 or plan_fill_units(len(s), L)["n_units"] > 5
    for flags in (0, FLAG_WIDE):
        with mf.fold([s], L, flags) as res:
            assert (res.hits(0), res.total(0)) == want, flags


@pytest.mark.gpu
def test_joined_locus_segmented_equals_oracle(oracle):
    """The L=150 joined locus folded in segments of one owned tile (a 1 MiB budget).  Every segment but the 3'-most one
    refills its halo tile, so the fill units counted show that the fold really ran in those segments."""
    from mir_prefer_b200.fold import plan_fill_units
    from test_segmented_loci import _seg_plan, budget_ctx
    L, n = JOINED[0]
    s, want = _joined_oracle(oracle, L, n)
    plan = _seg_plan(len(s), L, 1)
    assert len(plan) > 5 and (plan["tile_first"] == plan["tile_last"]).all()
    with budget_ctx(1) as ctx, ctx.fold([s], L) as res:
        assert (res.hits(0), res.total(0)) == want
        assert res.stats["fill_units"] == plan_fill_units(len(s), L)["n_units"] + int(plan["halo_tiles"].sum())


@pytest.mark.gpu
def test_records_cell_for_cell(mf, oracle):
    """c / fML / f3 of the first record of every family against the oracle's matrices, with both fill kernels."""
    seen = set()
    for fam, _, L, s in corpus():
        if fam in seen:
            continue
        seen.add(fam)
        o = oracle.fold(s, L, matrices=True)
        for flags in (0, FLAG_WIDE):
            c, m, f3 = mf.debug_matrices(s, L, flags=flags)
            assert (o["c"] == c).all(), (fam, flags)
            assert (np.minimum(o["m"], 1000000) == np.minimum(m, 1000000)).all(), (fam, flags)
            assert (o["f3"][:len(s) + 3] == f3[:len(s) + 3]).all(), (fam, flags)
