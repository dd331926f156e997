"""Search seeds for the designs of tests/test_loop_terms.py and write tests/golden/loop_corpus.json.

    python tools/loop_corpus.py [--seeds N] [--jobs J]

Every design is first built from its template (seed 0) and audited with the oracle's perturbations.  A design whose class
is not decisive gets the first seed in 1..N on which it is (loop designs: both their shape and ring class); seeds change
the helix lengths, the inner hairpin and the GC helices around the same loop.  A shape x parity class that no design
prints differently under its +1 mutant gets, on one of its designs, the first seed on which it does and both classes stay
decisive.  The file holds those seeds, the sha256 of the expanded corpus and the per-class counts (decisive,
printed-decisive, total) that the tests pin.  Results are deterministic: the generators are seeded and the oracle is exact."""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

import oracle as O  # noqa: E402
import test_loop_terms as T  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seeds", type=int, default=64)
    ap.add_argument("--jobs", type=int, default=os.cpu_count())
    ap.add_argument("--out", default=T.CORPUS_FILE)
    a = ap.parse_args()
    O.build()
    seeds = {}
    base = {(f, k): rows for f, k, rows, _ in T.audit([(f, k, T.design(f, k)) for f, k in T.design_keys()], a.jobs)}

    def search(keys, ok):
        """{(family, key): (first seed in 1..N whose audit rows satisfy ok, rows)}, all candidates of one seed audited in
        one batch; and the keys no seed satisfies."""
        found, left = {}, list(keys)
        for seed in range(1, a.seeds + 1):
            if not left:
                break
            for f, k, rows, _ in T.audit([(f, k, T.design(f, k, seed)) for f, k in left], a.jobs):
                if ok(rows):
                    found[f, k] = (seed, rows)
            left = [fk for fk in left if fk not in found]
        return found, left

    weak = [fk for fk, rows in base.items() if not all(r[1] for r in rows)]
    found, left = search(weak, lambda rows: all(r[1] for r in rows))
    for fk, (seed, rows) in found.items():
        seeds[T.seed_key(*fk)], base[fk] = seed, rows
    print("%d designs decisive at seed 0, %d more with a seed, %d with none" % (len(base) - len(weak), len(found), len(left)))

    printed = {}
    for (f, k), rows in base.items():
        if f == "loop":
            printed[rows[0][0][1:]] = printed.get(rows[0][0][1:], False) or rows[0][2]
    unprinted = {c for c, p in printed.items() if not p}
    cand = [(f, k) for f, k in base if f == "loop" and (k[0], k[1], k[2] % 2) in unprinted and T.seed_key(f, k) not in seeds]
    found, _ = search(cand, lambda rows: all(r[1] for r in rows) and rows[0][2])
    for f, k in sorted(found):
        c = (k[0], k[1], k[2] % 2)
        if c in unprinted:
            seeds[T.seed_key(f, k)] = found[f, k][0]
            unprinted.discard(c)
    if unprinted:
        print("no seed prints these shape classes: %s" % sorted(unprinted))

    ds = T.designs(seeds)
    counts, _, _ = T.class_counts(T.audit(ds, a.jobs))
    for name in sorted(counts):
        print("%-16s decisive %5d  printed %5d  of %5d" % (name, *counts[name]))
    with open(a.out, "w") as fh:
        json.dump({"generator": "tests/test_loop_terms.py", "search": "tools/loop_corpus.py --seeds %d" % a.seeds,
                   "designs": len(ds), "sha256": T.corpus_sha(ds), "counts": counts,
                   "seeds": dict(sorted(seeds.items()))}, fh)
        fh.write("\n")


if __name__ == "__main__":
    main()
