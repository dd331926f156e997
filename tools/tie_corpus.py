"""Search the seeded design families of tests/test_traceback_ties.py for records on which the oracle's tie-break mutants
(oracle.TIEBREAK) change the printed output, and write the (family, seed, span) list the tests fold to
tests/golden/tie_corpus.json.

    python tools/tie_corpus.py [--seeds N] [--target K] [--jobs J]

Every (family, seed, span) with seed < N is folded by the unmodified oracle and by each single-bit mutant.  Records are
then picked greedily, the one that catches most still-uncaught rules first, until every rule is caught by `target`
records; to these every family adds its first `--per-family` seeds (at each span) so that the shapes the families promise
stay in the corpus.  Results are deterministic: the generators are seeded and the oracle is exact."""
import argparse
import json
import os
import sys
from multiprocessing import Pool

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

import oracle as O  # noqa: E402
import test_traceback_ties as T  # noqa: E402


def caught_by(job):
    fam, seed, span = job
    s = T.FAMILIES[fam](seed)
    base = T.outcome(O, s, span)
    if base is None:
        raise RuntimeError("the unmodified oracle fails on %s" % (job,))
    return job, len(s), sorted(name for name, bit in O.TIEBREAK.items() if T.outcome(O, s, span, bit) != base)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seeds", type=int, default=48)
    ap.add_argument("--target", type=int, default=4)
    ap.add_argument("--per-family", type=int, default=8)
    ap.add_argument("--jobs", type=int, default=os.cpu_count())
    ap.add_argument("--out", default=T.CORPUS_FILE)
    a = ap.parse_args()
    O.build()
    jobs = [(f, s, L) for f in T.FAMILIES for s in range(a.seeds) for L in T.SPANS[f]]
    with Pool(a.jobs) as pool:
        found = pool.map(caught_by, jobs)
    rules = {job: set(c) for job, _, c in found}
    length = {job: n for job, n, _ in found}
    pick = [job for job in jobs if job[1] < a.per_family]
    count = {name: sum(name in rules[j] for j in pick) for name in O.TIEBREAK}
    unreached = sorted(name for name in O.TIEBREAK if not any(name in r for r in rules.values()))
    while True:
        short = {name for name, c in count.items() if c < a.target} - set(unreached)
        if not short:
            break
        best = max((j for j in jobs if j not in pick), key=lambda j: (len(rules[j] & short), -length[j] * j[2]))
        if not rules[best] & short:
            break
        pick.append(best)
        for name in rules[best]:
            count[name] += 1
    pick.sort(key=lambda j: (list(T.FAMILIES).index(j[0]), j[1], j[2]))
    for name in O.TIEBREAK:
        print("%-15s caught by %3d of %d searched, %d picked" % (name, sum(name in r for r in rules.values()), len(jobs), count[name]))
    if unreached:
        print("no searched record catches %s" % ", ".join(unreached))
    print("%d records, %d nt" % (len(pick), sum(length[j] for j in pick)))
    with open(a.out, "w") as fh:
        json.dump({"generator": "tests/test_traceback_ties.py", "search": "tools/tie_corpus.py --seeds %d --target %d --per-family %d"
                   % (a.seeds, a.target, a.per_family),
                   "records": [{"family": f, "seed": s, "span": L} for f, s, L in pick]}, fh, indent=1)
        fh.write("\n")


if __name__ == "__main__":
    main()
