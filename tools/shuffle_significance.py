#!/usr/bin/env python3
"""MFE significance test (MirFold.shuffle_test, dinucleotide shuffles, global folds) on the passing candidate precursors of
a seeded Arabidopsis-law run.

Workload: the generator of tools/genome_regions.py (seeded genome and records, --nrec / --mb scale it), the fused candidate
pass on the genome path, and the distinct precursors of the structures with at least one code-0 duplex verdict
(records.candidate_precursors, what records.hairpin_significance scores).  Per device count: one timed
shuffle_test(K = --k); host clock around a call that returns synchronised, plus the library's stats.

In the same call:
  * totals-only pass against plain mirfold_fold on the same sequences: shuffle_test(K = --k-plain) folds the natives and
    replicates 0..K-1; mirfold_fold folds exactly those sequences (the natives plus the device's exported replicates) at
    the same span.  Cells are equal by construction; the host-side tally of the plain fold's totals must equal the test.
  * a seeded sample of precursors scored with shuffle_test against the CPU oracle folding the exported replicates.

    python tools/shuffle_significance.py --gpus 1 8 --out profiles/<name>.json
"""
import argparse
import json
import os
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(ROOT, "tools"))

import mir_prefer_b200 as mp  # noqa: E402
from mir_prefer_b200 import records as R  # noqa: E402
from genome_regions import gpu_info, make_genome, make_records  # noqa: E402


def tally(native, totals_per_k):
    n_le = np.zeros(len(native), np.int64)
    s = np.zeros(len(native), np.int64)
    q = np.zeros(len(native), np.int64)
    for t in totals_per_k:
        t = np.asarray(t, np.int64)
        n_le += t <= native
        s += t
        q += t * t
    return n_le, s, q


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, nargs="+", default=[1, 8])
    ap.add_argument("--nrec", type=int, default=20000)
    ap.add_argument("--mb", type=int, default=12)
    ap.add_argument("--span", type=int, default=300, help="span of the candidate pass")
    ap.add_argument("--k", type=int, default=1000)
    ap.add_argument("--k-plain", type=int, default=100)
    ap.add_argument("--seed", type=int, default=2026)
    ap.add_argument("--out", required=True)
    a = ap.parse_args()
    rng = np.random.default_rng(a.seed)
    contigs = make_genome(rng, a.mb * 1000000, 5)
    recs = make_records(rng, contigs, a.nrec)
    out = {"gpus": gpu_info(), "workload": {"genome_nt": sum(len(s) for _, s in contigs), "records": len(recs), "span": a.span,
                                             "seed": a.seed, "K": a.k, "mode": "di", "fold": "global (span 0)"}, "runs": []}
    with tempfile.TemporaryDirectory() as tmp:
        fa = os.path.join(tmp, "genome.fa")
        with open(fa, "wb") as f:
            for name, s in contigs:
                f.write(b">" + name.encode() + b"\n")
                b = s.tobytes()
                f.write(b"\n".join(b[k:k + 80] for k in range(0, len(b), 80)) + b"\n")
        idx = mp.FastaIndex(fa)
    import torch
    ndev = torch.cuda.device_count()
    with mp.MirFold(devices=[0]) as mf, mf.upload_genome(idx) as g:
        _, _, cand = R.candidates_of_records(mf, recs, a.span, genome=g)
        uniq, rows, _ = R.candidate_precursors(cand, recs, genome=g)
    lens = np.array([len(p) for p in uniq], np.int64)
    out["workload"].update({"structures": cand.nstructs, "passing_structures": int(len(rows)), "precursors": len(uniq),
                            "precursor_nt": int(lens.sum()), "precursor_len_min_median_max": [int(lens.min()), float(np.median(lens)), int(lens.max())]})
    print(json.dumps(out["workload"]), flush=True)
    for G in a.gpus:
        if G > ndev:
            out["runs"].append({"n_gpus": G, "skipped": "only %d devices" % ndev})
            continue
        with mp.MirFold(devices=list(range(G))) as mf:
            mf.shuffle_test(uniq[:500], 5, seed=1)                         # warm-up: modules, buffers
            t = time.perf_counter()
            tab, st = mf.shuffle_test(uniq, a.k, seed=a.seed, mode="di", with_stats=True)
            wall = time.perf_counter() - t
            run = {"n_gpus": G, "wall_s": wall, "stats": st, "nt_per_s": st["nt"] / wall, "cells_per_s": st["cells"] / wall,
                   "p_le_0.05": int((tab["p_value"] <= 0.05).sum()), "median_z": float(np.nanmedian(tab["z"]))}
            print("N=%d: K=%d, %.3f s, %.3g nt/s, %.3g cells/s" % (G, a.k, wall, run["nt_per_s"], run["cells_per_s"]), flush=True)
            if G == 1:
                # totals-only vs plain mirfold_fold on the same sequences, alternated twice
                L = int(max(5, lens.max()))
                seqs = list(uniq)
                for k in range(a.k_plain):
                    seqs += mf.shuffle_sequences(uniq, k, seed=a.seed)
                cmp_ = []
                for rep in range(2):
                    t = time.perf_counter()
                    tt, st_t = mf.shuffle_test(uniq, a.k_plain, seed=a.seed, with_stats=True)
                    w_t = time.perf_counter() - t
                    t = time.perf_counter()
                    res = mf.fold(seqs, L)
                    w_p = time.perf_counter() - t
                    tot = np.asarray(res.total_mfe_dcal, np.int64).copy()
                    st_p = res.stats
                    res.close()
                    n = len(uniq)
                    n_le, s, q = tally(tot[:n], [tot[n * (k + 1):n * (k + 2)] for k in range(a.k_plain)])
                    assert tt["native_dcal"].tolist() == tot[:n].tolist() and tt["n_le"].tolist() == n_le.tolist()
                    assert tt["sum_dcal"].tolist() == s.tolist() and tt["sumsq_dcal"].tolist() == q.tolist()
                    assert st_t["cells"] == st_p["cells"]
                    cmp_.append({"totals_only_s": w_t, "plain_fold_s": w_p, "cells": st_p["cells"],
                                 "totals_only_cells_per_s": st_t["cells"] / w_t, "plain_fold_cells_per_s": st_p["cells"] / w_p,
                                 "totals_only_ms_device": st_t["ms_device"], "plain_fold_ms_device": st_p["ms_device"]})
                    print("  rep %d: totals-only %.3f s | plain fold %.3f s | equal tallies" % (rep, w_t, w_p), flush=True)
                run["totals_only_vs_plain_fold"] = {"K": a.k_plain, "span": L, "reps": cmp_}
                # seeded sample against the CPU oracle
                import oracle as O
                pick = sorted(np.random.default_rng(a.seed).choice(len(uniq), size=min(16, len(uniq)), replace=False).tolist())
                sample = [uniq[k] for k in pick]
                Ks = 20
                ts = mf.shuffle_test(sample, Ks, seed=a.seed + 1)
                fold = lambda xs: [O.fold(x, max(5, len(x)))["total"] for x in xs]   # noqa: E731
                native = np.array(fold(sample), np.int64)
                n_le, s, q = tally(native, [fold(mf.shuffle_sequences(sample, k, seed=a.seed + 1)) for k in range(Ks)])
                ok = (ts["native_dcal"].tolist() == native.tolist() and ts["n_le"].tolist() == n_le.tolist() and
                      ts["sum_dcal"].tolist() == s.tolist() and ts["sumsq_dcal"].tolist() == q.tolist())
                run["cpu_oracle_sample"] = {"precursors": len(sample), "K": Ks, "replicate_totals": len(sample) * (Ks + 1), "equal": ok}
                assert ok, "shuffle_test differs from the CPU oracle"
                print("  CPU oracle sample: %d precursors x %d shuffles equal" % (len(sample), Ks), flush=True)
            out["runs"].append(run)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
