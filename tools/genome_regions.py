#!/usr/bin/env python3
"""Host path vs genome path of the fused candidate pass (records.candidates_of_records) on an Arabidopsis-sized workload.

  host path  : FastaIndex.extend_region_sequence per record, then candidates_of_records (fold_sequence + pack +
               mirfold_fold_candidates)
  genome path: candidates_of_records(genome=g) (region table + mirfold_fold_candidates_regions); the genome is uploaded
               once per context (reported separately)

Workload (seeded): 5 contigs, 120 Mb, GC 0.36, lower-case masked stretches, N gaps, a planted hairpin in half of the
regions; 200 000 regions of the arabidopsis extend-region law (corpus._lengths), half on the minus strand, 30 % of them in
duplicated L/R pairs, 0-3 matures each.  One context per device count, the two paths alternated; candidates and verdicts
are asserted equal on every repetition.  Times are host clocks around calls that return synchronised, plus the library's
CUDA-event stats.  Writes one JSON file (--out); the FASTA goes to a temporary directory.

    python tools/genome_regions.py --gpus 1 8 --reps 3 --out profiles/<name>.json
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import mir_prefer_b200 as mp  # noqa: E402
from mir_prefer_b200 import records as R  # noqa: E402
from mir_prefer_b200.corpus import _lengths  # noqa: E402

_COMP = bytes.maketrans(b"ACGT", b"TGCA")


def make_genome(rng, total, ncontig):
    cuts = np.sort(rng.choice(np.arange(total // 10, total), size=ncontig - 1, replace=False))
    sizes = np.diff(np.concatenate([[0], cuts, [total]]))
    contigs = []
    for k, n in enumerate(sizes):
        n = int(n)
        s = np.frombuffer(b"ATGC", np.uint8)[rng.choice(4, size=n, p=[0.32, 0.32, 0.18, 0.18])].copy()
        for _ in range(n // 20000):                           # masked repeats: lower case
            a = int(rng.integers(0, n - 5000)); s[a:a + int(rng.integers(100, 5000))] |= 0x20
        for _ in range(n // 400000):                          # assembly gaps
            a = int(rng.integers(0, n - 50000)); s[a:a + int(rng.integers(100, 50000))] = ord("N")
        contigs.append(("Chr%d" % (k + 1), s))
    return contigs


def make_records(rng, contigs, nrec):
    lens = _lengths(rng, nrec, "arabidopsis")
    clen = np.array([len(s) for _, s in contigs], np.int64)
    which = rng.choice(len(contigs), size=nrec, p=clen / clen.sum())
    recs = []
    k = 0
    while k < nrec:
        c, n = int(which[k]), int(lens[k])
        name, seq = contigs[c]
        a = int(rng.integers(1, len(seq) - n))
        strand = "+-"[int(rng.integers(2))]
        if rng.random() < 0.5:                                # planted hairpin (plus-strand bases; minus records see it reversed)
            arm = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, size=int(rng.integers(20, 30)))]
            loop = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, size=int(rng.integers(6, 40)))]
            hp = np.concatenate([arm, loop, np.frombuffer(arm.tobytes().translate(_COMP)[::-1], np.uint8)])
            o = a - 1 + int(rng.integers(0, max(1, n - len(hp))))
            seq[o:o + len(hp)] = hp[:max(0, min(len(hp), len(seq) - o))]
        mats = []
        for _ in range(int(rng.integers(0, 4))):
            ml = int(rng.choice([20, 21, 22, 24, 25]))
            m0 = a + int(rng.integers(0, max(1, n - ml)))
            mats.append((m0, m0 + ml, strand, int(rng.integers(1, 500))))
        locus = (a + n // 3, a + n // 3 + 21)
        pair = rng.random() < 0.15 and k + 1 < nrec           # 15 % pairs -> 30 % of the records are duplicated L/R
        for tag in (("L", "R") if pair else ("0",)):
            recs.append(R.LocusRecord(name, (a, a + n), strand, locus, tag, [(locus[0], locus[1], strand)], mats, None))
        k += 2 if pair else 1
    return recs


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
    except (OSError, subprocess.SubprocessError) as e:
        return ["nvidia-smi unavailable: %s" % e]


def host_path(mf, idx, recs, span):
    t0 = time.perf_counter()
    filled = [r._replace(seq=idx.extend_region_sequence(r.seqid, r.region)) for r in recs]
    t1 = time.perf_counter()
    ss, table, cand = R.candidates_of_records(mf, filled, span)
    t2 = time.perf_counter()
    return ss, table, cand, {"extract_s": t1 - t0, "candidates_of_records_s": t2 - t1, "end_to_end_s": t2 - t0}


def genome_path(mf, g, recs, span):
    t0 = time.perf_counter()
    R.region_table(g, recs)                                   # timed alone too; candidates_of_records builds it again
    t1 = time.perf_counter()
    ss, table, cand = R.candidates_of_records(mf, recs, span, genome=g)
    t2 = time.perf_counter()
    return ss, table, cand, {"region_table_s": t1 - t0, "candidates_of_records_s": t2 - t1, "end_to_end_s": t2 - t1}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, nargs="+", default=[1, 8])
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--nrec", type=int, default=200000)
    ap.add_argument("--mb", type=int, default=120)
    ap.add_argument("--span", type=int, default=300)
    ap.add_argument("--seed", type=int, default=2026)
    ap.add_argument("--out", required=True)
    a = ap.parse_args()
    rng = np.random.default_rng(a.seed)
    t0 = time.perf_counter()
    contigs = make_genome(rng, a.mb * 1000000, 5)
    recs = make_records(rng, contigs, a.nrec)
    out = {"gpus": gpu_info(), "workload": {"genome_nt": sum(len(s) for _, s in contigs), "contigs": len(contigs), "records": len(recs),
                                             "minus": sum(r.strand == "-" for r in recs), "span": a.span, "seed": a.seed}, "runs": []}
    with tempfile.TemporaryDirectory() as tmp:
        fa = os.path.join(tmp, "genome.fa")
        with open(fa, "wb") as f:
            for name, s in contigs:
                f.write(b">" + name.encode() + b"\n")
                b = s.tobytes()
                f.write(b"\n".join(b[k:k + 80] for k in range(0, len(b), 80)) + b"\n")
        t1 = time.perf_counter()
        idx = mp.FastaIndex(fa)
        out["workload"]["make_s"], out["workload"]["fasta_index_s"] = t1 - t0, time.perf_counter() - t1
    out["workload"]["region_nt"] = int(sum(r.region[1] - r.region[0] for r in recs))
    print(json.dumps(out["workload"]), flush=True)
    import torch
    ndev = torch.cuda.device_count()
    for G in a.gpus:
        if G > ndev:
            out["runs"].append({"n_gpus": G, "skipped": "only %d devices" % ndev})
            continue
        with mp.MirFold(devices=list(range(G))) as mf:
            t = time.perf_counter()
            g = mf.upload_genome(idx)
            run = {"n_gpus": G, "genome_upload_s": time.perf_counter() - t, "host": [], "genome": []}
            with g:
                host_path(mf, idx, recs[:2000], a.span)       # warm-up of both paths (modules, pinned pools)
                genome_path(mf, g, recs[:2000], a.span)
                for rep in range(a.reps):
                    ss_h, tab_h, cand_h, th = host_path(mf, idx, recs, a.span)
                    ss_g, tab_g, cand_g, tg = genome_path(mf, g, recs, a.span)
                    assert ss_g == ss_h, "candidate structures differ"
                    assert tab_g._table == tab_h._table, "verdicts differ"
                    assert cand_g.nverdicts == cand_h.nverdicts and cand_g.nstructs == cand_h.nstructs
                    for t_, c_, key in ((th, cand_h, "host"), (tg, cand_g, "genome")):
                        t_["stats"] = c_.stats
                        t_["nstructs"], t_["nverdicts"] = c_.nstructs, c_.nverdicts
                        run[key].append(t_)
                    print("N=%d rep %d: host %.3f s (extract %.3f, call %.3f ms) | genome %.3f s (table %.3f, call %.3f ms) | equal" %
                          (G, rep, th["end_to_end_s"], th["extract_s"], cand_h.stats["ms_total"], tg["end_to_end_s"],
                           tg["region_table_s"], cand_g.stats["ms_total"]), flush=True)
            for key in ("host", "genome"):
                run[key + "_median_end_to_end_s"] = float(np.median([x["end_to_end_s"] for x in run[key]]))
            out["runs"].append(run)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({r["n_gpus"]: (r.get("host_median_end_to_end_s"), r.get("genome_median_end_to_end_s")) for r in out["runs"]}))


if __name__ == "__main__":
    main()
