#!/usr/bin/env python3
"""Whole contigs larger than device memory: segmented folds of long tiled loci (mirfold_plan_segments) on one GPU.

  chr1-sized : a seeded 30.4 Mb contig (the size of Arabidopsis chr1), both strands, at L = 300, folded from a resident
               genome in the default context: wall time, device ms, nt/s, DP cells/s and peak device bytes (the lowest
               free memory torch.cuda.mem_get_info sees, sampled every 20 ms during the call, against free memory before it)
  12 Mb A/B  : a 12 Mb locus at L = 300 (about 74 GB: one band in the default context), folded unsegmented (default
               context) and segmented (MIRFOLD_MEM_BUDGET_MB = 16384), alternated --reps times in this process; hits and
               totals asserted byte-identical every time
  maize-sized: a seeded 300 Mb contig, plus strand, if the host has room for its hits (--maize-min-host-gb)

The GPU's name and power limit are read in the same run.  Writes one JSON file (--out).

    python tools/segmented_fold.py --out profiles/r05_segmented_fold.json
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import mir_prefer_b200 as mp  # noqa: E402
from mir_prefer_b200.fold import plan_segments  # noqa: E402

L = 300


class PackedGenome:
    """What MirFold.upload_genome needs of a FastaIndex: the packed contigs."""

    def __init__(self, names, seqs):
        self.names, self.seqs = names, seqs

    def packed(self):
        off = np.zeros(len(self.seqs) + 1, np.uint64)
        off[1:] = np.cumsum([len(s) for s in self.seqs], dtype=np.uint64)
        return self.names, b"".join(self.seqs), off


def seeded_contig(seed, n):
    """ACGT with GC 0.36, planted GC stem-loops every ~2 kb and N runs every ~1 Mb."""
    rng = np.random.default_rng(seed)
    s = np.frombuffer(b"ACGT", np.uint8)[rng.choice(4, n, p=[0.32, 0.18, 0.18, 0.32])].copy()
    comp = bytes.maketrans(b"GC", b"CG")
    for a in rng.integers(0, n - 64, n // 2000).tolist():
        arm = np.frombuffer(b"GC", np.uint8)[rng.integers(0, 2, 12)].tobytes()
        hp = arm + b"TTCG" + arm.translate(comp)[::-1]
        s[a:a + len(hp)] = np.frombuffer(hp, np.uint8)
    for a in rng.integers(0, n - 500, max(1, n // 1_000_000)).tolist():
        s[a:a + int(rng.integers(50, 400))] = ord("N")
    return s.tobytes()


class FreeSampler:
    def __init__(self, torch):
        self.torch, self.low, self.stop = torch, None, False

    def __enter__(self):
        self.before = self.torch.cuda.mem_get_info()[0]
        self.low = self.before
        self.t = threading.Thread(target=self.run, daemon=True)
        self.t.start()
        return self

    def run(self):
        while not self.stop:
            self.low = min(self.low, self.torch.cuda.mem_get_info()[0])
            time.sleep(0.02)

    def __exit__(self, *a):
        self.stop = True
        self.t.join()

    @property
    def peak(self):
        return int(self.before - self.low)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,memory.total", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def contig_run(ctx, torch, name, seq, strands):
    g = ctx.upload_genome(PackedGenome([name], [seq]))
    n = len(seq)
    reg = g.regions([name] * len(strands), [1] * len(strands), [n + 1] * len(strands), strands)
    with FreeSampler(torch) as fs:
        t0 = time.perf_counter()
        res = g.fold_regions(reg, L)
        wall = time.perf_counter() - t0
    st = res.stats
    out = {"nt": int(st["nt"]), "strands": strands, "wall_s": wall, "ms_device": st["ms_device"], "ms_fill": st["ms_fill"],
           "ms_f3": st["ms_f3"], "ms_trace": st["ms_trace"], "ms_d2h": st["ms_d2h"], "cells": int(st["cells"]),
           "nt_per_s": st["nt"] / wall, "cells_per_s": st["cells"] / wall, "peak_device_bytes": fs.peak,
           "nhits": int(res.nhits), "ss_bytes": int(res.ss_bytes), "fill_units": int(st["fill_units"]),
           "kernel_launches": int(st["kernel_launches"]),
           "totals_dcal": [res.total(r) for r in range(len(strands))],
           "locus_bytes": int(plan_segments(n, L, 1 << 62)["device_bytes"][0]),
           "segments_default_lane": len(plan_segments(n, L, ctx_lane_bytes(torch)))}
    res.close()
    g.close()
    return out


def ctx_lane_bytes(torch):
    """A lane's share of the default context's budget (mirfold_open: min(60 % of free memory, 96 GB), two lanes)."""
    return min(int(torch.cuda.mem_get_info()[0] * 0.60), 96 << 30) // 2


def fold_budget(mb):
    old = os.environ.get("MIRFOLD_MEM_BUDGET_MB")
    if mb:
        os.environ["MIRFOLD_MEM_BUDGET_MB"] = str(mb)
    try:
        return mp.MirFold()
    finally:
        if old is None:
            os.environ.pop("MIRFOLD_MEM_BUDGET_MB", None)
        else:
            os.environ["MIRFOLD_MEM_BUDGET_MB"] = old


def ab_12mb(reps):
    n = 12_000_000
    s = seeded_contig(12, n).decode()
    out = {"n": n, "locus_bytes": int(plan_segments(n, L, 1 << 62)["device_bytes"][0]),
           "segments_16GB": len(plan_segments(n, L, (16384 << 20) // 2)), "unsegmented_s": [], "segmented_s": []}
    whole_ctx, seg_ctx = fold_budget(0), fold_budget(16384)
    want = None
    for _ in range(reps):
        for key, ctx in (("unsegmented_s", whole_ctx), ("segmented_s", seg_ctx)):
            t0 = time.perf_counter()
            res = ctx.fold([s], L)
            out[key].append(time.perf_counter() - t0)
            got = (res.hits(0), res.total(0))
            st = res.stats
            out.setdefault(key.replace("_s", "_stats"), {k: st[k] for k in ("ms_device", "ms_fill", "ms_f3", "ms_trace", "ms_d2h",
                                                                           "kernel_launches", "fill_units", "n_chunks")})
            res.close()
            if want is None:
                want = got
            assert got == want, key
    whole_ctx.close()
    seg_ctx.close()
    out["nhits"] = len(want[0])
    out["outputs_equal"] = True
    out["ratio_segmented_over_unsegmented_median"] = float(np.median(out["segmented_s"]) / np.median(out["unsegmented_s"]))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--maize-min-host-gb", type=float, default=40.0)
    a = ap.parse_args()
    import torch
    torch.cuda.init()
    rec = {"gpu": gpu_info(), "span": L, "note": "one GPU; times are host clocks around calls that return synchronised"}
    ctx = mp.MirFold()
    ctx.close()
    ctx = mp.MirFold()
    rec["chr1_30_4Mb"] = contig_run(ctx, torch, "chr1", seeded_contig(30, 30_400_000), ["+", "-"])
    ctx.close()
    rec["locus_12Mb_ab"] = ab_12mb(a.reps)
    avail = os.sysconf("SC_AVPHYS_PAGES") * os.sysconf("SC_PAGE_SIZE") / 2**30
    rec["host_available_gb"] = avail
    if avail >= a.maize_min_host_gb:
        ctx = mp.MirFold()
        rec["maize_chr1_300Mb"] = contig_run(ctx, torch, "chr1", seeded_contig(300, 300_000_000), ["+"])
        ctx.close()
    else:
        rec["maize_chr1_300Mb"] = "not run: %.1f GB of host memory available, %.0f GB asked for" % (avail, a.maize_min_host_gb)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps(rec, indent=1))


if __name__ == "__main__":
    main()
