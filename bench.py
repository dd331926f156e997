#!/usr/bin/env python3
"""bench.py -- fold-stage throughput on B200 (BASELINE.json metric: folded nt/sec, RNALfold -L 300, at 1/2/4/8 B200).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one pass of the hot path (encode -> c/fML band fill -> f3 -> plan/traceback/emission) over the whole
workload.  Workload = BASELINE.json configs[2] ("arabidopsis-200k": 200 000 loci of the reference's extend_region
length law, L=300, seed 1002, SURVEY.md 8d) -- the config the metric is quoted on -- folded through ONE libmirfold
context that owns all N GPUs (the product's own multi-GPU path: LPT sharding by DP cells, one host thread and two
pipeline lanes per device, no collective), i.e. STRONG scaling.  Under torchrun rank 0 drives the context; the other
ranks only take part in the barriers (loci are independent: there is no data-path exchange to give them).
`value` = nt/s with the raw sequences resident in HBM on every device and the results left in HBM (CUDA events on
the library's streams, max over devices); `e2e` = the same metric through the public host API mirfold_fold (host
buffers in, hit records out, all copies inside the timed region).  `weak` keeps round 1's line: every rank folds its
own parity-10k batch (BASELINE configs[1]) on its own GPU.

--dump-outputs DIR writes the result of the last timed step as DIR/<name>.npy (see dump_outputs()), so that two builds
run with the same arguments, hence on the same seeded inputs, can be compared output for output.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
from mir_prefer_b200.corpus import synth_loci  # noqa: E402  (pure generator; nothing under oracle/ is on the product arm's path)

METRIC = "folded nt/sec (RNALfold -L 300, bit-exact MFE)"
UNIT = "nt/s"
SPAN = 300


WORKLOADS = {   # SURVEY.md 8(d): name -> (length law, base seed, BASELINE configs index)
    "parity": ("parity", 1001, 1), "arabidopsis": ("arabidopsis", 1002, 2), "long": ("long", 1003, 3), "sweep": ("sweep", 1004, 4)}
WORKLOAD = "arabidopsis"
DEFAULT_LOCI = {"parity": 10000, "arabidopsis": 200000, "long": 1400, "sweep": 5000}


def workload(rank, nloci, name=None):
    law, seed, _ = WORKLOADS[name or WORKLOAD]
    return synth_loci(seed + rank, nloci, law)


def workload_packed(rank, nloci, name=None):
    """(uint8 buffer, uint64 offsets) of the workload; the generator is a sequential Python loop (30 s for 200 k
    loci), so the packed corpus is cached under the temp dir for the back-to-back runs of a scaling sweep."""
    law, seed, _ = WORKLOADS[name or WORKLOAD]
    fn = os.path.join(os.environ.get("MIRFOLD_CORPUS_DIR") or tempfile.gettempdir(), "mirfold_corpus_%s_%d_%d.npz" % (law, seed + rank, nloci))
    try:
        z = np.load(fn)
        return z["buf"], z["off"]
    except Exception:
        pass
    seqs = synth_loci(seed + rank, nloci, law)
    off = np.zeros(len(seqs) + 1, np.uint64)
    off[1:] = np.cumsum([len(s) for s in seqs], dtype=np.uint64)
    buf = np.frombuffer("".join(seqs).encode("ascii"), np.uint8)
    try:
        tmp = fn + ".%d.tmp.npz" % os.getpid()
        np.savez(tmp, buf=buf, off=off)
        os.replace(tmp, fn)
    except Exception:
        pass
    return buf, off


def unpack(buf, off, lo=0, hi=None):
    hi = len(off) - 1 if hi is None else hi
    raw = buf.tobytes()
    return [raw[int(off[k]):int(off[k + 1])].decode("ascii") for k in range(lo, hi)]


# ---------------------------------------------------------------------------------- work model
def g_of_d():
    G = np.zeros(4200, np.int64)
    for d in range(6, len(G)):
        K = min(30, d - 6)
        G[d] = sum(min(30 - u, d - u - 6) + 1 for u in range(K + 1))
    return G


def typed_fraction(seqs, span, sample=48):
    """rho = fraction of band cells (i,j) whose bases can pair (SURVEY 8d), on a seeded sample."""
    pair = np.zeros((8, 8), bool)
    for a, b in ((2, 3), (3, 2), (3, 4), (4, 3), (1, 4), (4, 1)):
        pair[a, b] = True
    code = np.zeros(256, np.int64)
    for ch, v in zip("ACGUT", (1, 2, 3, 4, 4)):
        code[ord(ch)] = v
        code[ord(ch.lower())] = v
    typed = cells = 0
    for s in seqs[:sample]:
        c = code[np.frombuffer(s.encode(), np.uint8)]
        n = len(c)
        for d in range(4, min(span, n - 1) + 1):
            cells += n - d
            if d < min(span, n):
                typed += int(pair[c[:n - d], c[d:]].sum())
    return typed / max(cells, 1)


def algorithmic_terms(lens, span, rho):
    """T_alg of SURVEY.md 8(d): sum over cells of max(0,d-8) + rho^2*G(d) + 16 min-plus terms."""
    G = g_of_d()
    tot = 0.0
    cells = 0
    uniq, counts = np.unique(np.asarray(lens, np.int64), return_counts=True)
    for n, mult in zip(uniq.tolist(), counts.tolist()):
        dmax = min(span, n - 1)
        if dmax < 4:
            continue
        d = np.arange(4, dmax + 1)
        cnt = n - d
        tot += mult * float((cnt * (np.maximum(0, d - 8) + rho * rho * G[d] + 16)).sum())
        cells += mult * int(cnt.sum())
    return tot, cells


# ---------------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")] + [time.time()])

    def window(self, t0, t1):
        """keep the samples taken inside [t0, t1] (the sampler is started early: nvidia-smi takes ~0.1 s to come up)"""
        inside = [r for r in self.rows if t0 <= r[-1] <= t1 + 0.05]
        if len(inside) >= 1:
            self.rows = inside

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                pass
        self.rows = [r[:-1] for r in self.rows]
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 9:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------- CPU reference arm
def _rlf_binary():
    rlf = os.path.join(ROOT, "oracle", "_ref", "RNALfold")
    if os.path.exists(rlf) and os.access(rlf, os.X_OK):
        return rlf, "reference"
    cli = os.path.join(ROOT, "oracle", "_build", "lfold_oracle")
    if not os.path.exists(cli):
        subprocess.run(["make", "-C", os.path.join(ROOT, "oracle"), "all"], check=True, stdout=subprocess.DEVNULL)
    return cli, "port"


def cpu_fold_stage(seqs, span, cores):
    """The reference's fold stage on host cores: P contiguous shards by locus count
    (num_each_piece = int(total/P)+1, miR_PREFeR.py:1329-1354), one `RNALfold -L span` process per
    shard, all concurrent (MP:3113-3118), output to tmpfs.  Returns (seconds, kind)."""
    binary, kind = _rlf_binary()
    P = max(1, min(cores, len(seqs)))
    per = len(seqs) // P + 1
    tmp = tempfile.mkdtemp(dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
    files = []
    for k in range(P):
        part = seqs[k * per:(k + 1) * per]
        if not part:
            continue
        fn = os.path.join(tmp, "in_%d.fa" % k)
        with open(fn, "w") as f:
            for r, s in enumerate(part):
                f.write(">r%d_%d\n%s\n" % (k, r, s))
        files.append(fn)
    t0 = time.perf_counter()
    procs = []
    for fn in files:
        procs.append(subprocess.Popen([binary, "-L", str(span)], stdin=open(fn), stdout=open(fn + ".out", "w")))
    for p in procs:
        if p.wait() != 0:
            raise RuntimeError("reference fold process failed")
    dt = time.perf_counter() - t0
    for fn in files:
        os.remove(fn)
        os.remove(fn + ".out")
    os.rmdir(tmp)
    return dt, kind, len(files)


def workload_name(nloci):
    law, seed, idx = WORKLOADS[WORKLOAD]
    shape = {"parity": "300-600 nt", "arabidopsis": "extend_region length law (70 % 300 nt, 5 % 299, 20 % 325, 5 % 301-350)",
             "long": "2-10 kb log-uniform", "sweep": "lognormal(400, 0.6) clipped [60, 5000]"}[law]
    return "%s-%s (BASELINE configs[%d]): %d loci, %s, GC 0.40, embedded hairpins, L=%d, seed %d" % (
        law, ("%dk" % (nloci // 1000)) if nloci % 1000 == 0 else str(nloci), idx, nloci, shape, SPAN, seed)


def run_reference(args, rank, world):
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    # bounded sample: RNALfold costs about 2 us per DP cell (0.09 s per 300-nt locus, 0.2 s per 450-nt locus); one
    # shard per core; keep the whole run near 100 s
    per_locus_s = {"parity": 0.2, "arabidopsis": 0.1, "long": 3.0, "sweep": 0.2}[WORKLOAD]
    per_core = int(max(4, min(args.ref_loci_per_core, 100.0 / (args.steps + 1) / per_locus_s)))
    per_step = max(cores, min(args.loci, cores * per_core))
    seqs = workload(0, per_step)
    nt = sum(len(s) for s in seqs)
    for _ in range(min(args.warmup, 1)):
        cpu_fold_stage(seqs[:cores], SPAN, cores)
    t = 0.0
    kind, used = "reference", cores
    for _ in range(args.steps):
        dt, kind, used = cpu_fold_stage(seqs, SPAN, cores)
        t += dt
    val = nt * args.steps / t
    sample = "first %d loci (%d nt) of the workload per step, %d concurrent RNALfold -L %d processes" % (per_step, nt, used, SPAN)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "int32", "data": "synthetic",
        "config": {"workload": workload_name(args.loci) + "; bounded sample per step", "span_L": SPAN, "loci_per_step": per_step},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": used, "kind": kind, "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


# ---------------------------------------------------------------------------------- ours
def text_sha256(mf, buf, off, span):
    """sha256 of the complete RNALfold-format text of the workload (headers as tools/bulk_parity.py wrote them)."""
    seqs = unpack(buf, off)
    text = "".join(">locus%d:%d-%d + 1-22 0 1,22,+\n%s\n" % (k, 1, len(x) + 1, x) for k, x in enumerate(seqs))
    out = mf.fold_text_bytes(text, span)
    return hashlib.sha256(out).hexdigest(), len(out)


def known_pin(nloci):
    law, seed, _ = WORKLOADS[WORKLOAD]
    try:
        pins = json.load(open(os.path.join(ROOT, "tests", "golden", "bulk_pins.json")))
    except Exception:
        return None
    for p in pins["pins"] + pins.get("full_size_pins_not_in_the_test_suite", []):
        if p["law"] == law and p["nloci"] == nloci and p["span"] == SPAN and p["seed"] == seed:
            return p
    return None


def weak_line(args, mp, torch, dist, rank, world, local_rank, barrier):
    """Round 1's line, kept as an extra key: every rank folds its own parity-10k batch on its own GPU."""
    buf, off = workload_packed(rank, 10000, "parity")
    nt = int(off[-1])
    mf = mp.MirFold(devices=[local_rank])
    steps = args.steps
    with mf.upload(buf, off, SPAN) as batch:
        batch.fold().close()
        barrier()
        t_dev = 0.0
        for _ in range(steps):
            with batch.fold() as r:
                t_dev += r.stats["ms_device"] * 1e-3
        barrier()
        mf.fold_packed(buf, off, SPAN).close()
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            mf.fold_packed(buf, off, SPAN).close()
        barrier()
        t_e2e = time.perf_counter() - t0
    mf.close()
    tt = torch.tensor([t_dev, t_e2e], dtype=torch.float64, device="cuda")
    tot = torch.tensor([float(nt)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    t_dev, t_e2e = tt.tolist()
    return {"scaling": "weak", "workload": "parity-10k (BASELINE configs[1]) per GPU, one single-device context per rank",
            "value": tot.item() * steps / t_dev, "e2e": tot.item() * steps / t_e2e, "unit": UNIT, "steps": steps,
            "ms_per_step": 1e3 * t_dev / steps, "e2e_ms_per_step": 1e3 * t_e2e / steps}


def run_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    import mir_prefer_b200 as mp
    from mir_prefer_b200 import _lib
    from mir_prefer_b200.fold import FLAG_SERIAL, plan_shards
    if not os.path.exists(_lib.LIB_PATH):
        raise RuntimeError("libmirfold.so missing (run python __graft_entry__.py); there is no CPU fallback")
    torch.cuda.set_device(local_rank)
    cpu_group = None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        dist.barrier()                                   # the NCCL communicator over all N ranks exists and works
        cpu_group = dist.new_group(backend="gloo")

    def barrier():
        # Ranks > 0 wait on the CPU (gloo): an NCCL barrier would park a spinning kernel on every waiting GPU, and those
        # are the GPUs rank 0's context is folding on (two processes time-slice a GPU: measured 2x slower at N = 2).
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier(group=cpu_group)

    out = None
    if rank == 0:
        buf, off = workload_packed(0, args.loci)
        lens = np.diff(off.astype(np.int64))
        nt = int(off[-1])
        mf = mp.MirFold(devices=list(range(world)))
        batch = mf.upload(buf, off, SPAN)
        sampler = ClockSampler(local_rank)
        sampler.start()
        for _ in range(args.warmup):
            batch.fold().close()
    barrier()
    # ---- device-resident timing (value): sequences in HBM on every device, results stay in HBM
    if rank == 0:
        t_w0 = time.time()
        t0 = time.perf_counter()
        dev_ms, launches = [], 0
        stage = {"ms_fill": 0.0, "ms_f3": 0.0, "ms_trace": 0.0}
        for _ in range(args.steps):
            with batch.fold() as r:
                dev_ms.append(r.stats["ms_device"])     # CUDA events on the library's streams, max over devices
                launches += r.stats["kernel_launches"]
                n_chunks, tracebacks, cells = r.stats["n_chunks"], r.stats["tracebacks"], r.stats["cells"]
                last_step = (r.nhits, r.ss_bytes)
        wall_resident = time.perf_counter() - t0
    barrier()
    if rank == 0:
        sampler.window(t_w0, time.time())
        clocks = sampler.stop()
        t_dev = float(np.sum(dev_ms)) * 1e-3
        # ---- end to end through the public API: host buffers in, hit records out
        for _ in range(min(args.warmup, 2)):
            mf.fold_packed(buf, off, SPAN).close()
    barrier()
    if rank == 0:
        t0 = time.perf_counter()
        for _ in range(args.steps):
            with mf.fold_packed(buf, off, SPAN) as r:
                h2d, d2h, nhits = r.stats["h2d_bytes"], r.stats["d2h_bytes"], r.nhits
                e2e_split = {k: r.stats[k] for k in ("ms_total", "ms_h2d", "ms_device", "ms_d2h")}
    barrier()
    if rank == 0:
        t_e2e = time.perf_counter() - t0
        # ---- per-kernel durations for the roofline: one pass with a single lane per device, so that the CUDA-event
        # brackets of the stages are disjoint (in the pipelined passes a chunk's fill shares the SMs with the previous
        # chunk's traceback)
        batch.fold(flags=FLAG_SERIAL).close()            # the single-lane chunking sizes its buffers once
        with batch.fold(flags=FLAG_SERIAL) as r:
            serial = {k: r.stats[k] for k in ("ms_fill", "ms_f3", "ms_trace", "ms_device")}
        _, shard_cells = plan_shards(lens, SPAN, world)
        rho = typed_fraction(unpack(buf, off, 0, 48), SPAN)
        t_alg, _ = algorithmic_terms(lens, SPAN, rho)
        peak_a, peak_dpx, peak_s16 = mf.int_peak2()
        peak = max(peak_a, peak_dpx)
        fill_s = serial["ms_fill"] * 1e-3                   # slowest device's fill kernels, all its chunks
        terms_dev = t_alg * float(shard_cells.max()) / max(float(shard_cells.sum()), 1.0)   # the same device's share
        achieved = terms_dev / fill_s
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
            hbm_peak, hbm_src = float(peaks["hbm_gbs"]), "measured"
        except Exception:
            hbm_peak, hbm_src = 6650.0, "fallback"
        band_bytes = float(shard_cells.max()) * 8.0  # c + fML written once, int32
        # DRAM bytes of the same fill launches: not measurable inside a timed run (ncu replays kernels), so the committed
        # ncu --set full capture of this build is scaled by DP cells and labelled static
        traffic, traffic_note = None, "not measured in this run (ncu --set full summaries are under profiles/)"
        try:
            tr = json.load(open(os.path.join(ROOT, "profiles", "fill_traffic.json")))
            if tr["workload"] == WORKLOAD and SPAN == 300:
                traffic = tr["dram_bytes_per_cell"] * float(shard_cells.max())
                traffic_note = "static: %.1f B/cell x the device's DP cells, from %s (%s)" % (tr["dram_bytes_per_cell"], tr["source"], tr["kernel"])
        except Exception:
            pass
        out = {
            "metric": METRIC, "value": nt * args.steps / t_dev, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * t_dev / args.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "int32", "data": "synthetic",
            "config": {"workload": workload_name(args.loci), "span_L": SPAN, "loci": args.loci, "nt": nt,
                       "dp_cells": int(cells), "devices": world, "context": "one libmirfold context over all devices, driven by rank 0",
                       "cache": "band workspace (%.1f GB per step) far larger than L2; no flush needed" % (float(cells) * 12 / 1e9),
                       "tracebacks_per_step": int(tracebacks), "chunks_per_step": int(n_chunks)},
            "dp_cells_per_s": float(cells) * args.steps / t_dev,
            "wall_ms_per_step_resident": 1e3 * wall_resident / args.steps,
            "e2e": {"value": nt * args.steps / t_e2e, "unit": UNIT, "h2d_bytes_per_step": int(h2d),
                    "d2h_bytes_per_step": int(d2h), "ms_per_step": 1e3 * t_e2e / args.steps, "hits_per_step": int(nhits),
                    "last_step_split": e2e_split},
            "gpu_launches": int(launches),
            "sharding": {"lpt_imbalance": float(shard_cells.max()) / max(float(shard_cells.mean()), 1.0),
                         "host_overhead_ms_per_step": 1e3 * (t_e2e - t_dev) / args.steps,
                         "note": "no merge pass: every device downloads straight into the call's shared pinned result buffers"},
            "stage_ms_serial_pass": serial,
            "clocks": clocks,
            "roofline": {"bound": "int32-issue", "kernel": "k_fill_s16 (all buckets of the slowest device, serial pass)",
                         "achieved": achieved / 1e12, "peak": peak / 1e12,
                         "unit": "Tterm/s (1 min-plus term = 1 add + 1 min)", "frac": achieved / peak,
                         "peak_source": "measured live (mirfold_int_peak2): add+min %.2f / VIADDMNMX s32 %.2f / VIADDMNMX.S16x2 %.2f Tterm/s"
                                        % (peak_a / 1e12, peak_dpx / 1e12, peak_s16 / 1e12),
                         "frac_of_s16x2_peak": achieved / max(peak_s16, 1.0),
                         "algorithmic_terms_per_launch": terms_dev, "terms_per_cell": t_alg / max(float(cells), 1.0), "rho": rho,
                         "kernel_ms": fill_s * 1e3, "kernel_share_of_step": fill_s / max(serial["ms_device"] * 1e-3, 1e-9),
                         "traffic": traffic, "traffic_note": traffic_note,
                         "hbm": {"bound": "hbm", "achieved": band_bytes / fill_s / 1e9, "peak": hbm_peak, "unit": "GB/s",
                                 "frac": band_bytes / fill_s / 1e9 / hbm_peak, "peak_source": hbm_src,
                                 "note": "band store of c+fML (8 B/cell) only; the kernel is integer-issue bound"}},
        }
        if not args.no_sha:
            pin = known_pin(args.loci)
            t0 = time.perf_counter()
            sha, nbytes = text_sha256(mf, buf, off, SPAN)
            out["parity_in_run"] = {"text_sha256": sha, "text_bytes": nbytes, "rnalfold_text_in_out_s": time.perf_counter() - t0,
                                    "pinned_sha256": pin["sha256"] if pin else None,
                                    "equal": (sha == pin["sha256"]) if pin else None,
                                    "pin_source": "tests/golden/bulk_pins.json (text of oracle/_ref/RNALfold on the same input)"}
            if pin and sha != pin["sha256"]:
                raise RuntimeError("parity broken: text sha256 %s != pinned %s" % (sha, pin["sha256"]))
        if world == 1 and not args.no_dropin:
            out["drop_in"] = drop_in_stages(mf, buf, off, lens)
        if args.dump_outputs:
            out["dump_outputs"] = dump_outputs(batch, last_step, lens, args.dump_outputs)
        batch.close()
        mf.close()
    barrier()
    if not args.no_weak and (world > 1 or args.weak):
        w = weak_line(args, mp, torch, dist, rank, world, local_rank, barrier)
        if rank == 0:
            out["weak"] = w
    if rank == 0:
        if world == 1 and not args.no_cpu:
            cores = os.cpu_count() or 1
            sample_n = max(cores, min(args.loci, cores * args.ref_loci_per_core))
            sample = unpack(buf, off, 0, sample_n)
            dt, kind, used = cpu_fold_stage(sample, SPAN, cores)
            snt = sum(len(s) for s in sample)
            one = sample[:12]                                   # SURVEY 8(d): also the P=1 figure
            dt1, _, _ = cpu_fold_stage(one, SPAN, 1)
            out["cpu_baseline"] = {"value": snt / dt, "unit": UNIT, "cores": used, "kind": kind,
                                   "sample": "first %d loci (%d nt) of the same workload, %d concurrent RNALfold -L %d "
                                             "processes, %.1f s" % (sample_n, snt, used, SPAN, dt),
                                   "single_core_value": sum(len(x) for x in one) / dt1,
                                   "dp_cells_per_s": snt / dt * (float(cells) / max(nt, 1))}
        print(json.dumps(out))
    if world > 1:
        torch.cuda.synchronize()
        dist.barrier()
        dist.destroy_process_group()


def drop_in_stages(mf, buf, off, lens):
    """The stage-1 / stage-3 boundaries on a 10 000-locus slice of the workload (informational, outside the timed regions)."""
    n = min(10000, len(off) - 1)
    sub_off = off[:n + 1] - off[0]
    sub_buf = buf[:int(sub_off[-1])]
    with mf.fold_packed(sub_buf, sub_off, SPAN) as r:
        t0 = time.perf_counter()
        per_rec = r.classify(55)
        nstruct = sum(len(x) for x in per_rec)
        t_cls = time.perf_counter() - t0
    # stage 3 on the same structures: one synthetic 21-nt mature on the 5' arm of every structure
    queries = [(ss, (fs + 8, fs + 29), fs, 1, int(lens[k]) + 1, "+") for k, recs_ in enumerate(per_rec) for (_, fs, ss, _) in recs_]
    t0 = time.perf_counter()
    verdicts = mf.duplex(queries)
    t_dup = time.perf_counter() - t0
    out = {"loci": n, "classify_structures_ms": 1e3 * t_cls, "structures": nstruct, "duplex_queries_ms": 1e3 * t_dup,
           "duplex_queries": len(queries), "duplex_pass": sum(1 for v in verdicts if not isinstance(v, str))}
    # the same two stages fused on the device after traceback (mirfold_fold_candidates): whole call vs the plain fold
    regions = np.stack([np.ones(n, np.int64), lens[:n].astype(np.int64) + 1], axis=1)
    matures = np.zeros(n, [("start", "<i4"), ("end", "<i4"), ("strand", "<i4"), ("depth", "<i4")])
    matures["start"], matures["end"], matures["strand"], matures["depth"] = 40, 61, ord("+"), 50
    moff = np.arange(n + 1, dtype=np.uint64)
    mf.fold_candidates(sub_buf, sub_off, SPAN, regions, matures, moff)
    t0 = time.perf_counter()
    cand = mf.fold_candidates(sub_buf, sub_off, SPAN, regions, matures, moff)
    t_fused = time.perf_counter() - t0
    t0 = time.perf_counter()
    with mf.fold_packed(sub_buf, sub_off, SPAN) as r:
        d2h_plain = r.stats["d2h_bytes"]
    t_plain = time.perf_counter() - t0
    out["fused"] = {"fold_candidates_ms": 1e3 * t_fused, "plain_fold_ms": 1e3 * t_plain, "stage1_3_on_device_ms": 1e3 * (t_fused - t_plain),
                    "structures": cand.nstructs, "verdicts": cand.nverdicts, "d2h_bytes": cand.stats["d2h_bytes"],
                    "d2h_bytes_plain_fold": d2h_plain}
    return out


DUMP_SEED = 0
DUMP_RECORDS = 1 << 20          # per-record arrays: every record up to this many, else a seeded sample of this size
DUMP_HIT_NT = 300000            # per-hit arrays: the hits of a seeded sample of records with about this many input nt
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(batch, last_step, lens, outdir):
    """Write the result of the timed path's last step under outdir as .npy files (float64; the dot-brackets float32).

    The timed steps leave their results in HBM, so the same batch is folded once more outside the timed region with
    the download on; the fold is deterministic, and its hit count and dot-bracket bytes must equal the last timed
    step's.  Records are sampled by a seeded permutation, so the same arguments dump the same records:
      records, total_mfe_dcal, hit_count         per record: its index, total MFE (dcal/mol), hairpin lines printed
      hit_records                                the records whose hits follow (a prefix of the same permutation)
      hit_start, hit_len, hit_mfe_dcal           their hits, record by record in RNALfold's print order
      hit_ss                                     the hits' dot-brackets concatenated: '(' = 1, ')' = -1, '.' = 0
    """
    with batch.fold(download=True) as res:
        if (res.nhits, res.ss_bytes) != last_step or res.nseq != len(lens):
            raise RuntimeError("the downloaded fold (%d hits, %d B) differs from the last timed step (%d hits, %d B)"
                               % ((res.nhits, res.ss_bytes) + tuple(last_step)))
        perm = np.random.default_rng(DUMP_SEED).permutation(res.nseq)
        rec = np.sort(perm[:DUMP_RECORDS])
        arrays = {"records": rec.astype(np.float64), "total_mfe_dcal": res.total_mfe_dcal[rec].astype(np.float64),
                  "hit_count": res.hit_count[rec].astype(np.float64)}
        budget = DUMP_MAX_BYTES - sum(a.nbytes for a in arrays.values()) - 4096      # 4096: the .npy headers
        k = max(1, int(np.searchsorted(np.cumsum(lens[perm]), DUMP_HIT_NT, side="right")))
        while True:
            hrec = np.sort(perm[:k])
            hb, hc = res.hit_begin[hrec].astype(np.int64), res.hit_count[hrec].astype(np.int64)
            rows = np.repeat(hb, hc) + (np.arange(int(hc.sum())) - np.repeat(np.cumsum(hc) - hc, hc))
            hits = res.hit_table[rows]
            n = hits["len"].astype(np.int64)
            if 8 * (len(hrec) + 3 * len(rows)) + 4 * int(n.sum()) <= budget or k == 1:
                break
            k //= 2
        chars = np.repeat(hits["ss_off"].astype(np.int64), n) + (np.arange(int(n.sum())) - np.repeat(np.cumsum(n) - n, n))
        code = np.zeros(256, np.float32)
        code[ord("(")], code[ord(")")] = 1, -1
        arrays.update({"hit_records": hrec.astype(np.float64), "hit_start": hits["start"].astype(np.float64),
                       "hit_len": n.astype(np.float64), "hit_mfe_dcal": hits["mfe_dcal"].astype(np.float64),
                       "hit_ss": code[res.arena[chars]]})
    os.makedirs(outdir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(outdir, name + ".npy"), a)
    return {"dir": os.path.abspath(outdir), "files": sorted(arrays), "bytes": sum(a.nbytes for a in arrays.values()),
            "records": len(rec), "hit_records": len(hrec), "hits": len(rows)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--loci", type=int, default=0, help="loci of the whole job (default: the workload's BASELINE size, 200000 for arabidopsis)")
    ap.add_argument("--ref-loci-per-core", type=int, default=96, help="CPU legs: loci per host core and step (about 10 s of RNALfold)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-sha", action="store_true", help="skip the in-run sha256 parity check of the full text")
    ap.add_argument("--no-dropin", action="store_true", help="skip the stage-1/3 figures")
    ap.add_argument("--no-weak", action="store_true", help="skip the weak-scaling extra line at N > 1")
    ap.add_argument("--weak", action="store_true", help="also run the weak line at N = 1")
    ap.add_argument("--workload", default="arabidopsis", choices=sorted(WORKLOADS),
                    help="length law of SURVEY 8(d); the bench line of record is the default (arabidopsis-200k, BASELINE configs[2])")
    ap.add_argument("--span", type=int, default=300, help="RNALfold -L (default 300)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's result as DIR/<name>.npy (at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the result of --impl ours")
    global WORKLOAD, SPAN
    WORKLOAD, SPAN = args.workload, args.span
    if args.loci <= 0:
        args.loci = DEFAULT_LOCI[WORKLOAD]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world == 1 and args.gpus > 1:
        # convenience: re-launch under torchrun
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus),
               "--master-addr", "127.0.0.1", "--master-port", "29513", os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
