"""The bench.py JSON contract, checked on the committed lines of the last GPU round (profiles/) and on a live
run of the CPU reference arm (a tiny sample)."""
import glob
import json
import os
import subprocess
import sys

import pytest

from conftest import ROOT

BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches"}


def _last(pattern):
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", pattern)))
    assert files, pattern
    return json.loads(open(files[-1]).read().strip().splitlines()[-1])


def test_committed_bench_line_has_every_contract_key():
    d = _last("r02_v*_bench.json")
    assert BASE_KEYS <= set(d) and {"roofline", "cpu_baseline", "clocks"} <= set(d)
    assert d["metric"].startswith("folded nt/sec") and d["unit"] == "nt/s" and d["higher_is_better"] is True
    assert d["scaling"] == "strong" and d["data"] == "synthetic" and d["vs_baseline"] is None
    assert "workload" in d["config"] and "model" not in d["config"] and "configs[2]" in d["config"]["workload"]
    assert d["n_gpus"] == 1 and d["warmup"] >= 3 and d["gpu_launches"] > 0
    assert abs(d["value"] - d["config"]["nt"] / (d["ms_per_step"] * 1e-3)) / d["value"] < 1e-6
    assert d["parity_in_run"]["equal"] is True and d["parity_in_run"]["text_bytes"] == 1235240762
    e = d["e2e"]
    assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(e)
    assert e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0 and e["value"] < d["value"]
    r = d["roofline"]
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(r)
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9 and 0 < r["frac"] < 1
    c = d["cpu_baseline"]
    assert {"value", "unit", "cores", "kind", "sample"} <= set(c) and c["kind"] in ("reference", "port")
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(d["clocks"])
    assert not set(d["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}


def test_committed_multi_gpu_lines_are_strong_scaling_through_one_context():
    one = _last("r02_v*_bench.json")
    for n in (2, 4, 8):
        d = _last("r02_v*_bench_%dgpu.json" % n)
        assert d["n_gpus"] == n and d["scaling"] == "strong" and d["config"]["devices"] == n
        assert d["config"]["nt"] == one["config"]["nt"]                       # the same job on more GPUs
        assert d["parity_in_run"]["equal"] is True                           # the multi-device result is the RNALfold text
        assert d["sharding"]["lpt_imbalance"] < 1.001
        assert d["e2e"]["value"] < d["value"] and d["weak"]["scaling"] == "weak"
        assert d["value"] > 0.85 * n * one["value"]                          # resident strong-scaling efficiency


def test_committed_reference_line():
    d = _last("r02_v*_bench_reference.json")
    assert d["impl"] == "reference" and BASE_KEYS <= set(d)
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]
    assert d["cpu_baseline"]["value"] == d["value"] and d["gpu_launches"] == 0


def test_reference_arm_runs_here():
    """bench.py --impl reference on a tiny sample (the reference's RNALfold, or the oracle port without it)."""
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--ref-loci-per-core", "1"], stdout=subprocess.PIPE, check=True, timeout=600).stdout.decode()
    d = json.loads(out.strip().splitlines()[-1])
    assert d["impl"] == "reference" and d["value"] > 0 and d["unit"] == "nt/s" and d["steps"] == 1


@pytest.mark.gpu
def test_dump_outputs_hold_the_oracles_result(oracle, tmp_path):
    """bench.py --dump-outputs on a small slice of the workload: the .npy files are the oracle's fold of the same loci."""
    import numpy as np
    from mir_prefer_b200.corpus import synth_loci
    dump = tmp_path / "dump"
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--loci", "64", "--steps", "2", "--warmup", "1", "--no-cpu",
                          "--no-sha", "--no-dropin", "--dump-outputs", str(dump)], stdout=subprocess.PIPE, check=True, timeout=600,
                         env=dict(os.environ, MIRFOLD_CORPUS_DIR=str(tmp_path))).stdout.decode()
    d = json.loads(out.strip().splitlines()[-1])
    assert d["steps"] == 2 and d["dump_outputs"]["records"] == 64 and d["dump_outputs"]["bytes"] <= 64 << 20
    a = {f.stem: np.load(f) for f in dump.glob("*.npy")}
    assert len(a) == 8 and all(x.dtype in (np.float32, np.float64) for x in a.values())
    want = [oracle.fold(s, 300) for s in synth_loci(1002, 64, "arabidopsis")]      # bench.WORKLOADS["arabidopsis"], rank 0
    assert a["records"].tolist() == a["hit_records"].tolist() == list(range(64))
    assert a["total_mfe_dcal"].tolist() == [o["total"] for o in want]
    assert a["hit_count"].tolist() == [len(o["hits"]) for o in want]
    hits = [h for o in want for h in o["hits"]]
    assert a["hit_start"].tolist() == [h[2] for h in hits] and a["hit_mfe_dcal"].tolist() == [h[1] for h in hits]
    assert a["hit_len"].tolist() == [len(h[0]) for h in hits]
    assert "".join(".()"[int(v)] for v in a["hit_ss"]) == "".join(h[0] for h in hits)   # codes 0, 1, -1
