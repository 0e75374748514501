"""CPU: the committed bench lines (profiles/r0N_bench_*.json, produced by bench.py on B200s) carry every key the
measurement contract asks for, and the numbers in them are self-consistent (value = proofs / time, frac = achieved / peak).
Round-2 lines additionally: identical `config` on both arms, the pageable-memory e2e figure, the whole-step roofline,
the pairing check of a timed proof, and the extras (BASELINE configs[2] and configs[4])."""
import glob
import json
import os

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LINES = sorted(glob.glob(os.path.join(ROOT, "profiles", "r0[12]_bench_*.json")))
R02 = sorted(glob.glob(os.path.join(ROOT, "profiles", "r02_bench_*.json")))


@pytest.mark.parametrize("path", LINES, ids=[os.path.basename(p) for p in LINES])
def test_bench_line_contract(path):
    d = json.load(open(path))
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches", "clocks", "roofline"):
        assert k in d, k
    assert d["metric"] == "groth16_proofs_per_sec" and d["unit"] == "proofs/s" and d["higher_is_better"] is True
    assert d["scaling"] == "weak" and d["vs_baseline"] is None and d["data"] == "synthetic"
    assert d["warmup"] >= 3 and d["gpu_launches"] > 0
    cfg = d["config"]
    assert "workload" in cfg and "model" not in cfg
    # value is the whole-job aggregate: proofs of all ranks / device time of the timed steps
    proofs = d["n_gpus"] * cfg["proofs_per_step_per_gpu"] * d["steps"]
    assert d["value"] == pytest.approx(proofs / (d["ms_per_step"] * d["steps"] / 1e3), rel=1e-6)
    e = d["e2e"]
    assert e["unit"] == "proofs/s" and 0 < e["value"] <= d["value"] * 1.02
    assert e["h2d_bytes_per_step"] == cfg["proofs_per_step_per_gpu"] * cfg["n_vars"] * 32 and e["d2h_bytes_per_step"] > 0
    r = d["roofline"]
    for k in ("bound", "achieved", "peak", "unit", "frac", "traffic"):
        assert k in r, k
    assert r["frac"] == pytest.approx(r["achieved"] / r["peak"], rel=1e-9) and 0 < r["frac"] < 1
    c = d["clocks"]
    assert not set(c["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
    assert c["sm_mhz"] >= 0.9 * c["sm_max_mhz"]
    if "cpu_baseline" in d:
        b = d["cpu_baseline"]
        assert b["kind"] in ("port", "reference") and b["cores"] >= 1 and b["value"] > 0 and b["sample"]
        assert d["proof_matches_cpu_port"] is True


def test_reference_arm_line():
    d = json.load(open(os.path.join(ROOT, "profiles", "r01_ref_n1.json")))
    assert d["impl"] == "reference" and d["metric"] == "groth16_proofs_per_sec" and d["value"] > 0
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["e2e"]["value"] == d["value"] and d["cpu_baseline"]["value"] == d["value"]
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1


@pytest.mark.parametrize("path", R02, ids=[os.path.basename(p) for p in R02])
def test_round2_line_additions(path):
    d = json.load(open(path))
    assert d["proof_verifies"] is True
    pg = d["e2e"]["pageable"]
    assert 0 < pg["value"] <= d["value"] * 1.02 and 0 < pg["value_driver_staged"] <= d["value"] * 1.02
    assert d["p50_latency_ms_pageable"] >= d["p50_latency_ms"] * 0.9
    rs = d["roofline_step"]
    tot = rs["canonical_fq_mul_per_proof"]
    assert tot["total"] == tot["bucket_additions"] + tot["per_window_bucket_reduction"] + tot["ntt"] + tot["r1cs_and_join"]
    per_gpu = d["value"] / d["n_gpus"]
    assert rs["achieved"] == pytest.approx(tot["total"] * per_gpu / 1e9, rel=1e-9)
    assert rs["frac"] == pytest.approx(rs["achieved"] / rs["peak"], rel=1e-9) and 0.5 < rs["frac_without_reduction_term"] < 1
    assert "traffic_source" in d["roofline"] and ("modes" in d or "modes" in d["config"])
    if "extras" in d:
        ex = d["extras"]
        c2, c4 = ex["config2_batch"], ex["config4_split_msm"]
        assert c2["proofs"] == 1024 and c2["scaling"] == "strong" and c2["n_gpus"] == d["n_gpus"]
        assert c2["proofs_per_s"] == pytest.approx(c2["proofs"] / c2["seconds"], rel=1e-9)
        assert c4["n_gpus"] == d["n_gpus"] and c4["points_per_gpu"] * d["n_gpus"] >= 1 << 24
        assert 0 < c4["kernel_ms_max_over_ranks"] <= c4["ms"]


def test_dump_outputs_hold_the_proofs_exactly(tmp_path):
    """bench.py --dump-outputs: the float64 limb arrays give back every byte of every proof, in order."""
    import random

    import numpy as np

    import bench
    rng = random.Random(3)
    proofs = [bytes(rng.randrange(256) for _ in range(256)) for _ in range(3)]
    bench.dump_proofs(str(tmp_path), proofs)
    a, b, c = (np.load(tmp_path / (n + ".npy")) for n in ("pi_a", "pi_b", "pi_c"))
    assert a.dtype == b.dtype == c.dtype == np.float64
    assert a.shape == c.shape == (3, 2, 8) and b.shape == (3, 2, 2, 8)
    limbs = np.concatenate([x.reshape(3, -1) for x in (a, b, c)], axis=1)
    assert [row.astype("<u4").tobytes() for row in limbs] == proofs


def test_round2_reference_arm_has_the_same_config():
    ref = os.path.join(ROOT, "profiles", "r02_ref_n1.json")
    main = os.path.join(ROOT, "profiles", "r02_bench_default.json")
    if not (os.path.exists(ref) and os.path.exists(main)):
        pytest.skip("round-2 records not committed yet")
    r, m = json.load(open(ref)), json.load(open(main))
    assert r["config"] == {k: v for k, v in m["config"].items() if k != "modes"}
    assert r["impl"] == "reference" and r["metric"] == m["metric"] and r["unit"] == m["unit"]
    assert r["cpu_baseline"]["kind"] == "port" and r["e2e"]["value"] == r["value"]
