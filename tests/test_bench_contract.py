"""bench.py contract: one JSON line with the keys the driver reads (metric/value/unit/n_gpus/steps/warmup/ms_per_step/..., `roofline`,
`cpu_baseline`, `e2e`, `clocks`, `gpu_launches`), for the engine arm (GPU) and the reference arm (CPU oracle, no GPU needed)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config"}


def run_bench(args, timeout=600):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, timeout=timeout, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, p.stdout
    return json.loads(lines[0])


def test_reference_arm_line():
    d = run_bench(["--impl", "reference", "--steps", "1", "--warmup", "1"])
    assert BASE_KEYS <= set(d) and d["impl"] == "reference" and d["metric"] == "candidates scored/sec" and d["unit"] == "candidates/s"
    assert d["value"] > 0 and d["higher_is_better"] is True and d["vs_baseline"] is None and "workload" in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "candidates_per_gpu_per_step" in d["config"]  # same key names as the engine arm's config
    cfg = d["configs"]  # the other BASELINE configs, CPU oracle on the same inputs
    assert cfg["C4_orbit_3x4x7_nnz"]["value"] > 0 and cfg["C4_orbit_3x4x7_G2"]["value"] > 0
    assert cfg["C3_sparsifier_4x4x4"]["search_1core"]["cores"] == 1 and cfg["C3_sparsifier_4x4x4"]["pipeline_c11"]["value"] > 0
    assert cfg["C5_mmcheck_32x32x32"]["all_correct"] and cfg["C5_mmcheck_32x32x32"]["unit"] == "samples/s"


def test_bad_arguments_are_refused():
    for args in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]):
        p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, timeout=120, cwd=ROOT)
        assert p.returncode == 2 and "error:" in p.stderr, (args, p.stderr)


@pytest.mark.gpu
def test_engine_arm_line(capi, tmp_path):
    d = run_bench(["--steps", "2", "--warmup", "3", "--batch-log2", "26", "--cpu-seconds", "1", "--dump-outputs", str(tmp_path)])
    assert BASE_KEYS <= set(d) and "impl" not in d
    assert d["n_gpus"] == 1 and d["steps"] == 2 and d["warmup"] == 3 and d["value"] > 1e9 and d["scaling"] == "weak"
    assert d["gpu_launches"] == 2 * 3  # sweep + final + slot-pack kernel per step
    r = d["roofline"]
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(r) and 0 < r["frac"] < 1 and r["peak"] > 1
    assert r["kernel"] == "orbit_sweep8x_kernel" and r["lanes_per_imad"] == 4  # frac is stated against lanes x the measured IMAD peak
    cfg = d["configs"]
    for key in ("C4_orbit_3x4x7_nnz", "C4_orbit_3x4x7_G2"):
        e = cfg[key]
        assert e["value"] > 1e8 and e["roofline"]["lanes_per_imad"] == 4 and 0 < e["roofline"]["frac"] < 1 and e["e2e"]["value"] > 0 and e["cpu_baseline"]["value"] > 0
    c3 = cfg["C3_sparsifier_4x4x4"]
    assert c3["search_c128"]["value"] > 1e10 and c3["search_c128"]["e2e"]["value"] > 1e10 and c3["pipeline_c11"]["consistent"]
    assert c3["pipeline_c11"]["value"] > 10 * c3["pipeline_c11"]["round1_value"] / 2
    c5 = cfg["C5_mmcheck_32x32x32"]
    assert c5["batch_4096"]["all_samples_agree"] and c5["batch_32"]["all_samples_agree"] and c5["batch_4096"]["value"] > 1e5
    assert cfg["C2_strong"]["scaling"] == "strong" and cfg["C2_strong"]["value"] > 1e9
    timed = [cfg["C2_strong"], cfg["C4_orbit_3x4x7_nnz"], cfg["C4_orbit_3x4x7_G2"], c3["search_c128"], c5["batch_4096"], c5["batch_32"]]
    assert [e["steps"] for e in timed] == [d["steps"]] * len(timed)  # --steps sets the timed steps of every path
    e = d["e2e"]
    assert e["value"] > 0 and e["h2d_bytes_per_step"] == 336 and e["d2h_bytes_per_step"] == 24
    c = d["clocks"]
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(c)
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["value"] > 0 and cb["cores"] >= 1
    assert d["best"]["score"] < 17.86  # the sweep improves on Winograd's growth factor (17.853)
    # --dump-outputs: what the last timed step of each path returned, float64
    import numpy as np
    out = {f[:-4]: np.load(tmp_path / f) for f in os.listdir(tmp_path)}
    assert sorted(out) == sorted(["C2", "C2_strong", "C4_orbit_3x4x7_nnz", "C4_orbit_3x4x7_G2", "C3_sparsifier_4x4x4_search_c128"] +
                                 [f"C5_mmcheck_32x32x32_batch_{b}_{x}" for b in (4096, 32) for x in ("verdict", "ok")])
    assert all(a.dtype == np.float64 for a in out.values()) and sum(a.nbytes for a in out.values()) <= 64 << 20
    score, nnz, nno, index = out["C2"]
    assert score >= d["best"]["score"] and nnz > 0 and (3 + 1) << 26 <= index < (3 + 2) << 26  # last step = the second timed one
    assert out["C2_strong"].tolist() == [cfg["C2_strong"]["best"][k] for k in ("score", "nnz", "nno", "index")]
    blocks = [[rl, cl, -1 if i is None else i] for rl, cl, i in cfg["C3_sparsifier_4x4x4"]["search_c128"]["best_per_block"]]
    assert out["C3_sparsifier_4x4x4_search_c128"].tolist() == blocks
    for b in (4096, 32):
        assert out[f"C5_mmcheck_32x32x32_batch_{b}_verdict"].tolist() == [0.0] and out[f"C5_mmcheck_32x32x32_batch_{b}_ok"].shape == (b,)
        assert out[f"C5_mmcheck_32x32x32_batch_{b}_ok"].all()
