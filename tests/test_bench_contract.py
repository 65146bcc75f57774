"""bench.py's output contract: the reference arm runs here (it is CPU work), our arm's line is checked on the committed
B200 result.  Keeps the keys the driver and the judge read from drifting."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches", "cpu_baseline"}


def _bench(*argv, env_extra=None):
    env = dict(os.environ, **(env_extra or {}))
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *argv], capture_output=True, text=True, env=env, timeout=600)


def _run(env_extra):
    return _bench("--impl", "reference", "--steps", "1", "--warmup", "0", "--cpu-pairs", "2", env_extra=env_extra)


def _line(r):
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, r.stdout[-400:]
    return json.loads(lines[0])


def test_reference_arm_prints_one_contract_line():
    r = _run({})
    assert r.returncode == 0, r.stderr[-400:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert BASE_KEYS <= set(d) and d["impl"] == "reference"
    assert d["metric"].startswith("frame-pairs/sec") and d["unit"] == "pairs/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["vs_baseline"] is None and d["data"] == "synthetic" and d["scaling"] == "weak"
    assert d["config"]["workload"].startswith("c3:")                    # headline: BASELINE.json configs[2], the GEMM of the metric
    assert d["extra"]["c2"]["config"]["workload"].startswith("c2:")     # BASELINE.json configs[1] rides along, complete line
    assert BASE_KEYS <= set(d["extra"]["c2"])
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0


def test_reference_arm_is_silent_on_other_ranks():
    r = _run({"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"})
    assert r.returncode == 0 and not [l for l in r.stdout.splitlines() if l.startswith("{")]


def test_bad_arguments_are_refused_before_any_work():
    for argv in (("--steps", "0"), ("--impl", "reference", "--dump-outputs", "unused")):
        r = _bench(*argv)
        assert r.returncode == 2 and "error" in r.stderr, (argv, r.stderr[-400:])


@pytest.mark.gpu
def test_dump_outputs_are_the_last_step_and_repeat_run_to_run(tmp_path):
    """--dump-outputs writes the timed path's outputs of its last step; two runs with the same arguments write the same
    arrays, and --steps sets the number of timed steps (one pass per step here: launches scale with it)."""
    small = ("--workload", "c1", "--pairs", "8", "--passes", "1", "--warmup", "1", "--no-cpu", "--no-api-rate",
             "--no-variants", "--allow-no-clocks")
    lines, dumps = [], []
    for k, steps in enumerate((2, 2, 1)):
        d = tmp_path / f"run{k}"
        r = _bench(*small, "--steps", str(steps), "--dump-outputs", str(d))
        assert r.returncode == 0, r.stderr[-800:]
        lines.append(_line(r))
        dumps.append({p.name: np.load(p) for p in sorted(d.iterdir())})
    names = {f"c1_{f}.npy" for f in ("T_rel", "rt", "n_matches", "n_corr", "n_inl", "status")}
    assert set(dumps[0]) == names
    assert dumps[0]["c1_T_rel.npy"].shape == (8, 4, 4) and all(a.dtype == np.float64 for a in dumps[0].values())
    assert (dumps[0]["c1_status.npy"] == 0).mean() >= 0.5 and (dumps[0]["c1_n_inl.npy"] > 20).any()
    for dump in dumps[1:]:
        assert set(dump) == names and all(np.array_equal(dumps[0][n], dump[n]) for n in names)
    assert [l["steps"] for l in lines] == [2, 2, 1] and all(l["config"]["passes_per_step"] == 1 for l in lines)
    assert lines[0]["gpu_launches"] == lines[1]["gpu_launches"] == 2 * lines[2]["gpu_launches"] > 0


def test_committed_b200_line_has_the_roofline_and_clock_keys():
    """The default line of this round as measured on a B200 (profiles/bench_default_r02j.json): the headline is workload c3 —
    the tcgen05 GEMM BASELINE.json's metric names — and the complete line of c2 rides in extra.c2."""
    d = json.loads(open(os.path.join(ROOT, "profiles", "bench_default_r02j.json")).read().strip().splitlines()[-1])
    for line, wl in ((d, "c3:"), (d["extra"]["c2"], "c2:")):
        assert BASE_KEYS <= set(line) and "impl" not in line
        assert line["n_gpus"] == 1 and line["warmup"] >= 3 and line["gpu_launches"] > 0
        assert line["config"]["workload"].startswith(wl) and "l2" in line["config"]
        assert line["config"]["timed_region_s"] >= 2.0 and line["e2e"]["timed_region_s"] >= 2.0
        roof = line["roofline"]
        assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(roof) and roof["bound"] in ("hbm", "tensor")
        assert abs(roof["frac"] - roof["achieved"] / roof["peak"]) < 1e-9
        e2e = line["e2e"]
        assert e2e["h2d_bytes_per_step"] > 0 and e2e["d2h_bytes_per_step"] > 0 and 0 < e2e["value"] < line["value"]
        assert e2e["equals_resident_bitwise"] is True and "precondition" in e2e
        clocks = line["clocks"]
        assert clocks["samples"] > 0 and clocks["sm_mhz"] and clocks["sm_max_mhz"]
        assert not set(clocks["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
        cb = line["cpu_baseline"]
        assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] > 0 and "pairs" in cb["sample"]
    roof = d["roofline"]
    assert "match_f32_tc_kernel" in roof["kernel"] and roof["bound"] == "tensor" and roof["unit"] == "TFLOP/s"
    assert 0.5 < roof["frac"] < 1.0 and roof["frac_of_cublas_tf32"] > 0.9                # tensor pipe rate, and cuBLAS TF32 of the same run
    assert 0.5 < d["extra"]["c2"]["roofline"]["binding_pipe"]["frac"] < 1.0                 # the POPC pipe bounds the Hamming kernel
