"""bench.py prints ONE JSON line with the contract's keys.  CPU: the reference arm (host port) with a tiny budget.
GPU: our arm, short."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "e2e", "cpu_baseline"}


def _run(*args):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-800:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    return json.loads(lines[0])


def test_reference_arm_line():
    d = _run("--impl", "reference", "--steps", "1", "--warmup", "0", "--cpu-budget-s", "0.3", "--no-reference-cuda")
    assert BASE_KEYS <= set(d) and d["impl"] == "reference"
    assert d["metric"] == "fe_path_steps_per_s" and d["unit"] == "path-steps/s" and d["value"] > 1e6
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and "sample" in d["cpu_baseline"]
    # generator initialisation is timed separately and excluded from value (the span of the GPU arm's timed region)
    assert d["cpu_baseline"]["init_s"] > 0 and d["cpu_baseline"]["value_incl_init"] < d["cpu_baseline"]["value"] * 1.5
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_dump_outputs_over_64_mb_is_refused():
    """--dump-outputs writes at most 64 MB: a grid whose c4 arrays would exceed that is rejected before any work."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--dump-outputs", "unused", "--c4-points", "130"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 2 and "more than 64 MB" in r.stderr, r.stderr[-400:]


@pytest.mark.gpu
@pytest.mark.parametrize("method,metric",[("fe", "fe_path_steps_per_s"), ("em", "em_paths_per_s")])
def test_our_arm_line(method, metric, tmp_path):
    d = _run("--method", method, "--steps", "3", "--warmup", "3", "--log2-paths", "20", "--cpu-budget-s", "0.3", "--no-reference-cuda",
             "--no-sub-records", "--dump-outputs", str(tmp_path))
    assert BASE_KEYS | {"gpu_launches", "clocks", "roofline", "kernel"} <= set(d)
    assert d["metric"] == metric and d["n_gpus"] == 1 and d["gpu_launches"] == 3 and d["value"] > 0
    assert set(d["roofline"]) >= {"bound", "achieved", "peak", "unit", "frac", "traffic"}
    assert set(d["clocks"]) >= {"sm_mhz", "sm_max_mhz", "reasons"}
    assert d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] == 16
    assert abs(d["result"]["E[X]"] - 0.1197325) < 5 * d["result"]["std_error"] + 2e-4
    # --dump-outputs: the FP64 sums of the last timed step, the ones the line's result is derived from
    assert sorted(os.listdir(tmp_path)) == ["moments.npy"]
    m = np.load(tmp_path / "moments.npy")
    assert m.dtype == np.float64 and m.shape == (2,)
    assert m[0] / (1 << 20) == d["result"]["E[X]"]
    # ... and they are call warmup + steps = 6 of the seeded stream, not a warm-up step or an earlier one
    from nmch_b200 import engine as E
    with E.Engine(NTPB=512, NB=(1 << 20) // 512, N=1000, method=E.METHOD_FE if method == "fe" else E.METHOD_EM,
                  rng=E.RNG_PHILOX) as e:
        e.init(1234)
        calls = [e.compute() for _ in range(6)]
    last, before = np.array([calls[5].sum_payoff, calls[5].sum_payoff_sq]), np.array([calls[4].sum_payoff, calls[4].sum_payoff_sq])
    np.testing.assert_allclose(m, last, rtol=1e-12)
    assert np.abs(m - before).max() > 1e-6 * np.abs(before).max()


def test_reference_arm_uses_every_host_thread_under_torchrun_env():
    """torch.distributed.run exports OMP_NUM_THREADS=1; the CPU arm must still use the cores the process may run on
    (round 1: SCALE's reference arm ran on one thread at N >= 2 and the driver's ratio was void)."""
    env = dict(os.environ, OMP_NUM_THREADS="1", RANK="0", WORLD_SIZE="2", LOCAL_RANK="0")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                        "--warmup", "0", "--cpu-budget-s", "0.3", "--no-reference-cuda"], capture_output=True, text=True,
                       timeout=600, env=env)
    assert r.returncode == 0, r.stderr[-800:]
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert d["cpu_baseline"]["cores"] == len(os.sched_getaffinity(0)) and d["n_gpus"] == 2
    # a rank other than 0 prints nothing and exits 0
    env["RANK"] = "1"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                        "--warmup", "0"], capture_output=True, text=True, timeout=600, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


@pytest.mark.gpu
def test_sub_records_em_and_c5_strong(tmp_path):
    d = _run("--steps", "3", "--warmup", "3", "--log2-paths", "20", "--c5-log2-paths", "22", "--c4-log2-paths", "14", "--c4-points", "6",
             "--no-cpu-baseline", "--no-reference-cuda", "--dump-outputs", str(tmp_path))
    assert d["metric"] == "fe_path_steps_per_s" and d["gpu_launches"] == 3
    em = d["em"]
    assert em["metric"] == "em_paths_per_s" and em["unit"] == "paths/s" and em["value"] > 0 and em["gpu_launches"] == em["steps"]
    assert set(em["roofline"]) >= {"bound", "achieved", "peak", "frac", "traffic", "traffic_source", "mix_bound_frac"}
    assert abs(em["result"]["E[X]"] - 0.1197325) < 5 * em["result"]["std_error"] + 2e-4
    assert em["e2e"]["d2h_bytes_per_step"] == 16
    c5 = d["c5_strong"]
    assert c5["scaling"] == "strong" and c5["global_paths"] == 1 << 22 and c5["steps"] == 3
    for m, u in (("fe", "path-steps/s"), ("em", "paths/s")):
        assert c5[m]["unit"] == u and c5[m]["value"] > 0 and c5[m]["gpu_launches"] == 3
        assert abs(c5[m]["result"]["E[X]"] - 0.1197325) < 5 * c5[m]["result"]["std_error"] + 2e-4
    assert d["roofline"]["traffic_source"].startswith("static")
    assert d["other_floor"]["floor"] == "plus" and d["other_floor"]["value"] > 0
    c4 = d["c4_sweep"]
    for m in ("fe", "em"):
        assert c4[m]["gpu_launches"] == 1 and c4[m]["all_finite"] and c4[m]["points"] == 200 and c4[m]["launch_ms"] > 0
    # --dump-outputs: one file per timed path
    assert sorted(os.listdir(tmp_path)) == sorted(f"{n}.npy" for n in ("moments", "em_moments", "c5_fe_moments", "c5_em_moments",
                                                                          "c4_fe_moments", "c4_em_moments"))
    assert np.load(tmp_path / "em_moments.npy")[0] / (1 << 22) == em["result"]["E[X]"]
    assert np.load(tmp_path / "c4_fe_moments.npy").shape == (200, 2)


@pytest.mark.gpu
def test_other_floor_record_carries_the_reference_build_with_the_plus_floor():
    """configs[1] names both floors; the (.)+ side of the reference is its CUDA build with the floor token changed while
    compiling (oracle/_ref/nmch_ref_harness_plus).  Same seed, same calls: 1e-5 on price and variance."""
    if not os.path.exists(os.path.join(ROOT, "oracle", "_ref", "nmch_ref_harness_plus")):
        pytest.skip("oracle/_ref/nmch_ref_harness_plus not shipped")
    d = _run("--steps", "3", "--warmup", "3", "--log2-paths", "18", "--c5-log2-paths", "20", "--c4-log2-paths", "12", "--c4-points", "4",
             "--no-cpu-baseline")
    ref = d["other_floor"]["reference_cuda"]
    for rng, tags in (("xorwow", ("ours_same_draws", "ours_same_stream_fast")), ("philox", ("ours_same_draws", "ours_native_same_words"))):
        assert ref[rng]["exec_ms"] > 0
        for tag in tags:
            assert ref[rng][tag]["max_rel_diff_E"] < 1e-5 and ref[rng][tag]["max_rel_diff_var"] < 1e-5, (rng, tag, ref[rng][tag])
