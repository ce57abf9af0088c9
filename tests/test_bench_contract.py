"""CPU-only checks of bench.py's output contract: the reference arm runs here (oracle on the host cores) and its JSON
line carries every key the driver reads; the CUDA arm must refuse to run without a GPU (no CPU fallback)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(*args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                          cwd=ROOT, env=e, timeout=600)


def test_reference_arm_json_line():
    r = run_bench("--impl", "reference", "--steps", "2", "--warmup", "1", "--n", "50000")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1  # ONE JSON line
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "point2point_linearized_residuals_per_sec" and d["unit"] == "Gres/s"
    assert d["higher_is_better"] is True and d["vs_baseline"] is None and d["data"] == "synthetic"
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["steps"] == 2 and d["n_gpus"] == 1
    assert set(d["cpu_baseline"]) >= {"value", "unit", "cores", "kind", "sample"} and d["cpu_baseline"]["kind"] == "port"
    assert d["cpu_baseline"]["value"] == d["value"] and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"] == {"value": d["value"], "unit": "Gres/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]
    # same workload keys as the GPU arm prints, W warm-up and K timed steps as requested, the whole --n per step
    sys.path.insert(0, ROOT)
    import bench
    assert d["config"] == bench.workload_config(50000, 50000) and d["warmup"] == 1 and d["cpu_sample_per_step"] == 50000


def test_reference_arm_other_ranks_stay_silent():
    r = run_bench("--impl", "reference", "--steps", "1", "--warmup", "0", "--n", "20000", "--gpus", "2",
                  env={"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_reference_arm_dump_outputs(tmp_path):
    """--dump-outputs writes the last timed step's H, b and sum r^T r; the seeded inputs make two runs agree."""
    import numpy as np
    dumps = []
    for k in range(2):
        d = tmp_path / f"run{k}"
        r = run_bench("--impl", "reference", "--steps", "2", "--warmup", "0", "--n", "30000", "--dump-outputs", str(d))
        assert r.returncode == 0, r.stderr[-2000:]
        line = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][0])
        assert sorted(os.listdir(d)) == ["H.npy", "b.npy", "sum_rtr.npy"]
        out = {name: np.load(d / f"{name}.npy") for name in ("H", "b", "sum_rtr")}
        assert out["H"].shape == (6, 6) and out["b"].shape == (6,) and out["sum_rtr"].shape == ()
        assert all(v.dtype == np.float64 for v in out.values())
        assert out["H"][0, 0] == line["check"]["H00"] and out["b"][0] == line["check"]["b0"]
        assert float(out["sum_rtr"]) == line["check"]["sum_rtr"]
        dumps.append(out)
    assert all(np.array_equal(dumps[0][k], dumps[1][k]) for k in dumps[0])


def test_steps_must_be_positive():
    r = run_bench("--impl", "reference", "--steps", "0", "--n", "1000")
    assert r.returncode != 0 and "--steps" in r.stderr


@pytest.mark.gpu
def test_cuda_arm_dump_outputs(tmp_path):
    """The CUDA arm's dump is the result of the timed pass: the same rows linearized again give the same H, b, sum."""
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    from moptimizer_0_b200 import capi
    from tests.common import rel_err
    n, steps = 1_000_003, 7
    r = run_bench("--steps", str(steps), "--warmup", "1", "--prewarm-steps", "10", "--n", str(n), "--no-cpu-baseline",
                  "--no-e2e", "--no-configs", "--no-peaks", "--no-lm", "--dump-outputs", str(tmp_path))
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][0])
    assert line["steps"] == steps and line["gpu_launches"] == steps
    H, b, s = (np.load(tmp_path / f"{name}.npy") for name in ("H", "b", "sum_rtr"))
    ctx = capi.Context(0)
    st = capi.Store(ctx, capi.MODEL_POINT2POINT, n, capi.F32)
    st.generate(seed=bench.SEED, gt=bench.X_GT, **bench.GEN)
    prob = capi.make_problem(capi.MODEL_POINT2POINT, capi.JAC_ANALYTICAL, capi.F32, loss=capi.LOSS_HUBER,
                             loss_param=bench.HUBER_K, variant=capi.P2P_EXACT)
    He, be, se = ctx.linearize(st, prob, np.zeros(6))
    st.close()
    ctx.close()
    assert rel_err(H, He) < 1e-12 and rel_err(b, be) < 1e-12 and abs(float(s) - se) <= 1e-12 * se


def test_cuda_arm_refuses_to_run_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    r = run_bench("--steps", "1")
    assert r.returncode != 0 and "no CPU fallback" in (r.stderr + r.stdout)


def test_committed_bench_lines_carry_the_contract_keys():
    """The round's recorded N = 1 line (profiles/) has the roofline / cpu_baseline / e2e / clocks objects."""
    path = os.path.join(ROOT, "profiles", "r1_bench_n1_final.json")
    d = json.loads(open(path).read().strip().splitlines()[-1])
    assert set(d["roofline"]) >= {"bound", "achieved", "peak", "unit", "frac", "traffic"} and d["roofline"]["bound"] == "hbm"
    assert abs(d["roofline"]["frac"] - d["roofline"]["achieved"] / d["roofline"]["peak"]) < 1e-12
    assert set(d["e2e"]) >= {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"}
    assert d["e2e"]["h2d_bytes_per_step"] == 24 * d["config"]["n_per_gpu"] and d["e2e"]["matches_resident"] is True
    assert set(d["clocks"]) >= {"sm_mhz", "sm_max_mhz", "reasons"} and d["gpu_launches"] == d["steps"]
    assert d["cpu_baseline"]["kind"] == "port" and d["dtype"] == "f32" and d["scaling"] == "weak"
    # algorithmic bytes vs measured DRAM traffic of the same launch: no wasted re-reads
    assert 1.0 <= d["roofline"]["traffic"] / d["roofline"]["algorithmic_bytes_per_launch"] < 1.01


def test_committed_round2_lines_cover_every_baseline_config():
    """Round 2's recorded lines: every BASELINE configuration with a roofline, measured ceilings, the same workload
    keys in both arms, and — at N > 1 — the exchanged result bit-identical to the single-GPU sums."""
    sys.path.insert(0, ROOT)
    import bench
    d = json.loads(open(os.path.join(ROOT, "profiles", "r2_bench_n1_allconfigs.json")).read().strip().splitlines()[-1])
    assert d["roofline"]["bound"] == "hbm" and d["roofline"]["frac"] > 1.0 and d["e2e"]["matches_resident"] is True
    assert set(d["configs"]) >= {"curve_10M_central", "camera_50M_P6_central", "camera_50M_P15_central", "fachada_lm"}
    for key in ("curve_10M_central", "camera_50M_P6_central", "camera_50M_P15_central"):
        c = d["configs"][key]
        assert c["ms"] > 0 and c["Gres_per_s"] > 0 and c["roofline"]["bound"] == "fp32_issue" and c["roofline"]["hbm_frac"] > 0
    assert d["configs"]["fachada_lm"]["status"] == "CONVERGED" and d["configs"]["fachada_lm"]["sequence"] == "AAAAA"
    assert d["peaks"]["fp32_fma_tflops"] > 10 and d["peaks"]["hbm_read_gbs"] > 1000 and d["e2e"]["frac_of_h2d_ceiling"] > 0.9
    ref = json.loads(open(os.path.join(ROOT, "profiles", "r2_bench_reference_arm.json")).read().strip().splitlines()[-1])
    assert ref["config"] == d["config"] == bench.workload_config(100_000_000, 100_000_000)
    assert abs(ref["check"]["sum_rtr"] - d["check"]["sum_rtr"]) <= 1e-8 * d["check"]["sum_rtr"]   # same 100 M rows
    for name in ("r2_bench_n2.json", "r2_bench_n8.json"):
        m = json.loads(open(os.path.join(ROOT, "profiles", name)).read().strip().splitlines()[-1])
        v = m["check"]["vs_single_gpu"]
        assert v["bit_identical"] is True and v["H_rel"] == 0.0 and v["b_rel"] == 0.0 and v["sum_rel"] == 0.0
        assert m["configs"]["p2p_1B_strong"]["n_total"] == 1_000_000_000 and m["lm"]["status"] == "SMALL_DELTA"
    # the issue-slot rooflines use instruction counts from a committed ncu capture of the same kernels
    counts = json.loads(open(os.path.join(ROOT, "profiles", "kernel_inst_counts.json")).read())
    assert counts["p2p_gen2_f32"]["issue_active_pct"] < 45 and counts["camera15_central_f32"]["tensor_pipe_pct"] > 0
    assert 1.0 <= counts["p2p_gen2_f32"]["dram_bytes_per_launch"] / 2.4e9 < 1.01
