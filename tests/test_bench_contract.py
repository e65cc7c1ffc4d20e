"""bench.py contract checks: the reference arm runs on host cores only, the committed bench lines carry every key of
the result line, and (on a GPU) --dump-outputs writes what the last timed step computed."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_runs_on_cpu_and_prints_one_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1"],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    rec = json.loads(lines[0])
    assert rec["impl"] == "reference" and rec["metric"].startswith("EM link-updates/sec") and rec["unit"] == "link-updates/s"
    assert rec["higher_is_better"] is True and rec["value"] > 0 and rec["gpu_launches"] == 0
    assert rec["steps"] == 2 and rec["warmup"] == 1          # the arm does the warm-up and step counts it was asked for
    # oracle/_ref (the unmodified reference script) is there in the build container and wherever the tree travelled with it
    want = "reference" if os.path.exists(os.path.join(ROOT, "oracle", "_ref", "TrigenicInteractionPredictor.py")) else "port"
    assert rec["cpu_baseline"]["kind"] == want and rec["cpu_baseline"]["cores"] >= 1 and rec["cpu_baseline"]["value"] == rec["value"]
    assert rec["e2e"] == {"value": rec["value"], "unit": rec["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


import pytest


@pytest.mark.parametrize("name", ["r1_bench_line.json", "r2_bench_line.json"])
def test_committed_bench_line_has_the_contract_keys(name):
    with open(os.path.join(ROOT, "profiles", name)) as fh:
        rec = json.loads(fh.read().strip().splitlines()[-1])
    if name.startswith("r2"):
        assert rec["cpu_baseline"]["kind"] == "reference" and rec["config"]["shape"] == "kuzmin"
        assert rec["roofline"]["kernel_ms"] <= rec["ms_per_step"] and rec["roofline"]["binding"]["frac"] < 1.0
        for key in ("cfg4_strong", "cfg3_samples", "value_uniform", "value_kuzmin"):
            assert key in rec, key
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "clocks", "e2e", "gpu_launches", "roofline", "cpu_baseline"):
        assert key in rec, key
    assert rec["dtype"] == "f64" and rec["vs_baseline"] is None and "workload" in rec["config"]
    for key in ("bound", "achieved", "peak", "unit", "frac", "traffic"):
        assert key in rec["roofline"], key
    assert abs(rec["roofline"]["frac"] - rec["roofline"]["achieved"] / rec["roofline"]["peak"]) < 1e-9
    for key in ("value", "unit", "cores", "kind", "sample"):
        assert key in rec["cpu_baseline"], key
    for key in ("value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"):
        assert key in rec["e2e"], key
    assert rec["e2e"]["h2d_bytes_per_step"] > 0 and rec["e2e"]["value"] < rec["value"]
    assert rec["gpu_launches"] >= rec["steps"]


@pytest.mark.gpu
def test_dump_outputs_are_the_parameters_after_the_last_timed_step(tmp_path):
    """--dump-outputs writes theta and pr as the headline leaves them after its warm-up and exactly --steps timed
    iterations: the same as that many eager iterations of the engine on bench.py's seeded inputs."""
    import numpy as np
    import torch
    from trigenicinteractionpredictor_b200 import synth
    from trigenicinteractionpredictor_b200.engine import EMEngine
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "3",
                          "--skip", "cfg4,cfg3,fp32,k3,e2e,cpu", "--dump-outputs", str(tmp_path / "dump")],
                         capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    rec = json.loads(lines[0])
    assert rec["steps"] == 2 and rec["warmup"] == 3
    assert sorted(os.listdir(tmp_path / "dump")) == ["pr.npy", "theta.npy"]
    theta, pr = np.load(tmp_path / "dump" / "theta.npy"), np.load(tmp_path / "dump" / "pr.npy")
    assert theta.dtype == np.float64 and pr.dtype == np.float64
    # bench.py's headline inputs: P=6000, K=10, 800,000 Kuzmin-shaped links of seed 100, parameters of default_rng(0)
    P, K, dev = 6000, 10, torch.device("cuda", 0)
    g1, g2, g3, lab = synth.kuzmin_links_soa(P, 800_000, seed=100, device=dev)
    g1[:P] = torch.arange(P, dtype=torch.int32, device=dev)
    rng = np.random.default_rng(0)
    theta0 = rng.dirichlet(np.ones(K), size=P)
    pr0 = rng.random((K, K, K, 2))
    pr0 /= pr0.sum(axis=3, keepdims=True)
    eng = EMEngine(P, K, device=dev)
    eng.set_train_links(g1, g2, g3, 1 - lab, lab)
    eng.set_params(theta0, pr0)
    for _ in range(3 + 2):
        eng.em_iteration()
    th, p = eng.get_params()
    assert theta.shape == th.shape and pr.shape == p.shape
    np.testing.assert_allclose(theta, th, rtol=1e-11, atol=0)
    np.testing.assert_allclose(pr, p, rtol=1e-11, atol=0)
