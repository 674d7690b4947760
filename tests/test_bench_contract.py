"""bench.py contract checks that need no GPU: the reference arm (CPU oracle port on the host cores) prints
exactly ONE JSON line on stdout with the keys the driver reads."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                        "--warmup", "1", "--ref-states", "256"], stdout=subprocess.PIPE, stderr=subprocess.PIPE,
                       text=True, cwd=ROOT, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["scaling"] == "weak"
    assert d["metric"].startswith("fwd+inv dynamics evals/s") and d["unit"] and d["value"] > 0
    assert d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] >= 3 and d["dtype"] == "f64"
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]


def test_bench_refuses_to_run_the_product_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        return
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1"],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, cwd=ROOT, timeout=600)
    assert r.returncode != 0 and not r.stdout.strip()   # no CPU fallback, no fake JSON line


def test_dump_sample_is_fixed_and_bounded():
    sys.path.insert(0, ROOT)
    from bench import DUMP_BYTES, dump_rows
    assert np.array_equal(dump_rows(1000, 48), np.arange(1000))
    rows = dump_rows(1 << 20, 48)
    assert 0 < len(rows) * 48 * 8 <= DUMP_BYTES and np.all(np.diff(rows) > 0) and rows[-1] < 1 << 20
    assert np.array_equal(rows, dump_rows(1 << 20, 48))


def test_reference_arm_dumps_the_outputs_of_its_last_step(oracle, tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2",
                        "--warmup", "1", "--ref-states", "256", "--dump-outputs", str(tmp_path)],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, cwd=ROOT, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads(r.stdout)["steps"] == 2
    assert sorted(os.listdir(tmp_path)) == ["tau_back.npy", "ydd.npy"]
    ydd, tau_back = np.load(tmp_path / "ydd.npy"), np.load(tmp_path / "tau_back.npy")
    assert ydd.dtype == np.float64 and ydd.shape == tau_back.shape == (256, 24)
    o = oracle.OracleModel("tello_with_arms")
    q, yd, tau = o.generate_states(256)
    ydd_o, tau_back_o = o.forward_dynamics(q, yd, tau), o.inverse_dynamics(q, yd, ydd)
    assert np.abs(ydd - ydd_o).max() <= 1e-12 * np.abs(ydd_o).max()
    assert np.abs(tau_back - tau_back_o).max() <= 1e-12 * np.abs(tau_back_o).max()


@pytest.mark.gpu
def test_gpu_bench_dumps_the_outputs_of_its_last_step(grbda, oracle, tmp_path):
    from test_gpu_parity import TOL64, relrows
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1",
                        "--batch", "4096", "--no-extras", "--no-e2e", "--no-cpu-baseline",
                        "--dump-outputs", str(tmp_path)],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, cwd=ROOT, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads(r.stdout)["steps"] == 2
    ydd, tau_back = np.load(tmp_path / "ydd.npy"), np.load(tmp_path / "tau_back.npy")
    assert ydd.dtype == np.float64 and ydd.shape == tau_back.shape == (4096, 24)
    # the dump is what the timed path computed: the same kernels on the same (device-generated) states, bit for bit
    m = grbda.ClusterTreeModel.from_robot("tello_with_arms")
    q, yd, tau, _ = m.generateStates(4096)
    ydd_m = m.forwardDynamics(q, yd, tau)
    assert np.array_equal(ydd, ydd_m.cpu().numpy())
    assert np.array_equal(tau_back, m.inverseDynamics(q, yd, ydd_m).cpu().numpy())
    # and forward dynamics agrees with the oracle (inverse dynamics of these accelerations is not compared with
    # the oracle: on ill-conditioned states tau = H ydd + C cancels large terms, so two correct implementations
    # differ by more than TOL64 of |tau|; test_gpu_parity checks inverse dynamics on accelerations in [-1, 1])
    n = 256
    qn, ydn, taun = q[:n].cpu().numpy(), yd[:n].cpu().numpy(), tau[:n].cpu().numpy()
    assert relrows(ydd[:n], oracle.OracleModel("tello_with_arms").forward_dynamics(qn, ydn, taun)) < TOL64
