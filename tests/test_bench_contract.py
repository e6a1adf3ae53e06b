"""bench.py prints exactly ONE JSON line with the keys the driver reads.  CPU: the reference arm
(`--impl reference`, the oracle port on the host cores) on a short sample.  GPU: our arm on a reduced
ensemble (same code path as the headline run)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"}


def _run(args, timeout):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True,
                       timeout=timeout, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout[-2000:]
    return json.loads(lines[0])


@pytest.mark.timeout(300)
def test_reference_arm_line():
    d = _run(["--impl", "reference", "--steps", "1", "--warmup", "0", "--cpu-seconds", "1.0", "--ess-steps", "600"], 280)
    assert BASE_KEYS <= set(d) and d["impl"] == "reference"
    assert d["unit"] == "chain-steps/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["e2e"]["value"] == d["value"] == d["cpu_baseline"]["value"]
    assert "workload" in d["config"] and "model" not in d["config"]
    # ESS/s is half of BASELINE.json's metric: the CPU arm reports it too, with the cores it used
    assert d["cpu_baseline"]["ess_per_s"] > 0 and d["ess"]["cores"] == d["cpu_baseline"]["cores"] == d["cores"]
    py = d["cpu_baseline"]["python_reference"]
    assert py["rk4_plugin"]["chain_steps_per_s_per_core"] > 0 and "NOT on this box" in py["measured_in"]


def test_dump_outputs_are_float64_and_capped(tmp_path, monkeypatch):
    """--dump-outputs writes one float64 .npy per array; above the cap, the same seeded sample of chains every time."""
    import numpy as np
    import bench
    n = 1000
    state = {"theta": np.arange(2.0 * n).reshape(2, n), "n_accept": np.arange(n, dtype=np.int64)}
    bench.dump_outputs(str(tmp_path / "full"), state)
    assert np.array_equal(np.load(tmp_path / "full" / "n_accept.npy"), np.arange(n))
    assert sorted(p.name for p in (tmp_path / "full").iterdir()) == ["n_accept.npy", "theta.npy"]
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 8 * 1024)
    for out in ("a", "b"):
        bench.dump_outputs(str(tmp_path / out), state, "_rank1")
    files = {p.name: np.load(p) for p in (tmp_path / "a").iterdir()}
    assert set(files) == {"theta_rank1.npy", "n_accept_rank1.npy", "chain_index_rank1.npy"}
    assert all(a.dtype == np.float64 for a in files.values()) and sum(a.nbytes for a in files.values()) <= 8 * 1024
    keep = files["chain_index_rank1.npy"].astype(np.int64)
    assert len(keep) > 0 and np.array_equal(files["theta_rank1.npy"], state["theta"][:, keep])
    assert np.array_equal(keep, np.load(tmp_path / "b" / "chain_index_rank1.npy"))


@pytest.mark.gpu
@pytest.mark.timeout(300)
def test_b200_arm_dumps_the_same_outputs_for_the_same_arguments(tmp_path):
    """Two runs with the same arguments compute the same chain state, bit for bit: what --dump-outputs writes can
    compare two builds of the project."""
    import numpy as np
    args = ["--steps", "2", "--warmup", "3", "--chains", "8192", "--transitions", "10",
            "--no-ess", "--no-e2e", "--no-cpu", "--no-configs", "--dump-outputs"]
    for out in ("a", "b"):
        d = _run(args + [str(tmp_path / out)], 280)
        assert d["steps"] == 2
    names = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert names == ["logpost.npy", "n_accept.npy", "theta.npy", "w_m2.npy", "w_mean.npy"]
    for name in names:
        a, b = np.load(tmp_path / "a" / name), np.load(tmp_path / "b" / name)
        assert a.dtype == np.float64 and a.shape[-1] == 8192 and np.array_equal(a, b, equal_nan=True), name
    theta = np.load(tmp_path / "a" / "theta.npy")
    assert theta.shape == (2, 8192) and np.isfinite(theta).all()


@pytest.mark.gpu
@pytest.mark.timeout(300)
def test_b200_arm_line():
    d = _run(["--steps", "2", "--warmup", "3", "--chains", "8192", "--transitions", "10", "--ess-steps", "300",
              "--cpu-seconds", "0.5", "--no-configs"], 280)
    assert BASE_KEYS | {"roofline", "gpu_launches", "clocks", "ess"} <= set(d)
    assert d["n_gpus"] == 1 and d["dtype"] == "f64" and d["gpu_launches"] >= 2 and d["value"] > 1e6
    rf = d["roofline"]
    assert rf["bound"] == "fp64" and abs(rf["frac"] - rf["achieved"] / rf["peak"]) < 1e-9
    assert 0.0 < rf["rk4_loop"]["frac"] < 1.0 and rf["executed"]["fp64_instr_per_rk4_step"] == 20
    assert abs(rf["frac_executed"] - rf["frac"] * 40.0 / 58.0) < 1e-9 and rf["frac_of_bare_rk4_loop"] == rf["rk4_loop"]["frac"]
    assert rf["traffic"] is None and "no committed ncu capture" in rf["traffic_source"]       # no capture at 8,192 chains
    e = d["e2e"]
    assert e["h2d_bytes_per_step"] == 8192 * 2 * 8 and e["d2h_bytes_per_step"] > 0 and 0 < e["value"] <= 1.05 * d["value"]
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["value"] > 0 and d["cpu_baseline"]["ess_per_s"] > 0
    assert d["cpu_cores"] == d["cpu_baseline"]["cores"] and d["scaling"] == "weak"
    assert d["ess"]["tuned"]["sub_chain_length"] == 8 and d["ess"]["tuned"]["over_example"] > 0.0   # > 2 at the real sizes (short test chains pay the burn-in)
    for arm in ("pooled", "adaptive", "tuned"):
        assert d["ess"][arm]["ess_per_s"] > 0 and d["ess"][arm]["degenerate_chains"] == 0
        assert all(abs(x - 1.0) < 0.05 for x in d["ess"][arm]["diagnostics"]["split_rhat"])
    dg = d["ess"]["diagnostics"]
    assert dg["n_chains"] == 8192 and all(abs(x - 1.0) < 0.05 for x in dg["rhat"] + dg["split_rhat"])
    assert "sm_mhz" in d["clocks"] and "reasons" in d["clocks"]
