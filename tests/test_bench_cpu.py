"""bench.py pieces that run without a GPU: the reference arm (CPU port of the path) and the learner's CPU baseline,
and the Q-network oracle's bf16-emulation mode (the checker of the tensor-core path)."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def test_reference_arm_prints_the_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    assert len(r.stdout.strip().splitlines()) == 1          # stdout carries the JSON line and nothing else
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "frames/s" and line["higher_is_better"] is True
    from oracle import ref_verbatim as rv
    kind = "reference" if rv.available() else "port"     # oracle/_ref staged by build(): the reference itself, verbatim
    assert line["value"] > 0 and line["cpu_baseline"]["kind"] == kind and line["cpu_baseline"]["cores"] >= 1
    assert line["cpu_baseline"]["c_port"]["kind"] == "port" and line["cpu_baseline"]["c_port"]["value"] > line["value"] * (1 if kind == "reference" else 0)
    assert "30 frames/s" in line["cpu_baseline"]["as_shipped"]
    assert line["e2e"] == {"value": line["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    import bench
    assert line["metric"] == bench.METRIC and line["config"]["workload"] == bench.WORKLOAD


def test_reference_arm_is_bounded_for_any_step_count():
    """each bench step is a bounded sample sized from K, so the driver's K (ours defaults to 2000) never makes the arm run long"""
    import time
    t0 = time.perf_counter()
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2000", "--warmup", "20",
                        "--reference-budget-s", "8"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    dt = time.perf_counter() - t0
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2000 and line["value"] > 0
    assert dt < 120, dt                     # 8 s of samples + interpreter / library start-up


def test_reference_arm_refuses_dump_outputs(tmp_path):
    """--dump-outputs writes the device path's outputs; the reference arm has none, so the combination is an error"""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                        "--dump-outputs", str(tmp_path / "out")], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 2 and "--dump-outputs" in r.stderr and r.stdout == ""
    assert not (tmp_path / "out").exists()


def test_learner_cpu_baseline_runs():
    import bench
    ups, n, dt = bench.cpu_port_updates_per_s(0.5)
    assert n >= 1 and ups > 0 and dt > 0


def test_oracle_bf16_emulation_is_close_to_exact_and_rounds_where_the_device_does():
    import torch
    from oracle import qnet_oracle as qo
    rng = np.random.default_rng(0)
    B = 4
    p = qo.init_params(512, False, seed=1) * np.float32(3.0)
    x = (rng.random((B, 5, 80, 80)) < 0.2).astype(np.uint8) * 255
    q, acts = qo.forward(torch.tensor(p.astype(np.float64)), x[:, 0:4], return_all=True)
    qe, acts_e = qo.forward(torch.tensor(p.astype(np.float64)), x[:, 0:4], return_all=True, emulate_bf16=True)
    assert np.abs((q - qe).numpy()).max() <= 2e-2 * np.abs(q.numpy()).max()
    for name in ("z1", "a2", "a3"):                      # stored activations are exactly bf16-representable
        t = acts_e[name]
        assert torch.equal(t, t.to(torch.float32).to(torch.bfloat16).to(torch.float64)), name
    a = rng.integers(0, 2, B).astype(np.uint8)
    r = np.array([0.1, 3.0, -3.0, 0.1], np.float32); term = (r == -3.0).astype(np.uint8)
    l0, g0, *_ = qo.loss_and_grads(1, p, p, x[:, 0:4], x[:, 1:5], a, r, term)
    l1, g1, *_ = qo.loss_and_grads(1, p, p, x[:, 0:4], x[:, 1:5], a, r, term, emulate_bf16=True)
    assert abs(l0 - l1) <= 5e-2 * abs(l0)
    assert np.linalg.norm(g1 - g0) <= 0.2 * np.linalg.norm(g0)


def test_reference_runs_verbatim_and_agrees_with_the_port():
    """oracle/_ref (staged by build() from the reference checkout, $FLAPPY_REFERENCE or /root/reference): the reference's env
    module on the pygame shim, its clock neutralised, gives the same rewards / terminals as the C port driven with the same
    gaps is checked in test_oracle_env; here: the staging is complete, the worker protocol works, and the reference's PER
    classes load and sample"""
    import pytest
    from oracle import ref_verbatim as rv
    if not rv.available():
        if not rv.stage():
            pytest.skip("no reference checkout ($FLAPPY_REFERENCE, default /root/reference) and oracle/_ref not staged")
    assert rv.available()
    segs = rv.env_segments(2, 12, 2)
    assert len(segs) == 2 and all(t > 0 for t in segs)
    SumTree, Memory = rv.load_per_classes()
    mem = Memory(64)
    for i in range(64):
        mem.store((i,))
    idx, batch, w = mem.sample(8)
    assert len(idx) == 8 and w.shape == (8, 1) and np.all(w > 0)
