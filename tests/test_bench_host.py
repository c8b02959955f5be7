"""Host-side checks of bench.py that need no GPU: the reference arm's JSON line (the contract the driver parses), its
behaviour under torchrun ranks, and the workload helpers shared by both arms."""
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
import odecol  # noqa: E402

TINY = ["--impl", "reference", "--steps", "1", "--warmup", "0", "--cpu-trials", "4", "--cpu-time-points", "4", "--columns", "2"]


def _run(extra_env=None):
    env = dict(os.environ, **(extra_env or {}))
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *TINY], env=env, capture_output=True, text=True, timeout=300)


def test_reference_arm_prints_the_contract_line():
    r = _run()
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == bench.METRIC and d["unit"] == bench.UNIT
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1 and d["vs_baseline"] is None
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["dtype"] == "f32" and d["data"] == "synthetic"
    assert "workload" in d["config"] and "model" not in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "4 trials x 3 rk4 steps" in cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": bench.UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0


def test_reference_arm_is_silent_on_the_other_ranks():
    r = _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_dump_outputs_is_refused_where_it_is_not_implemented_and_steps_must_be_positive(tmp_path):
    for extra in (["--dump-outputs", str(tmp_path)], ["--steps", "0"]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *TINY, *extra], capture_output=True, text=True, timeout=300)
        assert r.returncode == 2 and r.stdout == "", r.stderr[-2000:]
    assert not any(tmp_path.iterdir())


def test_dump_outputs_writes_a_seeded_float32_sample_within_the_budget(tmp_path):
    import numpy as np
    from types import SimpleNamespace
    g = torch.Generator().manual_seed(0)
    net = SimpleNamespace(recurrent_weights=SimpleNamespace(grad=torch.randn(16, 16, generator=g)),
                          input_weights=SimpleNamespace(grad=torch.randn(16, 2, generator=g)))
    traj = torch.randn(50, 40, 6, generator=g)
    trials = torch.randperm(40, generator=torch.Generator().manual_seed(0))
    for budget, shape, every in ((10**9, (50, 32, 6), 1), (12000, (50, 10, 6), 1), (600, (25, 1, 6), 2)):
        out = tmp_path / str(budget)
        bench.dump_outputs(torch, str(out), torch.tensor(0.25), net, traj, budget=budget)
        d = {p.stem: np.load(p) for p in out.iterdir()}
        assert set(d) == {"loss", "grad_recurrent_weights", "grad_input_weights", "trajectory_sample"}
        assert all(v.dtype == np.float32 for v in d.values()) and d["loss"] == np.float32(0.25)
        assert np.array_equal(d["grad_recurrent_weights"], net.recurrent_weights.grad.numpy())
        assert np.array_equal(d["grad_input_weights"], net.input_weights.grad.numpy())
        assert d["trajectory_sample"].shape == shape and d["trajectory_sample"].nbytes <= budget
        want = traj[::every, trials[:shape[1]].sort().values].numpy()
        assert np.array_equal(d["trajectory_sample"], want)


def test_loss_components_select_v_and_a_of_the_readout_populations_and_f_on_request():
    sel = bench.loss_components(torch, 4)
    n = 32
    assert sel.tolist() == [0, 8, 16, 24, n, n + 8, n + 16, n + 24]
    self_f = bench.loss_components(torch, 4, with_f=True)
    assert self_f[:8].tolist() == sel.tolist() and self_f[8:].tolist() == [2 * n, 2 * n + 8, 2 * n + 16, 2 * n + 24]


def test_huber_on_rates_ignores_the_f_components_that_ride_along():
    g = torch.Generator().manual_seed(0)
    cols = 3
    y = torch.randn(5, 2, 3 * cols, generator=g)
    target = torch.full((1, 1, cols), 0.5)
    with_f = bench.huber_on_rates(torch, odecol, y, target, cols)
    without = bench.huber_on_rates(torch, odecol, y[:, :, :2 * cols].contiguous(), target, cols)
    assert torch.equal(with_f, without)
    rate = odecol.compute_firing_rate(y[:, :, :cols] - y[:, :, cols:2 * cols])
    assert torch.allclose(with_f, torch.nn.functional.smooth_l1_loss(rate, target.expand_as(rate), beta=1.0))


def test_stimulus_chunks_are_seeded_by_their_first_global_trial_and_the_probe_by_one_global_draw():
    a = bench.make_stimulus(torch, 4, 2, 60, 1e-4, 8, "cpu")
    b = bench.make_stimulus(torch, 4, 2, 60, 1e-4, 8, "cpu")
    c = bench.make_stimulus(torch, 4, 2, 60, 1e-4, 12, "cpu")
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]) and not torch.equal(a[1], c[1])
    assert a[1].shape[0] == 4 and a[1].shape[2] == 2 and float(a[1].max()) <= 30.0 and float(a[1].min()) >= 0.0
    whole = bench.probe_amplitudes(torch, 16, 2)
    lo, hi = odecol.distributed.shard_bounds(16, 1, 4)
    assert torch.equal(bench.probe_amplitudes(torch, 16, 2)[lo:hi], whole[4:8])
