"""bench.py's engine arms executed end to end on the CPU emulator with the torch.cuda calls stubbed: a dry run of the HOST logic of the
bench (workload set-up, graph / e2e / per-kernel-timing loops, the JSON line's keys), at shrunken sizes.  Numbers are meaningless here;
the point is that a bench workload added without a GPU at hand does not fail on its first GPU visit for a host-side reason."""
import json
import os
import sys
import time
import types

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class _Event(object):
    def __init__(self, enable_timing=False):
        self.t = 0.0

    def record(self, stream=None):
        self.t = time.perf_counter()

    def elapsed_time(self, other):
        return max((other.t - self.t) * 1e3, 1e-3)

    def synchronize(self):
        pass


class _Stream(object):
    cuda_stream = 0

    def synchronize(self):
        pass

    def wait_stream(self, s):
        pass


@pytest.fixture()
def bench_mod(emu_engine, monkeypatch):
    sys.path.insert(0, ROOT)
    import bench
    monkeypatch.setattr(torch.cuda, "set_device", lambda *a, **k: None)
    monkeypatch.setattr(torch.cuda, "synchronize", lambda *a, **k: None)
    monkeypatch.setattr(torch.cuda, "Event", _Event)
    monkeypatch.setattr(torch.cuda, "current_stream", lambda *a, **k: _Stream())
    lines = []
    monkeypatch.setattr(bench, "emit", lambda line: lines.append(json.loads(json.dumps(line))))
    monkeypatch.setattr(bench.ClockSampler, "run", lambda self: None)
    for k, v in dict(PROFILE_REPS=1, PROFILE_INNER=2, E2E_MIN_STEPS=2, CPU_STEPS=2, E2E_WARM=1).items():
        monkeypatch.setattr(bench, k, v)
    bench._lines = lines
    threads = torch.get_num_threads()
    yield bench
    torch.set_num_threads(threads)          # the bench arms pin torch's thread count (1 for the engine arm, 8 for the CPU arms)


CONTRACT = ["metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config",
            "e2e", "gpu_launches", "roofline", "cpu_baseline", "clocks"]


def _dumped(d):
    return {p.stem: np.load(p) for p in d.glob("*.npy")}


def test_mlp_workload_dry_run(bench_mod, monkeypatch, tmp_path):
    bench = bench_mod
    monkeypatch.setitem(bench.MLP_WORKLOADS, "mqmix_mpe_spread", (3, 18, 5, 54, 24, 600))
    monkeypatch.setattr(bench, "mlp_best_threads", lambda *a: 1)
    args = types.SimpleNamespace(workload="mqmix_mpe_spread", impl="b200", gpus=1, steps=3, warmup=3, buffer=5000, quick=False, opt=[],
                                 dump_outputs=str(tmp_path))
    bench.run_mlp(args)
    out = _dumped(tmp_path)
    assert set(out) == {"loss", "grad_norm", "Q_tot", "sample_indices", "params", "target_params"} and out["sample_indices"].shape == (24,)
    line = bench._lines[-1]
    for k in CONTRACT:
        assert k in line, k
    assert line["config"]["workload"] == "mqmix_mpe_spread" and line["config"]["batch_transitions"] == 24
    assert line["gpu_launches"] > 0        # (kernels_per_step counts graph nodes: 0 on the emulator)
    assert set(line["e2e"]) >= {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} and line["e2e"]["h2d_bytes_per_step"] > 0
    assert line["roofline"]["kernel"] in line["kernels"] and line["roofline"]["frac"] is not None
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["value"] > 0
    args.quick = True
    bench.run_mlp(args)
    assert bench._lines[-1]["quick"] is True


@pytest.mark.parametrize("opts", [{}, {"wgrad_tc": 2}], ids=["default", "tc_backward"])
@pytest.mark.parametrize("workload,shape", [("qmix_mpe_spread", (3, 18, 5, 54, 5, 4, False))])
def test_recurrent_workload_dry_run(bench_mod, monkeypatch, emu_engine, workload, shape, opts):
    """The default bench arm (run_engine) at shrunken shapes: the MPE workload (no availability masks, reward normalisation)."""
    bench = bench_mod
    monkeypatch.setitem(bench.WORKLOADS, workload, shape)
    monkeypatch.setattr(bench, "best_cpu_threads", lambda *a, **k: 1)
    monkeypatch.setattr(torch.Tensor, "pin_memory", lambda self, *a, **k: self)

    def eager_gpu_baseline_fails(*a, **k):          # as it does without a CUDA device; on a GPU host it would run with the stubs above
        raise RuntimeError("no CUDA device")
    monkeypatch.setattr(bench, "torch_eager_gpu_steps_per_s", eager_gpu_baseline_fails)
    args = types.SimpleNamespace(workload=workload, impl="b200", gpus=1, steps=3, warmup=3, buffer=48, quick=False, opt=["%s=%d" % kv for kv in opts.items()],
                                 dump_outputs=None)
    for k, v in opts.items():
        emu_engine.lib().mx_set_option(k.encode(), v)
    try:
        bench.run_engine(args)
    finally:
        for k in opts:
            emu_engine.lib().mx_set_option(k.encode(), -1 if k == "wgrad_tc" else 0)
    line = bench._lines[-1]
    if opts.get("wgrad_tc") == 2:
        assert "k_wgrad_tc" in line["kernels"] and "k_front_bwd_tc" in line["kernels"] and "k_front_bwd" not in line["kernels"]
    for k in CONTRACT:
        assert k in line, k
    assert line["config"]["workload"] == workload
    assert line["gpu_launches"] > 0 and line["e2e"]["h2d_bytes_per_step"] > 0 and line["e2e"]["lagged_read_value"] > 0
    assert line["roofline"]["kernel"] in line["kernels"]
    assert line["torch_eager_gpu_baseline"]["value"] is None          # the secondary baseline failed: it is skipped, the line survives


def test_dump_outputs_repeat_and_follow_the_step_count(bench_mod, monkeypatch, emu_engine, tmp_path):
    """--dump-outputs on the default arm: float32 / float64 arrays of the last timed step, identical in two runs with the same arguments,
    different after one more timed step."""
    bench = bench_mod
    monkeypatch.setitem(bench.WORKLOADS, "qmix_mpe_spread", (3, 18, 5, 54, 5, 4, False))
    runs = []
    for k, steps in enumerate((3, 3, 4)):
        args = types.SimpleNamespace(workload="qmix_mpe_spread", impl="b200", gpus=1, steps=steps, warmup=3, buffer=48, quick=True, opt=[],
                                     dump_outputs=str(tmp_path / str(k)))
        bench.run_engine(args)
        runs.append(_dumped(tmp_path / str(k)))
    assert set(runs[0]) == {"loss", "grad_norm", "Q_tot", "sample_indices", "params", "target_params"}
    for name, a in runs[0].items():
        assert a.dtype in (np.float32, np.float64) and np.array_equal(a, runs[1][name]), name
    assert not np.array_equal(runs[0]["params"], runs[2]["params"])


@pytest.mark.parametrize("workload,shape", [("rmatd3_spread", (2, 6, 2, 8, 4, 4, True, False)), ("rmaddpg_spread_disc", (2, 6, 3, 8, 4, 4, False, True))])
def test_maddpg_workload_dry_run(bench_mod, monkeypatch, emu_engine, workload, shape, tmp_path):
    """The R-MADDPG / R-MATD3 bench arm (run_maddpg) at shrunken shapes: Box + TD3 target noise, Discrete + Gumbel noise.  The engine side
    takes its configuration from the package (factory.MaddpgLearnerConfig); the oracle is imported for the CPU baseline only."""
    bench = bench_mod
    monkeypatch.setitem(bench.MADDPG_WORKLOADS, workload, shape)
    monkeypatch.setattr(torch.Tensor, "pin_memory", lambda self, *a, **k: self)
    args = types.SimpleNamespace(workload=workload, impl="b200", gpus=1, steps=3, warmup=3, buffer=48, quick=False, opt=[], dump_outputs=str(tmp_path))
    bench.run_maddpg(args)
    out = _dumped(tmp_path)
    assert {"critic_loss", "critic_grad_norm", "sample_indices", "actor_params", "target_actor_params", "critic_params", "target_critic_params"} <= set(out)
    line = bench._lines[-1]
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "config", "e2e", "gpu_launches", "cpu_baseline"):
        assert k in line, k
    assert line["config"]["workload"] == workload and line["gpu_launches"] > 0
