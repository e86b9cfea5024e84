"""bench.py --dump-outputs: the actions of the last timed step, float32, within the size cap, identical for identical
arguments and equal to the last step of the same plan sequence run outside bench.py."""
import importlib.util
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench_module():
    spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def test_dump_outputs_keeps_a_fixed_row_sample_under_the_cap(tmp_path, monkeypatch):
    bench = _bench_module()
    monkeypatch.setattr(bench, "DUMP_BYTES", 2 * 1000 * 4 * 4)          # two arrays, 1000 rows of 4 floats each
    big = torch.arange(5000 * 4, dtype=torch.float64).reshape(5000, 4)
    small = torch.ones(10, 4, dtype=torch.float16)
    bench.dump_outputs(str(tmp_path / "a"), {"big": big, "small": small})
    bench.dump_outputs(str(tmp_path / "b"), {"big": big, "small": small})
    a, b = np.load(tmp_path / "a" / "big.npy"), np.load(tmp_path / "b" / "big.npy")
    assert a.dtype == np.float32 and a.shape == (1000, 4) and np.array_equal(a, b)
    rows = a[:, 0] / 4
    assert np.all(np.diff(rows) > 0) and np.array_equal(a, big.numpy()[rows.astype(int)])   # whole rows, in order
    s = np.load(tmp_path / "a" / "small.npy")
    assert s.dtype == np.float32 and s.shape == (10, 4) and np.all(s == 1)


def _replan(envs, warmup, steps):
    """bench.py's default path (workload c2, CUDA-graph replay, fp32-parity arithmetic, torch noise) replayed without it:
    the same weights, observations and generator seed; one t0 plan, warmup - 1 warm-up plans, then `steps` device-resident
    and `steps` end-to-end timed plans.  Returns every plan's actions."""
    from tdmpc2_b200.synth import synth_state_dict
    from tdmpc2_b200.tdmpc2 import TDMPC2
    dev = torch.device("cuda", 0)
    cfg = _bench_module().bench_cfg("c2", envs)
    cfg.cuda_graph, cfg.passes, cfg.rng = True, 3, "torch"
    agent = TDMPC2(cfg, device=dev)
    agent.load(synth_state_dict(cfg, seed=1))
    agent.generator = torch.Generator(device=dev).manual_seed(3)
    obs = torch.randn(envs, cfg.obs_shape["state"][0], generator=torch.Generator().manual_seed(2)).to(dev)
    outs = [agent._plan(obs, t0=True, eval_mode=False).cpu().numpy()]
    for _ in range(warmup - 1 + 2 * steps):
        outs.append(agent._plan(obs, t0=False, eval_mode=False).cpu().numpy())
    return outs


@pytest.mark.gpu
def test_bench_dumps_the_same_actions_for_the_same_arguments(tmp_path):
    """Two runs with the same arguments dump the same actions: those of the last timed step of the plan sequence."""
    envs, warmup, steps = 8, 3, 2
    args = ["--gpus", "1", "--steps", str(steps), "--warmup", str(warmup), "--envs", str(envs), "--no-parity",
            "--no-cpu-baseline", "--no-gpu-baseline"]
    for d in ("a", "b"):
        res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args, "--dump-outputs", str(tmp_path / d)],
                             capture_output=True, text=True, timeout=600)
        assert res.returncode == 0, res.stderr[-2000:]
        line = json.loads(res.stdout.strip().splitlines()[-1])
        assert line["steps"] == steps and line["value"] > 0
    a, b = np.load(tmp_path / "a" / "actions.npy"), np.load(tmp_path / "b" / "actions.npy")
    assert a.dtype == np.float32 and a.shape[0] == envs and np.all(np.isfinite(a)) and np.all(np.abs(a) <= 1)
    assert np.array_equal(a, b)
    outs = _replan(envs, warmup, steps)
    assert np.array_equal(a, outs[-1])                   # the last timed step ...
    assert not np.array_equal(a, outs[-2])               # ... and not the one before it
