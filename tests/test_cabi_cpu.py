"""CPU-side checks of the boundary: the C-ABI library loads, exports every symbol the
header declares, and refuses to run without a B200 (no CPU fallback)."""
import ctypes as C
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from tdmpc2_b200 import build, _cabi
    build.build()
    return _cabi.load()


def test_library_exports_every_header_symbol(lib):
    from tdmpc2_b200 import _cabi
    hdr = open(os.path.join(ROOT, "include", "tdmpc2_b200.h")).read()
    declared = set(re.findall(r"\b(tdmpc2_[a-z_0-9]+)\s*\(", hdr))
    declared -= {"tdmpc2_planner"}
    assert declared == set(_cabi.SYMBOLS), declared ^ set(_cabi.SYMBOLS)
    for s in declared:
        assert hasattr(lib, s), s
    want = int(re.search(r"#define TDMPC2_B200_ABI_VERSION (\d+)", hdr).group(1))
    assert lib.tdmpc2_abi_version() == want == _cabi.ABI_VERSION


def test_struct_layout_matches_header():
    from tdmpc2_b200 import _cabi
    assert C.sizeof(_cabi.Dims) == 18 * 4 + 5 * 4
    assert C.sizeof(_cabi.Linear) == 4 * 8
    assert C.sizeof(_cabi.Weights) == 8 + (_cabi.MAX_ENC_LAYERS + 12) * 32 + 4 * 8 + 3 * 32   # ... + termination[3]


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_no_cpu_fallback(lib):
    from tdmpc2_b200 import _cabi
    from tdmpc2_b200.config import workload
    from tdmpc2_b200.planner import Planner
    with pytest.raises(_cabi.CabiError):
        Planner(workload("tiny"), 1, "cpu")
    d = _cabi.Dims(num_envs=1, num_samples=128, num_pi_trajs=8, num_elites=16, horizon=3, iterations=2, obs_dim=8,
                   action_dim=4, latent_dim=64, mlp_dim=64, enc_dim=64, num_enc_layers=2, task_dim=0, num_tasks=1,
                   num_q=2, num_bins=101, simnorm_dim=8, episodic=0, temperature=0.5, min_std=0.05, max_std=2.0,
                   log_std_min=-10.0, log_std_dif=12.0)
    h = C.c_void_p()
    rc = lib.tdmpc2_planner_create(C.byref(d), C.byref(h))
    assert rc == -2 and b"no CUDA device" in lib.tdmpc2_last_error()       # TDMPC2_ERR_NO_DEVICE
    d.episodic = 1                                                           # termination head: accepted (single-task)
    assert lib.tdmpc2_planner_create(C.byref(d), C.byref(h)) == -2
    d.task_dim, d.num_tasks = 16, 3                                          # ... but not multi-task (world_model.py:136)
    assert lib.tdmpc2_planner_create(C.byref(d), C.byref(h)) == -5          # TDMPC2_ERR_UNSUPPORTED
    d.episodic = 2
    assert lib.tdmpc2_planner_create(C.byref(d), C.byref(h)) == -1          # TDMPC2_ERR_INVALID


def test_world_model_state_dict_layout():
    """WorldModel.state_dict() has exactly the reference's keys (SURVEY.md 8(b))."""
    from tdmpc2_b200.config import workload
    from tdmpc2_b200.synth import synth_state_dict
    from tdmpc2_b200.world_model import WorldModel, convert_legacy_checkpoint
    for wl, over in (("tiny", {}), ("tiny-mt", {}), ("tiny", {"episodic": True}), ("tiny-rgb", {})):
        cfg = workload(wl, **over)
        m = WorldModel(cfg)
        sd = m.state_dict()
        want = synth_state_dict(cfg, seed=3, perturb=True)
        meta = {k for k in sd if k.endswith(("__batch_size", "__device"))}
        assert meta == {p + s for p in ("_Qs.params.", "_detach_Qs_params.", "_target_Qs_params.")
                        for s in ("__batch_size", "__device")}
        assert set(sd) - meta == set(want)
        assert sd["_Qs.params.__batch_size"] == torch.Size([cfg.num_q])
        for k in want:
            assert tuple(sd[k].shape) == tuple(want[k].shape), k
        m.load_state_dict(want)
        got = m.state_dict()
        for k in want:
            assert torch.equal(got[k], want[k]), k
        # zero-init of the reward / Q output layers (world_model.py:32)
        fresh = WorldModel(cfg).state_dict()
        assert fresh["_reward.2.weight"].abs().sum() == 0 and fresh["_Qs.params.2.weight"].abs().sum() == 0
        assert fresh["_detach_Qs_params.0.weight"].data_ptr() == fresh["_Qs.params.0.weight"].data_ptr()
        # legacy (pre-compile API) checkpoints: _Qs.params.<n>, _target_Qs.params.<n>
        legacy = {k: v for k, v in want.items() if "Qs" not in k}
        names = ["weight", "bias", "ln.weight", "ln.bias"]
        for layer in range(3):
            for j, nm in enumerate(names):
                key = f"{layer}.{nm}"
                if "_Qs.params." + key in want:
                    legacy[f"_Qs.params.{4 * layer + j}"] = want["_Qs.params." + key]
                    legacy[f"_target_Qs.params.{4 * layer + j}"] = want["_target_Qs_params." + key]
        conv = convert_legacy_checkpoint(m.state_dict(), legacy)
        m2 = WorldModel(cfg)
        m2.load_state_dict(conv)
        for k in want:
            assert torch.equal(m2.state_dict()[k], want[k]), k


def test_pixel_model_keys_are_the_references(golden_dir):
    """cfg.obs == 'rgb': the container's keys and shapes are what the reference's own WorldModel registers, its encoder
    keys what layers.conv registers (_encoder.rgb.{2,4,6,8}.{weight,bias}, layers.py:136-150).  The reference's layout
    is stored in tests/golden/tiny_rgb_keys.npz (oracle/make_golden.py mints it from the reference model)."""
    import numpy as np
    from tdmpc2_b200.config import workload
    from tdmpc2_b200.synth import synth_state_dict
    f = np.load(os.path.join(golden_dir, "tiny_rgb_keys.npz"), allow_pickle=False)
    ref = {str(k): tuple(int(d) for d in str(s).split(",") if d) for k, s in zip(f["keys"], f["shapes"])}
    cfg = workload(str(f["workload"]))
    sd = synth_state_dict(cfg, seed=2)
    ours = {k: tuple(v.shape) for k, v in sd.items()        # the copies build_agent() leaves out of the reference model
            if not k.startswith(("_detach_Qs_params.", "_target_Qs_params.")) and "__" not in k}
    assert ours == ref
    ref_keys = {k for k in ref if k.startswith("_encoder.")}
    assert ref_keys == {k for k in sd if k.startswith("_encoder.")} == {
        f"_encoder.rgb.{i}.{n}" for i in (2, 4, 6, 8) for n in ("weight", "bias")}
    with pytest.raises(ValueError):                          # layers.conv flattens [num_channels, 4, 4]
        from tdmpc2_b200.world_model import WorldModel
        WorldModel(workload("tiny-rgb", latent_dim=64))


def test_graft_entry_build():
    """The driver's build check: __graft_entry__.build() compiles (or finds) the library, loads it, imports the package."""
    import importlib
    ge = importlib.import_module("__graft_entry__")
    ge.build()


def test_plain_c_host_links_and_reports_no_device(lib, tmp_path):
    """The boundary is a C ABI: a C11 program (examples/c_host.c) compiles against include/tdmpc2_b200.h, links the
    shared library without Python or torch, and -- on a machine without a B200 -- gets TDMPC2_ERR_NO_DEVICE."""
    import shutil, subprocess
    from tdmpc2_b200 import _cabi
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("no gcc")
    libdir = os.path.dirname(_cabi.LIB_PATH)
    exe = str(tmp_path / "c_host")
    subprocess.run([gcc, "-std=c11", "-Wall", "-Werror", "-I" + os.path.join(ROOT, "include"),
                    os.path.join(ROOT, "examples", "c_host.c"), "-L" + libdir, "-ltdmpc2_b200",
                    "-Wl,-rpath," + libdir, "-o", exe], check=True)
    res = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert res.returncode == 0, res.stdout + res.stderr
    assert "ABI version" in res.stdout
    if not torch.cuda.is_available():
        assert "no CUDA device" in res.stdout


def test_product_never_imports_the_oracle():
    """oracle/ is test infrastructure: nothing under tdmpc2_b200/ (or the drop-in shim) may import it, and bench.py
    only inside its CPU-baseline / reference-arm function."""
    import ast
    def imports_oracle(path):
        tree = ast.parse(open(path).read())
        hits = []
        for node in ast.walk(tree):
            names = []
            if isinstance(node, ast.Import):
                names = [a.name for a in node.names]
            elif isinstance(node, ast.ImportFrom):
                names = [node.module or ""]
            hits += [(n, node.lineno) for n in names if n == "oracle" or n.startswith("oracle.")]
        return hits
    for d in ("tdmpc2_b200", "dropin"):
        for fn in os.listdir(os.path.join(ROOT, d)):
            if fn.endswith(".py"):
                assert not imports_oracle(os.path.join(ROOT, d, fn)), fn
    src = open(os.path.join(ROOT, "bench.py")).read()
    tree = ast.parse(src)
    for fn in [n for n in tree.body if isinstance(n, ast.FunctionDef)]:
        uses = [n for n in ast.walk(fn) if isinstance(n, ast.ImportFrom) and (n.module or "").startswith("oracle")]
        if uses:
            # the CPU legs (cpu_baseline / --impl reference), the post-timing parity checker, and the on-box run of the
            # reference's own _plan for the gpu_baseline block; never main() / the timed step functions
            assert fn.name in ("_cpu_worker", "_ref_available", "parity_check", "gpu_baselines"), fn.name
    assert not [n for n in tree.body if isinstance(n, (ast.Import, ast.ImportFrom)) and "oracle" in ast.dump(n)]


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the oracle port on the host cores) needs no GPU: one JSON line with the contract keys."""
    import json, subprocess, sys
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600, env={**os.environ, "TDMPC2_CPU_THREADS": "8"})
    assert res.returncode == 0, res.stderr[-2000:]
    line = json.loads(res.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "steps/s" and line["value"] > 0 and line["higher_is_better"]
    assert line["cpu_baseline"]["kind"] in ("port", "reference") and line["cpu_baseline"]["cores"] >= 1
    assert line["cpu_baseline"]["host_cores"] == os.cpu_count()
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["gpu_launches"] == 0
    assert "workload" in line["config"]


def test_bench_reference_arm_times_exactly_the_steps_asked(monkeypatch, capsys):
    """`--impl reference --steps K --warmup W` plans W + K steps in every process: no cap on K, no time budget."""
    import argparse, importlib.util, json
    import oracle.plan_oracle as po
    spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    calls, real = [], po.plan_oracle
    monkeypatch.setattr(po, "plan_oracle", lambda *a, **k: calls.append(1) or real(*a, **k))
    monkeypatch.setattr(bench, "_ref_available", lambda: False)
    monkeypatch.setattr(os, "cpu_count", lambda: 8)          # one host layout: one process, in this interpreter
    bench.run_reference(argparse.Namespace(workload="c2", steps=23, warmup=2, gpus=1))
    line = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    assert len(calls) == 25 and line["steps"] == 23 and line["warmup"] == 2
