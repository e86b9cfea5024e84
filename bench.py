#!/usr/bin/env python
"""Benchmark of the TD-MPC2 planning hot path on B200 (contract: see DESIGN.md 'Measurement').

    python bench.py --gpus 1 --steps 10 --warmup 3                    # this build, workload c2 (BASELINE configs[1])
    python bench.py --workload c3|c4|c5 ...                           # the other BASELINE configs (per-GPU share)
    python bench.py --impl reference --steps 5 --warmup 3             # the reference's plan() on the host cores
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

A "step" is one full plan() over the batch of environments: noise draws, prologue (encode + policy-prior rollouts),
I CEM iterations, epilogue -- and the action all-gather when the environment axis is sharded (N > 1).
Metric (BASELINE.json): planning steps/sec = E * num_samples * horizon / t_plan.

Workloads (SURVEY.md section 8(d); synthetic weights / observations):
  c2  dog-run 5M, 256 envs per GPU, N=512, H=3, I=6          (default; the config the metric is quoted on at 1 GPU)
  c3  humanoid-walk 48M, 1024 envs per GPU, N=512, H=5, I=8
  c4  mt80 317M, 2048 envs over 8 GPUs = 256 envs per GPU, N=512, H=3, I=6
  c5  mt80 317M, 4096 envs over 8 GPUs = 512 envs per GPU, N=1024, H=8, I=10
Weak scaling: every rank plans its own share, so `--gpus 8` runs c4 / c5 exactly as BASELINE.json states them.

After the timed regions (never inside them) rank 0 adds: `parity_check` (environments OF THE TIMED BATCH re-planned
with explicit noise and compared with the CPU oracle), `cpu_baseline`, and `gpu_baseline` (the same algorithm as
batched eager PyTorch / cuBLAS on this GPU, and the reference's own `_plan` on this GPU when TDMPC2_REFERENCE_DIR names
a reference checkout).

--dump-outputs DIR writes what the last timed step returned to its caller: DIR/actions.npy, float32 [global envs,
action_dim].  Inputs (weights, observations, noise seeds) depend only on the arguments, so two builds run with the same
arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time
from typing import Optional

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from tdmpc2_b200.config import workload, flops_per_env      # noqa: E402
from tdmpc2_b200.synth import synth_state_dict              # noqa: E402

METRIC = "planning steps/sec (num_envs x num_samples x horizon per plan() call)"
UNIT = "steps/s"
WORKLOAD = "c2"
SHARDS = {"c2": 1, "c3": 1, "c4": 8, "c5": 8}               # BASELINE.json: c4 / c5 are stated for 8 GPUs
CPU_THREADS = int(os.environ.get("TDMPC2_CPU_THREADS", "8"))    # intra-op threads per reference process
DUMP_BYTES = 64 << 20                                        # --dump-outputs: most bytes written in all


def bench_cfg(name: str, envs=None):
    """The per-GPU share of a BASELINE workload (iterations = the effective loop count)."""
    cfg = workload(name, iterations_effective=True)
    per_gpu = cfg.num_envs // SHARDS.get(name, 1) if envs is None else envs
    cfg.num_envs = per_gpu
    return cfg


def describe(name: str, cfg, E_local: int) -> str:
    model = {"c2": "dog-run 5M", "c3": "humanoid-walk 48M", "c4": "mt80 317M", "c5": "mt80 317M"}.get(name, name)
    return (f"{name}: {model} model, {E_local} envs/GPU, num_samples={cfg.num_samples}, horizon={cfg.horizon}, "
            f"iterations={cfg.iterations}")


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """Each array as out_dir/<name>.npy in float32, DUMP_BYTES in all at most: an array over its share keeps a sample of
    its rows drawn from a fixed seed, so runs with the same arguments store the same rows."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_BYTES // len(arrays)
    for name, a in arrays.items():
        a = a.detach().to("cpu", torch.float32)
        if a.numel() * 4 > share:
            rows = max(1, share // (4 * a[0].numel()))
            a = a[torch.randperm(a.shape[0], generator=torch.Generator().manual_seed(0))[:rows].sort().values]
        np.save(os.path.join(out_dir, name + ".npy"), a.numpy())


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu, self.proc, self.path = gpu_index, None, None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 9:
                    continue
                try:
                    sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
                except ValueError:
                    continue
                for n, v in zip(names, f[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm),
                       power_w=statistics.median(pw))
        return out


# ------------------------------------------------------------------------------------------------ CPU reference legs
def _ref_available() -> bool:
    try:
        from oracle import ref_harness
        return ref_harness.available()
    except Exception:
        return False


def _cpu_worker(args):
    """One host process: plans `envs` environments one after another (the reference has no env axis) with `threads`
    intra-op threads; returns (seconds per env-plan, kind)."""
    wl, envs, steps, warmup, threads, budget_s, use_ref, seed = args
    import torch as th
    th.set_num_threads(threads)
    cfg = bench_cfg(wl, envs)
    sd = synth_state_dict(cfg, seed=1)
    g = th.Generator().manual_seed(2 + seed)
    obs = th.randn(envs, cfg.obs_shape["state"][0], generator=g)
    times, t_begin = [], time.perf_counter()
    if use_ref:
        # the reference's OWN unmodified _plan (tdmpc2.py:138-206) through the harness, eager, one env per call
        from oracle import ref_harness
        agent = ref_harness.build_agent(cfg, sd)
        th.manual_seed(3 + seed)
        for s in range(warmup + steps):
            if budget_s is not None and times and time.perf_counter() - t_begin > budget_s:
                break
            t = time.perf_counter()
            for e in range(envs):
                tk = th.tensor([e % len(cfg.tasks)]) if cfg.multitask else None
                agent._plan(obs[e].view(1, -1), t0=(s == 0), eval_mode=False, task=tk)
            if s >= warmup:
                times.append((time.perf_counter() - t) / envs)
        kind = "reference"
    else:
        from oracle.plan_oracle import OracleModel, draw_noise, plan_oracle
        model = OracleModel(cfg, sd)
        prev = th.zeros(envs, cfg.horizon, cfg.action_dim)
        for s in range(warmup + steps):
            if budget_s is not None and times and time.perf_counter() - t_begin > budget_s:
                break
            noise = draw_noise(cfg, 3 + 1000 * s + seed, envs)
            t = time.perf_counter()
            tr = plan_oracle(cfg, model, obs, t0=[s == 0] * envs, prev_mean=prev, noise=noise,
                             task=[e % len(cfg.tasks) for e in range(envs)] if cfg.multitask else None)
            dt = time.perf_counter() - t
            prev = tr.mean
            if s >= warmup:
                times.append(dt / envs)
        kind = "port"
    return sum(times) / len(times), kind


def _cpu_layout_run(wl, steps, warmup, budget_s, procs, threads, use_ref):
    import multiprocessing as mp
    cfg = bench_cfg(wl, 1)
    jobs = [(wl, 1, steps, warmup, threads, budget_s, use_ref, i) for i in range(procs)]
    if procs == 1:
        res = [_cpu_worker(jobs[0])]
    else:
        with mp.get_context("spawn").Pool(procs) as pool:
            res = pool.map(_cpu_worker, jobs)
    t_env = statistics.mean(r[0] for r in res)
    value = sum(cfg.num_samples * cfg.horizon / r[0] for r in res)
    return value, t_env, res[0][1]


def cpu_reference_run(wl: str, steps: int, warmup: int, budget_s: Optional[float]):
    """The reference's plan() on the host cores, with all the threads it can USE: eager PyTorch on these GEMM sizes
    stops scaling far below a 100+ core host (round 1: 128 threads in one process -> 53 s/plan, 16 -> 57 ms), and
    environments are independent, so the host layouts tried are processes x intra-op threads -- one process with
    16 threads, and process-parallel with 8 threads each over all cores -- and the BEST aggregate is reported.
    Every process plans its environments one after another (evaluate.py's loop; the reference has no env axis).
    budget_s bounds the time of a layout (a process stops after the step that crosses it, and the layouts after the
    first are skipped when they would exceed it); None times exactly `steps` steps after `warmup` in every layout.
    Returns (steps/s aggregate, seconds per env-plan of one process, cores used, kind, procs, all layouts tried)."""
    host = os.cpu_count() or 1
    use_ref = _ref_available()
    layouts = [(1, min(16, host))]
    if host >= 32:
        layouts += [(host // 32, 8), (host // 8, 8)]
    tried, best, t_first = [], None, None
    for procs, threads in layouts:
        if budget_s is not None and t_first is not None and 12.0 * t_first * (warmup + 1) > 2.0 * budget_s and procs > 1:
            tried.append({"procs": procs, "threads": threads, "skipped": "would exceed the time budget"})
            continue
        value, t_env, kind = _cpu_layout_run(wl, steps, warmup, budget_s, procs, threads, use_ref)
        t_first = t_env if t_first is None else t_first
        tried.append({"procs": procs, "threads": threads, "steps_per_s": round(value, 1), "s_per_env_plan": round(t_env, 3)})
        if best is None or value > best[0]:
            best = (value, t_env, procs * threads, kind, procs)
    return best + (tried,)


def run_reference(args):
    """`--impl reference`: the reference's own CPU implementation of the path on the box's host cores, all the threads
    it can use, on a bounded sample of the same workload: every process plans one environment for exactly --warmup,
    then --steps steps.  Under torchrun only rank 0 runs."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = args.workload
    cfg = bench_cfg(wl)
    value, t_env, cores, kind, procs, tried = cpu_reference_run(wl, args.steps, args.warmup, budget_s=None)
    src = ("the reference's own unmodified TDMPC2._plan (TDMPC2_REFERENCE_DIR via oracle/ref_harness.py)" if kind == "reference"
           else "oracle port of the reference algorithm (reference sources not on this box)")
    sample = (f"{procs} processes x {cores // procs} threads, each planning 1 environment of the workload per step, "
              f"sequentially inside a process (the reference has no env axis); {src}")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * t_env, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": describe(wl, cfg, cfg.num_envs) + " (reference algorithm, host CPU, eager PyTorch fp32)",
                   "envs_per_step": procs, "host_cores": os.cpu_count()},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample,
                         "host_cores": os.cpu_count(), "layouts_tried": tried},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------ parity of the timed batch
def parity_check(cfg, sd, obs_host, task_host, E_local, dev, engine, envs, budget_gflop=3000.0):
    """Re-plan the TIMED batch (same E, same engine, hence the same multi-trip persistent schedule) with explicit noise
    and compare the sampled environments with the CPU oracle (values 5e-5 + 1e-5 |v|, top-k indices exact where the
    oracle's sorted values are > 2*tol apart, refit mean 1e-4 while the elite set is unambiguous)."""
    from oracle.plan_oracle import draw_noise as oracle_noise, plan_oracle
    from tdmpc2_b200.planner import Planner, draw_noise
    torch.set_num_threads(max(1, min(16, os.cpu_count() or 1)))     # eager CPU PyTorch collapses on 100+ threads
    per_env = flops_per_env(cfg, heads_used=cfg.num_q) / 1e9
    envs = [e for e in envs if e < E_local][: max(1, int(budget_gflop // max(per_env, 1e-9)))]
    if per_env > budget_gflop:
        return {"skipped": f"oracle needs {per_env:.0f} GFLOP per environment on the host; run tests/test_gpu_multitrip.py"}
    atol, rtol = 5e-5, 1e-5                      # the tolerance of tests/test_gpu_parity.py, for every preset
    pl = Planner(cfg, E_local, dev, engine=engine)
    pl.pack(sd)
    g = torch.Generator(device=dev).manual_seed(1234)
    noise = draw_noise(cfg, E_local, dev, generator=g, reference_order=False)
    on = oracle_noise(cfg, 9000, len(envs))
    for j, e in enumerate(envs):
        noise.prior[e] = on.prior[j].to(dev)
        noise.r[:, e] = on.r[j].to(dev)
        noise.pi[:, e] = on.pi[j].to(dev)
        noise.qidx[:, e] = on.qidx[j].to(torch.int32).to(dev)
        noise.expo[e] = on.expo[j].to(dev)
        noise.final[e] = on.final[j].to(dev)
    gp = torch.Generator().manual_seed(77)
    prev = 0.3 * torch.randn(E_local, cfg.horizon, cfg.action_dim, generator=gp)
    t0 = torch.zeros(E_local, dtype=torch.uint8)
    taskv = None if task_host is None else task_host.to(torch.int32).to(dev)
    action, new_mean, tr = pl.plan(obs_host.to(dev), taskv, t0.to(dev), prev.to(dev), noise, trace=True)
    torch.cuda.synchronize()
    t_or = time.perf_counter()
    want = plan_oracle(cfg, sd, obs_host[envs], task=None if task_host is None else [int(task_host[e]) for e in envs],
                       t0=[False] * len(envs), prev_mean=prev[envs], noise=on)
    t_or = time.perf_counter() - t_or
    K = cfg.num_elites
    out = {"envs": envs, "value_tol": f"{atol} + {rtol} |v|", "max_abs_value_err": 0.0, "topk_positions_checked": 0, "topk_mismatches": 0,
           "refit_checked": 0, "max_abs_mean_err": 0.0, "max_abs_action_err": None, "oracle_s": round(t_or, 2)}
    ok = True
    for j, e in enumerate(envs):
        clean = True
        for it in range(cfg.iterations):
            v_got, v_want = tr["values"][e, it].cpu(), want.values[j, it]
            err = float((v_got - v_want).abs().max())
            out["max_abs_value_err"] = max(out["max_abs_value_err"], err)
            ok &= bool(torch.allclose(v_got, v_want, atol=atol, rtol=rtol))
            tol = atol + rtol * float(v_want.abs().max())
            top = torch.topk(v_want, K + 1).values
            gaps = top[:-1] - top[1:]
            sep = gaps > 2 * tol
            stable = sep & torch.cat([torch.ones(1, dtype=torch.bool), sep[:-1]])
            got_idx = tr["elite_idx"][e, it].cpu()
            mism = int((got_idx[stable] != want.elite_idx[j, it][stable]).sum())
            out["topk_positions_checked"] += int(stable.sum()); out["topk_mismatches"] += mism
            ok &= mism == 0
            if not bool(gaps[K - 1] > 2 * tol):
                clean = False
                break
            merr = float((tr["iter_mean"][e, it].cpu() - want.iter_mean[j, it]).abs().max())
            out["max_abs_mean_err"] = max(out["max_abs_mean_err"], merr); out["refit_checked"] += 1
            ok &= merr < 1e-4
        if clean:
            lg = want.score[j].log() - on.expo[j].log()
            t2 = torch.topk(lg, 2).values
            if float(t2[0] - t2[1]) > 1e-3:
                aerr = float((action[e].cpu() - want.action[j]).abs().max())
                out["max_abs_action_err"] = max(out["max_abs_action_err"] or 0.0, aerr)
                ok &= aerr < 1e-4
    out["ok"] = bool(ok and out["topk_positions_checked"] > 0)
    del pl
    return out


# ------------------------------------------------------------------------------------------------ GPU baselines (same box)
def gpu_baselines(wl, cfg, dev, budget_s=40.0):
    """SURVEY.md section 8(d)(ii)/(iii): what the library path does on the same B200 (never the product path)."""
    out = {}
    try:
        import importlib.util
        spec = importlib.util.spec_from_file_location("torch_gpu_baseline", os.path.join(ROOT, "scripts", "torch_gpu_baseline.py"))
        tb = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(tb)
        # bounded sample: the batched restatement keeps [num_q, E*N, mlp_dim] fp32 activations
        rows_budget = 6e9 / (4.0 * cfg.num_q * cfg.mlp_dim)                 # ~6 GB for the largest activation
        envs = int(max(1, min(cfg.num_envs, rows_budget // cfg.num_samples)))
        for tf32 in (False, True):
            r = tb.run(wl, envs=envs, steps=3, device=str(dev), tf32=tf32, budget_s=budget_s / 2)
            out["torch_batched_" + r["matmul"]] = {"value": r["value"], "unit": UNIT, "ms_per_step": r["ms_per_step"],
                                                   "envs_per_step": r["envs"], "impl": r["impl"]}
            torch.cuda.empty_cache()
    except Exception as e:                                                   # a baseline must never take the line down
        out["torch_batched_error"] = repr(e)[:300]
    try:
        from oracle import ref_harness
        if ref_harness.available():
            rcfg = bench_cfg(wl, 1)
            agent = ref_harness.build_agent(rcfg, synth_state_dict(rcfg, seed=1), device=dev)
            obs = torch.randn(1, rcfg.obs_shape["state"][0], device=dev)
            tk = torch.tensor([0], device=dev) if rcfg.multitask else None
            with torch.no_grad():
                agent._plan(obs, t0=True, eval_mode=False, task=tk)
                agent._plan(obs, t0=False, eval_mode=False, task=tk)
                torch.cuda.synchronize()
                times, t_begin = [], time.perf_counter()
                while len(times) < 10 and time.perf_counter() - t_begin < budget_s / 2:
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(); agent._plan(obs, t0=False, eval_mode=False, task=tk); e1.record()
                    torch.cuda.synchronize()
                    times.append(e0.elapsed_time(e1))
            ms = statistics.median(times)
            out["reference_plan_eager_gpu"] = {"value": rcfg.num_samples * rcfg.horizon / (ms * 1e-3), "unit": UNIT,
                                               "ms_per_env_plan": ms, "calls": len(times),
                                               "impl": "the reference's own unmodified TDMPC2._plan (TDMPC2_REFERENCE_DIR), eager, "
                                                       "one environment per call (it has no env axis), fp32"}
            del agent
            torch.cuda.empty_cache()
        else:
            out["reference_plan_eager_gpu"] = {"unavailable": "no reference checkout (TDMPC2_REFERENCE_DIR)"}
    except Exception as e:
        out["reference_plan_error"] = repr(e)[:300]
    return out


def act_latency_e1(wl, sd, dev, args, calls=20):
    """The reference's own call shape (evaluate.py:80): ONE environment per act(), CPU observation in, CPU action out; the
    launch chain runs with the reference-order noise draws on a side stream between the launches (Planner.plan_interleaved;
    --no-graph: all draws first, then eager launches).  Median wall-clock ms per call (perf_counter around act(); it ends
    with .cpu())."""
    from tdmpc2_b200.tdmpc2 import TDMPC2
    cfg1 = bench_cfg(wl, 1)
    cfg1.cuda_graph = not args.no_graph
    cfg1.passes = args.passes
    a1 = TDMPC2(cfg1, device=dev, engine=args.engine)
    a1.load(sd)
    obs = torch.randn(cfg1.obs_shape["state"][0]).pin_memory()
    task = 0 if cfg1.multitask else None
    a1.act(obs, t0=True, task=task)
    for _ in range(3):
        a1.act(obs, t0=False, task=task)
    torch.cuda.synchronize()
    ts = []
    for _ in range(calls):
        t = time.perf_counter()
        a1.act(obs, t0=False, task=task)
        ts.append(1e3 * (time.perf_counter() - t))
    del a1
    return {"ms_per_act_median": statistics.median(ts), "ms_per_act_min": min(ts), "calls": calls,
            "what": "TDMPC2.act(obs[obs_dim] on host) -> action on host, num_envs=1 (the reference's API shape), same model / planner settings"}


# ------------------------------------------------------------------------------------------------ this build
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--engine", default=None)
    ap.add_argument("--workload", default=WORKLOAD, choices=sorted(SHARDS))
    ap.add_argument("--envs", type=int, default=None, help="environments per GPU (default: the workload's share)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="launch the plan chain eagerly instead of replaying the CUDA graph")
    ap.add_argument("--rng", default="torch", choices=["torch", "philox"],
                    help="torch = the reference's noise draws (parity; the headline); philox = the DECLARED NON-PARITY throughput "
                         "mode: the two large noise tensors are generated inside the kernels (its own line; no oracle comparison)")
    ap.add_argument("--passes", type=int, default=3, choices=[1, 3],
                    help="3 = fp32-parity arithmetic (the headline); 1 = the DECLARED NON-PARITY fast mode (one fp16 MMA per "
                         "product): its own line, dtype f16, parity_check reports the elite-flip rate instead of gating")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the actions the last timed step returned to DIR/actions.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes the actions of this build's timed path; --impl reference has none to write")
        return run_reference(args)
    args.warmup = max(args.warmup, 3)

    import torch.distributed as dist
    from tdmpc2_b200.tdmpc2 import TDMPC2
    from tdmpc2_b200.sharded import ShardedActor

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the planner has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    assert world == args.gpus or world == 1, f"launched with WORLD_SIZE={world} but --gpus {args.gpus}"

    wl = args.workload
    cfg = bench_cfg(wl, args.envs)
    cfg.cuda_graph = not args.no_graph
    cfg.passes = args.passes
    cfg.rng = args.rng
    E_local = cfg.num_envs                       # weak scaling: per-GPU work is fixed
    E_total = E_local * world
    sd = synth_state_dict(cfg, seed=1)
    agent = TDMPC2(cfg, device=dev, engine=args.engine)
    agent.load(sd)
    gen = torch.Generator(device=dev).manual_seed(3 + rank)
    agent.generator = gen
    obs_dim, A = cfg.obs_shape["state"][0], cfg.action_dim
    g = torch.Generator().manual_seed(2)
    obs_host_all = torch.randn(E_total, obs_dim, generator=g)
    obs_host = obs_host_all[rank * E_local:(rank + 1) * E_local].clone().pin_memory()
    obs_dev = obs_host.to(dev)
    task_host = task_dev = None
    if cfg.multitask:
        task_host = torch.arange(rank * E_local, (rank + 1) * E_local) % len(cfg.tasks)
        task_dev = task_host.to(torch.int32).to(dev)
    actions_host = torch.empty(E_total, A).pin_memory()
    # environment-axis sharding: rank-local plan + ONE all-gather of the selected actions (only when world > 1)
    actor = ShardedActor(lambda o, t0, task: agent._plan(o, t0=t0, eval_mode=False, task=task), E_total)

    def step_device(t0):
        """plan() with inputs resident in HBM (+ the action all-gather when sharded)."""
        return actor.act_local(obs_dev, t0=t0, task=task_dev)

    def step_e2e(t0):
        """The user-facing call: HOST observations in (pinned), HOST actions out."""
        o = obs_host.to(dev, non_blocking=True)
        a = actor.act_local(o, t0=t0, task=task_dev)
        actions_host[: a.shape[0]].copy_(a, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return actions_host

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        """K steps between CUDA events, barrier + synchronize on both sides, max over ranks."""
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for _ in range(steps):
            fn(False)
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms / steps

    # ---- warm-up (first call t0=True, then steady-state warm starts; the first steady call captures the graph)
    step_device(True)
    for _ in range(args.warmup - 1):
        step_device(False)
    barrier()
    launches0 = agent.planner.launches
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms_step = timed(step_device, args.steps)
    launches = agent.planner.launches - launches0
    ms_e2e = timed(step_e2e, args.steps)
    clocks = sampler.stop() if rank == 0 else {}
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"actions": actions_host})

    # ---- dominant kernel: one CEM-iteration launch, timed alone with events on its stream
    from tdmpc2_b200.planner import draw_noise
    pl = agent.planner
    noise = draw_noise(cfg, E_local, dev, generator=gen, reference_order=False)
    t0v = torch.zeros(E_local, dtype=torch.uint8, device=dev)
    prev = agent._prev_mean.reshape(E_local, cfg.horizon, A).contiguous()
    pl.prologue(obs_dev, task_dev, t0v, prev, noise.prior)
    if pl.philox:
        its = [(i, noise.qidx[i]) for i in range(cfg.iterations)]
        pl.iterate = pl.iterate_rng                       # same timing loop, in-kernel noise
    else:
        its = [(noise.r[i], noise.pi[i], noise.qidx[i]) for i in range(cfg.iterations)]
    for a_ in its[:2]:
        pl.iterate(*a_)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 3 if ms_step < 500 else 1
    e0.record()
    for _ in range(reps):
        for a_ in its:
            pl.iterate(*a_)
    e1.record()
    torch.cuda.synchronize()
    ms_iter = e0.elapsed_time(e1) / (reps * cfg.iterations)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peaks, peak_src = load_peaks()
    traffic, traffic_src = None, None
    try:   # DRAM bytes per launch of the dominant kernel, from the committed ncu --set full capture of this workload
        sfx = "_pp" if agent.planner.iter_engine == "tcgen05pp" else ""       # one capture per engine
        with open(os.path.join(ROOT, "profiles", f"r02_traffic_{wl}{sfx}.json")) as f:
            tj = json.load(f)
        if int(tj.get("envs", -1)) == E_local and args.passes == 3:
            from tdmpc2_b200 import build as _b
            traffic = tj["dram_bytes_per_launch"]
            traffic_src = {"file": f"profiles/r02_traffic_{wl}{sfx}.json", "kernel_sources_unchanged_since_capture":
                           tj.get("lib_digest") == _b._digest()}
    except Exception:
        traffic = None
    L, M, A_, T, B = cfg.latent_dim, cfg.mlp_dim, cfg.action_dim, cfg.task_dim, cfg.num_bins
    D = L + T + A_
    w = lambda i, h, o: i * h + h * h + h * o
    flops_iter = 2.0 * E_local * cfg.num_samples * (cfg.horizon * (w(D, M, B) + w(D, M, L)) + w(L + T, M, 2 * A_) + 2 * w(D, M, B))
    achieved = flops_iter / (ms_iter * 1e-3) / 1e12
    peak = float(peaks["bf16_tflops"])
    steps_per_plan = E_total * cfg.num_samples * cfg.horizon
    value = steps_per_plan / (ms_step * 1e-3)
    e2e_value = steps_per_plan / (ms_e2e * 1e-3)
    noise_mb = 0.0 if args.rng != "torch" else 4 * E_local * cfg.iterations * (cfg.horizon * (cfg.num_samples - cfg.num_pi_trajs) + cfg.num_samples) * A_ / 1e6
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32" if args.passes == 3 else "f16", "data": "synthetic",
        "config": {"workload": describe(wl, cfg, E_local),
                   "global_envs": E_total, "parallelism": f"env-shard x{world}", "engine": agent.planner.iter_engine,
                   "arithmetic": "3-pass fp16-split operands on tcgen05 kind::f16, fp32 accumulate (fp32-parity mode)" if args.passes == 3
                                 else "DECLARED NON-PARITY fast mode: single-pass fp16 operands on tcgen05 kind::f16, fp32 accumulate",
                   "rng": "torch CUDA generator (reference draw semantics)" if args.rng == "torch"
                          else "DECLARED NON-PARITY: in-kernel Philox4x32-10 + Box-Muller for noise_r / noise_pi",
                   "launch": "CUDA-graph replay of prologue -> I x iter -> epilogue" if agent._use_graph and not args.no_graph
                             else "eager launch chain",
                   "l2": f"no flush: per-step inputs exceed L2 (fresh noise tensors, {noise_mb:.0f} MB/step/GPU)"
                         if noise_mb > 130 else f"no flush; fresh noise tensors {noise_mb:.0f} MB/step/GPU + weights",
                   "tflops_algorithmic": flops_per_env(cfg) * E_total / (ms_step * 1e-3) / 1e12,
                   "ms_outside_iter_kernels": ms_step - cfg.iterations * ms_iter},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": ms_e2e,
                "h2d_bytes_per_step": int(E_local * obs_dim * 4), "d2h_bytes_per_step": int(E_total * A_ * 4)},
        "gpu_launches": int(launches),
        "roofline": {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                     "frac_vs_sustained": achieved / float(peaks.get("bf16_tflops_sustained", peak)),
                     "traffic": traffic, "traffic_source": traffic_src,
                     "kernel": ("plan_pp_kernel" if agent.planner.iter_engine == "tcgen05pp" else "plan_kernel<tcgen05, pair>") + " (one CEM iteration)",
                     "ms_per_launch": ms_iter, "peak_source": f"MEASURED_PEAKS.json bf16_tflops ({peak_src}, burst)",
                     "flop_per_launch": flops_iter,
                     "note": ("achieved counts ALGORITHMIC flops (2 Q heads, 1x); the fp32-parity path issues 3 fp16 MMAs "
                              "per product, so its ceiling is peak/3") if args.passes == 3 else
                             "achieved counts ALGORITHMIC flops (2 Q heads, 1x); single-pass fast mode, ceiling = peak"},
    }
    if world == 1:
        del agent, actor, pl
        torch.cuda.empty_cache()
        try:
            line["e2e"]["act_latency_e1"] = act_latency_e1(wl, sd, dev, args)
        except Exception as e:
            line["e2e"]["act_latency_e1"] = {"error": repr(e)[:200]}
        torch.cuda.empty_cache()
        if args.rng != "torch":
            line["parity_check"] = {"skipped": "in-kernel noise stream: the oracle consumes torch's draws (declared non-parity mode)"}
        elif not args.no_parity:
            try:
                line["parity_check"] = parity_check(cfg, sd, obs_host.clone(), task_host, E_local, dev, args.engine,
                                                    envs=[0, E_local - 1, E_local // 2 + 1])
                if args.passes != 3:        # non-parity mode: the same comparison is a REPORT (elite-flip rate), not a gate
                    pc = line["parity_check"]
                    pc["mode"] = "declared non-parity fast mode: reported, not gated"
                    if pc.get("topk_positions_checked"):
                        pc["elite_flip_rate"] = pc["topk_mismatches"] / pc["topk_positions_checked"]
            except Exception as e:
                line["parity_check"] = {"ok": False, "error": repr(e)[:300]}
            torch.cuda.empty_cache()
        if not args.no_gpu_baseline:
            line["gpu_baseline"] = gpu_baselines(wl, cfg, dev)
        if not args.no_cpu_baseline:
            heavy = flops_per_env(cfg, heads_used=cfg.num_q) > 1e12
            v, t_env, cores, kind, procs, tried = cpu_reference_run(wl, steps=1 if heavy else 3, warmup=0 if heavy else 1, budget_s=15.0)
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": kind, "host_cores": os.cpu_count(), "layouts_tried": tried,
                                    "sample": f"{procs} processes x {cores // procs} threads, each planning 1 environment of the workload "
                                              f"per step (best of the host layouts tried), sequential inside a process (reference has no env axis), eager PyTorch fp32; "
                                              f"{1e3 * t_env:.1f} ms per env-plan per process"}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
