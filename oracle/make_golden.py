"""Mint golden vectors from the REFERENCE's own planner -- TEST INFRASTRUCTURE ONLY.

Needs a reference checkout (see oracle/ref_harness.py):

    TDMPC2_REFERENCE_DIR=<checkout>/tdmpc2 python -m oracle.make_golden     # writes tests/golden/*.npz

For each workload it builds synthetic weights (tdmpc2_b200.synth, seed in the
fixture), loads them into the reference WorldModel via oracle/ref_harness.py and
records what the reference's unmodified `TDMPC2._plan` returns for a chain of
calls (first call t0=True, later calls warm-started from the previous
`_prev_mean`), under torch.manual_seed(seed).  The fixtures carry only inputs,
seeds and outputs (a few KB each); weights are regenerated from the seed and
guarded by a checksum.
"""
from __future__ import annotations

import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tdmpc2_b200.config import workload            # noqa: E402
from tdmpc2_b200.synth import synth_state_dict, state_dict_checksum  # noqa: E402
from oracle import ref_harness as rh               # noqa: E402

# name -> (workload, overrides, weight seed, perturb, emb_scale, [(t0, eval_mode, task, noise seed), ...])
CASES = {
    "tiny": ("tiny", {}, 11, True, 1.0,
             [(True, False, None, 100), (False, False, None, 101), (False, True, None, 102)]),
    "tiny_mt": ("tiny-mt", {}, 12, True, 60.0,   # emb_scale 60 -> ||emb|| > 1 exercises max_norm renorm
                [(True, False, 0, 200), (False, False, 1, 201), (False, True, 3, 202), (True, True, 2, 203)]),
    "c1_dog5m": ("c1", {}, 1, False, 1.0,
                 [(True, False, None, 3), (False, False, None, 4), (False, True, None, 5)]),
    "c3_humanoid48m_e1": ("c3", {"num_envs": 1}, 1, False, 1.0,
                          [(True, False, None, 3), (False, False, None, 4)]),
    "c4_mt80_317m_e1": ("c4", {"num_envs": 1}, 1, False, 1.0,
                        [(True, False, 7, 3), (False, False, 41, 4)]),
    # cfg.episodic: termination head in the rollout (tdmpc2.py:126-136, world_model.py:28,132-141)
    "tiny_episodic": ("tiny", {"episodic": True}, 13, True, 1.0,
                      [(True, False, None, 300), (False, False, None, 301), (False, True, None, 302)]),
    "c1_dog5m_episodic": ("c1", {"episodic": True}, 2, True, 1.0,
                          [(True, False, None, 6), (False, False, None, 7)]),
    # cfg.obs == 'rgb': layers.conv encoder with ShiftAug inside encode() (layers.py:36-71,136-150)
    "tiny_rgb": ("tiny-rgb", {}, 14, True, 1.0,
                 [(True, False, None, 400), (False, False, None, 401), (False, True, None, 402)]),
    # branch / knob coverage of _plan on the test-sized model: no policy-prior trajectories (tdmpc2.py:149 skipped),
    # a one-step horizon (no warm-start shift at :169), and non-default planner knobs with a ragged sample count
    "tiny_nopi": ("tiny", {"num_pi_trajs": 0}, 15, True, 1.0,
                  [(True, False, None, 500), (False, False, None, 501), (False, True, None, 502)]),
    "tiny_h1": ("tiny", {"horizon": 1}, 16, True, 1.0,
                [(True, False, None, 510), (False, False, None, 511), (False, True, None, 512)]),
    "tiny_knobs": ("tiny", {"num_samples": 200, "num_elites": 7, "num_pi_trajs": 5, "temperature": 2.0, "min_std": 0.1,
                            "max_std": 1.5, "num_q": 5, "iterations": 4, "num_bins": 51, "vmin": -5, "vmax": 5}, 17, True, 1.0,
                   [(True, False, None, 520), (False, False, None, 521), (False, True, None, 522)]),
}


# name -> workload whose state-dict layout (keys, shapes) the reference's own WorldModel is recorded for
MODEL_KEY_CASES = {"tiny_rgb_keys": "tiny-rgb"}


def mint_model_keys(out_dir, name, wl):
    """The keys and shapes of the reference model for `wl`, in this project's naming (the harness stores the Q ensemble
    as `_Qs.p.<layer>/<param>`; written here as `_Qs.params.<layer>.<param>`).  build_agent() asserts that the synthetic
    state dict has exactly these keys and load_state_dict() that it has these shapes."""
    cfg = workload(wl)
    agent = rh.build_agent(cfg, synth_state_dict(cfg, seed=2))
    sd = {(("_Qs.params." + k[len("_Qs.p."):].replace("/", ".")) if k.startswith("_Qs.p.") else k): v
          for k, v in agent.model.state_dict().items()}
    keys = sorted(sd)
    np.savez_compressed(os.path.join(out_dir, name + ".npz"), workload=wl, keys=np.array(keys),
                        shapes=np.array([",".join(str(d) for d in sd[k].shape) for k in keys]),
                        torch_version=torch.__version__)
    print(f"{name}: {len(keys)} keys -> tests/golden/{name}.npz")


def main(only=None):
    out_dir = os.path.join(ROOT, "tests", "golden")
    os.makedirs(out_dir, exist_ok=True)
    for name, wl in MODEL_KEY_CASES.items():
        if not only or name in only:
            mint_model_keys(out_dir, name, wl)
    for name, (wl, over, wseed, perturb, emb_scale, calls) in CASES.items():
        if only and name not in only:
            continue
        t = time.time()
        cfg = workload(wl, **over)
        sd = synth_state_dict(cfg, seed=wseed, perturb=perturb, emb_scale=emb_scale)
        term_bias = None
        if cfg.episodic:      # synthetic termination logits all share one sign: centre them (see balance_termination)
            from oracle.plan_oracle import balance_termination
            term_bias = balance_termination(cfg, sd)
        agent = rh.build_agent(cfg, sd)
        g = torch.Generator().manual_seed(1000 + wseed)
        rgb = cfg.get("obs", "state") == "rgb"
        obs_dim = None if rgb else cfg.obs_shape["state"][0]
        rec = dict(workload=wl, overrides=repr(over), weight_seed=wseed, perturb=perturb, emb_scale=emb_scale,
                   weight_checksum=state_dict_checksum(sd), n_calls=len(calls),
                   torch_version=torch.__version__)
        if term_bias is not None:
            rec["term_bias"] = term_bias
        prev_mean = torch.zeros(cfg.horizon, cfg.action_dim)
        for i, (t0, ev, task, seed) in enumerate(calls):
            obs = (torch.randint(0, 256, tuple(cfg.obs_shape["rgb"]), generator=g).float() if rgb
                   else torch.randn(obs_dim, generator=g))
            out = rh.run_plan(agent, obs, seed=seed, t0=t0, eval_mode=ev, task=task, prev_mean=prev_mean)
            rec.update({f"c{i}_obs": obs.numpy(), f"c{i}_t0": t0, f"c{i}_eval_mode": ev,
                        f"c{i}_task": -1 if task is None else task, f"c{i}_seed": seed,
                        f"c{i}_prev_mean": prev_mean.numpy().copy(),
                        f"c{i}_action": out["action"].numpy(), f"c{i}_mean": out["mean"].numpy(),
                        f"c{i}_values": out["values"].squeeze(-1).numpy(),
                        f"c{i}_elite_idx": out["elite_idx"].numpy()})
            prev_mean = out["mean"]
        np.savez_compressed(os.path.join(out_dir, name + ".npz"), **rec)
        print(f"{name}: {len(calls)} calls in {time.time() - t:.1f}s -> tests/golden/{name}.npz")


if __name__ == "__main__":
    main(sys.argv[1:] or None)
