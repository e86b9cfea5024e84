"""Harness that executes the REFERENCE's own planner code on CPU -- TEST INFRASTRUCTURE ONLY.

Works only where a reference checkout is available: TDMPC2_REFERENCE_DIR names its
tdmpc2/ package directory (the one holding tdmpc2.py).  Nothing from the reference
is copied: its modules are imported from where they lie.  The recipe is the one
verified in SURVEY.md section 8(c) / Appendix A:

  1. import-only stubs for `tensordict` (not installable here) so that
     common/layers.py, common/world_model.py and tdmpc2.py import;
  2. a WorldModel subclass that only re-wires construction (the reference's
     own layers.enc / layers.mlp build every head) and replaces the
     tensordict-based `layers.Ensemble` (layers.py:8-33) by
     torch.func.stack_module_state + vmap(functional_call) in eval mode;
  3. the agent is created with TDMPC2.__new__ (its __init__ hard-codes cuda:0,
     tdmpc2.py:20,36,40).

Everything that runs afterwards -- TDMPC2._plan, _estimate_value,
WorldModel.encode/next/reward/pi/Q/task_emb, layers.mlp/NormedLinear/SimNorm,
math.* -- is the reference's unmodified code.
"""
from __future__ import annotations

import copy
import os
import sys
import types
from typing import Dict, Optional

import torch
import torch.nn as nn

REF_DIR = os.environ.get("TDMPC2_REFERENCE_DIR", "")


def available() -> bool:
    return bool(REF_DIR) and os.path.isfile(os.path.join(REF_DIR, "tdmpc2.py"))


_mods = None


def _import_reference():
    global _mods
    if _mods is not None:
        return _mods
    if not available():
        raise RuntimeError(f"reference checkout not found: set TDMPC2_REFERENCE_DIR (now {REF_DIR!r})")
    if "tensordict" not in sys.modules:
        td = types.ModuleType("tensordict"); td.from_modules = None; td.TensorDict = dict
        tdnn = types.ModuleType("tensordict.nn"); tdnn.TensorDictParams = None
        sys.modules["tensordict"], sys.modules["tensordict.nn"] = td, tdnn
    sys.path.insert(0, REF_DIR)
    try:
        from common import layers, init        # noqa: E402  (reference modules)
        from common.world_model import WorldModel
        import tdmpc2 as ref
    finally:
        sys.path.remove(REF_DIR)
    _mods = (layers, init, WorldModel, ref)
    return _mods


def build_agent(cfg, state_dict: Dict[str, torch.Tensor], device="cpu"):
    """Reference TDMPC2 agent on `device` (CPU for the oracle pins; cuda:0 for the on-box GPU baseline) carrying
    `state_dict` (reference key layout)."""
    layers, init, WorldModel, ref = _import_reference()

    class FuncEnsemble(nn.Module):                       # stands in for layers.Ensemble (layers.py:8-33)
        def __init__(self, mods):
            super().__init__()
            self.base = [copy.deepcopy(mods[0]).to("meta").eval()]   # eval(): Q layer 0 has Dropout(0.01)
            p, _ = torch.func.stack_module_state(mods)
            self.p = nn.ParameterDict({k.replace(".", "/"): nn.Parameter(v.detach().clone()) for k, v in p.items()})

        def forward(self, x):
            params = {k.replace("/", "."): v for k, v in self.p.items()}
            f = lambda pp, xx: torch.func.functional_call(self.base[0], pp, (xx,))
            return torch.vmap(f, (0, None), randomness="different")(params, x)

    class HarnessWorldModel(WorldModel):                 # every forward method is inherited unmodified
        def __init__(self, cfg):
            nn.Module.__init__(self)
            self.cfg = cfg
            if cfg.multitask:                            # world_model.py:20-24
                self._task_emb = nn.Embedding(len(cfg.tasks), cfg.task_dim, max_norm=1)
                self.register_buffer("_action_masks", torch.zeros(len(cfg.tasks), cfg.action_dim))
                for i in range(len(cfg.tasks)):
                    self._action_masks[i, :cfg.action_dims[i]] = 1.
            D = cfg.latent_dim + cfg.action_dim + cfg.task_dim
            self._encoder = layers.enc(cfg, out={})
            self._dynamics = layers.mlp(D, 2 * [cfg.mlp_dim], cfg.latent_dim, act=layers.SimNorm(cfg))
            self._reward = layers.mlp(D, 2 * [cfg.mlp_dim], max(cfg.num_bins, 1))
            self._termination = layers.mlp(cfg.latent_dim + cfg.task_dim, 2 * [cfg.mlp_dim], 1) if cfg.episodic else None   # world_model.py:28
            self._pi = layers.mlp(cfg.latent_dim + cfg.task_dim, 2 * [cfg.mlp_dim], 2 * cfg.action_dim)
            qs = [layers.mlp(D, 2 * [cfg.mlp_dim], max(cfg.num_bins, 1), dropout=cfg.dropout) for _ in range(cfg.num_q)]
            self._Qs = FuncEnsemble(qs)
            self.register_buffer("log_std_min", torch.tensor(cfg.log_std_min))
            self.register_buffer("log_std_dif", torch.tensor(cfg.log_std_max) - self.log_std_min)

        def init(self): pass
        def to(self, *a, **k): return nn.Module.to(self, *a, **k)
        def train(self, mode=True): return nn.Module.train(self, mode)

    model = HarnessWorldModel(cfg)
    own = model.state_dict()
    mapped = {}
    for k, v in state_dict.items():
        if k.startswith(("_detach_Qs_params.", "_target_Qs_params.")) or "__" in k:
            continue
        if k.startswith("_Qs.params."):
            k = "_Qs.p." + k[len("_Qs.params."):].replace(".", "/")
        mapped[k] = v
    missing = set(own) - set(mapped)
    extra = set(mapped) - set(own)
    assert not missing and not extra, f"state-dict mismatch: missing={sorted(missing)[:5]} extra={sorted(extra)[:5]}"
    model.load_state_dict(mapped)
    model.eval()
    device = torch.device(device)
    model.to(device)

    agent = ref.TDMPC2.__new__(ref.TDMPC2)
    nn.Module.__init__(agent)
    agent.cfg, agent.device = cfg, device
    agent.model = model
    if cfg.multitask:                                    # tdmpc2.py:35-37
        agent.discount = torch.tensor([ref.TDMPC2._get_discount(agent, ep) for ep in cfg.episode_lengths], device=device)
    else:
        agent.discount = ref.TDMPC2._get_discount(agent, cfg.episode_length)
    agent._prev_mean = torch.nn.Buffer(torch.zeros(cfg.horizon, cfg.action_dim, device=device))
    return agent


@torch.no_grad()
def run_plan(agent, obs: torch.Tensor, *, seed: int, t0: bool, eval_mode: bool,
             task: Optional[int], prev_mean: Optional[torch.Tensor] = None):
    """One unmodified reference `_plan` call under torch.manual_seed(seed),
    recording what it computes (top-k indices/values per iteration are captured
    by wrapping torch.topk for the duration of the call)."""
    if prev_mean is not None:
        agent._prev_mean.copy_(prev_mean)
    rec = {"values": [], "elite_idx": []}
    real_topk = torch.topk

    def spy(x, k, dim=0, **kw):
        out = real_topk(x, k, dim=dim, **kw)
        rec["values"].append(x.clone()); rec["elite_idx"].append(out.indices.clone())
        return out

    torch.manual_seed(seed)
    torch.topk = spy
    try:
        tk = None if task is None else torch.tensor([task])
        # tdmpc2.py:111: act() unsqueezes the observation -- [1, obs_dim] for states, [1, C, 64, 64] for pixels
        o = obs.unsqueeze(0) if agent.cfg.get("obs", "state") == "rgb" else obs.view(1, -1)
        a = agent._plan(o, t0=t0, eval_mode=eval_mode, task=tk)
    finally:
        torch.topk = real_topk
    return dict(action=a.clone(), mean=agent._prev_mean.detach().clone(),
                values=torch.stack(rec["values"]), elite_idx=torch.stack(rec["elite_idx"]))
