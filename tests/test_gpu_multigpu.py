"""Environment-axis sharding on real GPUs: 2 ranks (one process per GPU, NCCL) each plan their contiguous block of
environments with the fused kernels; the gathered actions must equal the single-GPU plan of the whole batch BIT FOR BIT
(an environment's arithmetic does not depend on the batch it runs in: tests/test_gpu_multitrip.py).
Needs >= 2 visible GPUs (skipped otherwise): python -m pytest tests/test_gpu_multigpu.py -m gpu on a multi-GPU machine."""
import os
import socket

import pytest
import torch

pytestmark = pytest.mark.gpu


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _problem(E):
    from tdmpc2_b200.config import workload
    from tdmpc2_b200.planner import draw_noise
    from tdmpc2_b200.synth import synth_state_dict
    cfg = workload("tiny-mt", num_envs=E, num_samples=256)      # 2 tiles per environment: the CTA-pair engine runs
    sd = synth_state_dict(cfg, seed=7, perturb=True)
    g = torch.Generator().manual_seed(5)
    obs = torch.randn(E, cfg.obs_shape["state"][0], generator=g)
    prev = 0.3 * torch.randn(E, cfg.horizon, cfg.action_dim, generator=g)
    t0 = torch.tensor([int(i % 2) for i in range(E)], dtype=torch.uint8)
    task = (torch.arange(E) * 3 + 1) % len(cfg.tasks)
    noise = draw_noise(cfg, E, "cpu", generator=torch.Generator().manual_seed(6), reference_order=False)
    return cfg, sd, obs, prev, t0, task, noise


def _plan_block(cfg, sd, obs, prev, t0, task, noise, lo, hi, dev):
    from tdmpc2_b200.planner import Noise, Planner
    E = hi - lo
    cfgl = cfg.replace(num_envs=E)
    pl = Planner(cfgl, E, dev)
    pl.pack(sd)
    mv = lambda t: t.to(dev).contiguous()
    nz = Noise(mv(noise.prior[lo:hi]), mv(noise.r[:, lo:hi]), mv(noise.pi[:, lo:hi]), mv(noise.qidx[:, lo:hi]),
               mv(noise.expo[lo:hi]), mv(noise.final[lo:hi]))
    a, m, _ = pl.plan(mv(obs[lo:hi]), mv(task[lo:hi].to(torch.int32)), mv(t0[lo:hi]), mv(prev[lo:hi]), nz)
    torch.cuda.synchronize(dev)
    return a, m


def _worker(rank, world, port, E, out_path):
    import torch.distributed as dist
    from tdmpc2_b200.sharded import ShardedActor
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        cfg, sd, obs, prev, t0, task, noise = _problem(E)
        actor = ShardedActor(lambda o, t, k: None, E)
        a, m = _plan_block(cfg, sd, obs, prev, t0, task, noise, actor.lo, actor.hi, dev)
        allact = actor.gather(a)                                   # the ONE collective of a sharded plan()
        assert allact.shape == (E, cfg.action_dim)
        if rank == 0:
            torch.save(allact.cpu(), out_path)
    finally:
        dist.destroy_process_group()


def test_two_rank_shard_equals_single_rank(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    E, out = 8, str(tmp_path / "gathered.pt")
    mp.spawn(_worker, args=(2, _free_port(), E, out), nprocs=2, join=True)
    gathered = torch.load(out)
    cfg, sd, obs, prev, t0, task, noise = _problem(E)
    a, _ = _plan_block(cfg, sd, obs, prev, t0, task, noise, 0, E, torch.device("cuda", 0))
    assert torch.equal(gathered, a.cpu()), (gathered - a.cpu()).abs().max()
