#!/usr/bin/env python
"""Secondary measurements for BASELINE configs 3-5 (parity-test cases, not the headline): sample + update throughput of
DQN+PER (2^20-transition HBM replay, B=512), SAC (1M replay, B=1024) and QMIX (5 agents x 72-d, T=60, 32 episodes)
on one B200, next to the oracle port of the reference's torch-CPU path on the host.  Also continuous-action PPO
(ppo_gaussian: configs/ppo/mujoco.yaml shapes, one GPU).  Prints one JSON object.

    python tools/algo_bench.py [--iters 200] [--cpu-iters 5] [--no-cpu] [--graph] [--only perdqn,sac,qmix,ppo_gaussian]
    torchrun --nnodes=1 --nproc-per-node G --master-addr 127.0.0.1 tools/algo_bench.py --no-cpu --graph    (G GPUs)

Multi-GPU (BASELINE configs 3 and 5 are multi-GPU configurations): one process per GPU; the replay is sharded (envs / episodes
per rank), every update takes batch/G rows from every rank, the gradient bucket (+ logged statistics) is all-reduced once per
update inside the captured graph; the time of an update is the max over ranks (barrier + synchronize on both sides) and the
global batch is fixed (strong scaling).
"""
import argparse
import json
import os
import sys
import time
from argparse import Namespace

import numpy as np
import torch
import torch.nn as nn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
RANK, WORLD, LOCAL = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))
DEV = "cuda:%d" % LOCAL


def timed(fn, iters, warm=10):
    import torch.distributed as dist
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    if WORLD > 1:
        dist.barrier()
        torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1) / 1e3 / iters], dtype=torch.float64, device=DEV)
    if WORLD > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def cpu_timed(fn, iters):
    fn()
    t0 = time.perf_counter()
    for _ in range(iters):
        fn()
    return (time.perf_counter() - t0) / iters


def bench_perdqn(args):
    from xuance_b200.common import PerOffPolicyBuffer, Box, Discrete, BaseCallback
    from xuance_b200.torch.rl_models import Basic_CNN, DeepQNetwork
    from xuance_b200.torch.learners import PerDQN_Learner
    N, S, B, A = 16 // WORLD, 65536, 512 // WORLD, 4          # this rank's envs and its share of the 512-row batch
    buf = PerOffPolicyBuffer(Box(0, 255, (84, 84, 4), np.uint8), Discrete(A), None, N, N * S, B, alpha=0.5, device=DEV)
    g = torch.Generator(device=DEV).manual_seed(RANK)
    for t in range(64):   # real stores through K1 + K5 insert, then the rest of the ring is declared filled
        o = torch.randint(0, 256, (N, 84, 84, 4), dtype=torch.uint8, device=DEV, generator=g)
        buf.store(o, torch.randint(0, A, (N,), device=DEV), torch.randn(N, device=DEV), torch.zeros(N, device=DEV), o)
    buf.size = S
    leaves = torch.rand((N, S), device=DEV) + 0.01
    cap = buf._it_capacity
    buf._it_sum[:, cap:cap + S], buf._it_min[:, cap:cap + S] = leaves, leaves
    lvl = cap // 2
    while lvl >= 1:
        buf._it_sum[:, lvl:2 * lvl] = buf._it_sum[:, 2 * lvl:4 * lvl:2] + buf._it_sum[:, 2 * lvl + 1:4 * lvl:2]
        buf._it_min[:, lvl:2 * lvl] = torch.minimum(buf._it_min[:, 2 * lvl:4 * lvl:2], buf._it_min[:, 2 * lvl + 1:4 * lvl:2])
        lvl //= 2
    rep = Basic_CNN(input_shape=(84, 84, 4), kernels=[8, 4, 3], strides=[4, 2, 1], filters=[32, 64, 64], activation=nn.ReLU, device=DEV)
    model = DeepQNetwork(rep, [512], Discrete(A), None, None, nn.ReLU, DEV).to(DEV)
    cfg = Namespace(distributed_training=WORLD > 1, episode_length=1000, use_grad_clip=False, grad_clip_norm=0.5, device=DEV,
                    model_dir="/tmp/x", running_steps=10**7, parallels=N * WORLD, learning_rate=1e-4, gamma=0.99,
                    sync_frequency=500, start_training=0, training_frequency=1, compute=args.compute, tc_planes=3)
    if args.compute != "fp32":
        rep.tc_planes = 3
        rep.set_compute(args.compute)
    cfg.use_cuda_graph = args.graph
    lrn = PerDQN_Learner(cfg, model, BaseCallback())

    def step():
        s = buf.sample(0.4)
        td, _ = lrn.update(sync=False, **s)
        buf.update_priorities(s["step_choices"], td)

    dt = timed(step, args.iters)
    out = {"config": "DQN+PER, 2^20-transition uint8 HBM replay (59 GB), 16 envs, B=512 (global), encoder compute=%s" % args.compute,
           "gpu_updates_per_s": 1 / dt, "gpu_transitions_per_s": B * WORLD / dt, "gpu_ms_per_update": dt * 1e3}
    if not args.no_cpu:
        from oracle.replay import PerReplayOracle
        from oracle.nets import DeepQNetworkOracle
        from oracle.learners import DQNLearnerOracle
        Sc = 1024   # the reference stores float32 image replay: 2^20 would need 226 GB of host RAM (SURVEY row P2)
        ob = PerReplayOracle((84, 84, 4), (), N, N * Sc, B, alpha=0.5, obs_dtype=np.uint8)
        rng = np.random.default_rng(0)
        for t in range(Sc):
            o = rng.integers(0, 256, size=(N, 84, 84, 4), dtype=np.uint8)
            ob.store(o, rng.integers(0, A, N), rng.normal(size=N).astype(np.float32), np.zeros(N, bool), o)
        ol = DQNLearnerOracle(DeepQNetworkOracle(A), per=True)

        def cstep():
            s = ob.sample(0.4)
            td, _ = ol.update(**s)
            ob.update_priorities(s["step_choices"], td)

        cdt = cpu_timed(cstep, args.cpu_iters)
        out.update(cpu_updates_per_s=1 / cdt, cpu_ms_per_update=cdt * 1e3, cpu_replay_capacity=N * Sc,
                   cpu_threads=torch.get_num_threads(), speedup=cdt / dt)
    return out


def bench_sac(args):
    from copy import deepcopy
    from xuance_b200.common import DummyOffPolicyBuffer, Box, BaseCallback
    from xuance_b200.torch.rl_models import Basic_Identical, SAC_GaussianActor, TwinActionValueCritic, SoftActorCritic
    from xuance_b200.torch.learners import REGISTRY_Learners
    N, S, B, od, ad = 4, 250000 // WORLD, 1024 // WORLD, 17, 6
    aspace = Box(-1, 1, (ad,), np.float32)
    buf = DummyOffPolicyBuffer(Box(-10, 10, (od,), np.float32), aspace, None, N, N * S, B, device=DEV)
    buf._obs.normal_(), buf._next_obs.normal_(), buf._act_rows.uniform_(-1, 1), buf._fields.normal_()
    buf.size = S
    rep = Basic_Identical((od,), device=DEV)
    model = SoftActorCritic(SAC_GaussianActor(rep, [256, 256], aspace, None, None, nn.LeakyReLU, nn.Tanh, DEV),
                            TwinActionValueCritic(deepcopy(rep), aspace, [256, 256], None, None, nn.LeakyReLU, DEV)).to(DEV)
    cfg = Namespace(distributed_training=WORLD > 1, episode_length=1000, use_grad_clip=False, grad_clip_norm=0.5, device=DEV,
                    model_dir="/tmp/x", running_steps=10**6, parallels=N, start_training=0, training_frequency=1,
                    learning_rate_actor=1e-3, learning_rate_critic=1e-3, tau=0.005, gamma=0.99, alpha=0.2,
                    use_automatic_entropy_tuning=True)
    cfg.use_cuda_graph = args.graph
    lrn = REGISTRY_Learners["SAC_Learner"](cfg, model, BaseCallback())
    dt = timed(lambda: lrn.update(sync=False, **buf.sample()), args.iters)
    out = {"config": "SAC, 17-d obs / 6-d act, 1M replay, B=1024 (global), MLP 256-256", "gpu_updates_per_s": 1 / dt,
           "gpu_transitions_per_s": B * WORLD / dt, "gpu_ms_per_update": dt * 1e3}
    if not args.no_cpu:
        from oracle.replay import UniformReplayOracle
        from oracle.sac import SACModelOracle, SACLearnerOracle
        ob = UniformReplayOracle((od,), (ad,), N, N * S, B)
        ob.observations[...] = np.random.default_rng(0).normal(size=ob.observations.shape)
        ob.size = S
        ol = SACLearnerOracle(SACModelOracle(od, ad))
        cdt = cpu_timed(lambda: ol.update(torch.randn(B, ad), torch.randn(B, ad), **ob.sample()), max(args.cpu_iters, 20))
        out.update(cpu_updates_per_s=1 / cdt, cpu_ms_per_update=cdt * 1e3, cpu_threads=torch.get_num_threads(), speedup=cdt / dt)
    return out


def bench_qmix(args, Be=32):
    from helpers import qmix_episode_stream
    from test_gpu_qmix import _product_model, _buffers
    from xuance_b200.common import BaseCallback
    from xuance_b200.torch.learners import REGISTRY_Learners
    n, od, A, S, T = 5, 72, 12, 98, 60
    Be_global, Be = Be, Be // WORLD                              # this rank's share of the episodes of an update
    keys, grouping, model = _product_model(n, od, A, S, device=DEV)
    n_envs, C = 8, max(256, 2 * Be)
    prod, ob = _buffers(keys, od, A, S, n_envs, C, Be, T, device=DEV)
    for ev in qmix_episode_stream(np.random.default_rng(RANK), keys, n_envs, T, od, A, S, C // n_envs):
        if ev[0] == 'store':
            prod.store(**ev[1]), ob.store(**ev[1])
        else:
            prod.finish_path(ev[1], **ev[2]), ob.finish_path(ev[1], **ev[2])
    cfg = Namespace(distributed_training=WORLD > 1, episode_length=T, use_grad_clip=False, grad_clip_norm=10.0, device=DEV,
                    model_dir="/tmp/x", running_steps=10**7, parallels=n_envs, use_parameter_sharing=True, use_rnn=True,
                    use_actions_mask=False, learning_rate=7e-4, sync_frequency=200, double_q=True, n_epochs=1,
                    start_training=0, gamma=0.99)
    cfg.use_cuda_graph = args.graph
    lrn = REGISTRY_Learners["QMIX_Learner"](cfg, grouping, model, BaseCallback())
    dt = timed(lambda: lrn.update(prod.sample(), sync=False), args.iters)
    out = {"config": f"QMIX, 5 agents x 72-d, S=98, A=12, T=60, {Be_global} episodes/update (global), GRU 64 + mixer 32/32",
           "gpu_updates_per_s": 1 / dt, "gpu_agent_steps_per_s": Be_global * T * n / dt, "gpu_ms_per_update": dt * 1e3}
    if not args.no_cpu:
        from oracle.qmix import QMIXModelOracle, QMIXLearnerOracle
        ol = QMIXLearnerOracle(QMIXModelOracle(n, od, A, S), keys, detach_q_eval=False)
        cdt = cpu_timed(lambda: ol.update(ob.sample()), max(args.cpu_iters, 10))
        out.update(cpu_updates_per_s=1 / cdt, cpu_ms_per_update=cdt * 1e3, cpu_threads=torch.get_num_threads(), speedup=cdt / dt)
    return out


def _card():
    """Name and power limit of the card the numbers were measured on (read-only query)."""
    import subprocess
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(LOCAL), "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return {"gpu": torch.cuda.get_device_name(LOCAL), "nvidia_smi_name_power_limit": q}


def bench_ppo_gaussian(args):
    """PPO-Clip with a Gaussian policy (K4-G in every update): configs/ppo/mujoco.yaml - 17-d obs, 6-d action, Basic_Identical
    + MLP 256-256, 16 epochs x 8 minibatches of a 16 x 256 rollout (B = 512) - and a large-batch row (256 x 256 rollout,
    B = 8192).  train_epochs runs on a filled buffer (GAE included); env-steps/s = rollout steps consumed per second of
    train_epochs.  The CPU arm is the oracle's update (torch on the host) at the same B."""
    from xuance_b200.common import Box
    from xuance_b200.common.common_tools import get_arguments
    from xuance_b200.torch.agents import PPO_Agent
    from oracle.gaussian import GaussianActorCriticOracle, PPOGaussianLearnerOracle
    od, ad = 17, 6
    out = {"card": _card()}
    for name, parallels in (("mujoco_B512", 16), ("large_B8192", 256)):
        cfg = get_arguments("ppo", "mujoco", parser_args=Namespace(device=DEV, parallels=parallels, logger=None,
                                                                    use_cuda_graph=args.graph, model_dir="/tmp/xb_bench"))
        agent = PPO_Agent(cfg, None, Box(-np.inf, np.inf, (od,), np.float32), Box(-1, 1, (ad,), np.float32))
        mem, N, T = agent.memory, agent.n_envs, agent.horizon_size
        g = torch.Generator(device=DEV).manual_seed(0)
        for t in range(T):
            mem.store(torch.randn((N, od), device=DEV, generator=g), torch.rand((N, ad), device=DEV, generator=g) * 2 - 1,
                      torch.randn(N, device=DEV, generator=g), torch.randn(N, device=DEV, generator=g),
                      torch.zeros(N, device=DEV), {"old_logp": torch.randn(N, device=DEV, generator=g) - 5.0})
        mem.finish_paths(np.zeros(N, np.float32))
        B = agent.batch_size
        n_upd = cfg.n_epochs * cfg.n_minibatch
        reps = max(1, args.iters // n_upd)
        dt = timed(lambda: agent.train_epochs(cfg.n_epochs), reps, warm=2)
        row = {"config": "PPO Gaussian, %d envs x %d steps, %d epochs x %d minibatches, B=%d, MLP 256-256, cuda_graph=%s"
                         % (N, T, cfg.n_epochs, cfg.n_minibatch, B, bool(args.graph)),
               "gpu_updates_per_s": n_upd / dt, "gpu_ms_per_update": dt / n_upd * 1e3,
               "gpu_train_epochs_s": dt, "gpu_env_steps_per_s": N * T / dt}
        if not args.no_cpu:
            torch.manual_seed(0)
            ol = PPOGaussianLearnerOracle(GaussianActorCriticOracle(od, ad), learning_rate=4e-4, ent_coef=0.0)
            rng = np.random.default_rng(0)
            s = {"obs": rng.normal(size=(B, od)).astype(np.float32), "actions": rng.uniform(-1, 1, (B, ad)).astype(np.float32),
                 "returns": rng.normal(size=B).astype(np.float32), "advantages": rng.normal(size=B).astype(np.float32),
                 "aux_batch": {"old_logp": (rng.normal(size=B) - 5.0).astype(np.float32)}}
            cdt = cpu_timed(lambda: ol.update(**s), max(args.cpu_iters, 20))
            row.update(cpu_updates_per_s=1 / cdt, cpu_ms_per_update=cdt * 1e3, cpu_threads=torch.get_num_threads(),
                       speedup=cdt / (dt / n_upd))
        out[name] = row
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--cpu-iters", type=int, default=5)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--only", default="", help="comma-separated subset of perdqn,sac,qmix,ppo_gaussian")
    ap.add_argument("--graph", action="store_true", help="capture the learners' device update in a CUDA graph")
    ap.add_argument("--compute", default="fp32", choices=["fp32", "tc"], help="pixel encoder of the PER-DQN network")
    args = ap.parse_args()
    torch.cuda.set_device(LOCAL)
    torch.manual_seed(0)          # identical initial weights on every rank
    if WORLD > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device(DEV))
        args.no_cpu = True
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.benchmark = True
    only = set(x for x in args.only.split(",") if x)
    res = {}
    if not only or "perdqn" in only:
        res["perdqn"] = bench_perdqn(args)
    if not only or "sac" in only:
        res["sac"] = bench_sac(args)
    if not only or "qmix" in only:
        res["qmix"] = bench_qmix(args)
        res["qmix_4096"] = bench_qmix(Namespace(**{**vars(args), "iters": 20, "no_cpu": True}), Be=1024)
    if (not only or "ppo_gaussian" in only) and WORLD == 1:
        res["ppo_gaussian"] = bench_ppo_gaussian(args)
    res["cuda_graph"] = bool(args.graph)
    res["n_gpus"] = WORLD
    if RANK == 0:
        print(json.dumps(res))
    if WORLD > 1:
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
