"""CPU: host-side logic - configs, vector envs, running statistics, sharding helpers, the multi-rank gradient identity
(world_size-2 gloo)."""
import os
from argparse import Namespace

import numpy as np
import pytest
import torch


def test_config_loader_merges_like_the_reference():
    from xuance_b200.common.common_tools import get_arguments, recursive_dict_update
    assert recursive_dict_update({'a': 1, 'b': 2}, {'a': 3, 'c': 4}) == {'a': 3, 'b': 2, 'c': 4}   # common_tools.py docstring
    c = get_arguments('ppo', 'atari', 'atari', parser_args=Namespace(parallels=64, device="cuda:1"))
    assert c.agent == "PPO" and c.parallels == 64 and c.device == "cuda:1" and c.horizon_size == 128
    assert c.kernels == [8, 4, 3] and c.fc_hidden_sizes == [512] and c.dl_toolbox == "torch"
    for algo, env in (('ppo', 'CartPole-v1'), ('perdqn', 'atari'), ('sac', 'mujoco'), ('qmix', '5m_vs_6m')):
        get_arguments(algo, env, env)    # the 5 BASELINE configs all resolve


@pytest.mark.parametrize("vec", ["DummyVecEnv", "SubprocVecEnv", "ShmSubprocVecEnv"])
def test_vector_env_contract(vec):
    from xuance_b200.environment import make_envs
    from xuance_b200.environment.vector_envs import AlreadySteppingError, NotSteppingError
    envs = make_envs(Namespace(env_id="CartPole-v1", vectorize=vec, parallels=4, env_seed=1))
    obs, infos = envs.reset()
    assert obs.shape == (4, 4) and obs.dtype == np.float32 and len(infos) == 4 and envs.num_envs == 4
    with pytest.raises(NotSteppingError):
        envs.step_wait()
    envs.step_async(np.zeros(4, np.int64))
    with pytest.raises(AlreadySteppingError):
        envs.step_async(np.zeros(4, np.int64))
    envs.step_wait()
    ended = 0
    for t in range(80):        # always pushing left ends every episode quickly
        obs, rew, term, trunc, infos = envs.step(np.zeros(4, np.int64))
        for i in range(4):
            assert infos[i]["episode_step"] >= 1
            if term[i] or trunc[i]:
                ended += 1
                assert "reset_obs" in infos[i] and infos[i]["reset_obs"].shape == (4,)
                assert infos[i]["episode_score"] == infos[i]["episode_step"]       # reward 1 per step
    assert ended >= 4 and rew.dtype == np.float32 and term.dtype == np.bool_
    envs.close()


def test_atari_vector_env_is_uint8():
    from xuance_b200.environment import make_envs
    envs = make_envs(Namespace(env_id="SyntheticAtari", vectorize="Dummy_Atari", parallels=2, env_seed=3))
    obs, _ = envs.reset()
    assert obs.dtype == np.uint8 and obs.shape == (2, 84, 84, 4) and envs.buf_obs.dtype == np.uint8
    envs.close()


def test_running_mean_std_matches_batch_statistics():
    from xuance_b200.common.statistic_tools import RunningMeanStd
    rng = np.random.default_rng(0)
    x = rng.normal(2.0, 3.0, size=(1000, 5)).astype(np.float32)
    rms = RunningMeanStd((5,))
    for i in range(0, 1000, 100):
        rms.update(x[i:i + 100])
    np.testing.assert_allclose(rms.mean, x.mean(0), rtol=1e-3, atol=1e-3)
    np.testing.assert_allclose(rms.std, x.std(0), rtol=1e-3)


def test_running_mean_std_matches_reference():
    """The reference's RunningMeanStd after the same seven updates (tests/golden/running_mean_std.npz)."""
    from xuance_b200.common.statistic_tools import RunningMeanStd
    a = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "running_mean_std.npz"))
    rng = np.random.default_rng(1)
    b = RunningMeanStd((3,))
    for _ in range(7):
        x = rng.normal(size=(8, 3)).astype(np.float32)
        b.update(x)
    assert np.array_equal(a["mean"], b.mean) and np.array_equal(a["var"], b.var) and a["count"] == b.count


def test_stratified_minibatches_partition_every_shard():
    from xuance_b200.torch.utils import stratified_minibatches, shard_bounds
    rng = np.random.default_rng(0)
    b = stratified_minibatches(4096, 4, rng)
    assert len(b) == 4 and all(len(x) == 1024 for x in b)
    assert np.array_equal(np.sort(np.concatenate(b)), np.arange(4096))
    assert shard_bounds(256, 3, 8) == (96, 128)


def _grad_worker(rank, world, port, out):
    """Each rank: PPO loss on ITS half of a global minibatch, scaled by 1/B_total, then a sum all-reduce."""
    import torch.distributed as dist
    from oracle.learners import ppo_clip_terms
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.manual_seed(0)
    B, A = 64, 4
    lin = torch.nn.Linear(8, A + 1)
    x, act = torch.randn(B, 8), torch.randint(0, A, (B,)).float()
    ret, adv, old = torch.randn(B), torch.randn(B), torch.randn(B) * 0.1 - 1.4
    lo, hi = rank * B // world, (rank + 1) * B // world
    o = lin(x[lo:hi])
    a, c, e, _ = ppo_clip_terms(o[:, :A], o[:, A], act[lo:hi], ret[lo:hi], adv[lo:hi], old[lo:hi], 0.2)
    loss = (a - 0.01 * e + 0.25 * c) * (hi - lo) / B          # mean over the GLOBAL batch
    loss.backward()
    flat = torch.cat([p.grad.reshape(-1) for p in lin.parameters()])
    dist.all_reduce(flat)                                       # the one collective
    if rank == 0:
        o = lin(x)
        a, c, e, _ = ppo_clip_terms(o[:, :A], o[:, A], act, ret, adv, old, 0.2)
        lin.zero_grad()
        (a - 0.01 * e + 0.25 * c).backward()
        full = torch.cat([p.grad.reshape(-1) for p in lin.parameters()])
        out.put(float((flat - full).abs().max()))
    dist.destroy_process_group()


def _offpolicy_grad_worker(rank, world, port, out):
    """DQN: mean squared TD error over the GLOBAL batch (dqn_learner.py:41-46; K6 scales by 1/B_total).  QMIX: masked
    squared TD error over the GLOBAL sum(filled) (qmix_learner.py:74-84) - the denominator is itself all-reduced."""
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.manual_seed(0)
    B, A = 48, 5
    net = torch.nn.Linear(6, A)
    x, act = torch.randn(B, 6), torch.randint(0, A, (B,))
    y, filled = torch.randn(B), (torch.rand(B) < 0.7).float()
    lo, hi = rank * B // world, (rank + 1) * B // world
    errs = []
    for kind in ("dqn", "qmix"):
        net.zero_grad()
        pred = net(x[lo:hi]).gather(1, act[lo:hi, None]).squeeze(1)
        if kind == "dqn":
            loss = ((pred - y[lo:hi]) ** 2).sum() / B
        else:
            denom = filled[lo:hi].sum().clone()
            dist.all_reduce(denom)                                   # global sum(filled): one float
            loss = (((pred - y[lo:hi]) * filled[lo:hi]) ** 2).sum() / denom
        loss.backward()
        flat = torch.cat([p.grad.reshape(-1) for p in net.parameters()])
        dist.all_reduce(flat)
        if rank == 0:
            net.zero_grad()
            pred = net(x).gather(1, act[:, None]).squeeze(1)
            full_loss = ((pred - y) ** 2).mean() if kind == "dqn" else (((pred - y) * filled) ** 2).sum() / filled.sum()
            full_loss.backward()
            full = torch.cat([p.grad.reshape(-1) for p in net.parameters()])
            errs.append(float((flat - full).abs().max()))
    if rank == 0:
        out.put(max(errs))
    dist.destroy_process_group()


def _run_world2(worker, port_base):
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = port_base + os.getpid() % 2000
    procs = [ctx.Process(target=worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    err = q.get(timeout=120)
    for p in procs:
        p.join(timeout=60)
    return err


def test_sharded_gradient_identity_gloo_world2():
    """sum over ranks of grad(local rows / B_total) == grad of the global minibatch: the identity the single
    NCCL all-reduce of the flat bucket relies on (K4/K6 take B_total for exactly this)."""
    assert _run_world2(_grad_worker, 29500) < 1e-6


def test_sharded_offpolicy_gradient_identities_gloo_world2():
    """The same identity for the DQN loss and for QMIX's masked loss with an all-reduced denominator."""
    assert _run_world2(_offpolicy_grad_worker, 31500) < 1e-6


def test_vector_envs_agree_step_for_step():
    """Dummy / Subproc / shared-memory Subproc produce identical trajectories for identical seeds and actions."""
    from xuance_b200.environment import make_envs
    rng = np.random.default_rng(0)
    acts = rng.integers(0, 2, size=(60, 6))
    traj = {}
    for vec in ("DummyVecEnv", "SubprocVecEnv", "ShmSubprocVecEnv"):
        envs = make_envs(Namespace(env_id="CartPole-v1", vectorize=vec, parallels=6, env_seed=5))
        obs, _ = envs.reset()
        out = [obs]
        for a in acts:
            obs, rew, term, trunc, infos = envs.step(a)
            out += [obs, rew, term.astype(np.float32), trunc.astype(np.float32),
                    np.array([i["episode_step"] for i in infos], np.float32)]
        traj[vec] = out
        envs.close()
    for vec in ("SubprocVecEnv", "ShmSubprocVecEnv"):
        for a, b in zip(traj["DummyVecEnv"], traj[vec]):
            assert np.array_equal(a, b), vec


def test_shm_vec_env_exposes_shared_block_without_copy():
    from xuance_b200.environment import make_envs
    envs = make_envs(Namespace(env_id="SyntheticAtari", vectorize="ShmSubproc_Atari", parallels=4, env_seed=3))
    envs.reset()
    envs.step_async(np.zeros(4, np.int64))
    obs, *_ = envs.step_wait(copy=False)
    assert obs is envs.buf_obs and obs.dtype == np.uint8 and obs.shape == (4, 84, 84, 4) and obs.any()
    envs.close()


def _ma_fns(n, kw):
    from xuance_b200.environment.ma_envs import SyntheticSMACEnv, XuanCeMultiAgentEnvWrapper
    return [lambda env_seed=0: XuanCeMultiAgentEnvWrapper(SyntheticSMACEnv(seed=env_seed, **kw)) for _ in range(n)]


@pytest.mark.parametrize("context,in_series", [("fork", 1), ("spawn", 2)])
def test_subproc_multi_agent_vector_env_equals_the_dummy_one(context, in_series):
    """SubprocVecMultiAgentEnv (subproc_vec_maenv.py:8-145): the same environments in worker processes give the same
    observations, rewards, terminations, infos (incl. reset_* at episode ends) and state / availability latches as
    DummyVecMultiAgentEnv, step for step; seeds env_seed + i; AlreadyStepping / NotStepping errors; idempotent close."""
    from xuance_b200.environment import REGISTRY_VEC_ENV, make_envs
    from xuance_b200.environment.vector_envs import (DummyVecMultiAgentEnv, SubprocVecMultiAgentEnv, AlreadySteppingError,
                                                     NotSteppingError)
    from helpers import same_structure as _same
    kw = dict(n_agents=3, obs_dim=16, state_dim=20, n_actions=5, episode_limit=6, p_death=0.1)
    n = 4
    dv, sv = DummyVecMultiAgentEnv(_ma_fns(n, kw), 7), SubprocVecMultiAgentEnv(_ma_fns(n, kw), 7, context=context, in_series=in_series)
    try:
        assert REGISTRY_VEC_ENV["Subproc_StarCraft2"] is SubprocVecMultiAgentEnv
        assert sv.num_envs == n and sv.agents == dv.agents and sv.max_episode_steps == dv.max_episode_steps
        assert sv.state_space.shape == dv.state_space.shape and sv.env_info["num_agents"] == 3
        _same(dv.reset(), sv.reset(), "reset")
        with pytest.raises(NotSteppingError):
            sv.step_wait()
        rng = np.random.default_rng(0)
        ends = 0
        for t in range(25):
            acts = [{a: int(rng.choice(np.flatnonzero(dv.buf_avail_actions[e][a]))) for a in dv.agents} for e in range(n)]
            sv.step_async(acts)
            with pytest.raises(AlreadySteppingError):
                sv.step_async(acts)
            r_s = sv.step_wait()
            r_d = dv.step(acts)
            _same(r_d, r_s, "t=%d" % t)
            _same(dv.buf_state, sv.buf_state, "state"), _same(dv.buf_avail_actions, sv.buf_avail_actions, "avail")
            ends += sum("reset_obs" in i for i in r_s[4])
        assert ends >= 4
    finally:
        sv.close(), sv.close(), dv.close()
    cfg = Namespace(env_name="StarCraft2", env_id="5m_vs_6m", vectorize="Subproc_StarCraft2", parallels=2, env_seed=3,
                    episode_limit=5)
    envs = make_envs(cfg)
    try:
        assert isinstance(envs, SubprocVecMultiAgentEnv) and envs.num_agents == 5 and envs.max_episode_steps == 5
        obs, infos = envs.reset()
        assert len(obs) == 2 and obs[0]["agent_0"].shape == (72,) and infos[1]["state"].shape == (98,)
    finally:
        envs.close()


def test_shipped_configs_define_every_key_their_classes_read():
    """Static check (the classes themselves need a GPU): every ``config.X`` an agent / learner of a shipped yaml reads without a
    getattr / hasattr default is a key of basic.yaml + that yaml - ``get_runner(algo, env)`` cannot die on an AttributeError."""
    import glob
    import re
    import yaml
    root = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "xuance_b200")
    rd = lambda *p: open(os.path.join(root, *p)).read()
    base = set(yaml.safe_load(rd("configs", "basic.yaml")))
    per_agent = {"QMIX": ["torch/agents/marl.py", "torch/learners/qmix_learner.py"],
                 "PPO": ["torch/agents/on_policy.py", "torch/agents/ppo_agent.py", "torch/learners/ppo_learner.py"],
                 "PerDQN": ["torch/agents/off_policy.py", "torch/agents/dqn_agent.py", "torch/learners/dqn_learner.py"],
                 "SAC": ["torch/agents/off_policy.py", "torch/agents/sac_agent.py", "torch/learners/sac_learner.py"]}
    common = ["torch/agents/agent.py", "torch/learners/learner.py"]
    seen = set()
    for y in sorted(glob.glob(os.path.join(root, "configs", "*", "*.yaml"))):
        cfg = yaml.safe_load(open(y))
        seen.add(cfg["agent"])
        src = "".join(rd(*f.split("/")) for f in per_agent[cfg["agent"]] + common)
        hard = set(re.findall(r"(?<![a-zA-Z_])(?:self\.)?config\.([a-zA-Z_][a-zA-Z0-9_]*)\b(?!\s*=[^=])", src))
        soft = set(re.findall(r"(?:getattr|hasattr)\((?:self\.)?config,\s*.([a-zA-Z_0-9]+).", src))
        missing = sorted(hard - soft - base - set(cfg))
        assert not missing, (os.path.relpath(y, root), missing)
    assert seen == set(per_agent)
