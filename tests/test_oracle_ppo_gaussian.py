"""CPU: continuous-action PPO without a GPU - the Gaussian oracle reproduces the reference (tests/golden/ppo_gaussian_update.npz,
written by tests/golden/make_golden_ppo_gaussian.py), the MuJoCo-shaped synthetic env keeps the vector-env contract, and the
K4-G / K10-G entry points validate their arguments before touching the device."""
import ctypes
import os

import numpy as np
import torch

from oracle.gaussian import GaussianActorCriticOracle, PPOGaussianLearnerOracle

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _golden_samples(g, it):
    return {"obs": g[f"in{it}/obs"], "actions": g[f"in{it}/actions"], "returns": g[f"in{it}/returns"],
            "advantages": g[f"in{it}/advantages"], "aux_batch": {"old_logp": g[f"in{it}/old_logp"]}}


def test_ppo_gaussian_update_matches_reference():
    g = np.load(os.path.join(G, "ppo_gaussian_update.npz"), allow_pickle=False)
    obs_dim, act_dim, B, seed = (int(x) for x in g["cfg"])
    torch.manual_seed(seed)
    model = GaussianActorCriticOracle(obs_dim, act_dim, actor_hidden=(64, 64), critic_hidden=(64, 64))
    for k, v in model.state_dict().items():   # same construction order => same initial weights as the reference
        d = g[f"init_digest/{k}"]
        np.testing.assert_allclose(v.double().abs().sum().item(), d[1], rtol=1e-6, err_msg=k)
        np.testing.assert_allclose(v.double().sum().item(), d[0], rtol=0, atol=1e-6 * d[1], err_msg=k)
    lrn = PPOGaussianLearnerOracle(model, end_factor_lr_decay=0.5, total_iters=int(g["total_iters"]))
    for it in range(2):
        info = lrn.update(**_golden_samples(g, it))
        got = [info["actor_loss"], info["critic_loss"], info["entropy"], info["learning_rate"], info["predict_value"],
               float(info["clip_ratio"])]
        np.testing.assert_allclose(got, g["infos"][it], rtol=1e-5, atol=1e-7)
    assert 0.0 < g["infos"][0][5] < 1.0          # the fixture exercises both sides of the clip
    for k, v in model.state_dict().items():
        flat = v.detach().reshape(-1)
        np.testing.assert_allclose(flat[:64].numpy(), g[f"final_head/{k}"], rtol=1e-4, atol=1e-7, err_msg=k)
        np.testing.assert_allclose(flat.double().abs().sum().item(), g[f"final_digest/{k}"][1], rtol=1e-6, err_msg=k)


def test_synthetic_mujoco_env_contract():
    from argparse import Namespace
    from xuance_b200.environment import REGISTRY_ENV, SyntheticMuJoCoEnv, make_envs
    assert REGISTRY_ENV["SyntheticMuJoCo"] is SyntheticMuJoCoEnv
    envs = make_envs(Namespace(env_id="SyntheticMuJoCo", vectorize="DummyVecEnv", parallels=3, env_seed=4))
    assert envs.observation_space.shape == (17,) and envs.action_space.shape == (6,)
    assert np.all(envs.action_space.low == -1.0) and np.all(envs.action_space.high == 1.0)
    obs, _ = envs.reset()
    assert obs.shape == (3, 17) and obs.dtype == np.float32
    trace = []
    for t in range(SyntheticMuJoCoEnv.max_episode_steps):
        nxt, rew, term, trunc, infos = envs.step(np.full((3, 6), 0.1, np.float32))
        assert nxt.shape == (3, 17) and nxt.dtype == np.float32 and rew.shape == (3,)
        assert not term.any() and trunc.all() == (t + 1 == SyntheticMuJoCoEnv.max_episode_steps)
        trace.append(rew.copy())
    assert all("reset_obs" in i and i["episode_step"] == SyntheticMuJoCoEnv.max_episode_steps for i in infos)
    # seeded: two envs built with the same seed produce the same observations and rewards
    a, b = SyntheticMuJoCoEnv(seed=7), SyntheticMuJoCoEnv(seed=7)
    oa, ob = a.reset()[0], b.reset()[0]
    assert np.array_equal(oa, ob)
    act = np.linspace(-3, 3, 6).astype(np.float32)
    assert a.step(act)[:2][1] == b.step(act)[:2][1]
    # actions are clipped to the bounds inside the env; the best action W o scores 0
    env = SyntheticMuJoCoEnv(seed=1)
    o = env.reset()[0]
    r_far = env.step(np.full(6, 50.0, np.float32))[1]
    env2 = SyntheticMuJoCoEnv(seed=1)
    env2.reset()
    assert env2.step(np.ones(6, np.float32))[1] == r_far
    env3 = SyntheticMuJoCoEnv(seed=1)
    o3 = env3.reset()[0]
    target = env3.W @ o3
    if np.all(np.abs(target) <= 1.0):
        assert env3.step(target)[1] == 0.0


def test_gaussian_entry_points_validate_before_touching_the_device():
    from xuance_b200 import _lib
    lib = _lib.load()
    P = ctypes.c_void_p
    junk = P(0x1000)          # never dereferenced: validation fails first
    EINVAL, ERANGE = -1, -3

    def loss(B=8, D=6, B_total=8, kind=0, old=junk, mu=junk, col=junk):
        return lib.xb_ppo_gaussian_loss_fwd_bwd(mu, junk, junk, junk, old, junk, junk, B, D, B_total, 0.2, 0.25, 0.01, kind,
                                                junk, junk, junk, junk, junk, col, None)
    assert loss(mu=None) == EINVAL
    assert loss(col=None) == EINVAL                 # the per-dimension scratch is required
    assert loss(old=None) == EINVAL                 # PPO-Clip needs old_logp
    assert loss(B=0) == EINVAL and loss(B=-3, B_total=8) == EINVAL
    assert loss(B=8, B_total=4) == EINVAL           # B_total < B
    assert loss(D=0) == EINVAL
    assert loss(D=65) == ERANGE
    assert loss(kind=2) == EINVAL and loss(kind=-1) == EINVAL
    assert lib.xb_gaussian_scratch_doubles(6) == 6 * lib.xb_gaussian_scratch_doubles(1) > 0
    assert lib.xb_gaussian_scratch_doubles(0) == 0 and lib.xb_gaussian_scratch_doubles(65) == 0

    def act(mu=junk, log_std=junk, N=8, D=6, out=junk, logp=junk):
        return lib.xb_gaussian_act(mu, log_std, junk, None, N, D, out, logp, None, None)
    assert act(mu=None) == EINVAL and act(log_std=None) == EINVAL
    assert act(N=0) == EINVAL and act(D=0) == EINVAL
    assert act(D=65) == ERANGE
    assert act(out=None, logp=None) == EINVAL       # no output requested
