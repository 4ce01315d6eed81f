"""GPU: continuous-action PPO - K4-G (xb_ppo_gaussian_loss_fwd_bwd) and K10-G (xb_gaussian_act) against torch autograd /
torch.distributions on the CPU, PPO_Learner on a Gaussian policy against the oracle and the reference fixture, the device
rollout's vector-action staging, CUDA-graph replay, and the MuJoCo-shaped runners end to end."""
import os
from argparse import Namespace

import numpy as np
import pytest
import torch
from torch.distributions import Normal

from helpers import ppo_config
from oracle.gaussian import GaussianActorCriticOracle, PPOGaussianLearnerOracle

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _inputs(rng, B, D, case):
    mu = np.tanh(rng.normal(size=(B, D))).astype(np.float32)
    log_std = (rng.normal(size=D) * 0.3 - 1.0).astype(np.float32)
    act = (mu + np.exp(log_std) * rng.normal(size=(B, D))).astype(np.float32)
    logp = Normal(torch.tensor(mu), torch.tensor(log_std).exp()).log_prob(torch.tensor(act)).sum(-1).numpy()
    spread = 1.0 if case == "clip_heavy" else 0.1
    old = (logp + rng.normal(size=B) * spread).astype(np.float32)
    value = rng.normal(size=B).astype(np.float32)
    ret = rng.normal(size=B).astype(np.float32)
    adv = np.zeros(B, np.float32) if case == "zero_adv" else rng.normal(size=B).astype(np.float32)
    adv[:3] = 0.0
    return mu, log_std, act, old, adv, ret, value


def _torch_reference(mu, log_std, act, old, adv, ret, value, clip, vf, ent, kind, B_total=None):
    """ppo_learner.py:46-60 (kind 0) / a2c_learner.py:46-52 (kind 1) on a Normal policy, autograd on the CPU."""
    mt, lt, vt = (torch.tensor(x, requires_grad=True) for x in (mu, log_std, value))
    dist = Normal(mt, lt.exp())
    logp = dist.log_prob(torch.tensor(act)).sum(-1)
    B = mu.shape[0]
    scale = B / (B_total or B)
    if kind == 0:
        ratio = (logp - torch.tensor(old)).exp()
        s1 = ratio.clamp(1 - clip, 1 + clip) * torch.tensor(adv)
        s2 = torch.tensor(adv) * ratio
        a_loss = -torch.minimum(s1, s2).mean() * scale
        cr = ((ratio < 1 - clip).sum() + (ratio > 1 + clip).sum()).item() / (B_total or B)
    else:
        a_loss = -(torch.tensor(adv) * logp).mean() * scale
        cr = 0.0
    c_loss = torch.nn.functional.mse_loss(vt, torch.tensor(ret)) * scale
    e_loss = dist.entropy().sum(-1).mean() * scale
    loss = a_loss - ent * e_loss + vf * c_loss
    loss.backward()
    stats = [a_loss.item(), c_loss.item(), e_loss.item(), vt.mean().item() * scale, cr, loss.item()]
    return stats, mt.grad.numpy(), vt.grad.numpy(), lt.grad.numpy()


def _k4g(mu, log_std, act, old, adv, ret, value, clip, vf, ent, kind, B_total=None, scratch=None, col=None):
    from xuance_b200 import _lib
    B, D = mu.shape
    t = [torch.tensor(x, device=DEV) for x in (mu, log_std, value, act, old, adv, ret)]
    dmu, dv = torch.empty((B, D), device=DEV), torch.empty(B, device=DEV)
    dls, stats = torch.empty(D, device=DEV), torch.zeros(8, device=DEV)
    scratch = _lib.scratch(torch.device(DEV)) if scratch is None else scratch
    if col is None:
        col = torch.zeros(_lib.load().xb_gaussian_scratch_doubles(D), dtype=torch.float64, device=DEV)
    _lib.call("xb_ppo_gaussian_loss_fwd_bwd", *[_lib.ptr(x) for x in t], B, D, B_total or B, clip, vf, ent, kind,
              _lib.ptr(dmu), _lib.ptr(dv), _lib.ptr(dls), _lib.ptr(stats), _lib.ptr(scratch), _lib.ptr(col))
    return stats.cpu().numpy(), dmu.cpu().numpy(), dv.cpu().numpy(), dls.cpu().numpy()


@pytest.mark.parametrize("B,D,case,kind", [(8192, 6, "plain", 0), (512, 6, "clip_heavy", 0), (257, 17, "plain", 0),
                                           (33, 1, "zero_adv", 0), (64, 64, "plain", 0), (512, 6, "plain", 1),
                                           (257, 17, "zero_adv", 1)])
def test_ppo_gaussian_loss_kernel_matches_torch_autograd(B, D, case, kind):
    from xuance_b200 import _lib
    rng = np.random.default_rng(B * 100 + D)
    inp = _inputs(rng, B, D, case)
    clip, vf, ent = 0.2, 0.25, 0.01
    ref_stats, g_mu, g_v, g_ls = _torch_reference(*inp, clip, vf, ent, kind)
    scratch = _lib.scratch(torch.device(DEV))
    col = torch.zeros(_lib.load().xb_gaussian_scratch_doubles(D), dtype=torch.float64, device=DEV)
    first = _k4g(*inp, clip, vf, ent, kind, scratch=scratch, col=col)
    second = _k4g(*inp, clip, vf, ent, kind, scratch=scratch, col=col)     # the ticket must re-arm
    for a, b in zip(first, second):
        assert np.array_equal(a, b)                                      # bit-identical run to run
    s, dmu, dv, dls = second
    for i in (0, 1, 2, 3, 5):
        np.testing.assert_allclose(s[i], ref_stats[i], rtol=1e-4, atol=1e-6, err_msg="stat %d" % i)
    np.testing.assert_allclose(s[4], ref_stats[4], rtol=0, atol=1e-7)
    if case == "clip_heavy":
        assert s[4] > 0.2
    assert s[6] == 0.0 and s[7] == 0.0
    np.testing.assert_allclose(dmu, g_mu, rtol=1e-4, atol=1e-9)
    np.testing.assert_allclose(dv, g_v, rtol=1e-5, atol=1e-10)
    np.testing.assert_allclose(dls, g_ls, rtol=1e-4, atol=1e-6)     # torch sums the B rows in float32, K4-G in double


def test_ppo_gaussian_loss_sharding_identity():
    """Two half-batch calls with B_total = B sum to the whole-batch call (a rank's shard gives correctly scaled gradients)."""
    rng = np.random.default_rng(3)
    B, D = 1000, 6
    inp = _inputs(rng, B, D, "plain")
    full = _k4g(*inp, 0.2, 0.25, 0.01, 0)
    h = B // 2
    rows = lambda sl: [x if i == 1 else x[sl] for i, x in enumerate(inp)]      # inp[1] is log_std [D]: shared
    lo = _k4g(*rows(slice(0, h)), 0.2, 0.25, 0.01, 0, B_total=B)
    hi = _k4g(*rows(slice(h, B)), 0.2, 0.25, 0.01, 0, B_total=B)
    np.testing.assert_allclose(lo[0][:6] + hi[0][:6], full[0][:6], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(np.concatenate([lo[1], hi[1]]), full[1], rtol=1e-6, atol=0)
    np.testing.assert_allclose(np.concatenate([lo[2], hi[2]]), full[2], rtol=1e-6, atol=0)
    np.testing.assert_allclose(lo[3] + hi[3], full[3], rtol=1e-5, atol=1e-6)


def test_gaussian_act_kernel():
    from xuance_b200.torch.utils.rollout_glue import gaussian_act
    rng = np.random.default_rng(0)
    for N, D in ((16, 6), (300, 17), (5, 1), (7, 64)):
        mu = torch.tensor(np.tanh(rng.normal(size=(N, D))).astype(np.float32), device=DEV)
        log_std = torch.tensor((rng.normal(size=D) * 0.5 - 1).astype(np.float32), device=DEV)
        noise = torch.tensor(rng.normal(size=(N, D)).astype(np.float32), device=DEV)
        out = gaussian_act(mu, log_std, noise=noise, entropy=torch.empty(N, device=DEV))
        sigma = log_std.exp().cpu().numpy()
        want = mu.cpu().numpy() + noise.cpu().numpy() * sigma            # float32 NumPy: product, then sum
        assert want.dtype == np.float32 and np.array_equal(out["actions"].cpu().numpy(), want)
        dist = Normal(mu.cpu(), log_std.cpu().exp())
        a = out["actions"].cpu()
        np.testing.assert_allclose(out["logp"].cpu().numpy(), dist.log_prob(a).sum(-1).numpy(), rtol=1e-5, atol=1e-5)
        np.testing.assert_allclose(out["entropy"].cpu().numpy(), dist.entropy().sum(-1).numpy(), rtol=1e-5)
        det = gaussian_act(mu, log_std)
        assert torch.equal(det["actions"], mu)
        np.testing.assert_allclose(det["logp"].cpu().numpy(), dist.log_prob(mu.cpu()).sum(-1).numpy(), rtol=1e-5)
        forced = torch.tensor(rng.uniform(-1, 1, (N, D)).astype(np.float32), device=DEV)
        f = gaussian_act(mu, log_std, forced_actions=forced)
        assert torch.equal(f["actions"], forced)
        np.testing.assert_allclose(f["logp"].cpu().numpy(), dist.log_prob(forced.cpu()).sum(-1).numpy(), rtol=1e-5, atol=1e-5)
    # torch.randn noise: the draws follow Normal(mu, sigma)
    N, D = 200000, 6
    mu = torch.linspace(-0.5, 0.5, D, device=DEV).repeat(N, 1).contiguous()
    log_std = torch.tensor([-2.0, -1.0, -0.5, 0.0, 0.3, -1.5], device=DEV)
    a = gaussian_act(mu, log_std, noise=torch.randn((N, D), device=DEV))["actions"].double()
    sigma = log_std.double().exp()
    assert torch.all((a.mean(0) - mu[0].double()).abs() <= 5 * sigma / N ** 0.5)      # 5 standard errors
    np.testing.assert_allclose(a.std(0).cpu().numpy(), sigma.cpu().numpy(), rtol=0.01)


def _product_gaussian_model(obs_dim, act_dim, hidden=(64, 64)):
    from xuance_b200.torch.rl_models import Basic_Identical, GaussianActorHead, ValueHead, SharedActorCritic
    rep = Basic_Identical((obs_dim,), device=DEV)
    actor = GaussianActorHead(obs_dim, list(hidden), act_dim, None, torch.nn.init.orthogonal_, torch.nn.LeakyReLU,
                              torch.nn.Tanh, DEV)
    critic = ValueHead(obs_dim, list(hidden), None, torch.nn.init.orthogonal_, torch.nn.LeakyReLU, DEV)
    return SharedActorCritic(rep, actor, critic).to(DEV)


def test_ppo_learner_gaussian_matches_oracle():
    """Four updates of PPO_Learner (K4-G) on a Gaussian MLP policy vs the torch-CPU oracle: info terms, then parameters."""
    from xuance_b200.torch.learners import PPO_Learner
    from xuance_b200.common import BaseCallback
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.manual_seed(2)
    od, ad, B = 17, 6, 512
    orc_model = GaussianActorCriticOracle(od, ad)
    model = _product_gaussian_model(od, ad, hidden=(256, 256))
    model.load_state_dict(orc_model.state_dict())
    cfg = ppo_config(DEV, running_steps=4096 * 50, learning_rate=4e-4)
    learner = PPO_Learner(cfg, model, BaseCallback())
    orc = PPOGaussianLearnerOracle(orc_model, learning_rate=4e-4, end_factor_lr_decay=0.5, total_iters=learner.total_iters)
    rng = np.random.default_rng(8)
    for it in range(4):
        obs = rng.normal(size=(B, od)).astype(np.float32)
        with torch.no_grad():
            dist, _ = orc_model(obs)
            acts = dist.sample().numpy()
            old = (dist.log_prob(torch.from_numpy(acts)).sum(-1).numpy() + rng.normal(size=B) * 0.2).astype(np.float32)
        s = {"obs": obs, "actions": acts, "returns": rng.normal(size=B).astype(np.float32),
             "advantages": rng.normal(size=B).astype(np.float32), "aux_batch": {"old_logp": old}}
        io, ip = orc.update(**s), learner.update(**s)
        for k in ("actor_loss", "critic_loss", "entropy", "predict_value"):
            np.testing.assert_allclose(ip[k], io[k], rtol=2e-4, atol=1e-5, err_msg=k)
        assert ip["learning_rate"] == io["learning_rate"]
        np.testing.assert_allclose(ip["clip_ratio"], float(io["clip_ratio"]), atol=1.0 / B + 1e-7)
    so, sp = orc_model.state_dict(), model.state_dict()
    assert set(so) == set(sp)
    for k in so:
        np.testing.assert_allclose(sp[k].cpu().numpy(), so[k].numpy(), rtol=1e-3, atol=1e-4, err_msg=k)


def test_ppo_learner_gaussian_matches_reference_fixture():
    from xuance_b200.torch.learners import PPO_Learner
    from xuance_b200.common import BaseCallback
    torch.backends.cuda.matmul.allow_tf32 = False
    g = np.load(os.path.join(G, "ppo_gaussian_update.npz"), allow_pickle=False)
    od, ad, B, seed = (int(x) for x in g["cfg"])
    torch.manual_seed(seed)
    init = GaussianActorCriticOracle(od, ad, actor_hidden=(64, 64), critic_hidden=(64, 64)).state_dict()
    model = _product_gaussian_model(od, ad)
    model.load_state_dict(init)
    cfg = ppo_config(DEV, running_steps=4096 * 10, parallels=32, horizon_size=128)
    learner = PPO_Learner(cfg, model, BaseCallback())
    assert learner.total_iters == int(g["total_iters"])
    for it in range(2):
        s = {k: g[f"in{it}/{k}"] for k in ("obs", "actions", "returns", "advantages")}
        info = learner.update(aux_batch={"old_logp": g[f"in{it}/old_logp"]}, **s)
        got = [info["actor_loss"], info["critic_loss"], info["entropy"], info["learning_rate"], info["predict_value"],
               float(info["clip_ratio"])]
        np.testing.assert_allclose(got, g["infos"][it], rtol=2e-4, atol=1e-5)
    for k, v in model.state_dict().items():
        flat = v.detach().reshape(-1).cpu()
        np.testing.assert_allclose(flat[:64].numpy(), g[f"final_head/{k}"], rtol=1e-3, atol=1e-4, err_msg=k)


def _agent_cfg(**kw):
    from xuance_b200.common.common_tools import get_arguments
    base = dict(device=DEV, parallels=8, horizon_size=32, n_epochs=2, n_minibatch=2, model_dir="/tmp/xb_models/ppo_g",
                logger=None, seed=3)
    base.update(kw)
    return get_arguments("ppo", "mujoco", parser_args=Namespace(**base))


def test_ppo_gaussian_train_epochs_cuda_graph_matches_eager():
    from xuance_b200.common import Box
    from xuance_b200.torch.agents import PPO_Agent
    torch.backends.cuda.matmul.allow_tf32 = False
    rng = np.random.default_rng(1)
    N, T, od, ad = 8, 32, 17, 6
    ro = [(rng.normal(size=(N, od)).astype(np.float32), rng.uniform(-1, 1, (N, ad)).astype(np.float32),
           rng.normal(size=N).astype(np.float32), rng.normal(size=N).astype(np.float32), rng.random(N) < 0.05,
           (rng.normal(size=N) - 5).astype(np.float32)) for _ in range(T)]
    results = []
    for graph in (False, True):
        agent = PPO_Agent(_agent_cfg(use_cuda_graph=graph), None, Box(-np.inf, np.inf, (od,), np.float32),
                          Box(-1, 1, (ad,), np.float32))
        for o, a, r, v, d, lp in ro:
            agent.memory.store(o, a, r, v, d, {"old_logp": lp})
        for i in range(N):
            agent.memory.finish_path(0.0, i)
        np.random.seed(11)
        agent.train_epochs(2)
        info = agent.train_epochs(2)                 # second call replays the captured graphs
        results.append((info, {k: v.clone() for k, v in agent.model.state_dict().items()}))
    (i0, p0), (i1, p1) = results
    for k in ("actor_loss", "critic_loss", "entropy", "predict_value", "clip_ratio"):
        np.testing.assert_allclose(i1[k], i0[k], rtol=1e-4, atol=1e-6, err_msg=k)
    for k in p0:
        np.testing.assert_allclose(p1[k].cpu().numpy(), p0[k].cpu().numpy(), rtol=1e-4, atol=1e-6, err_msg=k)


def test_store_staged_vector_actions_matches_store():
    from xuance_b200.common import DummyOnPolicyBuffer, Box
    N, T, od, ad = 4, 8, 17, 6
    spaces = (Box(-np.inf, np.inf, (od,), np.float32), Box(-1, 1, (ad,), np.float32))
    a_buf = DummyOnPolicyBuffer(*spaces, {"old_logp": ()}, N, T, device=DEV)
    b_buf = DummyOnPolicyBuffer(*spaces, {"old_logp": ()}, N, T, device=DEV)
    rng = np.random.default_rng(5)
    for t in range(T):
        obs = torch.tensor(rng.normal(size=(N, od)).astype(np.float32), device=DEV)
        acts = rng.uniform(-1, 1, (N, ad)).astype(np.float32)
        val, lp = rng.normal(size=N).astype(np.float32), rng.normal(size=N).astype(np.float32)
        rew, term = rng.normal(size=N).astype(np.float32), rng.random(N) < 0.2
        a_buf.store(obs, acts, rew, val, term, {"old_logp": lp})
        slots = b_buf.policy_slots()
        assert tuple(slots["actions"].shape) == (N, ad)
        slots["actions"].copy_(torch.from_numpy(acts))
        slots["values"].copy_(torch.from_numpy(val))
        slots["aux:old_logp"].copy_(torch.from_numpy(lp))
        b_buf.store_staged(obs, rew, term)
    torch.cuda.synchronize()
    assert a_buf.full and b_buf.full and a_buf.ptr == b_buf.ptr
    for name in ("_obs", "_act_rows", "_fields"):
        assert torch.equal(getattr(a_buf, name), getattr(b_buf, name)), name


@pytest.mark.parametrize("device_rollout", [False, True])
def test_ppo_mujoco_runner_learns(device_rollout):
    """24 rollouts of configs/ppo/mujoco.yaml; the test episodes act with the policy mean (the sampling noise alone costs
    ~80 per episode at the initial sigma), before and after training."""
    from xuance_b200 import get_runner
    steps = 16 * 256 * 24
    runner = get_runner("ppo", "mujoco", parser_args=Namespace(device=DEV, running_steps=steps, device_rollout=device_rollout,
                                                               model_dir="/tmp/xb_models/ppo_mujoco", logger=None,
                                                               deterministic_test=True))
    agent = runner.agent
    assert agent.n_envs == 16 and agent.memory.n_size == 256 and agent.batch_size == 512
    before = float(np.mean(agent.test(test_episodes=16)))
    runner.run("train", running_steps=steps)
    assert {"actor_loss", "critic_loss", "entropy", "learning_rate", "predict_value", "clip_ratio"} <= set(agent.logged)
    after = float(np.mean(agent.test(test_episodes=16)))
    runner.finish()
    assert after > before + 0.3 * abs(before), (before, after)


def test_sac_mujoco_runner_builds_and_trains():
    from xuance_b200 import get_runner
    runner = get_runner("sac", "mujoco", parser_args=Namespace(device=DEV, parallels=4, buffer_size=4000, batch_size=64,
                                                               start_training=40, running_steps=320,
                                                               model_dir="/tmp/xb_models/sac_mujoco", logger=None))
    info = runner.run("train", running_steps=320)
    runner.finish()
    assert np.isfinite(info["Qloss"]) and np.isfinite(info["Ploss"]) and info["alpha"] > 0
