"""Generate tests/golden/*.npz by running the UNMODIFIED reference (agi-brain/xuance v1.4.4 @ 4f0b05b).

Run in the build container only (needs /root/reference):   python tests/golden/make_golden.py
The reference is imported read-only with two import stubs (oracle/ref_stubs: gymnasium, pyglet).  Each fixture
stores the seeded inputs that cannot be re-derived cheaply plus the reference's outputs; the CPU tests re-run
the oracle on the same inputs and compare.  Environment of record is written into every file."""
import os
import random
import sys
from argparse import Namespace

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from oracle.ref_loader import import_reference  # noqa: E402

import_reference()
from gymnasium.spaces import Box, Discrete  # noqa: E402
from xuance.common import BaseCallback  # noqa: E402
from xuance.common.common_tools import discount_cumsum  # noqa: E402
from xuance.common.memory_tools import (DummyOnPolicyBuffer, DummyOnPolicyBuffer_Atari, PerOffPolicyBuffer,  # noqa
                                        DummyOffPolicyBuffer)
from xuance.torch.learners import PPO_Learner, DQN_Learner, PerDQN_Learner  # noqa: E402
from xuance.torch.rl_models.representations import AC_CNN_Atari, Basic_CNN  # noqa: E402
from xuance.torch.rl_models.heads import CategoricalActorHead, ValueHead  # noqa: E402
from xuance.torch.rl_models.architectures.single_agent.actor_critic import SharedActorCritic  # noqa: E402
from xuance.torch.rl_models.architectures.single_agent.deep_q_network import DeepQNetwork  # noqa: E402
from helpers import synth_rollout, fill_buffers  # noqa: E402

ENV = "torch %s / numpy %s / reference 4f0b05b" % (torch.__version__, np.__version__)


def golden_onpolicy():
    out = {"env": ENV}
    cases = [("vec_gae", 6, 24, (5,), False, True), ("vec_nstep", 6, 24, (5,), False, False),
             ("atari_gae", 4, 16, (8, 8, 4), True, True)]
    for name, N, T, shape, atari, use_gae in cases:
        rng = np.random.default_rng(hash(name) % 1000 if False else len(name) * 7 + N)
        ro = synth_rollout(rng, N, T, shape, obs_dtype=np.uint8 if atari else np.float32, p_term=0.08)
        cls = DummyOnPolicyBuffer_Atari if atari else DummyOnPolicyBuffer
        space = Box(0, 255, shape, np.uint8) if atari else Box(-10, 10, shape, np.float32)
        ref = cls(space, Discrete(4), {"old_logp": ()}, N, T, use_gae=use_gae)
        mids = [(T // 3, 1, np.float32(0.37)), (T // 2, 0, 0.0), (T // 2 + 1, 0, np.float32(-1.5))]
        fill_buffers([ref], ro, mids)
        idx = rng.permutation(N * T)[: N * T // 2]
        s = ref.sample(idx)
        for k, v in ro.items():
            out[f"{name}/in/{k}"] = v
        # 4th column: 1 if the bootstrap was a Python float (np.append then promotes the path to float64, as
        # happens for the reference's finish_path(0.0, i) calls), 0 if it was an np.float32 (model output)
        out[f"{name}/in/mids"] = np.array([(t, e, float(v), float(isinstance(v, float))) for t, e, v in mids])
        out[f"{name}/in/idx"] = idx
        out[f"{name}/returns"], out[f"{name}/advantages"] = ref.returns, ref.advantages
        out[f"{name}/start_ids"] = ref.start_ids
        for k in ("obs", "actions", "returns", "values", "advantages"):
            out[f"{name}/sample/{k}"] = s[k]
        out[f"{name}/sample/old_logp"] = s["aux_batch"]["old_logp"]
    out["kat/discount_cumsum"] = np.asarray(discount_cumsum(np.array([0, 1, 2, 2]), 0.99))
    np.savez_compressed(os.path.join(HERE, "onpolicy.npz"), **out)


def golden_per():
    """PER under the canonical float32 rule: the reference's float64 ``_max_priority`` array is replaced by a float32
    one right after construction (state change in the test harness, no reference source change) - see oracle/replay.py."""
    out = {"env": ENV}
    N, S, B, alpha = 4, 48, 32, 0.5
    rng = np.random.default_rng(42)
    ref = PerOffPolicyBuffer(Box(-1, 1, (3,)), Discrete(4), None, N, N * S, B, alpha=alpha)
    ref._max_priority = np.ones(N, np.float32)
    steps, samples = [], []
    for t in range(70):
        st = (rng.normal(size=(N, 3)).astype(np.float32), rng.integers(0, 4, N), rng.normal(size=N).astype(np.float32),
              rng.random(N) < 0.1, rng.normal(size=(N, 3)).astype(np.float32))
        ref.store(*st)
        steps.append(st)
        if t > 5 and t % 6 == 0:
            random.seed(t)
            u = np.array([[random.random() for _ in range(B // N)] for _ in range(N)])
            random.seed(t)
            s = ref.sample(0.4)
            td = np.abs(rng.normal(size=B)).astype(np.float32)
            td[2] = 0.0
            ref.update_priorities(s["step_choices"], td)
            samples.append(dict(t=t, u=u, step_choices=s["step_choices"], weights=s["weights"], td=td,
                                obs=s["obs"], rewards=s["rewards"],
                                sum_tree=np.array([np.array(tr._value, dtype=np.float64) for tr in ref._it_sum]),
                                min_tree=np.array([np.array(tr._value, dtype=np.float64) for tr in ref._it_min]),
                                max_priority=ref._max_priority.astype(np.float64).copy()))
    for i, name in enumerate(("obs", "acts", "rews", "terms", "next_obs")):
        out[f"in/{name}"] = np.stack([s[i] for s in steps])
    out["n_samples"] = len(samples)
    for j, s in enumerate(samples):
        for k, v in s.items():
            out[f"s{j}/{k}"] = v
    out["cfg"] = np.array([N, S, B, alpha])
    # the default (mixed float64/float32) behaviour of the reference under NumPy>=2, recorded for DESIGN.md
    ref2 = PerOffPolicyBuffer(Box(-1, 1, (3,)), Discrete(4), None, 2, 8, 2, alpha=alpha)
    ref2.store(np.zeros((2, 3)), np.zeros(2), np.zeros(2), np.zeros(2), np.zeros((2, 3)))
    ref2.store(np.zeros((2, 3)), np.zeros(2), np.zeros(2), np.zeros(2), np.zeros((2, 3)))
    ref2.update_priorities(np.array([[0], [1]]), np.array([0.3, 0.7], np.float32))
    out["note/default_leaf_dtypes"] = np.array([type(ref2._it_sum[0]._value[4]).__name__,
                                                type(ref2._it_sum[0]._value[5]).__name__])
    np.savez_compressed(os.path.join(HERE, "per.npz"), **out)


def _learner_cfg(**kw):
    cfg = dict(distributed_training=False, episode_length=1000, use_grad_clip=True, grad_clip_norm=0.5, device="cpu",
               model_dir="/tmp/xb_golden", running_steps=4096 * 10, parallels=32, learning_rate=2.5e-4,
               use_linear_lr_decay=True, end_factor_lr_decay=0.5, horizon_size=128, n_epochs=4, n_minibatch=4,
               vf_coef=0.25, ent_coef=0.01, clip_range=0.2, gamma=0.99, sync_frequency=2, start_training=0,
               training_frequency=1)
    cfg.update(kw)
    return Namespace(**cfg)


def golden_ppo():
    """Two PPO updates of the reference learner on the NatureCNN actor-critic at 84x84x4, B=24.  Initial weights are
    reproduced from torch.manual_seed (construction order is part of the oracle's contract); the fixture keeps
    inputs, info dicts and per-tensor digests of the parameters after the updates."""
    out = {"env": ENV}
    A, B = 6, 24
    torch.manual_seed(3)
    rep = AC_CNN_Atari(input_shape=(84, 84, 4), kernels=[8, 4, 3], strides=[4, 2, 1], filters=[32, 64, 64],
                       activation=torch.nn.ReLU, device="cpu", fc_hidden_sizes=[512])
    actor = CategoricalActorHead(512, [], A, None, torch.nn.init.orthogonal_, torch.nn.ReLU, "cpu")
    critic = ValueHead(512, [], None, torch.nn.init.orthogonal_, torch.nn.ReLU, "cpu")
    model = SharedActorCritic(rep, actor, critic)
    init = {k: v.clone() for k, v in model.state_dict().items()}
    learner = PPO_Learner(_learner_cfg(), model, BaseCallback())
    rng = np.random.default_rng(9)
    infos = []
    for it in range(2):
        s = {"obs": rng.integers(0, 256, size=(B, 84, 84, 4), dtype=np.uint8),
             "actions": rng.integers(0, A, size=B).astype(np.float32),
             "returns": rng.normal(size=B).astype(np.float32), "advantages": rng.normal(size=B).astype(np.float32),
             "aux_batch": {"old_logp": (rng.normal(size=B) * 0.05 - np.log(A)).astype(np.float32)}}
        info = learner.update(**s)
        infos.append([info["actor_loss"], info["critic_loss"], info["entropy"], info["learning_rate"],
                      info["predict_value"], float(info["clip_ratio"])])
    out["infos"] = np.array(infos, dtype=np.float64)
    out["total_iters"] = learner.total_iters
    for k, v in model.state_dict().items():
        out[f"init_digest/{k}"] = np.array([v_.double().sum().item() for v_ in (init[k], init[k].abs())])
        flat = v.detach().reshape(-1)
        out[f"final_head/{k}"] = flat[:64].numpy().copy()
        out[f"final_digest/{k}"] = np.array([flat.double().sum().item(), flat.double().abs().sum().item()])
    np.savez_compressed(os.path.join(HERE, "ppo_update.npz"), **out)


def golden_dqn():
    out = {"env": ENV}
    A, B = 5, 16
    torch.manual_seed(4)
    rep = Basic_CNN(input_shape=(84, 84, 4), kernels=[8, 4, 3], strides=[4, 2, 1], filters=[32, 64, 64],
                    activation=torch.nn.ReLU, device="cpu")
    model = DeepQNetwork(rep, [512], Discrete(A), None, None, torch.nn.ReLU, "cpu")
    learner = PerDQN_Learner(_learner_cfg(learning_rate=1e-4, use_grad_clip=False), model, BaseCallback())
    rng = np.random.default_rng(10)
    infos, tds = [], []
    for it in range(3):
        s = {"obs": rng.integers(0, 256, size=(B, 84, 84, 4), dtype=np.uint8).astype(np.float32),
             "actions": rng.integers(0, A, size=B).astype(np.float32),
             "obs_next": rng.integers(0, 256, size=(B, 84, 84, 4), dtype=np.uint8).astype(np.float32),
             "rewards": rng.normal(size=B).astype(np.float32), "terminals": (rng.random(B) < 0.2).astype(np.float32)}
        td, info = learner.update(**s)
        infos.append([info["Qloss"], info["learning_rate"], info["predictQ"]])
        tds.append(td)
    out["infos"], out["abs_td"] = np.array(infos, dtype=np.float64), np.stack(tds)
    for k, v in model.state_dict().items():
        flat = v.detach().reshape(-1)
        out[f"final_digest/{k}"] = np.array([flat.double().sum().item(), flat.double().abs().sum().item()])
    np.savez_compressed(os.path.join(HERE, "dqn_update.npz"), **out)


def golden_sac():
    """Three SAC updates of the reference learner (17-d obs / 6-d action, MLP 64-64, automatic entropy tuning).  The
    reference draws its reparameterisation noise from torch's global RNG; the fixture stores the noise it drew (the stream
    is replayed: randn(B, act) for the actor step, then randn(B, act) for the target step)."""
    from copy import deepcopy
    from xuance.torch.rl_models.representations.mlp import Basic_Identical
    from xuance.torch.rl_models.actors.gaussian_actors import SAC_GaussianActor
    from xuance.torch.rl_models.critics.twin_critics import TwinActionValueCritic
    from xuance.torch.rl_models.architectures.single_agent.actor_critic import SoftActorCritic
    from xuance.torch.learners import SAC_Learner
    out = {"env": ENV}
    torch.manual_seed(7)
    obs_dim, act_dim, B = 17, 6, 32
    aspace = Box(-1, 1, (act_dim,), np.float32)
    rep = Basic_Identical((obs_dim,), device='cpu')
    actor = SAC_GaussianActor(rep, [64, 64], aspace, None, None, torch.nn.LeakyReLU, torch.nn.Tanh, 'cpu')
    critic = TwinActionValueCritic(deepcopy(rep), aspace, [64, 64], None, None, torch.nn.LeakyReLU, 'cpu')
    model = SoftActorCritic(actor, critic)
    for k, v in model.state_dict().items():
        out[f"init/{k}"] = v.numpy().copy()
    cfg = _learner_cfg(learning_rate_actor=1e-3, learning_rate_critic=1e-3, tau=0.005, alpha=0.2, use_grad_clip=False,
                       use_automatic_entropy_tuning=True, end_factor_lr_decay=0.7, parallels=4, running_steps=100000)
    lrn = SAC_Learner(cfg, model, BaseCallback())
    out["total_iters"] = lrn.total_iters
    rng = np.random.default_rng(12)
    infos = []
    for it in range(3):
        s = {"obs": rng.normal(size=(B, obs_dim)).astype(np.float32),
             "actions": rng.uniform(-1, 1, size=(B, act_dim)).astype(np.float32),
             "obs_next": rng.normal(size=(B, obs_dim)).astype(np.float32),
             "rewards": rng.normal(size=B).astype(np.float32), "terminals": (rng.random(B) < 0.1).astype(np.float32)}
        torch.manual_seed(500 + it)
        out[f"noise_pi/{it}"] = torch.randn(B, act_dim).numpy()
        out[f"noise_next/{it}"] = torch.randn(B, act_dim).numpy()
        torch.manual_seed(500 + it)
        info = lrn.update(**s)
        for k, v in s.items():
            out[f"in{it}/{k}"] = v
        infos.append([info["Qloss"], info["Ploss"], info["Qvalue"], info["alpha_loss"], info["alpha"], info["actor_lr"]])
    out["infos"] = np.array(infos, dtype=np.float64)
    for k, v in model.state_dict().items():
        flat = v.detach().reshape(-1)
        out[f"final_head/{k}"] = flat[:32].numpy().copy()
        out[f"final_digest/{k}"] = np.array([flat.double().sum().item(), flat.double().abs().sum().item()])
    np.savez_compressed(os.path.join(HERE, "sac_update.npz"), **out)


def golden_qmix():
    """Episode replay + three QMIX updates of the reference (5 agents x 24-d obs, 7 actions, 30-d state, T=10, GRU 64,
    mixer 32/32, double-Q, use_actions_mask=False).  Pins BOTH reference behaviours recorded in DESIGN.md: the values and
    the fact that the agent networks do not move (q_eval is sliced under no_grad)."""
    from xuance.common import AgentGrouping
    from xuance.common.memory_tools_marl import MARL_OffPolicyBuffer_RNN
    from xuance.torch.rl_models.representations.rnn import Basic_RNN
    from xuance.torch.rl_models.representations.agent_feature import AgentFeatureEncoder
    from xuance.torch.rl_models.modules.identity_encoder import build_identity_encoder, IdentityFeatureFusion
    from xuance.torch.rl_models.critics.base_critics import DiscreteActionValueCritic
    from xuance.torch.rl_models.heads.q_mix_head import QMIX_Mixer
    from xuance.torch.rl_models.architectures.multi_agent.value_factorization import MixingQNetwork
    from xuance.torch.learners.multi_agent_rl.qmix_learner import QMIX_Learner
    from helpers import qmix_episode_stream
    out = {"env": ENV}
    torch.manual_seed(8)
    n, obs_dim, A, S, T = 5, 24, 7, 30, 10
    keys = [f"agent_{i}" for i in range(n)]
    rep = Basic_RNN(input_shape=(obs_dim,), hidden_sizes=None, initialize=torch.nn.init.orthogonal_,
                    activation=torch.nn.ReLU, device='cpu', fc_hidden_sizes=[64], recurrent_hidden_size=64,
                    N_recurrent_layers=1, dropout=0, rnn='GRU')
    enc = AgentFeatureEncoder(rep, build_identity_encoder(n, 'none', None, 'cpu'), IdentityFeatureFusion(64, 0, 'concat'))
    q = torch.nn.ModuleDict({'shared': DiscreteActionValueCritic(enc, Discrete(A), [64], None, torch.nn.init.orthogonal_,
                                                                   torch.nn.ReLU, 'cpu')})
    grouping = AgentGrouping.shared(keys)
    model = MixingQNetwork(grouping, q, QMIX_Mixer(S, 32, 32, n, 'cpu'), use_rnn=True, device='cpu')
    for k, v in model.state_dict().items():
        out[f"init/{k}"] = v.numpy().copy()
    cfg = _learner_cfg(episode_length=T, use_grad_clip=False, parallels=4, running_steps=100000,
                       use_parameter_sharing=True, use_rnn=True, use_actions_mask=False, learning_rate=7e-4,
                       sync_frequency=2, double_q=True, n_epochs=1, end_factor_lr_decay=0.5)
    lrn = QMIX_Learner(cfg, grouping, model, BaseCallback())
    out["total_iters"] = lrn.total_iters
    n_envs, C, Be = 3, 12, 6
    rb = MARL_OffPolicyBuffer_RNN(agent_keys=keys, state_space=Box(-1, 1, (S,)),
                                  obs_space={k: Box(-1, 1, (obs_dim,)) for k in keys},
                                  act_space={k: Discrete(A) for k in keys}, n_envs=n_envs, buffer_size=C, batch_size=Be,
                                  max_episode_steps=T, use_actions_mask=False)
    for ev in qmix_episode_stream(np.random.default_rng(21), keys, n_envs, T, obs_dim, A, S, 5):
        if ev[0] == 'store':
            rb.store(**ev[1])
        else:
            rb.finish_path(ev[1], **ev[2])
    out["cfg"] = np.array([n, obs_dim, A, S, T, n_envs, C, Be])
    out["buffer/ptr_size"] = np.array([rb.ptr, int(rb.size)])
    out["buffer/filled"], out["buffer/state"] = rb.data['filled'], rb.data['state']
    for kname in ('obs', 'actions', 'rewards', 'terminals', 'agent_mask'):
        out[f"buffer/{kname}"] = np.stack([rb.data[kname][a] for a in keys], axis=1)
    infos = []
    for it in range(3):
        np.random.seed(it)
        s = rb.sample()
        info = lrn.update(s)
        infos.append([info["loss_Q"], info["predictQ"], info["learning_rate"]])
    out["infos"] = np.array(infos, dtype=np.float64)
    for k, v in model.state_dict().items():
        flat = v.detach().reshape(-1)
        out[f"final_head/{k}"] = flat[:32].numpy().copy()
        out[f"final_digest/{k}"] = np.array([flat.double().sum().item(), flat.double().abs().sum().item()])
    np.savez_compressed(os.path.join(HERE, "qmix_update.npz"), **out)


def golden_rollout_glue():
    """RunningMeanStd + Agent._process_observation arithmetic (statistic_tools.py:117-185, agent.py:273-276) and
    CategoricalDistribution log_prob / entropy / deterministic_sample (distributions.py:128-162) of the reference."""
    from xuance.common.statistic_tools import RunningMeanStd
    from xuance.common.common_tools import EPS
    from xuance.torch.rl_models.modules.distributions import CategoricalDistribution
    out = {"env": ENV}
    rng = np.random.default_rng(33)
    for name, N, D in (("cartpole", 8, 4), ("wide", 256, 17)):
        rms = RunningMeanStd(shape=(D,))
        for it in range(6):
            x = (rng.normal(size=(N, D)) * (1.0 + 3.0 * it) + 0.5 * it).astype(np.float32)
            rms.update(x)
            y = np.clip((x - rms.mean) / (rms.std + EPS), -5, 5)
            out[f"rms/{name}/x{it}"], out[f"rms/{name}/y{it}"] = x, y
            out[f"rms/{name}/mean{it}"], out[f"rms/{name}/var{it}"] = rms.mean.copy(), rms.var.copy()
            out[f"rms/{name}/count{it}"] = np.float64(rms.count)
    for A in (2, 4, 18):
        logits = (rng.normal(size=(64, A)) * 2.0).astype(np.float32)
        acts = rng.integers(0, A, size=64)
        d = CategoricalDistribution(A)
        d.set_param(logits=torch.from_numpy(logits))
        out[f"cat/{A}/logits"], out[f"cat/{A}/actions"] = logits, acts
        out[f"cat/{A}/log_prob"] = d.log_prob(torch.from_numpy(acts)).numpy()
        out[f"cat/{A}/entropy"] = d.entropy().numpy()
        out[f"cat/{A}/argmax"] = d.deterministic_sample().numpy()
        out[f"cat/{A}/probs"] = d.probs.numpy()
    np.savez_compressed(os.path.join(HERE, "rollout_glue.npz"), **out)


QMIX_BUFFER_KEYS = ('obs', 'actions', 'rewards', 'terminals', 'agent_mask')   # digests: these x agents, then filled, state


def _ref_qmix_pair(n, obs_dim, A, S, T, lr_decay=0.5):
    """The reference's QMIX model (use_rnn, shared GRU agent) + learner, as tests/test_oracle_vs_reference.py builds the
    oracle's counterpart (QMIXModelOracle constructs the same initial weights from the same torch seed)."""
    from xuance.common import AgentGrouping
    from xuance.torch.rl_models.representations.rnn import Basic_RNN
    from xuance.torch.rl_models.representations.agent_feature import AgentFeatureEncoder
    from xuance.torch.rl_models.modules.identity_encoder import build_identity_encoder, IdentityFeatureFusion
    from xuance.torch.rl_models.critics.base_critics import DiscreteActionValueCritic
    from xuance.torch.rl_models.heads.q_mix_head import QMIX_Mixer
    from xuance.torch.rl_models.architectures.multi_agent.value_factorization import MixingQNetwork
    from xuance.torch.learners.multi_agent_rl.qmix_learner import QMIX_Learner
    nn = torch.nn
    keys = [f"agent_{i}" for i in range(n)]
    rep = Basic_RNN(input_shape=(obs_dim,), hidden_sizes=None, initialize=nn.init.orthogonal_, activation=nn.ReLU,
                    device='cpu', fc_hidden_sizes=[64], recurrent_hidden_size=64, N_recurrent_layers=1, dropout=0, rnn='GRU')
    enc = AgentFeatureEncoder(rep, build_identity_encoder(n, 'none', None, 'cpu'), IdentityFeatureFusion(64, 0, 'concat'))
    q = nn.ModuleDict({'shared': DiscreteActionValueCritic(enc, Discrete(A), [64], None, nn.init.orthogonal_, nn.ReLU, 'cpu')})
    grouping = AgentGrouping.shared(keys)
    model = MixingQNetwork(grouping, q, QMIX_Mixer(S, 32, 32, n, 'cpu'), use_rnn=True, device='cpu')
    cfg = Namespace(distributed_training=False, episode_length=T, use_grad_clip=False, grad_clip_norm=10, device='cpu',
                    model_dir='/tmp/x', running_steps=100000, parallels=4, use_parameter_sharing=True, use_rnn=True,
                    use_actions_mask=False, learning_rate=7e-4, sync_frequency=2, double_q=True, n_epochs=1,
                    start_training=0, gamma=0.99, end_factor_lr_decay=lr_decay)
    return keys, model, QMIX_Learner(cfg, grouping, model, BaseCallback())


def golden_oracle_vs_reference():
    """What tests/test_oracle_vs_reference.py compares the oracle with: the reference's buffers, learners and multi-agent
    vector env on the tests' own seeded inputs.  Large arrays are kept as sha256 digests (buffers) or as a fixed sample of
    elements plus sum / abs-sum digests (final weights); the initial weights as digests (the oracle rebuilds them from the
    same torch seed)."""
    from helpers import qmix_episode_stream, array_digest, structure_digest, record_state
    out = {"env": ENV}
    # on-policy buffer: test_onpolicy_buffer_live
    for seed, use_gae in [(0, True), (1, True), (2, False)]:
        rng = np.random.default_rng(seed)
        N, T = 5, 33
        ro = synth_rollout(rng, N, T, (3,), obs_dtype=np.float32, p_term=0.1)
        r = DummyOnPolicyBuffer(Box(-1, 1, (3,)), Discrete(4), {'old_logp': ()}, N, T, use_gae=use_gae)
        fill_buffers([r], ro, [(4, 1, np.float32(0.2)), (9, 3, 0.0), (20, 1, np.float32(-0.7))])
        p = f"onpolicy/{seed}"
        out[f"{p}/returns"], out[f"{p}/advantages"] = r.returns, r.advantages
        s = r.sample(rng.permutation(N * T)[:50])
        for k in ('obs', 'actions', 'returns', 'values', 'advantages'):
            out[f"{p}/sample/{k}"] = s[k]
    # PER: test_per_buffer_live (the sum / min trees as digests of their float64 leaf arrays)
    for alpha in (0.5, 0.6):
        rng = np.random.default_rng(int(alpha * 10))
        N, S, B = 4, 64, 32
        r = PerOffPolicyBuffer(Box(-1, 1, (3,)), Discrete(4), None, N, N * S, B, alpha=alpha)
        r._max_priority = np.ones(N, np.float32)
        rec = {k: [] for k in ("step_choices", "weights", "sum_tree", "min_tree", "max_priority")}
        for t in range(100):
            st = (rng.normal(size=(N, 3)).astype(np.float32), rng.integers(0, 4, N), rng.normal(size=N).astype(np.float32),
                  rng.random(N) < 0.1, rng.normal(size=(N, 3)).astype(np.float32))
            r.store(*st)
            if t > 10 and t % 3 == 0:
                random.seed(t)
                s = r.sample(0.4)
                rec["step_choices"].append(s['step_choices']), rec["weights"].append(s['weights'])
                td = np.abs(rng.normal(size=B)).astype(np.float32)
                td[3] = 0
                r.update_priorities(s['step_choices'], td)
                for name, trees in (("sum_tree", r._it_sum), ("min_tree", r._it_min)):
                    rec[name].append(array_digest(np.array([np.array(tr._value, dtype=np.float64) for tr in trees])))
                rec["max_priority"].append(np.array(r._max_priority, dtype=np.float64))
        for k, v in rec.items():
            out[f"per/{alpha}/{k}"] = np.array(v) if k.endswith("tree") else np.stack(v)
    # QMIX buffer + learner: test_qmix_buffer_and_learner_live
    from xuance.common.memory_tools_marl import MARL_OffPolicyBuffer_RNN
    torch.manual_seed(0)
    n, obs_dim, A, S, T = 5, 72, 12, 98, 12
    keys, model, lrn = _ref_qmix_pair(n, obs_dim, A, S, T)
    init = {k: v.clone() for k, v in model.state_dict().items()}
    record_state(out, "qmix/init", init, sample=False)
    out["qmix/total_iters"] = np.array(lrn.total_iters)
    n_envs, C, Be = 3, 12, 6
    rb = MARL_OffPolicyBuffer_RNN(agent_keys=keys, state_space=Box(-1, 1, (S,)),
                                  obs_space={k: Box(-1, 1, (obs_dim,)) for k in keys},
                                  act_space={k: Discrete(A) for k in keys}, n_envs=n_envs, buffer_size=C,
                                  batch_size=Be, max_episode_steps=T, use_actions_mask=False)
    for ev in qmix_episode_stream(np.random.default_rng(0), keys, n_envs, T, obs_dim, A, S, 5):
        if ev[0] == 'store':
            rb.store(**ev[1])
        else:
            rb.finish_path(ev[1], **ev[2])
    out["qmix/buffer/digests"] = np.array([array_digest(rb.data[k][a]) for k in QMIX_BUFFER_KEYS for a in keys]
                                    + [array_digest(rb.data['filled']), array_digest(rb.data['state'])])
    out["qmix/buffer/ptr_size"] = np.array([rb.ptr, int(rb.size)])
    infos = []
    for it in range(3):
        np.random.seed(it)
        i1 = lrn.update(rb.sample())
        infos.append([i1['loss_Q'], i1['predictQ'], i1['learning_rate']])
    out["qmix/infos"] = np.array(infos, dtype=np.float64)
    sd = model.state_dict()
    record_state(out, "qmix/final", sd)
    out["qmix/moved_agent_tensors"] = np.array(sorted(k for k in sd if k.startswith("individual_q_networks")
                                                      and not torch.equal(sd[k], init[k])), dtype=str)
    # SAC learner: test_sac_learner_live
    from copy import deepcopy
    from xuance.torch.rl_models.representations.mlp import Basic_Identical
    from xuance.torch.rl_models.actors.gaussian_actors import SAC_GaussianActor
    from xuance.torch.rl_models.critics.twin_critics import TwinActionValueCritic
    from xuance.torch.rl_models.architectures.single_agent.actor_critic import SoftActorCritic
    from xuance.torch.learners import SAC_Learner
    nn = torch.nn
    torch.manual_seed(0)
    obs_dim, act_dim, B = 17, 6, 64
    aspace = Box(-1, 1, (act_dim,), np.float32)
    rep = Basic_Identical((obs_dim,), device='cpu')
    actor = SAC_GaussianActor(rep, [256, 256], aspace, None, None, nn.LeakyReLU, nn.Tanh, 'cpu')
    critic = TwinActionValueCritic(deepcopy(rep), aspace, [256, 256], None, None, nn.LeakyReLU, 'cpu')
    model = SoftActorCritic(actor, critic)
    record_state(out, "sac/init", model.state_dict(), sample=False)
    cfg = Namespace(distributed_training=False, episode_length=1000, use_grad_clip=False, grad_clip_norm=0.5, device='cpu',
                    model_dir='/tmp/x', running_steps=100000, parallels=4, start_training=0, training_frequency=1,
                    learning_rate_actor=1e-3, learning_rate_critic=1e-3, tau=0.005, gamma=0.99, alpha=0.2,
                    use_automatic_entropy_tuning=True, end_factor_lr_decay=0.7)
    lrn = SAC_Learner(cfg, model, BaseCallback())
    out["sac/total_iters"] = np.array(lrn.total_iters)
    rng = np.random.default_rng(1)
    infos = []
    for it in range(3):
        s = {"obs": rng.normal(size=(B, obs_dim)).astype(np.float32),
             "actions": rng.uniform(-1, 1, size=(B, act_dim)).astype(np.float32),
             "obs_next": rng.normal(size=(B, obs_dim)).astype(np.float32),
             "rewards": rng.normal(size=B).astype(np.float32), "terminals": (rng.random(B) < 0.1).astype(np.float32)}
        torch.manual_seed(100 + it)
        i1 = lrn.update(**s)
        infos.append([float(i1[k]) for k in ("Qloss", "Ploss", "Qvalue", "alpha", "alpha_loss")])
    out["sac/infos"] = np.array(infos, dtype=np.float64)
    record_state(out, "sac/final", model.state_dict())
    # A2C / PG / DDQN: test_sibling_learners_live
    from xuance.torch.learners import A2C_Learner, PG_Learner, DDQN_Learner
    for kind in ("a2c", "pg", "ddqn"):
        torch.manual_seed(5)
        A, B = 5, 12
        cfg = Namespace(distributed_training=False, episode_length=1000, use_grad_clip=True, grad_clip_norm=0.5,
                        device="cpu", model_dir="/tmp/x", running_steps=4096 * 10, parallels=32, learning_rate=2.5e-4,
                        end_factor_lr_decay=0.5, horizon_size=128, n_epochs=4, n_minibatch=4, vf_coef=0.25, ent_coef=0.01,
                        gamma=0.99, sync_frequency=2, start_training=0, training_frequency=1)
        rng = np.random.default_rng(3)
        if kind == "ddqn":
            rep = Basic_CNN(input_shape=(84, 84, 4), kernels=[8, 4, 3], strides=[4, 2, 1], filters=[32, 64, 64],
                            activation=nn.ReLU, device="cpu")
            model = DeepQNetwork(rep, [512], Discrete(A), None, None, nn.ReLU, "cpu")
            lrn = DDQN_Learner(cfg, model, BaseCallback())
        else:
            rep = AC_CNN_Atari(input_shape=(84, 84, 4), kernels=[8, 4, 3], strides=[4, 2, 1], filters=[32, 64, 64],
                               activation=nn.ReLU, device="cpu", fc_hidden_sizes=[512])
            model = SharedActorCritic(rep, CategoricalActorHead(512, [], A, None, nn.init.orthogonal_, nn.ReLU, "cpu"),
                                      ValueHead(512, [], None, nn.init.orthogonal_, nn.ReLU, "cpu"))
            lrn = (A2C_Learner if kind == "a2c" else PG_Learner)(cfg, model, BaseCallback())
        record_state(out, f"sibling/{kind}/init", model.state_dict(), sample=False)
        out[f"sibling/{kind}/total_iters"] = np.array(lrn.total_iters)
        infos = []
        for it in range(3):
            s = {"obs": rng.integers(0, 256, size=(B, 84, 84, 4), dtype=np.uint8).astype(np.float32),
                 "actions": rng.integers(0, A, size=B).astype(np.float32),
                 "returns": rng.normal(size=B).astype(np.float32), "advantages": rng.normal(size=B).astype(np.float32),
                 "aux_batch": {"old_logp": np.zeros(B, np.float32)},
                 "obs_next": rng.integers(0, 256, size=(B, 84, 84, 4), dtype=np.uint8).astype(np.float32),
                 "rewards": rng.normal(size=B).astype(np.float32), "terminals": (rng.random(B) < 0.2).astype(np.float32)}
            i1 = lrn.update(**s)
            infos.append([i1["Qloss"]] if kind == "ddqn" else [i1["actor-loss"], i1["entropy"]])
        out[f"sibling/{kind}/infos"] = np.array(infos, dtype=np.float64)
        record_state(out, f"sibling/{kind}/final", model.state_dict())
    # multi-agent vector env: test_multi_agent_vector_env_live
    from xuance.environment.utils.wrapper import XuanCeMultiAgentEnvWrapper as RefWrapper
    from xuance.environment.vector_envs.dummy.dummy_vec_maenv import DummyVecMultiAgentEnv as RefVec
    from xuance_b200.environment.ma_envs import SyntheticSMACEnv
    kw = dict(n_agents=3, obs_dim=16, state_dim=20, n_actions=5, episode_limit=7, p_death=0.1)
    n_envs = 3
    rv = RefVec([lambda env_seed=0: RefWrapper(SyntheticSMACEnv(seed=env_seed, **kw)) for _ in range(n_envs)], 11)
    out["maenv/attrs"] = np.array([rv.num_envs, rv.num_agents, rv.max_episode_steps])
    out["maenv/agents"] = np.array(rv.agents, dtype=str)
    out["maenv/state_shape"] = np.array(rv.state_space.shape)
    names = ("obs", "rewards", "terminated", "truncated", "infos", "state", "avail")
    ro, ri = rv.reset()
    digests = [[structure_digest(ro), structure_digest(ri)] + [""] * (len(names) - 2)]
    rng = np.random.default_rng(2)
    ends = 0
    for t in range(40):
        acts = [{a: int(rng.choice(np.flatnonzero(rv.buf_avail_actions[e][a]))) for a in rv.agents} for e in range(n_envs)]
        r = rv.step(acts)
        digests.append([structure_digest(x) for x in tuple(r) + (rv.buf_state, rv.buf_avail_actions)])
        ends += sum("reset_obs" in i for i in r[4])
    out["maenv/names"] = np.array(names, dtype=str)
    out["maenv/digests"] = np.array(digests, dtype=str)       # row 0: reset (obs, info); row t + 1: step t
    out["maenv/episode_ends"] = np.array(ends)
    rv.close()
    _check_no_objects(out)
    np.savez_compressed(os.path.join(HERE, "oracle_vs_reference.npz"), **out)


def golden_qmix_action_mask():
    """tests/test_oracle_vs_reference.py::test_qmix_action_mask_variant_against_the_reference_with_its_slice_corrected: the
    unpatched reference learner raising on use_rnn + use_actions_mask, then three updates of the same learner with the one
    slice of iql_learner.py corrected in memory.  The reference buffer's availability masks are stored whole (they are
    small); its other contents as digests (the oracle buffer rebuilds them from the same seeded stream)."""
    import inspect
    import textwrap
    from xuance.common.memory_tools_marl import MARL_OffPolicyBuffer_RNN
    from xuance.torch.learners.multi_agent_rl import iql_learner as iql
    from helpers import qmix_episode_stream, array_digest, record_state
    out = {"env": ENV}
    torch.manual_seed(1)
    n, obs_dim, A, S, T = 4, 24, 7, 30, 9
    keys, model, lrn = _ref_qmix_pair(n, obs_dim, A, S, T)
    record_state(out, "init", model.state_dict(), sample=False)
    out["total_iters"] = np.array(lrn.total_iters)
    lrn.use_actions_mask = lrn.config.use_actions_mask = True
    n_envs, C, Be = 3, 12, 6
    rb = MARL_OffPolicyBuffer_RNN(agent_keys=keys, state_space=Box(-1, 1, (S,)),
                                  obs_space={k: Box(-1, 1, (obs_dim,)) for k in keys},
                                  act_space={k: Discrete(A) for k in keys}, n_envs=n_envs, buffer_size=C,
                                  batch_size=Be, max_episode_steps=T, use_actions_mask=True,
                                  avail_actions_shape={k: (A,) for k in keys})
    rng = np.random.default_rng(4)

    def avail(shape_prefix):
        a = rng.random(shape_prefix + (A,)) < 0.6
        a[..., 0] = True
        return a
    for ev in qmix_episode_stream(np.random.default_rng(3), keys, n_envs, T, obs_dim, A, S, 5):
        if ev[0] == 'store':
            rb.store(avail_actions={k: avail((n_envs,)) for k in keys}, **ev[1])
        else:
            rb.finish_path(ev[1], avail_actions={k: avail(()) for k in keys}, **ev[2])
    out["buffer/digests"] = np.array([array_digest(rb.data[k][a]) for k in QMIX_BUFFER_KEYS for a in keys]
                                    + [array_digest(rb.data['filled']), array_digest(rb.data['state'])])
    out["buffer/ptr_size"] = np.array([rb.ptr, int(rb.size)])
    out["buffer/avail_actions"] = np.stack([rb.data['avail_actions'][a] for a in keys])
    np.random.seed(0)
    sample = rb.sample()
    out["sample_avail_shape"] = np.array(sample['avail_actions'][keys[0]].shape)
    snap = {k: v.clone() for k, v in model.state_dict().items()}
    try:
        lrn.update(sample)
        out["unpatched_error"] = np.array("")
    except Exception as e:  # noqa: BLE001 - recorded, the test checks the type
        out["unpatched_error"] = np.array(type(e).__name__)
    model.load_state_dict(snap)
    lrn.iterations = 0
    src = textwrap.dedent(inspect.getsource(iql.IQL_Learner._forward_transitions))
    bad = "batch.avail_actions.group(group)[:, 1:]"
    out["bad_slice_count"] = np.array(src.count(bad))
    scope = {}
    exec(compile(src.replace(bad, "batch.avail_actions.group(group)[:, :, 1:]"), "iql_learner.py (slice corrected)", "exec"),
         vars(iql), scope)
    orig = iql.IQL_Learner._forward_transitions
    iql.IQL_Learner._forward_transitions = scope["_forward_transitions"]
    infos = []
    try:
        for it in range(3):
            np.random.seed(10 + it)
            i1 = lrn.update(rb.sample())
            infos.append([i1['loss_Q'], i1['predictQ']])
    finally:
        iql.IQL_Learner._forward_transitions = orig
    out["infos"] = np.array(infos, dtype=np.float64)
    record_state(out, "final", model.state_dict())
    np.savez_compressed(os.path.join(HERE, "qmix_action_mask.npz"), **out)


def golden_dropin():
    """tests/test_dropin_reference.py: what the INTEGRATION.md section A patch has to reach inside the reference (module
    paths and names), the keyword arguments the reference's OnPolicyAgent._build_memory passes to the patched buffer
    class, and the call sequence of its OnPolicyAgent.train_epochs."""
    import inspect
    import json
    import re
    from types import SimpleNamespace
    import xuance.torch.agents.core.on_policy as core
    import xuance.torch.learners as learners
    from xuance.torch.agents.base.agent import Agent
    out = {"env": ENV}
    md = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    code = re.search(r"```python\n(.*?)```", md[md.index("Registering inside an existing XuanCe checkout"):], re.S).group(1)
    mods = sorted(set(re.findall(r"(?:from|import)\s+(xuance(?:\.\w+)*)", code)))
    out["registry/modules"] = np.array(mods, dtype=str)
    out["registry/learner_names"] = np.array(sorted(learners.REGISTRY_Learners), dtype=str)
    out["registry/on_policy_buffers"] = np.array([n for n in ("DummyOnPolicyBuffer", "DummyOnPolicyBuffer_Atari")
                                                  if isinstance(getattr(core, n, None), type)], dtype=str)
    out["registry/build_learner_uses_registry"] = np.array(
        "REGISTRY_Learners[self.config.learner]" in inspect.getsource(Agent._build_learner))
    exec(compile(code, "INTEGRATION.md#A", "exec"), {})
    import xuance_b200.common as xc
    for atari in (False, True):
        cls = xc.DummyOnPolicyBuffer_Atari if atari else xc.DummyOnPolicyBuffer
        seen = {}
        real_init = cls.__init__

        def spy(self, *a, **kw):
            seen.update(kw, _n_positional=len(a))
            raise RuntimeError("recorded")
        cls.__init__ = spy
        obs_space = xc.Box(0, 255, (84, 84, 4), np.uint8) if atari else xc.Box(-1, 1, (4,), np.float32)
        agent = SimpleNamespace(observation_space=obs_space, action_space=xc.Discrete(4), n_envs=4, horizon_size=8,
                                n_minibatch=2, gamma=0.99, gae_lam=0.95, is_tensor_memory=False,
                                config=Namespace(use_gae=True, use_advnorm=True, env_name="Atari" if atari else "Classic"))
        try:
            core.OnPolicyAgent._build_memory(agent, {"old_logp": ()})
        except RuntimeError:
            pass
        finally:
            cls.__init__ = real_init
        kwargs = {k: ("agent." + k if v is getattr(agent, k, None) else v) for k, v in seen.items()}
        out[f"build_memory/{atari}/kwargs"] = np.array(json.dumps(kwargs, sort_keys=True))
        out[f"build_memory/{atari}/buffer_batch"] = np.array([agent.buffer_size, agent.batch_size])

    class Rec:
        def __init__(self):
            self.calls = []

        def sample(self, idx):
            self.calls.append(("sample", np.array(idx, copy=True)))
            return {"obs": idx[:1], "actions": idx[:1], "returns": idx[:1], "values": idx[:1], "advantages": idx[:1],
                    "aux_batch": {}, "batch_size": len(idx)}

        def update(self, **samples):
            self.calls.append(("update", ",".join(sorted(samples))))
            return {"n": len(self.calls)}
    for buffer_size, batch_size, n_epochs in [(64, 16, 4), (60, 16, 3)]:
        rec = Rec()
        np.random.seed(11)
        info = core.OnPolicyAgent.train_epochs(SimpleNamespace(buffer_size=buffer_size, batch_size=batch_size, memory=rec,
                                                               learner=rec), n_epochs)
        p = f"train_epochs/{buffer_size}_{batch_size}_{n_epochs}"
        out[f"{p}/kinds"] = np.array([k for k, _ in rec.calls], dtype=str)
        out[f"{p}/sample_idx"] = np.concatenate([v for k, v in rec.calls if k == "sample"])
        out[f"{p}/sample_len"] = np.array([len(v) for k, v in rec.calls if k == "sample"])
        out[f"{p}/update_keys"] = np.array([v for k, v in rec.calls if k == "update"], dtype=str)
        out[f"{p}/info_n"] = np.array(info["n"])
    np.savez_compressed(os.path.join(HERE, "dropin_reference.npz"), **out)


def golden_running_mean_std():
    """tests/test_host_logic.py::test_running_mean_std_matches_reference: the reference's RunningMeanStd after seven updates."""
    from xuance.common.statistic_tools import RunningMeanStd
    rng = np.random.default_rng(1)
    a = RunningMeanStd((3,))
    for _ in range(7):
        a.update(rng.normal(size=(8, 3)).astype(np.float32))
    np.savez_compressed(os.path.join(HERE, "running_mean_std.npz"), env=ENV, mean=a.mean, var=a.var, count=np.array(a.count))


def _check_no_objects(out):
    bad = [k for k, v in out.items() if np.asarray(v).dtype == object]
    assert not bad, bad


GOLDENS = {"onpolicy": golden_onpolicy, "per": golden_per, "ppo": golden_ppo, "dqn": golden_dqn, "sac": golden_sac,
           "qmix": golden_qmix, "rollout_glue": golden_rollout_glue, "oracle_vs_reference": golden_oracle_vs_reference,
           "qmix_action_mask": golden_qmix_action_mask, "dropin": golden_dropin, "running_mean_std": golden_running_mean_std}


if __name__ == "__main__":
    for name in sys.argv[1:] or GOLDENS:     # python tests/golden/make_golden.py [name ...]
        GOLDENS[name]()
    for f in sorted(os.listdir(HERE)):
        if f.endswith(".npz"):
            print(f, os.path.getsize(os.path.join(HERE, f)))
