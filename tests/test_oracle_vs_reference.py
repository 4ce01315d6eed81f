"""CPU: the oracle next to the unmodified reference on the seeded inputs of each test - the second way the oracle is
pinned (the first is tests/test_oracle_golden.py).  What the reference computed on these inputs is stored in
tests/golden/oracle_vs_reference.npz and tests/golden/qmix_action_mask.npz (tests/golden/make_golden.py writes both from the
reference): small results whole, buffer contents as sha256 digests, initial weights as digests (the oracle rebuilds them
from the same torch seed), final weights as a fixed element sample plus sum / abs-sum digests."""
import os
import random

import numpy as np
import pytest
import torch

from helpers import (synth_rollout, fill_buffers, qmix_episode_stream, array_digest, structure_digest, assert_same_init,
                     assert_state_close)

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
QMIX_BUFFER_KEYS = ('obs', 'actions', 'rewards', 'terminals', 'agent_mask')


@pytest.fixture(scope="module")
def ref():
    return np.load(os.path.join(G, "oracle_vs_reference.npz"), allow_pickle=False)


@pytest.mark.parametrize("seed,use_gae", [(0, True), (1, True), (2, False)])
def test_onpolicy_buffer_live(ref, seed, use_gae):
    from oracle.onpolicy import OnPolicyBufferOracle
    rng = np.random.default_rng(seed)
    N, T = 5, 33
    ro = synth_rollout(rng, N, T, (3,), obs_dtype=np.float32, p_term=0.1)
    o = OnPolicyBufferOracle((3,), (), {'old_logp': ()}, N, T, use_gae=use_gae)
    fill_buffers([o], ro, [(4, 1, np.float32(0.2)), (9, 3, 0.0), (20, 1, np.float32(-0.7))])
    p = "onpolicy/%d" % seed
    assert np.array_equal(ref[p + "/returns"], o.returns) and np.array_equal(ref[p + "/advantages"], o.advantages)
    idx = rng.permutation(N * T)[:50]
    s2 = o.sample(idx)
    for k in ('obs', 'actions', 'returns', 'values', 'advantages'):
        s1k = ref[p + "/sample/" + k]
        assert np.array_equal(s1k, s2[k]) and s1k.dtype == s2[k].dtype, k


@pytest.mark.parametrize("alpha", [0.5, 0.6])
def test_per_buffer_live(ref, alpha):
    """The reference ran with its float64 ``_max_priority`` replaced by a float32 one (canonical float32 rule,
    oracle/replay.py docstring); its sum / min trees are kept as digests of their float64 leaf arrays."""
    from oracle.replay import PerReplayOracle
    rng = np.random.default_rng(int(alpha * 10))
    N, S, B = 4, 64, 32
    o = PerReplayOracle((3,), (), N, N * S, B, alpha=alpha)
    g = {k: ref["per/%s/%s" % (alpha, k)] for k in ("step_choices", "weights", "sum_tree", "min_tree", "max_priority")}
    j = 0
    for t in range(100):
        st = (rng.normal(size=(N, 3)).astype(np.float32), rng.integers(0, 4, N), rng.normal(size=N).astype(np.float32),
              rng.random(N) < 0.1, rng.normal(size=(N, 3)).astype(np.float32))
        o.store(*st)
        if t > 10 and t % 3 == 0:
            random.seed(t)
            s2 = o.sample(0.4)
            assert np.array_equal(g["step_choices"][j], s2['step_choices']) and np.array_equal(g["weights"][j], s2['weights'])
            td = np.abs(rng.normal(size=B)).astype(np.float32)
            td[3] = 0
            o.update_priorities(s2['step_choices'], td)
            assert g["sum_tree"][j] == array_digest(np.array([o.sum[i].v.astype(np.float64) for i in range(N)]))
            assert g["min_tree"][j] == array_digest(np.array([o.min[i].v.astype(np.float64) for i in range(N)]))
            assert np.array_equal(g["max_priority"][j], o.max_priority)
            j += 1
    assert j == len(g["step_choices"])


def _qmix_oracle(n, obs_dim, A, S, total_iters, lr_decay=0.5):
    """The oracle pair of the reference's QMIX model (use_rnn, shared GRU agent, mixer 32/32) + learner; built right after
    torch.manual_seed it has the reference's initial weights (checked against the stored digests)."""
    from oracle.qmix import QMIXModelOracle, QMIXLearnerOracle
    keys = [f"agent_{i}" for i in range(n)]
    om = QMIXModelOracle(n, obs_dim, A, S)
    orc = QMIXLearnerOracle(om, keys, learning_rate=7e-4, sync_frequency=2, double_q=True, end_factor_lr_decay=lr_decay,
                            total_iters=total_iters, detach_q_eval=True)   # the reference as it is (see oracle/qmix.py)
    return keys, om, orc


def _fill_qmix_replay(ob, seed, keys, n_envs, T, obs_dim, A, S):
    for ev in qmix_episode_stream(np.random.default_rng(seed), keys, n_envs, T, obs_dim, A, S, 5):
        if ev[0] == 'store':
            ob.store(**ev[1])
        else:
            ob.finish_path(ev[1], **ev[2])


def _assert_qmix_replay(ob, keys, g, prefix):
    got = [array_digest(ob.data[k][a]) for k in QMIX_BUFFER_KEYS for a in keys]
    got += [array_digest(ob.data['filled']), array_digest(ob.data['state'])]
    names = ["%s/%s" % (k, a) for k in QMIX_BUFFER_KEYS for a in keys] + ["filled", "state"]
    for name, x, y in zip(names, g[prefix + "/digests"], got):
        assert x == y, name
    assert [ob.ptr, ob.size] == list(g[prefix + "/ptr_size"])


def test_qmix_buffer_and_learner_live(ref):
    from oracle.qmix import EpisodeReplayOracle
    torch.manual_seed(0)
    n, obs_dim, A, S, T = 5, 72, 12, 98, 12
    keys, om, orc = _qmix_oracle(n, obs_dim, A, S, int(ref["qmix/total_iters"]))
    assert_same_init(om.state_dict(), ref, "qmix/init")
    init = {k: v.clone() for k, v in om.state_dict().items()}
    n_envs, C, Be = 3, 12, 6
    ob = EpisodeReplayOracle(keys, obs_dim, S, n_envs, C, Be, T)
    _fill_qmix_replay(ob, 0, keys, n_envs, T, obs_dim, A, S)
    _assert_qmix_replay(ob, keys, ref, "qmix/buffer")
    for it in range(3):
        np.random.seed(it)
        i2 = orc.update(ob.sample())
        i1 = ref["qmix/infos"][it]
        np.testing.assert_allclose(i1[0], i2['loss_Q'], rtol=1e-5)
        np.testing.assert_allclose(i1[1], i2['predictQ'], rtol=1e-5, atol=1e-7)
        assert i1[2] == i2['learning_rate']
    sd2 = om.state_dict()
    assert_state_close(sd2, ref, "qmix/final", rtol=1e-5, atol=1e-6)
    # reference quirk pinned here: with use_rnn=True its agent networks never receive a gradient (only the mixer moves)
    assert len(ref["qmix/moved_agent_tensors"]) == 0, ref["qmix/moved_agent_tensors"]
    moved = {k for k in sd2 if k.startswith("individual_q_networks") and not torch.equal(sd2[k], init[k])}
    assert not moved, moved


def test_sac_learner_live(ref):
    """The reference's SAC learner (MLP 256-256, automatic entropy tuning) built after torch.manual_seed(0)."""
    from oracle.sac import SACModelOracle, SACLearnerOracle
    torch.manual_seed(0)
    obs_dim, act_dim, B = 17, 6, 64
    om = SACModelOracle(obs_dim, act_dim)
    assert_same_init(om.state_dict(), ref, "sac/init")
    orc = SACLearnerOracle(om, end_factor_lr_decay=0.7, total_iters=int(ref["sac/total_iters"]))
    rng = np.random.default_rng(1)
    for it in range(3):
        s = {"obs": rng.normal(size=(B, obs_dim)).astype(np.float32),
             "actions": rng.uniform(-1, 1, size=(B, act_dim)).astype(np.float32),
             "obs_next": rng.normal(size=(B, obs_dim)).astype(np.float32),
             "rewards": rng.normal(size=B).astype(np.float32), "terminals": (rng.random(B) < 0.1).astype(np.float32)}
        # the reference draws its noise from torch's global RNG: replay the same stream for the oracle
        torch.manual_seed(100 + it)
        n1 = torch.randn(B, act_dim)
        n2 = torch.randn(B, act_dim)
        i2 = orc.update(n1, n2, **s)
        for k, v in zip(("Qloss", "Ploss", "Qvalue", "alpha", "alpha_loss"), ref["sac/infos"][it]):
            np.testing.assert_allclose(i2[k], v, rtol=1e-5, atol=1e-6, err_msg=k)
    assert_state_close(om.state_dict(), ref, "sac/final", rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("kind", ["a2c", "pg", "ddqn"])
def test_sibling_learners_live(ref, kind):
    """A2C / PG / DDQN (SURVEY.md section 8f-3): oracle variants next to the reference learners (NatureCNN at 84x84x4,
    running_steps 40960, 32 envs, lr 2.5e-4 decaying to half, gradient clip 0.5, sync every 2 updates)."""
    from oracle.nets import SharedActorCriticOracle, DeepQNetworkOracle
    from oracle.learners import PPOLearnerOracle, DQNLearnerOracle
    torch.manual_seed(5)
    A, B = 5, 12
    p = "sibling/" + kind
    total_iters = int(ref[p + "/total_iters"])
    rng = np.random.default_rng(3)
    if kind == "ddqn":
        om = DeepQNetworkOracle(A)
        orc = DQNLearnerOracle(om, learning_rate=2.5e-4, sync_frequency=2, use_grad_clip=True, end_factor_lr_decay=0.5,
                               total_iters=total_iters, double_q=True)
    else:
        om = SharedActorCriticOracle(A)
        # a2c_learner.py:21: LinearLR(total_iters=config.running_steps); pg_learner.py:22: total_iters=self.total_iters
        orc = PPOLearnerOracle(om, end_factor_lr_decay=0.5, kind=kind, total_iters=4096 * 10 if kind == "a2c" else total_iters)
    assert_same_init(om.state_dict(), ref, p + "/init")
    for it in range(3):
        s = {"obs": rng.integers(0, 256, size=(B, 84, 84, 4), dtype=np.uint8).astype(np.float32),
             "actions": rng.integers(0, A, size=B).astype(np.float32),
             "returns": rng.normal(size=B).astype(np.float32), "advantages": rng.normal(size=B).astype(np.float32),
             "aux_batch": {"old_logp": np.zeros(B, np.float32)},
             "obs_next": rng.integers(0, 256, size=(B, 84, 84, 4), dtype=np.uint8).astype(np.float32),
             "rewards": rng.normal(size=B).astype(np.float32), "terminals": (rng.random(B) < 0.2).astype(np.float32)}
        i1, i2 = ref[p + "/infos"][it], orc.update(**s)
        if kind == "ddqn":
            np.testing.assert_allclose(i2["Qloss"], i1[0], rtol=1e-5)
        else:
            np.testing.assert_allclose(i2["actor_loss"], i1[0], rtol=1e-5, atol=1e-7)
            np.testing.assert_allclose(i2["entropy"], i1[1], rtol=1e-5)
    assert_state_close(om.state_dict(), ref, p + "/final", rtol=1e-5, atol=1e-6)


def test_multi_agent_vector_env_live(ref):
    """DummyVecMultiAgentEnv + XuanCeMultiAgentEnvWrapper (the QMIX caller side, vector_envs/dummy/dummy_vec_maenv.py:17-84,
    environment/utils/wrapper.py:141-226) next to the live reference classes over the SAME raw synthetic environments:
    identical observations, reward / terminated dicts, truncation flags and infos (episode_step, episode_score, agent_mask,
    avail_actions, state, reset_obs / reset_avail_actions / reset_state at episode ends) step for step.  The reference's
    results are stored as helpers.structure_digest of each, equal exactly when helpers.same_structure would hold."""
    from xuance_b200.environment.ma_envs import SyntheticSMACEnv, XuanCeMultiAgentEnvWrapper
    from xuance_b200.environment.vector_envs.dummy_vec_maenv import DummyVecMultiAgentEnv
    kw = dict(n_agents=3, obs_dim=16, state_dim=20, n_actions=5, episode_limit=7, p_death=0.1)
    n_envs = 3
    mk_own = [lambda env_seed=0: XuanCeMultiAgentEnvWrapper(SyntheticSMACEnv(seed=env_seed, **kw)) for _ in range(n_envs)]
    ov = DummyVecMultiAgentEnv(mk_own, 11)
    assert list(ref["maenv/attrs"]) == [ov.num_envs, ov.num_agents, ov.max_episode_steps]
    assert list(ref["maenv/agents"]) == list(ov.agents) and tuple(ref["maenv/state_shape"]) == ov.state_space.shape
    names, digests = list(ref["maenv/names"]), ref["maenv/digests"]
    oo, oi = ov.reset()
    assert digests[0][0] == structure_digest(oo), "reset obs"
    assert digests[0][1] == structure_digest(oi), "reset info"
    rng = np.random.default_rng(2)
    ends = 0
    for t in range(40):
        # a random AVAILABLE action per agent (the reference drew from the same availability, checked step by step)
        acts = [{a: int(rng.choice(np.flatnonzero(ov.buf_avail_actions[e][a]))) for a in ov.agents} for e in range(n_envs)]
        o = ov.step(acts)
        for name, x, y in zip(names, digests[t + 1], tuple(o) + (ov.buf_state, ov.buf_avail_actions)):
            assert x == structure_digest(y), "t=%d %s" % (t, name)
        ends += sum("reset_obs" in i for i in o[4])
    assert ends == int(ref["maenv/episode_ends"]) and ends >= 5   # episode ends (death of all agents / truncation) exercised
    ov.close()


def test_qmix_action_mask_variant_against_the_reference_with_its_slice_corrected():
    """use_rnn=True with use_actions_mask=True: the reference slices the AGENT axis of the availability mask
    (iql_learner.py:78, ``[:, 1:]``) and raises; the evidently intended statement slices the time axis (``[:, :, 1:]``).
    The oracle's masked variant (and through it xb_qmix_select_fwd's masked arg-max / target, tests/test_gpu_qmix.py) is pinned
    here against the reference learner with that ONE expression corrected in memory (tests/golden/qmix_action_mask.npz;
    nothing of the reference's source is stored in this repository).  The reference buffer's availability masks are stored
    whole; the oracle buffer rebuilds its other contents from the same seeded stream."""
    from oracle.qmix import EpisodeReplayOracle
    g = np.load(os.path.join(G, "qmix_action_mask.npz"), allow_pickle=False)
    torch.manual_seed(1)
    n, obs_dim, A, S, T = 4, 24, 7, 30, 9
    keys, om, orc = _qmix_oracle(n, obs_dim, A, S, int(g["total_iters"]))
    assert_same_init(om.state_dict(), g, "init")
    orc.use_actions_mask = True
    n_envs, C, Be = 3, 12, 6
    ob = EpisodeReplayOracle(keys, obs_dim, S, n_envs, C, Be, T)
    _fill_qmix_replay(ob, 3, keys, n_envs, T, obs_dim, A, S)
    _assert_qmix_replay(ob, keys, g, "buffer")
    avail = g["buffer/avail_actions"]                       # [n_agents, buffer_size, T + 1, A]
    assert avail.shape == (n, C, T + 1, A)

    def sample(seed):                                       # MARL_OffPolicyBuffer_RNN.sample: np.random.choice(size, batch)
        np.random.seed(seed)
        episodes = np.random.choice(ob.size, Be)
        s = ob.gather(episodes)
        s['avail_actions'] = {a: avail[i][episodes] for i, a in enumerate(keys)}
        return s
    assert tuple(g["sample_avail_shape"]) == sample(0)['avail_actions'][keys[0]].shape == (Be, T + 1, A)
    # 1. the reference as it is cannot run this configuration
    assert str(g["unpatched_error"]) in ("RuntimeError", "IndexError")
    assert int(g["bad_slice_count"]) == 1
    # 2. the same learner with the one slice corrected
    snap = {k: v.clone() for k, v in om.state_dict().items()}
    for it in range(3):
        i1, i2 = g["infos"][it], orc.update(sample(10 + it))
        np.testing.assert_allclose(i1[0], i2['loss_Q'], rtol=1e-5)
        np.testing.assert_allclose(i1[1], i2['predictQ'], rtol=1e-5, atol=1e-7)
    assert_state_close(om.state_dict(), g, "final", rtol=1e-5, atol=1e-6)
    # the masks mattered: the same first update without them has a different loss
    _, om_m, orc_m = _qmix_oracle(n, obs_dim, A, S, int(g["total_iters"]))
    _, om_u, orc_u = _qmix_oracle(n, obs_dim, A, S, int(g["total_iters"]))
    om_m.load_state_dict(snap, strict=True), om_u.load_state_dict(snap, strict=True)
    om_m.copy_target(), om_u.copy_target()
    orc_m.use_actions_mask = True
    s = sample(10)
    assert abs(orc_m.update(s)['loss_Q'] - orc_u.update(s)['loss_Q']) > 1e-6
