"""Shared builders for the parity tests."""
import numpy as np
import torch
import torch.nn as nn


def synth_rollout(rng, N, T, obs_shape=(84, 84, 4), n_actions=4, obs_dtype=np.uint8, p_term=0.01):
    """Synthetic rollout of SURVEY.md section 8d: uint8 frames, sign-clipped rewards, N(0,1) values, rare terminals."""
    if obs_dtype == np.uint8:
        obs = rng.integers(0, 256, size=(T, N) + tuple(obs_shape), dtype=np.uint8)
    else:
        obs = rng.normal(size=(T, N) + tuple(obs_shape)).astype(np.float32)
    acts = rng.integers(0, n_actions, size=(T, N))
    rews = rng.choice(np.array([-1.0, 0.0, 1.0], np.float32), size=(T, N), p=[0.05, 0.9, 0.05])
    vals = rng.normal(size=(T, N)).astype(np.float32)
    terms = rng.random((T, N)) < p_term
    logits = rng.normal(size=(T, N, n_actions)).astype(np.float32)
    lse = np.log(np.exp(logits).sum(-1))
    logp = (np.take_along_axis(logits, acts[..., None], -1)[..., 0] - lse).astype(np.float32)
    boot = rng.normal(size=N).astype(np.float32)
    return dict(obs=obs, acts=acts, rews=rews, vals=vals, terms=terms, logp=logp, boot=boot)


def fill_buffers(buffers, ro, mid_finishes=()):
    """Feed the same rollout to every buffer (oracle / product / reference share the API).
    mid_finishes: iterable of (t, env, val) - finish_path(val, env) issued right after step t is stored."""
    T = ro["rews"].shape[0]
    mids = {}
    for t, e, v in mid_finishes:
        mids.setdefault(t, []).append((e, v))
    for t in range(T):
        for b in buffers:
            b.store(ro["obs"][t], ro["acts"][t], ro["rews"][t], ro["vals"][t], ro["terms"][t],
                    {"old_logp": ro["logp"][t]})
        for e, v in mids.get(t, []):
            for b in buffers:
                b.finish_path(v, e)
    N = ro["rews"].shape[1]
    for i in range(N):
        val = 0.0 if ro["terms"][T - 1, i] else ro["boot"][i]
        for b in buffers:
            b.finish_path(val, i)


def build_product_ppo_model(n_actions, device, hwc=(84, 84, 4)):
    from xuance_b200.torch.rl_models import AC_CNN_Atari, CategoricalActorHead, ValueHead, SharedActorCritic
    rep = AC_CNN_Atari(input_shape=hwc, kernels=[8, 4, 3], strides=[4, 2, 1], filters=[32, 64, 64],
                       activation=nn.ReLU, device=device, fc_hidden_sizes=[512])
    actor = CategoricalActorHead(512, [], n_actions, None, nn.init.orthogonal_, nn.ReLU, device)
    critic = ValueHead(512, [], None, nn.init.orthogonal_, nn.ReLU, device)
    return SharedActorCritic(rep, actor, critic)


def ppo_config(device, **kw):
    from argparse import Namespace
    cfg = dict(distributed_training=False, episode_length=1000, use_grad_clip=True, grad_clip_norm=0.5,
               device=device, model_dir="/tmp/xb_models", running_steps=10_000_000, parallels=256,
               learning_rate=2.5e-4, use_linear_lr_decay=True, end_factor_lr_decay=0.5, horizon_size=128,
               n_epochs=4, n_minibatch=4, vf_coef=0.25, ent_coef=0.01, clip_range=0.2, gamma=0.99)
    cfg.update(kw)
    return Namespace(**cfg)


def qmix_episode_stream(rng, keys, n_envs, T, obs_dim, A, S, episodes):
    """Yields ('store', step_dict) / ('finish', env, terminal_dict) events of a synthetic SMAC-shaped rollout."""
    for ep in range(episodes):
        L = rng.integers(max(2, T // 3), T + 1, size=n_envs)
        for t in range(T):
            yield ('store', dict(
                obs={k: rng.normal(size=(n_envs, obs_dim)).astype(np.float32) for k in keys},
                actions={k: rng.integers(0, A, n_envs) for k in keys},
                rewards={k: rng.normal(size=n_envs).astype(np.float32) for k in keys},
                terminals={k: (rng.random(n_envs) < 0.1) for k in keys},
                agent_mask={k: np.ones(n_envs, bool) for k in keys},
                state=rng.normal(size=(n_envs, S)).astype(np.float32), episode_steps=np.full(n_envs, t)))
            for e in range(n_envs):
                if t + 1 == L[e]:
                    yield ('finish', e, dict(episode_step=t + 1,
                                             obs={k: rng.normal(size=obs_dim).astype(np.float32) for k in keys},
                                             state=rng.normal(size=S).astype(np.float32)))


def flatten(obj, path=""):
    """Nested dict / list / tuple / ndarray / scalar -> {path: ndarray}, the form the golden .npz files store results in."""
    out = {}
    if isinstance(obj, dict):
        for k in obj:
            out.update(flatten(obj[k], "%s/%s" % (path, k)))
    elif isinstance(obj, (list, tuple)):
        out[path + "#len"] = np.array(len(obj))
        for i, x in enumerate(obj):
            out.update(flatten(x, "%s[%d]" % (path, i)))
    else:
        out[path] = np.asarray(obj)
    return out


def array_digest(a):
    """sha256 of dtype, shape and bytes: a bit-exact stand-in for an array too large to store."""
    import hashlib
    a = np.ascontiguousarray(a)
    return hashlib.sha256(("%s%s" % (a.dtype.str, a.shape)).encode() + a.tobytes()).hexdigest()


def structure_digest(obj):
    """sha256 over the paths, shapes and values (as float64, or text) of a nested result: equal exactly when
    same_structure(a, b) holds for the two objects."""
    import hashlib
    h = hashlib.sha256()
    for path, v in sorted(flatten(obj).items()):
        v = v.astype(np.float64) if v.dtype.kind in "biuf" else v.astype(str)
        h.update(("%s%s%s" % (path, v.dtype.kind, v.shape)).encode() + np.ascontiguousarray(v).tobytes())
    return h.hexdigest()


def state_sample_index(n, size=64):
    """The fixed element sample of an n-element tensor that golden files keep (all of it when small)."""
    return np.arange(n) if n <= size else np.sort(np.random.default_rng(n).choice(n, size, replace=False))


def record_state(out, prefix, state_dict, sample=True):
    """Stores, per tensor (in state_dict order, under /keys), float64 sum and abs-sum digests and (sample=True) a fixed element sample."""
    out[prefix + "/keys"] = np.array(list(state_dict), dtype=str)
    flats = [v.detach().reshape(-1).numpy().astype(np.float64) for v in state_dict.values()]
    out[prefix + "/digest"] = np.array([[f.sum(), np.abs(f).sum()] for f in flats])
    if sample:
        out[prefix + "/val"] = np.concatenate([f[state_sample_index(f.size)] for f in flats]).astype(np.float32)


def assert_state_close(state_dict, g, prefix, rtol, atol):
    """Elementwise allclose on the recorded sample; the abs-sum over ALL elements within the bound elementwise closeness
    implies (n * atol + rtol * sum|expected|)."""
    keys = list(g[prefix + "/keys"])
    assert sorted(state_dict) == sorted(keys), (sorted(state_dict), sorted(keys))
    pos = 0
    for k, (_, ref_abs) in zip(keys, g[prefix + "/digest"]):
        flat = state_dict[k].detach().reshape(-1).cpu().numpy()
        idx = state_sample_index(flat.size)
        np.testing.assert_allclose(flat[idx], g[prefix + "/val"][pos:pos + idx.size], rtol=rtol, atol=atol, err_msg=k)
        pos += idx.size
        got_abs = np.abs(flat.astype(np.float64)).sum()
        assert abs(got_abs - ref_abs) <= flat.size * atol + rtol * ref_abs, (k, got_abs, ref_abs)


def assert_same_init(state_dict, g, prefix):
    """Initial weights rebuilt from the seed equal the reference's (float64 sum and abs-sum of every tensor).  rtol 1e-6:
    torch's orthogonal_ initialiser runs a LAPACK QR whose last bits depend on the host CPU; a different construction
    order changes the digests at order 1.  The signed sum cancels, so its tolerance is taken relative to the abs-sum."""
    keys = list(g[prefix + "/keys"])
    assert sorted(state_dict) == sorted(keys), (sorted(state_dict), sorted(keys))
    for k, (ref_sum, ref_abs) in zip(keys, g[prefix + "/digest"]):
        flat = state_dict[k].detach().reshape(-1).double()
        np.testing.assert_allclose(flat.abs().sum().item(), ref_abs, rtol=1e-6, err_msg=k)
        np.testing.assert_allclose(flat.sum().item(), ref_sum, rtol=0, atol=1e-6 * ref_abs, err_msg=k)


def same_structure(a, b, path=""):
    """Structural equality of nested dict / list / ndarray / scalar results."""
    if isinstance(a, dict):
        assert isinstance(b, dict) and set(a) == set(b), (path, sorted(a), sorted(b) if isinstance(b, dict) else b)
        for k in a:
            same_structure(a[k], b[k], path + "/" + str(k))
    elif isinstance(a, (list, tuple)):
        assert len(a) == len(b), path
        for i, (x, y) in enumerate(zip(a, b)):
            same_structure(x, y, path + "[%d]" % i)
    elif isinstance(a, np.ndarray) or isinstance(b, np.ndarray):
        assert np.array_equal(np.asarray(a), np.asarray(b)), path
    else:
        assert a == b, (path, a, b)
