"""Generate tests/golden/ppo_gaussian_update.npz by running the UNMODIFIED reference's PPO_Learner on a Gaussian policy.

Run in the build container only (needs the reference):   python tests/golden/make_golden_ppo_gaussian.py
Same conventions and digest format as the ``ppo`` fixture of make_golden.py (whose import set-up this reuses): two updates
of GaussianActorHead + ValueHead on Basic_Identical at 17-d observations / 6-d actions, B = 32; the inputs are stored, the
initial weights are rebuilt from torch.manual_seed by the oracle and pinned by per-tensor digests."""
import os

import numpy as np
import torch

from make_golden import ENV, HERE, _learner_cfg  # noqa: E402  (puts the reference on sys.path)
from xuance.common import BaseCallback  # noqa: E402
from xuance.torch.learners import PPO_Learner  # noqa: E402
from xuance.torch.rl_models.representations.mlp import Basic_Identical  # noqa: E402
from xuance.torch.rl_models.heads import GaussianActorHead, ValueHead  # noqa: E402
from xuance.torch.rl_models.architectures.single_agent.actor_critic import SharedActorCritic  # noqa: E402

OBS_DIM, ACT_DIM, B, SEED = 17, 6, 32, 5


def golden_ppo_gaussian():
    out = {"env": ENV}
    torch.manual_seed(SEED)
    rep = Basic_Identical((OBS_DIM,), device="cpu")
    actor = GaussianActorHead(OBS_DIM, [64, 64], ACT_DIM, None, torch.nn.init.orthogonal_, torch.nn.LeakyReLU,
                              torch.nn.Tanh, "cpu")
    critic = ValueHead(OBS_DIM, [64, 64], None, torch.nn.init.orthogonal_, torch.nn.LeakyReLU, "cpu")
    model = SharedActorCritic(rep, actor, critic)
    init = {k: v.clone() for k, v in model.state_dict().items()}
    learner = PPO_Learner(_learner_cfg(ent_coef=0.01), model, BaseCallback())
    rng = np.random.default_rng(11)
    infos = []
    for it in range(2):
        obs = rng.normal(size=(B, OBS_DIM)).astype(np.float32)
        with torch.no_grad():
            dist = model(torch.from_numpy(obs)).distributions
            mu = dist.mu.numpy()
        acts = (mu + np.exp(-1.0) * rng.normal(size=(B, ACT_DIM))).astype(np.float32)
        with torch.no_grad():
            logp = dist.log_prob(torch.from_numpy(acts)).numpy()
        # old_logp spread around the current log-prob: ratios both inside and outside the clip range
        old_logp = (logp + rng.normal(size=B) * 0.3).astype(np.float32)
        s = {"obs": obs, "actions": acts, "returns": rng.normal(size=B).astype(np.float32),
             "advantages": rng.normal(size=B).astype(np.float32), "aux_batch": {"old_logp": old_logp}}
        for k in ("obs", "actions", "returns", "advantages"):
            out[f"in{it}/{k}"] = s[k]
        out[f"in{it}/old_logp"] = old_logp
        info = learner.update(**s)
        infos.append([info["actor_loss"], info["critic_loss"], info["entropy"], info["learning_rate"],
                      info["predict_value"], float(info["clip_ratio"])])
    out["infos"] = np.array(infos, dtype=np.float64)
    out["total_iters"] = learner.total_iters
    out["cfg"] = np.array([OBS_DIM, ACT_DIM, B, SEED])
    for k, v in model.state_dict().items():
        out[f"init_digest/{k}"] = np.array([v_.double().sum().item() for v_ in (init[k], init[k].abs())])
        flat = v.detach().reshape(-1)
        out[f"final_head/{k}"] = flat[:64].numpy().copy()
        out[f"final_digest/{k}"] = np.array([flat.double().sum().item(), flat.double().abs().sum().item()])
    np.savez_compressed(os.path.join(HERE, "ppo_gaussian_update.npz"), **out)


if __name__ == "__main__":
    golden_ppo_gaussian()
