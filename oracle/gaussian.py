"""Torch-CPU restatement of the reference's Gaussian-policy PPO (continuous actions).  TEST INFRASTRUCTURE (see oracle/__init__).

  * Basic_Identical + GaussianActorHead + ValueHead ...... representations/mlp.py, heads/actor_head.py:45-72,
                                                          critic_head.py:9-30, wired by ppo_agent.py:40-93 (Box space)
  * SharedActorCritic ...................................... architectures/single_agent/actor_critic.py:40-72
  * DiagGaussianDistribution ............................... modules/distributions.py:165-197
  * PPO_Learner.update ...................................... learners/policy_gradient/ppo_learner.py:35-95
Modules are constructed in the reference's order (actor MLP layer by layer, then log_std, then the critic), so the same
torch.manual_seed gives the same initial weights; parameter names match the reference's state_dict.
"""
import torch
import torch.nn as nn
from torch.distributions import Normal

from .learners import PPOLearnerOracle


def _mlp(sizes, act, last_act, init=nn.init.orthogonal_):
    """mlp_block per layer (layers.py): Linear, initialiser on the weight, zero bias, then the activation (if any)."""
    mods = []
    for i in range(len(sizes) - 1):
        lin = nn.Linear(sizes[i], sizes[i + 1])
        init(lin.weight)
        nn.init.constant_(lin.bias, 0)
        mods.append(lin)
        a = act if i < len(sizes) - 2 else last_act
        if a is not None:
            mods.append(a())
    return nn.Sequential(*mods)


class GaussianActorCriticOracle(nn.Module):
    """Basic_Identical (no parameters) -> {mu MLP with activation_action, log_std = -1, value MLP}."""

    def __init__(self, obs_dim, act_dim, actor_hidden=(256, 256), critic_hidden=(256, 256), activation=nn.LeakyReLU,
                 activation_action=nn.Tanh):
        super().__init__()
        self.representation = nn.Module()
        self.actor = nn.Module()
        self.actor.mu = _mlp([obs_dim, *actor_hidden, act_dim], activation, activation_action)
        self.actor.log_std = nn.Parameter(-torch.ones((act_dim,)))
        self.critic = nn.Module()
        self.critic.values = _mlp([obs_dim, *critic_hidden, 1], activation, None)

    def forward(self, obs):
        """(DiagGaussianDistribution's Normal, values)."""
        z = torch.as_tensor(obs, dtype=torch.float32)
        return Normal(self.actor.mu(z), self.actor.log_std.exp()), self.critic.values(z).squeeze(-1)


class PPOGaussianLearnerOracle(PPOLearnerOracle):
    """PPOLearnerOracle for a GaussianActorCriticOracle: log-prob and entropy summed over the action dimensions."""

    def update(self, **samples):
        self.iterations += 1
        obs = torch.as_tensor(samples['obs'])
        act = torch.as_tensor(samples['actions'])
        ret = torch.as_tensor(samples['returns'])
        adv = torch.as_tensor(samples['advantages'])
        dist, v_pred = self.model(obs)
        log_prob = dist.log_prob(act).sum(-1)
        e_loss = dist.entropy().sum(-1).mean()
        c_loss = nn.functional.mse_loss(v_pred, ret.detach())
        if self.kind == "ppo":
            old_logp = torch.as_tensor(samples['aux_batch']['old_logp'])
            ratio = (log_prob - old_logp).exp().float()
            surrogate1 = ratio.clamp(1.0 - self.clip_range, 1.0 + self.clip_range) * adv
            surrogate2 = adv * ratio
            a_loss = -torch.minimum(surrogate1, surrogate2).mean()
        else:                      # a2c_learner.py:46-52 (w = advantages), pg_learner.py:44-47 (w = returns, no value term)
            a_loss = -((adv if self.kind == "a2c" else ret) * log_prob).mean()
            if self.kind == "pg":
                c_loss = torch.zeros(())
            ratio = torch.ones_like(log_prob)
        loss = a_loss - self.ent_coef * e_loss + self.vf_coef * c_loss
        self.optimizer.zero_grad()
        loss.backward()
        if self.use_grad_clip:
            torch.nn.utils.clip_grad_norm_(self.model.parameters(), self.grad_clip_norm)
        self.optimizer.step()
        self.scheduler.step()
        lr = self.optimizer.state_dict()['param_groups'][0]['lr']
        cr = ((ratio < 1 - self.clip_range).sum() + (ratio > 1 + self.clip_range).sum()) / ratio.shape[0]
        return {"actor_loss": a_loss.item(), "critic_loss": c_loss.item(), "entropy": e_loss.item(),
                "learning_rate": lr, "predict_value": v_pred.mean().item(), "clip_ratio": cr}
