"""Model architectures on the hot path (reference: xuance/torch/rl_models/architectures/single_agent/
{actor_critic,deep_q_network}.py, actors/gaussian_actors.py, critics/twin_critics.py).  Same attribute names
so reference checkpoints (``'policy'`` state_dict) load; no DistributedDataParallel wrappers - multi-GPU is ONE
flat-bucket all-reduce issued by the learner (DESIGN.md "Multi-GPU")."""
from copy import deepcopy

import torch
import torch.nn as nn

from ...common.spaces import is_discrete
from .heads import DuelingQValueHead, QValueHead, SAC_GaussianActorHead, GaussianActorHead, ValueHead
from .outputs import ModelOutput, StochasticActorOutput, TwinCriticOutput


class ActorCritic(nn.Module):
    """actor_critic.py:8-37 (separate actor / critic modules each owning a representation)."""

    def __init__(self, actor, critic, **kwargs):
        super().__init__()
        self.actor, self.critic = actor, critic

    def forward(self, observation, **kwargs):
        a, c = self.actor(observation, **kwargs), self.critic(observation, **kwargs)
        return ModelOutput(distributions=a.distributions, values=c.values, actor_rep_out=a.representations,
                           critic_rep_out=c.representations)

    def act(self, observation, deterministic=False, **kwargs):
        d = self.actor(observation, **kwargs).distributions
        return d.deterministic_sample() if deterministic else d.stochastic_sample()


class SharedActorCritic(nn.Module):
    """actor_critic.py:40-72: representation -> (actor head, critic head)."""

    def __init__(self, representation, actor, critic, **kwargs):
        super().__init__()
        self.representation, self.actor, self.critic = representation, actor, critic

    def forward(self, observation, **kwargs):
        rep_out = self.representation(observation, **kwargs)
        return ModelOutput(distributions=self.actor(rep_out.embeddings, **kwargs),
                           values=self.critic(rep_out.embeddings, **kwargs), rep_out=rep_out)

    def forward_raw(self, observation):
        """(logits, values) - or (mu, values) for a GaussianActorHead, whose log_std is ``self.actor.log_std`` - without
        building a torch.distributions object: the fused K4 / K4-G losses and K10 / K10-G consume these."""
        z = self.representation(observation).embeddings
        head = self.actor.mu if isinstance(self.actor, GaussianActorHead) else self.actor.logits
        return head(z), self.critic(z)

    def act(self, observation, deterministic=False, **kwargs):
        d = self.actor(self.representation(observation, **kwargs).embeddings, **kwargs)
        return d.deterministic_sample() if deterministic else d.stochastic_sample()


class DeepQNetwork(nn.Module):
    """deep_q_network.py:19-99: eval representation + Q head and their deep-copied targets."""

    q_head_cls = QValueHead

    def __init__(self, representation, hidden_size, action_space=None, normalizer=None, initializer=None,
                 activation=None, device=None, use_distributed_training=False, **kwargs):
        super().__init__()
        if not is_discrete(action_space):
            raise ValueError('action_space must be Discrete')
        self.n_actions = action_space.n
        self.device = device
        self.representation = representation
        self.target_representation = deepcopy(representation)
        self.representation_info_shape = representation.output_shapes
        self.eval_Q_head = self.q_head_cls(feature_dim=self.representation_info_shape['state'][0],
                                           hidden_size=hidden_size, n_actions=self.n_actions, normalizer=normalizer,
                                           initializer=initializer, activation=activation, device=device)
        self.target_Q_head = deepcopy(self.eval_Q_head)
        self.distributed_training = use_distributed_training

    def eval_parameters(self):
        return list(self.representation.parameters()) + list(self.eval_Q_head.parameters())

    def target_parameters(self):
        return list(self.target_representation.parameters()) + list(self.target_Q_head.parameters())

    def forward(self, observation, **kwargs):
        rep = self.representation(observation)
        q = self.eval_Q_head(rep.embeddings)
        return ModelOutput(actions=q.argmax(dim=-1), values=q, rep_out=rep)

    def act(self, observation, deterministic=True, epsilon_greedy=0.0, **kwargs):
        greedy = self(observation).actions
        if deterministic or epsilon_greedy <= 0.0:
            return greedy
        rand = torch.randint(low=0, high=self.n_actions, size=greedy.shape, device=greedy.device)
        mask = torch.rand(greedy.shape, device=greedy.device) < epsilon_greedy
        return torch.where(mask, rand, greedy)

    def target(self, observation, **kwargs):
        rep = self.target_representation(observation)
        return ModelOutput(values=self.target_Q_head(rep.embeddings))

    def copy_target(self):
        for ep, tp in zip(self.representation.parameters(), self.target_representation.parameters()):
            tp.data.copy_(ep)
        for ep, tp in zip(self.eval_Q_head.parameters(), self.target_Q_head.parameters()):
            tp.data.copy_(ep)


class DuelingDeepQNetwork(DeepQNetwork):
    """deep_q_network.py:102-103."""
    q_head_cls = DuelingQValueHead


class GaussianActor(nn.Module):
    """actors/gaussian_actors.py:10-52."""

    actor_head_cls = GaussianActorHead

    def __init__(self, representation, actor_hidden_size, action_space=None, normalizer=None, initializer=None,
                 activation=None, activation_action=None, device=None, **kwargs):
        super().__init__()
        self.action_space = action_space
        self.action_dim = action_space.shape[0]
        self.representation = representation
        self.representation_info_shape = representation.output_shapes
        self.actor_head = self.actor_head_cls(feature_dim=self.representation_info_shape['state'][0],
                                              hidden_size=actor_hidden_size, action_dim=self.action_dim,
                                              normalizer=normalizer, initializer=initializer, activation=activation,
                                              activation_action=activation_action, device=device)

    def forward(self, observation, avail_actions=None, **kwargs):
        rep_out = self.representation(observation, **kwargs)
        return StochasticActorOutput(representations=rep_out,
                                     distributions=self.actor_head(rep_out.embeddings, **kwargs))


class SAC_GaussianActor(GaussianActor):
    actor_head_cls = SAC_GaussianActorHead


class TwinActionValueCritic(nn.Module):
    """critics/twin_critics.py:11-62: two (representation, ValueHead) towers over concat(features, action)."""

    def __init__(self, representation, action_space, critic_hidden_size, normalizer=None, initializer=None,
                 activation=None, device=None, **kwargs):
        super().__init__()
        self.action_space = action_space
        self.action_dim = action_space.shape[-1]
        self.representation_1 = representation
        self.representation_2 = deepcopy(representation)
        self.representation_info_shape = representation.output_shapes
        self.feature_dim = self.representation_info_shape['state'][0] + self.action_dim
        kw = dict(feature_dim=self.feature_dim, hidden_size=critic_hidden_size, normalizer=normalizer,
                  initializer=initializer, activation=activation, device=device)
        self.critic_head_1 = ValueHead(**kw)
        self.critic_head_2 = ValueHead(**kw)

    def forward(self, observation, actions, **kwargs):
        r1, r2 = self.representation_1(observation), self.representation_2(observation)
        return TwinCriticOutput(
            representations_1=r1, representations_2=r2,
            values_1=self.critic_head_1(torch.concat([r1.embeddings, actions], dim=-1)),
            values_2=self.critic_head_2(torch.concat([r2.embeddings, actions], dim=-1)))


class SoftActorCritic(ActorCritic):
    """actor_critic.py:107-159."""

    def __init__(self, actor, critic, **kwargs):
        super().__init__(actor, critic, **kwargs)
        self.target_critic = deepcopy(critic)

    def forward(self, observation, **kwargs):
        a = self.actor(observation, **kwargs)
        c = self.critic(observation, a.actions, **kwargs)
        return ModelOutput(distributions=a.distributions, values=c, actor_rep_out=a.representations)

    def act(self, observation, deterministic=False, **kwargs):
        d = self.actor(observation, **kwargs).distributions
        return d.activated_deterministic_sample() if deterministic else d.activated_rsample()

    def Qpolicy(self, observation, noise=None):
        d = self.actor(observation).distributions
        act_sample, log_prob = d.activated_rsample_and_logprob(noise)
        v1, v2 = self.Qaction(observation, act_sample)
        return log_prob, v1, v2

    def Qtarget(self, observation, noise=None):
        d = self.actor(observation).distributions
        act_sample, log_prob = d.activated_rsample_and_logprob(noise)
        out = self.target_critic(observation, act_sample)
        return log_prob, torch.min(out.values_1, out.values_2)

    def Qaction(self, observation, action):
        out = self.critic(observation, action)
        return out.values_1, out.values_2

    def soft_update(self, tau=0.005):
        for ep, tp in zip(self.critic.parameters(), self.target_critic.parameters()):
            tp.data.mul_(1 - tau)
            tp.data.add_(tau * ep.data)
