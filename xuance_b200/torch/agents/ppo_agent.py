"""PPO-Clip agent - mirror of xuance/torch/agents/policy_gradient/ppo_agent.py:16-181."""
from copy import deepcopy

import numpy as np
import torch

from ...common.spaces import is_discrete, space2shape
from ..utils.rollout_glue import categorical_act, gaussian_act, DeviceRunningMeanStd, ActionReadback
from ..rl_models import CategoricalActorHead, GaussianActorHead, ValueHead, SharedActorCritic, ActivationFunctions
from .on_policy import OnPolicyAgent


class PPO_Agent(OnPolicyAgent):
    def __init__(self, config, envs=None, observation_space=None, action_space=None, callback=None):
        super().__init__(config, envs, observation_space, action_space, callback)
        self.model = self._build_model()
        self.memory = self._build_memory(self.auxiliary_info_shape)
        self.learner = self._build_learner(self.config, self.model, self.callback)

    def _build_model(self):
        """ppo_agent.py:40-93 (shared representation + categorical or Gaussian actor head + value head)."""
        if not getattr(self.config, "shared_representation", True):
            raise NotImplementedError("separate actor/critic representations are outside the hot path scope")
        rep = self._build_representation(self.config.representation, self.observation_space, self.config)
        kw = dict(normalizer=self.normalize_fn, initializer=self.initializer, activation=self.activation,
                  device=self.device)
        if is_discrete(self.action_space):
            actor = CategoricalActorHead(feature_dim=rep.output_shapes['state'][0],
                                         hidden_size=self.config.actor_hidden_size, action_dim=self.action_space.n, **kw)
        else:                                  # Box: tanh-style mu MLP + state-independent log_std (ppo_agent.py:54-57)
            act_fn = ActivationFunctions[getattr(self.config, "activation_action", "tanh")]
            actor = GaussianActorHead(feature_dim=rep.output_shapes['state'][0], hidden_size=self.config.actor_hidden_size,
                                      action_dim=self.action_space.shape[0], activation_action=act_fn, **kw)
        critic = ValueHead(feature_dim=rep.output_shapes['state'][0], hidden_size=self.config.critic_hidden_size, **kw)
        return SharedActorCritic(representation=rep, actor=actor, critic=critic).to(self.device)

    @property
    def auxiliary_info_shape(self):
        return {"old_logp": ()}

    def get_aux_info(self, policy_output=None):
        return {"old_logp": policy_output.log_probs}

    # ------------------------------------------------------------------ device-side rollout (SURVEY.md section 8f-1)
    def _device_rollout_state(self):
        """Lazily built: pinned observation staging, the device running mean/std and the action read-back ring."""
        if getattr(self, "_dr", None) is None:
            shape = tuple(space2shape(self.observation_space))
            dt = torch.uint8 if np.dtype(getattr(self.observation_space, "dtype", np.float32)) == np.uint8 \
                else torch.float32
            rb = ActionReadback(self.n_envs, self.device) if is_discrete(self.action_space) else \
                ActionReadback(self.n_envs, self.device, dtype=torch.float32, width=self.action_space.shape[0])
            self._dr = {"stage": torch.zeros((self.n_envs,) + shape, dtype=dt).pin_memory(),
                        "readback": rb,
                        "rms": DeviceRunningMeanStd(shape, self.device) if self.use_obsnorm else None}
            if self.use_obsnorm:      # continue from whatever the host statistics hold (fresh, or a loaded checkpoint)
                self._dr["rms"].load_state({'count': self.obs_rms.count, 'mean': self.obs_rms.mean,
                                            'var': self.obs_rms.var})
        return self._dr

    def _sync_obs_rms_to_host(self):
        dr = getattr(self, "_dr", None)
        if dr is not None and dr["rms"] is not None:
            st = dr["rms"].state()
            self.obs_rms.count, self.obs_rms.mean, self.obs_rms.var = st['count'], st['mean'], st['var']

    def save_model(self, model_name, save_buffer=False):
        self._sync_obs_rms_to_host()
        super().save_model(model_name, save_buffer)

    def load_model(self, path, model=None, load_buffer=False):
        super().load_model(path, model, load_buffer)
        dr = getattr(self, "_dr", None)
        if dr is not None and dr["rms"] is not None:
            dr["rms"].load_state({'count': self.obs_rms.count, 'mean': self.obs_rms.mean, 'var': self.obs_rms.var})

    @torch.no_grad()
    def _device_values(self, obs_host):
        """get_terminated_values (core/on_policy.py:109-126) for the device mode: normalise with the device statistics
        (no update), one forward, one [N] read-back.  Called once per rollout and on truncated episodes only."""
        dr = self._device_rollout_state()
        x = torch.as_tensor(np.ascontiguousarray(obs_host)).to(self.device)
        if dr["rms"] is not None:
            x = dr["rms"].normalize(x.float().contiguous(), self.obsnorm_range)
        return self.model.forward_raw(x)[1].reshape(-1).cpu().numpy()

    def _train_device(self, train_steps):
        """The loop of ``train`` with the per-step host work moved to the device: ONE upload of the observations (also
        the copy the buffer stores - the reference uploads them for the forward and stores a second host copy), K11
        running-statistics + normalise, the network, K10 sample + log-prob written into the buffer's K1 staging rows,
        ONE read-back of N int32 actions, K1.  Episode bookkeeping (rewards, terminals, infos) stays on the host, where
        the environments live.  Random stream: torch's device generator (``torch.rand``) - the reference's
        ``Categorical.sample`` stream cannot be reproduced by any fused kernel; distribution and log-prob are identical.
        A Gaussian policy takes K10-G with ``torch.randn`` noise instead and reads back N x D float32 actions."""
        dr = self._device_rollout_state()
        stage, rb, rms = dr["stage"], dr["readback"], dr["rms"]
        stage_np = stage.numpy()
        stage_np[...] = self.train_envs.buf_obs
        slots = self.memory.policy_slots()
        N = self.n_envs
        gaussian = isinstance(self.model.actor, GaussianActorHead)
        train_info = {}
        for _ in range(train_steps):
            obs_d = stage.to(self.device, non_blocking=True)
            obs_in = rms.update_and_normalize(obs_d, self.obsnorm_range) if rms is not None else obs_d
            with torch.no_grad():
                logits, values = self.model.forward_raw(obs_in)
                slots["values"].copy_(values.reshape(N))
                if gaussian:
                    act = gaussian_act(logits, self.model.actor.log_std, noise=torch.randn(logits.shape, device=self.device),
                                       actions=slots["actions"], logp=slots["aux:old_logp"])
                else:
                    act = categorical_act(logits, uniforms=torch.rand(N, device=self.device), actions_f32=slots["actions"],
                                          actions_i32=rb.dev, logp=slots["aux:old_logp"])
            rb.launch(slots["actions"] if gaussian else None)
            acts = rb.wait().copy() if gaussian else rb.wait().astype(np.int64)
            next_obs, rewards, terminals, truncations, infos = self.train_envs.step(acts)
            self.callback.on_train_step(self.current_step, envs=self.train_envs, policy=self.model, obs=obs_in,
                                        policy_out=act, acts=acts, vals=slots["values"], next_obs=next_obs,
                                        rewards=rewards, terminals=terminals, truncations=truncations, infos=infos,
                                        aux_info={"old_logp": slots["aux:old_logp"]}, train_steps=train_steps)
            self.memory.store_staged(obs_in, self._process_reward(rewards), terminals)
            if self.memory.full:
                vals = self._device_values(next_obs)
                for i in range(N):
                    self.memory.finish_path(0.0 if terminals[i] else vals[i], i)
                update_info = self.train_epochs(self.n_epochs)
                self.log_infos(update_info, self.current_step)
                train_info.update(update_info)
                self.callback.on_train_epochs_end(self.current_step, policy=self.model, memory=self.memory,
                                                  current_episode=self.current_episode, train_steps=train_steps,
                                                  update_info=update_info)
                self.memory.clear()
            self.returns = self.gamma * self.returns + rewards
            stage_np[...] = next_obs          # the reference's ``obs = deepcopy(next_obs)``: straight into pinned staging
            vals_trunc = None
            for i in range(N):
                if terminals[i] or truncations[i]:
                    self.ret_rms.update(self.returns[i:i + 1])
                    self.returns[i] = 0.0
                    if self.atari and (not truncations[i]):
                        continue
                    if terminals[i]:
                        self.memory.finish_path(0.0, i)
                    else:
                        if vals_trunc is None:
                            vals_trunc = self._device_values(next_obs)
                        self.memory.finish_path(vals_trunc[i], i)
                    stage_np[i] = infos[i]["reset_obs"]
                    self.train_envs.buf_obs[i] = infos[i]["reset_obs"]
                    self.current_episode[i] += 1
                    episode_info = {
                        f"Episode-Steps/rank_{self.rank}": {f"env-{i}": infos[i]["episode_step"]},
                        f"Train-Episode-Rewards/rank_{self.rank}": {f"env-{i}": infos[i]["episode_score"]}}
                    self.log_infos(episode_info, self.current_step)
                    train_info.update(episode_info)
                    self.callback.on_train_episode_info(envs=self.train_envs, policy=self.model, env_id=i, infos=infos,
                                                        rank=self.rank, use_wandb=self.use_wandb,
                                                        current_step=self.current_step,
                                                        current_episode=self.current_episode, train_steps=train_steps)
            self.current_step += N
            self.callback.on_train_step_end(self.current_step, envs=self.train_envs, policy=self.model,
                                            train_steps=train_steps, train_info=train_info)
        self._sync_obs_rms_to_host()
        return train_info

    def train(self, train_steps):
        """ppo_agent.py:111-181: one iteration = one vector-env step; update when the horizon is full.
        ``config.device_rollout = True`` selects the device-side glue of ``_train_device`` (same loop, same buffer
        contents up to the random stream)."""
        if getattr(self.config, "device_rollout", False):
            return self._train_device(train_steps)
        train_info = {}
        obs = self.train_envs.buf_obs
        for _ in range(train_steps):
            self.obs_rms.update(obs)
            obs = self._process_observation(obs)
            policy_out = self.get_actions(obs, return_dists=False, return_logpi=True)
            acts, value = policy_out.env_actions, policy_out.values
            next_obs, rewards, terminals, truncations, infos = self.train_envs.step(acts)
            aux_info = self.get_aux_info(policy_out)
            self.callback.on_train_step(self.current_step, envs=self.train_envs, policy=self.model, obs=obs,
                                        policy_out=policy_out, acts=acts, vals=value, next_obs=next_obs,
                                        rewards=rewards, terminals=terminals, truncations=truncations, infos=infos,
                                        aux_info=aux_info, train_steps=train_steps)
            self.memory.store(obs, acts, self._process_reward(rewards), value, terminals, aux_info)
            if self.memory.full:
                vals = self.get_terminated_values(next_obs)
                for i in range(self.n_envs):
                    self.memory.finish_path(0.0 if terminals[i] else vals[i], i)
                update_info = self.train_epochs(self.n_epochs)
                self.log_infos(update_info, self.current_step)
                train_info.update(update_info)
                self.callback.on_train_epochs_end(self.current_step, policy=self.model, memory=self.memory,
                                                  current_episode=self.current_episode, train_steps=train_steps,
                                                  update_info=update_info)
                self.memory.clear()
            self.returns = self.gamma * self.returns + rewards
            obs = deepcopy(next_obs)
            for i in range(self.n_envs):
                if terminals[i] or truncations[i]:
                    self.ret_rms.update(self.returns[i:i + 1])
                    self.returns[i] = 0.0
                    if self.atari and (not truncations[i]):
                        continue
                    if terminals[i]:
                        self.memory.finish_path(0.0, i)
                    else:
                        vals = self.get_terminated_values(next_obs)
                        self.memory.finish_path(vals[i], i)
                    obs[i] = infos[i]["reset_obs"]
                    self.train_envs.buf_obs[i] = obs[i]
                    self.current_episode[i] += 1
                    episode_info = {
                        f"Episode-Steps/rank_{self.rank}": {f"env-{i}": infos[i]["episode_step"]},
                        f"Train-Episode-Rewards/rank_{self.rank}": {f"env-{i}": infos[i]["episode_score"]}}
                    self.log_infos(episode_info, self.current_step)
                    train_info.update(episode_info)
                    self.callback.on_train_episode_info(envs=self.train_envs, policy=self.model, env_id=i, infos=infos,
                                                        rank=self.rank, use_wandb=self.use_wandb,
                                                        current_step=self.current_step,
                                                        current_episode=self.current_episode, train_steps=train_steps)
            self.current_step += self.n_envs
            self.callback.on_train_step_end(self.current_step, envs=self.train_envs, policy=self.model,
                                            train_steps=train_steps, train_info=train_info)
        return train_info
