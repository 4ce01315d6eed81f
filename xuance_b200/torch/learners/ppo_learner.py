"""PPO-Clip learner - mirror of xuance/torch/learners/policy_gradient/ppo_learner.py:12-95.

``update(**samples)`` keeps the reference's signature, info keys and numerics (fp32 tolerance, tests/), but runs
as: network forward (cuDNN/cuBLAS via torch) -> K4 fused loss forward+backward (one launch producing dlogits,
dvalue and the logged statistics; K4-G for a Gaussian policy, which also produces dlog_std) -> torch backward through
the network into the flat gradient bucket -> [one NCCL all-reduce] -> K7 fused clip-norm + Adam.  No ``.item()`` until the info dict is built (one D2H of
8 floats; skipped entirely with ``sync=False`` as train_epochs does for all but the last minibatch)."""
import torch

from ... import _lib
from ..utils import FusedAdam, allreduce_sum_
from .learner import Learner


class PPO_Learner(Learner):
    loss_kind = 0            # K4: 0 = PPO-Clip surrogate, 1 = plain policy gradient (A2C / PG subclasses)
    adv_key = "advantages"   # which sample field weights the log-probabilities
    info_names = ("actor_loss", "critic_loss", "entropy", "learning_rate", "predict_value", "clip_ratio")

    def __init__(self, config, model, callback):
        super().__init__(config, model, callback)
        self.optimizer = FusedAdam(self.model.parameters(), self.config.learning_rate, eps=1e-5)
        self.scheduler = torch.optim.lr_scheduler.LinearLR(self.optimizer, start_factor=1.0,
                                                           end_factor=self.end_factor_lr_decay,
                                                           total_iters=self._lr_total_iters())
        self.vf_coef, self.ent_coef = getattr(config, "vf_coef", 0.0), config.ent_coef
        self.clip_range = getattr(config, "clip_range", 0.0)
        self._stats = self.optimizer.bucket.tail[:8]      # the logged sums travel in the gradient bucket's tail
        self._scratch = _lib.scratch(self.device)
        # a Gaussian policy (GaussianActorHead: mu + state-independent log_std) selects K4-G, which also needs room for the
        # per-dimension partials of its log_std gradient
        self._log_std = getattr(getattr(self.model, "actor", None), "log_std", None)
        if self._log_std is not None:
            n = _lib.load().xb_gaussian_scratch_doubles(self._log_std.numel())
            if n <= 0:
                raise ValueError("K4-G supports 1..64 action dimensions, the policy has %d" % self._log_std.numel())
            self._col_scratch = torch.zeros(n, dtype=torch.float64, device=self.device)
        self._early = None
        self._hook_early_allreduce()

    def _hook_early_allreduce(self):
        """Optional (XB_EARLY_ALLREDUCE=1): the bulk of the gradient (the 6400->512 layer and the heads, 98 % of the parameters) is
        final before the convolution backward starts, so its all-reduce can be issued there (async, on NCCL's stream) and
        what remains - [statistics | convolution gradients], the front of the bucket - is one small all-reduce at the end.
        Measured on B200: no difference at 2 GPUs (65.4 ms per step either way); at 8 GPUs the early piece does NOT hide - the
        K12 launches are 148 persistent CTAs that hold every SM, NCCL's CTAs only run at launch boundaries, and the final piece
        then waits for it: 0.20 ms of collectives exposed per update against 0.09 ms for ONE all-reduce of the whole bucket
        issued at the end (profiles/r02_scale_n8.json: phases.nccl_all_reduce vs parity_vs_1gpu.allreduce_ms).  The default
        is therefore the single collective.  Needs an encoder that reports when those gradients are in place
        (BoxNatureCNN.grads_ready) and the bucket laid out in parameter order."""
        import os
        enc = getattr(getattr(self.model, "representation", None), "_tc", None)       # set by _PixelEncoder.set_compute("tc")
        if self.world_size <= 1 or enc is None or not hasattr(enc, "grads_ready") or os.environ.get("XB_EARLY_ALLREDUCE", "0") != "1":
            return
        bucket = self.optimizer.bucket

        def ready(first_param):
            if self.world_size <= 1 or self._early is not None:
                return
            off = bucket.offset_of(first_param)
            enc_ids = {id(p) for p in enc.parameters()}
            late = {id(p) for p in (enc.fc.weight, enc.fc.bias)}
            for p, o in zip(bucket.params, bucket.offsets):      # everything from `off` on must already be final
                if (o >= off) != (id(p) in late or id(p) not in enc_ids):
                    return
            import torch.distributed as dist
            self._early = (off, dist.all_reduce(bucket.grad[off:], op=dist.ReduceOp.SUM, async_op=True))
        enc.grads_ready = ready

    def _lr_total_iters(self):
        return self.total_iters

    def estimate_total_iterations(self):
        """ppo_learner.py:28-33."""
        buffer_size = self.config.horizon_size * self.config.parallels
        update_times = self.config.running_steps // buffer_size
        return update_times * self.config.n_epochs * self.config.n_minibatch

    def _f32(self, x):
        return torch.as_tensor(x, device=self.device).to(torch.float32).contiguous()

    def _device_update(self, obs, act, ret, adv, old_logp):
        """ppo_learner.py:43-65 on the device (no host synchronisation, static shapes: CUDA-graph capturable)."""
        B = act.shape[0]
        if hasattr(self.model, "forward_raw"):
            logits, v_pred = self.model.forward_raw(obs)
        else:
            out = self.model(obs)
            logits, v_pred = out.distributions.logits, out.values
        logits_c, v_c = logits.contiguous(), v_pred.contiguous()
        A = logits_c.shape[-1]
        dlogits = torch.empty_like(logits_c)
        dvalue = torch.empty_like(v_c)
        B_total = B * self.world_size
        if self._log_std is None:
            _lib.call("xb_ppo_loss_fwd_bwd", _lib.ptr(logits_c), _lib.ptr(v_c), _lib.ptr(act), _lib.ptr(old_logp),
                      _lib.ptr(adv), _lib.ptr(ret), B, A, B_total, float(self.clip_range), float(self.vf_coef),
                      float(self.ent_coef), self.loss_kind, _lib.ptr(dlogits), _lib.ptr(dvalue), _lib.ptr(self._stats),
                      _lib.ptr(self._scratch))
            self.optimizer.zero_grad()
            torch.autograd.backward([logits_c, v_c], [dlogits, dvalue])
        else:                                                # logits_c is the Gaussian mean mu [B, D], act [B, D]
            log_std = self._log_std
            dlog_std = torch.empty_like(log_std)
            _lib.call("xb_ppo_gaussian_loss_fwd_bwd", _lib.ptr(logits_c), _lib.ptr(log_std), _lib.ptr(v_c), _lib.ptr(act),
                      _lib.ptr(old_logp), _lib.ptr(adv), _lib.ptr(ret), B, A, B_total, float(self.clip_range),
                      float(self.vf_coef), float(self.ent_coef), self.loss_kind, _lib.ptr(dlogits), _lib.ptr(dvalue),
                      _lib.ptr(dlog_std), _lib.ptr(self._stats), _lib.ptr(self._scratch), _lib.ptr(self._col_scratch))
            self.optimizer.zero_grad()
            torch.autograd.backward([logits_c, v_c, log_std], [dlogits, dvalue, dlog_std])
        if self.world_size > 1:
            if self._early is not None:                      # the tail end of the bucket is already being reduced
                off, work = self._early
                self._early = None
                allreduce_sum_(self.optimizer.bucket.grad_all[:self.optimizer.bucket.TAIL + off])
                work.wait()
            else:
                allreduce_sum_(self.optimizer.bucket.grad_all)   # ONE collective: gradient + logged statistics
        self.optimizer.launch(max_norm=self.grad_clip_norm if self.use_grad_clip else None)

    def host_pre_step(self):
        """Host half before the device update (step counter + 16-byte hyper-parameter upload)."""
        self.iterations += 1
        self.optimizer.prepare()

    def host_post_step(self):
        if self.scheduler is not None:
            self.scheduler.step()

    def update(self, sync=True, **samples):
        obs = samples['obs']
        if not hasattr(obs, "fmt"):  # PreparedObs passes through; arrays / tensors go to the device
            obs = torch.as_tensor(obs, device=self.device)
        act = self._f32(samples['actions'])
        ret = self._f32(samples['returns'])
        adv = self._f32(samples[self.adv_key])
        old_logp = self._f32(samples['aux_batch']['old_logp']) if self.loss_kind == 0 else None
        self.host_pre_step()
        info = self.callback.on_update_start(self.iterations, policy=self.model, obs=obs, act=act, returns=ret,
                                             advantages=adv, old_logp=old_logp) or {}
        self._device_update(obs, act, ret, adv, old_logp)
        self.host_post_step()
        if sync:
            info.update(self.materialize_info())
            info.update(self.callback.on_update_end(self.iterations, policy=self.model, info=info) or {})
        return info

    def materialize_info(self):
        """The single device->host read of an update: 8 floats."""
        s = self._stats.tolist()
        lr = self.optimizer.param_groups[0]['lr']
        full = dict(zip(("actor_loss", "critic_loss", "entropy", "learning_rate", "predict_value", "clip_ratio"),
                        (s[0], s[1], s[2], lr, s[3], s[4])))
        vals = {name: full[name.replace("-", "_")] for name in self.info_names}
        if self.distributed_training:
            return {f"{k}/rank_{self.rank}": v for k, v in vals.items()}
        return vals


class A2C_Learner(PPO_Learner):
    """Advantage actor-critic - mirror of xuance/torch/learners/policy_gradient/a2c_learner.py:13-85:
    a_loss = -mean(adv * logp); same value / entropy terms, optimiser recipe and info keys (hyphenated, as the reference)."""
    loss_kind = 1
    info_names = ("actor-loss", "critic-loss", "entropy", "learning_rate", "predict_value")

    def _lr_total_iters(self):
        return self.config.running_steps   # a2c_learner.py:21 decays over running_steps, not over the update count


class PG_Learner(PPO_Learner):
    """Vanilla policy gradient - mirror of xuance/torch/learners/policy_gradient/pg_learner.py:12-75:
    loss = -mean(returns * logp) - ent_coef * entropy (no value term)."""
    loss_kind = 1
    adv_key = "returns"
    info_names = ("actor-loss", "entropy", "learning_rate")

    def __init__(self, config, model, callback):
        super().__init__(config, model, callback)
        self.vf_coef = 0.0
