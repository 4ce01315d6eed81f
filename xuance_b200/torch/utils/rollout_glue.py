"""Device-side rollout glue (SURVEY.md section 8f-1): what the reference's rollout loop does around the network on
the host, as single launches that leave their results in HBM.

* ``categorical_act``        - K10: sample / argmax / log-prob / entropy of a categorical policy from raw logits
                               (``OnPolicyAgent.get_actions``, core/on_policy.py:128-169 +
                               ``CategoricalDistribution``, modules/distributions.py:128-162).
* ``gaussian_act``           - K10-G: the same for a diagonal Gaussian policy from its mean and log-std
                               (``DiagGaussianDistribution``, modules/distributions.py:165-197).
* ``DeviceRunningMeanStd``   - K11: ``RunningMeanStd.update`` + ``Agent._process_observation``
                               (common/statistic_tools.py:117-185, agents/base/agent.py:262-279) on device arrays.
* ``ActionReadback``         - the one device->host transfer a vector-env step needs: N int32 actions (or N x D float32
                               continuous actions) into pinned memory.
"""
import numpy as np
import torch

from ... import _lib

EPS = 1e-8   # xuance/common/common_tools.py:8


def categorical_act(logits, uniforms=None, forced_actions=None, actions_f32=None, actions_i32=None, logp=None,
                    entropy=None):
    """One K10 launch over ``logits [N, A]`` (float32, contiguous, CUDA).  Mode: ``forced_actions`` given -> log-prob of
    those; else ``uniforms`` given -> inverse-CDF draw; else argmax.  Output tensors may be passed in (e.g. rows of the
    rollout buffer's K1 staging block); missing ones among (actions_f32, logp) are allocated.  Returns a dict."""
    if not logits.is_cuda:
        raise RuntimeError("categorical_act: logits must be a CUDA tensor (no CPU fallback)")
    logits = logits.contiguous()
    if logits.dtype != torch.float32:
        logits = logits.float()
    N, A = logits.shape
    dev = logits.device
    if actions_f32 is None:
        actions_f32 = torch.empty(N, dtype=torch.float32, device=dev)
    if logp is None:
        logp = torch.empty(N, dtype=torch.float32, device=dev)
    keep = [logits]
    if uniforms is not None:
        uniforms = uniforms.to(device=dev, dtype=torch.float32).contiguous()
        keep.append(uniforms)
    if forced_actions is not None:
        forced_actions = forced_actions.to(device=dev, dtype=torch.float32).contiguous()
        keep.append(forced_actions)
    _lib.call("xb_categorical_act", _lib.ptr(logits), _lib.ptr(uniforms) if uniforms is not None else None,
              _lib.ptr(forced_actions) if forced_actions is not None else None, N, A, _lib.ptr(actions_f32),
              _lib.ptr(actions_i32) if actions_i32 is not None else None, _lib.ptr(logp),
              _lib.ptr(entropy) if entropy is not None else None)
    return {"actions": actions_f32, "actions_i32": actions_i32, "logp": logp, "entropy": entropy, "_keep": keep}


def gaussian_act(mu, log_std, noise=None, forced_actions=None, actions=None, logp=None, entropy=None):
    """One K10-G launch over ``mu [N, D]`` and ``log_std [D]`` (float32, contiguous, CUDA).  Mode: ``forced_actions`` given ->
    log-prob of those; else ``noise`` (standard normal [N, D]) given -> mu + noise * exp(log_std); else mu.  Output tensors
    may be passed in (e.g. the rollout buffer's K1 staging); missing ones among (actions, logp) are allocated."""
    if not mu.is_cuda:
        raise RuntimeError("gaussian_act: mu must be a CUDA tensor (no CPU fallback)")
    mu = mu.contiguous().float()
    log_std = log_std.detach().contiguous().float()
    N, D = mu.shape
    if log_std.numel() != D:
        raise ValueError("gaussian_act: log_std has %d entries for %d action dimensions" % (log_std.numel(), D))
    if actions is None:
        actions = torch.empty((N, D), dtype=torch.float32, device=mu.device)
    if logp is None:
        logp = torch.empty(N, dtype=torch.float32, device=mu.device)
    keep = [mu, log_std]
    for t in (noise, forced_actions):
        if t is not None and (t.shape != mu.shape or t.dtype != torch.float32 or not t.is_contiguous()):
            raise ValueError("gaussian_act: noise / forced_actions must be contiguous float32 [N, D] like mu")
    _lib.call("xb_gaussian_act", _lib.ptr(mu), _lib.ptr(log_std), _lib.ptr(noise), _lib.ptr(forced_actions), N, D,
              _lib.ptr(actions), _lib.ptr(logp), _lib.ptr(entropy))
    return {"actions": actions, "logp": logp, "entropy": entropy, "_keep": keep}


class DeviceRunningMeanStd:
    """Running mean / variance held on the device; ``count`` stays a Python float as in the reference."""

    def __init__(self, shape, device, epsilon=1e-4):
        self.shape = tuple(shape)
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("DeviceRunningMeanStd lives on a CUDA device (the host version is "
                               "xuance_b200.common.statistic_tools.RunningMeanStd)")
        self.D = int(np.prod(self.shape, dtype=np.int64)) if self.shape else 1
        self.mean = torch.zeros(self.shape, dtype=torch.float32, device=self.device)
        self.var = torch.ones(self.shape, dtype=torch.float32, device=self.device)
        self.count = epsilon

    @property
    def std(self):
        return torch.sqrt(self.var)

    def _launch(self, x, update, out, clip_range):
        if not (x.is_cuda and x.dtype == torch.float32 and x.is_contiguous()):
            raise ValueError("DeviceRunningMeanStd: x must be a contiguous float32 CUDA tensor [N, *shape]")
        N = x.shape[0]
        if x.numel() != N * self.D:
            raise ValueError("DeviceRunningMeanStd: expected [N, %s], got %s" % (self.shape, tuple(x.shape)))
        _lib.call("xb_rms_update_normalize", _lib.ptr(x), N, self.D, _lib.ptr(self.mean), _lib.ptr(self.var),
                  float(self.count), 1 if update else 0, _lib.ptr(out) if out is not None else None,
                  float(clip_range), EPS)
        if update:
            self.count = self.count + N

    def update(self, x):
        """statistic_tools.py:117-185."""
        self._launch(x, True, None, 0.0)

    def normalize(self, x, clip_range=5, out=None):
        """agent.py:273-276 with the current statistics."""
        out = torch.empty_like(x) if out is None else out
        self._launch(x, False, out, clip_range)
        return out

    def update_and_normalize(self, x, clip_range=5, out=None):
        """``obs_rms.update(obs)`` followed by ``_process_observation(obs)`` (ppo_agent.py:115-116) in one launch."""
        out = torch.empty_like(x) if out is None else out
        self._launch(x, True, out, clip_range)
        return out

    # checkpoint format of Agent.save_model (obs_rms.npy: {'count', 'mean', 'var'}; agent.py:199-229)
    def state(self):
        return {'count': self.count, 'mean': self.mean.cpu().numpy(), 'var': self.var.cpu().numpy()}

    def load_state(self, d):
        self.count = float(d['count'])
        self.mean.copy_(torch.as_tensor(np.asarray(d['mean'], np.float32)).reshape(self.shape))
        self.var.copy_(torch.as_tensor(np.asarray(d['var'], np.float32)).reshape(self.shape))


class ActionReadback:
    """Double-buffered pinned block for the per-step actions: ``launch`` enqueues the D2H copy and records an event,
    ``wait`` blocks on that event only (not on the whole device) and hands out the NumPy view.  Defaults: N int32
    (discrete actions); ``dtype=torch.float32, width=D`` holds N x D continuous actions."""

    def __init__(self, n_envs, device, dtype=torch.int32, width=None):
        shape = (n_envs,) if width is None else (n_envs, width)
        self.dev = torch.zeros(shape, dtype=dtype, device=device)
        self.host = [torch.zeros(shape, dtype=dtype).pin_memory() for _ in range(2)]
        self.evt = [torch.cuda.Event(), torch.cuda.Event()]
        self.i = 0

    def launch(self, src=None):
        """Copies ``src`` (a device tensor shaped like ``dev``, e.g. a buffer staging view the policy kernel wrote) or ``dev``."""
        self.i ^= 1
        self.host[self.i].copy_(self.dev if src is None else src, non_blocking=True)
        self.evt[self.i].record()

    def wait(self):
        self.evt[self.i].synchronize()
        return self.host[self.i].numpy()
