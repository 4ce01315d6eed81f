"""HBM-resident rollout / replay buffers behind the reference's buffer API.

Drop-in mirror of ``xuance/common/memory_tools.py`` (reference v1.4.4): same class names, constructor
arguments, ``store / finish_path / sample / clear / full / ptr / size / start_ids`` surface and the same sample
dict keys - but the arrays live in device memory, laid out ``[n_envs, n_size, ...]`` exactly like the reference's
``create_memory`` (memory_tools.py:12-40) so a flat slot index ``env * n_size + step`` addresses both.
All data movement and arithmetic goes through the C-ABI (include/xb200.h): K1 store, K2 GAE scan, K3 gathers,
K5 prioritized-replay trees.  Returned batches are CUDA tensors; the reference learners wrap samples with
``torch.as_tensor(x, device=...)`` which is a no-op for them (SURVEY.md section 8b "Ownership").

Deliberate, documented departures (SURVEY.md appendix B): ``clear()`` resets cursors instead of re-allocating
(#6); image replay is stored as uint8 (#9); PER trees follow the canonical float32 rule (#10).
"""
import random
from abc import ABC, abstractmethod
from typing import Optional

import numpy as np
import torch

from .. import _lib
from .spaces import space2shape


def _as_device(x, device, dtype=None):
    """Host array / scalar / tensor -> device tensor."""
    if isinstance(x, torch.Tensor):
        t = x
    else:
        t = torch.from_numpy(np.ascontiguousarray(np.asarray(x)))
    if dtype is not None and t.dtype != dtype:
        t = t.to(dtype)
    return t if t.device == device else t.to(device, non_blocking=True)


class PreparedObs:
    """Observations already converted for the network (u8/255 -> float, layout chosen by the model)."""

    def __init__(self, tensor, fmt, hwc):
        self.tensor, self.fmt, self.hwc = tensor, fmt, hwc
        self._n = tensor.shape[1] if fmt in (_lib.OBS_PLANES2, _lib.OBS_PLANES3, _lib.OBS_PLANE_RAW) else tensor.shape[0]
        self.shape = (self._n,) + tuple(hwc)

    def __len__(self):
        return self._n


class Buffer(ABC):
    """Base class (reference memory_tools.py:87-142)."""

    def __init__(self, observation_space, action_space, auxiliary_info_shape, num_envs, buffer_size, device="cuda:0"):
        assert buffer_size % num_envs == 0, "buffer_size must be divisible by the number of envs (parallels)"
        self.observation_space, self.action_space = observation_space, action_space
        self.auxiliary_shape = auxiliary_info_shape
        self.n_envs, self.buffer_size = num_envs, buffer_size
        self.n_size = buffer_size // num_envs
        self.ptr, self.size = 0, 0
        self.device = torch.device(device if not isinstance(device, int) else "cuda:%d" % device)
        if self.device.type != "cuda":
            raise RuntimeError("xuance_b200 buffers are device-resident: device must be a CUDA device, got %s "
                               "(there is no CPU fallback)" % (self.device,))
        _lib.load()
        _lib.use_device(self.device)

    @property
    def full(self):
        return self.size >= self.n_size

    @abstractmethod
    def store(self, *args):
        raise NotImplementedError

    @abstractmethod
    def clear(self, *args):
        raise NotImplementedError

    @abstractmethod
    def sample(self, *args):
        raise NotImplementedError

    def finish_path(self, *args):
        pass

    # ------------------------------------------------------------------ checkpoint (SURVEY.md section 8f-4)
    # The reference never saves its buffers (learners/base/drl_learner.py:64-93 holds the policy and optimiser only), so a
    # resumed off-policy run starts from an empty replay.  ``state_dict`` / ``load_state_dict`` move the HBM arrays, the
    # ring cursors and (PER) the trees through host memory; ``Agent.save_model(..., save_buffer=True)`` writes them next
    # to the ``.pth``.
    _ckpt_tensors = ()      # attribute names of device tensors (None entries are skipped)
    _ckpt_host = ()         # attribute names of host tensors / NumPy arrays

    def state_dict(self):
        sd = {"class": type(self).__name__, "n_envs": self.n_envs, "n_size": self.n_size, "ptr": int(self.ptr),
              "size": int(self.size)}
        for name in self._ckpt_tensors:
            t = getattr(self, name, None)
            if t is not None:
                sd[name] = t.detach().cpu()
        for name in self._ckpt_host:
            v = getattr(self, name)
            sd[name] = v.clone() if isinstance(v, torch.Tensor) else np.array(v, copy=True)
        return sd

    def load_state_dict(self, sd):
        if sd.get("class") != type(self).__name__ or sd["n_envs"] != self.n_envs or sd["n_size"] != self.n_size:
            raise ValueError("buffer checkpoint is for %s[%s x %s], this buffer is %s[%d x %d]" % (
                sd.get("class"), sd.get("n_envs"), sd.get("n_size"), type(self).__name__, self.n_envs, self.n_size))
        for name in self._ckpt_tensors:
            t = getattr(self, name, None)
            if t is None:
                continue
            src = sd[name]
            if tuple(src.shape) != tuple(t.shape) or src.dtype != t.dtype:
                raise ValueError("buffer checkpoint field %s: %s %s, expected %s %s" % (
                    name, tuple(src.shape), src.dtype, tuple(t.shape), t.dtype))
            t.copy_(src)
        for name in self._ckpt_host:
            v = getattr(self, name)
            if isinstance(v, torch.Tensor):
                v.copy_(sd[name])
            else:
                v[...] = sd[name]
        self.ptr, self.size = int(sd["ptr"]), int(sd["size"])
        self._after_load()

    def _after_load(self):
        pass

    # ------------------------------------------------------------------ shared helpers
    def _alloc_rows(self, shape, dtype):
        return torch.zeros((self.n_envs, self.n_size) + tuple(shape), dtype=dtype, device=self.device)

    def _store_rows(self, dst, data, t):
        """dst[:, t] = data for a [N, T, *shape] buffer (K1 rows path)."""
        src = _as_device(data, self.device, dst.dtype).reshape(self.n_envs, -1)
        if not src.is_contiguous():
            src = src.contiguous()
        row_bytes = src.shape[1] * src.element_size()
        _lib.call("xb_rollout_store", _lib.ptr(dst), _lib.ptr(src), row_bytes, None, None, 0,
                  self.n_envs, self.n_size, int(t))

    def _gather_rows(self, src, flat_idx, out=None):
        row_shape = tuple(src.shape[2:])
        row_bytes = int(np.prod(row_shape, dtype=np.int64)) * src.element_size() if row_shape else src.element_size()
        B = flat_idx.numel()
        if out is None:
            out = torch.empty((B,) + row_shape, dtype=src.dtype, device=self.device)
        _lib.call("xb_gather_rows", _lib.ptr(src), _lib.ptr(flat_idx), B, row_bytes, _lib.ptr(out))
        return out

    def _index_tensor(self, idx):
        if isinstance(idx, torch.Tensor):
            return idx.to(device=self.device, dtype=torch.int64).contiguous()
        return _as_device(np.asarray(idx, dtype=np.int64), self.device)


# =====================================================================================================
# On-policy rollout buffer + GAE
# =====================================================================================================
class DummyOnPolicyBuffer(Buffer):
    """Device-resident mirror of DummyOnPolicyBuffer (reference memory_tools.py:182-287).

    Scalar fields live in ONE float32 tensor ``_fields[F, N, T]`` ordered
    ``rewards, terminals, actions*, values, aux..., returns, advantages`` (* only for a scalar action space) so
    that one K1 launch stores a step and one K3 launch gathers a minibatch.  ``finish_path`` only records the
    segment boundary (host side, pinned); the returns/advantages of ALL envs and segments are computed by one
    K2 launch the first time they are needed."""

    obs_dtype = torch.float32
    _ckpt_tensors = ("_obs", "_act_rows", "_fields")
    _ckpt_host = ("_seg_end_h", "_boot_h", "_covered_h", "start_ids")

    def _after_load(self):
        self._gae_dirty = True      # returns / advantages are recomputed from the restored segment bookkeeping

    def __init__(self, observation_space, action_space, auxiliary_shape, n_envs, horizon_size,
                 use_gae=True, use_advnorm=True, gamma=0.99, gae_lam=0.95, device="cuda:0"):
        self.buffer_size = horizon_size * n_envs
        super().__init__(observation_space, action_space, auxiliary_shape, n_envs, self.buffer_size, device)
        self.horizon_size = self.n_size = horizon_size
        self.use_gae, self.use_advnorm = use_gae, use_advnorm
        self.gamma, self.gae_lam = gamma, gae_lam
        self.start_ids = np.zeros(self.n_envs, np.int64)
        obs_shape = space2shape(self.observation_space)
        if isinstance(obs_shape, dict):
            raise NotImplementedError("dict observation spaces are outside the hot path (SURVEY.md section 8)")
        self._obs_shape = tuple(obs_shape)
        self._act_shape = tuple(space2shape(self.action_space))
        self._aux_keys = list((auxiliary_shape or {}).keys())
        for k in self._aux_keys:
            if tuple(auxiliary_shape[k]) != ():
                raise NotImplementedError("only scalar auxiliary infos are on the hot path (e.g. old_logp)")
        self._scalar_action = self._act_shape == ()
        names = ["rewards", "terminals"] + (["actions"] if self._scalar_action else []) + ["values"]
        names += ["aux:" + k for k in self._aux_keys]
        self._n_store = len(names)
        names += ["returns", "advantages"]
        self._names = names
        self._fid = {n: i for i, n in enumerate(names)}
        self._gather_first = 2  # gathered sub-block = everything after rewards, terminals
        N, T = self.n_envs, self.n_size
        self._obs = self._alloc_rows(self._obs_shape, self.obs_dtype)
        self._act_rows = None if self._scalar_action else self._alloc_rows(self._act_shape, torch.float32)
        self._fields = torch.zeros((len(names), N, T), dtype=torch.float32, device=self.device)
        # GAE bookkeeping: host (pinned) master copies + device mirrors uploaded when dirty
        self._seg_end_h = torch.zeros((N, T), dtype=torch.uint8).pin_memory()
        self._boot_h = torch.zeros((N, T), dtype=torch.float32).pin_memory()
        self._covered_h = torch.zeros((N,), dtype=torch.int32).pin_memory()
        self._seg_end = torch.zeros((N, T), dtype=torch.uint8, device=self.device)
        self._boot = torch.zeros((N, T), dtype=torch.float32, device=self.device)
        self._covered = torch.zeros((N,), dtype=torch.int32, device=self.device)
        self._gae_dirty = False
        # staging: double-buffered pinned host blocks for numpy inputs
        self._stage_i = 0
        self._stage_scal = [torch.zeros((self._n_store, N), dtype=torch.float32).pin_memory() for _ in range(2)]
        self._stage_obs = [torch.zeros((N,) + self._obs_shape, dtype=self.obs_dtype).pin_memory() for _ in range(2)]
        self._stage_evt = [None, None]
        self._scratch = _lib.scratch(self.device)
        self._stats = torch.zeros(2, dtype=torch.float32, device=self.device)
        self.ptr, self.size = 0, 0

    # -------- reference-shaped views (device tensors)
    @property
    def observations(self):
        return self._obs

    @property
    def actions(self):
        return self._fields[self._fid["actions"]] if self._scalar_action else self._act_rows

    @property
    def rewards(self):
        return self._fields[self._fid["rewards"]]

    @property
    def terminals(self):
        return self._fields[self._fid["terminals"]]

    @property
    def values(self):
        return self._fields[self._fid["values"]]

    @property
    def returns(self):
        self._ensure_gae()
        return self._fields[self._fid["returns"]]

    @property
    def advantages(self):
        self._ensure_gae()
        return self._fields[self._fid["advantages"]]

    @property
    def auxiliary_infos(self):
        return {k: self._fields[self._fid["aux:" + k]] for k in self._aux_keys}

    def clear(self):
        """Reference :221-230 re-allocates zeroed arrays; here the cursors and the GAE bookkeeping are reset and
        the two derived fields zeroed (contents of the other fields are overwritten before they are read)."""
        self.ptr, self.size = 0, 0
        self._seg_end_h.zero_()
        self._boot_h.zero_()
        self._covered_h.zero_()
        self._fields[self._fid["returns"]:].zero_()
        self._gae_dirty = True

    # -------- K1
    def store(self, obs, acts, rews, value, terminals, aux_info=None):
        """reference :232-240.  Inputs: numpy arrays (host, as produced by the vector env / get_actions) or CUDA
        tensors.  One K1 launch writes the observation rows and every scalar field of step ``ptr``."""
        N, T, t = self.n_envs, self.n_size, self.ptr
        aux_info = aux_info or {}
        scal_in = [rews, terminals] + ([acts] if self._scalar_action else []) + [value]
        scal_in += [aux_info[k] for k in self._aux_keys]
        on_dev = all(isinstance(x, torch.Tensor) and x.is_cuda for x in scal_in)
        if on_dev:
            scal = torch.stack([x.to(torch.float32).reshape(N) for x in scal_in])
        else:
            i = self._stage_i
            if self._stage_evt[i] is not None:
                self._stage_evt[i].synchronize()
            host = self._stage_scal[i].numpy()
            for f, x in enumerate(scal_in):
                host[f] = x.detach().cpu().numpy() if isinstance(x, torch.Tensor) else x
            scal = self._stage_scal[i].to(self.device, non_blocking=True)
        pinned = None
        if isinstance(obs, np.ndarray) and obs.flags["C_CONTIGUOUS"] and obs.dtype == np.dtype(str(self.obs_dtype).split(".")[-1]):
            cand = torch.from_numpy(obs)
            if cand.is_pinned():   # caller's array already lives in pinned memory: DMA straight from it
                pinned = cand
        if isinstance(obs, torch.Tensor) and obs.is_cuda:
            obs_d = obs.to(self.obs_dtype).reshape(N, -1).contiguous()
        elif pinned is not None:
            obs_d = pinned.to(self.device, non_blocking=True).reshape(N, -1)
        else:
            i = self._stage_i
            if self._stage_evt[i] is not None:
                self._stage_evt[i].synchronize()
            self._stage_obs[i].numpy()[...] = obs.cpu().numpy() if isinstance(obs, torch.Tensor) else obs
            obs_d = self._stage_obs[i].to(self.device, non_blocking=True).reshape(N, -1)
        row_bytes = obs_d.shape[1] * obs_d.element_size()
        _lib.call("xb_rollout_store", _lib.ptr(self._obs), _lib.ptr(obs_d), row_bytes,
                  _lib.ptr(self._fields), _lib.ptr(scal), self._n_store, N, T, t)
        if not on_dev or not (isinstance(obs, torch.Tensor) and obs.is_cuda):
            evt = torch.cuda.Event()
            evt.record()
            self._stage_evt[self._stage_i] = evt
            self._stage_i ^= 1
        if not self._scalar_action:
            self._store_rows(self._act_rows, acts, t)
        self.ptr = (self.ptr + 1) % self.n_size
        self.size = min(self.size + 1, self.n_size)

    # -------- device-side rollout (SURVEY.md section 8f-1): the policy kernel writes its outputs for the step being
    # collected straight into the K1 staging block; after the env step only rewards / terminals cross PCIe.
    def policy_slots(self):
        """float32 [N] device views {'actions', 'values', 'aux:<key>'...} of the persistent staging block that
        ``store_staged`` hands to K1.  Fill them (e.g. K10 ``xb_categorical_act``) before calling ``store_staged``.
        For a vector action space 'actions' is a float32 [N, *action_shape] staging tensor of its own (K10-G
        ``xb_gaussian_act`` writes it), stored with the same rows path ``store`` uses for vector actions."""
        if getattr(self, "_dev_scal", None) is None:
            N = self.n_envs
            self._dev_scal = torch.zeros((self._n_store, N), dtype=torch.float32, device=self.device)
            self._dev_act = None if self._scalar_action else \
                torch.zeros((N,) + self._act_shape, dtype=torch.float32, device=self.device)
            self._stage_rt = [torch.zeros((2, N), dtype=torch.float32).pin_memory() for _ in range(2)]
            self._stage_rt_evt = [None, None]
            self._stage_rt_i = 0
        slots = {n: self._dev_scal[self._fid[n]] for n in self._names[2:self._n_store]}
        if not self._scalar_action:
            slots["actions"] = self._dev_act
        return slots

    def store_staged(self, obs, rews, terminals):
        """``store`` for a step whose actions / values / aux already sit in ``policy_slots()``: ``obs`` is the CUDA
        tensor the policy just consumed (no second upload), ``rews`` / ``terminals`` are the env's host arrays."""
        self.policy_slots()
        N, T, t = self.n_envs, self.n_size, self.ptr
        if not (isinstance(obs, torch.Tensor) and obs.is_cuda):
            raise ValueError("store_staged: obs must be the CUDA tensor fed to the policy")
        i = self._stage_rt_i
        if self._stage_rt_evt[i] is not None:
            self._stage_rt_evt[i].synchronize()
        host = self._stage_rt[i].numpy()
        host[0], host[1] = rews, terminals
        self._dev_scal[0:2].copy_(self._stage_rt[i], non_blocking=True)
        evt = torch.cuda.Event()
        evt.record()
        self._stage_rt_evt[i] = evt
        self._stage_rt_i ^= 1
        obs_d = obs.to(self.obs_dtype).reshape(N, -1).contiguous()
        _lib.call("xb_rollout_store", _lib.ptr(self._obs), _lib.ptr(obs_d), obs_d.shape[1] * obs_d.element_size(),
                  _lib.ptr(self._fields), _lib.ptr(self._dev_scal), self._n_store, N, T, t)
        if not self._scalar_action:
            self._store_rows(self._act_rows, self._dev_act, t)
        self.ptr = (self.ptr + 1) % self.n_size
        self.size = min(self.size + 1, self.n_size)

    # -------- K2
    def finish_path(self, val, i):
        """reference :242-265 - records that env ``i``'s current path ends at the last stored step with bootstrap
        value ``val``; the arithmetic for all recorded segments runs in one K2 launch (``_ensure_gae``)."""
        end = self.n_size if self.full else self.ptr
        start = int(self.start_ids[i])
        if end > start:
            if isinstance(val, torch.Tensor):
                val = float(val)
            self._seg_end_h[i, end - 1] = 1
            self._boot_h[i, end - 1] = float(np.float32(val))
            self._covered_h[i] = end
            self._gae_dirty = True
        self.start_ids[i] = self.ptr

    def finish_paths(self, vals, mask=None):
        """Batched form: ``finish_path(vals[i], i)`` for every env (or those with mask[i])."""
        vals = vals.detach().float().cpu().numpy() if isinstance(vals, torch.Tensor) else np.asarray(vals, np.float32)
        end = self.n_size if self.full else self.ptr
        sel = np.ones(self.n_envs, bool) if mask is None else np.asarray(mask, bool).copy()
        env = np.flatnonzero(sel & (self.start_ids < end))        # paths with at least one stored step
        if env.size:
            self._seg_end_h.numpy()[env, end - 1] = 1
            self._boot_h.numpy()[env, end - 1] = vals.reshape(-1)[env].astype(np.float32)
            self._covered_h.numpy()[env] = end
            self._gae_dirty = True
        self.start_ids[np.flatnonzero(sel)] = self.ptr

    def _ensure_gae(self):
        if not self._gae_dirty:
            return
        self._seg_end.copy_(self._seg_end_h, non_blocking=True)
        self._boot.copy_(self._boot_h, non_blocking=True)
        self._covered.copy_(self._covered_h, non_blocking=True)
        f = self._fid
        _lib.call("xb_gae_scan", _lib.ptr(self._fields[f["rewards"]]), _lib.ptr(self._fields[f["values"]]),
                  _lib.ptr(self._fields[f["terminals"]]), _lib.ptr(self._seg_end), _lib.ptr(self._boot),
                  _lib.ptr(self._covered), _lib.ptr(self._fields[f["advantages"]]),
                  _lib.ptr(self._fields[f["returns"]]), self.n_envs, self.n_size,
                  float(self.gamma), float(self.gae_lam), 1 if self.use_gae else 0)
        self._gae_dirty = False

    # -------- K3
    def global_adv_stats(self, perm_d, n_minibatch):
        """Sharded runs: (mean, population std) of the advantages of every GLOBAL minibatch of one epoch, float32
        [n_minibatch, 2] on the device, from ONE all-reduce per epoch (3 doubles per minibatch) instead of one per
        minibatch.  ``perm_d``: this rank's slot permutation of the epoch, minibatch m = its m-th equal slice."""
        import torch.distributed as dist
        self._ensure_gae()
        a = self.advantages.reshape(-1)[perm_d].reshape(n_minibatch, -1).double()
        mom = torch.stack([a.sum(1), (a * a).sum(1), torch.full((n_minibatch,), float(a.shape[1]), dtype=torch.float64,
                                                               device=self.device)])
        if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            dist.all_reduce(mom)
        mean = mom[0] / mom[2]
        std = (mom[1] / mom[2] - mean * mean).clamp_min(0).sqrt()
        return torch.stack([mean, std], dim=1).float().contiguous()

    def _gather_fields(self, idx_t, adv_stats=None):
        B = idx_t.numel()
        g0 = self._gather_first
        F = len(self._names) - g0
        out = torch.empty((F, B), dtype=torch.float32, device=self.device)
        adv_field = (self._fid["advantages"] - g0) if self.use_advnorm else -1
        import torch.distributed as dist
        sharded = adv_field >= 0 and dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1
        _lib.call("xb_gather_scalars", _lib.ptr(self._fields[g0]), self.n_envs * self.n_size, _lib.ptr(idx_t), B, F,
                  _lib.ptr(out), -1 if sharded else adv_field, _lib.ptr(self._stats), _lib.ptr(self._scratch))
        if sharded and adv_stats is not None:      # global statistics of this minibatch, all-reduced once per epoch
            _lib.call("xb_adv_normalize", _lib.ptr(out[adv_field]), B, _lib.ptr(adv_stats))
        elif sharded:
            # this rank holds B of the B*world rows of the global minibatch: normalise with the GLOBAL mean / population
            # std (memory_tools.py:281-282 applied to the whole minibatch) - one 3-double all-reduce
            a = out[adv_field].double()
            mom = torch.stack([a.sum(), (a * a).sum(), torch.full((), float(B), dtype=torch.float64, device=self.device)])
            dist.all_reduce(mom)
            mean = mom[0] / mom[2]
            std = (mom[1] / mom[2] - mean * mean).clamp_min(0).sqrt()
            out[adv_field] = ((a - mean) / (std + 1e-8)).float()
        return out

    def _assemble(self, obs, idx_t, fields):
        g0 = self._gather_first
        row = lambda name: fields[self._fid[name] - g0]
        return {
            "obs": obs,
            "actions": row("actions") if self._scalar_action else self._gather_rows(self._act_rows, idx_t),
            "returns": row("returns"),
            "values": row("values"),
            "aux_batch": {k: row("aux:" + k) for k in self._aux_keys},
            "batch_size": idx_t.numel(),
            "advantages": row("advantages"),
        }

    def sample(self, indexes, adv_stats=None):
        """reference :267-287.  ``indexes`` are flat slots (env*T+step, as np.arange(buffer_size) shuffled by
        the agent); returns CUDA tensors with the reference's keys, shapes and dtypes."""
        assert self.full, "Not enough transitions for on-policy buffer to random sample"
        self._ensure_gae()
        idx_t = self._index_tensor(indexes)
        obs = self._gather_rows(self._obs, idx_t)
        return self._assemble(obs, idx_t, self._gather_fields(idx_t, adv_stats))

    def sample_prepared(self, indexes, fmt, adv_stats=None):
        """Fast path used by train_epochs: the observation gather also converts u8 -> float in the layout the
        network wants (K3 fused), skipping the u8 intermediate.  Only for uint8 image buffers."""
        assert self.full, "Not enough transitions for on-policy buffer to random sample"
        if self.obs_dtype != torch.uint8 or len(self._obs_shape) != 3 or fmt == _lib.OBS_U8:
            return self.sample(indexes, adv_stats)
        self._ensure_gae()
        idx_t = self._index_tensor(indexes)
        H, W, C = self._obs_shape
        B = idx_t.numel()
        if fmt in (_lib.OBS_PLANES2, _lib.OBS_PLANES3, _lib.OBS_PLANE_RAW):   # K12 input: bf16 planes of u8/255, or the raw
            P = {_lib.OBS_PLANES2: 2, _lib.OBS_PLANES3: 3, _lib.OBS_PLANE_RAW: 1}[fmt]    # pixel value as one exact plane
            out = torch.empty((P, B, H, W, C), dtype=torch.bfloat16, device=self.device)
            _lib.call("xb_gather_obs_planes", _lib.ptr(self._obs), _lib.ptr(idx_t), B, H * W * C, P, _lib.ptr(out))
            return self._assemble(PreparedObs(out, fmt, (H, W, C)), idx_t, self._gather_fields(idx_t, adv_stats))
        dt = {_lib.OBS_F32_NHWC: torch.float32, _lib.OBS_F32_NCHW: torch.float32,
              _lib.OBS_BF16_NHWC: torch.bfloat16, _lib.OBS_F16_NHWC: torch.float16}[fmt]
        shape = (B, C, H, W) if fmt == _lib.OBS_F32_NCHW else (B, H, W, C)
        out = torch.empty(shape, dtype=dt, device=self.device)
        _lib.call("xb_gather_obs", _lib.ptr(self._obs), _lib.ptr(idx_t), B, H, W, C, _lib.ptr(out), fmt)
        return self._assemble(PreparedObs(out, fmt, (H, W, C)), idx_t, self._gather_fields(idx_t, adv_stats))


class DummyOnPolicyBuffer_Atari(DummyOnPolicyBuffer):
    """uint8 observation storage (reference memory_tools.py:290-328)."""
    obs_dtype = torch.uint8


# =====================================================================================================
# Off-policy replay (uniform) and prioritized replay
# =====================================================================================================
class DummyOffPolicyBuffer(Buffer):
    """Device-resident mirror of DummyOffPolicyBuffer (reference memory_tools.py:331-387)."""

    obs_dtype = torch.float32
    _ckpt_tensors = ("_obs", "_next_obs", "_act_rows", "_fields")

    def __init__(self, observation_space, action_space, auxiliary_shape, n_envs, buffer_size, batch_size,
                 device="cuda:0"):
        super().__init__(observation_space, action_space, auxiliary_shape, n_envs, buffer_size, device)
        self.batch_size = batch_size
        obs_shape = space2shape(self.observation_space)
        if isinstance(obs_shape, dict):
            raise NotImplementedError("dict observation spaces are outside the hot path")
        self._obs_shape = tuple(obs_shape)
        self._act_shape = tuple(space2shape(self.action_space))
        self._scalar_action = self._act_shape == ()
        self._names = ["rewards", "terminals"] + (["actions"] if self._scalar_action else [])
        self._fid = {n: i for i, n in enumerate(self._names)}
        self._allocate()
        N = self.n_envs
        self._stage_i = 0
        self._stage_scal = [torch.zeros((len(self._names), N), dtype=torch.float32).pin_memory() for _ in range(2)]
        self._stage_obs = [torch.zeros((2, N) + self._obs_shape, dtype=self.obs_dtype).pin_memory() for _ in range(2)]
        self._stage_evt = [None, None]

    def _allocate(self):
        self._obs = self._alloc_rows(self._obs_shape, self.obs_dtype)
        self._next_obs = self._alloc_rows(self._obs_shape, self.obs_dtype)
        self._act_rows = None if self._scalar_action else self._alloc_rows(self._act_shape, torch.float32)
        self._fields = torch.zeros((len(self._names), self.n_envs, self.n_size), dtype=torch.float32,
                                   device=self.device)

    observations = property(lambda self: self._obs)
    next_observations = property(lambda self: self._next_obs)
    rewards = property(lambda self: self._fields[self._fid["rewards"]])
    terminals = property(lambda self: self._fields[self._fid["terminals"]])
    actions = property(lambda self: self._fields[self._fid["actions"]] if self._scalar_action else self._act_rows)

    def clear(self):
        self.ptr, self.size = 0, 0

    def _stage(self, obs, next_obs, scal_in):
        N = self.n_envs
        dev_obs = isinstance(obs, torch.Tensor) and obs.is_cuda and isinstance(next_obs, torch.Tensor) and next_obs.is_cuda
        dev_scal = all(isinstance(x, torch.Tensor) and x.is_cuda for x in scal_in)
        i = self._stage_i
        if not (dev_obs and dev_scal) and self._stage_evt[i] is not None:
            self._stage_evt[i].synchronize()
        if dev_scal:
            scal = torch.stack([x.to(torch.float32).reshape(N) for x in scal_in])
        else:
            host = self._stage_scal[i].numpy()
            for f, x in enumerate(scal_in):
                host[f] = x.detach().cpu().numpy() if isinstance(x, torch.Tensor) else x
            scal = self._stage_scal[i].to(self.device, non_blocking=True)
        if dev_obs:
            o = obs.to(self.obs_dtype).reshape(N, -1).contiguous()
            o2 = next_obs.to(self.obs_dtype).reshape(N, -1).contiguous()
        else:
            host = self._stage_obs[i].numpy()
            host[0] = obs.cpu().numpy() if isinstance(obs, torch.Tensor) else obs
            host[1] = next_obs.cpu().numpy() if isinstance(next_obs, torch.Tensor) else next_obs
            both = self._stage_obs[i].to(self.device, non_blocking=True)
            o, o2 = both[0].reshape(N, -1), both[1].reshape(N, -1)
        if not (dev_obs and dev_scal):
            evt = torch.cuda.Event()
            evt.record()
            self._stage_evt[i] = evt
            self._stage_i ^= 1
        return o, o2, scal

    def store(self, obs, acts, rews, terminals, next_obs):
        """reference :364-372."""
        N, T, t = self.n_envs, self.n_size, self.ptr
        scal_in = [rews, terminals] + ([acts] if self._scalar_action else [])
        o, o2, scal = self._stage(obs, next_obs, scal_in)
        row_bytes = o.shape[1] * o.element_size()
        _lib.call("xb_rollout_store", _lib.ptr(self._obs), _lib.ptr(o), row_bytes, _lib.ptr(self._fields),
                  _lib.ptr(scal), len(self._names), N, T, t)
        _lib.call("xb_rollout_store", _lib.ptr(self._next_obs), _lib.ptr(o2), row_bytes, None, None, 0, N, T, t)
        if not self._scalar_action:
            self._store_rows(self._act_rows, acts, t)
        self.ptr = (self.ptr + 1) % self.n_size
        self.size = min(self.size + 1, self.n_size)

    def _gather(self, flat_idx):
        B = flat_idx.numel()
        F = len(self._names)
        out = torch.empty((F, B), dtype=torch.float32, device=self.device)
        _lib.call("xb_gather_scalars", _lib.ptr(self._fields), self.n_envs * self.n_size, _lib.ptr(flat_idx), B, F,
                  _lib.ptr(out), -1, None, None)
        return {
            "obs": self._gather_rows(self._obs, flat_idx),
            "actions": out[self._fid["actions"]] if self._scalar_action else self._gather_rows(self._act_rows, flat_idx),
            "obs_next": self._gather_rows(self._next_obs, flat_idx),
            "rewards": out[self._fid["rewards"]],
            "terminals": out[self._fid["terminals"]],
        }

    def sample(self, batch_size=None):
        """reference :374-387: env and step drawn independently (with replacement) from NumPy's global RNG, in
        the reference's order, so ``np.random.seed(s)`` reproduces the reference's choices."""
        bs = self.batch_size if batch_size is None else batch_size
        env_choices = np.random.choice(self.n_envs, bs)
        step_choices = np.random.choice(self.size, bs)
        flat = self._index_tensor(env_choices.astype(np.int64) * self.n_size + step_choices.astype(np.int64))
        d = self._gather(flat)
        d["batch_size"] = bs
        return d


class DummyOffPolicyBuffer_Atari(DummyOffPolicyBuffer):
    """uint8 image replay (reference memory_tools.py:601-630)."""
    obs_dtype = torch.uint8


class PerOffPolicyBuffer(DummyOffPolicyBuffer):
    """Prioritized replay (reference memory_tools.py:471-598) with the segment trees of
    xuance/common/segtree_tool.py held in HBM: ``_it_sum`` / ``_it_min`` are ``[n_envs, 2*capacity]`` float32
    heaps (one pair per env, as the reference), driven by the K5 kernels.  Image observations are stored as
    uint8 when the observation space's dtype is uint8 (reference stores float32: appendix B #9)."""

    _ckpt_tensors = DummyOffPolicyBuffer._ckpt_tensors + ("_it_sum", "_it_min", "_max_priority")

    def __init__(self, observation_space, action_space, auxiliary_shape, n_envs, buffer_size, batch_size,
                 alpha=0.6, device="cuda:0"):
        if getattr(observation_space, "dtype", None) is not None and np.dtype(observation_space.dtype) == np.uint8:
            self.obs_dtype = torch.uint8
        super().__init__(observation_space, action_space, auxiliary_shape, n_envs, buffer_size, batch_size, device)
        self._alpha = alpha
        cap = 1
        while cap < self.n_size:
            cap *= 2
        self._it_capacity = cap
        self._it_sum = torch.zeros((n_envs, 2 * cap), dtype=torch.float32, device=self.device)
        self._it_min = torch.full((n_envs, 2 * cap), float("inf"), dtype=torch.float32, device=self.device)
        self._max_priority = torch.ones(n_envs, dtype=torch.float32, device=self.device)
        k = int(self.batch_size / self.n_envs)
        self._k = k
        self._u_host = [torch.zeros((n_envs, k), dtype=torch.float32).pin_memory() for _ in range(2)]
        self._u_evt = [None, None]
        self._u_i = 0

    def clear(self):
        super().clear()
        self._it_sum.zero_()
        self._it_min.fill_(float("inf"))

    def store(self, obs, acts, rews, terminals, next_obs):
        """reference :537-550: data store + leaf[ptr] = max_priority**alpha in both trees of every env."""
        t = self.ptr
        super().store(obs, acts, rews, terminals, next_obs)
        _lib.call("xb_per_insert", _lib.ptr(self._it_sum), _lib.ptr(self._it_min), _lib.ptr(self._max_priority),
                  self.n_envs, self._it_capacity, t, float(self._alpha))

    def sample(self, beta, uniforms=None):
        """reference :552-586.  ``uniforms`` ([n_envs, B/n_envs] in [0,1)) may be supplied; by default they are
        drawn with ``random.random()`` in the reference's order so ``random.seed(s)`` reproduces its batches."""
        assert beta > 0
        N, k = self.n_envs, self._k
        if self.size < 2:
            raise RuntimeError("PerOffPolicyBuffer.sample needs at least 2 stored steps (the reference's "
                               "sum(0, size-1) is undefined before that)")
        i = self._u_i
        if self._u_evt[i] is not None:
            self._u_evt[i].synchronize()
        host = self._u_host[i].numpy()
        if uniforms is None:             # N*k draws of random.random() in the reference's (env-major) order
            _rnd = random.random
            host.reshape(-1)[:] = [_rnd() for _ in range(N * k)]
        else:
            host[...] = np.asarray(uniforms, dtype=np.float64).reshape(N, k)
        u = self._u_host[i].to(self.device, non_blocking=True)
        evt = torch.cuda.Event()
        evt.record()
        self._u_evt[i] = evt
        self._u_i ^= 1
        step_choices = torch.empty((N, k), dtype=torch.int64, device=self.device)
        flat = torch.empty((N * k,), dtype=torch.int64, device=self.device)
        weights = torch.empty((N, k), dtype=torch.float64, device=self.device)
        spb = float(np.float32(self.size ** (-beta)))
        _lib.call("xb_per_sample", _lib.ptr(self._it_sum), _lib.ptr(self._it_min), _lib.ptr(u), N,
                  self._it_capacity, self.size, k, self.n_size, spb, _lib.ptr(step_choices), _lib.ptr(flat),
                  _lib.ptr(weights))
        d = self._gather(flat)
        d.update(weights=weights, step_choices=step_choices, batch_size=self.batch_size)
        return d

    def update_priorities(self, idxes, priorities):
        """reference :588-598.  ``idxes`` = the step_choices of the last sample, ``priorities`` = |td| [B]."""
        idx_t = idxes if isinstance(idxes, torch.Tensor) else _as_device(np.asarray(idxes, np.int64), self.device)
        idx_t = idx_t.to(device=self.device, dtype=torch.int64).contiguous()
        pr = priorities if isinstance(priorities, torch.Tensor) else _as_device(np.asarray(priorities, np.float32), self.device)
        pr = pr.to(device=self.device, dtype=torch.float32).contiguous()
        _lib.call("xb_per_update", _lib.ptr(self._it_sum), _lib.ptr(self._it_min), _lib.ptr(self._max_priority),
                  _lib.ptr(idx_t), _lib.ptr(pr), self.n_envs, self._it_capacity, self._k, float(self._alpha))
