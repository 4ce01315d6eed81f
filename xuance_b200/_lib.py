"""ctypes binding of libxb200.so (the C-ABI declared in include/xb200.h).

There is NO CPU or PyTorch fallback: if the library cannot be loaded, or a call returns a non-zero status,
this module raises.  Tensors are passed as raw device pointers (``tensor.data_ptr()``) plus sizes; the stream
is torch's current CUDA stream so launches interleave correctly with cuDNN/cuBLAS work issued by torch."""
import ctypes
import os
from ctypes import c_int, c_int64, c_float, c_double, c_void_p, c_char_p, POINTER

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libxb200.so")

OBS_U8, OBS_F32_NHWC, OBS_F32_NCHW, OBS_BF16_NHWC, OBS_F16_NHWC = 0, 1, 2, 3, 4
OBS_PLANES2, OBS_PLANES3, OBS_PLANE_RAW = 5, 6, 7   # bf16 plane tensors [P, B, H, W, C] for the K12 layers (xb_gather_obs_planes);
#                                                     RAW: one plane holding the uint8 value itself (exact in bf16)

_P = c_void_p
_SIGNATURES = {
    "xb_version": (c_int, []),
    "xb_error_string": (c_char_p, [c_int]),
    "xb_device_info": (c_int, [POINTER(c_int), POINTER(c_int), POINTER(c_int)]),
    "xb_rollout_store": (c_int, [_P, _P, c_int64, _P, _P, c_int, c_int, c_int, c_int, _P]),
    "xb_gae_scan": (c_int, [_P, _P, _P, _P, _P, _P, _P, _P, c_int, c_int, c_float, c_float, c_int, _P]),
    "xb_gather_rows": (c_int, [_P, _P, c_int64, c_int64, _P, _P]),
    "xb_gather_obs": (c_int, [_P, _P, c_int64, c_int, c_int, c_int, _P, c_int, _P]),
    "xb_scratch_doubles": (c_int64, []),
    "xb_gather_scalars": (c_int, [_P, c_int64, _P, c_int64, c_int, _P, c_int, _P, _P, _P]),
    "xb_adv_normalize": (c_int, [_P, c_int64, _P, _P]),
    "xb_ppo_loss_fwd_bwd": (c_int, [_P, _P, _P, _P, _P, _P, c_int64, c_int, c_int64, c_float, c_float, c_float,
                                    c_int, _P, _P, _P, _P, _P]),
    "xb_gaussian_scratch_doubles": (c_int64, [c_int]),
    "xb_ppo_gaussian_loss_fwd_bwd": (c_int, [_P, _P, _P, _P, _P, _P, _P, c_int64, c_int, c_int64, c_float, c_float,
                                             c_float, c_int, _P, _P, _P, _P, _P, _P, _P]),
    "xb_per_insert": (c_int, [_P, _P, _P, c_int, c_int, c_int, c_float, _P]),
    "xb_per_sample": (c_int, [_P, _P, _P, c_int, c_int, c_int, c_int, c_int64, c_float, _P, _P, _P, _P]),
    "xb_per_update": (c_int, [_P, _P, _P, _P, _P, c_int, c_int, c_int, c_float, _P]),
    "xb_dqn_td_fwd_bwd": (c_int, [_P, _P, _P, _P, _P, _P, c_int64, c_int, c_int64, c_float, _P, _P, _P, _P, _P]),
    "xb_grad_sumsq": (c_int, [_P, c_int64, c_float, _P, _P, _P]),
    "xb_adam_step": (c_int, [_P, _P, _P, _P, c_int64, _P, c_float, c_float, c_float, c_float, _P, c_float,
                             c_int, _P]),
    "xb_soft_update": (c_int, [_P, _P, c_int64, c_float, _P]),
    "xb_split_bf16": (c_int, [_P, c_int64, c_int, _P, _P]),
    "xb_gather_obs_planes": (c_int, [_P, _P, c_int64, c_int64, c_int, _P, _P]),
    "xb_pack_conv_weight": (c_int, [_P, c_int, c_int, c_int, c_int, c_int, c_float, _P, _P]),
    "xb_pack_weights": (c_int, [_P, c_int, _P]),
    "xb_gemm_gather_tc": (c_int, [c_int, c_int, _P, c_int64, _P, c_int64, _P, _P, c_int64, c_int] + [c_int] * 9
                          + [_P, _P, c_int, c_int, c_int, _P, c_int64, c_int, _P] + [c_int] * 6 + [c_int64, c_int, _P, _P]),
    "xb_gemm_box_tc": (c_int, [c_int, c_int, _P, c_int64, c_int, c_int, c_int64, c_int, c_int, c_int, c_int, c_int, _P, _P, _P,
                               _P, c_int64, _P, _P] + [c_int] * 9 + [_P, c_int64, c_int, _P]
                       + [c_int] * 6 + [c_int64, c_int, _P, _P]),
    "xb_gemm_halo_tc": (c_int, [c_int, c_int, _P, c_int64, c_int, c_int64, c_int, c_int, c_int, c_int, _P, _P, _P, c_int64, _P, _P,
                                c_int, c_int, c_int, c_int, c_int, _P, _P, c_int, c_int, _P, c_int64, c_int, _P, c_int, c_int,
                                c_int, c_int, _P, _P, c_int64, c_int, c_int, _P, _P]),
    "xb_debug_k12_timing": (c_int, [_P, c_int]),
    "xb_debug_tma_box": (c_int, [_P, c_int64] + [c_int] * 12 + [ctypes.c_uint32, _P, ctypes.c_uint32, _P]),
    "xb_wgrad_box_tc": (c_int, [c_int, c_int, _P, c_int64, c_int, c_int, c_int64, c_int, c_int, c_int, c_int, c_int, _P, _P, _P,
                                _P, c_int64, c_int64, c_int, c_int, _P, _P]),
    "xb_wgrad_gather_tc": (c_int, [c_int, c_int, _P, c_int64, _P, c_int64, c_int64] + [c_int] * 9 + [_P, _P, c_int, c_int, c_int,
                                   _P, _P]),
    "xb_wgrad_reduce": (c_int, [_P, c_int, c_int, c_int, c_int, c_int, c_float, _P, c_int, _P]),
    "xb_categorical_act": (c_int, [_P, _P, _P, c_int, c_int, _P, _P, _P, _P, _P]),
    "xb_gaussian_act": (c_int, [_P, _P, _P, _P, c_int, c_int, _P, _P, _P, _P]),
    "xb_rms_update_normalize": (c_int, [_P, c_int, c_int64, _P, _P, c_double, c_int, _P, c_float, c_float, _P]),
    "xb_sac_actor_loss": (c_int, [_P, _P, _P, _P, c_int64, c_int64, _P, _P, _P, _P, _P, _P]),
    "xb_sac_critic_loss": (c_int, [_P, _P, _P, _P, _P, _P, _P, c_float, c_int64, c_int64, _P, _P, _P, _P, _P, _P]),
    "xb_qmix_select_fwd": (c_int, [_P, _P, _P, _P, _P, _P, c_int, c_int, c_int, c_int, c_int, c_int, _P, _P, _P, _P, _P]),
    "xb_qmix_select_bwd": (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, c_int, _P, _P]),
    "xb_qmix_mix_fwd": (c_int, [_P, _P, _P, _P, _P, c_int64, c_int, c_int, _P, _P]),
    "xb_qmix_mix_bwd": (c_int, [_P, _P, _P, _P, _P, c_int64, c_int, c_int, _P, _P, _P, _P, _P]),
    "xb_qmix_td": (c_int, [_P, _P, _P, _P, _P, _P, c_int, c_int, c_int, c_float, c_float, _P, _P, _P, _P]),
    "xb_qmix_mix_fused_fwd": (c_int, [_P] * 10 + [c_int64, c_int, c_int, c_int, c_int, _P, _P]),
    "xb_powf_libm": (c_int, [_P, c_float, _P, c_int64, _P]),
}
_OPTIONAL = {}

_lib = None
launch_count = 0  # number of xb200 kernel-launching ABI calls issued (bench.py's gpu_launches evidence)


def exported_symbols():
    """Names include/xb200.h declares; tests check that each one resolves in the loaded library."""
    return [k for k, v in _SIGNATURES.items() if v is not None]


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "xuance_b200: %s is missing - build it with `python -m xuance_b200.build` (nvcc, sm_100a). "
            "There is no CPU fallback." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, sig in list(_SIGNATURES.items()) + list(_OPTIONAL.items()):
        if sig is None:
            continue
        try:
            fn = getattr(lib, name)
        except AttributeError:
            if name in _OPTIONAL:
                continue
            raise RuntimeError("xuance_b200: %s does not export %s" % (LIB_PATH, name))
        fn.restype, fn.argtypes = sig
    _lib = lib
    return lib


def error_string(code):
    return load().xb_error_string(int(code)).decode()


def check(code, what=""):
    if code != 0:
        raise RuntimeError("xb200 %s failed: %s (code %d)" % (what, error_string(code), code))


def ptr(t):
    """Device pointer of a tensor (None -> NULL).  Refuses CPU tensors: the ABI takes device memory only."""
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("xb200: expected a CUDA tensor, got a %s tensor (no CPU fallback)" % t.device)
    return t.data_ptr()


def use_device(device):
    """Make ``device`` the process's current CUDA device: ``call`` launches on the CURRENT device's current stream, so every
    owner of device memory (agents, buffers, learners) selects its device once at construction (one process drives one GPU)."""
    device = torch.device(device)
    if device.type == "cuda" and torch.cuda.is_available():
        torch.cuda.set_device(device if device.index is not None else torch.device("cuda", torch.cuda.current_device()))
    return device


def stream():
    return torch.cuda.current_stream().cuda_stream


_KERNELS_PER_CALL = {"xb_gather_scalars": 2}   # calls that launch more than one kernel (second one: normalise)
class XbPackJob(ctypes.Structure):
    """include/xb200.h ``XbPackJob`` (one operand form of one weight for ``xb_pack_weights``)."""
    _fields_ = [("w", ctypes.c_void_p), ("out", ctypes.c_void_p), ("N", c_int), ("C", c_int), ("KH", c_int), ("KW", c_int),
                ("mode", c_int), ("n_taps", c_int), ("kh", ctypes.c_int8 * 16), ("kw", ctypes.c_int8 * 16),
                ("scale", c_float), ("planes", c_int)]


PACK_FORWARD, PACK_TRANSPOSED, PACK_DGRAD = 0, 1, 2

profile = None   # optional {abi_name: [(start_event, end_event), ...]} filled when set (bench.py roofline timing)
nvtx = os.environ.get("XB_NVTX", "0") == "1"   # NVTX range per ABI call (nsys / ncu --nvtx timelines); off by default


def call(name, *args):
    """Invoke an ABI entry point, appending the current stream, and raise on a non-zero status."""
    global launch_count
    fn = getattr(load(), name)
    launch_count += _KERNELS_PER_CALL.get(name, 1)
    if nvtx:
        torch.cuda.nvtx.range_push(name)
        try:
            check(fn(*args, stream()), name)
        finally:
            torch.cuda.nvtx.range_pop()
        return
    if profile is not None and name in profile:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        check(fn(*args, stream()), name)
        e1.record()
        profile[name].append((e0, e1))
        return
    check(fn(*args, stream()), name)


def scratch(device):
    """Zeroed reduction scratch (doubles + ticket) for the deterministic grid reductions."""
    n = load().xb_scratch_doubles()
    return torch.zeros(n, dtype=torch.float64, device=device)
