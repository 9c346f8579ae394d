"""ctypes binding of the C ABI declared in include/hpc_rll_b200.h.

The CUDA library is the product: if it cannot be loaded this module raises -- nothing here falls
back to PyTorch ops, the CPU or the oracle.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "_lib", "libhpc_rll_b200.so")

c_f32p = ctypes.c_void_p
c_i64 = ctypes.c_int64
c_dbl = ctypes.c_double
c_int = ctypes.c_int
c_vp = ctypes.c_void_p
c_sz = ctypes.c_size_t

# name -> (restype, argtypes); mirrors include/hpc_rll_b200.h one to one
SIGNATURES = {
    "hpc_rll_version": (ctypes.c_char_p, []),
    "hpc_rll_last_error": (ctypes.c_char_p, []),
    "hpc_rll_launch_count": (ctypes.c_uint64, []),
    "hpc_rll_workspace_bytes": (c_sz, [c_int, c_i64, c_i64, c_i64]),
    "hpc_rll_debug_set_config": (c_int, [c_int, c_int]),
    "hpc_rll_axpby": (c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp]),
    "hpc_rll_gae_forward": (c_int, [c_vp, c_vp, c_vp, c_i64, c_i64, c_dbl, c_dbl, c_vp]),
    "hpc_rll_gae_backward": (c_int, [c_vp, c_vp, c_vp, c_i64, c_i64, c_dbl, c_dbl, c_vp]),
    "hpc_rll_gae_forward_moments": (c_int, [c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_dbl, c_dbl, c_vp, c_sz, c_vp]),
    "hpc_rll_adv_stats": (c_int, [c_vp, c_i64, c_vp, c_vp]),
    "hpc_rll_gae_forward_ld": (c_int, [c_vp, c_i64, c_vp, c_i64, c_vp, c_i64, c_i64, c_i64, c_dbl, c_dbl, c_vp]),
    "hpc_rll_gae_backward_ld": (c_int, [c_vp, c_i64, c_vp, c_i64, c_vp, c_i64, c_i64, c_i64, c_dbl, c_dbl, c_vp]),
    "hpc_rll_gae_fwd_bwd_host": (c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_dbl, c_dbl]),
    "hpc_rll_gae_forward_chunk": (c_int, [c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_i64, c_i64, c_dbl, c_dbl, c_vp]),
    "hpc_rll_gae_backward_chunk": (c_int, [c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_i64, c_i64, c_dbl, c_dbl, c_vp]),
    "hpc_rll_debug_host_schedule": (c_i64, [c_i64, c_i64, c_vp, c_i64]),
    "hpc_rll_device_numa_node": (c_int, [c_int]),
    "hpc_rll_bind_thread_to_device": (c_int, [c_int]),
    "hpc_rll_host_alloc": (c_vp, [c_sz, c_int]),
    "hpc_rll_host_free": (c_int, [c_vp]),
    "hpc_rll_td_lambda_forward": (c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_dbl, c_dbl, c_i64, c_vp,
                                          c_sz, c_vp]),
    "hpc_rll_td_lambda_backward": (c_int, [c_vp, c_vp, c_vp, c_i64, c_i64, c_vp]),
    "hpc_rll_vtrace_forward": (c_int, [c_vp] * 9 + [c_i64] * 3 + [c_dbl] * 5 + [c_i64, c_vp, c_sz, c_vp]),
    "hpc_rll_vtrace_backward": (c_int, [c_vp] * 10 + [c_i64] * 4 + [c_vp]),
    "hpc_rll_upgo_forward": (c_int, [c_vp] * 7 + [c_i64] * 4 + [c_vp, c_sz, c_vp]),
    "hpc_rll_upgo_backward": (c_int, [c_vp] * 5 + [c_i64] * 3 + [c_vp]),
    "hpc_rll_ppo_forward": (c_int, [c_vp] * 11 + [c_i64, c_i64, c_dbl, c_int, c_dbl, c_i64, c_vp, c_sz, c_vp]),
    "hpc_rll_ppo_forward_norm": (c_int, [c_vp] * 12 + [c_i64, c_i64, c_dbl, c_int, c_dbl, c_i64, c_vp, c_sz, c_vp]),
    "hpc_rll_ppo_backward": (c_int, [c_vp] * 10 + [c_i64] * 3 + [c_vp]),
    "hpc_rll_q_nstep_td_forward": (c_int, [c_vp] * 10 + [c_i64] * 3 + [c_dbl, c_int, c_i64, c_vp, c_sz, c_vp]),
    "hpc_rll_q_nstep_td_backward": (c_int, [c_vp] * 4 + [c_i64] * 2 + [c_vp]),
    "hpc_rll_dist_nstep_td_forward": (c_int, [c_vp] * 10 + [c_i64] * 4 + [c_dbl] * 3 + [c_i64, c_vp, c_sz, c_vp]),
    "hpc_rll_dist_nstep_td_backward": (c_int, [c_vp] * 4 + [c_i64] * 3 + [c_vp]),
    "hpc_rll_qrdqn_nstep_td_forward": (c_int, [c_vp] * 11 + [c_i64] * 4 + [c_dbl, c_i64, c_vp, c_sz, c_vp]),
    "hpc_rll_qrdqn_nstep_td_backward": (c_int, [c_vp] * 4 + [c_i64] * 3 + [c_vp]),
    "hpc_rll_iqn_nstep_td_forward": (c_int, [c_vp] * 12 + [c_i64] * 5 + [c_dbl, c_dbl, c_i64, c_vp, c_sz, c_vp]),
    "hpc_rll_iqn_nstep_td_backward": (c_int, [c_vp] * 4 + [c_i64] * 3 + [c_vp]),
    "hpc_rll_p2p_buffer_bytes": (c_sz, []),
    "hpc_rll_p2p_alloc": (c_int, [c_vp, c_vp]),
    "hpc_rll_p2p_open": (c_int, [c_vp, c_vp]),
    "hpc_rll_p2p_close": (c_int, [c_vp]),
    "hpc_rll_p2p_free": (c_int, [c_vp]),
    "hpc_rll_allreduce_scalars_p2p": (c_int, [c_vp, c_int, c_vp, c_int, c_int, c_vp]),
    "hpc_rll_pad_batch": (c_int, [c_vp] * 5 + [c_i64, c_int, c_vp]),
    "hpc_rll_unpad_batch": (c_int, [c_vp] * 4 + [c_i64, c_vp]),
    "hpc_rll_oracle_split_group": (c_int, [c_vp, c_i64, c_int, c_int, c_vp]),
    "hpc_rll_sample_split_group": (c_int, [c_vp, c_i64, c_int, c_int, ctypes.c_uint64, c_vp, c_vp]),
    "hpc_rll_scatter_connection_forward": (c_int, [c_vp] * 3 + [c_i64] * 5 + [c_int, c_vp]),
    "hpc_rll_scatter_connection_backward": (c_int, [c_vp] * 3 + [c_i64] * 5 + [c_vp]),
}

OP_GAE, OP_TD_LAMBDA, OP_VTRACE, OP_UPGO, OP_PPO, OP_Q_NSTEP_TD, OP_DIST_NSTEP_TD, OP_QRDQN_NSTEP_TD, \
    OP_IQN_NSTEP_TD, OP_GAE_MOMENTS, OP_SCATTER_CONNECTION = range(11)

_lib = None


class HpcRllError(RuntimeError):
    pass


def lib():
    """Load (once) and return the CDLL with typed entry points."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise HpcRllError(
                "libhpc_rll_b200.so not found at %s -- build it with `python -m di_hpc_b200.build` "
                "(or __graft_entry__.build()).  There is no fallback path." % LIB_PATH)
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)  # AttributeError if the library does not export a declared symbol
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = lib().hpc_rll_last_error()
        raise HpcRllError("%s failed (code %d): %s" % (what, rc, msg.decode() if msg else "?"))


def ptr(t):
    """Device/host pointer of a tensor as an int (None -> NULL)."""
    return None if t is None else t.data_ptr()


def stream_of(t) -> int:
    """The current CUDA stream of the tensor's device as a raw cudaStream_t."""
    return torch.cuda.current_stream(t.device).cuda_stream


class _NoGuard:
    def __enter__(self):
        return self

    def __exit__(self, *exc):
        return False


_NOGUARD = _NoGuard()


def on_device(device):
    """Device guard for the C-ABI calls (they act on the CURRENT device).  Free when the tensor already
    lives on the current device -- the common one-process-per-GPU case."""
    if device.index is None or device.index == torch.cuda.current_device():
        return _NOGUARD
    return torch.cuda.device(device)


def require_f32_cuda(name: str, t: torch.Tensor) -> torch.Tensor:
    """The reference assumes fp32 contiguous CUDA tensors (hpc_rll/rl_utils/gae.py:58-59 asserts
    is_cuda only); we check dtype and make the layout contiguous."""
    assert t.is_cuda, "%s must be a CUDA tensor (hpc version only supports cuda)" % name
    if t.dtype != torch.float32:
        raise TypeError("%s must be float32, got %s" % (name, t.dtype))
    return t.contiguous()


def require_i64_cuda(name: str, t: torch.Tensor) -> torch.Tensor:
    assert t.is_cuda, "%s must be a CUDA tensor (hpc version only supports cuda)" % name
    if t.dtype != torch.int64:
        raise TypeError("%s must be int64, got %s" % (name, t.dtype))
    return t.contiguous()


def workspace(op: int, T: int, B: int, N: int, device) -> torch.Tensor:
    """Allocate the scratch buffer an op asks for (torch caching allocator; stream-ordered reuse)."""
    with on_device(torch.device(device)):  # the size depends on the SM count of the tensor's device
        n = int(lib().hpc_rll_workspace_bytes(op, T, B, N))
    return torch.empty(max(n, 8), dtype=torch.uint8, device=device)


def grad_scalar(g: torch.Tensor, like: torch.Tensor) -> torch.Tensor:
    """Upstream gradient of a scalar loss as a 1-element fp32 device tensor (never read on the host)."""
    if g is None:
        return torch.zeros(1, dtype=torch.float32, device=like.device)
    return g.reshape(1).to(dtype=torch.float32, device=like.device).contiguous()


def launch_count() -> int:
    return int(lib().hpc_rll_launch_count())


def set_config(op: int, cfg: int) -> None:
    check(lib().hpc_rll_debug_set_config(op, cfg), "hpc_rll_debug_set_config")
