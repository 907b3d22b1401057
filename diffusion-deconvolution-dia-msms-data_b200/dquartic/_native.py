"""ctypes binding of the C-ABI in include/dquartic_b200.h (lib/libdquartic_b200.so, sm_100a).

There is no CPU fallback: if the library is missing, or a tensor is not a contiguous CUDA tensor of the expected
dtype, the call raises.  `launches` counts kernels launched through this module (bench.py reports it).
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
# DQ_B200_LIB: load another build of the same library (kernel A/B experiments, tools/)
LIB_PATH = os.environ.get("DQ_B200_LIB") or os.path.join(os.path.dirname(_HERE), "lib", "libdquartic_b200.so")

# signature mini-language: p = device pointer (torch tensor / None / int), i = int, l = long, f = float,
# s = stream (filled in automatically), h = host int array (sequence of python ints)
_SIGS = {
    "dq_qsample": ("pppppilis", 1),
    "dq_mix_affine": ("ppffffpls", 1),
    "dq_add_mul": ("pffpls", 1),
    "dq_ddim_step": ("pppffffils", 1),
    "dq_ddim_step_x0": ("ppppffffils", 1),
    "dq_dpm_step": ("pppppffiffffils", 1),
    "dq_scale_by": ("pppls", 1),
    "dq_cosine_sums": ("ppplis", 1),
    "dq_map_scores": ("ppppiiis", 2),
    "dq_sample_finalize": ("ppppls", 1),
    "dq_mse": ("ppppfls", 1),
    "dq_add_inplace": ("ppls", 1),
    "dq_conv1d_fwd": ("pipipippiiiiippiipppiiiis", 1),
    "dq_block_bwd": ("ppppiipppiiiis", 1),
    "dq_conv1d_bwd_data": ("pppiipiiiiiiiiiis", 1),
    "dq_conv1d_bwd_weight": ("ppipipippiiiiiiiiis", 1),
    "dq_conv_bwd_fused": ("ppppiipipipppipippppiiiiis", 1),
    "dq_conv_bwd_fused_res": ("pppp" + "ii" + "pipi" + "ppp" + "pppp" + "pppp" + "iiii" + "s", 1),
    "dq_initconv_bwd": ("pppp" + "i" + "ppppp" + "iiii" + "s", 2),
    "dq_resblock_fwd": ("pipippppipppppppppiiiis", 1),
    "dq_sample_dot": ("ppppilis", 1),
    "dq_upconv_bwd_fused": ("ppppippiiiiis", 1),
    "dq_downconv_bwd_fused": ("ppppippiiiiis", 1),
    "dq_upsample2x": ("ppls", 1),
    "dq_fold2x": ("pplis", 1),
    "dq_s2d": ("ppiiis", 1),
    "dq_d2s": ("ppiiiis", 1),
    "dq_down_w": ("ppiiis", 1),
    "dq_linattn_fwd": ("pppppppppppiiis", 3),
    "dq_linattn_bwd": ("pppppppppppppppppppiiis", 3),
    "dq_time_embed": ("ppiifs", 1),
    "dq_linear_fwd": ("ppppiiis", 1),
    "dq_linear_bwd": ("ppppppiiis", 2),
    "dq_act_fwd": ("ppils", 1),
    "dq_act_bwd": ("pppils", 1),
    "dq_ncl_nlc": ("ppiiiis", 1),
    "dq_gemm_bf16_tn": ("plllplllliplpiiiiihiiilis", 1),
    "dq_mid_pack": ("ppiiiis", 1),
    "dq_transpose_bf16": ("ppiilis", 1),
    "dq_cast_transpose": ("pppiis", 1),
    "dq_rownorm_fwd": ("pippiipppipiiis", 1),
    "dq_rownorm_bwd": ("pipippiipppipipppiiis", 2),
    "dq_colsum": ("ppiis", 1),
    "dq_attn_core_fwd": ("ppppppiis", 1),
    "dq_attn_core_bwd": ("ppppppppiis", 1),
    "dq_sumsq": ("plps", 1),
    "dq_clip_coef": ("pffps", 1),
    "dq_adamw": ("pppplpfffffffs", 1),
    "dq_adamw_ema": ("ppppplpffffffffs", 1),
    "dq_swap": ("ppls", 1),
    "dq_fill": ("pfls", 1),
    "dq_multiplex": ("ppippffpppppilis", 3),
}
_CT = {"p": ctypes.c_void_p, "i": ctypes.c_int, "l": ctypes.c_long, "f": ctypes.c_float, "s": ctypes.c_void_p,
       "h": ctypes.POINTER(ctypes.c_int)}

_lib = None
launches = 0
calls = 0


class NativeError(RuntimeError):
    pass


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise NativeError(
                f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a).  There is no CPU fallback for the dquartic hot path.")
        _lib = ctypes.CDLL(LIB_PATH)
        for name, (sig, _) in _SIGS.items():
            fn = getattr(_lib, name)
            fn.restype = ctypes.c_int
            fn.argtypes = [_CT[c] for c in sig]
        _lib.dq_la_nchunk.restype = ctypes.c_int
        _lib.dq_la_nchunk.argtypes = [ctypes.c_int]
        _lib.dq_map_scores_nblk.restype = ctypes.c_int
        _lib.dq_map_scores_nblk.argtypes = [ctypes.c_int]
        _lib.dq_gemm_last_error.restype = ctypes.c_int
        _lib.dq_gemm_last_error.argtypes = []
        _lib.dq_la_tc_last_error.restype = ctypes.c_int
        _lib.dq_la_tc_last_error.argtypes = [ctypes.POINTER(ctypes.c_uint)]
    return _lib


def exported_symbols():
    return sorted(list(_SIGS) + ["dq_la_nchunk", "dq_map_scores_nblk", "dq_gemm_last_error", "dq_la_tc_last_error"])


def _ptr(x):
    if x is None:
        return None
    if isinstance(x, int):
        return x
    if not x.is_cuda:
        raise NativeError("dquartic_b200 kernels need CUDA tensors (no CPU fallback)")
    if not x.is_contiguous():
        raise NativeError("non-contiguous tensor passed to a dquartic_b200 kernel")
    return x.data_ptr()


_OK_DTYPES = (torch.float32, torch.bfloat16, torch.int32, torch.int64)
_F64_ARGS = {"dq_sumsq", "dq_clip_coef", "dq_mse", "dq_map_scores"}   # the only entry points with a double* (accumulators)


def call(name, *args, allow=()):
    """Launch `name` on the current CUDA stream OF THE DEVICE THE TENSORS LIVE ON.  Raises on a non-zero return code
    (codes listed in `allow` are returned to the caller instead: "shape not covered by this kernel"), on tensors that
    are spread over several devices, and on dtypes no kernel of the library takes (fp16, int8, ...; the per-argument
    element type is the one include/dquartic_b200.h declares - callers pass fp32 unless the header says otherwise)."""
    global launches, calls
    sig, nk = _SIGS[name]
    fn = getattr(lib(), name)
    if len(args) != len(sig) - 1:
        raise TypeError(f"{name}: expected {len(sig) - 1} arguments, got {len(args)}")
    conv = []
    keep = []
    dev = None
    for c, a in zip(sig, args):
        if c == "p":
            if isinstance(a, torch.Tensor):
                if a.dtype not in _OK_DTYPES and not (a.dtype == torch.float64 and name in _F64_ARGS):
                    raise NativeError(f"{name}: unsupported tensor dtype {a.dtype}")
                if a.is_cuda:
                    if dev is None:
                        dev = a.device
                    elif a.device != dev:
                        raise NativeError(f"{name}: tensors on different devices ({dev} and {a.device})")
            conv.append(_ptr(a))
        elif c == "h":
            arr = (ctypes.c_int * len(a))(*[int(v) for v in a])
            keep.append(arr)
            conv.append(arr)
        elif c == "f":
            conv.append(float(a))
        else:
            conv.append(int(a))
    if dev is not None and dev.index != torch.cuda.current_device():
        with torch.cuda.device(dev):   # kernels, their static per-device state and the stream all belong to `dev`
            conv.append(torch.cuda.current_stream(dev).cuda_stream)
            rc = fn(*conv)
    else:
        conv.append(torch.cuda.current_stream().cuda_stream)
        rc = fn(*conv)
    if rc != 0 and rc in allow:
        return rc
    if rc != 0:
        raise NativeError(f"{name} failed with code {rc}" + (f" ({_cuda_err(rc)})" if rc > 0 else ""))
    launches += nk
    calls += 1
    return rc


def _cuda_err(rc):
    try:
        from torch.cuda import cudart
        return str(cudart().cudaGetErrorString(rc))
    except Exception:
        return "cuda error"


def la_nchunk(L):
    return int(lib().dq_la_nchunk(int(L)))


def map_scores_nblk(mz):
    """Column blocks of dq_map_scores per window: its scratch holds n_windows * map_scores_nblk(mz) * 9 doubles."""
    return int(lib().dq_map_scores_nblk(int(mz)))


def la_tc_last_error():
    """None when the tcgen05 LinearAttention pipelines ran clean since the last call, else the timeout record
    (wait code, blockIdx.x, blockIdx.y, threadIdx.x, barrier address, parity).  Synchronises with the device."""
    out = (ctypes.c_uint * 6)()
    rc = int(lib().dq_la_tc_last_error(out))
    if rc == 0:
        return None
    return (rc,) + tuple(int(v) for v in out)


def gemm_last_error():
    return int(lib().dq_gemm_last_error())
