"""ctypes binding of libso3d.so (C ABI declared in include/so3d.h).

There is no CPU fallback: if the library is missing, or a tensor is not a CUDA float32 tensor, the
call raises.  Build with ``python -m diffusion_extensions_b200.build`` (or ``__graft_entry__.build()``).
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
# SO3D_LIB_PATH: tuning aid, loads an alternative build of the same library (tests/tools/build_variant.py)
LIB_PATH = os.environ.get("SO3D_LIB_PATH") or os.path.join(_HERE, "libso3d.so")

_c_f = ctypes.c_void_p  # device pointers are passed as raw addresses
_i64 = ctypes.c_int64
_u64 = ctypes.c_uint64
_int = ctypes.c_int

# name -> argtypes (restype is always int); mirrors include/so3d.h one to one
SIGNATURES = {
    "so3d_log_f32": [_c_f, _c_f, _i64, _c_f],
    "so3d_logvec_f32": [_c_f, _c_f, _i64, _c_f],
    "so3d_rmat_to_aa_f32": [_c_f, _c_f, _c_f, _i64, _c_f],
    "so3d_aa_to_rmat_f32": [_c_f, _c_f, _c_f, _i64, _c_f],
    "so3d_expvec_f32": [_c_f, _c_f, _i64, _c_f],
    "so3d_scale_f32": [_c_f, _c_f, _int, _c_f, _i64, _c_f],
    "so3d_quat_to_rmat_f32": [_c_f, _c_f, _i64, _c_f],
    "so3d_rmat_to_quat_f32": [_c_f, _c_f, _i64, _c_f],
    "so3d_compose_f32": [_c_f, _int, _int, _c_f, _int, _int, _c_f, _i64, _c_f],
    "so3d_rmat_dist_f32": [_c_f, _c_f, _c_f, _i64, _c_f],
    "so3d_lerp_f32": [_c_f, _c_f, _c_f, _int, _c_f, _i64, _c_f],
    "so3d_log_bwd_f32": [_c_f, _c_f, _c_f, _i64, _c_f],
    "so3d_aa_to_rmat_bwd_f32": [_c_f, _c_f, _c_f, _c_f, _c_f, _i64, _c_f],
    "so3d_expvec_bwd_f32": [_c_f, _c_f, _c_f, _i64, _c_f],
    "so3d_scale_bwd_f32": [_c_f, _c_f, _int, _c_f, _c_f, _c_f, _i64, _c_f],
    "so3d_igso3_density_f32": [_c_f, _c_f, _int, _c_f, _i64, _int, _int, _c_f],
    "so3d_igso3_logp_score_f32": [_c_f, _c_f, _int, _c_f, _c_f, _c_f, _i64, _int, _int, _c_f],
    "so3d_igso3_logp_bwd_f32": [_c_f, _c_f, _c_f, _c_f, _i64, _c_f],
    "so3d_igso3_cdf_table_f32": [_c_f, _i64, _c_f, _c_f, _c_f, _int, _c_f],
    "so3d_igso3_sample_f32": [_c_f, _c_f, _c_f, _i64, _c_f, _i64, _c_f, _c_f, _u64, _u64, _u64, _c_f, _int, _c_f, _c_f, _c_f, _i64, _c_f],
    "so3d_igso3_sample_exact_f32": [_c_f, _int, _c_f, _c_f, _u64, _u64, _u64, _c_f, _int, _c_f, _c_f, _c_f, _i64, _c_f],
    "so3d_igso3_rsample_bwd_f32": [_c_f, _int, _c_f, _c_f, _c_f, _int, _c_f, _c_f, _u64, _u64, _u64, _c_f, _c_f, _i64, _c_f],
    "so3d_igso3_entropy_f32": [_c_f, _c_f, _c_f, _i64, _c_f],
    "so3d_q_sample_f32": [_c_f, _c_f, _c_f, _c_f, _i64, _c_f, _c_f, _c_f, _u64, _u64, _u64, _c_f, _c_f, _c_f, _c_f, _i64, _c_f],
    "so3d_q_sample_given_f32": [_c_f, _c_f, _c_f, _i64, _c_f, _c_f, _i64, _c_f],
    "so3d_p_sample_f32": [_c_f, _c_f, _c_f, _int, _c_f, _c_f, _c_f, _c_f, _i64, _c_f, _c_f, _c_f, _u64, _u64, _u64, _c_f, _c_f, _i64, _c_f],
    "so3d_q_sample_dseed_f32": [_c_f, _c_f, _c_f, _c_f, _i64, _c_f, _c_f, _c_f, _c_f, _u64, _u64, _c_f, _c_f, _i64, _c_f],
    "so3d_p_sample_dseed_f32": [_c_f, _c_f, _c_f, _c_f, _c_f, _c_f, _c_f, _i64, _c_f, _c_f, _c_f, _u64, _u64, _c_f, _i64, _c_f],
    "so3d_rotpredict_p_sample_dseed_f32": [_c_f, _c_f, _c_f, _c_f, _c_f, _c_f, _c_f, _c_f, _i64, _c_f, _c_f, _c_f, _u64, _u64, _c_f, _c_f, _i64, _c_f],
    "so3d_rotpredict_p_sample_loop_f32": [_c_f, _c_f, _c_f, _i64, _i64, _c_f, _c_f, _c_f, _c_f, _i64, _c_f, _c_f, _u64, _c_f, _u64, _c_f, _i64, _c_f],
    "so3d_p_sample_loop_f32": [_c_f, _c_f, _i64, _i64, _c_f, _c_f, _c_f, _c_f, _i64, _c_f, _c_f, _c_f, _u64, _u64, _u64, _c_f, _i64, _c_f],
    "so3d_igso3_cdf_guide": [_c_f, _i64, _c_f, _c_f],
    "so3d_se3_q_sample_f32": [_c_f, _c_f, _c_f, _c_f, _c_f, _i64, _c_f, _c_f, _c_f, ctypes.c_float, _u64, _u64, _u64, _c_f, _c_f, _c_f, _c_f, _i64, _c_f],
    "so3d_se3_p_sample_f32": [_c_f, _c_f, _c_f, _c_f, _c_f, _int, _c_f, _c_f, _c_f, _c_f, _c_f, _i64, _c_f, _c_f, _c_f, ctypes.c_float, _u64, _u64,
                              _u64, _c_f, _c_f, _i64, _c_f],
    "so3d_se3_q_sample_dseed_f32": [_c_f, _c_f, _c_f, _c_f, _c_f, _i64, _c_f, _c_f, _c_f, ctypes.c_float, _c_f, _u64, _u64, _c_f, _c_f, _c_f, _c_f,
                                    _i64, _c_f],
    "so3d_se3_p_sample_dseed_f32": [_c_f, _c_f, _c_f, _c_f, _c_f, _c_f, _c_f, _c_f, _c_f, _c_f, _i64, _c_f, _c_f, ctypes.c_float, _c_f, _u64, _u64,
                                    _c_f, _c_f, _i64, _c_f],
    "so3d_bingham_sample_f32": [_c_f, _c_f, _u64, _u64, _u64, _c_f, _c_f, _i64, _c_f],
    "so3d_rotpredict_pack_f32": [_c_f] * 11 + [_c_f],
    "so3d_rotpredict_p_sample_f32": [_c_f, _c_f, _c_f, _c_f, _c_f, _c_f, _c_f, _c_f, _i64, _c_f, _c_f, _u64, _u64, _u64, _c_f, _c_f, _i64, _c_f],
    "so3d_pair_kernel_sums_f32": [_c_f, _i64, _c_f, _i64, _int, _i64, _i64, _c_f, _i64, _c_f, _c_f],
}

MODE_SERIES, MODE_CLOSED, MODE_AUTO, MODE_SERIES_ADAPTIVE, MODE_SERIES_PURE = 0, 1, 2, 3, 4
MODES = {"series": MODE_SERIES, "closed": MODE_CLOSED, "auto": MODE_AUTO, "series_adaptive": MODE_SERIES_ADAPTIVE, "series_pure": MODE_SERIES_PURE}

PAIR_GAUSSIAN, PAIR_COSINE = 0, 1

_lib = None


def load():
    """Load libso3d.so once; raise loudly if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} not found: the sm_100a extension is not built. Run "
            "`python -m diffusion_extensions_b200.build`. There is no CPU fallback."
        )
    lib = ctypes.CDLL(LIB_PATH)
    lib.so3d_version.restype = ctypes.c_int
    lib.so3d_last_error.restype = ctypes.c_char_p
    for name, argtypes in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is missing
        fn.argtypes = argtypes
        fn.restype = ctypes.c_int
    _lib = lib
    return lib


def ptr(t):
    return None if t is None else t.data_ptr()


def stream_ptr(device=None):
    return torch.cuda.current_stream(device).cuda_stream


def check_f32(t, name, last=None):
    """Contiguous CUDA float32 tensor (copying only when needed)."""
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name} must be a torch.Tensor")
    if not t.is_cuda:
        raise RuntimeError(f"{name} must be a CUDA tensor (got {t.device}); this package has no CPU path")
    if t.dtype != torch.float32:
        raise TypeError(f"{name} must be float32 (got {t.dtype})")
    if last is not None and tuple(t.shape[-len(last):]) != tuple(last):
        raise ValueError(f"{name} must have trailing shape {tuple(last)} (got {tuple(t.shape)})")
    return t.contiguous()


_fn_cache = {}


def call(name, *args, device=None):
    """Invoke an entry point on the current stream of `device`; raise RuntimeError on failure.
    The launch happens under `device` as the current CUDA device; the context switch (a few microseconds of host time
    per call, which small launches feel) is skipped when `device` already is the current one."""
    fn = _fn_cache.get(name)
    if fn is None:
        fn = _fn_cache[name] = getattr(load(), name)
    idx = None if device is None else torch.device(device).index
    if idx is None or idx == torch.cuda.current_device():
        rc = fn(*args, torch.cuda.current_stream().cuda_stream)
    else:
        with torch.cuda.device(idx):
            rc = fn(*args, torch.cuda.current_stream(idx).cuda_stream)
    if rc != 0:
        msg = load().so3d_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"{name} failed (code {rc}): {msg}")
