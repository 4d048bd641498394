"""ctypes binding of the C-ABI in include/drakegpt_b200.h.

The shared library is built in-tree by ``drakegpt_b200/build.py`` (nvcc,
sm_100a).  There is no CPU or PyTorch-eager fallback: if the library is missing
or the device is not a B200-class GPU every op raises.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("DGPT_LIB") or os.path.join(_HERE, "csrc", "libdrakegpt_b200.so")  # DGPT_LIB: debug builds

F32, BF16 = 0, 1
MAJOR_K, MAJOR_MN = 0, 1

EXPORTS = [
    "dgpt_last_error", "dgpt_abi_version", "dgpt_device_check", "dgpt_sm_count", "dgpt_debug_clock_probe", "dgpt_debug_clock_stamps",
    "dgpt_dropout_keep_host", "dgpt_dropout_scale", "dgpt_cast_bf16", "dgpt_embed_fwd",
    "dgpt_embed_bwd", "dgpt_embed_ln_fwd", "dgpt_ln_fwd", "dgpt_ln_bwd", "dgpt_gemm", "dgpt_colsum", "dgpt_attn_fwd",
    "dgpt_attn_bwd", "dgpt_attn_bwd_scratch_bytes", "dgpt_cross_entropy", "dgpt_lmhead_ce", "dgpt_lmhead_ce_supported", "dgpt_gemm_res_ln", "dgpt_gemm_res_ln_supported", "dgpt_adamw", "dgpt_counter_add", "dgpt_sample",
    "dgpt_ipc_export", "dgpt_ipc_open", "dgpt_ipc_close", "dgpt_peer_copy", "dgpt_dp_adamw",
    "dgpt_decode_attn", "dgpt_decode_persistent", "dgpt_decode_persistent_scratch_floats",
    "dgpt_decode_persistent_max_batch", "dgpt_sample_ex", "dgpt_decode_persistent_ex",
    "dgpt_decode_persistent_supported",
]


class GemmArgs(C.Structure):
    _fields_ = [
        ("A", C.c_void_p), ("B", C.c_void_p), ("D", C.c_void_p), ("D2", C.c_void_p),
        ("bias", C.c_void_p), ("residual", C.c_void_p), ("relu_aux", C.c_void_p),
        ("M", C.c_int32), ("N", C.c_int32), ("K", C.c_int32),
        ("in_dtype", C.c_int32), ("d_dtype", C.c_int32), ("d2_dtype", C.c_int32), ("aux_dtype", C.c_int32),
        ("a_major", C.c_int32), ("b_major", C.c_int32),
        ("lda", C.c_int32), ("ldb", C.c_int32), ("ldd", C.c_int32), ("ldd2", C.c_int32),
        ("ldr", C.c_int32), ("ld_aux", C.c_int32),
        ("relu", C.c_int32), ("accumulate", C.c_int32), ("split_k", C.c_int32),
        ("dropout_p", C.c_float), ("site", C.c_uint32), ("seed", C.c_uint64), ("seed_dev", C.c_void_p),
        ("relu_mask_out", C.c_void_p), ("relu_mask_in", C.c_void_p), ("a_colsum", C.c_void_p),
    ]


class AttnArgs(C.Structure):
    _fields_ = [
        ("q", C.c_void_p), ("k", C.c_void_p), ("v", C.c_void_p), ("o", C.c_void_p), ("lse", C.c_void_p),
        ("d_o", C.c_void_p), ("dq", C.c_void_p), ("dk", C.c_void_p), ("dv", C.c_void_p), ("scratch", C.c_void_p),
        ("q_bs", C.c_int64), ("q_rs", C.c_int64), ("k_bs", C.c_int64), ("k_rs", C.c_int64),
        ("v_bs", C.c_int64), ("v_rs", C.c_int64), ("o_bs", C.c_int64), ("o_rs", C.c_int64),
        ("dq_bs", C.c_int64), ("dq_rs", C.c_int64), ("dk_bs", C.c_int64), ("dk_rs", C.c_int64),
        ("dv_bs", C.c_int64), ("dv_rs", C.c_int64), ("do_bs", C.c_int64), ("do_rs", C.c_int64),
        ("dtype", C.c_int32), ("B", C.c_int32), ("NH", C.c_int32), ("H", C.c_int32),
        ("Tq", C.c_int32), ("Tk", C.c_int32),
        ("scale", C.c_float), ("dropout_p", C.c_float), ("site", C.c_uint32), ("seed", C.c_uint64),
        ("seed_dev", C.c_void_p),
    ]


class KernelError(RuntimeError):
    pass


_lib = None


def _declare(lib):
    vp, i32, i64, u32, u64, f32 = C.c_void_p, C.c_int, C.c_int64, C.c_uint32, C.c_uint64, C.c_float
    lib.dgpt_last_error.restype = C.c_char_p
    lib.dgpt_last_error.argtypes = []
    for name in ("dgpt_abi_version", "dgpt_device_check", "dgpt_sm_count"):
        getattr(lib, name).restype = i32
        getattr(lib, name).argtypes = []
    lib.dgpt_debug_clock_probe.restype = i32
    lib.dgpt_debug_clock_probe.argtypes = [C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    lib.dgpt_debug_clock_stamps.restype = i32
    lib.dgpt_debug_clock_stamps.argtypes = [C.POINTER(C.c_uint64)]
    lib.dgpt_dropout_keep_host.restype = i32
    lib.dgpt_dropout_keep_host.argtypes = [u64, u32, u64, f32]
    sig = {
        "dgpt_dropout_scale": [vp, vp, vp, i32, i64, f32, u64, vp, u32, vp],
        "dgpt_cast_bf16": [vp, vp, i64, vp],
        "dgpt_embed_fwd": [vp, vp, vp, vp, i32, i32, i32, i32, i32, vp],
        "dgpt_embed_bwd": [vp, vp, vp, vp, i32, i32, i32, i32, i32, vp],
        "dgpt_ln_fwd": [vp, vp, vp, vp, i32, vp, vp, i32, i32, f32, vp],
        "dgpt_embed_ln_fwd": [vp, vp, vp, vp, vp, vp, vp, i32, vp, vp, i32, i32, i32, i32, i32, f32, vp],
        "dgpt_ln_bwd": [vp, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, vp, f32, u64, vp, u32, i32, i32, vp],
        "dgpt_gemm": [C.POINTER(GemmArgs), vp],
        "dgpt_colsum": [vp, i32, i32, i32, i32, vp, i32, vp],
        "dgpt_attn_fwd": [C.POINTER(AttnArgs), vp],
        "dgpt_attn_bwd": [C.POINTER(AttnArgs), vp],
        "dgpt_cross_entropy": [vp, i32, vp, vp, vp, i32, i32, vp, i32, i32, vp],
        "dgpt_lmhead_ce": [vp, i32, vp, i32, vp, vp, vp, vp, i32, vp, i32, vp, i32, i32, i32, vp],
        "dgpt_lmhead_ce_supported": [i32, i32],
        "dgpt_gemm_res_ln": [vp, i32, vp, i32, vp, vp, i32, vp, i32, vp, vp, vp, i32, vp, vp, i32, i32, i32, f32, f32, u64, vp, u32, vp],
        "dgpt_gemm_res_ln_supported": [i32, i32],
        "dgpt_adamw": [vp, vp, vp, vp, vp, i64, vp, vp, i32, vp],
        "dgpt_counter_add": [vp, u64, vp],
        "dgpt_decode_attn": [vp, vp, vp, vp, i64, i64, i64, i64, i64, i64, i32, i32, i32, i32, f32, vp],
        "dgpt_decode_persistent": [C.POINTER(C.c_void_p), i32, vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, i32,
                                   i32, i32, i32, i32, u64, vp, i32, vp],
        "dgpt_ipc_export": [vp, vp, C.POINTER(C.c_int64)],
        "dgpt_ipc_open": [vp, i64, C.POINTER(C.c_void_p)],
        "dgpt_ipc_close": [vp, i64],
        "dgpt_peer_copy": [vp, vp, i64, vp],
        "dgpt_dp_adamw": [C.POINTER(C.c_void_p), i32, i32, vp, vp, i64, i64, vp, vp, vp, vp, i32, vp],
        "dgpt_sample": [vp, i32, vp, i64, i32, i32, i32, i32, u64, vp, u32, vp],
        "dgpt_sample_ex": [vp, i32, vp, i64, i32, i32, i32, i32, u64, vp, u32, vp, vp],
        "dgpt_decode_persistent_ex": [C.POINTER(C.c_void_p), i32, vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, i32,
                                      i32, i32, i32, i32, i32, u64, vp, vp, i32, vp],
        "dgpt_decode_persistent_supported": [i32, i32, i32, i32, i32, i32, i32, i32, i32],
    }
    for name, args in sig.items():
        fn = getattr(lib, name)
        fn.restype = i32
        fn.argtypes = args
    lib.dgpt_decode_persistent_max_batch.restype = i32
    lib.dgpt_decode_persistent_max_batch.argtypes = []
    lib.dgpt_decode_persistent_scratch_floats.restype = i64
    lib.dgpt_decode_persistent_scratch_floats.argtypes = [i32, i32, i32, i32, i32]
    lib.dgpt_attn_bwd_scratch_bytes.restype = i64
    lib.dgpt_attn_bwd_scratch_bytes.argtypes = [C.POINTER(AttnArgs)]


def lib():
    """Load (once) and return the kernel library; raise if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise KernelError(
                f"{LIB_PATH} is missing: build it with `python -m drakegpt_b200.build` "
                "(drakegpt_b200 has no CPU / PyTorch-eager fallback)")
        handle = C.CDLL(LIB_PATH)
        _declare(handle)
        _lib = handle
    return _lib


def check(rc, what=""):
    if rc != 0:
        msg = lib().dgpt_last_error().decode("utf-8", "replace")
        raise KernelError(f"drakegpt_b200 kernel call {what} failed (code {rc}): {msg}")


def require_gpu():
    """Fail loudly unless the current CUDA device can run the sm_100a kernels."""
    check(lib().dgpt_device_check(), "dgpt_device_check")
