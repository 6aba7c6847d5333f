"""ctypes binding of libvpt_b200.so (the C ABI declared in include/vpt_b200.h).

There is NO fallback: if the shared library is missing or an entry point fails, this module raises.  The library is
built in-tree by `build()` (also called from `__graft_entry__.build()`), never JIT-cached elsewhere.
"""
import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
LIB_PATH = os.path.join(_HERE, "libvpt_b200.so")
SRC = os.path.join(_HERE, "csrc", "vpt_b200.cu")
HEADER = os.path.join(_ROOT, "include", "vpt_b200.h")

ABI_VERSION = 3  # == VPT_ABI_VERSION in include/vpt_b200.h (checked against the loaded library)

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-shared",
              "-Xcompiler", "-fPIC"]


def _sources():
    d = os.path.join(_HERE, "csrc")
    return [os.path.join(d, f) for f in sorted(os.listdir(d))] + [HEADER]


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile csrc/vpt_b200.cu (unity build) for sm_100a into libvpt_b200.so next to this file."""
    if not force and os.path.isfile(LIB_PATH):
        newest = max(os.path.getmtime(p) for p in _sources())
        if os.path.getmtime(LIB_PATH) >= newest:
            return LIB_PATH
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + [SRC, "-o", LIB_PATH]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + r.stdout + r.stderr)
    if verbose:
        print(r.stderr)
    return LIB_PATH


class GemmArgs(C.Structure):
    """struct vpt_gemm_args (include/vpt_b200.h)."""
    _fields_ = [
        ("A", C.c_void_p), ("B", C.c_void_p),
        ("M", C.c_int32), ("N", C.c_int32), ("K", C.c_int32),
        ("conv", C.c_int32), ("H", C.c_int32), ("W", C.c_int32), ("Cin", C.c_int32),
        ("mr", C.c_void_p), ("rows_per_group", C.c_int32),
        ("S1", C.c_void_p), ("S2", C.c_void_p),
        ("relu", C.c_int32), ("out_scale", C.c_float),
        ("residual", C.c_void_p), ("residual_f32", C.c_int32), ("ld_res", C.c_int64),
        ("out", C.c_void_p), ("out_f32", C.c_int32), ("ld_out", C.c_int64),
        ("seg_len", C.c_int32), ("seg_stride", C.c_int64), ("seg_off", C.c_int64),
        ("stat_part", C.c_void_p), ("stat_mode", C.c_int32), ("cluster", C.c_int32),
        ("ndst", C.c_int32), ("dst_n0", C.c_int32 * 4), ("dst_out", C.c_void_p * 4), ("dst_ld", C.c_int64 * 4), ("dst_f32", C.c_int32 * 4),
        ("dst_remap", C.c_int32 * 4),
    ]


class ConvZpArgs(C.Structure):
    """struct vpt_conv_zp_args (include/vpt_b200.h)."""
    _fields_ = [
        ("x", C.c_void_p), ("w", C.c_void_p),
        ("F", C.c_int32), ("H", C.c_int32), ("W", C.c_int32), ("Cin", C.c_int32), ("Cout", C.c_int32),
        ("mr", C.c_void_p), ("S1", C.c_void_p), ("S2", C.c_void_p),
        ("relu", C.c_int32), ("residual", C.c_void_p), ("out", C.c_void_p), ("stat_part", C.c_void_p),
        ("Ef", C.c_void_p), ("res_scale", C.c_void_p), ("res_shift", C.c_void_p),
    ]


_P, _I, _L, _F, _D = C.c_void_p, C.c_int32, C.c_int64, C.c_float, C.c_double

# name -> (restype, argtypes); every symbol include/vpt_b200.h declares
SIGNATURES = {
    "vpt_last_error": (C.c_char_p, []),
    "vpt_abi_version": (_I, []),
    "vpt_device_error": (_I, []),
    "vpt_num_sms": (_I, []),
    "vpt_gemm_bf16": (_I, [C.POINTER(GemmArgs), _P]),
    "vpt_gemm_stat_parts": (_I, [_I]),
    "vpt_set_default_cluster": (_I, [_I]),
    "vpt_conv3x3_zp": (_I, [C.POINTER(ConvZpArgs), _P]),
    "vpt_conv_zp_stat_parts": (_I, [_I, _I, _I, _I]),
    "vpt_conv_zp_t_stat_floats": (_L, [_I, _I, _I, _I]),
    "vpt_conv_zp_t_stats_finalize": (_I, [_P, _P, _I, _I, _I, _F, _P]),
    "vpt_set_conv_pair_mode": (_I, [_I]),
    "vpt_set_conv_swap_mode": (_I, [_I]),
    "vpt_set_wgrad_mode": (_I, [_I]),
    "vpt_set_pdl": (_I, [_I]),
    "vpt_debug_set": (_I, [_I, _I]),
    "vpt_firstconv_pool": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _P]),
    "vpt_firstconv_stat_parts": (_I, [_I, _I, _I, _I]),
    "vpt_set_firstconv_mode": (_I, [_I]),
    "vpt_conv3d_t5": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _P]),
    "vpt_group_stats_f32": (_I, [_P, _P, _L, _L, _F, _P]),
    "vpt_norm_split_f32": (_I, [_P, _P, _P, _P, _P, _P, _P, _L, _I, _L, _P]),
    "vpt_add_f32": (_I, [_P, _P, _P, _L, _I, _P]),
    "vpt_maxpool3s2_f32": (_I, [_P, _P, _L, _I, _I, _I, _P]),
    "vpt_attention_f32": (_I, [_P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "vpt_codec_to_env": (_I, [_P, _P, _P, _P, _P, _I, _I, _L, _P, _P, _P]),
    "vpt_codec_from_env": (_I, [_P, _P, _P, _I, _P, _L, _L, _P, _P]),
    "vpt_conv3d_stat_parts": (_I, [_I, _I, _I]),
    "vpt_maxpool3s2": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "vpt_norm2_fold": (_I, [_P, _I, _I, _L, _P, _P, _P, _P, _P, _P, _I, _F, _P, _P, _P, _P, _L, _P]),
    "vpt_pool_stat_parts": (_I, [_I, _I, _I, _I]),
    "vpt_pool_chan_parts": (_I, [_I, _I, _I, _I]),
    "vpt_affine_norm": (_I, [_P, _P, _P, _P, _P, _P, _P, _L, _I, _I, _P]),
    "vpt_affine_norm_zp": (_I, [_P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _P]),
    "vpt_norm_stat_parts": (_I, [_I, _I]),
    "vpt_stats_finalize": (_I, [_P, _P, _L, _I, _D, _F, _P]),
    "vpt_copy_rows": (_I, [_P, _I, _L, _L, _L, _P, _I, _L, _L, _L, _I, _I, _I, _P]),
    "vpt_copy_rows2": (_I, [_P, _P, _I, _L, _L, _L, _P, _P, _I, _L, _L, _L, _I, _I, _I, _P]),
    "vpt_state_mask_update": (_I, [_P, _P, _L, _P, _I, _I, _I, _P]),
    "vpt_attention": (_I, [_P, _P, _P, _P, _L, _P, _P, _L, _P, _P, _I, _I, _I, _I, _I, _I, _P]),
    "vpt_log_softmax": (_I, [_P, _L, _I, _I, _P, _L, _P]),
    "vpt_gumbel_argmax": (_I, [_P, _P, _P, _L, _I, _P]),
    "vpt_gather_logprob": (_I, [_P, _P, _P, _L, _I, _I, _P]),
    "vpt_resize_bilinear_u8": (_I, [_P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _P]),
    "vpt_composite_cursor_u8": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "vpt_adam_step": (_I, [_P, _P, _P, _P, _L, _F, _F, _F, _F, _F, _F, _I, _P]),
    # BC backward (training.py)
    "vpt_relu_mask": (_I, [_P, _P, _P, _L, _P]),
    "vpt_add_stats": (_I, [_P, _P, _P, _P, _L, _L, _P]),
    "vpt_add_stat_parts": (_I, [_L]),
    "vpt_wgrad_bf16": (_I, [_P, _L, _P, _L, _I, _I, _L, C.POINTER(C.c_int32), _I, _P, _P, _L, _P]),
    "vpt_wgrad_workspace_bytes": (_L, [_I, _I, _I, _L]),
    "vpt_group_sums": (_I, [_P, _P, _P, _P, _P, _P, _L, _I, _I, _D, _P]),
    "vpt_group_sums_parts": (_I, [_I, _I]),
    "vpt_col_sums": (_I, [_P, _L, _P, _P, _L, _I, _I, _P, _P, _P]),
    "vpt_col_sums_parts": (_I, [_L, _I]),
    "vpt_norm_sums": (_I, [_P, _P, _P, _P, _L, _I, _I, _D, _P, _P, _P, _P]),
    "vpt_norm_sums_workspace": (_L, [_L, _I, _I]),
    "vpt_norm_bwd_apply": (_I, [_P, _P, _P, _P, _P, _P, _P, _L, _I, _I, _I, _I, _I, _I, _P]),
    "vpt_maxpool3s2_bwd": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _P]),  # dy, x, dx, workspace
    "vpt_firstconv_bwd": (_I, [_P, _P, _P, _P, _P, _P, _P, _L, _I, _I, _I, _P]),
    "vpt_firstconv_bwd_parts": (_I, [_L, _I, _I]),
    "vpt_attention_bwd": (_I, [_P, _P, _P, _P, _L, _P, _P, _L, _P, _P, _P, _L, _P, _P, _I, _I, _I, _I, _I, _P]),
    "vpt_softmax_bwd": (_I, [_P, _P, _F, _P, _L, _I, _L, _I, _P]),
    # RL step (training.RLTrainer)
    "vpt_rl_heads_bwd": (_I, [C.POINTER(_P), C.POINTER(_P), C.POINTER(_P), C.POINTER(_I), C.POINTER(_I), _I, _P, _P, _P, _P, _P, _F, _F, _F, _F,
                              _F, _F, _P, _L, _I, _P, _L, _P]),
}

_lib = None


class NativeError(RuntimeError):
    pass


def lib():
    """The loaded library with argtypes set.  Raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise NativeError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                              "(there is no CPU / PyTorch fallback for the VPT forward path)")
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(l, name)  # AttributeError if the ABI is out of sync with the header
            fn.restype, fn.argtypes = res, args
        if l.vpt_abi_version() != ABI_VERSION:
            raise NativeError(f"libvpt_b200.so ABI version {l.vpt_abi_version()} != {ABI_VERSION} (rebuild: __graft_entry__.build())")
        _lib = l
    return _lib


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = lib().vpt_last_error()
        raise NativeError(f"{what} failed (rc={rc}): {msg.decode() if msg else ''}")


def device_check():
    """Synchronise and raise if a kernel recorded a device-side watchdog error (tests / debugging)."""
    check(lib().vpt_device_error(), "vpt_device_error")
