"""ctypes binding of libcnb200.so (include/cnb200.h).  PyTorch is used for device memory and streams only.

There is no CPU path: if the library cannot be loaded every op raises, and every op rejects non-CUDA tensors.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libcnb200.so")

MODE_F32, MODE_F16 = 0, 1
MAX_TAPS = 16
ROUTE_LEN = 16      # CNB_ROUTE_LEN

c_void_p, c_int, c_ll, c_float, c_u64 = ctypes.c_void_p, ctypes.c_int, ctypes.c_longlong, ctypes.c_float, ctypes.c_uint64


class ConvParams(ctypes.Structure):
    """Mirror of `struct cnb_conv_params` (include/cnb200.h)."""
    _fields_ = [
        ("inp", c_void_p), ("weight", c_void_p), ("weight_lp", c_void_p), ("bias", c_void_p),
        ("temb", c_void_p), ("residual", c_void_p), ("out", c_void_p),
        ("B", ctypes.c_int32), ("H", ctypes.c_int32), ("W", ctypes.c_int32), ("Cin", ctypes.c_int32),
        ("ldi", ctypes.c_int32), ("in_coff", ctypes.c_int32),
        ("OH", ctypes.c_int32), ("OW", ctypes.c_int32), ("OHf", ctypes.c_int32), ("OWf", ctypes.c_int32),
        ("oy_mul", ctypes.c_int32), ("oy_add", ctypes.c_int32), ("ox_mul", ctypes.c_int32), ("ox_add", ctypes.c_int32),
        ("Cout", ctypes.c_int32), ("ldo", ctypes.c_int32), ("out_coff", ctypes.c_int32),
        ("ldr", ctypes.c_int32), ("res_coff", ctypes.c_int32),
        ("stride", ctypes.c_int32), ("ntaps", ctypes.c_int32),
        ("dy", ctypes.c_int8 * MAX_TAPS), ("dx", ctypes.c_int8 * MAX_TAPS),
        ("temb_ld", ctypes.c_int32), ("temb_per_sample", ctypes.c_int32),
        ("act", ctypes.c_int32), ("mode", ctypes.c_int32), ("in_dtype", ctypes.c_int32), ("out_dtype", ctypes.c_int32), ("res_dtype", ctypes.c_int32),
        ("in2", c_void_p), ("Cin2", ctypes.c_int32), ("ldi2", ctypes.c_int32), ("in2_coff", ctypes.c_int32),
    ]


_SIGS = {
    "cnb_abi_version": (c_int, []),
    "cnb_sizeof_conv_params": (c_int, []),
    "cnb_last_error": (ctypes.c_char_p, []),
    "cnb_launch_count": (c_ll, []),
    "cnb_reset_launch_count": (None, []),
    "cnb_has_tcgen05": (c_int, []),
    "cnb_conv2d": (c_int, [ctypes.POINTER(ConvParams), c_void_p]),
    "cnb_conv2d_route": (c_int, [ctypes.POINTER(ConvParams), ctypes.POINTER(ctypes.c_int32)]),
    "cnb_pack_conv_weight": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "cnb_pack_convT_weight": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "cnb_cast_f16": (c_int, [c_void_p, c_void_p, c_ll, c_void_p]),
    "cnb_groupnorm": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_float, c_int,
                              c_int, c_int, c_void_p]),
    "cnb_groupnorm_workspace_bytes": (ctypes.c_size_t, [c_int, c_int, c_int, c_int, c_int]),
    "cnb_groupnorm_ws": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_float, c_int,
                                 c_int, c_int, c_void_p, ctypes.c_size_t, c_void_p]),
    "cnb_attention": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "cnb_attention_f16": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "cnb_attention_tmem": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "cnb_attention_mma": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "cnb_linear_small": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int,
                                 c_void_p]),
    "cnb_time_embedding": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "cnb_sched_step": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_ll, c_void_p, c_u64, c_u64,
                               c_void_p, c_u64, c_void_p]),
    "cnb_ddim_step": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_ll, c_void_p, c_int, c_u64, c_u64,
                              c_void_p, c_u64, c_void_p]),
    "cnb_dpm_solver_step": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_ll, c_void_p, c_int,
                                    c_u64, c_u64, c_void_p, c_u64, c_void_p]),
    "cnb_add_noise": (c_int, [c_void_p, c_void_p, c_void_p, c_ll, c_float, c_float, c_u64, c_u64, c_u64, c_void_p]),
    "cnb_inpaint_blend": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_ll, c_int, c_ll, c_int, c_void_p, c_ll,
                                  c_void_p, c_u64, c_u64, c_u64, c_void_p]),
    "cnb_mask_max_pool": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "cnb_philox_normal": (c_int, [c_void_p, c_ll, c_u64, c_u64, c_u64, c_void_p]),
    "cnb_gather_row": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    "cnb_sampler_prologue": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "cnb_bump_index": (c_int, [c_void_p, c_int, c_void_p]),
    "cnb_edm_coeffs": (c_int, [c_void_p, c_int, c_float, c_float, c_void_p, c_void_p, c_void_p, c_void_p]),
    "cnb_scale_rows": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_ll, c_void_p]),
    "cnb_x0_from_eps": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_int, c_ll,
                                c_void_p]),
    "cnb_scale_nchw_to_nhwc": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "cnb_edm_combine_to_nchw": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_int, c_int,
                                        c_int, c_int, c_void_p]),
    "cnb_nchw_to_nhwc": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "cnb_nhwc_to_nchw": (c_int, [c_void_p, c_int, c_int, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "cnb_copy_channels": (c_int, [c_void_p, c_int, c_int, c_void_p, c_int, c_int, c_ll, c_int, c_int, c_void_p]),
    "cnb_tc_error_flag": (c_int, []),
}

EXPORTS = tuple(_SIGS)
_lib = None


class CnbError(RuntimeError):
    pass


def lib():
    """Load (building first if the .so is absent and nvcc exists).  Raises if the native library is unavailable."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_LIB_PATH):
        from .build import build
        build()
    try:
        handle = ctypes.CDLL(_LIB_PATH)
    except OSError as e:   # fail loudly: there is no fallback implementation
        raise CnbError(f"libcnb200.so could not be loaded ({e}); run `python controlnet-pytorch_b200/build.py`") from e
    for name, (res, args) in _SIGS.items():
        fn = getattr(handle, name)
        fn.restype = res
        fn.argtypes = args
    if handle.cnb_sizeof_conv_params() != ctypes.sizeof(ConvParams):
        raise CnbError("ConvParams mirror is out of sync with include/cnb200.h (%d vs %d bytes)" % (
            ctypes.sizeof(ConvParams), handle.cnb_sizeof_conv_params()))
    _lib = handle
    return _lib


def check(rc):
    if rc != 0:
        msg = lib().cnb_last_error()
        raise CnbError(f"libcnb200 error {rc}: {msg.decode() if msg else ''}")


def stream():
    return torch.cuda.current_stream().cuda_stream


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise CnbError("controlnet-pytorch_b200 has no CPU path: tensors must live on a CUDA device "
                           "(got device=%s)" % t.device)


def ptr(t):
    return 0 if t is None else t.data_ptr()


# ---- global compute mode -----------------------------------------------------------------------------------
_MODE = None
_MODE_NAMES = {"fp32": MODE_F32, "f32": MODE_F32, "f16": MODE_F16, "fp16": MODE_F16,
               "tf32": MODE_F16}     # "tf32": the name this mode carried in round 1 (kept as an alias)


def set_mode(name):
    """'fp32' (CUDA-core exact path, 1e-4 gate) or 'f16' (tcgen05 tensor-core path: fp16 operands and activation
    stream, fp32 accumulators / statistics; 1e-2 gate).  There is no bf16 mode: bf16 operands measured 1.2e-2 .. 2e-2
    eps rel-L2 on the MNIST widths (SURVEY.md Appendix D), outside north_star's own 1e-2 gate, so it is rejected
    instead of silently running something else."""
    global _MODE
    if name in ("bf16", "bfloat16"):
        raise ValueError("bf16 mode is not implemented (bf16 operands miss the 1e-2 eps gate on the MNIST widths, "
                         "SURVEY.md Appendix D); use 'f16' (fp16 operands, fp32 accumulate) or 'fp32'")
    if name not in _MODE_NAMES:
        raise ValueError(f"unknown mode {name!r}; expected one of {sorted(_MODE_NAMES)}")
    _MODE = _MODE_NAMES[name]


def get_mode():
    global _MODE
    if _MODE is None:
        env = os.environ.get("CNB_MODE")
        if env:
            set_mode(env)
        else:
            _MODE = MODE_F16 if lib().cnb_has_tcgen05() else MODE_F32
    return _MODE


def mode_name(m=None):
    m = get_mode() if m is None else m
    return {MODE_F32: "fp32", MODE_F16: "f16"}[m]


def attention_kernel_name(L=784, d=16):
    """Name of the kernel cnb_attention_f16 dispatches to for (sequence length L, head dim d): the measured routing rule of
    csrc/attention_tmem.cu::attention_tmem_default (bench.py's roofline label)."""
    if d in (4, 8, 16, 24, 32, 48, 64) and L >= 128 and d >= 24:
        return "attention_tmem_kernel (tcgen05.mma SS + TS, S/P/O in TMEM, TMA)"
    return "attention_f16_kernel (mma.sync m16n8k16)"


def launch_count():
    return int(lib().cnb_launch_count())


def reset_launch_count():
    lib().cnb_reset_launch_count()
