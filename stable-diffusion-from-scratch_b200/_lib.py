"""ctypes binding of libsdb200.so (the C-ABI declared in include/sdb200.h).

There is no fallback: if the shared library is missing or a call fails, an exception is raised.
PyTorch is used only for device memory (`tensor.data_ptr()`) and the current CUDA stream.
"""
import ctypes as C
import os

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libsdb200.so")

F32, BF16 = 0, 1

_lib = None


class SdbError(RuntimeError):
    pass


class SimtArgs(C.Structure):
    _fields_ = [
        ("A", C.c_void_p), ("B", C.c_void_p), ("out", C.c_void_p),
        ("bias", C.c_void_p), ("rowvec", C.c_void_p), ("residual", C.c_void_p),
        ("lda", C.c_longlong), ("ldb", C.c_longlong), ("ldc", C.c_longlong), ("ldr", C.c_longlong), ("ldv", C.c_longlong),
        ("M", C.c_int), ("N", C.c_int), ("K", C.c_int),
        ("alpha", C.c_float),
        ("b_kn", C.c_int),
        ("nb1", C.c_int), ("nb2", C.c_int),
        ("sa1", C.c_longlong), ("sa2", C.c_longlong), ("sb1", C.c_longlong), ("sb2", C.c_longlong),
        ("sc1", C.c_longlong), ("sc2", C.c_longlong),
        ("kh", C.c_int), ("kw", C.c_int), ("stride", C.c_int), ("pad", C.c_int), ("up", C.c_int),
        ("NB", C.c_int), ("IH", C.c_int), ("IW", C.c_int), ("Cin", C.c_int), ("OH", C.c_int), ("OW", C.c_int),
        ("out_dtype", C.c_int),
    ]


class TcArgs(C.Structure):
    _fields_ = [
        ("A", C.c_void_p), ("B", C.c_void_p), ("out", C.c_void_p),
        ("bias", C.c_void_p), ("rowvec", C.c_void_p), ("residual", C.c_void_p),
        ("lda", C.c_longlong), ("ldb", C.c_longlong), ("ldc", C.c_longlong), ("ldr", C.c_longlong), ("ldv", C.c_longlong),
        ("M", C.c_int), ("N", C.c_int), ("K", C.c_int),
        ("out_dtype", C.c_int),
        ("geglu", C.c_int),
        ("col_group", C.c_int), ("col_group_stride", C.c_int),
        ("split_k", C.c_int),
        ("block_n", C.c_int),
        ("taps", C.c_int), ("kw", C.c_int),
        ("stride", C.c_int), ("pad_h", C.c_int), ("pad_w", C.c_int),
        ("NB", C.c_int), ("IH", C.c_int), ("IW", C.c_int), ("Cin", C.c_int), ("OH", C.c_int), ("OW", C.c_int),
        ("cout_pad", C.c_int),
        ("out_sh", C.c_int), ("out_sw", C.c_int), ("out_oh", C.c_int), ("out_ow", C.c_int), ("OHF", C.c_int), ("OWF", C.c_int),
        ("ws", C.c_void_p), ("ws_bytes", C.c_longlong),
        ("rows_per_item", C.c_int),
        ("variant", C.c_int),
        ("colstats", C.c_void_p), ("colstats_slots", C.c_longlong),
        ("b_const", C.c_int),
    ]


class AttnArgs(C.Structure):
    _fields_ = [
        ("q", C.c_void_p), ("k", C.c_void_p), ("v", C.c_void_p), ("out", C.c_void_p),
        ("q_bs", C.c_longlong), ("q_ss", C.c_longlong), ("q_hs", C.c_longlong),
        ("k_bs", C.c_longlong), ("k_ss", C.c_longlong), ("k_hs", C.c_longlong),
        ("v_bs", C.c_longlong), ("v_ss", C.c_longlong), ("v_hs", C.c_longlong),
        ("o_bs", C.c_longlong), ("o_ss", C.c_longlong), ("o_hs", C.c_longlong),
        ("B", C.c_int), ("H", C.c_int), ("Sq", C.c_int), ("Sk", C.c_int), ("d", C.c_int), ("dpad", C.c_int),
        ("scale", C.c_float),
        ("dense", C.c_int),
        ("causal", C.c_int),
    ]


# name -> (restype, argtypes); kept in one table so tests can check it against include/sdb200.h
_P, _I, _L, _F = C.c_void_p, C.c_int, C.c_longlong, C.c_float
SIGNATURES = {
    "sdb_version": (_I, []),
    "sdb_last_error_string": (C.c_char_p, []),
    "sdb_device_sm_count": (_I, []),
    "sdb_launch_count": (C.c_ulonglong, []),
    "sdb_pdl_skip_next": (_I, [_I]),
    "sdb_nchw_to_nhwc": (_I, [_P, _P, _I, _I, _I, _I, _I, _P]),
    "sdb_nchw_to_nhwc_split": (_I, [_P, _P, _I, _I, _I, _I, _P]),
    "sdb_nchw_concat_to_nhwc": (_I, [_P, _I, _P, _I, _P, _I, _I, _I, _I, _I, _P]),
    "sdb_nhwc_to_nchw": (_I, [_P, _P, _I, _I, _I, _P]),
    "sdb_groupnorm_ws_bytes": (_L, [_I, _I, _I, _I]),
    "sdb_groupnorm_nhwc": (_I, [_P, _I, _P, _I, _I, _I, _I, _F, _P, _P, _L, _I, _I, _P, _I, _P, _P, _P, _P]),
    "sdb_scale_shift_affine": (_I, [_P, _P, _P, _L, _I, _I, _P, _P, _P]),
    "sdb_avgpool2x2": (_I, [_P, _I, _I, _I, _I, _P, _I, _P]),
    "sdb_groupnorm_from_colstats": (_I, [_P, _I, _P, C.POINTER(C.c_longlong), _P, _I, _P, C.POINTER(C.c_longlong), _I, _I, _I, _F,
                                         _P, _P, _L, _I, _I, _P, _I, _P, _P, _P]),
    "sdb_layernorm": (_I, [_P, _I, _I, _F, _P, _P, _P, _I, _P]),
    "sdb_cast_concat": (_I, [_P, _I, _P, _I, _I, _I, _I, _I, _P, _I, _P]),
    "sdb_upsample_bilinear2x": (_I, [_P, _I, _I, _I, _I, _P, _I, _P]),
    "sdb_activation": (_I, [_P, _P, _I, _L, _I, _P]),
    "sdb_geglu": (_I, [_P, _I, _I, _P, _I, _P]),
    "sdb_softmax_rows": (_I, [_P, _L, _I, _L, _F, _P, _I, _L, _P]),
    "sdb_softmax_rows_causal": (_I, [_P, _L, _I, _I, _L, _F, _P, _I, _L, _P]),
    "sdb_add": (_I, [_P, _P, _P, _L, _P]),
    "sdb_add_rowvec": (_I, [_P, _P, _L, _I, _L, _I, _P, _I, _P]),
    "sdb_timestep_embedding": (_I, [_P, _P, _I, _I, _I, _P, _P]),
    "sdb_gather_rows": (_I, [_P, _P, _I, _I, _P, _P]),
    "sdb_skinny_linear": (_I, [_P, _I, _I, _P, _P, _I, _I, _I, _P, _P]),
    "sdb_skinny_linear_bf16w": (_I, [_P, _I, _I, _P, _P, _I, _I, _I, _P, _P]),
    "sdb_ddim_step": (_I, [_P, _P, _P, _F, _P, _F, _F, _F, _F, _F, _F, _P, _P, _L, _P]),
    "sdb_ddim_xprev": (_I, [_P, _P, _P, _F, _P, _F, _F, _F, _F, _P, _L, _P]),
    "sdb_ddpm_step": (_I, [_P, _P, _P, _P, _P, _P, _I, _I, _F, _P, _P, _I, _L, _P]),
    "sdb_inpaint_blend": (_I, [_P, _P, _P, _P, _P, _P, _I, _I, _I, _L, _P, _P]),
    "sdb_diag_gaussian": (_I, [_P, _P, _I, _I, _L, _P, _P, _P, _P, _P, _P]),
    "sdb_q_sample": (_I, [_P, _P, _P, _P, _I, _L, _P, _P]),
    "sdb_simt_contract": (_I, [C.POINTER(SimtArgs), _P]),
    "sdb_tc_contract": (_I, [C.POINTER(TcArgs), _P]),
    "sdb_tc_set_pair_kernel": (_I, [_I]),
    "sdb_tc_set_tma_epilogue": (_I, [_I]),
    "sdb_tc_set_tail_split": (_I, [_I]),
    "sdb_tc_workspace_bytes": (_L, [C.POINTER(TcArgs)]),
    "sdb_tc_colstats_layout": (_I, [C.POINTER(TcArgs), C.POINTER(C.c_longlong), C.POINTER(C.c_longlong)]),
    "sdb_attention_fwd": (_I, [C.POINTER(AttnArgs), _P]),
    "sdb_attention_set_short_key_kernel": (_I, [_I]),
    "sdb_attention_wide_fwd": (_I, [_P, _P, _P, _P, _L, _L, _L, _L, _L, _L, _L, _L, _I, _I, _I, _I, _F, _P]),
    "sdb_vq_ws_bytes": (_L, [_L, _I]),
    "sdb_vq_quantize": (_I, [_P, _I, _I, _I, _I, _P, _I, _F, _P, _I, _P, _P, _P, _P, _P]),
    "sdb_vq_codebook_gather": (_I, [_P, _L, _P, _I, _I, _P, _I, _I, _P]),
    "sdb_patch_unfold": (_I, [_P, _I, _I, _I, _I, _I, _I, _I, _I, _P, _P]),
    "sdb_patch_fold": (_I, [_P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _I, _P, _P, _I, _P, _P]),
}


def load(path=None):
    """Load libsdb200.so and attach signatures. Raises SdbError when it is absent."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    path = path or LIB_PATH
    if not os.path.exists(path):
        raise SdbError(
            "libsdb200.so not found at %s — build it with `python -c 'import __graft_entry__ as g; g.build()'`; "
            "there is no CPU or PyTorch fallback for the sdb200 hot path" % path)
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)   # AttributeError if the symbol is missing: loud on purpose
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc, what=""):
    if rc != 0:
        msg = load().sdb_last_error_string()
        raise SdbError("%s failed (rc=%d): %s" % (what or "sdb call", rc, msg.decode() if msg else "?"))


def stream_ptr():
    return torch.cuda.current_stream().cuda_stream


def stream_fence():
    """Call right after a cross-stream wait (fork to / join from a side stream): the next kernel launch is made without the
    programmatic-dependent-launch attribute, so it starts only once everything its stream waits for has completed."""
    load().sdb_pdl_skip_next(1)


def ptr(t):
    return 0 if t is None else t.data_ptr()


def dtype_code(dt):
    if dt == torch.float32:
        return F32
    if dt == torch.bfloat16:
        return BF16
    raise SdbError("unsupported dtype %s" % dt)


def require_cuda(*tensors):
    """Every operand must live on ONE CUDA device and that device must be the current one: kernels are enqueued on the
    current device's current stream (`stream_ptr`), so a tensor elsewhere would be dereferenced by the wrong GPU.  The
    module-level entry points (UNetModel.forward, AutoencoderKL.decode, ...) switch to their input's device themselves."""
    dev = None
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise SdbError("sdb200 kernels need CUDA tensors (got %s); there is no CPU fallback" % t.device)
        if dev is None:
            dev = t.device
        elif t.device != dev:
            raise SdbError("sdb200 op got operands on different devices (%s and %s)" % (dev, t.device))
    if dev is not None and dev.index != torch.cuda.current_device():
        raise SdbError("sdb200 op got tensors on %s while the current CUDA device is cuda:%d; wrap the call in "
                       "`with torch.cuda.device(tensor.device):`" % (dev, torch.cuda.current_device()))
