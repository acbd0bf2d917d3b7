"""ctypes binding of librvcb200.so (include/rvcb200.h).  Fails loudly: there is no CPU fallback."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("RVCB200_LIB") or os.path.join(HERE, "librvcb200.so")   # env override: kernel A/B experiments

MAX_UPS, MAX_RESK, MAX_DIL = 8, 4, 4
PREC = {"fp32": 0, "fp16": 1, "bf16": 2}
STATUS = {0: "ok", 1: "bad argument / unsupported configuration", 2: "missing tensor", 3: "workspace too small",
          4: "CUDA error", 5: "no CUDA device (no CPU fallback exists)"}


class RvcConfig(C.Structure):
    _fields_ = [
        ("feat_dim", C.c_int32), ("inter_channels", C.c_int32), ("hidden_channels", C.c_int32),
        ("filter_channels", C.c_int32), ("n_heads", C.c_int32), ("n_layers", C.c_int32),
        ("enc_kernel", C.c_int32), ("window_size", C.c_int32), ("flow_kernel", C.c_int32),
        ("flow_wn_layers", C.c_int32), ("n_flows", C.c_int32), ("resblock_kind", C.c_int32),
        ("n_res_kernels", C.c_int32), ("res_kernels", C.c_int32 * MAX_RESK), ("n_res_dils", C.c_int32 * MAX_RESK),
        ("res_dils", (C.c_int32 * MAX_DIL) * MAX_RESK), ("n_ups", C.c_int32), ("up_rates", C.c_int32 * MAX_UPS),
        ("up_kernels", C.c_int32 * MAX_UPS), ("up_init_channels", C.c_int32), ("gin_channels", C.c_int32),
        ("n_speakers", C.c_int32), ("sr", C.c_int32), ("no_f0", C.c_int32),
    ]


class RvcTap(C.Structure):
    _fields_ = [("name", C.c_char_p), ("dst", C.c_void_p), ("bytes", C.c_size_t)]


class ConvDesc(C.Structure):
    _fields_ = [
        ("x", C.c_void_p), ("x_bstride", C.c_int64), ("ldx", C.c_int32), ("L_in", C.c_int32),
        ("in_len", C.c_void_p), ("in_slope", C.c_float),
        ("w", C.c_void_p), ("bias", C.c_void_p), ("Cin", C.c_int32), ("Cout", C.c_int32), ("ntaps", C.c_int32),
        ("dil", C.c_int32), ("G", C.c_int32), ("g_off", C.c_int32 * 16),
        ("Lj", C.c_int32), ("out_stride", C.c_int32),
        ("y", C.c_void_p), ("y_bstride", C.c_int64), ("ldy", C.c_int32),
        ("cond", C.c_void_p), ("cond_bstride", C.c_int32),
        ("gather", C.c_void_p), ("gidx", C.c_void_p), ("gidx_bstride", C.c_int64),
        ("alpha", C.c_float), ("gate", C.c_int32),
        ("mask_pre", C.c_int32), ("mask_post", C.c_int32), ("out_len", C.c_void_p),
        ("res", C.c_void_p), ("res_bstride", C.c_int64), ("ldr", C.c_int32), ("res_mode", C.c_int32),
        ("out_slope", C.c_float), ("relu", C.c_int32),
        ("accum", C.c_int32), ("div", C.c_float),
    ]


class TcConvDesc(C.Structure):
    _fields_ = [
        ("x16", C.c_void_p), ("L_in", C.c_int32), ("padf", C.c_int32),
        ("w16", C.c_void_p), ("bias", C.c_void_p),
        ("Cin", C.c_int32), ("ntaps", C.c_int32), ("dil", C.c_int32), ("G", C.c_int32),
        ("g_off", C.c_int32 * 16),
        ("N", C.c_int32), ("Cout_total", C.c_int32), ("tmem_cols", C.c_int32),
        ("Lj", C.c_int32), ("out_stride", C.c_int32), ("Lp_out", C.c_int32),
        ("y32", C.c_void_p), ("y16", C.c_void_p), ("res32", C.c_void_p),
        ("cond", C.c_void_p), ("cond_bstride", C.c_int32),
        ("accum", C.c_int32), ("div", C.c_float), ("out_slope", C.c_float),
        ("in_bf16", C.c_int32), ("out_bf16", C.c_int32), ("a_mode", C.c_int32),
        ("batch", C.c_int32), ("na_stages", C.c_int32), ("nb_stages", C.c_int32), ("b_stationary", C.c_int32),
        ("generic", C.c_int32), ("ldx16", C.c_int32), ("f32_cl", C.c_int32),
        ("ldy32", C.c_int32), ("ldr32", C.c_int32), ("ldy16", C.c_int32),
        ("gather", C.c_void_p), ("gidx", C.c_void_p), ("gidx_bstride", C.c_int64),
        ("alpha", C.c_float), ("pre_slope", C.c_float), ("relu", C.c_int32), ("gate", C.c_int32),
        ("res_mode", C.c_int32), ("mask_pre", C.c_int32), ("mask_post", C.c_int32), ("mask16", C.c_int32),
        ("out_len", C.c_void_p), ("dbg_alt", C.c_int32),
        ("res16", C.c_void_p), ("res_neg_scale", C.c_float), ("a_fp16", C.c_int32), ("acc_f16", C.c_int32),
        ("tma_out", C.c_int32),
        ("tanh_out", C.c_void_p), ("acc_nostore", C.c_int32),
        ("inj_har", C.c_void_p), ("inj_w", C.c_void_p), ("inj_b", C.c_void_p),
        ("inj_k", C.c_int32), ("inj_s", C.c_int32), ("inj_pad", C.c_int32), ("inj_cn", C.c_int32), ("inj_Lhar", C.c_int64),
        ("gelu", C.c_int32), ("tap_w", C.c_int32), ("dil2", C.c_int32), ("pad_period", C.c_int32), ("pad_valid", C.c_int32),
        ("b_group", C.c_int32), ("a_nt_stride", C.c_int32), ("reserved1", C.c_int32),
    ]


# every symbol include/rvcb200.h declares: (restype, argtypes)
SYMBOLS = {
    "rvcb200_abi_version": (C.c_int32, []),
    "rvcb200_sizeof": (C.c_int64, [C.c_int32]),
    "rvcb200_create": (C.c_int, [C.POINTER(RvcConfig), C.POINTER(C.c_void_p)]),
    "rvcb200_destroy": (None, [C.c_void_p]),
    "rvcb200_set_tensor": (C.c_int, [C.c_void_p, C.c_char_p, C.c_void_p, C.c_int64, C.c_int32]),
    "rvcb200_set_scalar": (C.c_int, [C.c_void_p, C.c_char_p, C.c_float]),
    "rvcb200_finalize": (C.c_int, [C.c_void_p]),
    "rvcb200_workspace_bytes": (C.c_int64, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32]),
    "rvcb200_infer": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                C.c_void_p, C.c_int64, C.c_int32, C.POINTER(RvcTap), C.c_int32, C.c_void_p]),
    "rvcb200_infer_tail": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p]),
    "rvcb200_profile_enable": (C.c_int, [C.c_void_p, C.c_int32]),
    "rvcb200_profile_collect": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int64)]),
    "rvcb200_profile_launches": (C.c_int64, [C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_float),
                                           C.c_int64]),
    "rvcb200_last_launch_count": (C.c_int64, [C.c_void_p]),
    "rvcb200_last_error": (C.c_char_p, [C.c_void_p]),
    "rvcb200_op_conv_f32": (C.c_int, [C.POINTER(ConvDesc), C.c_int32, C.c_void_p]),
    "rvcb200_op_conv_tc": (C.c_int, [C.POINTER(TcConvDesc), C.c_int32, C.c_void_p]),
    "rvcb200_debug_trace_conv_tc": (C.c_int, [C.c_void_p]),
    "rvcb200_op_rmvpe_logmel": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_float,
                                          C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "rvcb200_op_rmvpe_pool": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                        C.c_void_p]),
    "rvcb200_op_rmvpe_shuffle": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                           C.c_int32, C.c_void_p]),
    "rvcb200_op_rmvpe_gru_pack": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p]),
    "rvcb200_op_rmvpe_gru": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "rvcb200_op_rmvpe_decode": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_float,
                                          C.c_void_p]),
    "rvcb200_op_rmvpe_mel_to_img": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_float, C.c_float, C.c_int32, C.c_int32,
                                              C.c_void_p]),
    "rvcb200_op_crepe_frames": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]),
    "rvcb200_op_crepe_bn_pool": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_int32,
                                           C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "rvcb200_op_crepe_decode": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                          C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_double, C.c_void_p, C.c_void_p,
                                          C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "rvcb200_op_rbconv_tc": (C.c_int, [C.POINTER(TcConvDesc), C.c_int32, C.c_void_p]),
    "rvcb200_op_rbpair_tc": (C.c_int, [C.POINTER(TcConvDesc), C.POINTER(TcConvDesc), C.c_int32, C.c_void_p]),
    "rvcb200_op_sine_scratch_bytes": (C.c_int64, [C.c_int32, C.c_int32, C.c_int32]),
    "rvcb200_op_sine_source": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                         C.c_int32, C.c_float, C.c_float, C.c_void_p, C.c_void_p]),
    "rvcb200_op_attention_f32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                           C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "rvcb200_op_attention_tc": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                          C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "rvcb200_op_layernorm": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32,
                                       C.c_float, C.c_void_p]),
    "rvcb200_op_prepare_feats": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                           C.c_int32, C.c_float, C.c_int32, C.c_void_p]),
    "rvcb200_op_absmax": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int32, C.c_void_p]),
    "rvcb200_op_to_int16": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "rvcb200_op_rms_halfblock": (C.c_int, [C.c_void_p, C.c_int32, C.c_int64, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p]),
    "rvcb200_op_rms_fold": (C.c_int, [C.c_void_p, C.c_int32, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p]),
    "rvcb200_op_rms_gain": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64,
                                      C.c_double, C.c_void_p]),
    "rvcb200_op_ivf_scratch_bytes": (C.c_int64, [C.c_int32, C.c_int32]),
    "rvcb200_op_ivf_assign": (C.c_int, [C.c_void_p, C.c_int32, C.c_int64, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32,
                                        C.c_void_p, C.c_void_p]),
    "rvcb200_op_ivf_scan": (C.c_int, [C.c_void_p, C.c_int32, C.c_int64, C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p,
                                      C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "rvcb200_op_index_blend": (C.c_int, [C.c_void_p, C.c_int32, C.c_int64, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.c_void_p, C.c_int64, C.c_int32, C.c_double, C.c_void_p, C.c_void_p]),
    "rvcb200_op_resample_poly": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int64, C.c_void_p, C.c_int64,
                                           C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int64,
                                           C.c_int64, C.c_void_p, C.c_void_p]),
    "rvcb200_op_hubert_conv0": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                          C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_float, C.c_int64, C.c_void_p]),
    "rvcb200_op_layernorm16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32,
                                         C.c_float, C.c_void_p]),
    "rvcb200_op_quiet_point": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "rvcb200_host_quiet_point": (C.c_int64, [C.c_void_p, C.c_int64, C.c_int64, C.c_int32, C.c_int32]),
    "rvcb200_host_filtfilt_pad": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int64,
                                            C.c_void_p, C.c_void_p]),
}

_lib = None


def load() -> C.CDLL:
    """Load the extension; raise (never fall back) if it is missing or stale."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -m comfy_rvc_b200.build` "
            "(or __graft_entry__.build()).  comfy_rvc_b200 has no CPU or PyTorch fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError if the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    if lib.rvcb200_abi_version() != 1:
        raise RuntimeError("librvcb200.so ABI version mismatch; rebuild")
    for which, mirror in enumerate((RvcConfig, RvcTap, ConvDesc, TcConvDesc)):
        if lib.rvcb200_sizeof(which) != C.sizeof(mirror):
            raise RuntimeError(f"librvcb200.so is stale: sizeof({mirror.__name__}) is {lib.rvcb200_sizeof(which)} in the library, "
                               f"{C.sizeof(mirror)} in _lib.py; rebuild with `python -m comfy_rvc_b200.build --force`")
    _lib = lib
    return lib


def check(status: int, ctx=None, what: str = ""):
    if status == 0:
        return
    msg = STATUS.get(status, f"status {status}")
    detail = ""
    if ctx:
        detail = load().rvcb200_last_error(ctx).decode(errors="replace")
    raise RuntimeError(f"rvcb200 {what}: {msg}{' — ' + detail if detail else ''}")
