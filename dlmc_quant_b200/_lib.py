"""ctypes binding of libdlmcq.so (the C ABI declared in include/dlmcq.h).

There is deliberately NO fallback: if the CUDA library is missing or fails to load, every
product entry point raises.  A CPU path would void the parity claims of this repo."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libdlmcq.so")

F32, BF16 = 0, 1
FORM_A1, FORM_AFFINE, FORM_ZP, FORM_SYM = 0, 1, 2, 3
STATS_PER_CHANNEL = 4
DIV_IEEE, DIV_CUDA_EAGER = 0, 1
SWEEP_CANDIDATES = 80
ROOTQ_STATE_FLOATS = 8
QGEMM_I8, QGEMM_E4M3 = 0, 1


class Layout(C.Structure):
    _fields_ = [("outer", C.c_int64), ("channels", C.c_int64), ("inner", C.c_int64), ("dtype", C.c_int32)]


class QParams(C.Structure):
    _fields_ = [("form", C.c_int32), ("lo", C.c_int32), ("hi", C.c_int32), ("g", C.c_float),
                ("scale", C.c_void_p), ("offset", C.c_void_p)]


class GroupItem(C.Structure):
    _fields_ = [("x", C.c_void_p), ("y", C.c_void_p), ("dy", C.c_void_p), ("scale", C.c_void_p),
                ("offset", C.c_void_p), ("dscale", C.c_void_p), ("channels", C.c_int64), ("inner", C.c_int64),
                ("form", C.c_int32), ("lo", C.c_int32), ("hi", C.c_int32), ("g", C.c_float)]


class FoldItem(C.Structure):
    _fields_ = ([(n, C.c_void_p) for n in ("w", "bias", "gamma", "beta", "mean", "var", "w1", "gamma1", "beta1", "mean1",
                                           "var1", "gamma_id", "beta_id", "mean_id", "var_id", "w_out", "bias_out",
                                           "stats")] +
                [("channels", C.c_int64), ("inner", C.c_int64), ("cin_g", C.c_int32), ("ksize", C.c_int32),
                 ("mode", C.c_int32), ("eps", C.c_float), ("eps1", C.c_float), ("eps_id", C.c_float)])


FOLD_MERGE_BN, FOLD_REPVGG = 0, 1


class RootqPrep(C.Structure):
    _fields_ = [("param_a", C.c_void_p), ("param_b", C.c_void_p), ("alpha", C.c_void_p), ("run_a", C.c_void_p),
                ("run_b", C.c_void_p), ("state", C.c_void_p), ("momentum", C.c_double), ("g", C.c_double),
                ("lo", C.c_int32), ("hi", C.c_int32), ("training", C.c_int32), ("is_weight", C.c_int32)]


class RootqItem(C.Structure):
    _fields_ = [("x", C.c_void_p), ("y", C.c_void_p), ("dy", C.c_void_p), ("state", C.c_void_p),
                ("grads", C.c_void_p), ("numel", C.c_int64)]


ROOTQ_UNIT = 2048


class FinalizeItem(C.Structure):
    _fields_ = [("partials", C.c_void_p), ("dscale", C.c_void_p)]


class SweepItem(C.Structure):
    _fields_ = [("x", C.c_void_p), ("scale", C.c_void_p), ("offset", C.c_void_p), ("channels", C.c_int64),
                ("inner", C.c_int64), ("n_bits", C.c_int32), ("is_signed", C.c_int32), ("wpr", C.c_int32),
                ("row_floats", C.c_int32), ("staged", C.c_int32), ("pad", C.c_int32), ("smem_bytes", C.c_int64),
                ("ctas", C.c_int64)]


class BnqDesc(C.Structure):
    _fields_ = [("rows", C.c_int64), ("channels", C.c_int64), ("dtype", C.c_int32), ("flags", C.c_int32),
                ("eps", C.c_float), ("momentum", C.c_float)]


BNQ_TRAINING, BNQ_RELU, BNQ_RESIDUAL = 1, 2, 4


class ConvGeom(C.Structure):
    _fields_ = ([(n, C.c_int64) for n in ("batch", "h", "w", "cin", "n")] +
                [(n, C.c_int32) for n in ("kh", "kw", "stride_h", "stride_w", "pad_h", "pad_w", "dil_h", "dil_w",
                                          "groups")])


class BnqTail(C.Structure):
    _fields_ = [("gamma", C.c_void_p), ("beta", C.c_void_p), ("running_mean", C.c_void_p), ("running_var", C.c_void_p),
                ("eps", C.c_float), ("relu", C.c_int32), ("inter_dtype", C.c_int32), ("qp", C.POINTER(QParams)),
                ("encoding", C.c_int32)]


class DlmcqError(RuntimeError):
    pass


_lib = None

_P, _I, _L, _F, _D, _Z = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_double, C.c_size_t
_LP, _QP = C.POINTER(Layout), C.POINTER(QParams)

# name -> (restype, argtypes); mirrors include/dlmcq.h one to one
SIGNATURES = {
    "dlmcq_version": (_I, []),
    "dlmcq_selftest_fastdiv": (_I, [C.c_uint64, _I, _I, _I, _P, _P]),
    "dlmcq_status_string": (C.c_char_p, [_I]),
    "dlmcq_last_cuda_error": (C.c_char_p, []),
    "dlmcq_workspace_bytes": (_Z, [_LP]),
    "dlmcq_fq_forward": (_I, [_P, _P, _P, _LP, _QP, _P]),
    "dlmcq_fq_backward": (_I, [_P, _P, _P, _P, _P, _LP, _QP, _P, _Z, _P]),
    "dlmcq_fq_partials_floats": (_Z, []),
    "dlmcq_fq_backward_partials": (_I, [_P, _P, _P, _LP, _QP, _P, _P]),
    "dlmcq_fq_finalize_many": (_I, [_P, _I, _P]),
    "dlmcq_capture_overlap_count": (_I, []),
    "dlmcq_dequantize": (_I, [_P, _P, _LP, _P, _P, _P]),
    "dlmcq_ste_value": (_I, [_P, _P, _L, _I, _I, _P]),
    "dlmcq_grad_scale_value": (_I, [_P, _P, _L, _F, _P]),
    "dlmcq_export_codes": (_I, [_P, _P, _LP, _QP, _I, _P]),
    "dlmcq_import_codes": (_I, [_P, _P, _LP, _QP, _I, _P]),
    "dlmcq_adaround_forward": (_I, [_P, _P, _P, _LP, _P, _I, _I, _I, _P]),
    "dlmcq_adaround_backward": (_I, [_P, _P, _P, _P, _P, _LP, _P, _I, _I, _P, _Z, _P]),
    "dlmcq_adaround_init_alpha": (_I, [_P, _P, _LP, _P, _P]),
    "dlmcq_rootq_act_prepare": (_I, [_P, _P, _D, _D, _I, _I, _I, _P, _P]),
    "dlmcq_rootq_act_forward": (_I, [_P, _P, _L, _I, _P, _P]),
    "dlmcq_rootq_act_backward": (_I, [_P, _P, _P, _P, _L, _I, _P, _P, _Z, _P]),
    "dlmcq_rootq_wt_prepare": (_I, [_P, _P, _P, _P, _P, _D, _D, _I, _I, _I, _P, _P]),
    "dlmcq_rootq_wt_forward": (_I, [_P, _P, _L, _I, _P, _P]),
    "dlmcq_rootq_wt_backward": (_I, [_P, _P, _P, _P, _L, _I, _P, _P, _Z, _P]),
    "dlmcq_rootq_prepare_many": (_I, [_P, _I, _P]),
    "dlmcq_rootq_wt_forward_grouped": (_I, [_P, _P, _I, _L, _I, _P]),
    "dlmcq_rootq_wt_backward_grouped": (_I, [_P, _P, _I, _L, _I, _P, _P]),
    "dlmcq_rootq_act_forward_grouped": (_I, [_P, _P, _I, _L, _I, _P]),
    "dlmcq_rootq_act_backward_grouped": (_I, [_P, _P, _I, _L, _I, _P, _P]),
    "dlmcq_obs_stats": (_I, [_P, _P, _LP, _I, _P, _Z, _P]),
    "dlmcq_obs_minmax_finalize": (_I, [_P, _P, _P, _L, _I, _I, _I, _P]),
    "dlmcq_obs_minmax_finalize_mode": (_I, [_P, _P, _P, _L, _I, _I, _I, _I, _P]),
    "dlmcq_obs_absmean_finalize": (_I, [_P, _P, _L, _D, _D, _D, _I, _P]),
    "dlmcq_obs_kth_state_bytes": (_Z, []),
    "dlmcq_obs_kth_begin": (_I, [_P, _L, _L, _P]),
    "dlmcq_obs_kth_hist": (_I, [_P, _L, _I, _I, _I, _P, _P]),
    "dlmcq_obs_kth_select": (_I, [_I, _P, _P]),
    "dlmcq_obs_kth_values": (_I, [_P, _P, _P]),
    "dlmcq_obs_kth_fast_workspace_bytes": (_Z, [_L]),
    "dlmcq_obs_kth_fast": (_I, [_P, _L, _I, _I, _L, _L, _P, _P, _P, _Z, _P]),
    "dlmcq_obs_kth_auto": (_I, [_P, _L, _I, _I, _L, _L, _P, _P, _P, _P, _Z, _P]),
    "dlmcq_obs_sweep_tensor_sse": (_I, [_P, _L, _I, _P, _I, _I, _P, _P, _Z, _P]),
    "dlmcq_obs_sweep_tensor_finalize": (_I, [_P, _P, _D, _I, _I, _P, _P, _P, _P]),
    "dlmcq_obs_sweep_channel": (_I, [_P, _L, _L, _I, _I, _I, _P, _P, _P]),
    "dlmcq_obs_sweep_channel_geom": (_I, [_P, _L, _L, _I, _I, _I, _L, _P, _P, _P]),
    "dlmcq_obs_sweep_channel_plan": (_I, [C.POINTER(SweepItem), _L]),
    "dlmcq_obs_sweep_channel_grouped": (_I, [_P, _P, _I, _L, _I, _L, _P]),
    "dlmcq_obs_l2norm_step": (_I, [_P, _L, _L, _I, _P, _P, _I, _I, _P, _P, _P, _P, _Z, _P]),
    "dlmcq_obs_l2norm_resident": (_I, [_P, _L, _L, _I, _P, _P, _I, _I, _I, _P, _P, _P, _P, _Z, _P]),
    "dlmcq_fq_forward_grouped": (_I, [_P, _P, _I, _L, _I, _P]),
    "dlmcq_fq_backward_grouped": (_I, [_P, _P, _P, _I, _L, _L, _I, _P, _P]),
    "dlmcq_fold_grouped": (_I, [_P, _P, _I, _L, _P]),
    "dlmcq_bnq_workspace_bytes": (_Z, [C.POINTER(BnqDesc)]),
    "dlmcq_bnq_forward": (_I, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, C.POINTER(BnqDesc), _QP, _P, _Z, _P]),
    "dlmcq_bnq_forward_codes": (_I, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, C.POINTER(BnqDesc), _QP, _I, _P, _Z,
                                     _P]),
    "dlmcq_bnq_backward": (_I, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, C.POINTER(BnqDesc), _QP, _P, _Z,
                                _P]),
    "dlmcq_host_ctx_create": (_I, [C.POINTER(C.c_void_p), _L]),
    "dlmcq_host_ctx_destroy": (_I, [_P]),
    "dlmcq_host_ctx_synchronize": (_I, [_P]),
    "dlmcq_host_ctx_fq_forward_backward": (_I, [_P, _P, _P, _P, _P, _P, _L, _I, _I, _I, _I, _F, _F, _F]),
    "dlmcq_host_ctx_fq_codes": (_I, [_P, _P, _P, _P, _P, _P, _L, _I, _I, _I, _I, _F, _F, _F, _I]),
    "dlmcq_codes_forward": (_I, [_P, _P, _LP, _QP, _I, _P]),
    "dlmcq_qgemm_prepare": (_I, [_P, _L, _L, _I, _QP, _QP, _L, _P, _P, _P, _P]),
    "dlmcq_qgemm": (_I, [_P, _P, _P, _P, _P, _L, _L, _L, _I, _I, _I, _I, _P]),
    "dlmcq_qconv_prepare": (_I, [_P, C.POINTER(ConvGeom), _I, _QP, _QP, _L, _P, _P, _P, _P]),
    "dlmcq_qconv": (_I, [_P, _P, _P, _P, _P, C.POINTER(ConvGeom), _I, _I, _I, _I, _P]),
    "dlmcq_qgemm_codes": (_I, [_P, _P, _P, _P, _P, _L, _L, _L, _I, _I, C.POINTER(BnqTail), _P]),
    "dlmcq_qconv_codes": (_I, [_P, _P, _P, _P, _P, C.POINTER(ConvGeom), _I, _I, C.POINTER(BnqTail), _P]),
}


def lib():
    """Load (once) and return the ctypes handle.  Raises if the library is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise DlmcqError(
            f"{LIB_PATH} not found: build it with `python -m dlmc_quant_b200.build` "
            "(nvcc, sm_100a).  There is no CPU fallback for this path.")
    h = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(h, name)          # AttributeError here = header and library disagree
        fn.restype, fn.argtypes = res, args
    if h.dlmcq_version() != 100:
        raise DlmcqError("libdlmcq.so version mismatch")
    _lib = h
    return h


def check(status):
    if status != 0:
        h = lib()
        msg = h.dlmcq_status_string(status).decode()
        if status == -4:
            msg += ": " + h.dlmcq_last_cuda_error().decode()
        raise DlmcqError(f"libdlmcq: {msg} (status {status})")
