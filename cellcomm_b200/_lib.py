"""ctypes binding of libcellcomm_b200.so (the C ABI declared in include/cellcomm_b200.h).

There is no CPU fallback: if the shared library cannot be found/built, `load()` raises.
"""
import ctypes as C
import os

from . import build as _build

_LIB = None

c_i32, c_i64, c_u32, c_u64, c_f32 = C.c_int32, C.c_int64, C.c_uint32, C.c_uint64, C.c_float
vp = C.c_void_p


class GemmDesc(C.Structure):
    """cc_gemm_desc"""
    _fields_ = [
        ("M", c_i32), ("N", c_i32),
        ("a_mn_major", c_i32), ("b_mn_major", c_i32),
        ("nseg", c_i32),
        ("a", vp * 4), ("lda", c_i64 * 4),
        ("b", vp * 4), ("ldb", c_i64 * 4),
        ("k", c_i32 * 4),
        ("alpha", c_f32),
        ("bias", vp), ("act", c_i32),
        ("dact_y", vp), ("ld_dact", c_i64), ("dact", c_i32),
        ("out16", vp), ("ld16", c_i64), ("beta16", c_i32),
        ("out32", vp), ("ld32", c_i64), ("beta32", c_i32),
        ("workspace", vp), ("workspace_elems", c_i64),
        ("force_splits", c_i32), ("force_bn", c_i32),
        ("rms_p32", vp), ("rms_ms", vp), ("rms_mom", vp), ("rms_p16", vp), ("rms_ld", c_i64),
        ("rms_lr", c_f32), ("rms_rho", c_f32), ("rms_momentum", c_f32), ("rms_eps", c_f32),
        ("route_world", c_i32), ("route_shard", c_i64), ("route_off0", c_i64),
        ("route_base", vp * 16),
        ("out16_lo", vp), ("ld16_lo", c_i64),
        ("rms_blocked", c_i32), ("rms_row0", c_i32), ("rms_p16_lo", vp),
    ]


class PeerRmspropDesc(C.Structure):
    """cc_peer_rmsprop_desc"""
    _fields_ = [
        ("world", c_i32), ("rank", c_i32),
        ("grad", vp * 16), ("p16", vp * 16),
        ("p32", vp), ("ms", vp), ("mom", vp),
        ("start", c_i64), ("count", c_i64),
        ("broadcast", c_i32),
        ("lr", c_f32), ("rho", c_f32), ("momentum", c_f32), ("eps", c_f32),
        ("ready", vp), ("epoch", c_u32),
        ("epoch_ctr", vp),
        ("p16_multicast", vp),
        ("p16lo", vp * 16), ("p16lo_multicast", vp),
        ("lo_begin", c_i64 * 2), ("lo_end", c_i64 * 2),
    ]


ENC_MAX_OPS = ENC_MAX_SLOTS = 32
ENC_DENSE, ENC_SPLIT, ENC_COPY, ENC_BN_INFER, ENC_SOFTMAX = range(5)


class EncOp(C.Structure):
    """cc_enc_op"""
    _fields_ = [
        ("kind", c_i32), ("n_in", c_i32),
        ("in_", c_i32 * 4), ("w_row", c_i32 * 4),
        ("out", c_i32), ("out2", c_i32),
        ("width", c_i32), ("act", c_i32),
        ("w16", vp), ("ldw", c_i64),
        ("bias", vp),
        ("gamma", vp), ("beta", vp), ("mean", vp), ("var", vp),
        ("eps", c_f32),
    ]


class EncodePlan(C.Structure):
    """cc_encode_plan"""
    _fields_ = [
        ("n_cols", c_i32), ("tile_rows", c_i32),
        ("n_slots", c_i32), ("n_ops", c_i32),
        ("slot_width", c_i32 * ENC_MAX_SLOTS),
        ("slot_fp32", c_i32 * ENC_MAX_SLOTS),
        ("ops", EncOp * ENC_MAX_OPS),
        ("scratch", vp), ("scratch_bytes", c_i64),
        ("workspace", vp), ("workspace_elems", c_i64),
    ]


# name -> (restype, argtypes); must list every symbol include/cellcomm_b200.h declares
SIGNATURES = {
    "cc_last_error": (C.c_char_p, []),
    "cc_version": (C.c_int, []),
    "cc_launch_count": (C.c_longlong, []),
    "cc_arch": (C.c_char_p, []),
    "cc_reload_env": (None, []),
    "cc_mtx_load_csr": (C.c_int, [C.c_char_p, C.POINTER(vp)]),
    "cc_coo_to_csr": (C.c_int, [vp, vp, vp, c_i64, C.POINTER(vp)]),
    "cc_csr_destroy": (None, [vp]),
    "cc_csr_rows": (c_i64, [vp]),
    "cc_csr_cols": (c_i64, [vp]),
    "cc_csr_nnz": (c_i64, [vp]),
    "cc_csr_rowptr": (vp, [vp]),
    "cc_csr_colidx": (vp, [vp]),
    "cc_csr_values": (vp, [vp]),
    "cc_csr_values64": (vp, [vp]),
    "cc_csr_row_ids": (vp, [vp]),
    "cc_csr_col_ids": (vp, [vp]),
    "cc_mtx_load_coo": (C.c_int, [C.c_char_p, C.POINTER(vp)]),
    "cc_coo_destroy": (None, [vp]),
    "cc_coo_nnz": (c_i64, [vp]),
    "cc_coo_gene": (vp, [vp]),
    "cc_coo_barcode": (vp, [vp]),
    "cc_coo_value": (vp, [vp]),
    "cc_coo_build_csr": (C.c_int, [vp, C.POINTER(vp)]),
    "cc_mtx_write": (C.c_int, [C.c_char_p, c_i64, c_i64, c_i64, vp, vp, vp, vp, vp]),
    "cc_encode_scratch_bytes": (c_i64, [C.POINTER(EncodePlan)]),
    "cc_encode_stream": (C.c_int, [vp, vp, vp, c_i64, c_i64, C.POINTER(EncodePlan), vp, c_i64, vp]),
    "cc_gather_rows": (C.c_int, [vp, vp, vp, vp, c_i64, c_i64, c_i64, vp, c_i64, vp, c_i64, vp]),
    "cc_gemm": (C.c_int, [C.POINTER(GemmDesc), vp]),
    "cc_gemm_workspace_elems": (c_i64, [c_i32, c_i32]),
    "cc_dense_fwd": (C.c_int, [c_i32, c_i32, c_i32, C.POINTER(vp), C.POINTER(c_i64),
                               C.POINTER(c_i32), C.POINTER(vp), C.POINTER(c_i64), vp, c_i32,
                               vp, c_i64, vp, c_i64, vp, c_i64, vp]),
    "cc_dense_dgrad": (C.c_int, [c_i32, c_i32, c_i32, C.POINTER(vp), C.POINTER(c_i64),
                                 C.POINTER(c_i32), C.POINTER(vp), C.POINTER(c_i64), vp, c_i64,
                                 c_i32, c_f32, vp, c_i64, c_i32, vp, c_i64, vp]),
    "cc_dense_wgrad": (C.c_int, [c_i32, c_i32, c_i32, vp, c_i64, vp, c_i64, vp, c_i64, c_i32, vp]),
    "cc_reduce_ws_floats": (c_i64, [c_i64, c_i64]),
    "cc_colsum": (C.c_int, [vp, c_i64, c_i64, c_i64, vp, c_i32, c_i32, vp]),
    "cc_colsum_ws": (C.c_int, [vp, c_i64, c_i64, c_i64, vp, c_i32, c_i32, vp, c_i64, vp]),
    "cc_bias_grad": (C.c_int, [vp, c_i64, vp, c_i64, c_i64, c_i64, c_i32, vp, c_i32, vp, c_i64, vp,
                               c_i64, c_i32, vp]),
    "cc_bias_grad_ws": (C.c_int, [vp, c_i64, vp, c_i64, c_i64, c_i64, c_i32, vp, c_i32, vp, c_i64,
                                  vp, c_i64, c_i32, vp, c_i64, vp]),
    "cc_split_bf16": (C.c_int, [vp, c_i64, vp, c_i64, vp, c_i64, c_i64, c_i64, c_i32, vp]),
    "cc_dropout": (C.c_int, [vp, c_i64, vp, c_i64, c_i64, c_i64, c_f32, vp, c_i64, c_u64, vp,
                             c_u32, c_i32, vp]),
    "cc_dropout_mask": (C.c_int, [vp, c_i64, c_i64, c_i64, c_f32, c_u64, vp, c_u32, vp]),
    "cc_uniform": (C.c_int, [vp, vp, c_i64, c_i64, c_i64, c_u64, vp, c_u32, vp]),
    "cc_counter_add": (C.c_int, [vp, c_u64, vp]),
    "cc_act_bwd": (C.c_int, [vp, c_i64, vp, c_i64, vp, c_i64, c_i64, c_i64, c_i32, c_i32, vp]),
    "cc_copy2d": (C.c_int, [vp, c_i64, vp, c_i64, c_i64, c_i64, c_i32, c_f32, c_i32, vp]),
    "cc_bn_stats": (C.c_int, [vp, c_i64, c_i64, c_i64, vp, c_i32, vp]),
    "cc_bn_stats_ws": (C.c_int, [vp, c_i64, c_i64, c_i64, vp, c_i32, vp, c_i64, vp]),
    "cc_bn_train_apply": (C.c_int, [vp, c_i64, vp, c_i64, c_i64, c_i64, vp, c_i64, vp, vp, c_f32,
                                    c_f32, vp, vp, vp, vp, c_i32, vp]),
    "cc_bn_infer": (C.c_int, [vp, c_i64, vp, c_i64, c_i64, c_i64, vp, vp, vp, vp, c_f32, c_i32,
                              vp]),
    "cc_bn_bwd_stats": (C.c_int, [vp, c_i64, vp, c_i64, c_i64, c_i64, vp, vp, vp, c_i32, vp]),
    "cc_bn_bwd_stats_ws": (C.c_int, [vp, c_i64, vp, c_i64, c_i64, c_i64, vp, vp, vp, c_i32, vp,
                                     c_i64, vp]),
    "cc_bn_bwd_apply": (C.c_int, [vp, c_i64, vp, c_i64, vp, c_i64, c_i64, c_i64, vp, vp, vp, vp,
                                  c_i64, vp, vp, c_i32, vp]),
    "cc_bn_infer_bwd": (C.c_int, [vp, c_i64, vp, c_i64, c_i64, c_i64, vp, vp, c_f32, c_i32, vp]),
    "cc_softmax_fwd": (C.c_int, [vp, c_i64, vp, c_i64, vp, c_i64, c_i64, c_i64, c_i32, vp]),
    "cc_softmax_bwd": (C.c_int, [vp, c_i64, vp, c_i64, vp, c_i64, c_i64, c_i64, c_i32, vp]),
    "cc_bce_fwd_bwd": (C.c_int, [vp, c_i64, c_i64, c_i32, c_f32, c_i64, vp, vp, c_i64, c_i32, vp]),
    "cc_mse_fwd_bwd": (C.c_int, [vp, c_i64, vp, c_i64, c_i64, c_i64, c_i64, vp, vp, c_i64, c_i32,
                                 vp]),
    "cc_mse_fwd_bwd_ws": (C.c_int, [vp, c_i64, vp, c_i64, c_i64, c_i64, c_i64, vp, vp, c_i64,
                                    c_i32, vp, c_i64, vp]),
    "cc_round_half_even": (C.c_int, [vp, c_i64, vp, c_i64, vp, c_i64, c_i64, c_i64, c_i32, vp]),
    "cc_round_csr_count": (C.c_int, [vp, c_i64, c_i64, c_i64, vp, vp]),
    "cc_round_csr_fill": (C.c_int, [vp, c_i64, c_i64, c_i64, vp, vp, vp, vp]),
    "cc_recon_sqerr": (C.c_int, [vp, c_i64, c_i64, c_i64, vp, vp, vp, c_i64, c_f32, vp, vp]),
    "cc_col_moments": (C.c_int, [vp, c_i64, c_i64, c_i64, c_i32, vp, vp, vp, vp, c_i64, vp]),
    "cc_col_moments_ws_bytes": (c_i64, [c_i64, c_i64]),
    "cc_log1p_features": (C.c_int, [vp, c_i64, c_i64, c_i64, c_i32, vp, c_i64, vp, vp, vp]),
    "cc_mmd_sums": (C.c_int, [vp, c_i64, c_i64, vp, c_i32, vp, c_i64, vp, vp, c_i64, vp]),
    "cc_mmd_sums_ws_bytes": (c_i64, [c_i64, c_i32, c_i64]),
    "cc_argmax_onehot": (C.c_int, [vp, c_i64, vp, c_i64, vp, c_i64, c_i64, c_i64, vp]),
    "cc_rmsprop_step": (C.c_int, [vp, vp, vp, vp, vp, c_i64, c_i64, c_i64, c_f32, c_f32, c_f32,
                                  c_f32, c_f32, vp]),
    "cc_bias_act": (C.c_int, [vp, c_i32, vp, c_i64, vp, c_i64, c_i64, c_i64, vp]),
    "cc_fill_f32": (C.c_int, [vp, c_f32, c_i64, vp]),
    "cc_peer_rmsprop": (C.c_int, [C.POINTER(PeerRmspropDesc), vp]),
    "cc_peer_signal": (C.c_int, [C.POINTER(vp), c_i32, c_u32, vp, vp]),
    "cc_peer_wait": (C.c_int, [vp, c_i32, c_u32, vp, c_i32, vp]),
    "cc_peer_allreduce": (C.c_int, [vp, c_i32, c_i32, c_i32, C.POINTER(vp), C.POINTER(vp), c_i64,
                                    c_u32, vp, vp]),
}


def lib_path():
    return _build.LIB


def load():
    """Load (building first when stale and nvcc is present) the C-ABI library.  Raises if absent."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = lib_path()
    if os.environ.get("CELLCOMM_B200_NO_BUILD") != "1":
        try:
            if _build.is_stale():
                _build.build_library()
        except Exception as exc:  # no nvcc on this box: fall through to the prebuilt file
            if not os.path.exists(path):
                raise RuntimeError(
                    f"libcellcomm_b200.so is missing and could not be built: {exc}") from exc
    if not os.path.exists(path):
        raise RuntimeError(f"libcellcomm_b200.so not found at {path}; run "
                           f"`python -m cellcomm_b200.build` (there is no CPU fallback)")
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the .so lacks a declared symbol
        fn.restype = res
        fn.argtypes = args
    _LIB = lib
    return lib


class CCError(RuntimeError):
    pass


def check(rc):
    if rc != 0:
        raise CCError(load().cc_last_error().decode("utf-8", "replace"))
