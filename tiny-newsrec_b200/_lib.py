"""ctypes binding of libtinyrec.so (the C ABI declared in include/tinyrec.h).

There is deliberately no fallback: if the shared object is missing or a call
fails, a ``TinyRecError`` is raised.
"""
import ctypes
import os
from ctypes import POINTER, Structure, c_char_p, c_float, c_int, c_int64, c_uint, c_void_p

PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(PKG, "libtinyrec.so")

ACT_NONE, ACT_GELU, ACT_TANH, ACT_DGELU, ACT_GELU_DAUX, ACT_MULAUX = 0, 1, 2, 3, 4, 5
BF16, F32 = 0, 1
SPLIT_ACT, SPLIT_WEIGHT = 0, 1      # tnr_split_bf16x3 layouts: [hi|lo|hi], [hi|hi|lo]


class TinyRecError(RuntimeError):
    pass


class Dropout(Structure):
    """tnr_dropout: DEVICE pointer to the uint64 seed, per-tensor site id, drop probability."""
    _fields_ = [("seed", c_void_p), ("site", c_uint), ("p", c_float)]


class UserEncoderIO(Structure):
    """tnr_user_encoder_io"""
    _fields_ = [(n, c_void_p) for n in ("vecs", "pad_doc", "W1", "b1", "w2", "b2", "user", "a_out", "e_out")]


class GemmArgs(Structure):
    _fields_ = [("M", c_int), ("N", c_int), ("K", c_int),
                ("A", c_void_p), ("lda", c_int), ("a_mn_major", c_int),
                ("B", c_void_p), ("ldb", c_int), ("b_mn_major", c_int),
                ("C", c_void_p), ("ldc", c_int), ("c_dtype", c_int),
                ("bias", c_void_p),
                ("residual", c_void_p), ("ldr", c_int),
                ("act", c_int),
                ("aux", c_void_p), ("ldaux", c_int),
                ("split_k", c_int),
                ("accumulate", c_int),
                ("drop", POINTER(Dropout)),
                ("colsum", c_void_p)]


P = c_void_p
_SIGNATURES = {
    "tnr_abi_version": ([], c_int),
    "tnr_device_check": ([POINTER(c_int)], c_int),
    "tnr_set_sm_reserve": ([c_int], c_int),
    "tnr_host_copy_mt": ([P, P, c_int64, c_int], c_int),
    "tnr_allreduce_p2p_flag_words": ([], c_int64),
    "tnr_allreduce_p2p": ([P, P, P, c_int, c_int, c_int64, c_int64, c_int, P], c_int),
    "tnr_gemm_bf16": ([POINTER(GemmArgs), P], c_int),
    "tnr_dropout_mask": ([POINTER(Dropout), c_int64, P, P], c_int),
    "tnr_embed_ln_fwd": ([P, c_int, c_int, c_int, c_int, P, c_int, P, P, P, P, c_float, c_int, P, POINTER(Dropout), P], c_int),
    "tnr_embed_ln_bwd_ws_bytes": ([c_int, c_int, c_int, c_int], c_int64),
    "tnr_embed_ln_bwd": ([P, c_int, c_int, c_int, c_int, P, c_int, P, P, P, c_float, c_int, P, P, P, P, P, P, P, c_int64,
                          POINTER(Dropout), P], c_int),
    "tnr_layernorm_fwd": ([P, c_int, c_int, P, P, c_float, P, P], c_int),
    "tnr_layernorm_bwd": ([P, P, c_int, c_int, P, c_float, P, P, P, P, P, POINTER(Dropout), P], c_int),
    "tnr_colsum_bf16": ([P, c_int, c_int, c_int, P, P], c_int),
    "tnr_attn_relpos_fwd": ([P, P, c_int, P, P, c_int, c_int, c_int, c_int, POINTER(Dropout), P], c_int),
    "tnr_attn_relpos_bwd": ([P, P, c_int, P, P, P, P, P, c_int, c_int, c_int, c_int, POINTER(Dropout), P], c_int),
    "tnr_attn_relpos_bwd_drel_ws_floats": ([c_int, c_int, c_int, c_int], c_int64),
    "tnr_attn_relpos_bwd_drel": ([P, P, c_int, P, P, P, P, P, c_int, c_int, c_int, c_int, POINTER(Dropout), P, c_int, P, P, P],
                                 c_int),
    "tnr_split_bf16x3": ([P, c_int, c_int, c_int, c_int, c_int, P, P], c_int),
    "tnr_embed_ln_fwd_f32": ([P, c_int, c_int, c_int, c_int, P, P, P, P, P, c_float, c_int, P, P], c_int),
    "tnr_add_layernorm_f32": ([P, P, c_int, c_int, P, P, c_float, P, P], c_int),
    "tnr_attn_relpos_fwd_f32": ([P, P, c_int, P, P, c_int, c_int, c_int, c_int, P], c_int),
    "tnr_attnpool_fwd_f32": ([P, P, c_int, c_int, P, P, P, c_int, c_int, c_int, P], c_int),
    "tnr_attnpool_fwd": ([P, P, c_int, c_int, P, P, P, P, P, c_int, c_int, c_int, P], c_int),
    "tnr_attnpool_bwd": ([P, P, c_int, c_int, P, P, P, P, P, P, P, c_int, c_int, c_int, P], c_int),
    "tnr_user_encoder_fwd": ([P, P, P, P, P, P, P, c_int, P, P, P, c_int, c_int, c_int, c_int, P], c_int),
    "tnr_user_encoder_fwd_multi": ([P, c_int, P, c_int, c_int, c_int, c_int, c_int, P], c_int),
    "tnr_user_encoder_fwd_gather": ([P, c_int64, P, P, P, P, P, P, P, c_int, P, P, c_int, c_int, c_int, c_int, P], c_int),
    "tnr_user_encoder_fwd_f32": ([P, P, P, P, P, P, P, c_int, P, P, P, c_int, c_int, c_int, c_int, P], c_int),
    "tnr_user_encoder_fwd_gather_f32": ([P, c_int64, P, P, P, P, P, P, P, c_int, P, P, c_int, c_int, c_int, c_int, P], c_int),
    "tnr_user_encoder_packed_w1_floats": ([c_int], c_int64),
    "tnr_user_encoder_pack_w1": ([P, P, P, P, P, c_int, c_int, P], c_int),
    "tnr_user_encoder_score_ws_bytes": ([c_int, c_int], c_int64),
    "tnr_user_encoder_score": ([P, c_int64, P, P, P, P, P, P, P, c_int, P, P, P, c_int, c_int, c_int, c_int, P], c_int),
    "tnr_user_encoder_bwd": ([P, P, P, P, P, c_int, P, P, P, P, P, P, P, P, P, P, c_int, c_int, c_int, c_int, P], c_int),
    "tnr_kd_loss_fwdbwd": ([P, P, P, P, P, c_int, c_int, c_int, c_int, c_int, c_float, c_float, c_int, P, P, P, P, P, P],
                           c_int),
    "tnr_sgemm_nt": ([P, P, P, P, c_int, c_int, c_int, c_int, c_int64, c_int64, c_int64, c_int64, P], c_int),
    "tnr_sgemm_nt_f32": ([P, P, P, P, c_int, c_int, c_int, c_int, c_int64, c_int64, c_int64, c_int64, P], c_int),
    "tnr_sgemm_tn_acc": ([P, P, P, P, c_int, c_int, c_int, c_int, c_int64, c_int64, c_int64, c_int64, P], c_int),
    "tnr_nrms_blend_fwd": ([P, P, P, P, c_int, c_int, P], c_int),
    "tnr_nrms_blend_bwd": ([P, P, P, P, c_int, c_int, P], c_int),
    "tnr_nrms_attn_fwd": ([P, P, P, P, P, c_int, c_int, c_int, P], c_int),
    "tnr_nrms_attn_bwd": ([P, P, P, P, P, P, P, P, c_int, c_int, c_int, P], c_int),
    "tnr_sgemm_nn": ([P, P, P, c_int, c_int, c_int, c_int, c_int64, c_int64, P], c_int),
    "tnr_adam_amsgrad": ([P, P, P, P, P, P, c_int64, c_float, c_float, c_float, c_float, c_int, c_float, P], c_int),
    "tnr_adam_amsgrad_devstep": ([P, P, P, P, P, P, c_int64, c_float, c_float, c_float, c_float, P, P, c_float, c_int, P], c_int),
    "tnr_cast_f32_bf16": ([P, P, c_int64, P], c_int),
    "tnr_gather_rows_i32_i64": ([P, c_int64, P, c_int64, c_int, P, P], c_int),
    "tnr_gather_rows_f32": ([P, c_int64, P, c_int64, c_int, P, c_int64, P], c_int),
    "tnr_train_batch_gather": ([P, c_int64, c_int, POINTER(c_void_p), POINTER(c_void_p), c_int, c_int, c_int64, P, c_int64, P,
                                c_int64, P, P], c_int),
    "tnr_doc_sim": ([P, c_int64, P, c_int64, c_int, P, P], c_int),
    "tnr_eval_metrics": ([P, c_int64, P, P, P, P, c_int64, c_int64, c_int, c_int, P, P, P, P], c_int),
    "tnr_predict_ranks": ([P, c_int64, P, P, P, c_int64, c_int64, c_int, c_int, P, P, P], c_int),
    "tnr_predict_format_ws_bytes": ([c_int64], c_int64),
    "tnr_predict_format_size": ([P, P, P, c_int64, P, P, c_int64, P], c_int),
    "tnr_predict_format_write": ([P, P, P, c_int64, P, P, P], c_int),
    "tnr_recommend_ws_bytes": ([c_int64, c_int, c_int, c_int], c_int64),
    "tnr_recommend_select": ([P, c_int64, P, c_int, c_int, P, P, c_int, c_int, c_int, P, c_int64, P], c_int),
    "tnr_recommend_merge": ([P, c_int64, P, c_int, c_int, c_int, c_int, c_int, P, P, P, P, c_int64, P], c_int),
    "tnr_recommend_filtered_ws_bytes": ([c_int64, c_int, c_int, c_int, c_int], c_int64),
    "tnr_recommend_select_filtered": ([P, c_int64, P, c_int, c_int, P, P, c_int, c_int, c_int, P, c_int, P, P, P, P, c_int64,
                                       P], c_int),
    "tnr_recommend_merge_filtered": ([P, c_int64, P, c_int, c_int, c_int, c_int, c_int, c_int, P, P, P, P, P, P, P, c_int64,
                                      P], c_int),
    "tnr_recommend_pool_ws_bytes": ([c_int64], c_int64),
    "tnr_recommend_pool": ([P, c_int64, P, P, P, P, P, c_int64, P], c_int),
}

_lib = None


def exported_names():
    return sorted(list(_SIGNATURES) + ["tnr_last_error"])


def load():
    """dlopen libtinyrec.so and attach argument types.  Raises if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise TinyRecError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). tiny-newsrec_b200 has no CPU or PyTorch fallback path.")
    lib = ctypes.CDLL(LIB_PATH)
    lib.tnr_last_error.argtypes = []
    lib.tnr_last_error.restype = c_char_p
    for name, (args, res) in _SIGNATURES.items():
        fn = getattr(lib, name)
        fn.argtypes = args
        fn.restype = res
    if lib.tnr_abi_version() != 6:
        raise TinyRecError("libtinyrec.so ABI version mismatch; rebuild")
    _lib = lib
    return lib


def check(rc, what):
    if rc != 0:
        msg = load().tnr_last_error().decode(errors="replace")
        raise TinyRecError(f"{what} failed (rc={rc}): {msg}")


_device_ok = set()


def require_device(index):
    """Fail loudly unless the current CUDA device is sm_100 (B200)."""
    if index in _device_ok:
        return
    n = c_int(0)
    check(load().tnr_device_check(ctypes.byref(n)), "tnr_device_check")
    _device_ok.add(index)
