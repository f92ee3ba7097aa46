"""ctypes binding of include/wlk_b200.h (the C-ABI boundary).

There is no CPU fallback: if the in-tree library is missing this raises, and
``wlk_engine_create`` itself fails when no sm_100 device is present.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "csrc", "libwlk_b200.so")


class wlk_dims(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "n_mels", "n_audio_ctx", "n_audio_state", "n_audio_head", "n_audio_layer",
        "n_vocab", "n_text_ctx", "n_text_state", "n_text_head", "n_text_layer")]


class wlk_qwen_dims(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "n_mels", "conv_channels", "d_model", "n_head", "n_layer", "ffn_dim", "out_dim", "max_positions",
        "chunk_frames", "block_frames", "left_context_steps", "block_bidirectional", "conv_out_bias", "mutable_tail_steps")]


class wlk_sf_dims(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "n_mels", "n_fft", "win_length", "hop", "conv_channels", "d_model", "n_head", "n_layer", "ff_mult", "conv_kernel",
        "tf_d_model", "tf_n_head", "tf_n_layer", "tf_inner", "n_spk", "spkcache_len", "fifo_len", "spkcache_update_period",
        "chunk_len", "subsampling_factor", "encoder_subsampling", "spkcache_sil_frames_per_spk")] + [(n, C.c_float) for n in (
        "pred_score_threshold", "scores_boost_latest", "sil_threshold", "strong_boost_rate", "weak_boost_rate",
        "min_pos_scores_rate")]


class wlk_config(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "device", "precision", "max_sessions", "max_batch", "gemm_backend", "attn_backend",
        "max_align_heads", "reserved")]


PREC_FP32, PREC_BF16, PREC_BF16X3 = 0, 1, 2
BACKEND_AUTO, BACKEND_SIMT, BACKEND_TCGEN05 = 0, 1, 2
KERNEL_CLASSES = ["mel", "gemm_enc", "attn_enc", "layernorm", "gemm_xkv", "gemm_dec",
                  "attn_dec_self", "attn_dec_cross", "logits", "align", "misc"]

_i32p = C.POINTER(C.c_int32)
_f32p = C.POINTER(C.c_float)
_i64p = C.POINTER(C.c_int64)
_vp = C.c_void_p

# name -> (restype, argtypes); every symbol declared in include/wlk_b200.h
SIGNATURES = {
    "wlk_last_error": (C.c_char_p, []),
    "wlk_abi_version": (C.c_int, []),
    "wlk_engine_create": (C.c_int, [C.POINTER(wlk_dims), C.POINTER(wlk_config), C.POINTER(_vp)]),
    "wlk_engine_destroy": (C.c_int, [_vp]),
    "wlk_engine_load_tensor": (C.c_int, [_vp, C.c_char_p, _vp, _i64p, C.c_int]),
    "wlk_engine_finalize_weights": (C.c_int, [_vp]),
    "wlk_engine_weight_blob": (C.c_int, [_vp, C.POINTER(_vp), C.POINTER(C.c_size_t)]),
    "wlk_engine_adopt_weights": (C.c_int, [_vp]),
    "wlk_engine_set_alignment_heads": (C.c_int, [_vp, _i32p, C.c_int]),
    "wlk_engine_stream": (C.c_int, [_vp, C.POINTER(_vp)]),
    "wlk_engine_sync": (C.c_int, [_vp]),
    "wlk_engine_memory": (C.c_int, [_vp, C.POINTER(C.c_size_t), C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]),
    "wlk_session_open": (C.c_int, [_vp, _i32p]),
    "wlk_session_close": (C.c_int, [_vp, C.c_int32]),
    "wlk_session_append_audio": (C.c_int, [_vp, C.c_int32, _vp, C.c_int64]),
    "wlk_session_drop_audio": (C.c_int, [_vp, C.c_int32, C.c_int64]),
    "wlk_session_clear_audio": (C.c_int, [_vp, C.c_int32]),
    "wlk_session_audio_len": (C.c_int, [_vp, C.c_int32, _i64p]),
    "wlk_session_reset_decoder": (C.c_int, [_vp, C.c_int32]),
    "wlk_qwen_create": (C.c_int, [_vp, _vp, _vp]),
    "wlk_qwen_destroy": (C.c_int, [_vp]),
    "wlk_qwen_load_tensor": (C.c_int, [_vp, C.c_char_p, _vp, _vp, C.c_int]),
    "wlk_qwen_finalize_weights": (C.c_int, [_vp]),
    "wlk_qwen_memory": (C.c_int, [_vp, _vp, _vp, _vp]),
    "wlk_qwen_session_open": (C.c_int, [_vp, _vp]),
    "wlk_qwen_session_close": (C.c_int, [_vp, C.c_int32]),
    "wlk_qwen_session_reset": (C.c_int, [_vp, C.c_int32]),
    "wlk_qwen_session_state": (C.c_int, [_vp, C.c_int32, _vp, _vp]),
    "wlk_qwen_session_mutable_steps": (C.c_int, [_vp, C.c_int32, _vp]),
    "wlk_qwen_forward_chunk": (C.c_int, [_vp, _vp, C.c_int, _vp, _vp, _vp, C.c_int64, _vp]),
    "wlk_qwen_append_audio": (C.c_int, [_vp, _vp, C.c_int, _vp, _vp, _vp, C.c_int64, _vp, C.c_int32]),
    "wlk_qwen_flush_pending": (C.c_int, [_vp, _vp, C.c_int, _vp, C.c_int64, _vp]),
    "wlk_select": (C.c_int, [_vp, _vp, C.c_int, _vp, C.c_int, _vp, C.c_int, _vp, _vp, _vp, _vp, C.c_int32, _vp, _vp, _vp]),
    "wlk_vad_create": (C.c_int, [C.c_int, C.c_int, _vp]),
    "wlk_vad_destroy": (C.c_int, [_vp]),
    "wlk_vad_load_tensor": (C.c_int, [_vp, C.c_char_p, _vp, C.c_int64]),
    "wlk_vad_session_open": (C.c_int, [_vp, _vp]),
    "wlk_vad_session_reset": (C.c_int, [_vp, C.c_int32]),
    "wlk_vad_session_close": (C.c_int, [_vp, C.c_int32]),
    "wlk_vad_forward": (C.c_int, [_vp, _vp, C.c_int, _vp, _vp, _vp]),
    "wlk_sf_create": (C.c_int, [_vp, _vp, _vp]),
    "wlk_sf_destroy": (C.c_int, [_vp]),
    "wlk_sf_load_tensor": (C.c_int, [_vp, C.c_char_p, _vp, _vp, C.c_int]),
    "wlk_sf_finalize_weights": (C.c_int, [_vp]),
    "wlk_sf_session_open": (C.c_int, [_vp, _vp]),
    "wlk_sf_session_close": (C.c_int, [_vp, C.c_int32]),
    "wlk_sf_session_reset": (C.c_int, [_vp, C.c_int32]),
    "wlk_sf_step_audio": (C.c_int, [_vp, _vp, C.c_int, _vp, _vp, _vp, _vp]),
    "wlk_sf_step_features": (C.c_int, [_vp, _vp, C.c_int, _vp, _vp, C.c_int32, C.c_int32, _vp, _vp]),
    "wlk_sf_total_preds": (C.c_int, [_vp, C.c_int32, _vp, _vp]),
    "wlk_sf_read_state": (C.c_int, [_vp, C.c_int32, _vp, _vp, _vp, _vp, _vp]),
    "wlk_sf_memory": (C.c_int, [_vp, _vp, _vp, _vp]),
    "wlk_diar_segments": (C.c_int, [C.c_int, _vp, _vp, _vp, C.c_int, C.c_int, C.c_int, _vp, _vp, C.c_int]),
    "wlk_session_append_pcm16": (C.c_int, [_vp, C.c_int32, _vp, C.c_int64]),
    "wlk_session_fork": (C.c_int, [_vp, C.c_int32, _vp]),
    "wlk_sessions_gather_decoder": (C.c_int, [_vp, _vp, _vp, C.c_int]),
    "wlk_encode": (C.c_int, [_vp, _vp, C.c_int, _vp]),
    "wlk_encode_incremental": (C.c_int, [_vp, _vp, C.c_int, _vp, _vp]),
    "wlk_session_reset_incremental": (C.c_int, [_vp, C.c_int32]),
    "wlk_decode": (C.c_int, [_vp, _vp, C.c_int, _vp, _vp, C.c_int32]),
    "wlk_encode_mel": (C.c_int, [_vp, C.c_int32, _vp, C.c_int32]),
    "wlk_decode_all_logits": (C.c_int, [_vp, C.c_int32, _vp, C.c_int, C.c_int32, _vp]),
    "wlk_read_align_rows": (C.c_int, [_vp, C.c_int32, _vp, C.c_int64, _i32p, _i32p]),
    "wlk_no_speech_prob": (C.c_int, [_vp, _vp, C.c_int, _vp]),
    "wlk_suppress": (C.c_int, [_vp, _vp, C.c_int, _vp, C.c_int]),
    "wlk_add_logit_bias": (C.c_int, [_vp, C.c_int32, _vp, _vp, C.c_int]),
    "wlk_greedy_and_align": (C.c_int, [_vp, _vp, C.c_int, C.c_int32, _vp, _vp, _vp]),
    "wlk_read_mel": (C.c_int, [_vp, C.c_int32, _vp]),
    "wlk_read_encoder": (C.c_int, [_vp, C.c_int32, _vp]),
    "wlk_read_logits": (C.c_int, [_vp, C.c_int32, C.c_int32, _vp]),
    "wlk_read_align_attn": (C.c_int, [_vp, C.c_int32, _vp, C.c_int64, _i32p, _i32p]),
    "wlk_op_gemm": (C.c_int, [_vp, C.c_int, _vp, C.c_int, C.c_int64, _vp, C.c_int, C.c_int64, _vp,
                              _vp, C.c_int, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_int]),
    "wlk_op_encoder_attention": (C.c_int, [_vp, C.c_int, _vp, C.c_int, C.c_int, _vp]),
    "wlk_op_decoder_attention": (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, C.c_int, _vp, C.c_int, _vp, _vp, _vp, _vp,
                                           _vp, _vp]),
    "wlk_op_encoder_attention_trace": (C.c_int, [_vp, _vp, C.c_int, _vp, _vp]),
    "wlk_op_median_filter": (C.c_int, [_vp, _vp, _vp, C.c_int, C.c_int, C.c_int]),
    "wlk_op_dtw": (C.c_int, [_vp, _vp, C.c_int, C.c_int, _vp, _vp, _i32p]),
    "wlk_timer_record": (C.c_int, [_vp, C.c_int]),
    "wlk_timer_elapsed_ms": (C.c_int, [_vp, C.c_int, C.c_int, _f32p]),
    "wlk_profile_enable": (C.c_int, [_vp, C.c_int]),
    "wlk_profile_reset": (C.c_int, [_vp]),
    "wlk_profile_read": (C.c_int, [_vp, C.c_int, C.POINTER(C.c_double), _i64p, C.POINTER(C.c_double),
                                   C.POINTER(C.c_double)]),
    "wlk_profile_class_name": (C.c_int, [C.c_int, C.POINTER(C.c_char_p)]),
}

_lib = None


class WlkError(RuntimeError):
    pass


def load():
    """Load csrc/libwlk_b200.so (built by whisperlivekit_b200.build / __graft_entry__.build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise WlkError(
            f"{LIB_PATH} is missing: build it with `python -m whisperlivekit_b200.build` "
            "(nvcc, sm_100a). The B200 engine has no CPU or PyTorch fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if lib.wlk_abi_version() != 1:
        raise WlkError("ABI version mismatch")
    _lib = lib
    return lib


def check(rc: int):
    if rc != 0:
        raise WlkError(load().wlk_last_error().decode("utf-8", "replace"))
