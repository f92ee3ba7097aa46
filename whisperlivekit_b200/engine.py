"""Python host wrapper over the C-ABI engine (include/wlk_b200.h).

``WhisperEngine`` exposes the session API the AlignAtt host code drives
(``alignatt.StreamingAlignAtt`` / ``AlignAttHooks``); every method is one C call
into hand-written sm_100a CUDA.  Inputs are host numpy arrays (the reference's
callers hand CPU float32 PCM, SURVEY.md §8b); device memory is owned by the
engine.  There is no fallback path: construction raises without the library or
without a B200.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np

from . import _lib as L
from .dims import ModelDimensions, SpecialTokens, default_alignment_heads
from .weights import hann_window, mel_filterbank


def _i32(a) -> np.ndarray:
    return np.ascontiguousarray(np.asarray(a, dtype=np.int32))


def _ptr(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


class WhisperEngine:
    backend = "b200-cuda"

    def __init__(self, dims: ModelDimensions, state_dict: Optional[Dict[str, np.ndarray]] = None,
                 align_heads: Optional[Sequence[Tuple[int, int]]] = None, *, precision: str = "bf16",
                 device: int = 0, max_sessions: int = 8, max_batch: int = 8,
                 gemm_backend: str = "auto", attn_backend: str = "auto"):
        self.lib = L.load()
        self.dims = dims
        self.specials = SpecialTokens.for_dims(dims)
        self.precision = precision
        self.device = int(device)
        heads = list(align_heads) if align_heads is not None else default_alignment_heads(dims)
        self.align_heads = [tuple(int(v) for v in h) for h in heads]
        be = {"auto": L.BACKEND_AUTO, "simt": L.BACKEND_SIMT, "tcgen05": L.BACKEND_TCGEN05}
        cdims = L.wlk_dims(*dims.as_tuple())
        cfg = L.wlk_config(device=device, precision={"fp32": L.PREC_FP32, "bf16": L.PREC_BF16, "bf16x3": L.PREC_BF16X3}[precision],
                           max_sessions=max_sessions, max_batch=max_batch,
                           gemm_backend=be[gemm_backend], attn_backend=be[attn_backend],
                           max_align_heads=max(len(self.align_heads), 1), reserved=0)
        self.max_batch = max_batch
        h = C.c_void_p()
        L.check(self.lib.wlk_engine_create(C.byref(cdims), C.byref(cfg), C.byref(h)))
        self.h = h
        self._closed = False
        self.load_tensor("mel_filters", mel_filterbank(dims.n_mels))
        self.load_tensor("hann_window", hann_window())
        pairs = _i32(self.align_heads).reshape(-1)
        L.check(self.lib.wlk_engine_set_alignment_heads(self.h, pairs.ctypes.data_as(C.POINTER(C.c_int32)),
                                                        len(self.align_heads)))
        if state_dict is not None:
            self.load_state_dict(state_dict)

    # -- weights -----------------------------------------------------------------
    def load_tensor(self, name: str, arr) -> None:
        a = np.ascontiguousarray(np.asarray(arr, dtype=np.float32))
        shape = (C.c_int64 * a.ndim)(*a.shape)
        L.check(self.lib.wlk_engine_load_tensor(self.h, name.encode(), _ptr(a), shape, a.ndim))

    def load_state_dict(self, sd: Dict[str, np.ndarray]) -> None:
        for k, v in sd.items():
            if k.endswith("alignment_heads") or k.endswith(".mask"):
                continue
            self.load_tensor(k, v)
        L.check(self.lib.wlk_engine_finalize_weights(self.h))

    def weight_blob(self) -> Tuple[int, int]:
        """(device pointer, nbytes) of the packed weights -- broadcast target for NCCL at init."""
        p, n = C.c_void_p(), C.c_size_t()
        L.check(self.lib.wlk_engine_weight_blob(self.h, C.byref(p), C.byref(n)))
        return int(p.value), int(n.value)

    def adopt_weights(self) -> None:
        L.check(self.lib.wlk_engine_adopt_weights(self.h))

    def memory(self) -> Dict[str, int]:
        w, s, k = C.c_size_t(), C.c_size_t(), C.c_size_t()
        L.check(self.lib.wlk_engine_memory(self.h, C.byref(w), C.byref(s), C.byref(k)))
        return dict(weights=w.value, sessions=s.value, workspace=k.value)

    def stream(self) -> int:
        p = C.c_void_p()
        L.check(self.lib.wlk_engine_stream(self.h, C.byref(p)))
        return int(p.value or 0)

    def sync(self) -> None:
        L.check(self.lib.wlk_engine_sync(self.h))

    # -- sessions ------------------------------------------------------------------
    def open_session(self) -> int:
        sid = C.c_int32()
        L.check(self.lib.wlk_session_open(self.h, C.byref(sid)))
        return int(sid.value)

    def close_session(self, sid: int) -> None:
        L.check(self.lib.wlk_session_close(self.h, sid))

    def append_audio(self, sid: int, pcm) -> None:
        a = np.ascontiguousarray(np.asarray(pcm, dtype=np.float32).reshape(-1))
        L.check(self.lib.wlk_session_append_audio(self.h, sid, _ptr(a), a.shape[0]))

    def append_pcm16(self, sid: int, pcm) -> None:
        """s16le samples (bytes or int16 array), converted to fp32 / 32768 on the device (audio_processor.py:416-418)."""
        a = np.frombuffer(pcm, dtype=np.int16) if isinstance(pcm, (bytes, bytearray, memoryview)) else np.ascontiguousarray(pcm, np.int16)
        L.check(self.lib.wlk_session_append_pcm16(self.h, sid, _ptr(a), a.shape[0]))

    def drop_audio(self, sid: int, n: int) -> None:
        L.check(self.lib.wlk_session_drop_audio(self.h, sid, int(n)))

    def clear_audio(self, sid: int) -> None:
        L.check(self.lib.wlk_session_clear_audio(self.h, sid))

    def audio_len(self, sid: int) -> int:
        n = C.c_int64()
        L.check(self.lib.wlk_session_audio_len(self.h, sid, C.byref(n)))
        return int(n.value)

    def reset_decoder(self, sid: int) -> None:
        L.check(self.lib.wlk_session_reset_decoder(self.h, sid))

    # -- hot path --------------------------------------------------------------------
    def fork_session(self, parent: int) -> int:
        """A beam of ``parent``: own self-K/V, logits and alignment rows; shared encoder output and cross-K/V."""
        sid = C.c_int32()
        L.check(self.lib.wlk_session_fork(self.h, parent, C.byref(sid)))
        return sid.value

    def gather_decoder(self, sids: Sequence[int], source_indices: Sequence[int]) -> None:
        """BeamPyTorchInference.rearrange_kv_cache (reference beam.py:15-19) over a group of sessions."""
        a, b = _i32(sids), _i32(source_indices)
        if len(a) != len(b):
            raise ValueError("sids and source_indices differ in length")
        L.check(self.lib.wlk_sessions_gather_decoder(self.h, _ptr(a), _ptr(b), len(a)))

    incremental_encoder = False     # engine-wide default of ``encode``: True selects the labelled approximate mode

    def encode(self, sids: Sequence[int], incremental: Optional[bool] = None) -> List[int]:
        """AlignAtt._encode for a batch of sessions.  incremental=True (default: ``self.incremental_encoder``): the
        labelled approximate mode that retains the encoder K/V across chunks and runs only the appended frames
        (wlk_encode_incremental); the rows it encoded per session are left in ``self.last_block_rows``."""
        s = _i32(sids)
        out = np.zeros(len(s), np.int32)
        if self.incremental_encoder if incremental is None else incremental:
            rows = np.zeros(len(s), np.int32)
            L.check(self.lib.wlk_encode_incremental(self.h, _ptr(s), len(s), _ptr(out), _ptr(rows)))
            self.last_block_rows = [int(v) for v in rows]
        else:
            L.check(self.lib.wlk_encode(self.h, _ptr(s), len(s), _ptr(out)))
        return [int(v) for v in out]

    def reset_incremental(self, sid: int) -> None:
        """The next incremental encode of this session takes the whole window as its block (bounds the drift)."""
        L.check(self.lib.wlk_session_reset_incremental(self.h, int(sid)))

    def decode(self, sids: Sequence[int], tokens: Sequence[Sequence[int]], sot_index: int = 0) -> None:
        s = _i32(sids)
        offs = np.zeros(len(s) + 1, np.int32)
        offs[1:] = np.cumsum([len(t) for t in tokens])
        flat = _i32([t for ts in tokens for t in ts])
        L.check(self.lib.wlk_decode(self.h, _ptr(s), len(s), _ptr(flat), _ptr(offs), int(sot_index)))

    # -- LocalAgreement path ---------------------------------------------------------
    def encode_mel(self, sid: int, mel, content_mel_len: int = 1500) -> None:
        m = np.ascontiguousarray(np.asarray(mel, dtype=np.float32))
        assert m.shape == (self.dims.n_mels, 3000), m.shape
        L.check(self.lib.wlk_encode_mel(self.h, int(sid), _ptr(m), int(content_mel_len)))

    def decode_all_logits(self, sid: int, tokens: Sequence[int], sot_index: int = 0) -> np.ndarray:
        t = _i32(tokens)
        out = np.zeros((len(t), self.dims.n_vocab), np.float32)
        L.check(self.lib.wlk_decode_all_logits(self.h, int(sid), _ptr(t), len(t), int(sot_index), _ptr(out)))
        return out

    def read_align_rows(self, sid: int) -> np.ndarray:
        cap = max(1, len(self.align_heads)) * self.dims.n_text_ctx * 1500
        out = np.zeros(cap, np.float32)
        a, r = C.c_int32(), C.c_int32()
        L.check(self.lib.wlk_read_align_rows(self.h, int(sid), _ptr(out), cap, C.byref(a), C.byref(r)))
        return out[: a.value * r.value * 1500].reshape(a.value, r.value, 1500).copy()

    def no_speech_prob(self, sids: Sequence[int]) -> List[float]:
        s = _i32(sids)
        out = np.zeros(len(s), np.float32)
        L.check(self.lib.wlk_no_speech_prob(self.h, _ptr(s), len(s), _ptr(out)))
        return [float(v) for v in out]

    def suppress(self, sids: Sequence[int], token_ids: Sequence[int]) -> None:
        s, t = _i32(sids), _i32(token_ids)
        L.check(self.lib.wlk_suppress(self.h, _ptr(s), len(s), _ptr(t), len(t)))

    def add_logit_bias(self, sid: int, token_ids: Sequence[int], biases: Sequence[float]) -> None:
        t = _i32(token_ids)
        b = np.ascontiguousarray(np.asarray(biases, np.float32))
        L.check(self.lib.wlk_add_logit_bias(self.h, int(sid), _ptr(t), _ptr(b), len(t)))

    def greedy_and_align(self, sids: Sequence[int], window_iters: int = 16):
        s = _i32(sids)
        tok = np.zeros(len(s), np.int32)
        lp = np.zeros(len(s), np.float32)
        fr = np.zeros(len(s), np.int32)
        L.check(self.lib.wlk_greedy_and_align(self.h, _ptr(s), len(s), int(window_iters), _ptr(tok), _ptr(lp), _ptr(fr)))
        return [(int(tok[i]), float(lp[i]), int(fr[i])) for i in range(len(s))]

    def select(self, sids: Sequence[int], suppress: Sequence[int], first_ids: Sequence[int] = (),
               first_mask: Optional[Sequence[bool]] = None, biases: Optional[Sequence[Sequence[Tuple[int, float]]]] = None,
               window_iters: int = 16):
        """suppress (+ first-iteration set where first_mask) -> DRY biases -> greedy token / logprob -> attended frame,
        one C call (wlk_select).  biases[i] = [(token, value_to_add)] of session i."""
        s, sup, fst = _i32(sids), _i32(suppress), _i32(first_ids)
        n = len(s)
        mask = np.ascontiguousarray(first_mask if first_mask is not None else np.zeros(n), np.uint8)
        offs = np.zeros(n + 1, np.int32)
        bt, bv = [], []
        if biases is not None:
            for i, b in enumerate(biases):
                offs[i + 1] = offs[i] + len(b)
                bt += [int(t) for t, _ in b]; bv += [float(v) for _, v in b]
        btok, bval = _i32(bt), np.ascontiguousarray(bv, np.float32)
        tok = np.zeros(n, np.int32); lp = np.zeros(n, np.float32); fr = np.zeros(n, np.int32)
        L.check(self.lib.wlk_select(self.h, _ptr(s), n, _ptr(sup), len(sup), _ptr(fst), len(fst), _ptr(mask),
                                    _ptr(btok) if len(bt) else None, _ptr(bval) if len(bt) else None,
                                    _ptr(offs) if len(bt) else None, int(window_iters), _ptr(tok), _ptr(lp), _ptr(fr)))
        return [(int(tok[i]), float(lp[i]), int(fr[i])) for i in range(n)]

    # -- debug taps -------------------------------------------------------------------
    def read_mel(self, sid: int) -> np.ndarray:
        out = np.zeros((self.dims.n_mels, 3000), np.float32)
        L.check(self.lib.wlk_read_mel(self.h, sid, _ptr(out)))
        return out

    def read_encoder(self, sid: int) -> np.ndarray:
        out = np.zeros((1500, self.dims.n_audio_state), np.float32)
        L.check(self.lib.wlk_read_encoder(self.h, sid, _ptr(out)))
        return out

    def read_logits(self, sid: int) -> np.ndarray:
        out = np.zeros(self.dims.n_vocab, np.float32)
        L.check(self.lib.wlk_read_logits(self.h, sid, 0, _ptr(out)))
        return out

    def read_sot_logits(self, sid: int) -> np.ndarray:
        out = np.zeros(self.dims.n_vocab, np.float32)
        L.check(self.lib.wlk_read_logits(self.h, sid, 1, _ptr(out)))
        return out

    def read_align_attn(self, sid: int) -> np.ndarray:
        cap = self.dims.n_text_ctx * 1500
        out = np.zeros(cap, np.float32)
        r, c = C.c_int32(), C.c_int32()
        L.check(self.lib.wlk_read_align_attn(self.h, sid, _ptr(out), cap, C.byref(r), C.byref(c)))
        return out[: r.value * c.value].reshape(r.value, c.value).copy()

    # -- timers / profile ---------------------------------------------------------------
    def timer_record(self, slot: int) -> None:
        L.check(self.lib.wlk_timer_record(self.h, slot))

    def timer_elapsed_ms(self, a: int, b: int) -> float:
        ms = C.c_float()
        L.check(self.lib.wlk_timer_elapsed_ms(self.h, a, b, C.byref(ms)))
        return float(ms.value)

    def profile_enable(self, on: bool) -> None:
        L.check(self.lib.wlk_profile_enable(self.h, int(on)))

    def profile_reset(self) -> None:
        L.check(self.lib.wlk_profile_reset(self.h))

    def profile_read(self) -> Dict[str, dict]:
        out = {}
        for i, name in enumerate(L.KERNEL_CLASSES):
            ms, n, fl, by = C.c_double(), C.c_int64(), C.c_double(), C.c_double()
            L.check(self.lib.wlk_profile_read(self.h, i, C.byref(ms), C.byref(n), C.byref(fl), C.byref(by)))
            out[name] = dict(ms=ms.value, launches=n.value, flops=fl.value, bytes=by.value)
        return out

    # -- op-level (device pointers, e.g. torch tensors' data_ptr()) ----------------------
    def op_gemm(self, backend: str, A_ptr, a_type, lda, W_ptr, w_type, ldw, bias_ptr, C_ptr, c_type, ldc,
                M, N, K, gelu=False):
        be = {"simt": L.BACKEND_SIMT, "tcgen05": L.BACKEND_TCGEN05, "tcgen05_1cta": 3, "tcgen05_pair": 4}[backend]
        L.check(self.lib.wlk_op_gemm(self.h, be, A_ptr, a_type, lda, W_ptr, w_type, ldw, bias_ptr, C_ptr, c_type,
                                     ldc, M, N, K, int(gelu)))

    def op_encoder_attention(self, backend: str, qkv_ptr, dtype_code, batch, out_ptr):
        """dtype_code 0 = fp32, 1 = bf16, 2 = split bf16 planes (hi, lo right behind it; fp32 out)."""
        be = {"simt": L.BACKEND_SIMT, "tcgen05": L.BACKEND_TCGEN05, "tcgen05_1tile": 3}[backend]
        L.check(self.lib.wlk_op_encoder_attention(self.h, be, qkv_ptr, dtype_code, batch, out_ptr))

    def op_decoder_attention(self, kind: str, backend: str, dtype_code: int, layer: int, q_ptr, n_rows: Sequence[int],
                             offsets: Sequence[int], kv_ptrs: Sequence[int], out_ptr,
                             align_row0: Optional[Sequence[int]] = None, align_ptrs: Optional[Sequence[int]] = None):
        """One decoder layer's attention (wlk_op_decoder_attention) over caller-owned caches: kind "self" (causal) or
        "cross"; q / out packed [sum n_rows][n_text_state] by job, job i's rows at positions offsets[i] + t."""
        k = {"self": 0, "cross": 1}[kind]
        be = {"simt": L.BACKEND_SIMT, "tcgen05": L.BACKEND_TCGEN05}[backend]
        n = len(n_rows)
        nr, off = _i32(n_rows), _i32(offsets)
        kv = (C.c_void_p * n)(*[int(p) for p in kv_ptrs])
        a0 = _i32(align_row0) if align_row0 is not None else None
        al = (C.c_void_p * n)(*[int(p) for p in align_ptrs]) if align_ptrs is not None else None
        L.check(self.lib.wlk_op_decoder_attention(self.h, k, be, int(dtype_code), int(layer), q_ptr, n, _ptr(nr), _ptr(off),
                                                  _ptr(a0) if a0 is not None else None, kv, al, out_ptr))

    def op_median_filter(self, x_ptr, out_ptr, rows: int, cols: int, width: int = 7) -> None:
        L.check(self.lib.wlk_op_median_filter(self.h, x_ptr, out_ptr, rows, cols, width))

    def op_dtw(self, x_ptr, n_tokens: int, n_frames: int):
        """-> (text_indices, time_indices) like whisper.timing.dtw (reference timing.py:141-151)."""
        ti = np.zeros(n_tokens + n_frames, np.int32)
        fi = np.zeros(n_tokens + n_frames, np.int32)
        n = C.c_int32()
        L.check(self.lib.wlk_op_dtw(self.h, x_ptr, n_tokens, n_frames, _ptr(ti), _ptr(fi), C.byref(n)))
        return ti[: n.value].copy(), fi[: n.value].copy()

    def median_filter_host(self, x: np.ndarray, width: int = 7) -> np.ndarray:
        """whisper.timing.median_filter on a host array [..., cols] (reflect pad, odd width): H2D, wlk_op_median_filter,
        D2H.  Staging goes through torch's allocator (plumbing); the arithmetic is the native kernel."""
        import torch
        x = np.ascontiguousarray(x, np.float32)
        cols = x.shape[-1]
        xd = torch.from_numpy(x.reshape(-1, cols)).to(f"cuda:{self.device}")
        od = torch.empty_like(xd)
        torch.cuda.synchronize()
        self.op_median_filter(xd.data_ptr(), od.data_ptr(), xd.shape[0], cols, width)
        self.sync()
        return od.cpu().numpy().reshape(x.shape)

    def dtw_host(self, x: np.ndarray):
        """whisper.timing.dtw on a host cost matrix [n_tokens, n_frames] -> (text_indices, time_indices)."""
        import torch
        x = np.ascontiguousarray(x, np.float32)
        xd = torch.from_numpy(x).to(f"cuda:{self.device}")
        torch.cuda.synchronize()
        return self.op_dtw(xd.data_ptr(), x.shape[0], x.shape[1])

    # -- lifetime ------------------------------------------------------------------------
    def close(self) -> None:
        if not self._closed:
            self._closed = True
            L.check(self.lib.wlk_engine_destroy(self.h))

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
