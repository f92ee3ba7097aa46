/*
 * wlk_b200.h -- C ABI of the B200-native streaming-Whisper engine.
 *
 * The reference (QuentinFuxa/WhisperLiveKit) has no FFI: its plugin surface for
 * this path is Python duck-typing (SURVEY.md §8b).  This header is the boundary a
 * maintainer would bind (ctypes, see INTEGRATION.md) underneath those seams; each
 * entry point names the reference interface it replaces.  Conventions:
 *   - every function returns 0 on success, non-zero on failure; the message is
 *     available from wlk_last_error() (thread-local);
 *   - no exceptions, no C++/torch types cross the boundary: plain pointers+sizes;
 *   - "host" pointers are caller-owned host memory, "dev" pointers device memory
 *     on the engine's device; the engine owns all device state it allocates;
 *   - calls on one engine are serialised internally (one mutex, one CUDA stream);
 *     concurrency comes from batching sessions into one call.
 */
#ifndef WLK_B200_H
#define WLK_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define WLK_ABI_VERSION 1

typedef struct wlk_engine wlk_engine;

/* ModelDimensions, reference whisperlivekit/whisper/model.py:25-36 */
typedef struct wlk_dims {
    int32_t n_mels, n_audio_ctx, n_audio_state, n_audio_head, n_audio_layer;
    int32_t n_vocab, n_text_ctx, n_text_state, n_text_head, n_text_layer;
} wlk_dims;

enum { WLK_PREC_FP32 = 0,     /* SIMT fp32 kernels end to end: the 1e-3-on-logits parity mode                    */
       WLK_PREC_BF16 = 1,     /* bf16 operands / fp32 accumulate + fp32 residual: the serving mode                */
       WLK_PREC_BF16X3 = 2 }; /* tcgen05 with split operands (x = hi + lo, both bf16; A_hi W_hi + A_lo W_hi +    *
                               * A_hi W_lo into one fp32 accumulator): 1e-3 on logits at tensor-core speed / 3;   *
                               * activations, softmax, LayerNorm and K/V caches stay fp32                         */
enum { WLK_BACKEND_AUTO = 0, WLK_BACKEND_SIMT = 1, WLK_BACKEND_TCGEN05 = 2 };

typedef struct wlk_config {
    int32_t device;          /* CUDA ordinal */
    int32_t precision;       /* WLK_PREC_* */
    int32_t max_sessions;    /* device state is pooled for this many sessions */
    int32_t max_batch;       /* sessions per encode/decode call */
    int32_t gemm_backend;    /* WLK_BACKEND_* (AUTO: tcgen05 in bf16 mode, SIMT in fp32 mode) */
    int32_t attn_backend;    /* WLK_BACKEND_* for the encoder self-attention */
    int32_t max_align_heads; /* capacity of the alignment-head export */
    int32_t reserved;
} wlk_config;

const char* wlk_last_error(void);
int wlk_abi_version(void);

/* ---- engine lifetime + weights: replaces whisper.load_model()/Whisper.__init__
 *      (reference whisperlivekit/whisper/__init__.py:466-596, model.py:335-361)            */
int wlk_engine_create(const wlk_dims* dims, const wlk_config* cfg, wlk_engine** out);
int wlk_engine_destroy(wlk_engine* e);
/* name = reference state_dict key ("encoder.blocks.0.attn.query.weight", ...), plus
 * "mel_filters" [n_mels,201] and "hann_window" [400]; data = host fp32, row-major.        */
int wlk_engine_load_tensor(wlk_engine* e, const char* name, const float* host, const int64_t* shape, int ndim);
int wlk_engine_finalize_weights(wlk_engine* e);
/* packed device weight blob (for an NCCL broadcast done by the host at init)             */
int wlk_engine_weight_blob(wlk_engine* e, void** dev, size_t* nbytes);
int wlk_engine_adopt_weights(wlk_engine* e);   /* after the blob was filled by a broadcast */
/* (layer, head) pairs, reference model.alignment_heads (model.py:357-370) iteration order */
int wlk_engine_set_alignment_heads(wlk_engine* e, const int32_t* layer_head_pairs, int n_pairs);
int wlk_engine_stream(wlk_engine* e, void** cuda_stream);
int wlk_engine_sync(wlk_engine* e);
int wlk_engine_memory(wlk_engine* e, size_t* weights, size_t* sessions, size_t* workspace);

/* ---- per-session state: replaces DecoderState + AlignAtt.insert_audio
 *      (reference simul_whisper/decoder_state.py:7-91, simul_whisper.py:219-237)           */
int wlk_session_open(wlk_engine* e, int32_t* sid);
int wlk_session_close(wlk_engine* e, int32_t sid);
int wlk_session_append_audio(wlk_engine* e, int32_t sid, const float* pcm_host, int64_t n);
/* ingest step before the path (SURVEY.md section 8f item 3): the wire format is s16le PCM, which the reference
 * converts on the host (audio_processor.py:416-418: int16 / 32768.0); here half the bytes cross PCIe and the
 * conversion runs on the device straight into the session's ring.                                             */
int wlk_session_append_pcm16(wlk_engine* e, int32_t sid, const int16_t* pcm_host, int64_t n);
int wlk_session_drop_audio(wlk_engine* e, int32_t sid, int64_t n_front_samples);
int wlk_session_clear_audio(wlk_engine* e, int32_t sid);
int wlk_session_audio_len(wlk_engine* e, int32_t sid, int64_t* n);
/* DecoderState.clean_cache (reference decoder_state.py:51-59): forget the self-KV and the
 * alignment rows of the current epoch but keep the encoder output / cross-K/V.           */
int wlk_session_reset_decoder(wlk_engine* e, int32_t sid);
/* Beam search (reference simul_whisper/beam.py:8-32, whisper/decoding.py:289-376; AlignAtt with
 * decoder_type "beam", simul_whisper.py:182-192,240-243).  The reference runs the decoder on
 * beam_size rows that share one encoder output; here a beam is a session forked from the stream's
 * session: it has its own self-K/V, logits and alignment rows but reads the parent's encoder
 * output and cross-K/V (no copy, 245.8 MB per session at large-v3 stay shared).  A fork holds no
 * audio; it must be closed before its parent; encoding the parent starts a new epoch for its forks. */
int wlk_session_fork(wlk_engine* e, int32_t parent, int32_t* child_sid);
/* BeamPyTorchInference.rearrange_kv_cache (beam.py:15-19): for every i the self-K/V (and its
 * length) of sessions[i] becomes that of sessions[source_indices[i]] as it was before the call.
 * The alignment rows are NOT moved: the reference keeps its accumulated cross-attention per beam
 * row, not per hypothesis (align_att_base.py:222-224 appends whole [beam, ...] tensors).          */
int wlk_sessions_gather_decoder(wlk_engine* e, const int32_t* sessions, const int32_t* source_indices, int n);

/* ---- hot path, batched over sessions -------------------------------------------------
 * wlk_encode: AlignAtt._encode (simul_whisper.py:299-352) = log_mel_spectrogram
 *   (whisper/audio.py:110-157) + AudioEncoder.forward (model.py:238-254), plus the cross-
 *   attention K/V projection the reference does lazily (model.py:116-125).  Starts a new
 *   inference epoch for the session (the reference drops its KV cache after every infer,
 *   align_att_base.py:312).  content_mel_len_out[i] as simul_whisper.py:350.              */
int wlk_encode(wlk_engine* e, const int32_t* sids, int n, int32_t* content_mel_len_out);
/* wlk_encode_incremental: the same hook in the LABELLED APPROXIMATE incremental mode (north_star item 2; SURVEY.md
 *   section 7 H1): the K/V of every encoder layer are retained per session, and per call only a block of positions --
 *   two left of the old content end, the appended frames, two of padding (plus the vacated tail after a slide of the
 *   rolling window, simul_whisper.py:224-236) -- runs through the conv stem and the layers, attending to the retained
 *   K/V of every other position.  The first call of a stream takes the whole window as its block and equals wlk_encode;
 *   buffers are ring-addressed after a slide (nothing is moved).  Not bit- or 1e-3-comparable with the reference by
 *   construction: graded by token / attended-frame agreement with the parity mode.  bf16 tcgen05 mode only.
 *   block_rows_out[i] (may be NULL) = positions that went through the encoder for session i.                          */
int wlk_encode_incremental(wlk_engine* e, const int32_t* sids, int n, int32_t* content_mel_len_out, int32_t* block_rows_out);
/* forget the retained encoder K/V of a session: its next wlk_encode_incremental takes the whole window as its block
 * (= the parity computation); a host calls this to bound the drift of the approximate mode (also: WLK_INC_REFRESH=k
 * makes every k-th chunk such a block).                                                                              */
int wlk_session_reset_incremental(wlk_engine* e, int32_t sid);
/* wlk_decode: AlignAtt._get_logits_and_cross_attn (simul_whisper.py:357-368) =
 *   TextDecoder.forward with kv_cache + return_cross_attn (model.py:281-332).  Feeds
 *   tokens[offsets[i]..offsets[i+1]) to session i at its current self-KV offset.  Keeps
 *   the last-row logits (and, on the first call of an epoch, the row at sot_index) and
 *   the alignment heads' softmaxed cross-attention rows on the device.                    */
int wlk_decode(wlk_engine* e, const int32_t* sids, int n, const int32_t* tokens, const int32_t* offsets,
               int32_t sot_index);
/* ---- LocalAgreement path (whisper.transcribe(), reference whisper/transcribe.py:21-497) -------------
 * wlk_encode_mel: Whisper.encoder(mel) (model.py:238-254) for a log-mel the CALLER computed
 *   (transcribe.py:122 builds it on the host), mel_host = [n_mels, 3000] fp32; same epoch semantics as
 *   wlk_encode.
 * wlk_decode_all_logits: TextDecoder.forward returning the logits of EVERY fed position, as the word-timestamp
 *   pass needs (whisper/timing.py:197-201); logits_host = [n_tokens, n_vocab] fp32.
 * wlk_read_align_rows: softmax(qk) rows of the alignment heads accumulated in the current epoch,
 *   out = [n_align, rows, 1500] fp32 (what the cross-attention hooks of timing.py:186-192 capture).      In the incremental encoder mode the 1500 columns of a row are
 * ring slots, not frames: frame f is column (f + rot) mod 1500 (wlk_read_align_attn and the attended frames are in frame order). */
int wlk_encode_mel(wlk_engine* e, int32_t sid, const float* mel_host, int32_t content_mel_len);
int wlk_decode_all_logits(wlk_engine* e, int32_t sid, const int32_t* tokens, int n_tokens, int32_t sot_index,
                          float* logits_host);
int wlk_read_align_rows(wlk_engine* e, int32_t sid, float* out, int64_t capacity, int32_t* n_align, int32_t* rows);

/* AlignAtt._check_no_speech (simul_whisper.py:370-377)                                     */
int wlk_no_speech_prob(wlk_engine* e, const int32_t* sids, int n, float* prob_out);
/* _suppress_blank_tokens / SuppressTokens.apply (simul_whisper.py:379-385, decoding.py:427) */
int wlk_suppress(wlk_engine* e, const int32_t* sids, int n, const int32_t* token_ids, int n_tokens);
/* logits[tok] += bias: device half of _apply_dry_penalty (align_att_base.py:492-537)       */
int wlk_add_logit_bias(wlk_engine* e, int32_t sid, const int32_t* token_ids, const float* bias, int n);
/* GreedyDecoder.update (decoding.py:271-287) + _process_cross_attention +
 * _get_attended_frames (simul_whisper.py:390-437) over the last window_iters decode
 * calls of the epoch; one device->host copy of 3 scalars per session.                     */
int wlk_greedy_and_align(wlk_engine* e, const int32_t* sids, int n, int32_t window_iters,
                         int32_t* token_out, float* logprob_out, int32_t* frame_out);

/* One call for the "pick" half of a policy iteration (align_att_base.py:229-243): for every session first the
 * first-iteration set first_ids (where first_mask[i] != 0: _suppress_blank_tokens), then suppress_ids
 * (_apply_token_suppression), then logits[bias_tokens[k]] += bias_values[k] for k in [bias_offsets[i], bias_offsets[i+1])
 * (_apply_dry_penalty), then exactly what wlk_greedy_and_align does.  Same results as the separate calls in that order;
 * one lock acquisition, one staging upload and one device->host sync instead of four.  bias_* may be null.            */
int wlk_select(wlk_engine* e, const int32_t* sids, int n, const int32_t* suppress_ids, int n_suppress,
               const int32_t* first_ids, int n_first, const uint8_t* first_mask, const int32_t* bias_tokens,
               const float* bias_values, const int32_t* bias_offsets, int32_t window_iters, int32_t* token_out,
               float* logprob_out, int32_t* frame_out);

/* ---- debug taps for parity tests (device -> host fp32) ---------------------------------*/
int wlk_read_mel(wlk_engine* e, int32_t sid, float* out /* [n_mels,3000] */);
int wlk_read_encoder(wlk_engine* e, int32_t sid, float* out /* [1500,d] */);
int wlk_read_logits(wlk_engine* e, int32_t sid, int32_t which /* 0 last, 1 sot row */, float* out /* [V] */);
int wlk_read_align_attn(wlk_engine* e, int32_t sid, float* out, int64_t capacity, int32_t* rows, int32_t* cols);

/* ---- op-level entry points (kernel tests, roofline benches). Device pointers.
 *      backend: WLK_BACKEND_SIMT, WLK_BACKEND_TCGEN05 (auto tile choice), 3 = force the one-CTA tcgen05 kernel,
 *      4 = force the CTA-pair (cta_group::2) kernel.
 *      a_type/w_type/c_type: 0 = fp32, 1 = bf16.  C[M,N] = act(A[M,K] W[N,K]^T + bias); `gelu` is a flag
 *      word: bit 0 = erf-GELU, bit 1 = accumulate into the fp32 C in place (C += A W^T + bias).
 *      w_type 2 = the WLK_PREC_BF16X3 split operands (tcgen05 backends only): W is the bf16 hi plane, the lo plane
 *      sits right behind it at W + N * ldw; A is fp32 and is split on the fly.                                */
int wlk_op_gemm(wlk_engine* e, int backend, const void* A, int a_type, int64_t lda,
                const void* W, int w_type, int64_t ldw, const float* bias,
                void* C, int c_type, int64_t ldc, int M, int N, int K, int gelu);
/* encoder self-attention over qkv [batch * 1500, 3 * n_audio_state] (q, k pre-scaled by 64^-0.25) -> out
 * [batch * 1500, n_audio_state].  backend 3 = force the one-query-tile tcgen05 kernel.  type 0 = fp32, 1 = bf16,
 * 2 = split planes (tcgen05): qkv is the bf16 hi plane with the lo plane right behind it, out is fp32.             */
int wlk_op_encoder_attention(wlk_engine* e, int backend, const void* qkv, int type, int batch, void* out);
/* One decoder layer's attention over caches the caller owns, with the dispatch wlk_decode runs (backend
 * WLK_BACKEND_SIMT or WLK_BACKEND_TCGEN05 = the bf16 prefill kernels; type 0 = fp32, 1 = bf16).
 *   kind 0: causal self-attention, kv[i] = [n_text_layer][2][n_text_head][n_text_ctx][64];
 *   kind 1: cross-attention, kv[i] = [n_text_layer][2][n_text_head][1500][64]; the softmaxed rows of the engine's
 *           alignment heads go to align[i] = [n_align][n_text_ctx][1500] fp32 from row align_row0[i] on.
 * q and out are [sum n_rows][n_text_state], packed by job; row t of job i is at position offsets[i] + t.           */
int wlk_op_decoder_attention(wlk_engine* e, int kind, int backend, int type, int layer, const void* q, int n_jobs,
                             const int32_t* n_rows, const int32_t* offsets, const int32_t* align_row0,
                             const void* const* kv, float* const* align, void* out);

/* ---- word-timestamp kernels of the LocalAgreement path: native replacements of the reference's Triton
 *      median_kernel / dtw_kernel (whisper/triton_ops.py:13-103) with the semantics of its CPU path
 *      (whisper/timing.py:19-54 median_filter; :57-105 dtw_cpu + backtrace).  x is device fp32.
 *      wlk_op_dtw: x[N tokens, M frames] -> alignment path (text_idx[i], time_idx[i]), i < *len <= N+M.   */
/* diagnostic: the tcgen05 encoder attention with one CTA stamping clock64() at its pipeline hand-offs, [12 key tiles][8]:
 * MMA warp before S_j / before P_j V, softmax warp after S ready / exponentials done / arrive (tools/attn_trace.py)      */
int wlk_op_encoder_attention_trace(wlk_engine* e, const void* qkv_dev, int batch, void* out_dev, int64_t* stamps_host);
int wlk_op_median_filter(wlk_engine* e, const float* x_dev, float* out_dev, int rows, int cols, int width);
int wlk_op_dtw(wlk_engine* e, const float* x_dev, int N, int M, int32_t* text_idx_host, int32_t* time_idx_host,
               int32_t* len_out);

/* ---- device timers + per-kernel-class profile (CUDA events on the engine stream) ------- */
int wlk_timer_record(wlk_engine* e, int slot);                 /* slot in [0,16) */
int wlk_timer_elapsed_ms(wlk_engine* e, int from_slot, int to_slot, float* ms);
int wlk_profile_enable(wlk_engine* e, int on);
int wlk_profile_reset(wlk_engine* e);
/* class ids: see WLK_KC_*; returns accumulated device ms, launches, algorithmic flops and bytes */
int wlk_profile_read(wlk_engine* e, int kernel_class, double* ms, int64_t* launches, double* flops, double* bytes);
int wlk_profile_class_name(int kernel_class, const char** name);
enum { WLK_KC_MEL = 0, WLK_KC_GEMM_ENC, WLK_KC_ATTN_ENC, WLK_KC_LN, WLK_KC_GEMM_XKV, WLK_KC_GEMM_DEC,
       WLK_KC_ATTN_DEC_SELF, WLK_KC_ATTN_DEC_CROSS, WLK_KC_LOGITS, WLK_KC_ALIGN, WLK_KC_MISC, WLK_KC_COUNT };

/* =====================================================================================
 * Qwen3-ASR causal-KV audio tower (SURVEY.md section 8 row a17).  Replaces
 * QwenAudioCausalKVEncoder (reference third_party/qwen3-asr-causal/src/qwen3_asr_causal/causal.py:60-782):
 * append-only execution of the pretrained audio tower -- every mel frame transits conv stem and layers exactly
 * once, per-layer K/V of the bounded left window stay on the device, block-bidirectional or causal mask.
 * Tensor names are the tower's own state_dict names (conv2d1.weight ... layers.N.self_attn.q_proj.weight ...
 * ln_post.weight, proj1.weight, proj2.weight), fp32 on the host.
 * ===================================================================================== */
typedef struct wlk_qwen wlk_qwen;
typedef struct {
    int32_t n_mels;              /* 128 */
    int32_t conv_channels;       /* conv2d1/2/3 output channels (3x3, stride 2, pad 1) */
    int32_t d_model, n_head, n_layer, ffn_dim;
    int32_t out_dim;             /* proj2 output width */
    int32_t max_positions;       /* rows of the sinusoid table; the closed form is used beyond (causal.py:204-228) */
    int32_t chunk_frames;        /* 8: mel frames per encoder step */
    int32_t block_frames;        /* fixed attention block in mel frames (config.py:31-36); 0 = consume per chunk */
    int32_t left_context_steps;  /* K/V kept per layer (causal.py:103-106) */
    int32_t block_bidirectional; /* 1: queries see their whole block (causal.py:336-341) */
    int32_t conv_out_bias;
    int32_t mutable_tail_steps;  /* bounded mutable tail (causal.py:101-113, _encode_mutable_tail :548-640): > 0 requires
                                  * block_frames == 0; every call re-encodes the tail steps together with the new ones over
                                  * the frozen K/V prefix and returns hidden rows for ALL of them                          */
} wlk_qwen_dims;

int wlk_qwen_create(const wlk_qwen_dims* dims, const wlk_config* cfg, wlk_qwen** out);
int wlk_qwen_destroy(wlk_qwen* q);
int wlk_qwen_load_tensor(wlk_qwen* q, const char* name, const float* host, const int64_t* shape, int ndim);
int wlk_qwen_finalize_weights(wlk_qwen* q);
int wlk_qwen_memory(wlk_qwen* q, size_t* weights, size_t* sessions, size_t* workspace);
/* QwenAudioCausalKVState (causal.py:44-57): pending mel frames, per-layer K/V, emitted steps */
int wlk_qwen_session_open(wlk_qwen* q, int32_t* sid);
int wlk_qwen_session_close(wlk_qwen* q, int32_t sid);
int wlk_qwen_session_reset(wlk_qwen* q, int32_t sid);
int wlk_qwen_session_state(wlk_qwen* q, int32_t sid, int32_t* pending_frames, int64_t* emitted_steps);
/* QwenAudioCausalKVState.mutable_steps (causal.py:53-57): steps of the bounded mutable tail; emitted_steps counts frozen ones */
int wlk_qwen_session_mutable_steps(wlk_qwen* q, int32_t sid, int32_t* mutable_steps);
/* forward_chunk (causal.py:713-782) for n sessions at once.  mels_host holds the new mel frames of all sessions
 * back to back ([frames][n_mels] fp32, session i = rows frame_offsets[i] .. frame_offsets[i+1]); every complete
 * block (or chunk) is encoded; the newly emitted rows [steps][out_dim] of session i land in
 * out_host[out_row_offsets[i] .. out_row_offsets[i+1]).                                                       */
int wlk_qwen_forward_chunk(wlk_qwen* q, const int32_t* sids, int n, const float* mels_host, const int32_t* frame_offsets,
                           float* out_host, int64_t out_capacity_rows, int32_t* out_row_offsets);

/* StreamingMelExtractor.append (flush = 0) / .flush (flush = 1), reference features.py:86-110, for n sessions: the
 * raw sample window of every stream stays on the device; the call featurizes the windows (Hugging Face
 * WhisperFeatureExtractor semantics: reflect-padded 400-point STFT, hop 160, Slaney mel bank loaded as tensor
 * "mel_filters" [n_mels][201], log10, clamp to the window's max - 8, (x + 4) / 4) and returns the newly determined
 * frames [frames][n_mels] of session i in mel_out_host[frame_offsets_out[i] .. frame_offsets_out[i+1]).           */
int wlk_qwen_append_audio(wlk_qwen* q, const int32_t* sids, int n, const float* pcm_host, const int64_t* sample_offsets,
                          float* mel_out_host, int64_t out_capacity_frames, int32_t* frame_offsets_out, int32_t flush);
/* flush_pending (causal.py:687-711), end of stream: the buffered whole 8-frame chunks of each session are encoded as
 * one piece (whatever the block size), a sub-chunk remainder is dropped.                                          */
int wlk_qwen_flush_pending(wlk_qwen* q, const int32_t* sids, int n, float* out_host, int64_t out_capacity_rows,
                           int32_t* out_row_offsets);

/* =====================================================================================
 * Step after the diarization forward (SURVEY.md section 8f item 4).  Replaces SortformerDiarizationOnline.
 * _process_predictions (reference whisperlivekit/diarization/sortformer_backend.py:313-363): for every stream the last
 * len_prediction[i] frames of its device-resident predictions preds_dev[i] = [n_frames_total[i]][n_spk] fp32 are reduced
 * to argmax over the first max_speakers channels and run-length encoded; only the segments are copied to the host:
 * seg_out_host[i][k] = (speaker, first frame, end frame) in frames of the chunk, k < seg_count_host[i] <= max_seg.
 * Times are the caller's (round(base_time + frame * frame_duration, 2), :343-361).  n_spk < max_speakers is the
 * reference's RuntimeError (:316-319).
 * ===================================================================================== */
int wlk_diar_segments(int device, const float* const* preds_dev, const int32_t* n_frames_total,
                      const int32_t* len_prediction, int n_streams, int n_spk, int max_speakers,
                      int32_t* seg_out_host, int32_t* seg_count_host, int max_seg);

/* =====================================================================================
 * Ingest step before the path (SURVEY.md section 8f item 3): Silero VAD forward, batched over streams.  Replaces the
 * per-stream, per-window call of the scripted model that VADIterator / FixedVADIterator make (reference
 * whisperlivekit/silero_vad_iterator.py:20-29 init_jit_model, :288-331 FixedVADIterator.__call__ -> model(x[512], 16000)).
 * Tensor names are the scripted model's state_dict keys ("_model.stft.forward_basis_buffer", "_model.encoder.N.
 * reparam_conv.weight|bias", "_model.decoder.rnn.weight_ih|weight_hh|bias_ih|bias_hh", "_model.decoder.decoder.2.weight|
 * bias"; the "_model." prefix is optional).  A session holds what the model keeps between windows: the 64-sample context
 * and the LSTM (h, c).  wlk_vad_forward: session i consumes windows [window_offsets[i], window_offsets[i+1]) of pcm_host
 * ([windows][512] fp32, 16 kHz) in order and gets one speech probability per window in probs_host at the same index.
 * ===================================================================================== */
typedef struct wlk_vad wlk_vad;
int wlk_vad_create(int device, int max_sessions, wlk_vad** out);
int wlk_vad_destroy(wlk_vad* v);
int wlk_vad_load_tensor(wlk_vad* v, const char* name, const float* host, int64_t n);
int wlk_vad_session_open(wlk_vad* v, int32_t* sid);
int wlk_vad_session_reset(wlk_vad* v, int32_t sid);       /* model.reset_states() */
int wlk_vad_session_close(wlk_vad* v, int32_t sid);
int wlk_vad_forward(wlk_vad* v, const int32_t* sids, int n, const float* pcm_host, const int32_t* window_offsets,
                    float* probs_host);

/* =====================================================================================
 * Streaming Sortformer diarizer forward (SURVEY.md section 8 row a16, seam 8b-3).  Replaces what
 * SortformerDiarizationOnline.diarize() runs per 1.0 s chunk and stream (reference whisperlivekit/diarization/
 * sortformer_backend.py:253-311): AudioToMelSpectrogramPreprocessor.get_features (:181-188, :273), the 99-frame overlap
 * with the previous chunk (:277-283) and NeMo's SortformerEncLabelModel.forward_streaming_step (:293-300) with the
 * streaming parameters of :120-126 and the per-stream state of :212-234 (speaker cache, FIFO, silence profile).  The
 * arithmetic is NeMo's (absent from the reference tree); it is restated in oracle/sortformer_oracle.py, PARITY UNPINNED.
 * Tensor names are the NeMo state_dict keys ("encoder.pre_encode.conv.0.weight", "encoder.layers.N.self_attn.linear_q.
 * weight", "transformer_encoder.layers.N.first_sub_layer.query_net.weight", "sortformer_modules.encoder_proj.weight", ...)
 * plus "mel_filters" [n_mels][n_fft/2+1].  Sessions hold the state the reference keeps in StreamingSortformerState +
 * _previous_chunk_features + total_preds; many streams are served by one call.
 * ===================================================================================== */
typedef struct wlk_sf wlk_sf;
typedef struct wlk_sf_dims {
    int32_t n_mels, n_fft, win_length, hop;                 /* front end: 128, 512, 400, 160                            */
    int32_t conv_channels, d_model, n_head, n_layer, ff_mult, conv_kernel;   /* FastConformer: 256, 512, 8, 17, 4, 9    */
    int32_t tf_d_model, tf_n_head, tf_n_layer, tf_inner, n_spk;              /* Transformer + head: 192, 8, 18, 768, 4  */
    int32_t spkcache_len, fifo_len, spkcache_update_period, chunk_len, subsampling_factor;   /* :120-126                */
    int32_t encoder_subsampling, spkcache_sil_frames_per_spk;                /* 8, 3                                    */
    float pred_score_threshold, scores_boost_latest, sil_threshold;          /* SortformerModules defaults 0.25, 0.05,  */
    float strong_boost_rate, weak_boost_rate, min_pos_scores_rate;           /* 0.2, 0.75, 1.5, 0.5                     */
} wlk_sf_dims;
int wlk_sf_create(const wlk_sf_dims* dims, const wlk_config* cfg, wlk_sf** out);    /* SortformerDiarization._load_model :68-128 */
int wlk_sf_destroy(wlk_sf* q);
int wlk_sf_load_tensor(wlk_sf* q, const char* name, const float* host, const int64_t* shape, int ndim);
int wlk_sf_finalize_weights(wlk_sf* q);
int wlk_sf_session_open(wlk_sf* q, int32_t* sid);          /* SortformerDiarizationOnline.__init__ / _init_streaming_state :151-234 */
int wlk_sf_session_close(wlk_sf* q, int32_t sid);
int wlk_sf_session_reset(wlk_sf* q, int32_t sid);
/* diarize() (:253-311) for n streams: stream i hands in exactly chunk_len * subsampling_factor * hop samples
 * (pcm_host[sample_offsets[i] .. sample_offsets[i+1])); chunk_preds of stream i -- the rows forward_streaming_step
 * appends to total_preds -- land in chunk_preds_host[row_offsets_out[i] .. row_offsets_out[i+1]) x n_spk (may be NULL:
 * the rows also stay on the device, see wlk_sf_total_preds).  row_offsets_out has n + 1 entries.                       */
int wlk_sf_step_audio(wlk_sf* q, const int32_t* sids, int n, const float* pcm_host, const int64_t* sample_offsets,
                      float* chunk_preds_host, int32_t* row_offsets_out);
/* forward_streaming_step (:293-300) itself: time-major features [frames][n_mels] per stream (frame_offsets, n + 1
 * entries), left_offset / right_offset in feature frames as the reference passes them.                                 */
int wlk_sf_step_features(wlk_sf* q, const int32_t* sids, int n, const float* feats_host, const int32_t* frame_offsets,
                         int32_t left_offset, int32_t right_offset, float* chunk_preds_host, int32_t* row_offsets_out);
/* device-resident total_preds [n_rows][n_spk] of a stream (the tail the reference keeps, :301-305): feed it to
 * wlk_diar_segments so only segments cross PCIe.                                                                       */
int wlk_sf_total_preds(wlk_sf* q, int32_t sid, const float** preds_dev, int32_t* n_rows);
/* parity taps: lengths[4] = spkcache rows, fifo rows, n_sil_frames, chunk index; buffers may be NULL                   */
int wlk_sf_read_state(wlk_sf* q, int32_t sid, int32_t* lengths, float* spkcache_host, float* spkcache_preds_host,
                      float* fifo_host, float* mean_sil_host);
int wlk_sf_memory(wlk_sf* q, size_t* weights, size_t* sessions, size_t* workspace);

#ifdef __cplusplus
}
#endif
#endif /* WLK_B200_H */
