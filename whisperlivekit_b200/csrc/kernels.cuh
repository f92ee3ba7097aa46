// Host-callable launchers of the non-GEMM kernels (mel front end, LayerNorm, encoder / decoder
// attention, logits post-processing, AlignAtt reduction).  `type` is a wlk::DType: the activation
// type of the engine's precision mode.
#pragma once
#include "common.cuh"

namespace wlk {

constexpr int MEL_ROWS = 3002;      // 3000 frames + one zero row either side (conv padding)
constexpr int N_FRAMES = 3000;
constexpr int N_CTX = 1500;
constexpr int N_FREQ = 201;
constexpr int N_FFT = 400;
constexpr int HOP = 160;
constexpr int MEL_FRAMES_PER_CTA = 16;
constexpr int MEL_STORE_FRAMES = 3008;                  // rows of MelJob.raw (N_FRAMES + 2, rounded up to whole CTAs)
constexpr int MEL_MAX_PARTS = 8;                        // partial maxima over the stored rows (mel_max_kernel)
constexpr int MEL_MAX_FRAMES = 2 * N_FRAMES + 2;        // a session may buffer up to 60 s: every frame joins the global max
constexpr int MEL_MAX_CTAS = (MEL_MAX_FRAMES + MEL_FRAMES_PER_CTA - 1) / MEL_FRAMES_PER_CTA;   // 376

struct MelJob {                 // one per session in the batch (device array)
    const float* audio;         // device, n samples
    float* raw;                 // [MEL_STORE_FRAMES][n_mels] fp32 log10(max(mel,1e-10)) for frames < min(n_compute, MEL_STORE_FRAMES)
    float* blockmax;            // [MEL_MAX_CTAS + MEL_MAX_PARTS]: per-CTA maxima of the frames computed in this pass, then
                                // the partial maxima over ALL stored rows (kept + recomputed)
    void* out;                  // [MEL_ROWS][n_mels] activation type, time-major, zero pad rows
    int32_t n;                  // samples
    int32_t n_compute;          // frames whose window touches audio (others are the silence constant); frames past
                                // MEL_STORE_FRAMES only feed the global maximum (audio.py:154-155 takes it over the whole
                                // padded spectrogram, before pad_or_trim cuts it to 3000 frames)
    int32_t n_total;            // floor((n + 480000) / 160): frames the reference's STFT keeps
    int32_t pad;
    // incremental log-mel: rows [keep_lo, keep_hi) of `raw` already hold this window's values (same samples, same
    // arithmetic as a full pass: bit-identical) and are not recomputed
    int32_t keep_lo, keep_hi;
};

// max_frames: the largest n_compute in the batch (sizes the grid)
void mel_forward(const MelJob* jobs_dev, int batch, int n_mels, const float* filtT, const float* window,
                 const float2* twiddle, const int2* filt_span, int out_type, int max_frames, cudaStream_t st);

// streaming-window variant (Qwen3 front end): MelJob.pad = 1, n_compute = n_total = window frames; emits frames
// [ranges[i].x, ranges[i].y) of job i as fp32 [frames][n_mels] at row out_off[i] of `out`
void mel_window_forward(const MelJob* jobs_dev, const int2* ranges_dev, const int64_t* out_off_dev, float* out_dev, int batch,
                        int n_mels, const float* filtT, const float* window, const float2* twiddle, const int2* filt_span,
                        int max_frames, cudaStream_t st);

void mel_import(const float* mel_dev /*[n_mels,3000]*/, void* out /*[3002,n_mels]*/, int out_type, int n_mels, cudaStream_t st);

void zero_rows(void* base, int type, int64_t row_elems, const int64_t* row_index_dev, int n_rows, cudaStream_t st);

// incremental encoder (engine.cu encode_incremental): operand gathers for the conv stem over a block of positions, and
// row scatters into a session's ring-addressed buffers
struct IncJob {                 // one per session in the batch (device array)
    const void* mel;            // [MEL_ROWS][n_mels] time-major log-mel of the window (activation type, zero pad rows)
    void* xa;                   // session encoder output [1500][d]
    int32_t p0, p1;             // block of logical positions [p0, p1)
    int32_t rot;                // slot = (position + rot) % 1500
    int32_t row1_off;           // first conv1 row of the block in the packed buffers (frames 2 p0 - 1 .. 2 p1 - 1)
    int32_t row_off;            // first position row of the block in the packed buffers
    int32_t pad;
};
void inc_gather_conv1(const IncJob* jobs, int n, int max_rows1, int n_mels, void* A1, int type, cudaStream_t st);
void inc_gather_conv2(const IncJob* jobs, int n, int max_rows, int d, const void* H1, void* A2, const float* enc_pos, float* posbuf,
                      int32_t* row_slot, int32_t* row_pos, int type, cudaStream_t st);
void inc_scatter_rows(const IncJob* jobs, int n, int max_rows, int d, const void* src, int type, cudaStream_t st);

void layernorm(const float* x, int64_t ldx, const float* w, const float* b, void* out, int out_type, int64_t ldo,
               int rows, int d, const int32_t* row_index_dev, cudaStream_t st);

void embed_tokens(const int32_t* tokens_dev, const int32_t* pos_dev, const float* emb, const float* pos_emb, float* x,
                  int rows, int d, cudaStream_t st);

// encoder self-attention over the fused qkv buffer [batch*1500, 3d] (q,k pre-scaled by d_head^-0.25)
void enc_attention_simt(const void* qkv, int type, int batch, int n_head, int d_model, void* out, cudaStream_t st);
void enc_attention_tcgen05(const void* qkv, int batch, int n_head, int d_model, void* out, cudaStream_t st, int num_sms,
                           long long* trace_dev = nullptr);   // trace_dev: [12 tiles][8] clock64 stamps of one CTA (diagnostic)
// always the one-query-tile CTA of attn_tc.cu (the kernel body the decoder prefills and the split-operand mode run)
void enc_attention_tcgen05_one_tile(const void* qkv, int batch, int n_head, int d_model, void* out, cudaStream_t st,
                                    long long* trace_dev = nullptr);
void enc_attention_tcgen05_x3(const void* qkv_hi, const void* qkv_lo, int batch, int n_head, int d_model, float* out, cudaStream_t st);
// fp32 -> (hi, lo) bf16 planes on the stream (gemm_tc.cu)
void split_f32_planes_async(const float* src, bf16* hi, bf16* lo, int64_t n, cudaStream_t st);

struct DecJob {                 // one per session in a decode batch (device array)
    void* self_kv;              // [L][2][H][n_text_ctx][64]
    const void* cross_kv;       // [L][2][H][1500][64]
    float* align;               // [n_align][n_text_ctx][1500] softmaxed cross-attention rows
    float* logits_last;         // [V]
    float* logits_sot;          // [V]
    int32_t row_off;            // first row of this session in the packed row buffers
    int32_t n_rows;             // Tq
    int32_t offset;             // self-KV length before this call (position of row 0)
    int32_t align_row0;         // first alignment row this call writes (rows accumulated in the epoch)
    int32_t slot;               // session slot (index of its cross-K/V tensor map)
    int32_t pad0, pad1, pad2;
};

void dec_self_attention(const void* q, int type, const DecJob* jobs, int n_jobs, int layer, int n_head, int d_model,
                        int n_text_ctx, void* out, int max_rows, cudaStream_t st);
// align_rank[layer * n_head + head] = rank of the alignment head or -1
void dec_cross_attention(const void* q, int type, const DecJob* jobs, int n_jobs, int layer, int n_head, int d_model,
                         int n_text_ctx, const int32_t* align_rank, void* out, int max_rows, bool only_align_heads,
                         cudaStream_t st);
// tensor-core prefill path (bf16): every head that is not an alignment head
void dec_cross_attention_tcgen05(const void* q, int total_rows, const DecJob* jobs, int n_jobs, int max_rows, int layer,
                                 int n_head, int d_model, const void* kv_maps_dev, const int32_t* align_rank, void* out,
                                 cudaStream_t st);
void make_cross_kv_tmap(void* tmap_out_host /* 128 bytes */, const void* cross_kv, int n_layer, int n_head);
// tensor-core causal prefill of the decoder self-attention (bf16)
void dec_self_attention_tcgen05(const void* q, int total_rows, const DecJob* jobs, int n_jobs, int max_rows, int layer,
                                int n_head, int d_model, int n_text_ctx, const void* kv_maps_dev, void* out, cudaStream_t st);
void make_self_kv_tmap(void* tmap_out_host /* 128 bytes */, const void* self_kv, int n_layer, int n_head, int n_text_ctx);

struct LogitJob {               // one per session (device array)
    float* logits_last;
    float* logits_sot;
    const float* align;         // [n_align][n_text_ctx][1500]
    float* attn_out;            // [n_text_ctx][1500] scratch/tap: processed attention rows
    float* stats;               // [n_align][1500][2] scratch: mean, 1/(std+1e-8)
    int32_t row_begin, row_end; // retained alignment rows [begin, end)
    int32_t content_len;
    int32_t full;               // 1: produce every retained row (debug tap); 0: last row only
    int32_t rot;                // ring offset of the encoder output (incremental encoder): frame f sits in slot (f + rot) % 1500
    int32_t pad;
};
struct StepResult { int32_t token; float logprob; int32_t frame; float no_speech; };

void no_speech_prob(const LogitJob* jobs, int n, int n_vocab, int no_speech_token, StepResult* res, cudaStream_t st);
void suppress_tokens(const LogitJob* jobs, int n, const int32_t* tokens_dev, int n_tokens, cudaStream_t st);
void add_logit_bias(float* logits, const int32_t* tokens_dev, const float* bias_dev, int n, cudaStream_t st);
// entry i adds bias[i] to logits_last[tokens[i]] of job job_of[i] (tokens are distinct within a job)
void add_logit_bias_jobs(const LogitJob* jobs, const int32_t* job_of_dev, const int32_t* tokens_dev, const float* bias_dev, int n,
                         cudaStream_t st);
void greedy_pick(const LogitJob* jobs, int n, int n_vocab, StepResult* res, cudaStream_t st);
void align_reduce(const LogitJob* jobs, int n, int n_align, int n_text_ctx, StepResult* res, cudaStream_t st);

// word-timestamp kernels (LocalAgreement path)
void median_filter(const float* x, float* out, int rows, int cols, int width, cudaStream_t st);
struct DtwJobHost { const float* x; uint8_t* trace; int32_t* path; int32_t* path_len; int32_t N, M; };
void dtw_batch(const void* jobs_dev, int n_jobs, int max_tokens, cudaStream_t st);

void convert_f32_to(const float* src, void* dst, int dst_type, int64_t n, cudaStream_t st);
void convert_to_f32(const void* src, int src_type, float* dst, int64_t n, cudaStream_t st);
// WLK_PREC_BF16X3 weights: hi = bf16(x), lo = bf16(x - hi)
void split_f32_to_planes(const float* src, bf16* hi, bf16* lo, int64_t n, cudaStream_t st);
void pcm16_to_f32(const int16_t* src_dev, float* dst_dev, int64_t n, cudaStream_t st);
// conv weight [c_out, c_in, 3] -> [c_out, 3 * c_in] (tap-major) in the destination type
void pack_conv_weight(const float* w, void* dst, int dst_type, int c_out, int c_in, cudaStream_t st);

}  // namespace wlk
