// Engine: weights arena, per-session device state, batched encode/decode orchestration and the C ABI
// declared in include/wlk_b200.h.  One CUDA stream per engine; calls are serialised by a mutex and
// concurrency comes from batching sessions into one call.
#include <algorithm>
#include <cmath>
#include <map>
#include <mutex>
#include <set>
#include <vector>

#include "../../include/wlk_b200.h"
#include "kernels.cuh"

namespace wlk {

bool pdl_enabled() {
    static const bool on = [] {
        const char* v = getenv("WLK_PDL");
        return !(v && v[0] == '0');
    }();
    return on;
}


static thread_local std::string g_last_error;
void set_last_error(const std::string& msg) { g_last_error = msg; }

namespace {

constexpr int AUDIO_CAP = 2 * 480000;       // samples a session may buffer (reference keeps <= 30 s + one chunk)
constexpr size_t ALIGN = 256;

static const char* kClassNames[WLK_KC_COUNT] = {"mel", "gemm_enc", "attn_enc", "layernorm", "gemm_xkv", "gemm_dec",
                                                "attn_dec_self", "attn_dec_cross", "logits", "align", "misc"};

struct Arena {                       // bump allocator over one device allocation (the weight blob)
    uint8_t* base = nullptr;
    size_t cap = 0, used = 0;
    void* take(size_t bytes) {
        size_t off = (used + ALIGN - 1) / ALIGN * ALIGN;
        used = off + bytes;
        return base ? base + off : reinterpret_cast<void*>(off);   // dry run when base == nullptr
    }
};

struct EncLayerW { float *ln1w, *ln1b, *bqkv, *bo, *ln2w, *ln2b, *b1, *b2; void *Wqkv, *Wo, *W1, *W2; };
struct DecLayerW {
    float *ln1w, *ln1b, *bqkv, *bo, *lncw, *lncb, *bqc, *boc, *ln2w, *ln2b, *b1, *b2;
    void *Wqkv, *Wo, *Wqc, *Woc, *W1, *W2;
};
struct Weights {
    float *filtT, *window; float2* twiddle; int2* filt_span;
    void *Wc1, *Wc2; float *bc1, *bc2, *enc_pos;
    std::vector<EncLayerW> enc;
    float *lnpw, *lnpb;
    float* emb_f32; void* emb_act; float* dec_pos;
    std::vector<DecLayerW> dec;
    float *lnw, *lnb;
    void* Wxkv; float* bxkv;          // all decoder layers' cross K/V projections: [L*2*dt, d_audio]
};

struct Session {
    bool open = false;
    float* audio = nullptr; int64_t audio_len = 0;
    float* mel_raw = nullptr; float* mel_blockmax = nullptr;
    // incremental log-mel: mel_raw holds the raw log-mel of the window as it was when audio_len was mel_n, minus
    // mel_dropped samples dropped at the front since (-1: nothing cached)
    int64_t mel_n = -1, mel_dropped = 0;
    void* xa = nullptr; void* cross_kv = nullptr; void* self_kv = nullptr;
    float* align = nullptr; float* logits_last = nullptr; float* logits_sot = nullptr;
    float* attn_out = nullptr; float* stats = nullptr;
    int self_len = 0, align_rows = 0, content_len = 0;
    bool encoded = false;
    std::vector<int> iter_row_start;
    size_t bytes = 0;
    int parent = -1;      // >= 0: a beam fork -- audio/mel are null, xa / cross_kv alias the parent's buffers
    int n_forks = 0;      // open forks reading this session's encoder output
    // incremental encoder (labelled approximate mode, encode_incremental): encoder K/V of every layer retained across
    // chunks [L_enc][2][H][1500][64], ring-addressed: logical position p of the window lives in slot (p + rot) % 1500
    void* enc_kv = nullptr;
    bool inc_valid = false;
    int rot = 0;
    int inc_content = 0;          // positions of content covered by the last incremental encode
    int64_t inc_dropped = 0;      // samples dropped at the front since then
    int inc_chunks = 0;           // incremental encodes since the last full-window block
};

struct ProfRec { int cls; cudaEvent_t a, b; double flops, bytes; };

}  // namespace
}  // namespace wlk

using namespace wlk;

struct wlk_engine {
    wlk_dims dims{};
    wlk_config cfg{};
    int act = DT_F32;                 // activation type (and type of every session buffer)
    int wt = DT_F32;                  // weight-matrix type: = act, or DT_BF16X2 (hi + lo bf16 planes) in WLK_PREC_BF16X3
    void* a_split = nullptr; size_t a_split_elems = 0;   // BF16X3: (hi, lo) planes of a GEMM's fp32 activation operand
    int gemm_backend = WLK_BACKEND_SIMT, attn_backend = WLK_BACKEND_SIMT;
    int num_sms = 148;
    cudaStream_t st = nullptr;
    std::mutex mu;
    // token-step CUDA graphs: the ~390 launches of one decoder step depend only on the batch size (every per-session
    // quantity travels in the staged job arrays), so they are captured once per batch size and replayed
    bool graphs_on = true;
    bool mel_incremental = true;      // WLK_MEL_INCREMENTAL=0: recompute every frame of the window at every encode
    struct GraphSlot { cudaGraphExec_t exec; uint64_t last_use; };
    std::map<uint64_t, GraphSlot> dec_graphs;     // LRU-bounded: under the batching shim the batch size varies in 1..max_batch
    std::set<uint64_t> dec_graph_seen;
    uint64_t dec_graph_tick = 0;

    Arena arena;
    Weights w;
    std::set<std::string> loaded;
    bool finalized = false;
    float* stage_f32 = nullptr; size_t stage_cap = 0;

    std::vector<Session> sess;
    std::vector<int32_t> align_rank_host;     // [L*H] -> rank or -1
    int32_t* align_rank_dev = nullptr;
    uint8_t* kv_maps_dev = nullptr;           // [max_sessions] CUtensorMap (128 B each) over each session's cross-K/V
    uint8_t* self_maps_dev = nullptr;         // [max_sessions] CUtensorMap over each session's self-K/V cache
    uint8_t* enc_maps_dev = nullptr;          // [max_sessions] CUtensorMap over each session's retained encoder K/V
    int32_t* enc_norank_dev = nullptr;        // [L_enc * H_enc] all -1: no head of the encoder is an alignment head
    int32_t *inc_row_slot = nullptr, *inc_row_pos = nullptr;   // [max_batch * 1500] row maps of an incremental block
    int inc_refresh = 0;                      // WLK_INC_REFRESH: a full-window block every this many chunks (0: never)
    int n_align = 0;

    // encoder workspace (max_batch streams)
    void *mel_t = nullptr, *h1 = nullptr, *xn = nullptr, *qkv = nullptr, *att = nullptr, *hid = nullptr;
    float* x = nullptr;
    int64_t* pad_rows_dev = nullptr;          // rows of h1 to re-zero after the conv1 GEMM
    void** xptrs_dev = nullptr;               // x + b*1500*d
    float* audio_scratch = nullptr;
    void* beam_scratch = nullptr; size_t beam_scratch_cap = 0;   // staging for wlk_sessions_gather_decoder
    float* sk_scratch = nullptr; int* sk_counters = nullptr;     // this engine's split-K workspace (GemmArgs)
    float* mel_scratch = nullptr;             // fp32 [MEL_ROWS][n_mels] for the read_mel tap
    // decoder workspace
    int dec_rows_max = 0;
    float* dx = nullptr; void *dxn = nullptr, *dq = nullptr, *datt = nullptr, *dhid = nullptr, *dsel = nullptr;
    // staging (pinned host mirror + device copy)
    uint8_t *stg_host = nullptr, *stg_dev = nullptr; size_t stg_bytes = 0;
    cudaEvent_t stg_done = nullptr;
    StepResult *res_dev = nullptr, *res_host = nullptr;
    float* tap_host = nullptr; size_t tap_cap = 0;
    float* all_logits_dev = nullptr; size_t all_logits_cap = 0;

    cudaEvent_t timers[16] = {};
    bool prof_on = false;
    std::vector<ProfRec> prof;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> ev_pool;
    size_t bytes_weights = 0, bytes_sessions = 0, bytes_workspace = 0;

    size_t es() const { return dtype_size(act); }
    size_t wes() const { return dtype_size(wt); }
};

namespace wlk {
namespace {

template <typename T>
T* dmalloc(wlk_engine* e, size_t count, size_t* acct) {
    void* p = nullptr;
    size_t bytes = count * sizeof(T);
    if (bytes == 0) bytes = 16;
    CUDA_CHECK(cudaMalloc(&p, bytes));
    if (acct) *acct += bytes;
    return reinterpret_cast<T*>(p);
}
void* dmalloc_bytes(size_t bytes, size_t* acct) {
    void* p = nullptr;
    if (bytes == 0) bytes = 16;
    CUDA_CHECK(cudaMalloc(&p, bytes));
    if (acct) *acct += bytes;
    return p;
}

// ---------------------------------------------------------------------------------------
// profiling
// ---------------------------------------------------------------------------------------
struct ProfScope {
    wlk_engine* e; int idx = -1;
    ProfScope(wlk_engine* e_, int cls, double flops = 0, double bytes = 0) : e(e_) {
        if (!e->prof_on) return;
        std::pair<cudaEvent_t, cudaEvent_t> ev;
        if (!e->ev_pool.empty()) { ev = e->ev_pool.back(); e->ev_pool.pop_back(); }
        else { CUDA_CHECK(cudaEventCreate(&ev.first)); CUDA_CHECK(cudaEventCreate(&ev.second)); }
        CUDA_CHECK(cudaEventRecord(ev.first, e->st));
        e->prof.push_back({cls, ev.first, ev.second, flops, bytes});
        idx = (int)e->prof.size() - 1;
    }
    ~ProfScope() {
        if (idx >= 0) cudaEventRecord(e->prof[idx].b, e->st);
    }
};

// ---------------------------------------------------------------------------------------
// weights
// ---------------------------------------------------------------------------------------
void layout_weights(wlk_engine* e) {
    const wlk_dims& D = e->dims;
    Arena& A = e->arena;
    Weights& W = e->w;
    const size_t es = e->wes();
    const int d = D.n_audio_state, dt = D.n_text_state;
    auto f32 = [&](size_t n) { return reinterpret_cast<float*>(A.take(n * 4)); };
    auto mat = [&](size_t n) { return A.take(n * es); };
    W.filtT = f32((size_t)N_FREQ * D.n_mels);
    W.window = f32(N_FFT);
    W.twiddle = reinterpret_cast<float2*>(A.take(N_FFT * 8));
    W.filt_span = reinterpret_cast<int2*>(A.take((size_t)D.n_mels * 8));
    W.Wc1 = mat((size_t)d * 3 * D.n_mels); W.bc1 = f32(d);
    W.Wc2 = mat((size_t)d * 3 * d); W.bc2 = f32(d);
    W.enc_pos = f32((size_t)D.n_audio_ctx * d);
    W.enc.resize(D.n_audio_layer);
    for (auto& l : W.enc) {
        l.ln1w = f32(d); l.ln1b = f32(d);
        l.Wqkv = mat((size_t)3 * d * d); l.bqkv = f32(3 * d);
        l.Wo = mat((size_t)d * d); l.bo = f32(d);
        l.ln2w = f32(d); l.ln2b = f32(d);
        l.W1 = mat((size_t)4 * d * d); l.b1 = f32(4 * d);
        l.W2 = mat((size_t)4 * d * d); l.b2 = f32(d);
    }
    W.lnpw = f32(d); W.lnpb = f32(d);
    W.emb_f32 = f32((size_t)D.n_vocab * dt);
    W.emb_act = (e->wt == DT_F32) ? (void*)W.emb_f32 : mat((size_t)D.n_vocab * dt);
    W.dec_pos = f32((size_t)D.n_text_ctx * dt);
    W.dec.resize(D.n_text_layer);
    for (auto& l : W.dec) {
        l.ln1w = f32(dt); l.ln1b = f32(dt);
        l.Wqkv = mat((size_t)3 * dt * dt); l.bqkv = f32(3 * dt);
        l.Wo = mat((size_t)dt * dt); l.bo = f32(dt);
        l.lncw = f32(dt); l.lncb = f32(dt);
        l.Wqc = mat((size_t)dt * dt); l.bqc = f32(dt);
        l.Woc = mat((size_t)dt * dt); l.boc = f32(dt);
        l.ln2w = f32(dt); l.ln2b = f32(dt);
        l.W1 = mat((size_t)4 * dt * dt); l.b1 = f32(4 * dt);
        l.W2 = mat((size_t)4 * dt * dt); l.b2 = f32(dt);
    }
    W.lnw = f32(dt); W.lnb = f32(dt);
    W.Wxkv = mat((size_t)D.n_text_layer * 2 * dt * d);
    W.bxkv = f32((size_t)D.n_text_layer * 2 * dt);
}

float* stage_reserve(wlk_engine* e, size_t n) {
    if (n > e->stage_cap) {
        if (e->stage_f32) CUDA_CHECK(cudaFree(e->stage_f32));
        size_t cap = n < (1u << 20) ? (1u << 20) : n;
        CUDA_CHECK(cudaMalloc(&e->stage_f32, cap * 4));
        e->stage_cap = cap;
    }
    return e->stage_f32;
}
float* stage(wlk_engine* e, const float* host, size_t n) {
    float* s = stage_reserve(e, n);
    CUDA_CHECK(cudaMemcpyAsync(s, host, n * 4, cudaMemcpyHostToDevice, e->st));
    return s;
}
void put_f32(wlk_engine* e, float* dst, const float* host, size_t n) {
    CUDA_CHECK(cudaMemcpyAsync(dst, host, n * 4, cudaMemcpyHostToDevice, e->st));
    CUDA_CHECK(cudaStreamSynchronize(e->st));
}
// device fp32 -> `n` elements at element offset `off` of a weight matrix of `total` elements (planar in DT_BF16X2)
void store_mat(wlk_engine* e, void* base, size_t total, size_t off, const float* src_dev, size_t n) {
    if (e->wt == DT_BF16X2) {
        bf16* hi = reinterpret_cast<bf16*>(base) + off;
        split_f32_to_planes(src_dev, hi, hi + total, (int64_t)n, e->st);
    } else {
        convert_f32_to(src_dev, reinterpret_cast<uint8_t*>(base) + off * e->wes(), e->wt, (int64_t)n, e->st);
    }
    CUDA_CHECK(cudaStreamSynchronize(e->st));
}
void put_mat(wlk_engine* e, void* base, size_t total, size_t off, const float* host, size_t n) {
    store_mat(e, base, total, off, stage(e, host, n), n);
}
uint8_t* offs(void* p, size_t elems, size_t es) { return reinterpret_cast<uint8_t*>(p) + elems * es; }
// conv weight [c_out, c_in, 3] -> tap-major [c_out, 3 * c_in] in the weight type (via an fp32 staging copy in BF16X3)
void put_conv(wlk_engine* e, void* dst, const float* host, int c_out, int c_in) {
    const size_t n = (size_t)c_out * c_in * 3;
    float* s = stage_reserve(e, 2 * n);                         // second half: the packed fp32 copy
    CUDA_CHECK(cudaMemcpyAsync(s, host, n * 4, cudaMemcpyHostToDevice, e->st));
    if (e->wt == DT_BF16X2) {
        pack_conv_weight(s, s + n, DT_F32, c_out, c_in, e->st);
        store_mat(e, dst, n, 0, s + n, n);
    } else {
        pack_conv_weight(s, dst, e->wt, c_out, c_in, e->st);
        CUDA_CHECK(cudaStreamSynchronize(e->st));
    }
}

int64_t numel(const int64_t* shape, int ndim) {
    int64_t n = 1;
    for (int i = 0; i < ndim; ++i) n *= shape[i];
    return n;
}

void load_tensor(wlk_engine* e, const std::string& name, const float* host, const int64_t* shape, int ndim) {
    const wlk_dims& D = e->dims;
    Weights& W = e->w;
    const int d = D.n_audio_state, dt = D.n_text_state;
    const size_t es = e->es();
    const int64_t n = numel(shape, ndim);
    auto expect = [&](int64_t want) {
        WLK_CHECK(n == want, "tensor %s has %lld elements, expected %lld", name.c_str(), (long long)n, (long long)want);
    };
    if (name == "mel_filters") {
        expect((int64_t)D.n_mels * N_FREQ);
        std::vector<float> t((size_t)n);
        for (int m = 0; m < D.n_mels; ++m)
            for (int k = 0; k < N_FREQ; ++k) t[(size_t)k * D.n_mels + m] = host[(size_t)m * N_FREQ + k];
        put_f32(e, W.filtT, t.data(), n);
        std::vector<int2> span(D.n_mels);                     // non-zero span of every (triangular) filter
        for (int m = 0; m < D.n_mels; ++m) {
            int lo = N_FREQ, hi = 0;
            for (int k = 0; k < N_FREQ; ++k)
                if (host[(size_t)m * N_FREQ + k] != 0.f) { if (k < lo) lo = k; hi = k + 1; }
            if (lo >= hi) { lo = 0; hi = 0; }
            span[m] = make_int2(lo, hi);
        }
        CUDA_CHECK(cudaMemcpyAsync(W.filt_span, span.data(), span.size() * 8, cudaMemcpyHostToDevice, e->st));
        CUDA_CHECK(cudaStreamSynchronize(e->st));
    } else if (name == "hann_window") {
        expect(N_FFT);
        put_f32(e, W.window, host, n);
    } else if (name == "encoder.conv1.weight") {
        expect((int64_t)d * D.n_mels * 3);
        put_conv(e, W.Wc1, host, d, D.n_mels);
    } else if (name == "encoder.conv2.weight") {
        expect((int64_t)d * d * 3);
        put_conv(e, W.Wc2, host, d, d);
    } else if (name == "encoder.conv1.bias") { expect(d); put_f32(e, W.bc1, host, n);
    } else if (name == "encoder.conv2.bias") { expect(d); put_f32(e, W.bc2, host, n);
    } else if (name == "encoder.positional_embedding") { expect((int64_t)D.n_audio_ctx * d); put_f32(e, W.enc_pos, host, n);
    } else if (name == "encoder.ln_post.weight") { expect(d); put_f32(e, W.lnpw, host, n);
    } else if (name == "encoder.ln_post.bias") { expect(d); put_f32(e, W.lnpb, host, n);
    } else if (name == "decoder.token_embedding.weight") {
        expect((int64_t)D.n_vocab * dt);
        put_f32(e, W.emb_f32, host, n);
        if (e->wt != DT_F32) store_mat(e, W.emb_act, (size_t)n, 0, W.emb_f32, (size_t)n);
    } else if (name == "decoder.positional_embedding") { expect((int64_t)D.n_text_ctx * dt); put_f32(e, W.dec_pos, host, n);
    } else if (name == "decoder.ln.weight") { expect(dt); put_f32(e, W.lnw, host, n);
    } else if (name == "decoder.ln.bias") { expect(dt); put_f32(e, W.lnb, host, n);
    } else if (name.rfind("encoder.blocks.", 0) == 0 || name.rfind("decoder.blocks.", 0) == 0) {
        const bool is_dec = name[0] == 'd';
        size_t p0 = strlen("encoder.blocks.");
        size_t p1 = name.find('.', p0);
        int li = std::stoi(name.substr(p0, p1 - p0));
        std::string rest = name.substr(p1 + 1);
        const int dm = is_dec ? dt : d;
        WLK_CHECK(li >= 0 && li < (is_dec ? D.n_text_layer : D.n_audio_layer), "layer index out of range in %s", name.c_str());
        if (!is_dec) {
            EncLayerW& L = W.enc[li];
            if (rest == "attn.query.weight") { expect((int64_t)dm * dm); put_mat(e, L.Wqkv, (size_t)3 * dm * dm, 0, host, n); }
            else if (rest == "attn.key.weight") { expect((int64_t)dm * dm); put_mat(e, L.Wqkv, (size_t)3 * dm * dm, (size_t)dm * dm, host, n); }
            else if (rest == "attn.value.weight") { expect((int64_t)dm * dm); put_mat(e, L.Wqkv, (size_t)3 * dm * dm, (size_t)2 * dm * dm, host, n); }
            else if (rest == "attn.query.bias") { expect(dm); put_f32(e, L.bqkv, host, n); }
            else if (rest == "attn.value.bias") { expect(dm); put_f32(e, L.bqkv + 2 * dm, host, n); }
            else if (rest == "attn.out.weight") { expect((int64_t)dm * dm); put_mat(e, L.Wo, (size_t)dm * dm, 0, host, n); }
            else if (rest == "attn.out.bias") { expect(dm); put_f32(e, L.bo, host, n); }
            else if (rest == "attn_ln.weight") { expect(dm); put_f32(e, L.ln1w, host, n); }
            else if (rest == "attn_ln.bias") { expect(dm); put_f32(e, L.ln1b, host, n); }
            else if (rest == "mlp.0.weight") { expect((int64_t)4 * dm * dm); put_mat(e, L.W1, (size_t)4 * dm * dm, 0, host, n); }
            else if (rest == "mlp.0.bias") { expect(4 * dm); put_f32(e, L.b1, host, n); }
            else if (rest == "mlp.2.weight") { expect((int64_t)4 * dm * dm); put_mat(e, L.W2, (size_t)4 * dm * dm, 0, host, n); }
            else if (rest == "mlp.2.bias") { expect(dm); put_f32(e, L.b2, host, n); }
            else if (rest == "mlp_ln.weight") { expect(dm); put_f32(e, L.ln2w, host, n); }
            else if (rest == "mlp_ln.bias") { expect(dm); put_f32(e, L.ln2b, host, n); }
            else WLK_CHECK(false, "unknown tensor %s", name.c_str());
        } else {
            DecLayerW& L = W.dec[li];
            const size_t xrow = (size_t)li * 2 * dt;      // row offset inside Wxkv / bxkv
            if (rest == "attn.query.weight") { expect((int64_t)dm * dm); put_mat(e, L.Wqkv, (size_t)3 * dm * dm, 0, host, n); }
            else if (rest == "attn.key.weight") { expect((int64_t)dm * dm); put_mat(e, L.Wqkv, (size_t)3 * dm * dm, (size_t)dm * dm, host, n); }
            else if (rest == "attn.value.weight") { expect((int64_t)dm * dm); put_mat(e, L.Wqkv, (size_t)3 * dm * dm, (size_t)2 * dm * dm, host, n); }
            else if (rest == "attn.query.bias") { expect(dm); put_f32(e, L.bqkv, host, n); }
            else if (rest == "attn.value.bias") { expect(dm); put_f32(e, L.bqkv + 2 * dm, host, n); }
            else if (rest == "attn.out.weight") { expect((int64_t)dm * dm); put_mat(e, L.Wo, (size_t)dm * dm, 0, host, n); }
            else if (rest == "attn.out.bias") { expect(dm); put_f32(e, L.bo, host, n); }
            else if (rest == "attn_ln.weight") { expect(dm); put_f32(e, L.ln1w, host, n); }
            else if (rest == "attn_ln.bias") { expect(dm); put_f32(e, L.ln1b, host, n); }
            else if (rest == "cross_attn.query.weight") { expect((int64_t)dm * dm); put_mat(e, L.Wqc, (size_t)dm * dm, 0, host, n); }
            else if (rest == "cross_attn.query.bias") { expect(dm); put_f32(e, L.bqc, host, n); }
            else if (rest == "cross_attn.key.weight") { expect((int64_t)dt * d); put_mat(e, W.Wxkv, (size_t)D.n_text_layer * 2 * dt * d, xrow * d, host, n); }
            else if (rest == "cross_attn.value.weight") { expect((int64_t)dt * d); put_mat(e, W.Wxkv, (size_t)D.n_text_layer * 2 * dt * d, (xrow + dt) * d, host, n); }
            else if (rest == "cross_attn.value.bias") { expect(dt); put_f32(e, W.bxkv + xrow + dt, host, n); }
            else if (rest == "cross_attn.out.weight") { expect((int64_t)dm * dm); put_mat(e, L.Woc, (size_t)dm * dm, 0, host, n); }
            else if (rest == "cross_attn.out.bias") { expect(dm); put_f32(e, L.boc, host, n); }
            else if (rest == "cross_attn_ln.weight") { expect(dm); put_f32(e, L.lncw, host, n); }
            else if (rest == "cross_attn_ln.bias") { expect(dm); put_f32(e, L.lncb, host, n); }
            else if (rest == "mlp.0.weight") { expect((int64_t)4 * dm * dm); put_mat(e, L.W1, (size_t)4 * dm * dm, 0, host, n); }
            else if (rest == "mlp.0.bias") { expect(4 * dm); put_f32(e, L.b1, host, n); }
            else if (rest == "mlp.2.weight") { expect((int64_t)4 * dm * dm); put_mat(e, L.W2, (size_t)4 * dm * dm, 0, host, n); }
            else if (rest == "mlp.2.bias") { expect(dm); put_f32(e, L.b2, host, n); }
            else if (rest == "mlp_ln.weight") { expect(dm); put_f32(e, L.ln2w, host, n); }
            else if (rest == "mlp_ln.bias") { expect(dm); put_f32(e, L.ln2b, host, n); }
            else WLK_CHECK(false, "unknown tensor %s", name.c_str());
        }
    } else {
        WLK_CHECK(false, "unknown tensor %s", name.c_str());
    }
    e->loaded.insert(name);
}

std::vector<std::string> required_tensors(const wlk_dims& D) {
    std::vector<std::string> r = {"mel_filters", "hann_window", "encoder.conv1.weight", "encoder.conv1.bias",
                                  "encoder.conv2.weight", "encoder.conv2.bias", "encoder.positional_embedding",
                                  "encoder.ln_post.weight", "encoder.ln_post.bias", "decoder.token_embedding.weight",
                                  "decoder.positional_embedding", "decoder.ln.weight", "decoder.ln.bias"};
    const char* att[] = {"query.weight", "query.bias", "key.weight", "value.weight", "value.bias", "out.weight", "out.bias"};
    const char* com[] = {"attn_ln.weight", "attn_ln.bias", "mlp.0.weight", "mlp.0.bias", "mlp.2.weight", "mlp.2.bias",
                         "mlp_ln.weight", "mlp_ln.bias"};
    for (int l = 0; l < D.n_audio_layer; ++l) {
        std::string p = "encoder.blocks." + std::to_string(l) + ".";
        for (auto a : att) r.push_back(p + "attn." + a);
        for (auto c : com) r.push_back(p + c);
    }
    for (int l = 0; l < D.n_text_layer; ++l) {
        std::string p = "decoder.blocks." + std::to_string(l) + ".";
        for (auto a : att) { r.push_back(p + "attn." + a); r.push_back(p + "cross_attn." + a); }
        for (auto c : com) r.push_back(p + c);
        r.push_back(p + "cross_attn_ln.weight"); r.push_back(p + "cross_attn_ln.bias");
    }
    return r;
}

// ---------------------------------------------------------------------------------------
// GEMM dispatch
// ---------------------------------------------------------------------------------------
void run_gemm(wlk_engine* e, GemmArgs& g, int cls) {
    ProfScope ps(e, cls, 2.0 * g.M * (double)g.N * g.K,
                 (double)g.M * g.K * dtype_size(g.a_type) + (double)g.N * g.K * dtype_size(g.w_type) +
                     (double)g.M * g.N * dtype_size(g.epi.c_type));
    g.sk_scratch = e->sk_scratch; g.sk_scratch_floats = SK_SCRATCH_FLOATS;
    g.sk_counters = e->sk_counters; g.sk_max_tiles = SK_MAX_TILES;
    if (e->wt == DT_BF16X2) {
        // every weight matrix is one whole [N, ldw] allocation: the lo plane sits right behind the hi plane
        g.W_lo = reinterpret_cast<const bf16*>(g.W) + (size_t)g.N * g.ldw;
        g.a_split = e->a_split; g.a_split_elems = e->a_split_elems;
        std::string why;
        WLK_CHECK(gemm_tcgen05_supported(g, &why), "bf16x3 GEMM (M=%d N=%d K=%d): %s", g.M, g.N, g.K, why.c_str());
        gemm_tcgen05(g, e->st, e->num_sms);
        return;
    }
    bool tc = e->gemm_backend == WLK_BACKEND_TCGEN05 && gemm_tcgen05_supported(g, nullptr);
    if (tc) gemm_tcgen05(g, e->st, e->num_sms);
    else gemm_simt(g, e->st);
}

// ---------------------------------------------------------------------------------------
// staging: a pinned host block mirrored on the device, carved per call
// ---------------------------------------------------------------------------------------
struct Stager {
    wlk_engine* e; size_t used = 0;
    explicit Stager(wlk_engine* e_) : e(e_) { CUDA_CHECK(cudaEventSynchronize(e->stg_done)); }
    template <typename T> T* host(size_t count, T** dev) {
        size_t off = (used + 255) / 256 * 256;
        size_t bytes = count * sizeof(T);
        WLK_CHECK(off + bytes <= e->stg_bytes, "staging buffer overflow (%zu + %zu > %zu)", off, bytes, e->stg_bytes);
        used = off + bytes;
        *dev = reinterpret_cast<T*>(e->stg_dev + off);
        return reinterpret_cast<T*>(e->stg_host + off);
    }
    void upload() {
        if (used) CUDA_CHECK(cudaMemcpyAsync(e->stg_dev, e->stg_host, used, cudaMemcpyHostToDevice, e->st));
        CUDA_CHECK(cudaEventRecord(e->stg_done, e->st));
    }
};

Session& get_session(wlk_engine* e, int32_t sid) {
    WLK_CHECK(sid >= 0 && sid < (int)e->sess.size() && e->sess[sid].open, "invalid session id %d", sid);
    return e->sess[sid];
}
// the session whose encoder output / cross-K/V / content length `s` decodes against (itself unless a beam fork)
Session& enc_owner(wlk_engine* e, Session& s) { return s.parent >= 0 ? e->sess[s.parent] : s; }
Session& get_root_session(wlk_engine* e, int32_t sid, const char* what) {
    Session& s = get_session(e, sid);
    WLK_CHECK(s.parent < 0, "session %d is a beam fork of session %d: %s belongs to the parent", sid, s.parent, what);
    return s;
}

// ---------------------------------------------------------------------------------------
// encode: log-mel -> conv stem -> L encoder blocks -> ln_post -> cross-K/V for every decoder layer
// ---------------------------------------------------------------------------------------
void run_encoder(wlk_engine* e, const int32_t* sids, int n, void** xkv_dev);

// One session's log-mel job (shared by the parity and the incremental encode): fills `mj`, moves the reusable raw rows of
// the incremental log-mel, sets s.content_len.
void fill_mel_job(wlk_engine* e, Session& s, MelJob& mj, int i, int& max_frames) {
    const int nm = e->dims.n_mels;
    const size_t es = e->es();
    const int64_t N = s.audio_len;
    const int64_t n_total = (N + 480000) / HOP;                 // torch.stft frames minus the dropped last one
    int64_t n_compute = (N + 199) / HOP + 1;                   // frames whose window overlaps [0, N): all of them
    if (n_compute > MEL_MAX_FRAMES) n_compute = MEL_MAX_FRAMES; // join the global max, also beyond the 30 s kept
    if (n_compute > max_frames) max_frames = (int)n_compute;
    mj.audio = s.audio; mj.raw = s.mel_raw; mj.blockmax = s.mel_blockmax;
    mj.out = offs(e->mel_t, (size_t)i * MEL_ROWS * nm, es);
    mj.n = (int32_t)N; mj.n_compute = (int32_t)n_compute; mj.n_total = (int32_t)n_total; mj.pad = 0;
    mj.keep_lo = mj.keep_hi = 0;
    // Incremental log-mel (exact).  Frame f of the window reads samples [160 f - 200, 160 f + 200).  After the window
    // slid by d = mel_dropped / 160 whole frames and grew at the end, new frame f equals old frame f + d bit for bit
    // as long as neither touches an edge: f >= 2 (no reflection at the new left edge; f + d >= 2 follows) and
    // 160 f + 200 <= old end (the old pass saw the same samples, not the zero padding).  Those rows are moved, the
    // two leading frames and the ~50 trailing ones are recomputed.
    if (e->mel_incremental && s.mel_n >= 0 && s.mel_dropped % HOP == 0 && s.mel_dropped <= s.mel_n &&
        n_compute <= MEL_STORE_FRAMES && (s.mel_n + 199) / HOP + 1 <= MEL_STORE_FRAMES) {
        const int64_t d = s.mel_dropped / HOP;
        const int64_t old_end = s.mel_n - s.mel_dropped;                   // old audio end in new coordinates
        const int64_t lo = d == 0 ? 0 : 2;
        int64_t hi = old_end >= 200 ? (old_end - 200) / HOP + 1 : 0;       // exclusive
        if (hi > n_compute) hi = n_compute;
        if (hi > lo) {
            if (d > 0) {
                const size_t bytes = (size_t)(hi - lo) * nm * 4;
                CUDA_CHECK(cudaMemcpyAsync(e->mel_scratch, s.mel_raw + (size_t)(lo + d) * nm, bytes, cudaMemcpyDeviceToDevice, e->st));
                CUDA_CHECK(cudaMemcpyAsync(s.mel_raw + (size_t)lo * nm, e->mel_scratch, bytes, cudaMemcpyDeviceToDevice, e->st));
            }
            mj.keep_lo = (int32_t)lo; mj.keep_hi = (int32_t)hi;
        }
    }
    s.mel_n = N; s.mel_dropped = 0;
    s.content_len = (int)((n_total - N_FRAMES) / 2);            // simul_whisper.py:350 (unclamped: the policy's
}                                                               // frame_threshold test needs the true value)

void encode_batch(wlk_engine* e, const int32_t* sids, int n, int32_t* content_out) {
    const wlk_dims& D = e->dims;
    Weights& W = e->w;
    const int nm = D.n_mels;
    const size_t es = e->es();
    WLK_CHECK(n >= 1 && n <= e->cfg.max_batch, "encode batch %d outside [1, %d]", n, e->cfg.max_batch);
    // first pass: validation only (no session state is touched until the whole batch is known to be good)
    for (int i = 0; i < n; ++i) {
        Session& s = get_root_session(e, sids[i], "encode");
        WLK_CHECK(s.audio_len > 0, "session %d has no audio", sids[i]);
        for (int j = 0; j < i; ++j) WLK_CHECK(sids[j] != sids[i], "session %d appears twice in the batch", sids[i]);
    }
    Stager sg(e);
    MelJob* mj_dev; MelJob* mj = sg.host<MelJob>(n, &mj_dev);
    void** xkv_dev; void** xkv = sg.host<void*>(n, &xkv_dev);
    int max_frames = 1;
    for (int i = 0; i < n; ++i) {
        Session& s = e->sess[sids[i]];
        fill_mel_job(e, s, mj[i], i, max_frames);
        content_out[i] = s.content_len;
        xkv[i] = s.cross_kv;
    }
    sg.upload();

    {   ProfScope ps(e, WLK_KC_MEL, 0, (double)n * (480000.0 * 4 + 3000.0 * nm * es));
        mel_forward(mj_dev, n, nm, W.filtT, W.window, W.twiddle, W.filt_span, e->act, max_frames, e->st); }
    run_encoder(e, sids, n, xkv_dev);
}

// conv stem -> L encoder blocks -> ln_post -> cross-K/V, from the time-major mel of `n` streams in e->mel_t
void run_encoder(wlk_engine* e, const int32_t* sids, int n, void** xkv_dev) {
    const wlk_dims& D = e->dims;
    Weights& W = e->w;
    const int d = D.n_audio_state, dt = D.n_text_state, nm = D.n_mels;
    const size_t es = e->es();

    // conv1 (k=3, pad=1) as a GEMM over overlapping rows of the time-major mel: row t = frames t-1..t+1
    {   GemmArgs g;
        g.A = e->mel_t; g.a_type = e->act; g.lda = nm;
        g.W = W.Wc1; g.w_type = e->wt; g.ldw = 3 * nm;
        g.M = n * MEL_ROWS - 2; g.N = d; g.K = 3 * nm;
        g.epi.bias = W.bc1; g.epi.gelu = 1;
        g.epi.C = offs(e->h1, (size_t)d, es); g.epi.c_type = e->act; g.epi.ldc = d;
        run_gemm(e, g, WLK_KC_GEMM_ENC);
        zero_rows(e->h1, e->act, d, e->pad_rows_dev, 2 * n, e->st); }
    // conv2 (k=3, stride 2, pad=1): row t = padded rows 2t..2t+2 -> pitch 2d, then GELU and + positional
    {   GemmArgs g;
        g.A = e->h1; g.a_type = e->act; g.lda = 2 * d;
        g.W = W.Wc2; g.w_type = e->wt; g.ldw = 3 * d;
        g.M = n * (N_CTX + 1) - 1; g.N = d; g.K = 3 * d;
        g.epi.bias = W.bc2; g.epi.gelu = 1; g.epi.residual = W.enc_pos; g.epi.ldr = d;
        g.epi.mode = EPI_ROWPTR; g.epi.batch_ptrs = e->xptrs_dev; g.epi.rows_per_batch = N_CTX + 1;
        g.epi.rows_valid = N_CTX; g.epi.c_type = DT_F32; g.epi.ldc = d;
        run_gemm(e, g, WLK_KC_GEMM_ENC); }

    const int M = n * N_CTX;
    const float qk_scale = powf(64.0f, -0.25f);                     // model.py:152
    for (int li = 0; li < D.n_audio_layer; ++li) {
        EncLayerW& L = W.enc[li];
        {   ProfScope ps(e, WLK_KC_LN, 0, (double)M * d * (4 + es));
            layernorm(e->x, d, L.ln1w, L.ln1b, e->xn, e->act, d, M, d, nullptr, e->st); }
        {   GemmArgs g;
            g.A = e->xn; g.a_type = e->act; g.lda = d; g.W = L.Wqkv; g.w_type = e->wt; g.ldw = d;
            g.M = M; g.N = 3 * d; g.K = d;
            g.epi.bias = L.bqkv; g.epi.col_scale = qk_scale; g.epi.scale_cols = 2 * d;
            g.epi.C = e->qkv; g.epi.c_type = e->act; g.epi.ldc = 3 * d;
            run_gemm(e, g, WLK_KC_GEMM_ENC); }
        {   ProfScope ps(e, WLK_KC_ATTN_ENC, 4.0 * n * D.n_audio_head * (double)N_CTX * N_CTX * 64,
                         (double)M * 4 * d * es);
            if (e->attn_backend == WLK_BACKEND_TCGEN05 && e->wt == DT_BF16X2) {
                // split the fp32 q|k|v into (hi, lo) planes (the GEMM operand scratch is idle between GEMMs)
                bf16* hi = reinterpret_cast<bf16*>(e->a_split);
                bf16* lo = hi + e->a_split_elems;
                split_f32_planes_async(reinterpret_cast<const float*>(e->qkv), hi, lo, (int64_t)M * 3 * d, e->st);
                enc_attention_tcgen05_x3(hi, lo, n, D.n_audio_head, d, reinterpret_cast<float*>(e->att), e->st);
            } else if (e->attn_backend == WLK_BACKEND_TCGEN05)
                enc_attention_tcgen05(e->qkv, n, D.n_audio_head, d, e->att, e->st, e->num_sms);
            else
                enc_attention_simt(e->qkv, e->act, n, D.n_audio_head, d, e->att, e->st); }
        {   GemmArgs g;
            g.A = e->att; g.a_type = e->act; g.lda = d; g.W = L.Wo; g.w_type = e->wt; g.ldw = d;
            g.M = M; g.N = d; g.K = d;
            g.epi.bias = L.bo; g.epi.residual = e->x; g.epi.ldr = d;
            g.epi.C = e->x; g.epi.c_type = DT_F32; g.epi.ldc = d;
            run_gemm(e, g, WLK_KC_GEMM_ENC); }
        {   ProfScope ps(e, WLK_KC_LN, 0, (double)M * d * (4 + es));
            layernorm(e->x, d, L.ln2w, L.ln2b, e->xn, e->act, d, M, d, nullptr, e->st); }
        {   GemmArgs g;
            g.A = e->xn; g.a_type = e->act; g.lda = d; g.W = L.W1; g.w_type = e->wt; g.ldw = d;
            g.M = M; g.N = 4 * d; g.K = d;
            g.epi.bias = L.b1; g.epi.gelu = 1;
            g.epi.C = e->hid; g.epi.c_type = e->act; g.epi.ldc = 4 * d;
            run_gemm(e, g, WLK_KC_GEMM_ENC); }
        {   GemmArgs g;
            g.A = e->hid; g.a_type = e->act; g.lda = 4 * d; g.W = L.W2; g.w_type = e->wt; g.ldw = 4 * d;
            g.M = M; g.N = d; g.K = 4 * d;
            g.epi.bias = L.b2; g.epi.residual = e->x; g.epi.ldr = d;
            g.epi.C = e->x; g.epi.c_type = DT_F32; g.epi.ldc = d;
            run_gemm(e, g, WLK_KC_GEMM_ENC); }
    }
    {   ProfScope ps(e, WLK_KC_LN, 0, (double)M * d * (4 + es));
        layernorm(e->x, d, W.lnpw, W.lnpb, e->xn, e->act, d, M, d, nullptr, e->st); }
    for (int i = 0; i < n; ++i) {
        Session& s = e->sess[sids[i]];
        CUDA_CHECK(cudaMemcpyAsync(s.xa, offs(e->xn, (size_t)i * N_CTX * d, es), (size_t)N_CTX * d * es,
                                   cudaMemcpyDeviceToDevice, e->st));
    }
    // cross-attention K/V of every decoder layer in one GEMM, scattered head-major into each session
    {   GemmArgs g;
        g.A = e->xn; g.a_type = e->act; g.lda = d; g.W = W.Wxkv; g.w_type = e->wt; g.ldw = d;
        g.M = M; g.N = D.n_text_layer * 2 * dt; g.K = d;
        g.epi.bias = W.bxkv; g.epi.col_scale = qk_scale; g.epi.scale_cols = dt; g.epi.scale_period = 2 * dt;
        g.epi.mode = EPI_XKV; g.epi.batch_ptrs = xkv_dev; g.epi.rows_per_batch = N_CTX;
        g.epi.n_head = D.n_text_head; g.epi.d_model = dt; g.epi.kv_len = N_CTX; g.epi.c_type = e->act;
        run_gemm(e, g, WLK_KC_GEMM_XKV); }
    for (int i = 0; i < n; ++i) {
        Session& s = e->sess[sids[i]];
        s.self_len = 0; s.align_rows = 0; s.iter_row_start.clear(); s.encoded = true;
        s.inc_valid = false; s.rot = 0;                  // the parity encode writes every buffer in logical order
        if (s.n_forks)                                   // a new epoch for the beams of this stream as well
            for (auto& f : e->sess)
                if (f.open && f.parent == sids[i]) { f.self_len = 0; f.align_rows = 0; f.iter_row_start.clear(); }
    }
}

// ---------------------------------------------------------------------------------------
// Incremental encoder -- LABELLED APPROXIMATE (north_star item 2: "KV retained across chunk extensions so only the
// appended frames are re-encoded"; SURVEY.md section 7 H1 explains why this cannot equal the reference's full re-encode:
// Whisper's encoder is bidirectional, so new audio changes every position's output from layer 1 on).
//   * every encoder layer's K/V of a stream is retained ([L][2][H][1500][64], like the cross-K/V);
//   * per chunk only a BLOCK of positions runs through the conv stem and the layers: the two positions left of the old
//     content end (conv receptive field), the new content and two positions of padding behind it -- ~29 rows instead of
//     1500; the block attends to all 1500 slots: the retained K/V of everything outside the block (frozen as computed when
//     those positions were last in a block) and the block's own fresh K/V (written by the QKV GEMM's scatter epilogue first);
//   * the first encode of a stream (and every `inc_refresh`-th, and whenever the bookkeeping does not fit) takes the whole
//     window as its block: that IS the parity computation (same kernels as the decoder's cross-attention prefill);
//   * when the window slides by whole positions the buffers are not moved: position p lives in ring slot (p + rot) % 1500,
//     rot advances by the dropped positions, and the vacated slots -- now the logical tail -- join the block.  Attention is
//     order-free over keys; the two consumers of frame ORDER (the median-7 / argmax of the alignment reduction) read
//     through `rot`.  Positional embeddings are taken by slot: a frame keeps the embedding it was encoded with, frames
//     stay cyclically ordered, the wrap point travels through the window (the approximation's second source of error).
// Evaluated by token / attended-frame agreement against the parity mode (tests/test_gpu_incremental.py, bench.py).
// ---------------------------------------------------------------------------------------
void ensure_incremental(wlk_engine* e, Session& s, int sid) {
    const wlk_dims& D = e->dims;
    if (!e->enc_maps_dev) {
        size_t* acct = &e->bytes_workspace;
        e->enc_maps_dev = reinterpret_cast<uint8_t*>(dmalloc_bytes((size_t)e->cfg.max_sessions * 128, acct));
        std::vector<int32_t> none((size_t)D.n_audio_layer * D.n_audio_head, -1);
        e->enc_norank_dev = dmalloc<int32_t>(e, none.size(), acct);
        CUDA_CHECK(cudaMemcpy(e->enc_norank_dev, none.data(), none.size() * 4, cudaMemcpyHostToDevice));
        e->inc_row_slot = dmalloc<int32_t>(e, (size_t)e->cfg.max_batch * N_CTX, acct);
        e->inc_row_pos = dmalloc<int32_t>(e, (size_t)e->cfg.max_batch * N_CTX, acct);
        const char* v = getenv("WLK_INC_REFRESH");
        e->inc_refresh = v ? atoi(v) : 0;
    }
    if (!s.enc_kv) {
        const size_t bytes = (size_t)D.n_audio_layer * 2 * N_CTX * D.n_audio_state * e->es();
        s.enc_kv = dmalloc_bytes(bytes, &s.bytes);
        e->bytes_sessions += bytes;
        CUDA_CHECK(cudaMemsetAsync(s.enc_kv, 0, bytes, e->st));
        alignas(64) uint8_t tmap[128];
        make_cross_kv_tmap(tmap, s.enc_kv, D.n_audio_layer, D.n_audio_head);
        CUDA_CHECK(cudaMemcpy(e->enc_maps_dev + (size_t)sid * 128, tmap, 128, cudaMemcpyHostToDevice));
        s.inc_valid = false;
    }
}

void encode_incremental(wlk_engine* e, const int32_t* sids, int n, int32_t* content_out, int32_t* block_rows_out) {
    const wlk_dims& D = e->dims;
    Weights& W = e->w;
    const int d = D.n_audio_state, dt = D.n_text_state, nm = D.n_mels, H = D.n_audio_head;
    const size_t es = e->es();
    WLK_CHECK(e->act == DT_BF16 && e->wt == DT_BF16 && e->attn_backend == WLK_BACKEND_TCGEN05 && e->gemm_backend == WLK_BACKEND_TCGEN05,
              "the incremental encoder runs in the bf16 tcgen05 mode only");
    WLK_CHECK(n >= 1 && n <= e->cfg.max_batch, "encode batch %d outside [1, %d]", n, e->cfg.max_batch);
    for (int i = 0; i < n; ++i) {
        Session& s = get_root_session(e, sids[i], "encode");
        WLK_CHECK(s.audio_len > 0, "session %d has no audio", sids[i]);
        for (int j = 0; j < i; ++j) WLK_CHECK(sids[j] != sids[i], "session %d appears twice in the batch", sids[i]);
    }
    for (int i = 0; i < n; ++i) ensure_incremental(e, e->sess[sids[i]], sids[i]);

    Stager sg(e);
    MelJob* mj_dev; MelJob* mj = sg.host<MelJob>(n, &mj_dev);
    IncJob* ij_dev; IncJob* ij = sg.host<IncJob>(n, &ij_dev);
    DecJob* dj_dev; DecJob* dj = sg.host<DecJob>(n, &dj_dev);
    void** ekv_dev; void** ekv = sg.host<void*>(n, &ekv_dev);
    void** xkv_dev; void** xkv = sg.host<void*>(n, &xkv_dev);
    int max_frames = 1, R = 0, R1 = 0, max_rows = 0;
    std::vector<int> new_rot(n), new_chunks(n);
    for (int i = 0; i < n; ++i) {
        Session& s = e->sess[sids[i]];
        fill_mel_job(e, s, mj[i], i, max_frames);
        content_out[i] = s.content_len;
        const int C = std::min(s.content_len, N_CTX);
        int p0 = 0, p1 = N_CTX, rot = 0, chunks = 0;
        const bool whole = !s.inc_valid || s.inc_dropped % 320 != 0 || s.inc_dropped / 320 > s.inc_content ||
                           (e->inc_refresh > 0 && s.inc_chunks + 1 >= e->inc_refresh);
        if (!whole) {
            const int dpos = (int)(s.inc_dropped / 320);
            rot = (s.rot + dpos) % N_CTX;
            const int old_end = s.inc_content - dpos;                      // old content end in the new coordinates
            p0 = std::max(0, std::min(old_end, C) - 2);
            p1 = dpos > 0 ? N_CTX : std::min(N_CTX, std::max(C, old_end) + 2);   // a slide hands the vacated tail slots to the block
            chunks = s.inc_chunks + 1;
        }
        new_rot[i] = rot; new_chunks[i] = chunks;
        const int len = p1 - p0;
        ij[i].mel = mj[i].out; ij[i].xa = s.xa; ij[i].p0 = p0; ij[i].p1 = p1; ij[i].rot = rot;
        ij[i].row1_off = R1; ij[i].row_off = R; ij[i].pad = 0;
        memset(&dj[i], 0, sizeof(DecJob));
        dj[i].row_off = R; dj[i].n_rows = len; dj[i].slot = sids[i];
        ekv[i] = s.enc_kv; xkv[i] = s.cross_kv;
        if (block_rows_out) block_rows_out[i] = len;
        R += len; R1 += 2 * len + 1;
        max_rows = std::max(max_rows, len);
    }
    sg.upload();
    {   ProfScope ps(e, WLK_KC_MEL, 0, (double)n * (480000.0 * 4 + 3000.0 * nm * es));
        mel_forward(mj_dev, n, nm, W.filtT, W.window, W.twiddle, W.filt_span, e->act, max_frames, e->st); }

    // conv stem over the block: gathered operand rows, two ordinary GEMMs
    void* A1 = e->h1; void* H1 = e->qkv; void* A2 = e->hid;
    float* posbuf = reinterpret_cast<float*>(e->h1);                      // A1 is dead once conv1 has run
    {   ProfScope ps(e, WLK_KC_MISC);
        inc_gather_conv1(ij_dev, n, 2 * max_rows + 1, nm, A1, e->act, e->st); }
    {   GemmArgs g;
        g.A = A1; g.a_type = e->act; g.lda = 3 * nm; g.W = W.Wc1; g.w_type = e->wt; g.ldw = 3 * nm;
        g.M = R1; g.N = d; g.K = 3 * nm;
        g.epi.bias = W.bc1; g.epi.gelu = 1; g.epi.C = H1; g.epi.c_type = e->act; g.epi.ldc = d;
        run_gemm(e, g, WLK_KC_GEMM_ENC); }
    {   ProfScope ps(e, WLK_KC_MISC);
        inc_gather_conv2(ij_dev, n, max_rows, d, H1, A2, W.enc_pos, posbuf, e->inc_row_slot, e->inc_row_pos, e->act, e->st); }
    {   GemmArgs g;
        g.A = A2; g.a_type = e->act; g.lda = 3 * d; g.W = W.Wc2; g.w_type = e->wt; g.ldw = 3 * d;
        g.M = R; g.N = d; g.K = 3 * d;
        g.epi.bias = W.bc2; g.epi.gelu = 1; g.epi.residual = posbuf; g.epi.ldr = d;
        g.epi.C = e->x; g.epi.c_type = DT_F32; g.epi.ldc = d;
        run_gemm(e, g, WLK_KC_GEMM_ENC); }

    const float qk_scale = powf(64.0f, -0.25f);
    for (int li = 0; li < D.n_audio_layer; ++li) {
        EncLayerW& L = W.enc[li];
        {   ProfScope ps(e, WLK_KC_LN, 0, (double)R * d * (4 + es));
            layernorm(e->x, d, L.ln1w, L.ln1b, e->xn, e->act, d, R, d, nullptr, e->st); }
        {   GemmArgs g;                                                   // q -> packed rows, k / v -> the ring slots
            g.A = e->xn; g.a_type = e->act; g.lda = d; g.W = L.Wqkv; g.w_type = e->wt; g.ldw = d;
            g.M = R; g.N = 3 * d; g.K = d;
            g.epi.bias = L.bqkv; g.epi.col_scale = qk_scale; g.epi.scale_cols = 2 * d;
            g.epi.mode = EPI_SELF_QKV; g.epi.C = e->qkv; g.epi.ldc = d; g.epi.c_type = e->act;
            g.epi.batch_ptrs = ekv_dev; g.epi.row_slot = e->inc_row_slot; g.epi.row_pos = e->inc_row_pos;
            g.epi.layer = li; g.epi.n_head = H; g.epi.d_model = d; g.epi.kv_len = N_CTX;
            run_gemm(e, g, WLK_KC_GEMM_ENC); }
        {   ProfScope ps(e, WLK_KC_ATTN_ENC, 4.0 * H * (double)R * N_CTX * 64, (double)n * 2 * d * N_CTX * es);
            dec_cross_attention_tcgen05(e->qkv, R, dj_dev, n, max_rows, li, H, d, e->enc_maps_dev, e->enc_norank_dev, e->att, e->st); }
        {   GemmArgs g;
            g.A = e->att; g.a_type = e->act; g.lda = d; g.W = L.Wo; g.w_type = e->wt; g.ldw = d;
            g.M = R; g.N = d; g.K = d;
            g.epi.bias = L.bo; g.epi.residual = e->x; g.epi.ldr = d; g.epi.C = e->x; g.epi.c_type = DT_F32; g.epi.ldc = d;
            run_gemm(e, g, WLK_KC_GEMM_ENC); }
        {   ProfScope ps(e, WLK_KC_LN, 0, (double)R * d * (4 + es));
            layernorm(e->x, d, L.ln2w, L.ln2b, e->xn, e->act, d, R, d, nullptr, e->st); }
        {   GemmArgs g;
            g.A = e->xn; g.a_type = e->act; g.lda = d; g.W = L.W1; g.w_type = e->wt; g.ldw = d;
            g.M = R; g.N = 4 * d; g.K = d;
            g.epi.bias = L.b1; g.epi.gelu = 1; g.epi.C = e->hid; g.epi.c_type = e->act; g.epi.ldc = 4 * d;
            run_gemm(e, g, WLK_KC_GEMM_ENC); }
        {   GemmArgs g;
            g.A = e->hid; g.a_type = e->act; g.lda = 4 * d; g.W = L.W2; g.w_type = e->wt; g.ldw = 4 * d;
            g.M = R; g.N = d; g.K = 4 * d;
            g.epi.bias = L.b2; g.epi.residual = e->x; g.epi.ldr = d; g.epi.C = e->x; g.epi.c_type = DT_F32; g.epi.ldc = d;
            run_gemm(e, g, WLK_KC_GEMM_ENC); }
    }
    {   ProfScope ps(e, WLK_KC_LN, 0, (double)R * d * (4 + es));
        layernorm(e->x, d, W.lnpw, W.lnpb, e->xn, e->act, d, R, d, nullptr, e->st); }
    {   ProfScope ps(e, WLK_KC_MISC);
        inc_scatter_rows(ij_dev, n, max_rows, d, e->xn, e->act, e->st); }
    {   GemmArgs g;                                                       // cross-K/V of the block's rows only
        g.A = e->xn; g.a_type = e->act; g.lda = d; g.W = W.Wxkv; g.w_type = e->wt; g.ldw = d;
        g.M = R; g.N = D.n_text_layer * 2 * dt; g.K = d;
        g.epi.bias = W.bxkv; g.epi.col_scale = qk_scale; g.epi.scale_cols = dt; g.epi.scale_period = 2 * dt;
        g.epi.mode = EPI_XKV; g.epi.batch_ptrs = xkv_dev; g.epi.rows_per_batch = N_CTX;
        g.epi.row_slot = e->inc_row_slot; g.epi.row_pos = e->inc_row_pos;
        g.epi.n_head = D.n_text_head; g.epi.d_model = dt; g.epi.kv_len = N_CTX; g.epi.c_type = e->act;
        run_gemm(e, g, WLK_KC_GEMM_XKV); }
    for (int i = 0; i < n; ++i) {
        Session& s = e->sess[sids[i]];
        s.self_len = 0; s.align_rows = 0; s.iter_row_start.clear(); s.encoded = true;
        s.inc_valid = true; s.rot = new_rot[i]; s.inc_chunks = new_chunks[i];
        s.inc_content = std::min(s.content_len, N_CTX); s.inc_dropped = 0;
        if (s.n_forks)
            for (auto& f : e->sess)
                if (f.open && f.parent == sids[i]) { f.self_len = 0; f.align_rows = 0; f.iter_row_start.clear(); }
    }
}

// ---------------------------------------------------------------------------------------
// decoder attention of one layer over the jobs' caches (decode_batch and wlk_op_decoder_attention): `q` / `out` are
// the packed rows [R][n_text_state] of `type`, max_rows the largest n_rows of a job.  tensor_cores: the bf16 tcgen05
// prefill kernels, which read the caches through the tensor maps at maps_dev[job.slot].
// ---------------------------------------------------------------------------------------
void dec_self_attention_layer(wlk_engine* e, const void* q, int type, int R, const DecJob* jobs_dev, int n, int max_rows,
                              int layer, const void* self_maps_dev, void* out, bool tensor_cores) {
    const wlk_dims& D = e->dims;
    // prefills on the tensor cores (causal, per-session cache planes through TMA); token steps and the fp32 modes on
    // the SIMT kernel
    if (tensor_cores)
        dec_self_attention_tcgen05(q, R, jobs_dev, n, max_rows, layer, D.n_text_head, D.n_text_state, D.n_text_ctx,
                                   self_maps_dev, out, e->st);
    else
        dec_self_attention(q, type, jobs_dev, n, layer, D.n_text_head, D.n_text_state, D.n_text_ctx, out, max_rows, e->st);
}
void dec_cross_attention_layer(wlk_engine* e, const void* q, int type, int R, const DecJob* jobs_dev, int n, int max_rows,
                               int layer, const void* cross_maps_dev, void* out, bool tensor_cores) {
    const wlk_dims& D = e->dims;
    if (tensor_cores)     // all non-alignment heads on the tensor cores; alignment heads need the exported rows
        dec_cross_attention_tcgen05(q, R, jobs_dev, n, max_rows, layer, D.n_text_head, D.n_text_state, cross_maps_dev,
                                    e->align_rank_dev, out, e->st);
    dec_cross_attention(q, type, jobs_dev, n, layer, D.n_text_head, D.n_text_state, D.n_text_ctx, e->align_rank_dev, out,
                        max_rows, tensor_cores, e->st);
}

// ---------------------------------------------------------------------------------------
// decode: one TextDecoder.forward over packed rows of several sessions
// ---------------------------------------------------------------------------------------
void decode_batch(wlk_engine* e, const int32_t* sids, int n, const int32_t* tokens, const int32_t* offsets,
                  int32_t sot_index, float* all_logits_dev = nullptr) {
    const wlk_dims& D = e->dims;
    Weights& W = e->w;
    const int dt = D.n_text_state, H = D.n_text_head, ctx = D.n_text_ctx;
    const size_t es = e->es();
    WLK_CHECK(n >= 1 && n <= e->cfg.max_batch, "decode batch %d outside [1, %d]", n, e->cfg.max_batch);
    const int R = offsets[n] - offsets[0];
    WLK_CHECK(R >= n && R <= e->dec_rows_max, "decode rows %d outside [%d, %d]", R, n, e->dec_rows_max);

    Stager sg(e);
    DecJob* dj_dev; DecJob* dj = sg.host<DecJob>(n, &dj_dev);
    int32_t *tok_dev, *pos_dev, *slot_dev, *sel_dev;
    int32_t* tok = sg.host<int32_t>(R, &tok_dev);
    int32_t* pos = sg.host<int32_t>(R, &pos_dev);
    int32_t* slot = sg.host<int32_t>(R, &slot_dev);
    int32_t* sel = sg.host<int32_t>(2 * n, &sel_dev);
    void** skv_dev; void** skv = sg.host<void*>(n, &skv_dev);
    void** lptr_dev; void** lptr = sg.host<void*>(2 * n, &lptr_dev);
    int n_sel = 0, r = 0, max_tq = 0;
    for (int i = 0; i < n; ++i) {
        Session& s = get_session(e, sids[i]);
        for (int j = 0; j < i; ++j) WLK_CHECK(sids[j] != sids[i], "session %d appears twice in the batch", sids[i]);
        WLK_CHECK(enc_owner(e, s).encoded, "session %d: decode before encode", sids[i]);
        const int tq = offsets[i + 1] - offsets[i];
        WLK_CHECK(tq >= 1, "session %d: empty token list", sids[i]);
        if (tq > max_tq) max_tq = tq;
        WLK_CHECK(s.self_len + tq <= ctx, "session %d: %d + %d tokens exceed n_text_ctx %d", sids[i], s.self_len, tq, ctx);
        const bool first = s.iter_row_start.empty();
        if (first) WLK_CHECK(sot_index >= 0 && sot_index < tq, "sot_index %d outside the %d fed tokens", sot_index, tq);
        dj[i].self_kv = s.self_kv; dj[i].cross_kv = enc_owner(e, s).cross_kv; dj[i].align = s.align;
        dj[i].logits_last = s.logits_last; dj[i].logits_sot = s.logits_sot;
        dj[i].row_off = r; dj[i].n_rows = tq; dj[i].offset = s.self_len; dj[i].align_row0 = s.align_rows;
        dj[i].slot = sids[i]; dj[i].pad0 = dj[i].pad1 = dj[i].pad2 = 0;
        skv[i] = s.self_kv;
        for (int t = 0; t < tq; ++t, ++r) {
            int32_t tk = tokens[offsets[i] - offsets[0] + t];
            WLK_CHECK(tk >= 0 && tk < D.n_vocab, "token %d out of range", tk);
            tok[r] = tk; pos[r] = s.self_len + t; slot[r] = i;
        }
        if (first) { sel[n_sel] = dj[i].row_off + sot_index; lptr[n_sel] = s.logits_sot; ++n_sel; }
        sel[n_sel] = r - 1; lptr[n_sel] = s.logits_last; ++n_sel;
    }
    sg.upload();

    const bool tc_prefill = e->attn_backend == WLK_BACKEND_TCGEN05 && e->act == DT_BF16 && max_tq >= 16;
    auto launch_all = [&]() {
    {   ProfScope ps(e, WLK_KC_MISC);
        embed_tokens(tok_dev, pos_dev, W.emb_f32, W.dec_pos, e->dx, R, dt, e->st); }
    const float qk_scale = powf(64.0f, -0.25f);
    for (int li = 0; li < D.n_text_layer; ++li) {
        DecLayerW& L = W.dec[li];
        {   ProfScope ps(e, WLK_KC_LN);
            layernorm(e->dx, dt, L.ln1w, L.ln1b, e->dxn, e->act, dt, R, dt, nullptr, e->st); }
        {   GemmArgs g;
            g.A = e->dxn; g.a_type = e->act; g.lda = dt; g.W = L.Wqkv; g.w_type = e->wt; g.ldw = dt;
            g.M = R; g.N = 3 * dt; g.K = dt;
            g.epi.bias = L.bqkv; g.epi.col_scale = qk_scale; g.epi.scale_cols = 2 * dt;
            g.epi.mode = EPI_SELF_QKV; g.epi.C = e->dq; g.epi.ldc = dt; g.epi.c_type = e->act;
            g.epi.batch_ptrs = skv_dev; g.epi.row_slot = slot_dev; g.epi.row_pos = pos_dev;
            g.epi.layer = li; g.epi.n_head = H; g.epi.d_model = dt; g.epi.kv_len = ctx;
            run_gemm(e, g, WLK_KC_GEMM_DEC); }
        {   ProfScope ps(e, WLK_KC_ATTN_DEC_SELF);
            dec_self_attention_layer(e, e->dq, e->act, R, dj_dev, n, max_tq, li, e->self_maps_dev, e->datt, tc_prefill); }
        {   GemmArgs g;
            g.A = e->datt; g.a_type = e->act; g.lda = dt; g.W = L.Wo; g.w_type = e->wt; g.ldw = dt;
            g.M = R; g.N = dt; g.K = dt;
            g.epi.bias = L.bo; g.epi.residual = e->dx; g.epi.ldr = dt; g.epi.C = e->dx; g.epi.c_type = DT_F32; g.epi.ldc = dt;
            run_gemm(e, g, WLK_KC_GEMM_DEC); }
        {   ProfScope ps(e, WLK_KC_LN);
            layernorm(e->dx, dt, L.lncw, L.lncb, e->dxn, e->act, dt, R, dt, nullptr, e->st); }
        {   GemmArgs g;
            g.A = e->dxn; g.a_type = e->act; g.lda = dt; g.W = L.Wqc; g.w_type = e->wt; g.ldw = dt;
            g.M = R; g.N = dt; g.K = dt;
            g.epi.bias = L.bqc; g.epi.col_scale = qk_scale; g.epi.scale_cols = dt;
            g.epi.C = e->dq; g.epi.c_type = e->act; g.epi.ldc = dt;
            run_gemm(e, g, WLK_KC_GEMM_DEC); }
        {   ProfScope ps(e, WLK_KC_ATTN_DEC_CROSS, 0, (double)n * 2 * H * N_CTX * 64 * es);
            dec_cross_attention_layer(e, e->dq, e->act, R, dj_dev, n, max_tq, li, e->kv_maps_dev, e->datt, tc_prefill); }
        {   GemmArgs g;
            g.A = e->datt; g.a_type = e->act; g.lda = dt; g.W = L.Woc; g.w_type = e->wt; g.ldw = dt;
            g.M = R; g.N = dt; g.K = dt;
            g.epi.bias = L.boc; g.epi.residual = e->dx; g.epi.ldr = dt; g.epi.C = e->dx; g.epi.c_type = DT_F32; g.epi.ldc = dt;
            run_gemm(e, g, WLK_KC_GEMM_DEC); }
        {   ProfScope ps(e, WLK_KC_LN);
            layernorm(e->dx, dt, L.ln2w, L.ln2b, e->dxn, e->act, dt, R, dt, nullptr, e->st); }
        {   GemmArgs g;
            g.A = e->dxn; g.a_type = e->act; g.lda = dt; g.W = L.W1; g.w_type = e->wt; g.ldw = dt;
            g.M = R; g.N = 4 * dt; g.K = dt;
            g.epi.bias = L.b1; g.epi.gelu = 1; g.epi.C = e->dhid; g.epi.c_type = e->act; g.epi.ldc = 4 * dt;
            run_gemm(e, g, WLK_KC_GEMM_DEC); }
        {   GemmArgs g;
            g.A = e->dhid; g.a_type = e->act; g.lda = 4 * dt; g.W = L.W2; g.w_type = e->wt; g.ldw = 4 * dt;
            g.M = R; g.N = dt; g.K = 4 * dt;
            g.epi.bias = L.b2; g.epi.residual = e->dx; g.epi.ldr = dt; g.epi.C = e->dx; g.epi.c_type = DT_F32; g.epi.ldc = dt;
            run_gemm(e, g, WLK_KC_GEMM_DEC); }
    }
    if (all_logits_dev) {
        // word-timestamp pass (find_alignment, timing.py:197-201) reads the logits of EVERY fed position
        WLK_CHECK(n == 1, "all-logits decode is single-session");
        {   ProfScope ps(e, WLK_KC_LN);
            layernorm(e->dx, dt, W.lnw, W.lnb, e->dxn, e->act, dt, R, dt, nullptr, e->st); }
        GemmArgs g;
        g.A = e->dxn; g.a_type = e->act; g.lda = dt; g.W = W.emb_act; g.w_type = e->wt; g.ldw = dt;
        g.M = R; g.N = D.n_vocab; g.K = dt;
        g.epi.C = all_logits_dev; g.epi.c_type = DT_F32; g.epi.ldc = D.n_vocab;
        run_gemm(e, g, WLK_KC_LOGITS);
    }
    // logits only for the rows the policy reads (last row; sot row on the first call of the epoch)
    {   ProfScope ps(e, WLK_KC_LN);
        layernorm(e->dx, dt, W.lnw, W.lnb, e->dsel, e->act, dt, n_sel, dt, sel_dev, e->st); }
    {   GemmArgs g;
        g.A = e->dsel; g.a_type = e->act; g.lda = dt; g.W = W.emb_act; g.w_type = e->wt; g.ldw = dt;
        g.M = n_sel; g.N = D.n_vocab; g.K = dt;
        g.epi.mode = EPI_ROWPTR; g.epi.batch_ptrs = lptr_dev; g.epi.rows_per_batch = 1; g.epi.c_type = DT_F32;
        g.epi.ldc = D.n_vocab;
        run_gemm(e, g, WLK_KC_LOGITS); }
    };   // launch_all

    // Token steps (one row per session): replay a captured graph.  The key is everything that shapes the launches --
    // batch size and number of logits rows; pointers into the staging block are a function of those two.  A key is
    // run eagerly the first time (lazy one-time initialisations happen outside capture) and captured the second.
    const bool graphable = e->graphs_on && max_tq == 1 && !all_logits_dev && !e->prof_on;
    if (!graphable) {
        launch_all();
    } else {
        const uint64_t key = ((uint64_t)n << 32) | (uint32_t)n_sel;
        auto it = e->dec_graphs.find(key);
        if (it == e->dec_graphs.end() && !e->dec_graph_seen.count(key)) {
            e->dec_graph_seen.insert(key);
            launch_all();
        } else {
            if (it == e->dec_graphs.end()) {
                cudaGraph_t graph = nullptr;
                CUDA_CHECK(cudaStreamBeginCapture(e->st, cudaStreamCaptureModeRelaxed));
                try {
                    launch_all();
                } catch (...) {
                    cudaStreamEndCapture(e->st, &graph);
                    if (graph) cudaGraphDestroy(graph);
                    throw;
                }
                CUDA_CHECK(cudaStreamEndCapture(e->st, &graph));
                cudaGraphExec_t exec = nullptr;
                CUDA_CHECK(cudaGraphInstantiate(&exec, graph, 0));
                cudaGraphDestroy(graph);
                const size_t cap = (size_t)2 * e->cfg.max_batch + 8;   // (n, n_sel) pairs in use: n_sel is n or 2n
                if (e->dec_graphs.size() >= cap) {               // evict the least recently used entry only
                    auto lru = e->dec_graphs.begin();
                    for (auto jt = e->dec_graphs.begin(); jt != e->dec_graphs.end(); ++jt)
                        if (jt->second.last_use < lru->second.last_use) lru = jt;
                    CUDA_CHECK(cudaStreamSynchronize(e->st));    // its last replay may still be in flight
                    cudaGraphExecDestroy(lru->second.exec);
                    e->dec_graphs.erase(lru);
                }
                it = e->dec_graphs.emplace(key, wlk_engine::GraphSlot{exec, 0}).first;
            }
            it->second.last_use = ++e->dec_graph_tick;
            CUDA_CHECK(cudaGraphLaunch(it->second.exec, e->st));
        }
    }
    for (int i = 0; i < n; ++i) {
        Session& s = e->sess[sids[i]];
        const int tq = offsets[i + 1] - offsets[i];
        s.iter_row_start.push_back(s.align_rows);
        s.align_rows += tq;
        s.self_len += tq;
    }
}

LogitJob make_logit_job(wlk_engine* e, Session& s, int window_iters, int full) {
    LogitJob j{};
    j.logits_last = s.logits_last; j.logits_sot = s.logits_sot; j.align = s.align;
    j.attn_out = s.attn_out; j.stats = s.stats;
    const int ni = (int)s.iter_row_start.size();
    const int first = ni > window_iters ? ni - window_iters : 0;
    j.row_begin = ni ? s.iter_row_start[first] : 0;
    j.row_end = s.align_rows;
    // the reference slices a 1500-wide tensor ([:, :, :content_mel_len], simul_whisper.py:433): frames >= 1500 do not exist
    j.content_len = std::min(enc_owner(e, s).content_len, N_CTX);
    j.full = full;
    j.rot = enc_owner(e, s).rot;
    return j;
}

void alloc_session(wlk_engine* e, Session& s) {
    const wlk_dims& D = e->dims;
    const size_t es = e->es();
    size_t* acct = &s.bytes;
    s.bytes = 0;
    s.audio = dmalloc<float>(e, AUDIO_CAP, acct);
    s.mel_raw = dmalloc<float>(e, (size_t)MEL_STORE_FRAMES * D.n_mels, acct);
    s.mel_blockmax = dmalloc<float>(e, MEL_MAX_CTAS + MEL_MAX_PARTS, acct);
    s.mel_n = -1; s.mel_dropped = 0;
    s.xa = dmalloc_bytes((size_t)N_CTX * D.n_audio_state * es, acct);
    s.cross_kv = dmalloc_bytes((size_t)D.n_text_layer * 2 * N_CTX * D.n_text_state * es, acct);
    s.self_kv = dmalloc_bytes((size_t)D.n_text_layer * 2 * D.n_text_ctx * D.n_text_state * es, acct);
    s.align = dmalloc<float>(e, (size_t)(e->n_align > 0 ? e->n_align : 1) * D.n_text_ctx * N_CTX, acct);
    s.logits_last = dmalloc<float>(e, D.n_vocab, acct);
    s.logits_sot = dmalloc<float>(e, D.n_vocab, acct);
    s.attn_out = dmalloc<float>(e, (size_t)D.n_text_ctx * N_CTX, acct);
    s.stats = dmalloc<float>(e, (size_t)(e->n_align > 0 ? e->n_align : 1) * N_CTX * 2, acct);
    e->bytes_sessions += s.bytes;
    if (e->act == DT_BF16) {
        alignas(64) uint8_t tmap[128];
        make_cross_kv_tmap(tmap, s.cross_kv, D.n_text_layer, D.n_text_head);
        const size_t slot = (size_t)(&s - e->sess.data());
        CUDA_CHECK(cudaMemcpy(e->kv_maps_dev + slot * 128, tmap, 128, cudaMemcpyHostToDevice));
        make_self_kv_tmap(tmap, s.self_kv, D.n_text_layer, D.n_text_head, D.n_text_ctx);
        CUDA_CHECK(cudaMemcpy(e->self_maps_dev + slot * 128, tmap, 128, cudaMemcpyHostToDevice));
        // the tensor-core prefill reads whole 128-key tiles of the cache: rows past the current length take part in the
        // MMAs with probability exactly 0, so they must hold finite values (0 x NaN would poison the accumulator)
        CUDA_CHECK(cudaMemsetAsync(s.self_kv, 0, (size_t)D.n_text_layer * 2 * D.n_text_ctx * D.n_text_state * es, e->st));
    }
}
void free_session(wlk_engine* e, Session& s) {
    if (s.parent >= 0) {                                  // a fork owns its decoder-side buffers only
        e->sess[s.parent].n_forks -= 1;
        s.xa = nullptr; s.cross_kv = nullptr;
    }
    void* ptrs[] = {s.audio, s.mel_raw, s.mel_blockmax, s.xa, s.cross_kv, s.self_kv, s.align, s.logits_last,
                    s.logits_sot, s.attn_out, s.stats, s.enc_kv};
    for (void* p : ptrs) if (p) cudaFree(p);
    e->bytes_sessions -= s.bytes;
    s = Session{};
}
// a beam: decoder-side buffers of its own, encoder output and cross-K/V of `parent` (reference: beam_size decoder rows
// over one encoder output, simul_whisper.py:240-243)
void alloc_fork(wlk_engine* e, Session& s, int parent) {
    const wlk_dims& D = e->dims;
    const size_t es = e->es();
    Session& p = e->sess[parent];
    size_t* acct = &s.bytes;
    s.bytes = 0;
    s.self_kv = dmalloc_bytes((size_t)D.n_text_layer * 2 * D.n_text_ctx * D.n_text_state * es, acct);
    s.align = dmalloc<float>(e, (size_t)(e->n_align > 0 ? e->n_align : 1) * D.n_text_ctx * N_CTX, acct);
    s.logits_last = dmalloc<float>(e, D.n_vocab, acct);
    s.logits_sot = dmalloc<float>(e, D.n_vocab, acct);
    s.attn_out = dmalloc<float>(e, (size_t)D.n_text_ctx * N_CTX, acct);
    s.stats = dmalloc<float>(e, (size_t)(e->n_align > 0 ? e->n_align : 1) * N_CTX * 2, acct);
    s.xa = p.xa; s.cross_kv = p.cross_kv; s.parent = parent;
    p.n_forks += 1;
    e->bytes_sessions += s.bytes;
    if (e->act == DT_BF16) {
        alignas(64) uint8_t tmap[128];
        make_cross_kv_tmap(tmap, p.cross_kv, D.n_text_layer, D.n_text_head);
        const size_t slot = (size_t)(&s - e->sess.data());
        CUDA_CHECK(cudaMemcpy(e->kv_maps_dev + slot * 128, tmap, 128, cudaMemcpyHostToDevice));
        make_self_kv_tmap(tmap, s.self_kv, D.n_text_layer, D.n_text_head, D.n_text_ctx);
        CUDA_CHECK(cudaMemcpy(e->self_maps_dev + slot * 128, tmap, 128, cudaMemcpyHostToDevice));
        CUDA_CHECK(cudaMemsetAsync(s.self_kv, 0, (size_t)D.n_text_layer * 2 * D.n_text_ctx * D.n_text_state * es, e->st));
    }
}

void create_engine(const wlk_dims* dims, const wlk_config* cfg, wlk_engine** out) {
    WLK_CHECK(dims && cfg && out, "null argument");
    WLK_CHECK(dims->n_audio_ctx == N_CTX, "n_audio_ctx must be 1500");
    WLK_CHECK(dims->n_audio_state % 64 == 0 && dims->n_audio_state / dims->n_audio_head == 64, "audio heads must be 64 wide");
    WLK_CHECK(dims->n_text_state % 64 == 0 && dims->n_text_state / dims->n_text_head == 64, "text heads must be 64 wide");
    WLK_CHECK(dims->n_mels % 8 == 0 && dims->n_mels <= 128, "n_mels must be 80 or 128");
    WLK_CHECK(cfg->max_sessions >= 1 && cfg->max_batch >= 1, "max_sessions / max_batch must be >= 1");
    int ndev = 0;
    cudaError_t ce = cudaGetDeviceCount(&ndev);
    WLK_CHECK(ce == cudaSuccess && ndev > 0, "no CUDA device available (%s): the B200 engine has no CPU fallback",
              cudaGetErrorString(ce));
    WLK_CHECK(cfg->device >= 0 && cfg->device < ndev, "device %d out of range (%d devices)", cfg->device, ndev);
    CUDA_CHECK(cudaSetDevice(cfg->device));
    cudaDeviceProp prop;
    CUDA_CHECK(cudaGetDeviceProperties(&prop, cfg->device));
    WLK_CHECK(prop.major == 10, "this library contains sm_100a code only; device %d is sm_%d%d", cfg->device, prop.major, prop.minor);

    auto* e = new wlk_engine();
    e->dims = *dims; e->cfg = *cfg;
    e->num_sms = prop.multiProcessorCount;
    WLK_CHECK(cfg->precision == WLK_PREC_FP32 || cfg->precision == WLK_PREC_BF16 || cfg->precision == WLK_PREC_BF16X3,
              "unknown precision %d", cfg->precision);
    e->act = cfg->precision == WLK_PREC_BF16 ? DT_BF16 : DT_F32;
    e->wt = cfg->precision == WLK_PREC_BF16X3 ? DT_BF16X2 : e->act;
    e->gemm_backend = cfg->gemm_backend != WLK_BACKEND_AUTO ? cfg->gemm_backend
                      : (e->act == DT_BF16 ? WLK_BACKEND_TCGEN05 : WLK_BACKEND_SIMT);
    e->attn_backend = cfg->attn_backend != WLK_BACKEND_AUTO ? cfg->attn_backend
                      : (e->act == DT_BF16 ? WLK_BACKEND_TCGEN05 : WLK_BACKEND_SIMT);
    if (e->act != DT_BF16) { e->gemm_backend = WLK_BACKEND_SIMT; e->attn_backend = WLK_BACKEND_SIMT; }
    // BF16X3: fp32 activations, LayerNorm and decoder attention; every GEMM and the encoder attention on the tensor
    // cores with split operands (WLK_BACKEND_SIMT for the attention keeps the fp32 SIMT kernel: a test reference)
    if (e->wt == DT_BF16X2) {
        e->gemm_backend = WLK_BACKEND_TCGEN05;
        e->attn_backend = cfg->attn_backend == WLK_BACKEND_SIMT ? WLK_BACKEND_SIMT : WLK_BACKEND_TCGEN05;
    }
    CUDA_CHECK(cudaStreamCreateWithFlags(&e->st, cudaStreamNonBlocking));
    {   const char* v = getenv("WLK_GRAPHS"); e->graphs_on = !(v && v[0] == '0'); }
    {   const char* v = getenv("WLK_MEL_INCREMENTAL"); e->mel_incremental = !(v && v[0] == '0'); }
    for (auto& t : e->timers) CUDA_CHECK(cudaEventCreate(&t));
    CUDA_CHECK(cudaEventCreateWithFlags(&e->stg_done, cudaEventDisableTiming));
    CUDA_CHECK(cudaEventRecord(e->stg_done, e->st));

    // weights arena: dry run for the size, then the real layout
    layout_weights(e);
    const size_t wbytes = e->arena.used + ALIGN;
    e->arena = Arena{};
    e->arena.base = reinterpret_cast<uint8_t*>(dmalloc_bytes(wbytes, &e->bytes_weights));
    e->arena.cap = wbytes;
    CUDA_CHECK(cudaMemsetAsync(e->arena.base, 0, wbytes, e->st));
    layout_weights(e);
    {   // DFT twiddles exp(-2 pi i t / 400) in double -> float
        std::vector<float2> tw(N_FFT);
        for (int t = 0; t < N_FFT; ++t) {
            double a = 2.0 * M_PI * t / N_FFT;
            tw[t] = make_float2((float)cos(a), (float)-sin(a));
        }
        CUDA_CHECK(cudaMemcpyAsync(e->w.twiddle, tw.data(), N_FFT * 8, cudaMemcpyHostToDevice, e->st));
        CUDA_CHECK(cudaStreamSynchronize(e->st));
    }

    const wlk_dims& D = e->dims;
    const size_t es = e->es();
    const int B = cfg->max_batch, d = D.n_audio_state, dt = D.n_text_state;
    size_t* acct = &e->bytes_workspace;
    e->mel_t = dmalloc_bytes((size_t)B * MEL_ROWS * D.n_mels * es, acct);
    e->h1 = dmalloc_bytes(((size_t)B * MEL_ROWS + 2) * d * es, acct);
    e->x = dmalloc<float>(e, (size_t)B * N_CTX * d, acct);
    e->xn = dmalloc_bytes((size_t)B * N_CTX * d * es, acct);
    e->qkv = dmalloc_bytes((size_t)B * N_CTX * 3 * d * es, acct);
    e->att = dmalloc_bytes((size_t)B * N_CTX * d * es, acct);
    e->hid = dmalloc_bytes((size_t)B * N_CTX * 4 * d * es, acct);
    e->audio_scratch = dmalloc<float>(e, AUDIO_CAP, acct);
    e->mel_scratch = dmalloc<float>(e, (size_t)MEL_STORE_FRAMES * D.n_mels, acct);
    if (e->gemm_backend == WLK_BACKEND_TCGEN05) {
        e->sk_scratch = dmalloc<float>(e, SK_SCRATCH_FLOATS, acct);
        e->sk_counters = dmalloc<int>(e, SK_MAX_TILES, acct);
        CUDA_CHECK(cudaMemset(e->sk_counters, 0, SK_MAX_TILES * 4));
    }
    {
        std::vector<int64_t> rows(2 * B);
        std::vector<void*> xp(B);
        for (int b = 0; b < B; ++b) {
            rows[2 * b] = (int64_t)b * MEL_ROWS;
            rows[2 * b + 1] = (int64_t)b * MEL_ROWS + MEL_ROWS - 1;
            xp[b] = e->x + (size_t)b * N_CTX * d;
        }
        e->pad_rows_dev = dmalloc<int64_t>(e, 2 * B, acct);
        e->xptrs_dev = dmalloc<void*>(e, B, acct);
        CUDA_CHECK(cudaMemcpy(e->pad_rows_dev, rows.data(), rows.size() * 8, cudaMemcpyHostToDevice));
        CUDA_CHECK(cudaMemcpy(e->xptrs_dev, xp.data(), xp.size() * sizeof(void*), cudaMemcpyHostToDevice));
    }
    e->dec_rows_max = B * D.n_text_ctx;
    const size_t R = e->dec_rows_max;
    e->dx = dmalloc<float>(e, R * dt, acct);
    e->dxn = dmalloc_bytes(R * dt * es, acct);
    e->dq = dmalloc_bytes(R * dt * es, acct);
    e->datt = dmalloc_bytes(R * dt * es, acct);
    e->dhid = dmalloc_bytes(R * 4 * dt * es, acct);
    e->dsel = dmalloc_bytes((size_t)2 * B * dt * es, acct);
    if (e->wt == DT_BF16X2) {
        size_t m = (size_t)B * N_CTX * 4 * d;                                  // fc2's operand (the MLP hidden)
        m = std::max(m, R * 4 * dt);                                           // decoder MLP hidden
        m = std::max(m, ((size_t)B * MEL_ROWS + 2) * (size_t)std::max(d, D.n_mels) + 3 * (size_t)d);   // conv views
        e->a_split_elems = (m + 7) / 8 * 8;
        e->a_split = dmalloc_bytes(e->a_split_elems * 2 * 2, acct);
    }
    e->stg_bytes = (size_t)B * 2048 + R * 16 + 65536 + 1024 * 8 * 4;
    CUDA_CHECK(cudaMallocHost(&e->stg_host, e->stg_bytes));
    e->stg_dev = reinterpret_cast<uint8_t*>(dmalloc_bytes(e->stg_bytes, acct));
    e->res_dev = dmalloc<StepResult>(e, B, acct);
    CUDA_CHECK(cudaMallocHost(&e->res_host, sizeof(StepResult) * B));
    e->sess.resize(cfg->max_sessions);
    e->kv_maps_dev = reinterpret_cast<uint8_t*>(dmalloc_bytes((size_t)cfg->max_sessions * 128, acct));
    e->self_maps_dev = reinterpret_cast<uint8_t*>(dmalloc_bytes((size_t)cfg->max_sessions * 128, acct));
    e->align_rank_host.assign((size_t)D.n_text_layer * D.n_text_head, -1);
    e->align_rank_dev = dmalloc<int32_t>(e, e->align_rank_host.size(), acct);
    CUDA_CHECK(cudaMemcpy(e->align_rank_dev, e->align_rank_host.data(), e->align_rank_host.size() * 4, cudaMemcpyHostToDevice));
    *out = e;
}

void destroy_engine(wlk_engine* e) {
    cudaStreamSynchronize(e->st);
    for (auto& s : e->sess) if (s.open && s.parent >= 0) free_session(e, s);     // forks before their parents
    for (auto& s : e->sess) if (s.open) free_session(e, s);
    void* ptrs[] = {e->arena.base, e->stage_f32, e->mel_t, e->h1, e->x, e->xn, e->qkv, e->att, e->hid, e->audio_scratch, e->mel_scratch, e->beam_scratch, e->sk_scratch, e->sk_counters, e->a_split,
                    e->pad_rows_dev, e->xptrs_dev, e->dx, e->dxn, e->dq, e->datt, e->dhid, e->dsel, e->stg_dev,
                    e->res_dev, e->align_rank_dev, e->kv_maps_dev, e->self_maps_dev, e->all_logits_dev};
    for (void* p : ptrs) if (p) cudaFree(p);
    if (e->stg_host) cudaFreeHost(e->stg_host);
    if (e->res_host) cudaFreeHost(e->res_host);
    if (e->tap_host) cudaFreeHost(e->tap_host);
    for (auto& t : e->timers) if (t) cudaEventDestroy(t);
    for (auto& p : e->prof) { cudaEventDestroy(p.a); cudaEventDestroy(p.b); }
    for (auto& p : e->ev_pool) { cudaEventDestroy(p.first); cudaEventDestroy(p.second); }
    if (e->stg_done) cudaEventDestroy(e->stg_done);
    for (auto& kv : e->dec_graphs) cudaGraphExecDestroy(kv.second.exec);
    cudaStreamDestroy(e->st);
    delete e;
}

float* tap_buffer(wlk_engine* e, size_t n) {
    if (n > e->tap_cap) {
        if (e->tap_host) cudaFreeHost(e->tap_host);
        CUDA_CHECK(cudaMallocHost(&e->tap_host, n * 4));
        e->tap_cap = n;
    }
    return e->tap_host;
}

// per-call device memory of an op-level entry point: freed once the engine's stream has drained (also when the call
// fails half-way)
struct CallBuffers {
    wlk_engine* e;
    std::vector<void*> bufs;
    explicit CallBuffers(wlk_engine* e_) : e(e_) {}
    void* take(size_t bytes) { bufs.push_back(dmalloc_bytes(bytes, nullptr)); return bufs.back(); }
    ~CallBuffers() {
        if (bufs.empty()) return;
        cudaStreamSynchronize(e->st);
        for (void* p : bufs) cudaFree(p);
    }
};

bool aligned16(const void* p) { return p != nullptr && reinterpret_cast<uintptr_t>(p) % 16 == 0; }

}  // namespace
}  // namespace wlk

// =========================================================================================
// C ABI
// =========================================================================================
#define WLK_API_BEGIN try {
#define WLK_API_END                                              \
    return 0;                                                    \
    } catch (const wlk::Error& err) {                            \
        wlk::set_last_error(err.msg);                            \
        return 1;                                                \
    } catch (const std::exception& ex) {                         \
        wlk::set_last_error(std::string("exception: ") + ex.what()); \
        return 2;                                                \
    } catch (...) {                                              \
        wlk::set_last_error("unknown exception");                \
        return 3;                                                \
    }
#define LOCK(e) WLK_CHECK((e) != nullptr, "null engine"); std::lock_guard<std::mutex> _lk((e)->mu); \
                CUDA_CHECK(cudaSetDevice((e)->cfg.device))

extern "C" {

const char* wlk_last_error(void) { return wlk::g_last_error.c_str(); }
int wlk_abi_version(void) { return WLK_ABI_VERSION; }

int wlk_engine_create(const wlk_dims* dims, const wlk_config* cfg, wlk_engine** out) {
    WLK_API_BEGIN
    create_engine(dims, cfg, out);
    WLK_API_END
}
int wlk_engine_destroy(wlk_engine* e) {
    WLK_API_BEGIN
    WLK_CHECK(e != nullptr, "null engine");
    CUDA_CHECK(cudaSetDevice(e->cfg.device));
    destroy_engine(e);
    WLK_API_END
}
int wlk_engine_load_tensor(wlk_engine* e, const char* name, const float* host, const int64_t* shape, int ndim) {
    WLK_API_BEGIN
    LOCK(e);
    WLK_CHECK(name && host && shape && ndim >= 1, "bad arguments");
    load_tensor(e, name, host, shape, ndim);
    WLK_API_END
}
int wlk_engine_finalize_weights(wlk_engine* e) {
    WLK_API_BEGIN
    LOCK(e);
    std::string missing;
    int nmiss = 0;
    for (auto& r : required_tensors(e->dims))
        if (!e->loaded.count(r)) { if (nmiss++ < 5) missing += r + " "; }
    WLK_CHECK(nmiss == 0, "%d tensors missing, e.g. %s", nmiss, missing.c_str());
    if (e->stage_f32) { CUDA_CHECK(cudaFree(e->stage_f32)); e->stage_f32 = nullptr; e->stage_cap = 0; }
    e->finalized = true;
    WLK_API_END
}
int wlk_engine_weight_blob(wlk_engine* e, void** dev, size_t* nbytes) {
    WLK_API_BEGIN
    LOCK(e);
    WLK_CHECK(dev && nbytes, "null out pointer");
    CUDA_CHECK(cudaStreamSynchronize(e->st));
    *dev = e->arena.base; *nbytes = e->arena.cap;
    WLK_API_END
}
int wlk_engine_adopt_weights(wlk_engine* e) {
    WLK_API_BEGIN
    LOCK(e);
    e->finalized = true;
    WLK_API_END
}
int wlk_engine_set_alignment_heads(wlk_engine* e, const int32_t* pairs, int n_pairs) {
    WLK_API_BEGIN
    LOCK(e);
    WLK_CHECK(n_pairs >= 1 && n_pairs <= e->cfg.max_align_heads, "%d alignment heads outside [1, max_align_heads=%d]",
              n_pairs, e->cfg.max_align_heads);
    for (auto& s : e->sess) WLK_CHECK(!s.open, "set alignment heads before opening sessions");
    std::fill(e->align_rank_host.begin(), e->align_rank_host.end(), -1);
    for (int i = 0; i < n_pairs; ++i) {
        int l = pairs[2 * i], h = pairs[2 * i + 1];
        WLK_CHECK(l >= 0 && l < e->dims.n_text_layer && h >= 0 && h < e->dims.n_text_head, "alignment head (%d,%d) out of range", l, h);
        e->align_rank_host[(size_t)l * e->dims.n_text_head + h] = i;
    }
    e->n_align = n_pairs;
    CUDA_CHECK(cudaStreamSynchronize(e->st));
    for (auto& kv : e->dec_graphs) cudaGraphExecDestroy(kv.second.exec);  // captured launches bake the head count in
    e->dec_graphs.clear(); e->dec_graph_seen.clear();
    CUDA_CHECK(cudaMemcpy(e->align_rank_dev, e->align_rank_host.data(), e->align_rank_host.size() * 4, cudaMemcpyHostToDevice));
    WLK_API_END
}
int wlk_engine_stream(wlk_engine* e, void** cuda_stream) {
    WLK_API_BEGIN
    WLK_CHECK(e && cuda_stream, "null argument");
    *cuda_stream = e->st;
    WLK_API_END
}
int wlk_engine_sync(wlk_engine* e) {
    WLK_API_BEGIN
    LOCK(e);
    CUDA_CHECK(cudaStreamSynchronize(e->st));
    WLK_API_END
}
int wlk_engine_memory(wlk_engine* e, size_t* weights, size_t* sessions, size_t* workspace) {
    WLK_API_BEGIN
    LOCK(e);
    if (weights) *weights = e->bytes_weights;
    if (sessions) *sessions = e->bytes_sessions;
    if (workspace) *workspace = e->bytes_workspace;
    WLK_API_END
}

int wlk_session_open(wlk_engine* e, int32_t* sid) {
    WLK_API_BEGIN
    LOCK(e);
    WLK_CHECK(sid, "null out pointer");
    WLK_CHECK(e->finalized, "weights not finalized");
    WLK_CHECK(e->n_align > 0, "alignment heads not set");
    int found = -1;
    for (int i = 0; i < (int)e->sess.size(); ++i) if (!e->sess[i].open) { found = i; break; }
    WLK_CHECK(found >= 0, "all %d sessions in use", (int)e->sess.size());
    alloc_session(e, e->sess[found]);
    e->sess[found].open = true;
    *sid = found;
    WLK_API_END
}
int wlk_session_close(wlk_engine* e, int32_t sid) {
    WLK_API_BEGIN
    LOCK(e);
    Session& s = get_session(e, sid);
    WLK_CHECK(s.n_forks == 0, "session %d still has %d beam fork(s): close them first", sid, s.n_forks);
    CUDA_CHECK(cudaStreamSynchronize(e->st));
    free_session(e, s);
    WLK_API_END
}
int wlk_session_fork(wlk_engine* e, int32_t parent, int32_t* child) {
    WLK_API_BEGIN
    LOCK(e);
    WLK_CHECK(child, "null out pointer");
    get_root_session(e, parent, "forking");
    int found = -1;
    for (int i = 0; i < (int)e->sess.size(); ++i) if (!e->sess[i].open) { found = i; break; }
    WLK_CHECK(found >= 0, "all %d sessions in use", (int)e->sess.size());
    alloc_fork(e, e->sess[found], parent);
    e->sess[found].open = true;
    *child = found;
    WLK_API_END
}
int wlk_sessions_gather_decoder(wlk_engine* e, const int32_t* sids, const int32_t* src, int n) {
    WLK_API_BEGIN
    LOCK(e);
    WLK_CHECK(sids && src && n >= 1, "bad argument");
    const wlk_dims& D = e->dims;
    const size_t es = e->es();
    const size_t pitch = (size_t)D.n_text_ctx * 64 * es;                 // one (layer, k|v, head) plane of the self-K/V
    const size_t planes = (size_t)D.n_text_layer * 2 * D.n_text_head;
    std::vector<int> moved;
    for (int i = 0; i < n; ++i) {
        Session& d = get_session(e, sids[i]);
        WLK_CHECK(src[i] >= 0 && src[i] < n, "source index %d out of range", src[i]);
        Session& s = get_session(e, sids[src[i]]);
        WLK_CHECK(&enc_owner(e, d) == &enc_owner(e, s), "sessions %d and %d do not share an encoder output", sids[i], sids[src[i]]);
        for (int j = 0; j < i; ++j) WLK_CHECK(sids[j] != sids[i], "session %d appears twice", sids[i]);
        if (src[i] != i) moved.push_back(i);
    }
    if (moved.empty()) return 0;
    const size_t per = planes * pitch;
    if (e->beam_scratch_cap < moved.size() * per) {
        if (e->beam_scratch) { CUDA_CHECK(cudaStreamSynchronize(e->st)); cudaFree(e->beam_scratch); e->beam_scratch = nullptr; }
        CUDA_CHECK(cudaMalloc(&e->beam_scratch, moved.size() * per));
        e->beam_scratch_cap = moved.size() * per;
    }
    // stage every source that moves (only its valid prefix), then scatter: sources may be overwritten by other moves
    std::vector<int> new_len(n);
    for (int i = 0; i < n; ++i) new_len[i] = e->sess[sids[src[i]]].self_len;
    for (size_t k = 0; k < moved.size(); ++k) {
        Session& s = e->sess[sids[src[moved[k]]]];
        if (s.self_len)
            CUDA_CHECK(cudaMemcpy2DAsync((char*)e->beam_scratch + k * per, pitch, s.self_kv, pitch, (size_t)s.self_len * 64 * es,
                                         planes, cudaMemcpyDeviceToDevice, e->st));
    }
    for (size_t k = 0; k < moved.size(); ++k) {
        Session& d = e->sess[sids[moved[k]]];
        const int len = new_len[moved[k]];
        if (len)
            CUDA_CHECK(cudaMemcpy2DAsync(d.self_kv, pitch, (char*)e->beam_scratch + k * per, pitch, (size_t)len * 64 * es, planes,
                                         cudaMemcpyDeviceToDevice, e->st));
    }
    for (int i = 0; i < n; ++i) e->sess[sids[i]].self_len = new_len[i];
    WLK_API_END
}
int wlk_session_append_audio(wlk_engine* e, int32_t sid, const float* pcm, int64_t n) {
    WLK_API_BEGIN
    LOCK(e);
    Session& s = get_root_session(e, sid, "the audio ring");
    WLK_CHECK(n >= 0 && (n == 0 || pcm), "bad audio chunk");
    WLK_CHECK(s.audio_len + n <= AUDIO_CAP, "audio buffer overflow: %lld + %lld > %d samples", (long long)s.audio_len, (long long)n, AUDIO_CAP);
    if (n) CUDA_CHECK(cudaMemcpyAsync(s.audio + s.audio_len, pcm, (size_t)n * 4, cudaMemcpyHostToDevice, e->st));
    s.audio_len += n;
    WLK_API_END
}
int wlk_session_append_pcm16(wlk_engine* e, int32_t sid, const int16_t* pcm, int64_t n) {
    WLK_API_BEGIN
    LOCK(e);
    Session& s = get_root_session(e, sid, "the audio ring");
    WLK_CHECK(n >= 0 && (n == 0 || pcm), "bad audio chunk");
    WLK_CHECK(s.audio_len + n <= AUDIO_CAP, "audio buffer overflow: %lld + %lld > %d samples", (long long)s.audio_len, (long long)n, AUDIO_CAP);
    if (n) {
        // the raw bytes land in the (idle between calls) audio scratch, the conversion writes the ring in place
        CUDA_CHECK(cudaMemcpyAsync(e->audio_scratch, pcm, (size_t)n * 2, cudaMemcpyHostToDevice, e->st));
        pcm16_to_f32(reinterpret_cast<const int16_t*>(e->audio_scratch), s.audio + s.audio_len, n, e->st);
    }
    s.audio_len += n;
    WLK_API_END
}
int wlk_session_drop_audio(wlk_engine* e, int32_t sid, int64_t n) {
    WLK_API_BEGIN
    LOCK(e);
    Session& s = get_root_session(e, sid, "the audio ring");
    WLK_CHECK(n >= 0 && n <= s.audio_len, "cannot drop %lld of %lld samples", (long long)n, (long long)s.audio_len);
    const int64_t keep = s.audio_len - n;
    if (n && keep) {
        CUDA_CHECK(cudaMemcpyAsync(e->audio_scratch, s.audio + n, (size_t)keep * 4, cudaMemcpyDeviceToDevice, e->st));
        CUDA_CHECK(cudaMemcpyAsync(s.audio, e->audio_scratch, (size_t)keep * 4, cudaMemcpyDeviceToDevice, e->st));
    }
    if (s.mel_n >= 0) s.mel_dropped += n;
    if (s.inc_valid) s.inc_dropped += n;
    s.audio_len = keep;
    WLK_API_END
}
int wlk_session_clear_audio(wlk_engine* e, int32_t sid) {
    WLK_API_BEGIN
    LOCK(e);
    Session& s = get_session(e, sid);
    s.audio_len = 0; s.mel_n = -1; s.mel_dropped = 0; s.inc_valid = false;
    WLK_API_END
}
int wlk_session_audio_len(wlk_engine* e, int32_t sid, int64_t* n) {
    WLK_API_BEGIN
    LOCK(e);
    WLK_CHECK(n, "null out pointer");
    *n = get_session(e, sid).audio_len;
    WLK_API_END
}

int wlk_session_reset_decoder(wlk_engine* e, int32_t sid) {
    WLK_API_BEGIN
    LOCK(e);
    Session& s = get_session(e, sid);
    s.self_len = 0; s.align_rows = 0; s.iter_row_start.clear();
    WLK_API_END
}

int wlk_encode(wlk_engine* e, const int32_t* sids, int n, int32_t* content_out) {
    WLK_API_BEGIN
    LOCK(e);
    WLK_CHECK(sids && content_out, "null argument");
    encode_batch(e, sids, n, content_out);
    WLK_API_END
}
int wlk_encode_incremental(wlk_engine* e, const int32_t* sids, int n, int32_t* content_out, int32_t* block_rows_out) {
    WLK_API_BEGIN
    LOCK(e);
    WLK_CHECK(sids && content_out, "null argument");
    WLK_CHECK(e->finalized, "weights not finalized");
    encode_incremental(e, sids, n, content_out, block_rows_out);
    WLK_API_END
}
int wlk_session_reset_incremental(wlk_engine* e, int32_t sid) {
    WLK_API_BEGIN
    LOCK(e);
    Session& s = get_root_session(e, sid, "the encoder K/V");
    s.inc_valid = false;                       // the next incremental encode takes the whole window as its block
    WLK_API_END
}
int wlk_decode(wlk_engine* e, const int32_t* sids, int n, const int32_t* tokens, const int32_t* offsets, int32_t sot_index) {
    WLK_API_BEGIN
    LOCK(e);
    WLK_CHECK(sids && tokens && offsets, "null argument");
    decode_batch(e, sids, n, tokens, offsets, sot_index);
    WLK_API_END
}
int wlk_encode_mel(wlk_engine* e, int32_t sid, const float* mel_host, int32_t content_mel_len) {
    WLK_API_BEGIN
    LOCK(e);
    Session& s = get_root_session(e, sid, "encode");
    WLK_CHECK(mel_host && content_mel_len >= 0, "bad arguments");
    const int nm = e->dims.n_mels;
    Stager sg(e);
    void** xkv_dev; void** xkv = sg.host<void*>(1, &xkv_dev);
    xkv[0] = s.cross_kv;
    sg.upload();
    CUDA_CHECK(cudaMemcpyAsync(e->mel_scratch, mel_host, (size_t)nm * N_FRAMES * 4, cudaMemcpyHostToDevice, e->st));
    {   ProfScope ps(e, WLK_KC_MEL);
        mel_import(e->mel_scratch, e->mel_t, e->act, nm, e->st); }
    run_encoder(e, &sid, 1, xkv_dev);
    s.mel_n = -1;                                    // the caller's mel: nothing of this window is cached in mel_raw
    s.content_len = content_mel_len > N_CTX ? N_CTX : content_mel_len;
    CUDA_CHECK(cudaStreamSynchronize(e->st));        // mel_host may be reused by the caller
    WLK_API_END
}
int wlk_decode_all_logits(wlk_engine* e, int32_t sid, const int32_t* tokens, int n_tokens, int32_t sot_index,
                          float* logits_host) {
    WLK_API_BEGIN
    LOCK(e);
    WLK_CHECK(tokens && logits_host && n_tokens >= 1 && n_tokens <= e->dims.n_text_ctx, "bad arguments");
    const size_t need = (size_t)n_tokens * e->dims.n_vocab;
    if (need > e->all_logits_cap) {
        if (e->all_logits_dev) CUDA_CHECK(cudaFree(e->all_logits_dev));
        CUDA_CHECK(cudaMalloc(&e->all_logits_dev, need * 4));
        e->all_logits_cap = need;
    }
    int32_t offs[2] = {0, n_tokens};
    decode_batch(e, &sid, 1, tokens, offs, sot_index, e->all_logits_dev);
    CUDA_CHECK(cudaMemcpyAsync(logits_host, e->all_logits_dev, need * 4, cudaMemcpyDeviceToHost, e->st));
    CUDA_CHECK(cudaStreamSynchronize(e->st));
    WLK_API_END
}
int wlk_read_align_rows(wlk_engine* e, int32_t sid, float* out, int64_t capacity, int32_t* n_align, int32_t* rows) {
    WLK_API_BEGIN
    LOCK(e);
    Session& s = get_session(e, sid);
    WLK_CHECK(out && n_align && rows, "null argument");
    const int R = s.align_rows, A = e->n_align;
    WLK_CHECK((int64_t)A * R * N_CTX <= capacity, "output buffer too small: need %d x %d x %d", A, R, N_CTX);
    for (int a = 0; a < A; ++a)
        CUDA_CHECK(cudaMemcpyAsync(out + (size_t)a * R * N_CTX, s.align + (size_t)a * e->dims.n_text_ctx * N_CTX,
                                   (size_t)R * N_CTX * 4, cudaMemcpyDeviceToHost, e->st));
    CUDA_CHECK(cudaStreamSynchronize(e->st));
    *n_align = A; *rows = R;
    WLK_API_END
}

int wlk_no_speech_prob(wlk_engine* e, const int32_t* sids, int n, float* prob_out) {
    WLK_API_BEGIN
    LOCK(e);
    WLK_CHECK(sids && prob_out && n >= 1 && n <= e->cfg.max_batch, "bad arguments");
    Stager sg(e);
    LogitJob* lj_dev; LogitJob* lj = sg.host<LogitJob>(n, &lj_dev);
    for (int i = 0; i < n; ++i) {
        Session& s = get_session(e, sids[i]);
        WLK_CHECK(!s.iter_row_start.empty(), "session %d: no decode call in this epoch", sids[i]);
        lj[i] = make_logit_job(e, s, 16, 0);
    }
    sg.upload();
    const int no_speech = (e->dims.n_vocab >= 51865 ? 50257 : 50256) + 2 + (e->dims.n_vocab - 51765 - (e->dims.n_vocab >= 51865 ? 1 : 0)) + 4;
    {   ProfScope ps(e, WLK_KC_LOGITS);
        no_speech_prob(lj_dev, n, e->dims.n_vocab, no_speech, e->res_dev, e->st); }
    CUDA_CHECK(cudaMemcpyAsync(e->res_host, e->res_dev, sizeof(StepResult) * n, cudaMemcpyDeviceToHost, e->st));
    CUDA_CHECK(cudaStreamSynchronize(e->st));
    for (int i = 0; i < n; ++i) prob_out[i] = e->res_host[i].no_speech;
    WLK_API_END
}
int wlk_suppress(wlk_engine* e, const int32_t* sids, int n, const int32_t* token_ids, int n_tokens) {
    WLK_API_BEGIN
    LOCK(e);
    WLK_CHECK(sids && n >= 1 && n <= e->cfg.max_batch && n_tokens >= 0 && n_tokens <= 4096, "bad arguments");
    Stager sg(e);
    LogitJob* lj_dev; LogitJob* lj = sg.host<LogitJob>(n, &lj_dev);
    int32_t* tk_dev; int32_t* tk = sg.host<int32_t>(n_tokens > 0 ? n_tokens : 1, &tk_dev);
    for (int i = 0; i < n; ++i) lj[i] = make_logit_job(e, get_session(e, sids[i]), 16, 0);
    for (int i = 0; i < n_tokens; ++i) {
        WLK_CHECK(token_ids[i] >= 0 && token_ids[i] < e->dims.n_vocab, "token %d out of range", token_ids[i]);
        tk[i] = token_ids[i];
    }
    sg.upload();
    {   ProfScope ps(e, WLK_KC_LOGITS);
        suppress_tokens(lj_dev, n, tk_dev, n_tokens, e->st); }
    WLK_API_END
}
int wlk_add_logit_bias(wlk_engine* e, int32_t sid, const int32_t* token_ids, const float* bias, int n) {
    WLK_API_BEGIN
    LOCK(e);
    Session& s = get_session(e, sid);
    WLK_CHECK(n >= 0 && n <= 4096, "bad count");
    if (n) {
        Stager sg(e);
        int32_t* tk_dev; int32_t* tk = sg.host<int32_t>(n, &tk_dev);
        float* b_dev; float* b = sg.host<float>(n, &b_dev);
        for (int i = 0; i < n; ++i) {
            WLK_CHECK(token_ids[i] >= 0 && token_ids[i] < e->dims.n_vocab, "token %d out of range", token_ids[i]);
            tk[i] = token_ids[i]; b[i] = bias[i];
        }
        sg.upload();
        add_logit_bias(s.logits_last, tk_dev, b_dev, n, e->st);
    }
    WLK_API_END
}
int wlk_greedy_and_align(wlk_engine* e, const int32_t* sids, int n, int32_t window_iters, int32_t* token_out,
                         float* logprob_out, int32_t* frame_out) {
    WLK_API_BEGIN
    LOCK(e);
    WLK_CHECK(sids && token_out && logprob_out && frame_out && n >= 1 && n <= e->cfg.max_batch && window_iters >= 1, "bad arguments");
    Stager sg(e);
    LogitJob* lj_dev; LogitJob* lj = sg.host<LogitJob>(n, &lj_dev);
    for (int i = 0; i < n; ++i) {
        Session& s = get_session(e, sids[i]);
        WLK_CHECK(!s.iter_row_start.empty(), "session %d: no decode call in this epoch", sids[i]);
        lj[i] = make_logit_job(e, s, window_iters, 0);
    }
    sg.upload();
    {   ProfScope ps(e, WLK_KC_LOGITS);
        greedy_pick(lj_dev, n, e->dims.n_vocab, e->res_dev, e->st); }
    {   ProfScope ps(e, WLK_KC_ALIGN);
        align_reduce(lj_dev, n, e->n_align, e->dims.n_text_ctx, e->res_dev, e->st); }
    CUDA_CHECK(cudaMemcpyAsync(e->res_host, e->res_dev, sizeof(StepResult) * n, cudaMemcpyDeviceToHost, e->st));
    CUDA_CHECK(cudaStreamSynchronize(e->st));
    for (int i = 0; i < n; ++i) {
        token_out[i] = e->res_host[i].token; logprob_out[i] = e->res_host[i].logprob; frame_out[i] = e->res_host[i].frame;
    }
    WLK_API_END
}

// The whole "pick" half of a policy iteration in one call (one lock, one staging upload, one sync): suppression sets,
// DRY biases, greedy token + logprob, alignment reduction and attended frame.
int wlk_select(wlk_engine* e, const int32_t* sids, int n, const int32_t* suppress_ids, int n_suppress,
               const int32_t* first_ids, int n_first, const uint8_t* first_mask, const int32_t* bias_tokens,
               const float* bias_values, const int32_t* bias_offsets, int32_t window_iters, int32_t* token_out,
               float* logprob_out, int32_t* frame_out) {
    WLK_API_BEGIN
    LOCK(e);
    WLK_CHECK(sids && token_out && logprob_out && frame_out && n >= 1 && n <= e->cfg.max_batch && window_iters >= 1, "bad arguments");
    WLK_CHECK(n_suppress >= 0 && n_suppress <= 4096 && n_first >= 0 && n_first <= 64, "bad suppression lists");
    const int n_bias = bias_offsets ? bias_offsets[n] : 0;
    WLK_CHECK(n_bias >= 0 && n_bias <= 64 * n, "bad bias lists");
    Stager sg(e);
    LogitJob* lj_dev; LogitJob* lj = sg.host<LogitJob>(n, &lj_dev);
    LogitJob* fj_dev; LogitJob* fj = sg.host<LogitJob>(n, &fj_dev);
    int32_t* sup_dev; int32_t* sup = sg.host<int32_t>(n_suppress > 0 ? n_suppress : 1, &sup_dev);
    int32_t* fst_dev; int32_t* fst = sg.host<int32_t>(n_first > 0 ? n_first : 1, &fst_dev);
    int32_t* bj_dev; int32_t* bj = sg.host<int32_t>(n_bias > 0 ? n_bias : 1, &bj_dev);
    int32_t* bt_dev; int32_t* bt = sg.host<int32_t>(n_bias > 0 ? n_bias : 1, &bt_dev);
    float* bv_dev; float* bv = sg.host<float>(n_bias > 0 ? n_bias : 1, &bv_dev);
    int nf = 0;
    for (int i = 0; i < n; ++i) {
        Session& s = get_session(e, sids[i]);
        WLK_CHECK(!s.iter_row_start.empty(), "session %d: no decode call in this epoch", sids[i]);
        for (int j = 0; j < i; ++j) WLK_CHECK(sids[j] != sids[i], "session %d appears twice in the batch", sids[i]);
        lj[i] = make_logit_job(e, s, window_iters, 0);
        if (first_mask && first_mask[i]) fj[nf++] = lj[i];
        if (n_bias) {
            WLK_CHECK(bias_offsets[i + 1] >= bias_offsets[i], "bias offsets must be non-decreasing");
            for (int k = bias_offsets[i]; k < bias_offsets[i + 1]; ++k) {
                WLK_CHECK(bias_tokens[k] >= 0 && bias_tokens[k] < e->dims.n_vocab, "token %d out of range", bias_tokens[k]);
                bj[k] = i; bt[k] = bias_tokens[k]; bv[k] = bias_values[k];
            }
        }
    }
    auto check_ids = [&](const int32_t* ids, int cnt, int32_t* dst) {
        for (int i = 0; i < cnt; ++i) {
            WLK_CHECK(ids[i] >= 0 && ids[i] < e->dims.n_vocab, "token %d out of range", ids[i]);
            dst[i] = ids[i];
        }
    };
    check_ids(suppress_ids, n_suppress, sup);
    check_ids(first_ids, n_first, fst);
    sg.upload();
    {   ProfScope ps(e, WLK_KC_LOGITS);
        if (nf && n_first) suppress_tokens(fj_dev, nf, fst_dev, n_first, e->st);
        suppress_tokens(lj_dev, n, sup_dev, n_suppress, e->st);
        add_logit_bias_jobs(lj_dev, bj_dev, bt_dev, bv_dev, n_bias, e->st);
        greedy_pick(lj_dev, n, e->dims.n_vocab, e->res_dev, e->st); }
    {   ProfScope ps(e, WLK_KC_ALIGN);
        align_reduce(lj_dev, n, e->n_align, e->dims.n_text_ctx, e->res_dev, e->st); }
    CUDA_CHECK(cudaMemcpyAsync(e->res_host, e->res_dev, sizeof(StepResult) * n, cudaMemcpyDeviceToHost, e->st));
    CUDA_CHECK(cudaStreamSynchronize(e->st));
    for (int i = 0; i < n; ++i) {
        token_out[i] = e->res_host[i].token; logprob_out[i] = e->res_host[i].logprob; frame_out[i] = e->res_host[i].frame;
    }
    WLK_API_END
}

// ---- debug taps ---------------------------------------------------------------------------
int wlk_read_mel(wlk_engine* e, int32_t sid, float* out) {
    WLK_API_BEGIN
    LOCK(e);
    Session& s = get_root_session(e, sid, "the mel");
    WLK_CHECK(out && s.encoded, "session not encoded");
    const int nm = e->dims.n_mels;
    // re-run the finalize pass into an fp32 time-major scratch (att is free between calls)
    Stager sg(e);
    MelJob* mj_dev; MelJob* mj = sg.host<MelJob>(1, &mj_dev);
    const int64_t N = s.audio_len;
    int64_t n_compute = (N + 199) / HOP + 1;
    if (n_compute > MEL_MAX_FRAMES) n_compute = MEL_MAX_FRAMES;
    float* scratch = e->mel_scratch;
    mj[0].audio = s.audio; mj[0].raw = s.mel_raw; mj[0].blockmax = s.mel_blockmax; mj[0].out = scratch;
    mj[0].n = (int32_t)N; mj[0].n_compute = (int32_t)n_compute; mj[0].n_total = (int32_t)((N + 480000) / HOP); mj[0].pad = 0;
    WLK_CHECK(s.mel_n == N && s.mel_dropped == 0, "read_mel: the audio changed since the last encode");
    // the tap shows what the encoder consumed: the session's cached raw rows (however they were produced -- moved or
    // recomputed) go through the clamp / scale pass again; only audio longer than the stored rows is recomputed
    mj[0].keep_lo = 0; mj[0].keep_hi = n_compute <= MEL_STORE_FRAMES ? (int32_t)n_compute : 0;
    sg.upload();
    mel_forward(mj_dev, 1, nm, e->w.filtT, e->w.window, e->w.twiddle, e->w.filt_span, DT_F32, (int)n_compute, e->st);
    float* h = tap_buffer(e, (size_t)MEL_ROWS * nm);
    CUDA_CHECK(cudaMemcpyAsync(h, scratch, (size_t)MEL_ROWS * nm * 4, cudaMemcpyDeviceToHost, e->st));
    CUDA_CHECK(cudaStreamSynchronize(e->st));
    for (int m = 0; m < nm; ++m)
        for (int f = 0; f < N_FRAMES; ++f) out[(size_t)m * N_FRAMES + f] = h[(size_t)(f + 1) * nm + m];
    WLK_API_END
}
int wlk_read_encoder(wlk_engine* e, int32_t sid, float* out) {
    WLK_API_BEGIN
    LOCK(e);
    Session& s = enc_owner(e, get_session(e, sid));
    WLK_CHECK(out && s.encoded, "session not encoded");
    const size_t n = (size_t)N_CTX * e->dims.n_audio_state;
    float* h = tap_buffer(e, n);
    convert_to_f32(s.xa, e->act, e->x, (int64_t)n, e->st);
    CUDA_CHECK(cudaMemcpyAsync(h, e->x, n * 4, cudaMemcpyDeviceToHost, e->st));
    CUDA_CHECK(cudaStreamSynchronize(e->st));
    const size_t dd = e->dims.n_audio_state, head = (size_t)(N_CTX - s.rot) * dd;      // ring slot -> logical position
    memcpy(out, h + (size_t)s.rot * dd, head * 4);
    memcpy(out + head, h, (n - head) * 4);
    WLK_API_END
}
int wlk_read_logits(wlk_engine* e, int32_t sid, int32_t which, float* out) {
    WLK_API_BEGIN
    LOCK(e);
    Session& s = get_session(e, sid);
    WLK_CHECK(out && !s.iter_row_start.empty(), "no decode call in this epoch");
    CUDA_CHECK(cudaMemcpyAsync(out, which ? s.logits_sot : s.logits_last, (size_t)e->dims.n_vocab * 4, cudaMemcpyDeviceToHost, e->st));
    CUDA_CHECK(cudaStreamSynchronize(e->st));
    WLK_API_END
}
int wlk_read_align_attn(wlk_engine* e, int32_t sid, float* out, int64_t capacity, int32_t* rows, int32_t* cols) {
    WLK_API_BEGIN
    LOCK(e);
    Session& s = get_session(e, sid);
    WLK_CHECK(out && rows && cols && !s.iter_row_start.empty(), "no decode call in this epoch");
    Stager sg(e);
    LogitJob* lj_dev; LogitJob* lj = sg.host<LogitJob>(1, &lj_dev);
    lj[0] = make_logit_job(e, s, 16, 1);
    const int T = lj[0].row_end - lj[0].row_begin, C = lj[0].content_len;
    WLK_CHECK((int64_t)T * C <= capacity, "output buffer too small: need %d x %d", T, C);
    sg.upload();
    align_reduce(lj_dev, 1, e->n_align, e->dims.n_text_ctx, e->res_dev, e->st);
    float* h = tap_buffer(e, (size_t)T * N_CTX);
    CUDA_CHECK(cudaMemcpyAsync(h, s.attn_out, (size_t)T * N_CTX * 4, cudaMemcpyDeviceToHost, e->st));
    CUDA_CHECK(cudaStreamSynchronize(e->st));
    for (int t = 0; t < T; ++t) memcpy(out + (size_t)t * C, h + (size_t)t * N_CTX, (size_t)C * 4);
    *rows = T; *cols = C;
    WLK_API_END
}

// ---- op-level entry points ---------------------------------------------------------------------
int wlk_op_gemm(wlk_engine* e, int backend, const void* A, int a_type, int64_t lda, const void* Wm, int w_type, int64_t ldw,
                const float* bias, void* C, int c_type, int64_t ldc, int M, int N, int K, int gelu) {
    WLK_API_BEGIN
    LOCK(e);
    WLK_CHECK(A && Wm && C, "null argument");
    WLK_CHECK(M >= 1 && N >= 1 && K >= 1, "empty problem %d x %d x %d", M, N, K);
    CallBuffers cb(e);
    GemmArgs g;
    g.A = A; g.a_type = a_type; g.lda = lda; g.W = Wm; g.w_type = w_type; g.ldw = ldw; g.M = M; g.N = N; g.K = K;
    g.epi.bias = bias; g.epi.gelu = gelu & 1; g.epi.C = C; g.epi.c_type = c_type; g.epi.ldc = ldc;
    g.sk_scratch = e->sk_scratch; g.sk_scratch_floats = SK_SCRATCH_FLOATS;
    g.sk_counters = e->sk_counters; g.sk_max_tiles = SK_MAX_TILES;
    if (gelu & 2) { WLK_CHECK(c_type == DT_F32, "in-place accumulation needs an fp32 output"); g.epi.residual = (const float*)C; g.epi.ldr = ldc; }
    if (w_type == DT_BF16X2) {
        // split operands (the bf16x3 mode): W is the hi plane with the lo plane right behind it, as run_gemm lays out
        // the weights; the fp32 A is split into (hi, lo) planes over its whole range (M - 1) lda + K (overlapping
        // conv views included), in the engine's scratch when it is large enough, else in per-call memory
        WLK_CHECK(backend == WLK_BACKEND_TCGEN05 || backend == 3 || backend == 4,
                  "the bf16x3 GEMM runs on the tensor cores only (backend 2, 3 or 4)");
        WLK_CHECK(lda >= 1 && ldw >= K, "bad row pitch");
        g.W_lo = reinterpret_cast<const bf16*>(Wm) + (size_t)N * ldw;
        const size_t need = ((size_t)(M - 1) * lda + K + 7) / 8 * 8;   // whole 16-byte units: the lo plane stays aligned
        if (e->a_split && need <= e->a_split_elems) { g.a_split = e->a_split; g.a_split_elems = e->a_split_elems; }
        else { g.a_split = cb.take(need * 2 * sizeof(bf16)); g.a_split_elems = need; }
    }
    ProfScope ps(e, WLK_KC_MISC, 2.0 * M * (double)N * K, 0);
    if (backend == WLK_BACKEND_TCGEN05) gemm_tcgen05(g, e->st, e->num_sms, 0);
    else if (backend == 3) gemm_tcgen05(g, e->st, e->num_sms, 1);
    else if (backend == 4) gemm_tcgen05(g, e->st, e->num_sms, 2);
    else gemm_simt(g, e->st);
    WLK_API_END
}
int wlk_op_encoder_attention(wlk_engine* e, int backend, const void* qkv, int type, int batch, void* out) {
    WLK_API_BEGIN
    LOCK(e);
    WLK_CHECK(aligned16(qkv) && aligned16(out), "qkv and out must be non-null and 16-byte aligned");
    WLK_CHECK(batch >= 1, "batch %d < 1", batch);
    const int H = e->dims.n_audio_head, d = e->dims.n_audio_state;
    ProfScope ps(e, WLK_KC_MISC, 4.0 * batch * H * (double)N_CTX * N_CTX * 64, 0);
    if (type == DT_BF16X2) {
        // split planes (the bf16x3 mode): qkv is the hi plane [batch * 1500, 3d] bf16, the lo plane right behind it;
        // out is fp32
        WLK_CHECK(backend == WLK_BACKEND_TCGEN05 || backend == 3, "split-plane attention runs on the tensor cores (backend 2 or 3)");
        const bf16* hi = reinterpret_cast<const bf16*>(qkv);
        enc_attention_tcgen05_x3(hi, hi + (size_t)batch * N_CTX * 3 * d, batch, H, d, reinterpret_cast<float*>(out), e->st);
    } else if (backend == WLK_BACKEND_TCGEN05 || backend == 3) {
        WLK_CHECK(type == DT_BF16, "tcgen05 attention needs bf16");
        if (backend == 3) enc_attention_tcgen05_one_tile(qkv, batch, H, d, out, e->st);   // 3 = force the one-tile CTA
        else enc_attention_tcgen05(qkv, batch, H, d, out, e->st, e->num_sms);
    } else {
        WLK_CHECK(backend == WLK_BACKEND_SIMT, "backend %d: 1 = SIMT, 2 = tcgen05, 3 = one-tile tcgen05", backend);
        WLK_CHECK(type == DT_F32 || type == DT_BF16, "type %d: 0 = fp32, 1 = bf16, 2 = split bf16 planes", type);
        enc_attention_simt(qkv, type, batch, H, d, out, e->st);
    }
    WLK_API_END
}

int wlk_op_decoder_attention(wlk_engine* e, int kind, int backend, int type, int layer, const void* q, int n_jobs,
                             const int32_t* n_rows, const int32_t* offsets, const int32_t* align_row0,
                             const void* const* kv, float* const* align, void* out) {
    WLK_API_BEGIN
    LOCK(e);
    const wlk_dims& D = e->dims;
    const int ctx = D.n_text_ctx;
    WLK_CHECK(kind == 0 || kind == 1, "kind %d: 0 = causal self-attention, 1 = cross-attention", kind);
    WLK_CHECK(backend == WLK_BACKEND_SIMT || backend == WLK_BACKEND_TCGEN05, "backend %d: 1 = SIMT, 2 = tcgen05", backend);
    WLK_CHECK(type == DT_F32 || type == DT_BF16, "type %d: 0 = fp32, 1 = bf16", type);
    WLK_CHECK(backend == WLK_BACKEND_SIMT || type == DT_BF16, "the tcgen05 decoder attention needs bf16");
    WLK_CHECK(layer >= 0 && layer < D.n_text_layer, "layer %d outside [0, %d)", layer, D.n_text_layer);
    WLK_CHECK(n_jobs >= 1 && n_jobs <= 65535, "%d jobs outside [1, 65535]", n_jobs);
    WLK_CHECK(n_rows && offsets && kv, "null argument");
    WLK_CHECK(aligned16(q) && aligned16(out), "q and out must be non-null and 16-byte aligned");
    const bool cross = kind == 1;
    if (cross) WLK_CHECK(align_row0 && align, "cross-attention needs align_row0 and align");
    std::vector<DecJob> jobs(n_jobs);
    int R = 0, max_rows = 0;
    for (int i = 0; i < n_jobs; ++i) {
        const int nr = n_rows[i], off = offsets[i];
        WLK_CHECK(nr >= 1 && off >= 0 && off <= ctx - nr, "job %d: rows at positions [%d, %d + %d) outside n_text_ctx %d",
                  i, off, off, nr, ctx);
        WLK_CHECK(aligned16(kv[i]), "job %d: kv must be non-null and 16-byte aligned", i);
        DecJob& j = jobs[i];
        memset(&j, 0, sizeof(DecJob));
        j.row_off = R; j.n_rows = nr; j.offset = off; j.slot = i;     // slot: the job's tensor map in this call's array
        if (cross) {
            const int a0 = align_row0[i];
            WLK_CHECK(a0 >= 0 && a0 <= ctx - nr, "job %d: alignment rows [%d, %d + %d) outside n_text_ctx %d", i, a0, a0, nr, ctx);
            WLK_CHECK(aligned16(align[i]), "job %d: align must be non-null and 16-byte aligned", i);
            j.cross_kv = kv[i]; j.align = align[i]; j.align_row0 = a0;
        } else {
            j.self_kv = const_cast<void*>(kv[i]);
        }
        R += nr;
        max_rows = std::max(max_rows, nr);
    }
    const bool tc = backend == WLK_BACKEND_TCGEN05;
    CallBuffers cb(e);
    DecJob* jobs_dev = reinterpret_cast<DecJob*>(cb.take(jobs.size() * sizeof(DecJob)));
    CUDA_CHECK(cudaMemcpyAsync(jobs_dev, jobs.data(), jobs.size() * sizeof(DecJob), cudaMemcpyHostToDevice, e->st));
    uint8_t* maps_dev = nullptr;
    if (tc) {
        std::vector<uint8_t> maps((size_t)n_jobs * 128);
        for (int i = 0; i < n_jobs; ++i) {
            alignas(64) uint8_t tmap[128];
            if (cross) make_cross_kv_tmap(tmap, kv[i], D.n_text_layer, D.n_text_head);
            else make_self_kv_tmap(tmap, kv[i], D.n_text_layer, D.n_text_head, ctx);
            memcpy(maps.data() + (size_t)i * 128, tmap, 128);
        }
        maps_dev = reinterpret_cast<uint8_t*>(cb.take(maps.size()));
        CUDA_CHECK(cudaMemcpyAsync(maps_dev, maps.data(), maps.size(), cudaMemcpyHostToDevice, e->st));
    }
    ProfScope ps(e, cross ? WLK_KC_ATTN_DEC_CROSS : WLK_KC_ATTN_DEC_SELF);
    if (cross) dec_cross_attention_layer(e, q, type, R, jobs_dev, n_jobs, max_rows, layer, maps_dev, out, tc);
    else dec_self_attention_layer(e, q, type, R, jobs_dev, n_jobs, max_rows, layer, maps_dev, out, tc);
    WLK_API_END
}

int wlk_op_encoder_attention_trace(wlk_engine* e, const void* qkv, int batch, void* out, int64_t* stamps_host /*[12][8]*/) {
    WLK_API_BEGIN
    LOCK(e);
    WLK_CHECK(qkv && out && stamps_host, "null argument");
    long long* dev = nullptr;
    CUDA_CHECK(cudaMalloc(&dev, 96 * 8));
    CUDA_CHECK(cudaMemsetAsync(dev, 0, 96 * 8, e->st));
    enc_attention_tcgen05(qkv, batch, e->dims.n_audio_head, e->dims.n_audio_state, out, e->st, e->num_sms, dev);
    CUDA_CHECK(cudaMemcpyAsync(stamps_host, dev, 96 * 8, cudaMemcpyDeviceToHost, e->st));
    CUDA_CHECK(cudaStreamSynchronize(e->st));
    cudaFree(dev);
    WLK_API_END
}

int wlk_op_median_filter(wlk_engine* e, const float* x_dev, float* out_dev, int rows, int cols, int width) {
    WLK_API_BEGIN
    LOCK(e);
    WLK_CHECK(x_dev && out_dev && rows >= 1 && cols >= 1, "bad arguments");
    ProfScope ps(e, WLK_KC_ALIGN);
    median_filter(x_dev, out_dev, rows, cols, width, e->st);
    WLK_API_END
}
int wlk_op_dtw(wlk_engine* e, const float* x_dev, int N, int M, int32_t* text_idx_host, int32_t* time_idx_host,
               int32_t* len_out) {
    WLK_API_BEGIN
    LOCK(e);
    WLK_CHECK(x_dev && text_idx_host && time_idx_host && len_out, "null argument");
    WLK_CHECK(N >= 1 && N <= 4096 && M >= 1 && M <= 8192, "dtw: shape %d x %d out of range", N, M);
    size_t acct = 0;
    uint8_t* trace = dmalloc<uint8_t>(e, (size_t)(N + 1) * (M + 1), &acct);
    int32_t* path = dmalloc<int32_t>(e, (size_t)4 * (N + M) + 4, &acct);
    int32_t* plen = dmalloc<int32_t>(e, 1, &acct);
    DtwJobHost* job_dev = dmalloc<DtwJobHost>(e, 1, &acct);
    DtwJobHost job{x_dev, trace, path, plen, N, M};
    CUDA_CHECK(cudaMemcpyAsync(job_dev, &job, sizeof(job), cudaMemcpyHostToDevice, e->st));
    {   ProfScope ps(e, WLK_KC_ALIGN);
        dtw_batch(job_dev, 1, N, e->st); }
    std::vector<int32_t> host((size_t)2 * (N + M));
    int32_t n = 0;
    CUDA_CHECK(cudaMemcpyAsync(&n, plen, 4, cudaMemcpyDeviceToHost, e->st));
    CUDA_CHECK(cudaMemcpyAsync(host.data(), path, host.size() * 4, cudaMemcpyDeviceToHost, e->st));
    CUDA_CHECK(cudaStreamSynchronize(e->st));
    cudaFree(trace); cudaFree(path); cudaFree(plen); cudaFree(job_dev);
    WLK_CHECK(n >= 1 && n <= N + M, "dtw: bad path length %d", n);
    memcpy(text_idx_host, host.data(), (size_t)n * 4);
    memcpy(time_idx_host, host.data() + (N + M), (size_t)n * 4);
    *len_out = n;
    WLK_API_END
}

// ---- timers / profile ------------------------------------------------------------------------
int wlk_timer_record(wlk_engine* e, int slot) {
    WLK_API_BEGIN
    LOCK(e);
    WLK_CHECK(slot >= 0 && slot < 16, "timer slot out of range");
    CUDA_CHECK(cudaEventRecord(e->timers[slot], e->st));
    WLK_API_END
}
int wlk_timer_elapsed_ms(wlk_engine* e, int from_slot, int to_slot, float* ms) {
    WLK_API_BEGIN
    LOCK(e);
    WLK_CHECK(from_slot >= 0 && from_slot < 16 && to_slot >= 0 && to_slot < 16 && ms, "bad arguments");
    CUDA_CHECK(cudaEventSynchronize(e->timers[to_slot]));
    CUDA_CHECK(cudaEventElapsedTime(ms, e->timers[from_slot], e->timers[to_slot]));
    WLK_API_END
}
int wlk_profile_enable(wlk_engine* e, int on) {
    WLK_API_BEGIN
    LOCK(e);
    e->prof_on = on != 0;
    WLK_API_END
}
int wlk_profile_reset(wlk_engine* e) {
    WLK_API_BEGIN
    LOCK(e);
    CUDA_CHECK(cudaStreamSynchronize(e->st));
    for (auto& p : e->prof) e->ev_pool.push_back({p.a, p.b});
    e->prof.clear();
    WLK_API_END
}
int wlk_profile_read(wlk_engine* e, int cls, double* ms, int64_t* launches, double* flops, double* bytes) {
    WLK_API_BEGIN
    LOCK(e);
    WLK_CHECK(cls >= 0 && cls < WLK_KC_COUNT, "class out of range");
    CUDA_CHECK(cudaStreamSynchronize(e->st));
    double t = 0, f = 0, b = 0; int64_t n = 0;
    for (auto& p : e->prof) {
        if (p.cls != cls) continue;
        float m = 0;
        CUDA_CHECK(cudaEventElapsedTime(&m, p.a, p.b));
        t += m; f += p.flops; b += p.bytes; ++n;
    }
    if (ms) *ms = t;
    if (launches) *launches = n;
    if (flops) *flops = f;
    if (bytes) *bytes = b;
    WLK_API_END
}
int wlk_profile_class_name(int cls, const char** name) {
    if (cls < 0 || cls >= WLK_KC_COUNT || !name) { wlk::set_last_error("class out of range"); return 1; }
    *name = wlk::kClassNames[cls];
    return 0;
}

}  // extern "C"
