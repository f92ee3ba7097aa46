// Fused encoder self-attention on the 5th-gen tensor cores (sm_100a).
//   O = softmax(Q K^T) V over all 1500 positions, no mask (reference whisper/model.py:148-173);
//   q and k arrive pre-scaled by d_head^-0.25 from the QKV GEMM epilogue.
//
// One CTA per (128-query tile, head, stream); two CTAs are co-resident per SM (80 KB smem, 256 TMEM
// columns each) so one CTA's exponentials overlap the other's MMAs.
//   warp 0     TMA producer : Q tile once, then 128-key K and V tiles (128B-swizzled) through a
//                             2-stage mbarrier ring, straight out of the fused [rows, 3d] qkv buffer
//   warp 1     MMA issuer   : S = Q K^T   (tcgen05.mma SS, M128 N128 K16 x4)      -> TMEM cols [0,128)
//                             O_j = P V   (tcgen05.mma TS: P from TMEM, V MN-major smem, N64, K16 x8)
//                                                                                  -> TMEM cols [128,192)
//   warps 2-9  softmax      : two threads per query row (64 keys of the tile each). tcgen05.ld S in 16-column
//                             chunks, ONE pass: exp2 against the row's reference maximum, row sum, and the
//                             tile's true maximum on the side; P packed to bf16 and written back to TMEM
//                             (cols [192,256)) with tcgen05.st.  O stays in TMEM across key tiles and is only
//                             rescaled when the reference maximum has to move (rare); final O / l as bf16.
#include <cudaTypedefs.h>

#include <type_traits>

#include "kernels.cuh"
#include "ptx.cuh"

namespace wlk {

bool make_tmap_bf16_2d(CUtensorMap* tm, const void* ptr, uint64_t rows, uint64_t cols, uint64_t ld,
                       uint32_t box_rows, uint32_t box_cols, std::string* err);

namespace {

constexpr int BQ = 128, BKV = 128, DH = 64;
constexpr int ATT_THREADS = 320;          // TMA warp, MMA warp, 8 softmax warps
constexpr uint32_t TILE_BYTES = BQ * DH * 2;          // 16 KB: Q, K and V tiles all are 128 x 64 bf16
// Shared-memory / TMEM layout.  X3 (WLK_PREC_BF16X3): every operand is two bf16 planes (hi, lo); Q K^T and P V are each
// three MMAs (hi hi + lo hi + hi lo) into the same fp32 accumulator, P is split like the other operands, the output is
// fp32.  Twice the tiles and 320 TMEM columns: one CTA per SM instead of two.
template <bool X3> struct AttLayout {
    static constexpr uint32_t NP = X3 ? 2 : 1;                               // planes per operand
    static constexpr uint32_t SM_Q = 0;                                      // [NP] tiles
    static constexpr uint32_t SM_K = NP * TILE_BYTES;                        // [2 stages][NP]
    static constexpr uint32_t SM_V = SM_K + 2 * NP * TILE_BYTES;             // [2 stages][NP]
    static constexpr uint32_t SM_BAR = SM_V + 2 * NP * TILE_BYTES;
    static constexpr uint32_t SM_XCH = SM_BAR + 128;                         // row-half exchange: [2][2][128] floats
    static constexpr uint32_t SMEM = SM_XCH + 2 * 2 * BQ * 4 + 1024;
    static constexpr uint32_t TM_COLS = X3 ? 512 : 256;
};
constexpr uint32_t TM_S = 0, TM_O = 128, TM_P = 192, TM_PLO = 256;
constexpr float LOG2E = 1.4426950408889634f;

__device__ __forceinline__ float fast_exp2(float x) {      // MUFU.EX2, flush-to-zero, exp2(-inf) = 0
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

__device__ __forceinline__ void tmem_st_32x16(uint32_t taddr, const uint32_t* r) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, "
        "%15, %16};"
        ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
          "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
        : "memory");
}
__device__ __forceinline__ void tmem_st_32x32(uint32_t taddr, const uint32_t* r) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
        "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
        ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
          "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]),
          "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]),
          "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
        : "memory");
}
__device__ __forceinline__ void tmem_st_32x8(uint32_t taddr, const uint32_t* r) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
                 ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
                 : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]
__device__ __forceinline__ void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc,
                                             uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
        ::"r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}

// MODE 0: encoder self-attention, Q/K/V tiles all come out of the fused qkv buffer (tensor map `tm`).
// MODE 1: decoder cross-attention of a prefill (many query rows per session): Q tiles from the packed
//         query buffer (`tm`), K/V tiles from the session's head-major cross-K/V planes through a
//         per-session tensor map kept in global memory (`kv_maps[job.slot]`).  Alignment heads are
//         skipped here: their rows need the exactly normalised probabilities exported, which the
//         SIMT kernel produces.
// MODE 2: decoder SELF-attention of a prefill, causal: Q as in mode 1, K/V tiles from the session's self-K/V
//         cache planes [L][2][H][n_text_ctx][64] (per-session tensor map); query row at position p sees keys
//         0..p -- the mask is applied per row where the probabilities are formed (masked keys get exactly 0),
//         and only the key tiles up to the tile's last position are visited.  A long context prefix (the
//         reference keeps up to n_text_ctx - 20 = 428 tokens, align_att_base.py:100-113) costs ~90 k query
//         rows x 32 layers per tick at 48 streams: on the SIMT kernel that was half of the tick.
constexpr int MODE_ENC = 0, MODE_CROSS = 1, MODE_SELF = 2;
template <int MODE, bool X3>
__global__ void __launch_bounds__(ATT_THREADS, X3 ? 1 : 2)
attn_tc_kernel(const __grid_constant__ CUtensorMap tm, const __grid_constant__ CUtensorMap tm_lo,
               const CUtensorMap* __restrict__ kv_maps,
               const DecJob* __restrict__ jobs, int layer, const int32_t* __restrict__ align_rank,
               int n_head, int d_model, int kv_len, void* __restrict__ out_ptr, long long* __restrict__ trace = nullptr) {
    // diagnostic (tools/attn_trace.py): one CTA in the middle of the grid stamps clock64() at its pipeline hand-offs
    const bool tr = trace != nullptr && blockIdx.x == 3 && blockIdx.y == 1 && blockIdx.z == gridDim.z / 2;
    constexpr bool CROSS = MODE != MODE_ENC;              // Q from the packed query buffer, K/V through a per-session map
    static_assert(!(CROSS && X3), "the split-operand variant serves the encoder only");
    using AL = AttLayout<X3>;
    constexpr uint32_t SM_Q = AL::SM_Q, SM_K = AL::SM_K, SM_V = AL::SM_V, SM_BAR = AL::SM_BAR, SM_XCH = AL::SM_XCH;
    constexpr uint32_t TM_COLS = AL::TM_COLS, NP = AL::NP;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t sbase = (ptx::smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t* sgen = smem_raw + (sbase - ptx::smem_u32(smem_raw));
    const uint32_t bar_q = sbase + SM_BAR;
    const uint32_t bar_kv_full = bar_q + 8;       // [2]
    const uint32_t bar_kv_empty = bar_q + 24;     // [2]
    const uint32_t bar_s_full = bar_q + 40;
    const uint32_t bar_s_free = bar_q + 48;
    const uint32_t bar_p_full = bar_q + 56;
    const uint32_t bar_o_full = bar_q + 64;
    const uint32_t tmem_slot = bar_q + 72;
    volatile uint32_t* tmem_slot_gen = reinterpret_cast<volatile uint32_t*>(sgen + SM_BAR + 72);

    ptx::griddep_launch();                   // programmatic dependent launch: see launch_pdl (common.cuh)
    ptx::griddep_wait();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int q0 = blockIdx.x * BQ, h = blockIdx.y, b = blockIdx.z;
    int NT = (N_CTX + BKV - 1) / BKV;                    // 12 key tiles (encoder, cross)
    int pos0 = 0;                                        // MODE_SELF: position of the tile's first query row
    // tile origins (tensor-map coordinates) and the number of query rows this CTA owns
    const CUtensorMap* tm_kv = &tm;
    int q_row, q_col = h * DH, k_row, k_col, v_row, v_col, out_row, n_q;
    if constexpr (CROSS) {
        const DecJob job = jobs[b];
        if (q0 >= job.n_rows) return;                                            // uniform: before any barrier / TMEM use
        if (MODE == MODE_CROSS && align_rank[layer * n_head + h] >= 0) return;
        tm_kv = kv_maps + job.slot;
        q_row = job.row_off + q0;
        k_row = (((layer * 2 + 0) * n_head) + h) * kv_len; k_col = 0;
        v_row = (((layer * 2 + 1) * n_head) + h) * kv_len; v_col = 0;
        out_row = job.row_off + q0;
        n_q = min(BQ, job.n_rows - q0);
        if (MODE == MODE_SELF) {
            pos0 = job.offset + q0;
            NT = (pos0 + n_q + BKV - 1) / BKV;                                   // keys 0 .. position of the last row
        }
    } else {
        q_row = b * N_CTX + q0;
        k_row = b * N_CTX; k_col = d_model + h * DH;
        v_row = b * N_CTX; v_col = 2 * d_model + h * DH;
        out_row = b * N_CTX + q0;
        n_q = min(BQ, N_CTX - q0);
    }

    if (warp == 0 && lane == 0) {
        ptx::prefetch_tensormap(&tm);
        if (X3) ptx::prefetch_tensormap(&tm_lo);
        if (CROSS) ptx::prefetch_tensormap(tm_kv);
        ptx::mbar_init(bar_q, 1);
        for (int i = 0; i < 2; ++i) { ptx::mbar_init(bar_kv_full + 8 * i, 1); ptx::mbar_init(bar_kv_empty + 8 * i, 1); }
        ptx::mbar_init(bar_s_full, 1);
        ptx::mbar_init(bar_s_free, 256);
        ptx::mbar_init(bar_p_full, 256);
        ptx::mbar_init(bar_o_full, 1);
        ptx::fence_barrier_init();
    }
    if (warp == 1) { ptx::tmem_alloc(tmem_slot, TM_COLS); ptx::tmem_relinquish(); }
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem = *tmem_slot_gen;

    if (warp == 0) {
        if (lane == 0) {
            ptx::mbar_arrive_expect_tx(bar_q, NP * TILE_BYTES);
            ptx::tma_load_2d(sbase + SM_Q, &tm, bar_q, q_col, q_row);
            if (X3) ptx::tma_load_2d(sbase + SM_Q + TILE_BYTES, &tm_lo, bar_q, q_col, q_row);
            for (int j = 0; j < NT; ++j) {
                const uint32_t s = j & 1, ph = (j >> 1) & 1;
                ptx::mbar_wait(bar_kv_empty + 8 * s, ph ^ 1);
                ptx::mbar_arrive_expect_tx(bar_kv_full + 8 * s, 2 * NP * TILE_BYTES);
                ptx::tma_load_2d(sbase + SM_K + s * NP * TILE_BYTES, tm_kv, bar_kv_full + 8 * s, k_col, k_row + j * BKV);
                ptx::tma_load_2d(sbase + SM_V + s * NP * TILE_BYTES, tm_kv, bar_kv_full + 8 * s, v_col, v_row + j * BKV);
                if (X3) {
                    ptx::tma_load_2d(sbase + SM_K + (s * NP + 1) * TILE_BYTES, &tm_lo, bar_kv_full + 8 * s, k_col, k_row + j * BKV);
                    ptx::tma_load_2d(sbase + SM_V + (s * NP + 1) * TILE_BYTES, &tm_lo, bar_kv_full + 8 * s, v_col, v_row + j * BKV);
                }
            }
        }
    } else if (warp == 1) {
        constexpr uint32_t idesc_s = ptx::umma_idesc_bf16(BQ, BKV, 0, 0);   // A=Q K-major, B=K K-major
        constexpr uint32_t idesc_o = ptx::umma_idesc_bf16(BQ, DH, 0, 1);    // A=P (TMEM), B=V MN-major
        ptx::mbar_wait(bar_q, 0);
        // Issue order: S_{j+1} = Q K_{j+1}^T goes to the tensor pipe BEFORE P_j V_j.  Both become issuable at the same
        // moment (the softmax warps arrive on s_free and p_full together), and the softmax of tile j+1 only needs S_{j+1}:
        // with P V first it sat behind ~750 clk of P V issue plus ~550 clk of barrier round trips per tile (measured with
        // tools/attn_trace.py: tile period 3 950 clk, of which the exponentials are 2 050).  P and O are single-buffered,
        // so the softmax warps wait for P_j V_j (bar_o_full) before their first write of tile j+1.
        auto issue_s = [&](int j) {
            const uint32_t s = j & 1;
            if (tr && lane == 0) trace[j * 8 + 0] = clock64();
            if (lane == 0) {
                const uint64_t dq = ptx::umma_desc_kmajor_sw128(sbase + SM_Q);
                const uint64_t dk = ptx::umma_desc_kmajor_sw128(sbase + SM_K + s * NP * TILE_BYTES);
                const uint64_t dql = ptx::umma_desc_kmajor_sw128(sbase + SM_Q + TILE_BYTES);
                const uint64_t dkl = ptx::umma_desc_kmajor_sw128(sbase + SM_K + (s * NP + 1) * TILE_BYTES);
#pragma unroll
                for (int k = 0; k < DH / 16; ++k) {
                    ptx::umma_bf16_ss(tmem + TM_S, dq + 2 * k, dk + 2 * k, idesc_s, k > 0 ? 1u : 0u);
                    if (X3) {
                        ptx::umma_bf16_ss(tmem + TM_S, dql + 2 * k, dk + 2 * k, idesc_s, 1u);
                        ptx::umma_bf16_ss(tmem + TM_S, dq + 2 * k, dkl + 2 * k, idesc_s, 1u);
                    }
                }
                ptx::umma_commit(bar_s_full);
            }
            __syncwarp();
        };
        ptx::mbar_wait(bar_kv_full, 0);
        ptx::tc_fence_after();
        issue_s(0);
        for (int j = 0; j < NT; ++j) {
            const uint32_t s = j & 1;
            if (j + 1 < NT) {
                ptx::mbar_wait(bar_kv_full + 8 * ((j + 1) & 1), ((j + 1) >> 1) & 1);
                if (tr && lane == 0) trace[(j + 1) * 8 + 5] = clock64();
                ptx::mbar_wait(bar_s_free, j & 1);            // the softmax threads have read S of tile j
                ptx::tc_fence_after();
                issue_s(j + 1);
            }
            ptx::mbar_wait(bar_p_full, j & 1);                // P of tile j is in TMEM
            ptx::tc_fence_after();
            if (tr && lane == 0) trace[j * 8 + 1] = clock64();
            if (lane == 0) {
                const uint64_t dv = ptx::umma_desc_mnmajor_sw128(sbase + SM_V + s * NP * TILE_BYTES, BKV * 128);
                const uint64_t dvl = ptx::umma_desc_mnmajor_sw128(sbase + SM_V + (s * NP + 1) * TILE_BYTES, BKV * 128);
#pragma unroll
                for (int k = 0; k < BKV / 16; ++k) {           // 16 keys = 16 V rows of 128 B = 2048 B = +128 encoded
                    umma_bf16_ts(tmem + TM_O, tmem + TM_P + 8 * k, dv + 128 * k, idesc_o, (j > 0 || k > 0) ? 1u : 0u);
                    if (X3) {
                        umma_bf16_ts(tmem + TM_O, tmem + TM_PLO + 8 * k, dv + 128 * k, idesc_o, 1u);
                        umma_bf16_ts(tmem + TM_O, tmem + TM_P + 8 * k, dvl + 128 * k, idesc_o, 1u);
                    }
                }
                ptx::umma_commit(bar_o_full);
                ptx::umma_commit(bar_kv_empty + 8 * s);
            }
            __syncwarp();
            if (tr && lane == 0) trace[j * 8 + 7] = clock64();
        }
    } else {
        // ---- softmax: two threads per query row (warps w and w+4 share a TMEM lane quadrant; each owns 64 of
        // the tile's 128 keys), eight warps per CTA, sixteen per SM: enough warps per scheduler to cover the
        // tcgen05.ld round trips with other rows' exponentials.
        const int qd = warp & 3;
        const int half = (warp - 2) >> 2;
        const int r = qd * 32 + lane;                         // query row within the tile == TMEM lane
        const uint32_t lane_addr = static_cast<uint32_t>(qd * 32) << 16;
        const uint32_t s_addr = tmem + lane_addr + TM_S + half * (BKV / 2);
        const uint32_t p_addr = tmem + lane_addr + TM_P + half * (BKV / 4);
        const uint32_t plo_addr = tmem + lane_addr + TM_PLO + half * (BKV / 4);
        const uint32_t o_addr = tmem + lane_addr + TM_O + half * (DH / 2);
        float* xch = reinterpret_cast<float*>(sgen + SM_XCH);  // [2 parities][2 halves][128 rows]
        uint32_t xn = 0;
        // combine a per-thread value with the row's other half (named barrier of the two warps of a quadrant)
        auto exchange = [&](float v) -> float {
            float* slot = xch + (xn & 1) * 2 * BQ;
            ++xn;
            slot[half * BQ + r] = v;
            switch (qd) {                                      // literal ids: ptxas then reserves 5 barriers, not all 16
                case 0: asm volatile("bar.sync 1, 64;" ::: "memory"); break;
                case 1: asm volatile("bar.sync 2, 64;" ::: "memory"); break;
                case 2: asm volatile("bar.sync 3, 64;" ::: "memory"); break;
                default: asm volatile("bar.sync 4, 64;" ::: "memory"); break;
            }
            return slot[(half ^ 1) * BQ + r];
        };
        float m = -INFINITY, l = 0.f;                         // reference max (log2 domain), this half's running sum
        // One pass per key tile.  Probabilities are taken against the row's reference maximum `m`, which is
        // only moved (and O, l rescaled in place in TMEM) when a tile's true maximum -- found during the same
        // pass -- exceeds it by more than 2^8; in that rare case the tile's probabilities are recomputed
        // against the new reference before anything consumes them.  Until then values may exceed 1 by at most
        // 2^8, which bf16 / fp32 hold without loss.  The steady-state tile has no per-element predicates
        // (MASKED only for the last, 92-key tile) and exp2 is a bare MUFU.
        auto tile = [&](int j, auto masked_tag) {
            constexpr bool MASKED = decltype(masked_tag)::value;
            // valid keys among this thread's 64 (MASKED only): the tail of the 1500 frames, or -- causal -- keys up to
            // the row's own position
            const int n_valid = MODE == MODE_SELF ? (pos0 + r + 1) - j * BKV - half * (BKV / 2)
                                                  : N_CTX - j * BKV - half * (BKV / 2);
            ptx::mbar_wait(bar_s_full, j & 1);
            if (j > 0) ptx::mbar_wait(bar_o_full, (j - 1) & 1);   // P_{j-1} V_{j-1} has read P and updated O (it was issued after
            ptx::tc_fence_after();                            // Q K_j^T: see the issue order in the MMA warp)
            if (tr && lane == 0 && warp == 2) trace[j * 8 + 2] = clock64();
            uint32_t va[16], vb[16];
            if (j == 0) {                                     // first tile: a true row maximum seeds the reference
                float mx = -INFINITY;
#pragma unroll 1
                for (int c = 0; c < 4; c += 2) {
                    ptx::tmem_ld_32x16(s_addr + c * 16, va);
                    ptx::tmem_ld_32x16(s_addr + c * 16 + 16, vb);
                    ptx::tmem_ld_wait();
#pragma unroll
                    for (int i = 0; i < 16; ++i) {
                        if (!MASKED || c * 16 + i < n_valid) mx = fmaxf(mx, __uint_as_float(va[i]));
                        if (!MASKED || c * 16 + 16 + i < n_valid) mx = fmaxf(mx, __uint_as_float(vb[i]));
                    }
                }
                m = fmaxf(mx, exchange(mx)) * LOG2E;
            }
#pragma unroll 1
            for (;;) {
                float rs = 0.f, mx = -INFINITY;
                auto emit = [&](const uint32_t* v, int c) {   // 16 scores -> 8 packed words of P
                    uint32_t pk[8];
                    uint32_t pl[X3 ? 8 : 1];
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const float s0 = __uint_as_float(v[2 * i]), s1 = __uint_as_float(v[2 * i + 1]);
                        float p0 = fast_exp2(fmaf(s0, LOG2E, -m));
                        float p1 = fast_exp2(fmaf(s1, LOG2E, -m));
                        if (MASKED) {
                            if (c * 16 + 2 * i >= n_valid) p0 = 0.f; else mx = fmaxf(mx, s0);
                            if (c * 16 + 2 * i + 1 >= n_valid) p1 = 0.f; else mx = fmaxf(mx, s1);
                        } else {
                            mx = fmaxf(mx, fmaxf(s0, s1));
                        }
                        rs += p0 + p1;
                        __nv_bfloat162 hb = __floats2bfloat162_rn(p0, p1);
                        pk[i] = *reinterpret_cast<uint32_t*>(&hb);
                        if (X3) {                             // P = hi + lo like every other operand of this mode
                            __nv_bfloat162 lb = __floats2bfloat162_rn(p0 - __low2float(hb), p1 - __high2float(hb));
                            pl[i] = *reinterpret_cast<uint32_t*>(&lb);
                        }
                    }
                    tmem_st_32x8(p_addr + c * 8, pk);
                    if (X3) tmem_st_32x8(plo_addr + c * 8, pl);
                };
                ptx::tmem_ld_32x16(s_addr, va);
                ptx::tmem_ld_wait();
                ptx::tmem_ld_32x16(s_addr + 16, vb);
                emit(va, 0);
                ptx::tmem_ld_wait();
                ptx::tmem_ld_32x16(s_addr + 32, va);
                emit(vb, 1);
                ptx::tmem_ld_wait();
                ptx::tmem_ld_32x16(s_addr + 48, vb);
                emit(va, 2);
                ptx::tmem_ld_wait();
                emit(vb, 3);
                if (tr && lane == 0 && warp == 2) trace[j * 8 + 3] = clock64();
                const float mx2 = fmaxf(mx, exchange(mx)) * LOG2E;    // the whole row's maximum in this tile
                const bool need = mx2 > m + 8.0f;
                if (!__any_sync(0xffffffffu, need)) { l += rs; break; }   // both warps of the row decide alike
                // rare: move the reference, rescale this half of O and l, then redo the tile's probabilities
                const float alpha = need ? fast_exp2(m - mx2) : 1.0f;
                if (j > 0) {
                    uint32_t o[32];
                    ptx::tmem_ld_32x32(o_addr, o);
                    ptx::tmem_ld_wait();
#pragma unroll
                    for (int i = 0; i < 32; ++i) o[i] = __float_as_uint(__uint_as_float(o[i]) * alpha);
                    tmem_st_32x32(o_addr, o);
                }
                l *= alpha;
                if (need) m = mx2;
            }
            ptx::tc_fence_before();
            ptx::mbar_arrive(bar_s_free);     // S fully consumed (every load has been waited for): the next Q K^T may overwrite
            ptx::tmem_st_wait();              // it while this thread's P stores are still draining
            ptx::tc_fence_before();
            ptx::mbar_arrive(bar_p_full);     // P written, O rescaled if needed: P V may run
            if (tr && lane == 0 && (warp == 2 || warp == 9)) trace[j * 8 + (warp == 2 ? 4 : 6)] = clock64();
        };
        if (MODE == MODE_SELF) {
#pragma unroll 1
            for (int j = 0; j < NT; ++j) tile(j, std::true_type{});
        } else {
#pragma unroll 1
            for (int j = 0; j < NT - 1; ++j) tile(j, std::false_type{});
            tile(NT - 1, std::true_type{});
        }
        ptx::mbar_wait(bar_o_full, (NT - 1) & 1);
        ptx::tc_fence_after();
        const float inv = 1.0f / (l + exchange(l));
        uint32_t v[32];
        ptx::tmem_ld_32x32(o_addr, v);                        // warp-collective: before the row predicate
        ptx::tmem_ld_wait();
        if (X3) {
            float* o = reinterpret_cast<float*>(out_ptr) + (int64_t)(out_row + r) * d_model + h * DH + half * (DH / 2);
            if (r < n_q) {
#pragma unroll
                for (int e4 = 0; e4 < 8; ++e4)
                    reinterpret_cast<float4*>(o)[e4] = make_float4(__uint_as_float(v[e4 * 4 + 0]) * inv, __uint_as_float(v[e4 * 4 + 1]) * inv,
                                                                   __uint_as_float(v[e4 * 4 + 2]) * inv, __uint_as_float(v[e4 * 4 + 3]) * inv);
            }
        } else if (r < n_q) {
            bf16* o = reinterpret_cast<bf16*>(out_ptr) + (int64_t)(out_row + r) * d_model + h * DH + half * (DH / 2);
#pragma unroll
            for (int e8 = 0; e8 < 4; ++e8) {
                uint4 u;
                __nv_bfloat162 h0 = __floats2bfloat162_rn(__uint_as_float(v[e8 * 8 + 0]) * inv, __uint_as_float(v[e8 * 8 + 1]) * inv);
                __nv_bfloat162 h1 = __floats2bfloat162_rn(__uint_as_float(v[e8 * 8 + 2]) * inv, __uint_as_float(v[e8 * 8 + 3]) * inv);
                __nv_bfloat162 h2 = __floats2bfloat162_rn(__uint_as_float(v[e8 * 8 + 4]) * inv, __uint_as_float(v[e8 * 8 + 5]) * inv);
                __nv_bfloat162 h3 = __floats2bfloat162_rn(__uint_as_float(v[e8 * 8 + 6]) * inv, __uint_as_float(v[e8 * 8 + 7]) * inv);
                u.x = *reinterpret_cast<uint32_t*>(&h0); u.y = *reinterpret_cast<uint32_t*>(&h1);
                u.z = *reinterpret_cast<uint32_t*>(&h2); u.w = *reinterpret_cast<uint32_t*>(&h3);
                reinterpret_cast<uint4*>(o)[e8] = u;
            }
        }
    }
    ptx::tc_fence_before();
    __syncthreads();
    if (warp == 1) ptx::tmem_dealloc(tmem, TM_COLS);
}

}  // namespace

void enc_attention_tcgen05_two_tile(const void* qkv, int batch, int n_head, int d_model, void* out, cudaStream_t st);   // attn_tc2.cu

void enc_attention_tcgen05(const void* qkv, int batch, int n_head, int d_model, void* out, cudaStream_t st, int num_sms,
                           long long* trace_dev) {
    (void)num_sms;
    // the serving kernel is the two-query-tile CTA of attn_tc2.cu; WLK_ATTN2=0 (and the pipeline trace) keep this file's
    // one-tile CTA, which also serves the decoder prefills and the split-operand mode
    static const bool two_tile = [] { const char* v = getenv("WLK_ATTN2"); return !(v && v[0] == '0'); }();
    if (two_tile && trace_dev == nullptr) { enc_attention_tcgen05_two_tile(qkv, batch, n_head, d_model, out, st); return; }
    enc_attention_tcgen05_one_tile(qkv, batch, n_head, d_model, out, st, trace_dev);
}

void enc_attention_tcgen05_one_tile(const void* qkv, int batch, int n_head, int d_model, void* out, cudaStream_t st,
                                    long long* trace_dev) {
    CUtensorMap tm;
    std::string err;
    WLK_CHECK(make_tmap_bf16_2d(&tm, qkv, (uint64_t)batch * N_CTX, (uint64_t)3 * d_model, (uint64_t)3 * d_model, BQ, DH, &err),
              "qkv tensor map: %s", err.c_str());
    static bool seen[64] = {};
    if (first_on_device(seen))
        CUDA_CHECK(cudaFuncSetAttribute(attn_tc_kernel<MODE_ENC, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)AttLayout<false>::SMEM));
    dim3 grid((N_CTX + BQ - 1) / BQ, n_head, batch);
    attn_tc_kernel<MODE_ENC, false><<<grid, ATT_THREADS, AttLayout<false>::SMEM, st>>>(tm, tm, nullptr, nullptr, 0, nullptr, n_head, d_model, N_CTX, out, trace_dev);
    CUDA_CHECK(cudaGetLastError());
}

// WLK_PREC_BF16X3: qkv arrives as two bf16 planes [batch*1500, 3d] (hi, lo) -- the split of the fp32 QKV GEMM output --
// and the result is fp32 [batch*1500, d].
void enc_attention_tcgen05_x3(const void* qkv_hi, const void* qkv_lo, int batch, int n_head, int d_model, float* out, cudaStream_t st) {
    CUtensorMap tm, tml;
    std::string err;
    WLK_CHECK(make_tmap_bf16_2d(&tm, qkv_hi, (uint64_t)batch * N_CTX, (uint64_t)3 * d_model, (uint64_t)3 * d_model, BQ, DH, &err),
              "qkv tensor map: %s", err.c_str());
    WLK_CHECK(make_tmap_bf16_2d(&tml, qkv_lo, (uint64_t)batch * N_CTX, (uint64_t)3 * d_model, (uint64_t)3 * d_model, BQ, DH, &err),
              "qkv lo tensor map: %s", err.c_str());
    static bool seen[64] = {};
    if (first_on_device(seen))
        CUDA_CHECK(cudaFuncSetAttribute(attn_tc_kernel<MODE_ENC, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)AttLayout<true>::SMEM));
    dim3 grid((N_CTX + BQ - 1) / BQ, n_head, batch);
    attn_tc_kernel<MODE_ENC, true><<<grid, ATT_THREADS, AttLayout<true>::SMEM, st>>>(tm, tml, nullptr, nullptr, 0, nullptr, n_head, d_model, N_CTX, out);
    CUDA_CHECK(cudaGetLastError());
}

// tensor map over one session's cross-K/V planes viewed as [L * 2 * H * 1500 rows, 64] bf16
void make_cross_kv_tmap(void* tmap_out_host, const void* cross_kv, int n_layer, int n_head) {
    std::string err;
    WLK_CHECK(make_tmap_bf16_2d(reinterpret_cast<CUtensorMap*>(tmap_out_host), cross_kv,
                                (uint64_t)n_layer * 2 * n_head * N_CTX, DH, DH, BKV, DH, &err),
              "cross-K/V tensor map: %s", err.c_str());
}

void dec_cross_attention_tcgen05(const void* q, int total_rows, const DecJob* jobs, int n_jobs, int max_rows, int layer,
                                 int n_head, int d_model, const void* kv_maps_dev, const int32_t* align_rank, void* out,
                                 cudaStream_t st) {
    CUtensorMap tm;
    std::string err;
    WLK_CHECK(make_tmap_bf16_2d(&tm, q, (uint64_t)total_rows, (uint64_t)d_model, (uint64_t)d_model, BQ, DH, &err),
              "query tensor map: %s", err.c_str());
    static bool seen[64] = {};
    if (first_on_device(seen))
        CUDA_CHECK(cudaFuncSetAttribute(attn_tc_kernel<MODE_CROSS, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)AttLayout<false>::SMEM));
    dim3 grid((max_rows + BQ - 1) / BQ, n_head, n_jobs);
    CUDA_CHECK(launch_pdl(attn_tc_kernel<MODE_CROSS, false>, grid, dim3(ATT_THREADS), (size_t)AttLayout<false>::SMEM, st, tm, tm,
                          reinterpret_cast<const CUtensorMap*>(kv_maps_dev), jobs, layer, align_rank, n_head, d_model, N_CTX, out,
                          (long long*)nullptr));
}

// tensor map over one session's self-K/V cache viewed as [L * 2 * H * n_text_ctx rows, 64] bf16
void make_self_kv_tmap(void* tmap_out_host, const void* self_kv, int n_layer, int n_head, int n_text_ctx) {
    std::string err;
    WLK_CHECK(make_tmap_bf16_2d(reinterpret_cast<CUtensorMap*>(tmap_out_host), self_kv,
                                (uint64_t)n_layer * 2 * n_head * n_text_ctx, DH, DH, BKV, DH, &err),
              "self-K/V tensor map: %s", err.c_str());
}

// causal self-attention of a decoder prefill on the tensor cores (bf16): every head, rows [0, n_rows) of each job at
// positions job.offset + row; the cache rows of this call were written by the QKV GEMM's scatter epilogue just before
void dec_self_attention_tcgen05(const void* q, int total_rows, const DecJob* jobs, int n_jobs, int max_rows, int layer,
                                int n_head, int d_model, int n_text_ctx, const void* kv_maps_dev, void* out, cudaStream_t st) {
    CUtensorMap tm;
    std::string err;
    WLK_CHECK(make_tmap_bf16_2d(&tm, q, (uint64_t)total_rows, (uint64_t)d_model, (uint64_t)d_model, BQ, DH, &err),
              "query tensor map: %s", err.c_str());
    static bool seen[64] = {};
    if (first_on_device(seen))
        CUDA_CHECK(cudaFuncSetAttribute(attn_tc_kernel<MODE_SELF, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)AttLayout<false>::SMEM));
    dim3 grid((max_rows + BQ - 1) / BQ, n_head, n_jobs);
    CUDA_CHECK(launch_pdl(attn_tc_kernel<MODE_SELF, false>, grid, dim3(ATT_THREADS), (size_t)AttLayout<false>::SMEM, st, tm, tm,
                          reinterpret_cast<const CUtensorMap*>(kv_maps_dev), jobs, layer, (const int32_t*)nullptr, n_head, d_model,
                          n_text_ctx, out, (long long*)nullptr));
}

}  // namespace wlk
