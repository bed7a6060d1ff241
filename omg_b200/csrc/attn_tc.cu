// Flash attention on tcgen05 for the SDXL transformer blocks (head_dim 64): self-attention (N = 1024 / 4096 keys)
// and cross-attention (77 text keys, 16 IP-adapter keys), never materialising the probability matrix.
//
// Prompt-to-prompt control and decoupled (IP-adapter) attention are expressed through the descriptor instead of
// through a probability callback (reference: src/pipelines/lora_pipeline.py:114-116 + src/prompt_attention/
// p2p_attention.py:124-138, src/ip_adapter/attention_processor.py:370-409):
//   * every output batch row names the batch rows its Q, K and V come from  -> "replace self-attention"
//     out_1 = softmax(Q_0 K_0^T) V_1 is a pointer remap;
//   * `accumulate` + `out_weight` add a second separately-normalised term    -> txt + scale * ip, and the general
//     cross-attention edit  P_0 (M diag(a) V_1) + P_1 (diag(1-a) V_1).
//
// CTA = one (item, head, 128-query tile), two CTAs per SM (template G = 1; G = 2 puts two tiles into one CTA): 256
// threads = warp 0 TMA, warp 1 tcgen05.mma issuer (setmaxnreg gives their registers away), warps 4-7 softmax (one
// query row per thread: TMEM lane == row, so no shuffles are needed).  While one CTA's softmax runs the tensor core
// works for the co-resident CTA, and within a CTA S is double-buffered (S(j+2) and P.V(j) run during softmax(j+1)).
// KV blocks are 64 keys; TMEM per tile: S_g[2] (2 x 64 columns of fp32 scores, double-buffered), O_g (64 columns, the
// running P.V accumulator) and P_g[2] (2 x 32 columns: the probabilities as fp16 pairs).  P never touches shared
// memory: P.V is a TS-MMA with the A operand in TMEM (the SS form moved 32 KB more shared-memory traffic per tile and
// KV block and was shared-memory-bandwidth bound: 529 -> 597 TFLOP/s at N = 4096).
// Softmax follows the lazy-rescale scheme: O stays in TMEM and is accumulated by the tensor core across KV blocks;
// the running maximum is allowed to go stale by up to 2^8 and O is only rescaled (TMEM load-scale-store) when a row
// maximum grows beyond that, which after the first blocks is rare.  The arithmetic is packed fp32x2 (FFMA2 / FADD2);
// exp2 runs on the MUFU for 14 of 16 element pairs and as a degree-3 polynomial on the FMA pipe for the other 2
// (MUFU only: 529 TFLOP/s; ncu in profiles/r01_ncu_full_summary.csv).
#include <cuda_fp16.h>

#include <algorithm>
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include "../../include/omg_b200.h"
#include "host_common.h"
#include "ptx.cuh"

// which of the 16 element pairs of a 32-column chunk take the polynomial exp2 (FMA pipe) instead of the MUFU:
// balances issue slots (5 per polynomial value) against the MUFU's 16 lanes / clk / SM.  Round 1 (one CTA per tile) settled
// on 5 of 16; with the persistent kernel a same-box sweep (profiles/r02_attn_variants.jsonl) has 2 of 16 ahead on all four
// SDXL shapes (+2..4 %; all-MUFU is best at B = 4 and worst at B = 8, where the longer launch runs into the power cap)
#ifndef OMG_ATT_POLY_MASK
#define OMG_ATT_POLY_MASK 0x0101
#endif

namespace omg {

constexpr int ATT_BQ = 128;       // rows per softmax group (= one Q tile)
constexpr int ATT_BKV = 64;       // keys per block
constexpr int ATT_D = 64;
constexpr int ATT_Q_BYTES = ATT_BQ * ATT_D * 2;    // 16 KB
constexpr int ATT_K_BYTES = ATT_BKV * ATT_D * 2;   // 8 KB (K) ; V same

// G = Q tiles per CTA.  G = 1 (256 TMEM columns, 66-98 KB smem, two CTAs per SM) is what runs: the co-resident CTA
// hides the prologue / epilogue latencies.  G = 2 (one CTA per SM, the two tiles share every K/V load) is kept for
// measurements (OMG_ATTN_TILES=2); since P moved to TMEM the shared K/V load no longer pays for the lock-step.
template <int G, int KV_STAGES_>
struct AttCfg {
    static constexpr int THREADS = 128 + 128 * G;  // warpgroup 0: TMA + MMA issuer warps, then one softmax warpgroup per tile
    static constexpr int KV_STAGES = KV_STAGES_;
    static constexpr int SMEM = 1024 + G * ATT_Q_BYTES + KV_STAGES * 2 * ATT_K_BYTES + 512;
    static constexpr int TMEM_COLS = G == 2 ? 512 : 256;
    static constexpr int O_COL0 = G * 2 * 64;      // S_g[b] at (g*2+b)*64, O_g at O_COL0 + g*64
    static constexpr int P_COL0 = O_COL0 + G * 64;  // P_g[b] (fp16 pairs, 32 columns) at P_COL0 + (g*2+b)*32
    static constexpr int SOFTMAX_REGS = G == 2 ? 224 : 200;
};

struct alignas(64) AttnParams {
    CUtensorMap q_map, k_map, v_map;  // 3D (cols, tokens, batch), box (64, 128 | 64, 1), SWIZZLE_128B
    __half* out;
    int out_ld;
    long long out_bs;
    int n_q, n_kv, heads;
    int q_col0, k_col0, v_col0, out_col0;
    int n_items;
    int out_b[OMG_ATTN_MAX_ITEMS], q_b[OMG_ATTN_MAX_ITEMS], k_b[OMG_ATTN_MAX_ITEMS], v_b[OMG_ATTN_MAX_ITEMS];
    float scale_log2;  // softmax scale * log2(e)
    float out_weight;
    int accumulate;
    int causal;  // cross kernel only: key index > query index is masked
#ifdef OMG_ATT_TRACE
    long long* trace;  // [cta < 2][role 2][block 512][8] clock stamps (diagnostic build only)
#endif
};

// Pipeline (per 128-row tile g, KV block j, buffer b = j & 1):
//   MMA:      S_g[b] = Q_g K_j^T  (issued two blocks ahead)   ->  s_full[g][b]
//   softmax:  read S_g[b], (rare) rescale O_g, P = exp2(S*scale - m), P_g[b] -> TMEM (fp16 pairs)  ->  p_full[g][b]
//   MMA:      S_g[b] = Q_g K_{j+2}^T ; O_g += P_g[b] V_j  ->  p_empty[g][b]
// S and P are double-buffered, so the softmax warps never wait for the tensor core in steady state and vice versa.
template <int G, int KVS>
__global__ void __launch_bounds__(AttCfg<G, KVS>::THREADS, G == 1 ? 2 : 1) attn_tc_kernel(const __grid_constant__ AttnParams p) {
    using Cfg = AttCfg<G, KVS>;
    constexpr int ATT_KV_STAGES = KVS;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* q_smem = smem;                                          // G x 16 KB
    uint8_t* kv_smem = q_smem + G * ATT_Q_BYTES;                     // stages x (K 8 KB | V 8 KB)
    uint64_t* bars = reinterpret_cast<uint64_t*>(kv_smem + ATT_KV_STAGES * 2 * ATT_K_BYTES);
    uint64_t* q_full = bars;                        // 1
    uint64_t* kv_full = bars + 1;                   // STAGES
    uint64_t* kv_empty = kv_full + ATT_KV_STAGES;   // STAGES
    uint64_t* s_full = kv_empty + ATT_KV_STAGES;    // [g*2 + b]
    uint64_t* p_full = s_full + 4;                  // [g*2 + b]
    uint64_t* p_empty = p_full + 4;                 // [g*2 + b]: P.V of the block that used buffer b has completed
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(p_empty + 4);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int slab = blockIdx.x;  // slab of G * 128 queries
    const int head = blockIdx.y;
    const int item = blockIdx.z;
    const int nkv = (p.n_kv + ATT_BKV - 1) / ATT_BKV;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&p.q_map);
        tma_prefetch_desc(&p.k_map);
        tma_prefetch_desc(&p.v_map);
        mbar_init(q_full, 1);
        for (int i = 0; i < ATT_KV_STAGES; ++i) {
            mbar_init(&kv_full[i], 1);
            mbar_init(&kv_empty[i], G);  // one commit per tile's MMA issuer
        }
        for (int i = 0; i < 2 * G; ++i) {
            mbar_init(&s_full[i], 1);
            mbar_init(&p_full[i], 4);
            mbar_init(&p_empty[i], 1);
        }
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc(tmem_slot, Cfg::TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    griddep_launch_dependents();
    griddep_wait();
    // TMEM columns: S_g[b] at (g*2 + b)*64, O_g at O_COL0 + g*64
    if (warp < 4) {
      asm volatile("setmaxnreg.dec.sync.aligned.u32 56;");
      if (warp == 0) {
        // ------------------------------------------------------------------ TMA producer
        if (lane == 0) {
            mbar_arrive_expect_tx(q_full, G * ATT_Q_BYTES);
            const int qb = p.q_b[item];
            for (int g = 0; g < G; ++g)
                tma_load_3d(q_smem + g * ATT_Q_BYTES, &p.q_map, q_full, p.q_col0 + head * ATT_D,
                            slab * (G * ATT_BQ) + g * ATT_BQ, qb);
            int stage = 0;
            uint32_t phase = 0;
            const int kb = p.k_b[item], vb = p.v_b[item];
            for (int j = 0; j < nkv; ++j) {
                mbar_wait(&kv_empty[stage], phase ^ 1);
                uint8_t* kd = kv_smem + stage * 2 * ATT_K_BYTES;
                mbar_arrive_expect_tx(&kv_full[stage], 2 * ATT_K_BYTES);
                tma_load_3d(kd, &p.k_map, &kv_full[stage], p.k_col0 + head * ATT_D, j * ATT_BKV, kb);
                tma_load_3d(kd + ATT_K_BYTES, &p.v_map, &kv_full[stage], p.v_col0 + head * ATT_D, j * ATT_BKV, vb);
                if (++stage == ATT_KV_STAGES) {
                    stage = 0;
                    phase ^= 1;
                }
            }
        }
      } else if (warp >= 1 && warp <= G) {
        // ------------------------------------------------------------------ MMA issuers: warp 1 -> tile 0, warp 2 -> tile 1
        // (a single issuing thread would serialise both tiles' barrier round-trips; the tensor work per event is
        // only 256 cycles)
        if (lane == 0) {
            const int g = warp - 1;
            constexpr uint32_t idesc_s = umma_idesc_f16(128, ATT_BKV, false, false);  // S = Q K^T
            constexpr uint32_t idesc_o = umma_idesc_f16(128, ATT_D, false, true);     // O += P V (V is N-major)
            const uint64_t q_desc = umma_desc_sw128(smem_u32(q_smem + g * ATT_Q_BYTES), 1024, 16);
            const uint64_t k_desc0 = umma_desc_sw128(smem_u32(kv_smem), 1024, 16);
            const uint64_t v_desc0 = umma_desc_sw128(smem_u32(kv_smem + ATT_K_BYTES), 1024, 1024);
            const uint32_t p_tmem_g = tmem_base + Cfg::P_COL0 + g * 64;
            const uint32_t o_tmem_g = tmem_base + Cfg::O_COL0 + g * 64;
            auto issue_s = [&](int jb) {  // scores of block jb into S_g[jb & 1]
                const uint64_t kd = k_desc0 + (uint64_t)((jb % ATT_KV_STAGES) * ((2 * ATT_K_BYTES) >> 4));
#pragma unroll
                for (int k = 0; k < ATT_D / 16; ++k)
                    tc_mma_f16_ss(tmem_base + (g * 2 + (jb & 1)) * 64, q_desc + 2 * k, kd + 2 * k, idesc_s, k > 0);
                tc_commit(&s_full[g * 2 + (jb & 1)]);
            };
            auto wait_kv = [&](int jb) { mbar_wait(&kv_full[jb % ATT_KV_STAGES], (jb / ATT_KV_STAGES) & 1); };
            mbar_wait(q_full, 0);
            for (int jb = 0; jb < 2 && jb < nkv; ++jb) {
                wait_kv(jb);
                tc_fence_after();
                issue_s(jb);
            }
            for (int j = 0; j < nkv; ++j) {
                const int b = j & 1;
                const int st = j % ATT_KV_STAGES;
                mbar_wait(&p_full[g * 2 + b], (j >> 1) & 1);  // P_g[b] is in TMEM and S_g[b] has been read out
                tc_fence_after();
                if (j + 2 < nkv) {  // refill the score buffer that was just released
                    wait_kv(j + 2);
                    tc_fence_after();
                    issue_s(j + 2);
                }
                const uint64_t vd = v_desc0 + (uint64_t)(st * ((2 * ATT_K_BYTES) >> 4));
#pragma unroll
                for (int k = 0; k < ATT_BKV / 16; ++k) {
                    // A = P from TMEM (16 keys = 8 packed columns per K step; P never touches shared memory);
                    // B = V: 16 key rows (2 KB) per K step, N-major
                    tc_mma_f16_ts(o_tmem_g, p_tmem_g + b * 32 + 8 * k, vd + 128 * k, idesc_o, (j > 0 || k > 0) ? 1u : 0u);
                }
                tc_commit(&p_empty[g * 2 + b]);
                tc_commit(&kv_empty[st]);
            }
        }
      }
    } else {
        // ------------------------------------------------------------------ softmax groups
        if constexpr (G == 2) asm volatile("setmaxnreg.inc.sync.aligned.u32 224;");
        else asm volatile("setmaxnreg.inc.sync.aligned.u32 200;");
        const int g = (warp - 4) >> 2;
        const int q = warp & 3;
        const int row = q * 32 + lane;
        const uint32_t lane_base = (uint32_t)(q * 32) << 16;
        const uint32_t s_tmem = tmem_base + g * 128 + lane_base;
        const uint32_t o_tmem = tmem_base + Cfg::O_COL0 + g * 64 + lane_base;
        const uint32_t p_tmem = tmem_base + Cfg::P_COL0 + g * 64 + lane_base;
        float m = -INFINITY, l = 0.f;
        constexpr float kRescaleThreshold = 8.0f;  // log2 domain: P may reach 2^8 before O is rescaled

        for (int j = 0; j < nkv; ++j) {
            const int b = j & 1;
            mbar_wait(&s_full[g * 2 + b], (j >> 1) & 1);
            tc_fence_after();
            const int kv_left = p.n_kv - j * ATT_BKV;  // valid keys in this block (>= 1)
            uint32_t sr[2][32];
            tmem_ld_32x32(s_tmem + b * 64, sr[0]);
            tmem_ld_32x32(s_tmem + b * 64 + 32, sr[1]);
            tc_wait_ld();
            if (kv_left < ATT_BKV) {  // partial last block: keys beyond n_kv (zero-filled K rows) are excluded
#pragma unroll
                for (int c = 0; c < 2; ++c)
#pragma unroll
                    for (int i = 0; i < 32; ++i)
                        if (c * 32 + i >= kv_left) sr[c][i] = __float_as_uint(-INFINITY);
            }
            float mx = -INFINITY;
#pragma unroll
            for (int c = 0; c < 2; ++c)
#pragma unroll
                for (int i = 0; i < 32; i += 2) mx = fmax3(mx, __uint_as_float(sr[c][i]), __uint_as_float(sr[c][i + 1]));
            const float m_cand = fmaxf(m, mx * p.scale_log2);
            if (j == 0) {
                m = m_cand;
            } else {
                const bool need = (m_cand - m) > kRescaleThreshold;
                if (__any_sync(0xffffffffu, need)) {
                    // O_g holds blocks < j relative to the stale maximum: rescale it once P.V(j-1) has landed.
                    // (p_empty of the OTHER buffer: this is next block's regular wait done early, so no mbarrier
                    // phase is skipped - a waiter may never fall two phases behind a parity barrier.)
                    mbar_wait(&p_empty[g * 2 + (b ^ 1)], ((j - 1) >> 1) & 1);
                    tc_fence_after();
                    const float corr = need ? fast_exp2(m - m_cand) : 1.0f;
                    if (need) m = m_cand;
                    l *= corr;
#pragma unroll
                    for (int c = 0; c < 2; ++c) {
                        uint32_t r[32];
                        tmem_ld_32x32(o_tmem + c * 32, r);
                        tc_wait_ld();
#pragma unroll
                        for (int i = 0; i < 32; ++i) r[i] = __float_as_uint(__uint_as_float(r[i]) * corr);
                        tmem_st_32x32(o_tmem + c * 32, r);
                    }
                    tc_wait_st();
                }
            }
            // P_g[b] must have been consumed by P.V(j-2)
            mbar_wait(&p_empty[g * 2 + b], ((j >> 1) & 1) ^ 1);
            uint64_t sum2 = pack_f32x2(0.f, 0.f);
            const uint64_t scale2 = pack_f32x2(p.scale_log2, p.scale_log2);
            const uint64_t negm2 = pack_f32x2(-m, -m);
            uint32_t pk[32];  // this row's 64 probabilities as fp16 pairs = the A operand of P.V, kept in TMEM
#pragma unroll
            for (int c = 0; c < 2; ++c) {
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    // packed fp32x2 arithmetic: one issue slot per two elements for the scale/shift and the row sum
                    const uint64_t x2 = ffma2(pack_f32x2(__uint_as_float(sr[c][2 * i]), __uint_as_float(sr[c][2 * i + 1])),
                                              scale2, negm2);
                    float x0, x1, p0, p1;
                    unpack_f32x2(x2, x0, x1);
                    if ((OMG_ATT_POLY_MASK >> i) & 1) {  // this pair on the FMA pipe, the others on the MUFU
                        poly_exp2_x2(x0, x1, p0, p1);
                    } else {
                        p0 = fast_exp2(x0);
                        p1 = fast_exp2(x1);
                    }
                    sum2 = fadd2(sum2, pack_f32x2(p0, p1));
                    pk[c * 16 + i] = pack_half2(p0, p1);
                }
            }
            tmem_st_32x32(p_tmem + b * 32, pk);
            float sum, sum_hi;
            unpack_f32x2(sum2, sum, sum_hi);
            sum += sum_hi;
            l += sum;
            tc_wait_st();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&p_full[g * 2 + b]);
        }
        // all P.V of this tile have landed: the last user of each P buffer
        if (nkv >= 2) mbar_wait(&p_empty[g * 2 + ((nkv - 2) & 1)], ((nkv - 2) >> 1) & 1);
        mbar_wait(&p_empty[g * 2 + ((nkv - 1) & 1)], ((nkv - 1) >> 1) & 1);
        tc_fence_after();
        float o_acc[ATT_D];
#pragma unroll
        for (int c = 0; c < 2; ++c) {
            uint32_t r[32];
            tmem_ld_32x32(o_tmem + c * 32, r);
            tc_wait_ld();
#pragma unroll
            for (int i = 0; i < 32; ++i) o_acc[c * 32 + i] = __uint_as_float(r[i]);
        }

        // finalise: out = (accumulate ? out : 0) + w * O / l
        const int qrow = slab * (G * ATT_BQ) + g * ATT_BQ + row;
        if (qrow < p.n_q) {
            const float inv = p.out_weight / l;
            __half* op = p.out + (long long)p.out_b[item] * p.out_bs + (long long)qrow * p.out_ld + p.out_col0 +
                         head * ATT_D;
            uint4* op4 = reinterpret_cast<uint4*>(op);
#pragma unroll
            for (int t = 0; t < 8; ++t) {
                float v[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) v[i] = o_acc[t * 8 + i] * inv;
                if (p.accumulate) {
                    const uint4 u = op4[t];
                    const __half2* h2 = reinterpret_cast<const __half2*>(&u);
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const float2 f = __half22float2(h2[i]);
                        v[2 * i] += f.x;
                        v[2 * i + 1] += f.y;
                    }
                }
                op4[t] = make_uint4(pack_half2(v[0], v[1]), pack_half2(v[2], v[3]), pack_half2(v[4], v[5]),
                                    pack_half2(v[6], v[7]));
            }
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
}


// ---------------------------------------------------------------------------------------------------------------------
// Persistent form of the single-stream kernel.  A CTA of the per-tile kernel costs ~6 us of setup and drain (CTA launch,
// barrier init, TMEM allocation, first Q/K/V round trip, pipeline ramp, epilogue, dealloc) - a third of an N = 1024
// tile (16 KV blocks x ~0.75 us) - measured as the intercept of round time over KV blocks between N = 4096 and N = 1024.
// Here 2 x #SM CTAs each walk tiles  t = blockIdx.x, blockIdx.x + gridDim.x, ...  as ONE stream of KV blocks: barriers
// and TMEM live for the whole kernel, the TMA warp runs ahead into the next tile (Q is double-buffered), the MMA issuer
// starts the next tile's Q.K^T while the softmax group is still in the current tile's epilogue, and only the first
// P.V of a tile waits for the softmax group to have read the previous tile's O out of tensor memory (o_free).
// Barrier phases are tracked with running counters, so tiles with odd block counts need no special case.
template <int KVS_, int QB_>
struct AttPCfg {
    static constexpr int THREADS = 256;
    static constexpr int KV_STAGES = KVS_;
    static constexpr int Q_BUFS = QB_;
    // no alignment slack: two CTAs per SM leave 115 712 B each; the dynamic window is 1024 B aligned in practice (checked)
    static constexpr int SMEM = Q_BUFS * ATT_Q_BYTES + KV_STAGES * 2 * ATT_K_BYTES + 512;
    static constexpr int TMEM_COLS = 256;
    static constexpr int O_COL0 = 128, P_COL0 = 192;
};

template <int KVS_, int QB>
__global__ void __launch_bounds__(256, 2) attn_p_kernel(const __grid_constant__ AttnParams p, int n_tiles, int n_slabs) {
    using Cfg = AttPCfg<KVS_, QB>;
    constexpr int KVS = Cfg::KV_STAGES;
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = smem_raw;
    if ((smem_u32(smem) & 1023u) != 0) __trap();  // the swizzled tiles need 1024 B alignment
    uint8_t* q_smem = smem;                                   // 2 x 16 KB
    uint8_t* kv_smem = q_smem + QB * ATT_Q_BYTES;
    uint64_t* bars = reinterpret_cast<uint64_t*>(kv_smem + KVS * 2 * ATT_K_BYTES);
    uint64_t* q_full = bars;                 // [2]
    uint64_t* q_empty = bars + 2;            // [2] every Q.K^T of the tile that used the buffer has completed
    uint64_t* kv_full = bars + 4;            // [KVS]
    uint64_t* kv_empty = kv_full + KVS;      // [KVS]
    uint64_t* s_full = kv_empty + KVS;       // [2]
    uint64_t* p_full = s_full + 2;           // [2]
    uint64_t* p_empty = p_full + 2;          // [2]
    uint64_t* o_free = p_empty + 2;          // the softmax group has read the finished tile's O out of TMEM
    uint64_t* o_done = o_free + 1;           // the last P.V of a tile has completed
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(o_done + 1);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int nkv = (p.n_kv + ATT_BKV - 1) / ATT_BKV;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&p.q_map);
        tma_prefetch_desc(&p.k_map);
        tma_prefetch_desc(&p.v_map);
        for (int i = 0; i < 2; ++i) {
            mbar_init(&q_full[i], 1);
            mbar_init(&q_empty[i], 1);
            mbar_init(&s_full[i], 1);
            mbar_init(&p_full[i], 4);
            mbar_init(&p_empty[i], 1);
        }
        for (int i = 0; i < KVS; ++i) {
            mbar_init(&kv_full[i], 1);
            mbar_init(&kv_empty[i], 1);
        }
        mbar_init(o_free, 4);
        mbar_init(o_done, 1);
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc(tmem_slot, Cfg::TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    griddep_launch_dependents();
    griddep_wait();
    if (warp < 4) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 56;");
        if (warp == 0) {
            if (lane == 0) {  // ------------------------------------------------------------ TMA producer
                uint32_t gj = 0;  // running KV-block counter of this CTA
                int ti = 0;       // running tile counter
                for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++ti) {
                    const int slab = tile % n_slabs, head = (tile / n_slabs) % p.heads, item = tile / (n_slabs * p.heads);
                    const int qb = ti % QB;
                    mbar_wait(&q_empty[qb], ((ti / QB) & 1) ^ 1);
                    mbar_arrive_expect_tx(&q_full[qb], ATT_Q_BYTES);
                    tma_load_3d(q_smem + qb * ATT_Q_BYTES, &p.q_map, &q_full[qb], p.q_col0 + head * ATT_D, slab * ATT_BQ, p.q_b[item]);
                    const int kb = p.k_b[item], vb = p.v_b[item];
                    for (int j = 0; j < nkv; ++j, ++gj) {
                        const int stage = gj % KVS;  // KVS is a compile-time constant
                        mbar_wait(&kv_empty[stage], ((gj / KVS) & 1) ^ 1);
                        uint8_t* kd = kv_smem + stage * 2 * ATT_K_BYTES;
                        mbar_arrive_expect_tx(&kv_full[stage], 2 * ATT_K_BYTES);
                        tma_load_3d(kd, &p.k_map, &kv_full[stage], p.k_col0 + head * ATT_D, j * ATT_BKV, kb);
                        tma_load_3d(kd + ATT_K_BYTES, &p.v_map, &kv_full[stage], p.v_col0 + head * ATT_D, j * ATT_BKV, vb);
                    }
                }
            }
        } else if (warp == 1) {
            if (lane == 0) {  // ------------------------------------------------------------ MMA issuer
                constexpr uint32_t idesc_s = umma_idesc_f16(128, ATT_BKV, false, false);
                constexpr uint32_t idesc_o = umma_idesc_f16(128, ATT_D, false, true);
                const uint64_t k_desc0 = umma_desc_sw128(smem_u32(kv_smem), 1024, 16);
                const uint64_t v_desc0 = umma_desc_sw128(smem_u32(kv_smem + ATT_K_BYTES), 1024, 1024);
                // every tile contributes nkv blocks to ONE running sequence g = ti * nkv + j; S / P buffers alternate with g
                int n_my = 0;
                for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) ++n_my;
                const uint32_t total = (uint32_t)n_my * (uint32_t)nkv;
                uint32_t sg = 0;       // running block the next Q.K^T belongs to, and its (tile, block) coordinates
                int s_ti = 0, s_j = 0;
                auto issue_s = [&]() {  // scores of running block sg into S[sg & 1]
                    const int qb = s_ti % QB;
                    if (s_j == 0) {
                        mbar_wait(&q_full[qb], (s_ti / QB) & 1);
                        tc_fence_after();
                    }
                    const uint32_t st = sg % KVS;
                    mbar_wait(&kv_full[st], (sg / KVS) & 1);
                    tc_fence_after();
                    const uint64_t q_desc = umma_desc_sw128(smem_u32(q_smem + qb * ATT_Q_BYTES), 1024, 16);
                    const uint64_t kd = k_desc0 + (uint64_t)(st * ((2 * ATT_K_BYTES) >> 4));
#pragma unroll
                    for (int k = 0; k < ATT_D / 16; ++k)
                        tc_mma_f16_ss(tmem_base + (sg & 1) * 64, q_desc + 2 * k, kd + 2 * k, idesc_s, k > 0);
                    tc_commit(&s_full[sg & 1]);
                    if (s_j == nkv - 1) tc_commit(&q_empty[qb]);  // last Q.K^T of the tile: its Q buffer may be refilled
                    ++sg;
                    if (++s_j == nkv) {
                        s_j = 0;
                        ++s_ti;
                    }
                };
                for (uint32_t g = 0; g < 2 && g < total; ++g) issue_s();
                int ti = 0, j = 0;
                for (uint32_t g = 0; g < total; ++g) {
                    const int b = g & 1;
#ifdef OMG_ATT_TRACE
                    const bool tr = p.trace && (blockIdx.x == 0 || blockIdx.x == 148) && g < 512;
                    long long* tp = tr ? p.trace + (((blockIdx.x ? 1 : 0) * 2 + 1) * 512 + g) * 8 : nullptr;
                    if (tr) tp[0] = clock64();
#endif
                    mbar_wait(&p_full[b], (g >> 1) & 1);
                    tc_fence_after();
#ifdef OMG_ATT_TRACE
                    if (tr) tp[1] = clock64();
#endif
                    if (sg < total) issue_s();
#ifdef OMG_ATT_TRACE
                    if (tr) tp[2] = clock64();
#endif
                    if (j == 0 && ti > 0) {  // O still holds the previous tile until the softmax group has read it
                        mbar_wait(o_free, (ti - 1) & 1);
                        tc_fence_after();
                    }
                    const uint64_t vd = v_desc0 + (uint64_t)((g % KVS) * ((2 * ATT_K_BYTES) >> 4));
#pragma unroll
                    for (int k = 0; k < ATT_BKV / 16; ++k)
                        tc_mma_f16_ts(tmem_base + Cfg::O_COL0, tmem_base + Cfg::P_COL0 + b * 32 + 8 * k, vd + 128 * k, idesc_o,
                                      (j > 0 || k > 0) ? 1u : 0u);
                    tc_commit(&p_empty[b]);
                    tc_commit(&kv_empty[g % KVS]);
                    if (j == nkv - 1) tc_commit(o_done);
#ifdef OMG_ATT_TRACE
                    if (tr) tp[3] = clock64();
#endif
                    if (++j == nkv) {
                        j = 0;
                        ++ti;
                    }
                }
            }
        }
    } else {
        // ---------------------------------------------------------------------------------- softmax group
        asm volatile("setmaxnreg.inc.sync.aligned.u32 200;");
        const int q = warp & 3;
        const int row = q * 32 + lane;
        const uint32_t lane_base = (uint32_t)(q * 32) << 16;
        const uint32_t s_tmem = tmem_base + lane_base;
        const uint32_t o_tmem = tmem_base + Cfg::O_COL0 + lane_base;
        const uint32_t p_tmem = tmem_base + Cfg::P_COL0 + lane_base;
        constexpr float kRescaleThreshold = 8.0f;
        const uint64_t scale2 = pack_f32x2(p.scale_log2, p.scale_log2);
        uint32_t g = 0;
        int ti = 0;
        for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++ti) {
            const int slab = tile % n_slabs, head = (tile / n_slabs) % p.heads, item = tile / (n_slabs * p.heads);
            float m = -INFINITY, l = 0.f;
            for (int j = 0; j < nkv; ++j, ++g) {
                const int b = g & 1;
#ifdef OMG_ATT_TRACE
                const bool tr = p.trace && warp == 4 && lane == 0 && (blockIdx.x == 0 || blockIdx.x == 148) && g < 512;
                long long* tp = tr ? p.trace + (((blockIdx.x ? 1 : 0) * 2 + 0) * 512 + g) * 8 : nullptr;
                if (tr) tp[0] = clock64();
#endif
                mbar_wait(&s_full[b], (g >> 1) & 1);
                tc_fence_after();
#ifdef OMG_ATT_TRACE
                if (tr) tp[1] = clock64();
#endif
                const int kv_left = p.n_kv - j * ATT_BKV;
                uint32_t sr[2][32];
                tmem_ld_32x32(s_tmem + b * 64, sr[0]);
                tmem_ld_32x32(s_tmem + b * 64 + 32, sr[1]);
                tc_wait_ld();
#ifdef OMG_ATT_TRACE
                if (tr) tp[2] = clock64() + (long long)(sr[0][0] & 0u);
#endif
                if (kv_left < ATT_BKV) {
#pragma unroll
                    for (int c = 0; c < 2; ++c)
#pragma unroll
                        for (int i = 0; i < 32; ++i)
                            if (c * 32 + i >= kv_left) sr[c][i] = __float_as_uint(-INFINITY);
                }
                float mx = -INFINITY;
#pragma unroll
                for (int c = 0; c < 2; ++c)
#pragma unroll
                    for (int i = 0; i < 32; i += 2) mx = fmax3(mx, __uint_as_float(sr[c][i]), __uint_as_float(sr[c][i + 1]));
                const float m_cand = fmaxf(m, mx * p.scale_log2);
                if (j == 0) {
                    m = m_cand;
                } else {
                    const bool need = (m_cand - m) > kRescaleThreshold;
                    if (__any_sync(0xffffffffu, need)) {
                        // P.V of the previous block (same tile: j >= 1) must have landed before O is rescaled
                        mbar_wait(&p_empty[b ^ 1], ((g - 1) >> 1) & 1);
                        tc_fence_after();
                        const float corr = need ? fast_exp2(m - m_cand) : 1.0f;
                        if (need) m = m_cand;
                        l *= corr;
#pragma unroll
                        for (int c = 0; c < 2; ++c) {
                            uint32_t r[32];
                            tmem_ld_32x32(o_tmem + c * 32, r);
                            tc_wait_ld();
#pragma unroll
                            for (int i = 0; i < 32; ++i) r[i] = __float_as_uint(__uint_as_float(r[i]) * corr);
                            tmem_st_32x32(o_tmem + c * 32, r);
                        }
                        tc_wait_st();
                    }
                }
#ifdef OMG_ATT_TRACE
                if (tr) tp[3] = clock64() + (long long)(__float_as_uint(m) & 0u);
#endif
                if (g >= 2) mbar_wait(&p_empty[b], ((g >> 1) & 1) ^ 1);  // P[b] consumed by the P.V of running block g - 2
#ifdef OMG_ATT_TRACE
                if (tr) tp[4] = clock64();
#endif
                uint64_t sum2 = pack_f32x2(0.f, 0.f);
                const uint64_t negm2 = pack_f32x2(-m, -m);
                uint32_t pk[32];
#pragma unroll
                for (int c = 0; c < 2; ++c) {
#pragma unroll
                    for (int i = 0; i < 16; ++i) {
                        const uint64_t x2 = ffma2(pack_f32x2(__uint_as_float(sr[c][2 * i]), __uint_as_float(sr[c][2 * i + 1])),
                                                  scale2, negm2);
                        float x0, x1, p0, p1;
                        unpack_f32x2(x2, x0, x1);
                        if ((OMG_ATT_POLY_MASK >> i) & 1) {
                            poly_exp2_x2(x0, x1, p0, p1);
                        } else {
                            p0 = fast_exp2(x0);
                            p1 = fast_exp2(x1);
                        }
                        sum2 = fadd2(sum2, pack_f32x2(p0, p1));
                        pk[c * 16 + i] = pack_half2(p0, p1);
                    }
                }
#ifdef OMG_ATT_TRACE
                if (tr) tp[5] = clock64() + (long long)(pk[31] & 0u);
#endif
                tmem_st_32x32(p_tmem + b * 32, pk);
                float sum, sum_hi;
                unpack_f32x2(sum2, sum, sum_hi);
                l += sum + sum_hi;
                tc_wait_st();
#ifdef OMG_ATT_TRACE
                if (tr) tp[6] = clock64();
#endif
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&p_full[b]);
#ifdef OMG_ATT_TRACE
                if (tr) tp[7] = clock64();
#endif
            }
            // tile epilogue: O is complete once the last P.V has landed; read it out and hand TMEM back at once
            mbar_wait(o_done, ti & 1);
            tc_fence_after();
            float o_acc[ATT_D];
#pragma unroll
            for (int c = 0; c < 2; ++c) {
                uint32_t r[32];
                tmem_ld_32x32(o_tmem + c * 32, r);
                tc_wait_ld();
#pragma unroll
                for (int i = 0; i < 32; ++i) o_acc[c * 32 + i] = __uint_as_float(r[i]);
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(o_free);
            const int qrow = slab * ATT_BQ + row;
            if (qrow < p.n_q) {
                const float inv = p.out_weight / l;
                __half* op = p.out + (long long)p.out_b[item] * p.out_bs + (long long)qrow * p.out_ld + p.out_col0 +
                             head * ATT_D;
                uint4* op4 = reinterpret_cast<uint4*>(op);
#pragma unroll
                for (int t = 0; t < 8; ++t) {
                    float v[8];
#pragma unroll
                    for (int i = 0; i < 8; ++i) v[i] = o_acc[t * 8 + i] * inv;
                    if (p.accumulate) {
                        const uint4 u = op4[t];
                        const __half2* h2 = reinterpret_cast<const __half2*>(&u);
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            const float2 f = __half22float2(h2[i]);
                            v[2 * i] += f.x;
                            v[2 * i + 1] += f.y;
                        }
                    }
                    op4[t] = make_uint4(pack_half2(v[0], v[1]), pack_half2(v[2], v[3]), pack_half2(v[4], v[5]),
                                        pack_half2(v[6], v[7]));
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
}

// ---------------------------------------------------------------------------------------------------------------------
// Cross-attention (77 text keys, 16 IP-adapter keys, <= 128 keys in general): the whole key sequence is ONE block, so a
// head needs one Q.K^T, one softmax and one P.V.  Launched as one CTA per (query tile, head) - 640 CTAs of ~3 us at
// N = 1024 - the old kernel spent most of its time in per-CTA setup (barrier init, TMEM allocation, pipeline fill):
// 22-35 us per launch for ~3 us of HBM traffic.  Here a CTA walks a GROUP of heads of its 128-query tile: Q_h / K_h / V_h
// of the next head are fetched by TMA while the current head is in its softmax, the TMEM allocation and the barriers
// live for the whole group, and the two co-resident CTAs of an SM fill each other's bubbles.
//   NK = padded key count (16 | 80 | 128): S is 128 x NK fp32 in TMEM, P (fp16 pairs) overwrites it in place,
//   O is 128 x 64.  256 TMEM columns per CTA, two CTAs per SM.
template <int NK>
struct AttXCfg {
    static constexpr int THREADS = 256;
    static constexpr int STAGES = 2;
    static constexpr int KV_BYTES = NK * ATT_D * 2;
    static constexpr int STAGE_BYTES = ATT_Q_BYTES + 2 * ((KV_BYTES + 1023) / 1024 * 1024);
    static constexpr int SMEM = 1024 + STAGES * STAGE_BYTES + 256;
    static constexpr int TMEM_COLS = 256;
    static constexpr int O_COL0 = 128;
};

template <int NK>
__global__ void __launch_bounds__(256, 2) attn_cross_kernel(const __grid_constant__ AttnParams p, int heads_per_cta) {
    using Cfg = AttXCfg<NK>;
    constexpr int KV_PAD = (Cfg::KV_BYTES + 1023) / 1024 * 1024;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Cfg::STAGES * Cfg::STAGE_BYTES);
    uint64_t* full = bars;                    // [stage] Q, K, V of a head have landed
    uint64_t* empty = bars + Cfg::STAGES;     // [stage] both MMAs of that head have completed
    uint64_t* s_full = empty + Cfg::STAGES;   // scores ready
    uint64_t* p_full = s_full + 1;            // probabilities written (and the previous head's O read out)
    uint64_t* o_full = p_full + 1;            // P.V complete
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(o_full + 1);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int slab = blockIdx.x, item = blockIdx.z;
    const int h0 = blockIdx.y * heads_per_cta;
    const int nh = min(heads_per_cta, p.heads - h0);

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&p.q_map);
        tma_prefetch_desc(&p.k_map);
        tma_prefetch_desc(&p.v_map);
        for (int i = 0; i < Cfg::STAGES; ++i) {
            mbar_init(&full[i], 1);
            mbar_init(&empty[i], 1);
        }
        mbar_init(s_full, 1);
        mbar_init(p_full, 4);
        mbar_init(o_full, 1);
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc(tmem_slot, Cfg::TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    griddep_launch_dependents();
    griddep_wait();
    if (warp < 4) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 56;");
        if (warp == 0) {
            if (lane == 0) {  // ------------------------------------------------------------ TMA producer
                const int qb = p.q_b[item], kb = p.k_b[item], vb = p.v_b[item];
                for (int i = 0; i < nh; ++i) {
                    const int st = i % Cfg::STAGES;
                    mbar_wait(&empty[st], ((i / Cfg::STAGES) & 1) ^ 1);
                    uint8_t* base = smem + st * Cfg::STAGE_BYTES;
                    const int col = (h0 + i) * ATT_D;
                    mbar_arrive_expect_tx(&full[st], ATT_Q_BYTES + 2 * Cfg::KV_BYTES);
                    tma_load_3d(base, &p.q_map, &full[st], p.q_col0 + col, slab * ATT_BQ, qb);
                    tma_load_3d(base + ATT_Q_BYTES, &p.k_map, &full[st], p.k_col0 + col, 0, kb);
                    tma_load_3d(base + ATT_Q_BYTES + KV_PAD, &p.v_map, &full[st], p.v_col0 + col, 0, vb);
                }
            }
        } else if (warp == 1) {
            if (lane == 0) {  // ------------------------------------------------------------ MMA issuer
                constexpr uint32_t idesc_s = umma_idesc_f16(128, NK, false, false);
                constexpr uint32_t idesc_o = umma_idesc_f16(128, ATT_D, false, true);
                for (int i = 0; i < nh; ++i) {
                    const int st = i % Cfg::STAGES;
                    const uint32_t base = smem_u32(smem + st * Cfg::STAGE_BYTES);
                    const uint64_t q_desc = umma_desc_sw128(base, 1024, 16);
                    const uint64_t k_desc = umma_desc_sw128(base + ATT_Q_BYTES, 1024, 16);
                    const uint64_t v_desc = umma_desc_sw128(base + ATT_Q_BYTES + KV_PAD, 1024, 1024);
                    mbar_wait(&full[st], (i / Cfg::STAGES) & 1);
                    tc_fence_after();
                    // behind the previous head's P.V in issue order, so its P (aliased on S) has been consumed
#pragma unroll
                    for (int k = 0; k < ATT_D / 16; ++k) tc_mma_f16_ss(tmem_base, q_desc + 2 * k, k_desc + 2 * k, idesc_s, k > 0);
                    tc_commit(s_full);
                    mbar_wait(p_full, i & 1);  // P_i in TMEM; the softmax group has also finished reading O_(i-1)
                    tc_fence_after();
#pragma unroll
                    for (int k = 0; k < NK / 16; ++k)
                        tc_mma_f16_ts(tmem_base + Cfg::O_COL0, tmem_base + 8 * k, v_desc + 128 * k, idesc_o, k > 0 ? 1u : 0u);
                    tc_commit(o_full);
                    tc_commit(&empty[st]);
                }
            }
        }
    } else {
        // ---------------------------------------------------------------------------------- softmax + epilogue
        asm volatile("setmaxnreg.inc.sync.aligned.u32 200;");
        const int q = warp & 3;
        const int row = q * 32 + lane;
        const uint32_t lane_base = (uint32_t)(q * 32) << 16;
        const uint32_t s_tmem = tmem_base + lane_base;
        const uint32_t o_tmem = tmem_base + Cfg::O_COL0 + lane_base;
        const int qrow = slab * ATT_BQ + row;
        const uint64_t scale2 = pack_f32x2(p.scale_log2, p.scale_log2);
        for (int i = 0; i < nh; ++i) {
            mbar_wait(s_full, i & 1);
            tc_fence_after();
            constexpr int NCH = (NK + 31) / 32;
            uint32_t sr[NCH][32];
#pragma unroll
            for (int c = 0; c < NCH; ++c) {
                if (NK - c * 32 >= 32) {
                    tmem_ld_32x32(s_tmem + c * 32, sr[c]);
                } else {
                    uint32_t t16[16];
                    tmem_ld_32x16(s_tmem + c * 32, t16);
#pragma unroll
                    for (int t = 0; t < 16; ++t) sr[c][t] = t16[t];
                }
            }
            tc_wait_ld();
            float mx = -INFINITY;
#pragma unroll
            for (int c = 0; c < NCH; ++c)
#pragma unroll
                for (int t = 0; t < 32; ++t)
                    if (c * 32 + t < NK) {
                        if (c * 32 + t >= p.n_kv || (p.causal && c * 32 + t > qrow)) sr[c][t] = __float_as_uint(-INFINITY);
                        mx = fmaxf(mx, __uint_as_float(sr[c][t]));
                    }
            const float m = mx * p.scale_log2;
            const uint64_t negm2 = pack_f32x2(-m, -m);
            uint64_t sum2 = pack_f32x2(0.f, 0.f);
#pragma unroll
            for (int c = 0; c < NCH; ++c) {
                constexpr int dummy = 0;
                (void)dummy;
                const int npair = (NK - c * 32 >= 32) ? 16 : (NK - c * 32) / 2;
                uint32_t pk[16];
#pragma unroll
                for (int t = 0; t < 16; ++t) {
                    if (t < npair) {
                        const uint64_t x2 = ffma2(pack_f32x2(__uint_as_float(sr[c][2 * t]), __uint_as_float(sr[c][2 * t + 1])), scale2, negm2);
                        float x0, x1;
                        unpack_f32x2(x2, x0, x1);
                        const float p0 = fast_exp2(x0), p1 = fast_exp2(x1);  // exp2(-inf) = 0 for the masked keys
                        sum2 = fadd2(sum2, pack_f32x2(p0, p1));
                        pk[t] = pack_half2(p0, p1);
                    } else {
                        pk[t] = 0u;
                    }
                }
                if (npair == 16) {
                    tmem_st_32x16(s_tmem + c * 16, pk);
                } else {
                    uint32_t p8[8];
#pragma unroll
                    for (int t = 0; t < 8; ++t) p8[t] = pk[t];
                    tmem_st_32x8(s_tmem + c * 16, p8);
                }
            }
            float l, l_hi;
            unpack_f32x2(sum2, l, l_hi);
            l += l_hi;
            tc_wait_st();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(p_full);
            mbar_wait(o_full, i & 1);
            tc_fence_after();
            float o_acc[ATT_D];
#pragma unroll
            for (int c = 0; c < 2; ++c) {
                uint32_t r[32];
                tmem_ld_32x32(o_tmem + c * 32, r);
                tc_wait_ld();
#pragma unroll
                for (int t = 0; t < 32; ++t) o_acc[c * 32 + t] = __uint_as_float(r[t]);
            }
            if (qrow < p.n_q) {
                const float inv = p.out_weight / l;
                __half* op = p.out + (long long)p.out_b[item] * p.out_bs + (long long)qrow * p.out_ld + p.out_col0 +
                             (h0 + i) * ATT_D;
                uint4* op4 = reinterpret_cast<uint4*>(op);
#pragma unroll
                for (int t = 0; t < 8; ++t) {
                    float v[8];
#pragma unroll
                    for (int e = 0; e < 8; ++e) v[e] = o_acc[t * 8 + e] * inv;
                    if (p.accumulate) {
                        const uint4 u = op4[t];
                        const __half2* h2 = reinterpret_cast<const __half2*>(&u);
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            const float2 f = __half22float2(h2[e]);
                            v[2 * e] += f.x;
                            v[2 * e + 1] += f.y;
                        }
                    }
                    op4[t] = make_uint4(pack_half2(v[0], v[1]), pack_half2(v[2], v[3]), pack_half2(v[4], v[5]),
                                        pack_half2(v[6], v[7]));
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
}

template <int NK>
static int launch_cross(AttnParams& p, const omg_attn_desc* d, cudaStream_t stream, int max_qb, int max_kb, int max_vb) {
    static bool configured = false;
    if (!configured) {
        OMG_CUDA(cudaFuncSetAttribute(attn_cross_kernel<NK>, cudaFuncAttributeMaxDynamicSharedMemorySize, AttXCfg<NK>::SMEM));
        configured = true;
    }
    (void)max_qb;
    const int cols = d->heads * 64;
    // K / V boxes cover the whole (padded) key sequence; rows beyond n_kv are zero-filled by TMA and masked
    {
        const uint64_t dims[3] = {(uint64_t)(d->k_col0 + cols), (uint64_t)d->n_kv, (uint64_t)(max_kb + 1)};
        const uint64_t strides[3] = {1, (uint64_t)d->k_ld, (uint64_t)d->k_bs};
        const uint32_t box[3] = {64, NK, 1};
        if (make_tmap_16b(&p.k_map, d->k, 3, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B)) return 1;
    }
    {
        const uint64_t dims[3] = {(uint64_t)(d->v_col0 + cols), (uint64_t)d->n_kv, (uint64_t)(max_vb + 1)};
        const uint64_t strides[3] = {1, (uint64_t)d->v_ld, (uint64_t)d->v_bs};
        const uint32_t box[3] = {64, NK, 1};
        if (make_tmap_16b(&p.v_map, d->v, 3, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B)) return 1;
    }
    // heads per CTA: as many as keep the grid at >= ~1.5 CTAs per SM slot pair (148 SMs x 2), at most 8
    const int tiles = ((d->n_q + ATT_BQ - 1) / ATT_BQ) * d->n_items;
    int hpc = 1;
    while (hpc < 8 && hpc * 2 <= d->heads && (long)tiles * ((d->heads + 2 * hpc - 1) / (2 * hpc)) >= 148) hpc *= 2;
    if (d->heads % 5 == 0 && hpc == 4 && (long)tiles * (d->heads / 5) >= 128) hpc = 5;  // 10 / 20 heads: 5 per CTA, no tail group
    {
        static int force_hpc = -1;
        if (force_hpc < 0) {
            const char* e = getenv("OMG_ATTN_HPC");  // heads per CTA of the cross-attention kernel (measurements)
            force_hpc = e ? atoi(e) : 0;
        }
        if (force_hpc > 0) hpc = std::min(force_hpc, d->heads);
    }
    dim3 grid((d->n_q + ATT_BQ - 1) / ATT_BQ, (d->heads + hpc - 1) / hpc, d->n_items);
    OMG_CUDA(launch_pdl(attn_cross_kernel<NK>, grid, dim3(256), AttXCfg<NK>::SMEM, stream, p, hpc));
    return check_launch("attn_cross_kernel");
}

static int make_attn_map(CUtensorMap* m, const void* ptr, int cols, int ld, int tokens, long long bs, int nb,
                         uint32_t box_rows) {
    const uint64_t dims[3] = {(uint64_t)cols, (uint64_t)tokens, (uint64_t)nb};
    const uint64_t strides[3] = {1, (uint64_t)ld, (uint64_t)bs};
    const uint32_t box[3] = {64, box_rows, 1};
    return make_tmap_16b(m, ptr, 3, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B);
}

}  // namespace omg

using namespace omg;

static int attention_impl(const omg_attn_desc* d, void* stream_) {
    cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
    OMG_CHECK(d != nullptr, "omg_attention: null descriptor");
    OMG_CHECK(d->head_dim == 64, "omg_attention: head_dim %d unsupported (SDXL uses 64)", d->head_dim);
    OMG_CHECK(d->n_items >= 1 && d->n_items <= OMG_ATTN_MAX_ITEMS, "omg_attention: n_items=%d out of range",
              d->n_items);
    OMG_CHECK(d->n_q >= 1 && d->n_kv >= 1 && d->heads >= 1, "omg_attention: empty problem");
    OMG_CHECK(d->q && d->k && d->v && d->out, "omg_attention: null pointer");
    OMG_CHECK(d->out_ld % 8 == 0 && d->out_col0 % 8 == 0 && d->out_bs % 8 == 0,
              "omg_attention: output must be 16 B aligned per row");
    static bool configured = false;
    static int force_g = 0;
    static bool cross_kernel = true;
    static bool persistent = true;
    static int p_stages = 0;
    static int num_sms = 148;
    if (!configured) {
        OMG_CUDA(cudaFuncSetAttribute(attn_tc_kernel<1, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, AttCfg<1, 3>::SMEM));
        OMG_CUDA(cudaFuncSetAttribute(attn_tc_kernel<1, 5>, cudaFuncAttributeMaxDynamicSharedMemorySize, AttCfg<1, 5>::SMEM));
        OMG_CUDA(cudaFuncSetAttribute(attn_tc_kernel<2, 6>, cudaFuncAttributeMaxDynamicSharedMemorySize, AttCfg<2, 6>::SMEM));
        OMG_CUDA(cudaFuncSetAttribute(attn_p_kernel<5, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, AttPCfg<5, 2>::SMEM));
        OMG_CUDA(cudaFuncSetAttribute(attn_p_kernel<6, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, AttPCfg<6, 1>::SMEM));
        const char* e7 = getenv("OMG_ATTN_PSTAGES");  // 5 | 6: force the (KV stages, Q buffers) = (5, 2) | (6, 1) variant
        p_stages = e7 ? atoi(e7) : 0;
        const char* e6 = getenv("OMG_ATTN_PERSISTENT");  // 0: one CTA per tile
        persistent = !(e6 && atoi(e6) == 0);
        {
            int dev = 0;
            OMG_CUDA(cudaGetDevice(&dev));
            OMG_CUDA(cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev));
        }
        const char* e = getenv("OMG_ATTN_TILES");  // 1 | 2: force the tiles-per-CTA variant (measurements)
        force_g = e ? atoi(e) : 0;
        const char* e3 = getenv("OMG_ATTN_CROSS");  // 0: cross-attention through the per-(tile, head) kernel
        cross_kernel = !(e3 && atoi(e3) == 0);
        configured = true;
    }
    AttnParams p;
    memset(&p, 0, sizeof(p));
    int max_qb = 0, max_kb = 0, max_vb = 0;
    for (int i = 0; i < d->n_items; ++i) {
        p.out_b[i] = d->out_b[i];
        p.q_b[i] = d->q_b[i];
        p.k_b[i] = d->k_b[i];
        p.v_b[i] = d->v_b[i];
        max_qb = d->q_b[i] > max_qb ? d->q_b[i] : max_qb;
        max_kb = d->k_b[i] > max_kb ? d->k_b[i] : max_kb;
        max_vb = d->v_b[i] > max_vb ? d->v_b[i] : max_vb;
        OMG_CHECK(d->out_b[i] >= 0 && d->q_b[i] >= 0 && d->k_b[i] >= 0 && d->v_b[i] >= 0,
                  "omg_attention: negative batch index in item %d", i);
    }
    const int cols = d->heads * 64;
    if (make_attn_map(&p.q_map, d->q, d->q_col0 + cols, d->q_ld, d->n_q, d->q_bs, max_qb + 1, ATT_BQ)) return 1;
    if (make_attn_map(&p.k_map, d->k, d->k_col0 + cols, d->k_ld, d->n_kv, d->k_bs, max_kb + 1, ATT_BKV)) return 1;
    if (make_attn_map(&p.v_map, d->v, d->v_col0 + cols, d->v_ld, d->n_kv, d->v_bs, max_vb + 1, ATT_BKV)) return 1;
    p.out = static_cast<__half*>(d->out);
    p.out_ld = d->out_ld;
    p.out_bs = d->out_bs;
    p.n_q = d->n_q;
    p.n_kv = d->n_kv;
    p.heads = d->heads;
    p.q_col0 = d->q_col0;
    p.k_col0 = d->k_col0;
    p.v_col0 = d->v_col0;
    p.out_col0 = d->out_col0;
    p.n_items = d->n_items;
    p.scale_log2 = d->scale * 1.4426950408889634f;
    p.out_weight = d->out_weight;
    p.accumulate = d->accumulate;
    p.causal = d->causal;
#ifdef OMG_ATT_TRACE
    {
        const char* e = getenv("OMG_ATT_TRACE_PTR");
        p.trace = e ? reinterpret_cast<long long*>(strtoull(e, nullptr, 0)) : nullptr;
    }
#endif
    OMG_CHECK(!d->causal || (d->n_kv <= 128 && d->n_q <= 128), "omg_attention: causal masking is available for sequences of <= 128 tokens");
    // Single-tile CTAs, two per SM, for every shape: two independent CTAs overlap each other's prologue / epilogue
    // with the other's main loop, which the two-tile CTA (tiles start and end together) cannot (measured, 5 KV
    // stages each: 604 vs 569 TFLOP/s at N = 4096, 388 vs 362 at N = 1024).  Short key sequences (cross-attention,
    // one or two KV blocks) take the 3-stage variant: less shared memory to set up per CTA.
    const int tiles = force_g ? force_g : 1;
    if ((!force_g && cross_kernel && d->n_kv <= 128) || d->causal) {
        if (d->n_kv <= 16) return launch_cross<16>(p, d, stream, max_qb, max_kb, max_vb);
        if (d->n_kv <= 80) return launch_cross<80>(p, d, stream, max_qb, max_kb, max_vb);
        return launch_cross<128>(p, d, stream, max_qb, max_kb, max_vb);
    }
    if (!force_g && persistent && d->n_kv > 2 * ATT_BKV) {
        const int n_slabs = (d->n_q + ATT_BQ - 1) / ATT_BQ;
        const int n_tiles = n_slabs * d->heads * d->n_items;
        const int grid = std::min(n_tiles, 2 * num_sms);
        const bool deep = p_stages == 6 || (p_stages == 0 && false);
        if (deep)
            OMG_CUDA(launch_pdl(attn_p_kernel<6, 1>, dim3(grid), dim3(256), AttPCfg<6, 1>::SMEM, stream, p, n_tiles, n_slabs));
        else
            OMG_CUDA(launch_pdl(attn_p_kernel<5, 2>, dim3(grid), dim3(256), AttPCfg<5, 2>::SMEM, stream, p, n_tiles, n_slabs));
        return check_launch("attn_p_kernel");
    }
    if (tiles == 1) {
        dim3 grid((d->n_q + ATT_BQ - 1) / ATT_BQ, d->heads, d->n_items);
        if (d->n_kv <= 2 * ATT_BKV)
            OMG_CUDA(launch_pdl(attn_tc_kernel<1, 3>, grid, dim3(AttCfg<1, 3>::THREADS), AttCfg<1, 3>::SMEM, stream, p));
        else
            OMG_CUDA(launch_pdl(attn_tc_kernel<1, 5>, grid, dim3(AttCfg<1, 5>::THREADS), AttCfg<1, 5>::SMEM, stream, p));
    } else {
        dim3 grid((d->n_q + 2 * ATT_BQ - 1) / (2 * ATT_BQ), d->heads, d->n_items);
        OMG_CUDA(launch_pdl(attn_tc_kernel<2, 6>, grid, dim3(AttCfg<2, 6>::THREADS), AttCfg<2, 6>::SMEM, stream, p));
    }
    return check_launch("attn_tc_kernel");
}

// C-ABI entry points: launch, and - while this thread records a launch plan (omg_plan_record_begin) - remember the call
extern "C" int omg_attention(const omg_attn_desc* d, void* stream_) {
    const int rc = attention_impl(d, stream_);
    if (rc == 0 && ::omg::plan_recording()) {
        const omg_attn_desc c = *d;  // by value: a plan outlives the caller's descriptor
        ::omg::plan_note([c](void* s) { return attention_impl(&c, s); });
    }
    return rc;
}
