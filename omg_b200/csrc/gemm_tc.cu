// Persistent tcgen05 implicit-GEMM for every Linear / Conv2d / LoRA / GEGLU of the SDXL UNet.
//
//   out[pix, n] = epi( sum_seg sum_k A_seg[pix + (dx,dy), k] * W[n, b_k0 + k] + bias[n] + rowvec[b, n] ) + residual
//
// * Activations are channels-last, so a 3x3 conv is 9 K-segments whose A tiles are the SAME tensor read
//   through TMA at shifted pixel coordinates (hardware zero-fill = padding); no im2col buffer exists.
//   Stride-2 convs and nearest-2x-upsample convs use strided "phase" views of the tensor as A / D maps.
//   A ResBlock's 1x1 shortcut and a LoRA delta  s*B(Ax)  are just more K-segments of the same accumulator.
// * One CTA per SM, 320 threads: warp 0 = TMA producer, warp 1 = tcgen05.mma issuer (single thread) + TMEM
//   owner, warps 2..9 = epilogue (TMEM -> registers -> swizzled smem -> TMA store).  Two TMEM accumulator
//   stages so the epilogue of tile i overlaps the mainloop of tile i+1.  Large GEMMs run as CTA pairs
//   (cta_group::2, 256 x 256 tiles, each CTA stages half of the weight tile).
// * Tile 128 (pixels) x BN (channels) x 64 (K); operands land in smem in the 128B-swizzled K-major layout
//   the UMMA descriptors expect.
//
// Roofline: tensor-bound (ridge ~227 flop/B); algorithmic FLOPs per launch = 2 * pixels * N * sum(k_len).
#include <cuda_fp16.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <type_traits>

#include "../../include/omg_b200.h"
#include "host_common.h"
#include "ptx.cuh"

namespace omg {

constexpr int BM = 128;
constexpr int BK = 64;
constexpr int GEMM_THREADS = 320;  // warp 0 TMA, warp 1 MMA, warps 2..9 epilogue
constexpr int STAGING_BYTES = 8 * 2048;  // 8 epilogue warps x (32 rows x 64 B)

struct SegDev {
    int a_map, dx, dy, a_c0, k_blocks, b_k0, b_map;
};

struct alignas(64) GemmParams {
    CUtensorMap a_maps[OMG_MAX_A];
    CUtensorMap b_maps[2];
    CUtensorMap d_map;
    SegDev segs[OMG_MAX_SEGS];
    int n_segs;
    int m_tiles, n_tiles;
    int tw, th, tiles_w, tiles_h;
    int store_w, store_h;
    int img_w, img_h, img_b;
    int N, N_out;
    const void* bias;          // element type of the kernel instantiation (fp16 | bf16)
    const void* rowvec;
    int rowvec_ld;
    const void* residual;
    int residual_ld;
    int act_silu;
    // LayerNorm folded into the GEMM pair (see omg_gemm_desc): statistics written by the producer's epilogue ...
    float* stats_out;          // [n_tiles][rows][2] partial (sum, sum of squares) of this GEMM's output rows, or null
    // ... and consumed by the next GEMM's epilogue: out = rstd * (acc - mean * c1[n]) + c2[n]
    const float* stats_in;     // [stats_parts][rows][2] or null
    int stats_parts;
    long long stats_rows;      // rows per part (both directions)
    float ln_inv_dim, ln_eps;
    const float* col_c1;       // [N] fp32: row sums of the gamma-folded weights
    const float* col_c2;       // [N] fp32: W beta + bias
    int n_col_groups;          // c1/c2 are [n_col_groups][N]; row group g = rows [col_group_end[g-1], col_group_end[g])
    long long col_group_end[8];
    int w_group_rows;          // > 0: the weight matrix holds one [N, K] plane per row group (per-stream merged LoRA)
    // fp32 master copy of the residual trunk: the addend is read from / the result also written to fp32 twins, so the
    // chain h <- h + f(h) accumulates in fp32 while every GEMM / norm input stays the fp16 copy
    const float* residual_f32;
    long long residual_f32_ld;
    float* out_f32;
    long long out_f32_ld;
    float4* col_stats;         // GroupNorm statistics of the output: [B][cs_rb_total][N] float2 (sum, sumsq), or null
    int cs_rb0, cs_rb_total;
};

// CTAS = 2: a CTA pair (cluster of 2, cta_group::2) works on a 256 x BN tile; each CTA stages its own 128 A rows and
// HALF of the B tile, so the L2 -> smem traffic per flop drops by a third (the mainloop is TMA-latency bound: ncu shows
// lts/xbar at ~50 % with the tensor pipe at 62 % for the 128 x 256 single-CTA tile).
// MT = 2 ("tall tile", single CTA): two 128-row sub-tiles share every weight tile -> a third less L2 -> smem traffic
// per flop WITHOUT a cluster, and half as many work units.  The narrow-N GEMMs at c = 1280 (out-proj, q, FF-out,
// N = 1280, M = 4096: 256 tiles of 128 x 160 on 148 SMs, L2-latency bound) become 128 tiles of 256 x 160 = one wave.
// Both accumulators fill the TMEM (no second stage): the epilogue is exposed, acceptable for 1-2 tiles per CTA.
template <int BN, int CTAS = 1, int MT = 1>
struct GemmCfg {
    static constexpr int A_BYTES = MT * BM * BK * 2;
    static constexpr int B_BYTES = (BN / CTAS) * BK * 2;
    static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
    // per-column epilogue vectors (bias | c1), one plane per sub-tile
    static constexpr int VEC_PLANE = MT == 2 ? BN : (BN > 256 ? BN : 256);
    static constexpr int VEC_BYTES = 2 * MT * VEC_PLANE * 4;
    // tall tiles need the last KB for a 4th stage: they rely on the (in practice guaranteed, checked at run time)
    // 1024 B alignment of the dynamic shared memory window instead of reserving alignment slack
    static constexpr int ALIGN_SLACK = MT == 2 ? 0 : 1024;
    static constexpr int BUDGET = 227 * 1024 - ALIGN_SLACK - STAGING_BYTES - VEC_BYTES - 256 /*bars*/;
    static constexpr int STAGES_RAW = BUDGET / STAGE_BYTES;
    static constexpr int STAGES = STAGES_RAW > 8 ? 8 : STAGES_RAW;
    static constexpr int SMEM_BYTES = ALIGN_SLACK + STAGES * STAGE_BYTES + STAGING_BYTES + VEC_BYTES + 256;
    // BN = 320 (CTA pairs only): a 256 x 320 pair tile = two N = 160 MMAs per K step into one 320-column accumulator
    // (operand bytes per MMA cycle: 128x256 tiles 96 B/clk, tall 256x160 83, 256x256 pairs 64, 256x320 pairs 56).
    static constexpr int ACC_STRIDE = BN <= 64 ? 64 : (BN <= 128 ? 128 : (BN <= 256 ? 256 : 512));  // TMEM columns per accumulator
    static constexpr int TMEM_COLS = BN > 256 ? 512 : 2 * ACC_STRIDE;
    static constexpr int ACC_STAGES = (MT == 2 || BN > 256) ? 1 : 2;  // MT = 2: the two accumulators ARE the two sub-tiles
};

// GEGLU / erf-GELU use libdevice's erff: measured on one box against a branch-free Abramowitz-Stegun form (rcp + ex2 on the
// MUFU): 91 vs 94-98 us on FF1 4096 x 10240 x 1280 and 109-112 vs 147-157 us on 16384 x 5120 x 640 (the epilogue of a short-K
// tile is MUFU-bound with the two-transcendental form), so erff stays.
__device__ __forceinline__ float gelu_exact(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752f)); }

// FEAT selects what the epilogue carries besides bias / time-embedding vector / residual / LayerNorm fold / row statistics:
//   0  nothing else (the linears of the transformer blocks: the hot instantiations stay as lean as they were in round 1 -
//      same-box A/B: the all-in-one epilogue cost +3..17 % on these launches, profiles/r02_gemm_builds_ab.jsonl)
//   1  + GroupNorm column statistics (convs, proj_out)
//   2  + activations (SiLU, quick-GELU, erf / tanh GELU) and the fp32 residual-trunk twins (once-per-call MLPs, CLIP / SAM
//      towers, OMG_TRUNK_F32)
// T is the 16-bit element type of every operand and of the output: __half, or __nv_bfloat16 (instantiated only with
// FEAT 0 and OMG_EPI_NONE, what the VAE decoder uses).
template <int BN, int EPI, int CTAS, int MT, int FEAT, typename T = __half>
__global__ void __launch_bounds__(GEMM_THREADS, 1) gemm_tc_kernel(const __grid_constant__ GemmParams p) {
    constexpr bool kStats = FEAT >= 1, kExtra = FEAT >= 2;
    using T2 = typename Pair<T>::type;
    static_assert(MT == 1 || CTAS == 1, "tall tiles are a single-CTA variant");
    static_assert(BN <= 256 || (CTAS == 2 && BN == 320 && EPI != OMG_EPI_GEGLU), "BN = 320 exists as a CTA-pair tile only");
    using Cfg = GemmCfg<BN, CTAS, MT>;
    constexpr int MSUB = CTAS * MT;  // 128-row m-tiles per work unit
    constexpr int STAGES = Cfg::STAGES;
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    if constexpr (Cfg::ALIGN_SLACK == 0) {
        if (smem != smem_raw) __trap();  // dynamic smem window not 1024 B aligned: the swizzled tiles would be garbage
    }
    uint8_t* staging = smem + STAGES * Cfg::STAGE_BYTES;
    float* s_bias = reinterpret_cast<float*>(staging + STAGING_BYTES);
    float* s_c1 = s_bias + MT * Cfg::VEC_PLANE;
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(s_c1 + MT * Cfg::VEC_PLANE);
    uint64_t* empty_bar = full_bar + STAGES;
    uint64_t* tfull_bar = empty_bar + STAGES;
    uint64_t* tempty_bar = tfull_bar + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    // work unit = (group of CTAS consecutive m-tiles, n-tile); CTA `cta_rank` of the pair owns m-tile unit_m*CTAS+rank
    const uint32_t cta_rank = (CTAS == 2) ? cluster_ctarank() : 0u;
    const bool leader = cta_rank == 0;
    const int total_tiles = ((p.m_tiles + MSUB - 1) / MSUB) * p.n_tiles;
    const int unit0 = blockIdx.x / CTAS, unit_step = gridDim.x / CTAS;
    const int tiles_per_img = p.tiles_w * p.tiles_h;

    if (warp == 0 && lane == 0) {
        for (int i = 0; i < OMG_MAX_A; ++i) tma_prefetch_desc(&p.a_maps[i]);
        tma_prefetch_desc(&p.b_maps[0]);
        tma_prefetch_desc(&p.b_maps[1]);
        tma_prefetch_desc(&p.d_map);
        for (int i = 0; i < STAGES; ++i) {
            mbar_init(&full_bar[i], 1);
            mbar_init(&empty_bar[i], 1);
        }
        for (int i = 0; i < 2; ++i) {
            mbar_init(&tfull_bar[i], 1);
            mbar_init(&tempty_bar[i], 8 * CTAS);  // epilogue warps of every CTA of the pair arrive on the leader's
        }
        fence_barrier_init();
    }
    if (warp == 1) {
        if constexpr (CTAS == 2) tmem_alloc_pair(tmem_slot, Cfg::TMEM_COLS);
        else tmem_alloc(tmem_slot, Cfg::TMEM_COLS);
    }
    tc_fence_before();
    if constexpr (CTAS == 2) cluster_sync();
    else __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    griddep_launch_dependents();  // the prologue above overlaps the previous kernel's tail
    griddep_wait();               // operands / residual / output buffers belong to earlier kernels until here

    if (warp == 0) {
        // ------------------------------------------------------------- TMA producer
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            for (int tile = unit0; tile < total_tiles; tile += unit_step) {
                const int m_tile = (tile / p.n_tiles) * MSUB + (int)cta_rank * MT, n_tile = tile % p.n_tiles;
                const int b = m_tile / tiles_per_img;  // >= img_b for the odd m-tile of the last pair: TMA zero-fills
                const int rem = m_tile % tiles_per_img;
                const int h0 = (rem / p.tiles_w) * p.th, w0 = (rem % p.tiles_w) * p.tw;
                // second 128-row sub-tile of a tall tile (the next m-tile in (w, h, image) order)
                const int b1 = (m_tile + 1) / tiles_per_img, rem1 = (m_tile + 1) % tiles_per_img;
                const int h1 = (rem1 / p.tiles_w) * p.th, w1 = (rem1 % p.tiles_w) * p.tw;
                // this CTA's slice of the B tile (BN = 320: two 80-row slices, one per N = 160 MMA)
                int n0 = n_tile * BN + (int)cta_rank * (BN > 256 ? 80 : BN / CTAS);
                if (p.w_group_rows > 0) {  // multi-stream launch: this tile's stream selects the weight plane
                    const long long tile_pix0 = ((long long)b * p.img_h + h0) * p.img_w + w0;
                    for (int g2 = 0; g2 + 1 < p.n_col_groups; ++g2)
                        if (tile_pix0 >= p.col_group_end[g2]) n0 += p.w_group_rows;
                }
                for (int s = 0; s < p.n_segs; ++s) {
                    const SegDev sg = p.segs[s];
                    for (int kb = 0; kb < sg.k_blocks; ++kb) {
                        mbar_wait(&empty_bar[stage], phase ^ 1);
                        uint8_t* a_dst = smem + stage * Cfg::STAGE_BYTES;
                        uint8_t* b_dst = a_dst + Cfg::A_BYTES;
                        if constexpr (CTAS == 2) {
                            // both CTAs' bytes are counted on the leader's barrier
                            if (leader) mbar_arrive_expect_tx(&full_bar[stage], 2 * Cfg::STAGE_BYTES);
                            tma_load_4d_pair(a_dst, &p.a_maps[sg.a_map], &full_bar[stage], sg.a_c0 + kb * BK,
                                             w0 + sg.dx, h0 + sg.dy, b);
                            tma_load_2d_pair(b_dst, &p.b_maps[sg.b_map], &full_bar[stage], sg.b_k0 + kb * BK, n0);
                            if constexpr (BN > 256)
                                tma_load_2d_pair(b_dst + 80 * BK * 2, &p.b_maps[sg.b_map], &full_bar[stage], sg.b_k0 + kb * BK,
                                                 n0 + 160);
                        } else {
                            mbar_arrive_expect_tx(&full_bar[stage], Cfg::STAGE_BYTES);
                            tma_load_4d(a_dst, &p.a_maps[sg.a_map], &full_bar[stage], sg.a_c0 + kb * BK, w0 + sg.dx,
                                        h0 + sg.dy, b);
                            if constexpr (MT == 2)
                                tma_load_4d(a_dst + BM * BK * 2, &p.a_maps[sg.a_map], &full_bar[stage], sg.a_c0 + kb * BK,
                                            w1 + sg.dx, h1 + sg.dy, b1);
                            tma_load_2d(b_dst, &p.b_maps[sg.b_map], &full_bar[stage], sg.b_k0 + kb * BK, n0);
                        }
                        if (++stage == STAGES) {
                            stage = 0;
                            phase ^= 1;
                        }
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------- MMA issuer (one thread)
        if (lane == 0 && leader) {
            constexpr uint32_t idesc = umma_idesc_f16(BM * CTAS, BN > 256 ? 160 : BN, false, false,
                                                      std::is_same<T, __nv_bfloat16>::value);
            int stage = 0;
            uint32_t phase = 0;
            int acc = 0;
            uint32_t acc_phase = 0;
            for (int tile = unit0; tile < total_tiles; tile += unit_step) {
                mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + acc * Cfg::ACC_STRIDE;  // (ACC_STAGES == 1 for tall tiles: acc == 0)
                uint32_t accumulate = 0;
                for (int s = 0; s < p.n_segs; ++s) {
                    const int kbs = p.segs[s].k_blocks;
                    for (int kb = 0; kb < kbs; ++kb) {
                        mbar_wait(&full_bar[stage], phase);
                        tc_fence_after();
                        const uint32_t a_addr = smem_u32(smem + stage * Cfg::STAGE_BYTES);
                        const uint64_t a_desc = umma_desc_sw128(a_addr, 1024, 16);
                        const uint64_t b_desc = umma_desc_sw128(a_addr + Cfg::A_BYTES, 1024, 16);
#pragma unroll
                        for (int k = 0; k < BK / 16; ++k) {
                            // +32 B per K=16 step inside the 128 B swizzle atom (start-address field is >>4)
                            if constexpr (CTAS == 2) tc_mma_f16_ss_pair(d_tmem, a_desc + 2 * k, b_desc + 2 * k, idesc, accumulate);
                            else tc_mma_f16_ss(d_tmem, a_desc + 2 * k, b_desc + 2 * k, idesc, accumulate);
                            if constexpr (BN > 256)  // second N = 160 half: the next 80-row slice of B, columns 160..319
                                tc_mma_f16_ss_pair(d_tmem + 160, a_desc + 2 * k, b_desc + ((80 * BK * 2) >> 4) + 2 * k, idesc,
                                                   accumulate);
                            if constexpr (MT == 2)  // second sub-tile: A rows 128..255 (+16 KB), accumulator + ACC_STRIDE
                                tc_mma_f16_ss(d_tmem + Cfg::ACC_STRIDE, a_desc + ((BM * BK * 2) >> 4) + 2 * k, b_desc + 2 * k,
                                              idesc, accumulate);
                            accumulate = 1;
                        }
                        if constexpr (CTAS == 2) tc_commit_pair(&empty_bar[stage]);
                        else tc_commit(&empty_bar[stage]);
                        if (++stage == STAGES) {
                            stage = 0;
                            phase ^= 1;
                        }
                    }
                }
                if constexpr (CTAS == 2) tc_commit_pair(&tfull_bar[acc]);
                else tc_commit(&tfull_bar[acc]);
                if (++acc == Cfg::ACC_STAGES) {
                    acc = 0;
                    acc_phase ^= 1;
                }
            }
        }
    } else {
        // ------------------------------------------------------------- epilogue warps
        // 8 warps: TMEM lane quarter q = warp % 4 (hardware rule), and within a quarter the two warps split the
        // tile's 32-column chunks by parity.  (With 4 warps the epilogue of short-K tiles - K <= 1280 at BN 160 - took
        // as long as their mainloop and throttled the tensor core through the 2-stage accumulator ring.)
        const int ew = warp - 2;
        const int q = warp & 3;
        const int half = ew >> 2;
        const int et = q * 32 + lane;  // row of the (sub-)tile owned by this thread
        // MT == 1: the two warps of a lane quarter split the column chunks by parity.  MT == 2: warp `half` owns
        // sub-tile `half` (its own accumulator) and walks all of its chunks.
        constexpr int CH_STEP = MT == 2 ? 1 : 2;
        const int ch0 = MT == 2 ? 0 : half;
        const int sub = MT == 2 ? half : 0;
        uint8_t* sbuf = staging + (q * 2 + half) * 2048;
        int acc = 0;
        uint32_t acc_phase = 0;
        constexpr int ACC_PER_CHUNK = (EPI == OMG_EPI_GEGLU) ? 64 : 32;
        constexpr int NCH = BN / ACC_PER_CHUNK;
        constexpr int NIT = (NCH + CH_STEP - 1) / CH_STEP;  // chunks per warp
        for (int tile = unit0; tile < total_tiles; tile += unit_step) {
            const int m_tile = (tile / p.n_tiles) * MSUB + (int)cta_rank * MT + sub, n_tile = tile % p.n_tiles;
            const int b = m_tile / tiles_per_img;
            const int rem = m_tile % tiles_per_img;
            const int h0 = (rem / p.tiles_w) * p.th, w0 = (rem % p.tiles_w) * p.tw;
            const int n0 = n_tile * BN;

            asm volatile("bar.sync 1, 256;" ::: "memory");  // previous tile's s_bias readers are done
            const bool ln = p.stats_in != nullptr;
            // tiles never straddle row groups (host guarantees 128-row alignment): pick this tile's c1/c2 plane
            size_t cg = 0;
            if (ln && p.n_col_groups > 1) {
                const long long tile_pix0 = ((long long)b * p.img_h + h0) * p.img_w + w0;
                for (int g2 = 0; g2 + 1 < p.n_col_groups; ++g2)
                    if (tile_pix0 >= p.col_group_end[g2]) cg = g2 + 1;
                cg *= (size_t)p.N;
            }
            // per-column vectors of THIS warp group's sub-tile (tall tiles: each half fills its own 256-entry plane,
            // the two sub-tiles may belong to different images / streams)
            float* sbias = s_bias + sub * Cfg::VEC_PLANE;
            float* sc1 = s_c1 + sub * Cfg::VEC_PLANE;
            for (int j = (MT == 2 ? q * 32 + lane : ew * 32 + lane); j < BN; j += (MT == 2 ? 128 : 256)) {
                float v = 0.f, c1 = 0.f;
                const int n = n0 + j;
                if (n < p.N) {
                    if (ln) {
                        v = p.col_c2[cg + n];
                        c1 = p.col_c1[cg + n];
                    } else {
                        if (p.bias) v += to_float(static_cast<const T*>(p.bias)[n]);
                        if (p.rowvec && b < p.img_b) v += to_float(static_cast<const T*>(p.rowvec)[(size_t)b * p.rowvec_ld + n]);
                    }
                }
                sbias[j] = v;
                sc1[j] = c1;
            }
            asm volatile("bar.sync 1, 256;" ::: "memory");

            const int ph = h0 + et / p.tw, pw = w0 + et % p.tw;
            const bool row_valid = (ph < p.img_h) && (pw < p.img_w) && (b < p.img_b);
            const size_t pix = ((size_t)b * p.img_h + ph) * p.img_w + pw;
            // folded LayerNorm: this row's mean / rstd from the producer's partial sums (one row per thread, so no
            // cross-thread reduction is needed); out = ln_a * acc + (ln_k * c1 + c2), ln_k = -rstd * mean
            float ln_a = 1.0f, ln_k = 0.f;
            if (ln && row_valid) {
                float sa = 0.f, sq = 0.f;
                for (int t = 0; t < p.stats_parts; ++t) {
                    const float2 st = __ldg(reinterpret_cast<const float2*>(p.stats_in) + (size_t)t * p.stats_rows + pix);
                    sa += st.x;
                    sq += st.y;
                }
                const float mu = sa * p.ln_inv_dim;
                ln_a = rsqrtf(fmaxf(sq * p.ln_inv_dim - mu * mu, 0.f) + p.ln_eps);
                ln_k = -ln_a * mu;
            }
            float row_sum = 0.f, row_sq = 0.f;  // statistics of THIS GEMM's output row (stats_out), this warp's chunks
            // pixel origin of this warp's 32-row store box
            const int sh = h0 + (q * 32) / p.tw, sw = w0 + (q * 32) % p.tw;

            // residual rows are fetched two of this warp's chunks ahead (the first two before the accumulator is even
            // ready), so their HBM/L2 latency hides behind the mainloop / the previous chunks
            uint4 res[2][4];
            const bool has_res = (EPI != OMG_EPI_GEGLU) && p.residual != nullptr && row_valid;
            const T* res_row = has_res ? static_cast<const T*>(p.residual) + pix * (size_t)p.residual_ld + n0 : nullptr;
            auto load_res = [&](int c, uint4(&dst)[4]) {
                if (has_res && c < NCH && n0 + c * 32 < p.N) {
                    const uint4* rp = reinterpret_cast<const uint4*>(res_row + c * 32);
#pragma unroll
                    for (int j = 0; j < 4; ++j) dst[j] = __ldg(rp + j);
                }
            };
            if constexpr (EPI != OMG_EPI_GEGLU) {
                load_res(ch0, res[0]);
                load_res(ch0 + CH_STEP, res[1]);
            }

            mbar_wait(&tfull_bar[acc], acc_phase);
            tc_fence_after();
            const uint32_t t_row = tmem_base + (acc + sub) * Cfg::ACC_STRIDE + ((uint32_t)(q * 32) << 16);

            // One 32-column chunk of the accumulator.  The chunk loop below is NOT fully unrolled: fully unrolled the
            // epilogue was ~90 KB of straight-line code executed once per tile and spent 60 % of its time in
            // instruction-fetch stalls (ncu, profiles/r01_ncu_full_summary.csv); two bodies (one per residual
            // prefetch buffer) stay hot in the instruction cache.
            auto chunk = [&](const int it, uint4(&resb)[4]) {
                const int c = CH_STEP * it + ch0;
                if (c >= NCH) return;
                const int nacc0 = n0 + c * ACC_PER_CHUNK;
                if (nacc0 >= p.N) return;
                uint32_t outp[16];
                if constexpr (EPI == OMG_EPI_GEGLU) {
                    uint32_t r0[32], r1[32];
                    tmem_ld_32x32(t_row + c * 64, r0);
                    tmem_ld_32x32(t_row + c * 64 + 32, r1);
                    tc_wait_ld();
                    const float* sb = sbias + c * 64;
                    const float* sc = sc1 + c * 64;
                    auto pair_out = [&](const uint32_t(&r)[32], int off, int i) {
                        float a, g;
                        if (ln) {
                            a = fmaf(ln_a, __uint_as_float(r[i]), fmaf(ln_k, sc[off + i], sb[off + i]));
                            g = fmaf(ln_a, __uint_as_float(r[i + 1]), fmaf(ln_k, sc[off + i + 1], sb[off + i + 1]));
                        } else {
                            a = __uint_as_float(r[i]) + sb[off + i];
                            g = __uint_as_float(r[i + 1]) + sb[off + i + 1];
                        }
                        return a * gelu_exact(g);
                    };
#pragma unroll
                    for (int j = 0; j < 8; ++j)  // columns (4j, 4j+1) and (4j+2, 4j+3) are (value, gate) pairs
                        outp[j] = pack2<T>(pair_out(r0, 0, 4 * j), pair_out(r0, 0, 4 * j + 2));
#pragma unroll
                    for (int j = 0; j < 8; ++j)
                        outp[8 + j] = pack2<T>(pair_out(r1, 32, 4 * j), pair_out(r1, 32, 4 * j + 2));
                } else {
                    uint32_t r[32];
                    tmem_ld_32x32(t_row + c * 32, r);
                    tc_wait_ld();
                    const float* sb = sbias + c * 32;
                    float v[32];
                    if (ln) {
                        const float* sc = sc1 + c * 32;
#pragma unroll
                        for (int j = 0; j < 32; ++j) v[j] = fmaf(ln_a, __uint_as_float(r[j]), fmaf(ln_k, sc[j], sb[j]));
                    } else {
#pragma unroll
                        for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]) + sb[j];
                    }
                    if constexpr (kExtra) {
                        if (p.act_silu == 1) {
    #pragma unroll
                            for (int j = 0; j < 32; ++j) v[j] = v[j] / (1.0f + __expf(-v[j]));
                        } else if (p.act_silu == 2) {  // quick_gelu
    #pragma unroll
                            for (int j = 0; j < 32; ++j) v[j] = v[j] / (1.0f + __expf(-1.702f * v[j]));
                        } else if (p.act_silu == 3) {  // erf-gelu
    #pragma unroll
                            for (int j = 0; j < 32; ++j) v[j] = gelu_exact(v[j]);
                        } else if (p.act_silu == 4) {  // tanh-gelu (EfficientViT-SAM): 0.5 x (1 + tanh(sqrt(2/pi)(x + 0.044715 x^3)))
    #pragma unroll
                            for (int j = 0; j < 32; ++j) {
                                const float u = 0.7978845608028654f * fmaf(0.044715f * v[j] * v[j], v[j], v[j]);
                                v[j] = 0.5f * v[j] * (2.0f - __fdividef(2.0f, 1.0f + __expf(2.0f * u)));
                            }
                        }
                    }
                    if (has_res) {
#pragma unroll
                        for (int j4 = 0; j4 < 4; ++j4) {
                            const uint4 u = resb[j4];
                            const T2* h2 = reinterpret_cast<const T2*>(&u);
#pragma unroll
                            for (int t = 0; t < 4; ++t) {
                                const float2 f = to_float2(h2[t]);
                                v[j4 * 8 + 2 * t] += f.x;
                                v[j4 * 8 + 2 * t + 1] += f.y;
                            }
                        }
                        load_res(c + 2 * CH_STEP, resb);
                    }
                    if constexpr (kExtra) {
                    if (p.residual_f32 != nullptr && row_valid) {  // fp32 addend (prefetching it a chunk ahead was measured: no gain)
                        const float4* rp = reinterpret_cast<const float4*>(p.residual_f32 + pix * (size_t)p.residual_f32_ld + nacc0);
#pragma unroll
                        for (int j4 = 0; j4 < 8; ++j4) {
                            const float4 f = __ldg(rp + j4);
                            v[j4 * 4] += f.x;
                            v[j4 * 4 + 1] += f.y;
                            v[j4 * 4 + 2] += f.z;
                            v[j4 * 4 + 3] += f.w;
                        }
                    }
                    if (p.out_f32 != nullptr && row_valid) {
                        float4* op = reinterpret_cast<float4*>(p.out_f32 + pix * (size_t)p.out_f32_ld + nacc0);
#pragma unroll
                        for (int j4 = 0; j4 < 8; ++j4) op[j4] = make_float4(v[j4 * 4], v[j4 * 4 + 1], v[j4 * 4 + 2], v[j4 * 4 + 3]);
                    }
                    }
                    if (p.stats_out != nullptr) {
                        if (nacc0 + 32 <= p.N) {
#pragma unroll
                            for (int j = 0; j < 32; ++j) {
                                row_sum += v[j];
                                row_sq = fmaf(v[j], v[j], row_sq);
                            }
                        } else {
#pragma unroll
                            for (int j = 0; j < 32; ++j) {
                                if (nacc0 + j < p.N) {
                                    row_sum += v[j];
                                    row_sq = fmaf(v[j], v[j], row_sq);
                                }
                            }
                        }
                    }
#pragma unroll
                    for (int j = 0; j < 16; ++j) outp[j] = pack2<T>(v[2 * j], v[2 * j + 1]);
                }
                if constexpr (EPI != OMG_EPI_GEGLU && kStats) {
                    if (p.col_stats != nullptr && !row_valid) {  // rows outside the image count as zeros
#pragma unroll
                        for (int j = 0; j < 16; ++j) outp[j] = 0u;
                    }
                }
                // this warp's staging buffer was last read by the TMA store of its previous chunk
                if (lane == 0) tma_store_wait_read<0>();
                __syncwarp();
                // 64 B rows, SWIZZLE_64B: 16 B chunk j of row r lives at chunk j ^ ((r >> 1) & 3)
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int pj = j ^ ((lane >> 1) & 3);
                    *reinterpret_cast<uint4*>(sbuf + lane * 64 + pj * 16) =
                        make_uint4(outp[4 * j], outp[4 * j + 1], outp[4 * j + 2], outp[4 * j + 3]);
                }
                fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) {
                    const int nout0 = (EPI == OMG_EPI_GEGLU) ? (nacc0 >> 1) : nacc0;
                    tma_store_4d(&p.d_map, sbuf, nout0, sw, sh, b);
                    tma_store_commit();
                }
                if constexpr (EPI != OMG_EPI_GEGLU && kStats) {
                    if (p.col_stats != nullptr && b < p.img_b) {
                        // per-channel (sum, sumsq) of the 32 rows x 32 channels just staged (the fp16-rounded values the
                        // consumer GroupNorm will see): lane = (row parity, channel pair); 16 conflict-free LDS.32
                        const int cp = lane & 15, hp = lane >> 4;
                        float s0 = 0.f, q0 = 0.f, s1 = 0.f, q1 = 0.f;
#pragma unroll
                        for (int i = 0; i < 16; ++i) {
                            const int r = 2 * i + hp;
                            const T2 h2 = *reinterpret_cast<const T2*>(
                                sbuf + r * 64 + (((cp >> 2) ^ (i & 3)) << 4) + ((cp & 3) << 2));
                            const float2 f = to_float2(h2);
                            s0 += f.x;
                            q0 = fmaf(f.x, f.x, q0);
                            s1 += f.y;
                            q1 = fmaf(f.y, f.y, q1);
                        }
                        s0 += __shfl_xor_sync(0xffffffffu, s0, 16);
                        q0 += __shfl_xor_sync(0xffffffffu, q0, 16);
                        s1 += __shfl_xor_sync(0xffffffffu, s1, 16);
                        q1 += __shfl_xor_sync(0xffffffffu, q1, 16);
                        const int col = nacc0 + 2 * cp;
                        if (hp == 0 && col < p.N) {
                            const size_t rb = (size_t)b * p.cs_rb_total + p.cs_rb0 + (size_t)rem * 4 + q;
                            p.col_stats[(rb * p.N + col) >> 1] = make_float4(s0, q0, s1, q1);
                        }
                    }
                }
            };
#pragma unroll 1
            for (int it = 0; it < NIT; it += 2) {
                chunk(it, res[0]);
                if (it + 1 < NIT) chunk(it + 1, res[1]);
            }
            if (p.stats_out != nullptr && row_valid) {  // two partial planes per n-tile
                float2* so = reinterpret_cast<float2*>(p.stats_out);
                if constexpr (MT == 2) {  // this thread covered the whole row of its sub-tile
                    so[(size_t)(n_tile * 2) * p.stats_rows + pix] = make_float2(row_sum, row_sq);
                    so[(size_t)(n_tile * 2 + 1) * p.stats_rows + pix] = make_float2(0.f, 0.f);
                } else if constexpr (BN > 256) {  // same plane count as two 160-wide tiles (what omg_gemm_plan promised)
                    so[(size_t)(n_tile * 4 + half) * p.stats_rows + pix] = make_float2(row_sum, row_sq);
                    so[(size_t)(n_tile * 4 + 2 + half) * p.stats_rows + pix] = make_float2(0.f, 0.f);
                } else {
                    so[(size_t)(n_tile * 2 + half) * p.stats_rows + pix] = make_float2(row_sum, row_sq);
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) {
                if (leader) mbar_arrive(&tempty_bar[acc]);
                else mbar_arrive_remote(&tempty_bar[acc], 0);  // the pair's MMA issuer lives in the leader CTA
            }
            if (++acc == Cfg::ACC_STAGES) {
                acc = 0;
                acc_phase ^= 1;
            }
        }
        // the staging buffers must stay intact until the bulk stores have READ them; their global writes complete
        // before the grid does (kernel-boundary ordering), so nothing waits for them here
        if (lane == 0) tma_store_wait_read<0>();
    }

    tc_fence_before();
    if constexpr (CTAS == 2) {
        cluster_sync();  // the peer may still arrive on / multicast into this CTA's barriers
        if (warp == 1) tmem_dealloc_pair(tmem_base, Cfg::TMEM_COLS);
    } else {
        __syncthreads();
        if (warp == 1) tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
    }
}

// ------------------------------------------------------------------------------------------------ host
static int view_to_tmap(CUtensorMap* m, const omg_view4& v, uint32_t box_c, uint32_t box_w, uint32_t box_h,
                        CUtensorMapSwizzle sw, CUtensorMapDataType dt) {
    const uint64_t dims[4] = {(uint64_t)v.C, (uint64_t)v.W, (uint64_t)v.H, (uint64_t)v.B};
    const uint64_t strides[4] = {1, (uint64_t)v.sw, (uint64_t)v.sh, (uint64_t)v.sb};
    const uint32_t box[4] = {box_c, box_w, box_h, 1};
    return make_tmap_16b(m, v.ptr, 4, dims, strides, box, sw, dt);
}

template <int BN, int EPI, int CTAS, int MT, int FEAT, typename T = __half>
static int launch_gemm_f(const GemmParams& p, cudaStream_t stream) {
    using Cfg = GemmCfg<BN, CTAS, MT>;
    static bool configured = false;
    static int num_sms = 0;
    if (!configured) {
        OMG_CUDA(cudaFuncSetAttribute(gemm_tc_kernel<BN, EPI, CTAS, MT, FEAT, T>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      Cfg::SMEM_BYTES));
        int dev = 0;
        OMG_CUDA(cudaGetDevice(&dev));
        OMG_CUDA(cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev));
        configured = true;
    }
    const int units = ((p.m_tiles + CTAS * MT - 1) / (CTAS * MT)) * p.n_tiles;
    const int grid = CTAS * std::min(units, num_sms / CTAS);
    OMG_CUDA(launch_cluster(gemm_tc_kernel<BN, EPI, CTAS, MT, FEAT, T>, dim3(grid), dim3(GEMM_THREADS), Cfg::SMEM_BYTES, stream, CTAS, p));
    return check_launch("gemm_tc_kernel");
}

// FEAT dispatch: 0 lean, 1 + GroupNorm column statistics, 2 + activations / fp32 twins (GEGLU launches are always lean).
// bf16 exists as the lean OMG_EPI_NONE variant only (gemm_impl rejects every other feature in bf16 mode): a larger
// epilogue cost the hot fp16 instantiations 3..17 %, and the VAE decoder needs none of it.
template <int BN, int EPI, int CTAS, int MT = 1, typename T = __half>
static int launch_gemm(const GemmParams& p, cudaStream_t stream) {
    if constexpr (std::is_same<T, __nv_bfloat16>::value) {
        static_assert(EPI == OMG_EPI_NONE, "bf16 GEMMs have no activation epilogue");
        return launch_gemm_f<BN, EPI, CTAS, MT, 0, T>(p, stream);
    } else if constexpr (EPI == OMG_EPI_GEGLU) {
        return launch_gemm_f<BN, EPI, CTAS, MT, 0>(p, stream);
    } else {
        if (p.act_silu != 0 || p.residual_f32 != nullptr || p.out_f32 != nullptr) return launch_gemm_f<BN, EPI, CTAS, MT, 2>(p, stream);
        if (p.col_stats != nullptr) return launch_gemm_f<BN, EPI, CTAS, MT, 1>(p, stream);
        return launch_gemm_f<BN, EPI, CTAS, MT, 0>(p, stream);
    }
}

static bool use_tall_tiles(long m_tiles, long n_tiles, long k_blocks) {
    if (m_tiles < 2 || k_blocks < 16) return false;
    const long t1 = m_tiles * n_tiles, t2 = ((m_tiles + 1) / 2) * n_tiles;
    const double e1 = (double)t1 / (double)(((t1 + 147) / 148) * 148);
    const double e2 = (double)t2 / (double)(((t2 + 147) / 148) * 148);
    return e2 * 1.20 >= e1;  // measured: a tall tile runs ~1.2x faster per row than two 128-row tiles
}

// CTA pairs pay off when the pair-tiles still fill the 74 SM pairs about as well as single tiles fill 148 SMs
static bool use_cta_pair(long m_tiles, long n_tiles, long k_blocks) {
    // measured (profiles/, kernel_bench): +5..9 % for K >= 1280 (ff1/ff2/qkv at c = 1280), -8 % for K = 640 where
    // the short mainloop cannot amortise the pair's cluster synchronisation and doubled epilogue per launch slot
    if (m_tiles < 2 || k_blocks < 16) return false;
    const long t1 = m_tiles * n_tiles, t2 = ((m_tiles + 1) / 2) * n_tiles;
    const double e1 = (double)t1 / (double)(((t1 + 147) / 148) * 148);
    const double e2 = (double)t2 / (double)(((t2 + 73) / 74) * 74);
    return e2 * 1.12 >= e1;
}

// k_plan: K blocks the choice is made for; k_blocks: K blocks of this launch.  Row-statistics producers of one consumer
// must all emit the same number of partials (= 2 * n_tiles), so they - and omg_gemm_plan - choose with k_plan = "long"
// whatever their own K; whether a 160-wide choice then runs as tall or as 128-row tiles does not change n_tiles.
constexpr long K_PLAN_LONG = 1000;
static int pick_block_n(int N, int epilogue, long m_tiles, long k_plan, long k_blocks, bool* prefer_tall) {
    if (prefer_tall) *prefer_tall = false;
    if (epilogue == OMG_EPI_GEGLU) return 256;
    // time ~ waves * per-tile cost.  Per-tile costs are empirical (kernel_bench on B200, profiles/): narrow tiles
    // re-read the A tile from shared memory once per BN columns, so cost per column rises as BN shrinks; a tall
    // (256 x 160) tile costs ~1.2x less than two 128 x 160 tiles.
    const int cands[5] = {256, 160, 128, 64, 160};
    const double cost[5] = {256.0, 200.0, 175.0, 110.0, 333.0};
    int best = 256;
    double best_t = 1e30;
    for (int i = 0; i < 5; ++i) {
        const bool tall = i == 4;
        if (tall && (k_plan < 16 || m_tiles < 2)) continue;
        const long nt = (N + cands[i] - 1) / cands[i];
        const long mt = tall ? (m_tiles + 1) / 2 : m_tiles;
        const long waves = (nt * mt + 147) / 148;
        double t = (double)waves * cost[i];
        if (i == 0 && k_plan >= 16 && m_tiles >= 2) t /= 1.07;  // CTA pairs (measured +5..9 %)
        if (t < best_t - 1e-9) {
            best_t = t;
            best = cands[i];
            if (prefer_tall) *prefer_tall = tall && k_blocks >= 16;
        }
    }
    return best;
}

// the non-GEGLU tile shapes: CTA pairs (block_n 160 | 256 | 320), tall 256 x 160 tiles, single 128 x block_n tiles
template <typename T>
static int launch_tiles(const GemmParams& p, int bn, bool pair, bool tall, cudaStream_t stream) {
    if (pair) {
        if (bn == 320) return launch_gemm<320, OMG_EPI_NONE, 2, 1, T>(p, stream);
        if (bn == 160) return launch_gemm<160, OMG_EPI_NONE, 2, 1, T>(p, stream);
        return launch_gemm<256, OMG_EPI_NONE, 2, 1, T>(p, stream);
    }
    if (tall) return launch_gemm<160, OMG_EPI_NONE, 1, 2, T>(p, stream);
    switch (bn) {
        case 64: return launch_gemm<64, OMG_EPI_NONE, 1, 1, T>(p, stream);
        case 128: return launch_gemm<128, OMG_EPI_NONE, 1, 1, T>(p, stream);
        case 160: return launch_gemm<160, OMG_EPI_NONE, 1, 1, T>(p, stream);
        default: return launch_gemm<256, OMG_EPI_NONE, 1, 1, T>(p, stream);
    }
}

}  // namespace omg

using namespace omg;

extern "C" int omg_gemm_plan(int N, int epilogue, int W, int H, int B, int* block_n, int* n_tiles) {
    OMG_CHECK(N >= 8 && W >= 1 && H >= 1 && B >= 1, "omg_gemm_plan: bad arguments");
    int tw = 128;
    while (tw / 2 >= W && tw > 1) tw /= 2;
    const int th = 128 / tw;
    const long m_tiles = (long)((W + tw - 1) / tw) * ((H + th - 1) / th) * B;
    const int bn = pick_block_n(N, epilogue, m_tiles, K_PLAN_LONG, 0, nullptr);
    if (block_n) *block_n = bn;
    if (n_tiles) *n_tiles = 2 * ((N + bn - 1) / bn);  // row-statistics partials: one per (n-tile, chunk parity)
    return 0;
}

extern "C" int omg_gemm_colstats_blocks(int W, int H) {
    if (W < 1 || H < 1) return 0;
    int tw = 128;
    while (tw / 2 >= W && tw > 1) tw /= 2;
    const int th = 128 / tw;
    return ((W + tw - 1) / tw) * ((H + th - 1) / th) * 4;
}

static int gemm_impl(const omg_gemm_desc* d, void* stream_) {
    cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
    OMG_CHECK(d != nullptr, "omg_gemm: null descriptor");
    OMG_CHECK(d->dtype == OMG_DTYPE_F16 || d->dtype == OMG_DTYPE_BF16, "omg_gemm: unknown dtype %d", d->dtype);
    const bool bf16 = d->dtype == OMG_DTYPE_BF16;
    if (bf16) {  // exactly what the VAE decoder uses; see launch_gemm
        OMG_CHECK(d->epilogue == OMG_EPI_NONE, "omg_gemm: bf16 supports no epilogue activation (GEGLU, SiLU, GELU): epilogue %d",
                  d->epilogue);
        OMG_CHECK(!d->row_stats_out && !d->row_stats_in, "omg_gemm: bf16 does not support the folded LayerNorm (row_stats_*)");
        OMG_CHECK(!d->col_stats_out, "omg_gemm: bf16 does not support col_stats_out");
        OMG_CHECK(!d->rowvec, "omg_gemm: bf16 does not support rowvec");
        OMG_CHECK(d->w_group_planes == 0 && d->n_col_groups <= 1, "omg_gemm: bf16 does not support weight planes or column groups");
        OMG_CHECK(!d->residual_f32 && !d->out_f32, "omg_gemm: bf16 does not support the fp32 twins (residual_f32 / out_f32)");
    }
    const CUtensorMapDataType dt = bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
    OMG_CHECK(d->n_a >= 1 && d->n_a <= OMG_MAX_A, "omg_gemm: n_a=%d out of range", d->n_a);
    OMG_CHECK(d->n_segs >= 1 && d->n_segs <= OMG_MAX_SEGS, "omg_gemm: n_segs=%d out of range", d->n_segs);
    OMG_CHECK(d->w && d->d.ptr, "omg_gemm: null weight/output pointer");
    OMG_CHECK(d->N >= 8 && d->N % 8 == 0, "omg_gemm: N=%d must be a positive multiple of 8", d->N);
    OMG_CHECK(d->Ktot % 8 == 0, "omg_gemm: Ktot=%d must be a multiple of 8", d->Ktot);
    const bool geglu = d->epilogue == OMG_EPI_GEGLU;
    const bool silu = d->epilogue == OMG_EPI_SILU;
    const int act = silu ? 1 : (d->epilogue == OMG_EPI_QUICK_GELU ? 2 : (d->epilogue == OMG_EPI_GELU ? 3 : (d->epilogue == OMG_EPI_GELU_TANH ? 4 : 0)));
    OMG_CHECK(d->epilogue == OMG_EPI_NONE || geglu || act, "omg_gemm: unknown epilogue %d", d->epilogue);
    const int N_out = geglu ? d->N / 2 : d->N;
    OMG_CHECK(d->d.C == N_out, "omg_gemm: output view has %d channels, expected %d", d->d.C, N_out);
    OMG_CHECK(!geglu || (d->N % 64 == 0 && !d->residual && !d->rowvec),
              "omg_gemm: GEGLU needs N %% 64 == 0 and no residual/rowvec");
    OMG_CHECK(!d->residual || (N_out % 32 == 0 && d->residual_ld % 8 == 0),
              "omg_gemm: residual needs N %% 32 == 0 and ld %% 8 == 0");

    GemmParams p;
    memset(&p, 0, sizeof(p));
    const int W = d->d.W, H = d->d.H, B = d->d.B;
    OMG_CHECK(W >= 1 && H >= 1 && B >= 1, "omg_gemm: empty output grid");
    int tw = 128;
    while (tw / 2 >= W && tw > 1) tw /= 2;  // smallest power of two >= W, capped at 128
    const int th = 128 / tw;
    p.tw = tw;
    p.th = th;
    p.tiles_w = (W + tw - 1) / tw;
    p.tiles_h = (H + th - 1) / th;
    p.store_w = std::min(tw, 32);
    p.store_h = 32 / p.store_w;
    p.img_w = W;
    p.img_h = H;
    p.img_b = B;
    p.m_tiles = p.tiles_w * p.tiles_h * B;
    p.N = d->N;
    p.N_out = N_out;
    bool prefer_tall = false;
    const long k_blocks_hint = (long)(d->Ktot + (d->w2 ? d->K2tot : 0)) / 64;
    int bn = d->block_n ? d->block_n
                        : pick_block_n(d->N, d->epilogue, p.m_tiles, d->row_stats_out ? K_PLAN_LONG : k_blocks_hint,
                                       k_blocks_hint, &prefer_tall);
    // block_n = 320 (256 x 320 CTA-pair tiles, two N = 160 MMAs per K step) is available on request and through
    // OMG_GEMM_320=1 (every 160-wide choice that allows it); never chosen by default: measured equal to the tall 256 x 160
    // tiles on the linears and 4-7 % slower on the convs (profiles/r02_gemm_tile_ab.jsonl) although it moves a third fewer
    // operand bytes per MMA cycle - these mainloops are not bound by the L2 -> shared-memory bandwidth.
    static int allow_320 = -1;
    if (allow_320 < 0) {
        const char* e = getenv("OMG_GEMM_320");
        allow_320 = (e && atoi(e) == 1) ? 1 : 0;
    }
    if (allow_320) {
        bool pair_ok0 = true;
        for (int i = 0; i + 1 < (d->n_col_groups > 0 ? d->n_col_groups : 1); ++i) pair_ok0 = pair_ok0 && (d->col_group_end[i] % 256 == 0);
        if (!d->block_n && d->cta_pair == 0 && bn == 160 && !geglu && d->N % 320 == 0 && pair_ok0 && p.m_tiles >= 2 &&
            k_blocks_hint >= 8)
            bn = 320;
    }
    OMG_CHECK(bn == 64 || bn == 128 || bn == 160 || bn == 256 || bn == 320, "omg_gemm: block_n=%d unsupported", bn);
    OMG_CHECK(bn != 320 || (!geglu && d->N % 320 == 0), "omg_gemm: block_n=320 needs N %% 320 == 0 and no GEGLU");
    if (geglu) bn = 256;
    p.n_tiles = (d->N + bn - 1) / bn;
    p.bias = d->bias;
    p.rowvec = d->rowvec;
    p.rowvec_ld = d->rowvec_ld;
    p.residual = d->residual;
    p.residual_ld = d->residual_ld;
    p.act_silu = act;  // 0 none, 1 SiLU, 2 quick_gelu, 3 erf-gelu, 4 tanh-gelu
    p.stats_out = static_cast<float*>(d->row_stats_out);
    p.stats_in = static_cast<const float*>(d->row_stats_in);
    p.stats_parts = d->row_stats_parts;
    p.stats_rows = d->row_stats_stride > 0 ? d->row_stats_stride : (long long)W * H * B;
    p.ln_inv_dim = d->ln_dim > 0 ? 1.0f / (float)d->ln_dim : 0.f;
    p.ln_eps = d->ln_eps;
    p.col_c1 = static_cast<const float*>(d->col_c1);
    p.col_c2 = static_cast<const float*>(d->col_c2);
    p.n_col_groups = d->n_col_groups > 0 ? d->n_col_groups : 1;
    p.w_group_rows = d->w_group_planes > 0 ? d->N : 0;
    OMG_CHECK(d->w_group_planes == 0 || d->w_group_planes == p.n_col_groups, "omg_gemm: w_group_planes must equal n_col_groups");
    OMG_CHECK(p.n_col_groups <= 8, "omg_gemm: at most 8 column-vector row groups");
    for (int i = 0; i < 8; ++i) {
        p.col_group_end[i] = d->col_group_end[i];
        OMG_CHECK(i + 1 >= p.n_col_groups || d->col_group_end[i] % 128 == 0,
                  "omg_gemm: row-group boundary %lld is not a multiple of the 128-row tile", (long long)d->col_group_end[i]);
    }
    OMG_CHECK(!p.stats_in || (p.col_c1 && p.col_c2 && d->ln_dim > 0 && d->row_stats_parts >= 1 && !d->rowvec),
              "omg_gemm: folded LayerNorm needs col_c1, col_c2, ln_dim, row_stats_parts and no rowvec");
    OMG_CHECK(!p.stats_out || !geglu, "omg_gemm: row statistics cannot be emitted by the GEGLU epilogue");
    p.residual_f32 = static_cast<const float*>(d->residual_f32);
    p.residual_f32_ld = d->residual_f32_ld;
    p.out_f32 = static_cast<float*>(d->out_f32);
    p.out_f32_ld = d->out_f32_ld;
    OMG_CHECK((!p.residual_f32 && !p.out_f32) || (!geglu && d->N % 32 == 0 && !(d->residual && d->residual_f32)),
              "omg_gemm: fp32 residual / output twins need a non-GEGLU epilogue, N %% 32 == 0, and replace the fp16 residual");
    OMG_CHECK((!p.residual_f32 || d->residual_f32_ld % 4 == 0) && (!p.out_f32 || d->out_f32_ld % 4 == 0),
              "omg_gemm: fp32 twin row strides must be multiples of 4");
    OMG_CHECK((!p.residual_f32 && !p.out_f32) || (d->d.sw == d->d.C && d->d.sh == (int64_t)d->d.sw * W && d->d.sb == d->d.sh * H),
              "omg_gemm: fp32 twins need a contiguous output view (rows are indexed by pixel)");
    p.col_stats = static_cast<float4*>(d->col_stats_out);
    p.cs_rb0 = d->col_stats_rb0;
    p.cs_rb_total = d->col_stats_rb_total;
    OMG_CHECK(!p.col_stats || (!geglu && d->N % 32 == 0 && d->col_stats_rb0 >= 0 &&
                               d->col_stats_rb0 + p.tiles_w * p.tiles_h * 4 <= d->col_stats_rb_total),
              "omg_gemm: column statistics need a non-GEGLU epilogue, N %% 32 == 0 and rb0 + blocks <= rb_total");
    OMG_CHECK((!p.stats_out && !p.stats_in) || (d->d.sw == d->d.C && d->d.sh == (int64_t)d->d.sw * W && d->d.sb == d->d.sh * H),
              "omg_gemm: row statistics need a contiguous output view");

    for (int i = 0; i < d->n_a; ++i) {
        OMG_CHECK(d->a[i].ptr != nullptr, "omg_gemm: A view %d is null", i);
        if (view_to_tmap(&p.a_maps[i], d->a[i], BK, tw, th, CU_TENSOR_MAP_SWIZZLE_128B, dt)) return 1;
    }
    for (int i = d->n_a; i < OMG_MAX_A; ++i) p.a_maps[i] = p.a_maps[0];
    {
        const uint64_t planes = d->w_group_planes > 0 ? (uint64_t)d->w_group_planes : 1;
        const uint64_t dims[2] = {(uint64_t)d->Ktot, (uint64_t)d->N * planes};
        const uint64_t strides[2] = {1, (uint64_t)d->Ktot};
        const uint32_t box[2] = {BK, (uint32_t)std::min(bn, 256)};
        if (make_tmap_16b(&p.b_maps[0], d->w, 2, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B, dt)) return 1;
        p.b_maps[1] = p.b_maps[0];
    }
    if (d->w2 != nullptr) {
        OMG_CHECK(d->K2tot >= 8 && d->K2tot % 8 == 0, "omg_gemm: K2tot=%d must be a positive multiple of 8", d->K2tot);
        const uint64_t dims[2] = {(uint64_t)d->K2tot, (uint64_t)d->N};
        const uint64_t strides[2] = {1, (uint64_t)d->K2tot};
        const uint32_t box[2] = {BK, (uint32_t)std::min(bn, 256)};
        if (make_tmap_16b(&p.b_maps[1], d->w2, 2, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B, dt)) return 1;
    }
    if (view_to_tmap(&p.d_map, d->d, 32, p.store_w, p.store_h, CU_TENSOR_MAP_SWIZZLE_64B, dt)) return 1;

    p.n_segs = d->n_segs;
    for (int s = 0; s < d->n_segs; ++s) {
        const omg_seg& sg = d->segs[s];
        OMG_CHECK(sg.a_idx >= 0 && sg.a_idx < d->n_a, "omg_gemm: segment %d references A view %d", s, sg.a_idx);
        OMG_CHECK(sg.k_len > 0 && sg.a_c0 >= 0 && sg.b_k0 >= 0 && sg.a_c0 + sg.k_len <= d->a[sg.a_idx].C,
                  "omg_gemm: segment %d has a bad K range", s);
        OMG_CHECK(sg.b_idx == 0 || (sg.b_idx == 1 && d->w2 != nullptr), "omg_gemm: segment %d has a bad b_idx", s);
        const int ktot_s = sg.b_idx ? d->K2tot : d->Ktot;
        OMG_CHECK(sg.b_k0 + sg.k_len <= ktot_s, "omg_gemm: segment %d exceeds weight K (%d + %d > %d)", s, sg.b_k0,
                  sg.k_len, ktot_s);
        // A K-tail (k_len % 64 != 0) is only legal when the over-read of A is zero-filled, i.e. the segment ends
        // at the end of the A view's channel range.
        OMG_CHECK(sg.k_len % BK == 0 || sg.a_c0 + sg.k_len == d->a[sg.a_idx].C,
                  "omg_gemm: segment %d: K tail must end at the A view's last channel", s);
        p.segs[s] = SegDev{sg.a_idx, sg.dx, sg.dy, sg.a_c0, (sg.k_len + BK - 1) / BK, sg.b_k0, sg.b_idx};
    }

    // the TMA box of the weight tile is this CTA's slice: BN rows, or BN/2 for a CTA pair
    long k_blocks = 0;
    for (int i = 0; i < p.n_segs; ++i) k_blocks += p.segs[i].k_blocks;
    bool pair_ok = true;  // both CTAs of a pair must belong to the same stream
    for (int i = 0; i + 1 < p.n_col_groups; ++i) pair_ok = pair_ok && (p.col_group_end[i] % 256 == 0);
    // BN = 160 pairs are available on request but never chosen: measured 0..-8 % (profiles/r01_kernel_bench.json)
    OMG_CHECK(bn != 320 || (pair_ok && p.m_tiles >= 2 && d->cta_pair != 1 && d->cta_pair != 3),
              "omg_gemm: block_n=320 runs as CTA pairs only (>= 2 m-tiles, 256-row aligned stream boundaries)");
    const bool pair = bn == 320 || ((bn == 256 || (bn == 160 && !geglu)) && pair_ok &&
                      (d->cta_pair == 2 || (d->cta_pair == 0 && bn == 256 && use_cta_pair(p.m_tiles, p.n_tiles, k_blocks))));
    if (pair) {
        for (int i = 0; i < 2; ++i) {
            const void* wp = i == 0 ? d->w : d->w2;
            if (!wp) continue;
            const int kt = i == 0 ? d->Ktot : d->K2tot;
            const uint64_t planes = (i == 0 && d->w_group_planes > 0) ? (uint64_t)d->w_group_planes : 1;
            const uint64_t dims[2] = {(uint64_t)kt, (uint64_t)d->N * planes};
            const uint64_t strides[2] = {1, (uint64_t)kt};
            const uint32_t box[2] = {BK, (uint32_t)(bn == 320 ? 80 : bn / 2)};
            if (make_tmap_16b(&p.b_maps[i], wp, 2, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B, dt)) return 1;
        }
        if (!d->w2) p.b_maps[1] = p.b_maps[0];
        if (geglu) return launch_gemm<256, OMG_EPI_GEGLU, 2>(p, stream);
        return bf16 ? launch_tiles<__nv_bfloat16>(p, bn, true, false, stream) : launch_tiles<__half>(p, bn, true, false, stream);
    }
    // tall tiles (256 x 160 per CTA): the narrow-N, long-enough-K GEMMs whose 128 x 160 tiles are L2-latency bound
    const bool tall = bn == 160 && !geglu && pair_ok &&
                      (d->cta_pair == 3 ||
                       (d->cta_pair == 0 && (prefer_tall || use_tall_tiles(p.m_tiles, p.n_tiles, k_blocks))));
    if (geglu) return launch_gemm<256, OMG_EPI_GEGLU, 1>(p, stream);
    return bf16 ? launch_tiles<__nv_bfloat16>(p, bn, false, tall, stream) : launch_tiles<__half>(p, bn, false, tall, stream);
}

// C-ABI entry points: launch, and - while this thread records a launch plan (omg_plan_record_begin) - remember the call
extern "C" int omg_gemm(const omg_gemm_desc* d, void* stream_) {
    const int rc = gemm_impl(d, stream_);
    if (rc == 0 && ::omg::plan_recording()) {
        const omg_gemm_desc c = *d;  // by value: a plan outlives the caller's descriptor
        ::omg::plan_note([c](void* s) { return gemm_impl(&c, s); });
    }
    return rc;
}
