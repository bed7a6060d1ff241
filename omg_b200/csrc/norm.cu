// GroupNorm(32) [+SiLU] and LayerNorm over channels-last fp16 activations.  HBM-bound: each element is read
// twice (statistics, apply) and written once; algorithmic bytes per launch pair = 3 * B*HW*C * 2 B.
//
// GroupNorm reads from up to two sources that are concatenated along channels (the UNet decoder's
// cat([hidden, skip], dim=1), diffusers UNet2DConditionModel up-blocks [3P]); the concatenation is never
// materialised un-normalised: the apply pass writes the normalised, activated, concatenated tensor that the
// following conv consumes through TMA.
//
// The normalising GroupNorm (omg_groupnorm) also exists for bf16 activations (omg_groupnorm_bf16, the VAE decoder with
// weights that overflow fp16); the statistics are fp32 sums in both cases.
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <type_traits>

#include "../../include/omg_b200.h"
#include "host_common.h"
#include "ptx.cuh"

namespace omg {

template <typename T = __half>
struct GnSrc {
    const T* x1;
    const T* x2;
    int C1, C2;  // channels of each source (C2 = 0 when unused); both multiples of 8
};

template <typename T>
__device__ __forceinline__ uint4 gn_load8(const GnSrc<T>& s, size_t pix, int c) {
    // c is a multiple of 8 and an 8-vector never straddles the two sources
    if (c < s.C1) return *reinterpret_cast<const uint4*>(s.x1 + pix * s.C1 + c);
    return *reinterpret_cast<const uint4*>(s.x2 + pix * s.C2 + (c - s.C1));
}

// Deterministic (atomic-free, batch-invariant) statistics:
//   pass 1  partial[b][split][g] = {sum, sumsq} over the CTA's rows    grid = (splits, B), block = (C/8, rows_par)
//   pass 2  stats[b][g] = {mean, rstd}, partials summed in split order  grid = B, block = 32
// Identical images in a batch therefore get bit-identical results (the reference's stage-1 rows are identical).
template <typename T>
__global__ void gn_partial_kernel(GnSrc<T> s, int HW, int cpg, int rows_per_cta, float* __restrict__ partial) {
    extern __shared__ float s_red[];  // [rows_par][C] sums, then [rows_par][C] squares
    griddep_launch_dependents();
    griddep_wait();
    const int C = s.C1 + s.C2;
    const int b = blockIdx.y;
    const int c = threadIdx.x * 8;
    const int r0 = blockIdx.x * rows_per_cta;
    const int r1 = min(r0 + rows_per_cta, HW);
    float a[8], q[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) a[i] = q[i] = 0.f;
    auto acc8 = [&](const uint4& u) {
        const auto* h2 = reinterpret_cast<const typename Pair<T>::type*>(&u);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float2 f = to_float2(h2[i]);
            a[2 * i] += f.x;
            q[2 * i] += f.x * f.x;
            a[2 * i + 1] += f.y;
            q[2 * i + 1] += f.y * f.y;
        }
    };
    int r = r0 + threadIdx.y;
    const int step = blockDim.y;
    for (; r + 3 * step < r1; r += 4 * step) {  // four independent 16 B loads in flight per thread
        const uint4 u0 = gn_load8(s, (size_t)b * HW + r, c);
        const uint4 u1 = gn_load8(s, (size_t)b * HW + r + step, c);
        const uint4 u2 = gn_load8(s, (size_t)b * HW + r + 2 * step, c);
        const uint4 u3 = gn_load8(s, (size_t)b * HW + r + 3 * step, c);
        acc8(u0);
        acc8(u1);
        acc8(u2);
        acc8(u3);
    }
    for (; r < r1; r += step) acc8(gn_load8(s, (size_t)b * HW + r, c));
    float* s_sum = s_red;
    float* s_sq = s_red + blockDim.y * C;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        s_sum[threadIdx.y * C + c + i] = a[i];
        s_sq[threadIdx.y * C + c + i] = q[i];
    }
    __syncthreads();
    if (threadIdx.y == 0) {  // fold the row-parallel copies in a fixed order
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            float sa = a[i], sq = q[i];
            for (int y = 1; y < blockDim.y; ++y) {
                sa += s_sum[y * C + c + i];
                sq += s_sq[y * C + c + i];
            }
            s_sum[c + i] = sa;
            s_sq[c + i] = sq;
        }
    }
    __syncthreads();
    const int tid = threadIdx.y * blockDim.x + threadIdx.x;
    if (tid < 32) {
        float sa = 0.f, sq = 0.f;
        for (int k = 0; k < cpg; ++k) {
            sa += s_sum[tid * cpg + k];
            sq += s_sq[tid * cpg + k];
        }
        float* o = partial + (((size_t)b * gridDim.x + blockIdx.x) * 32 + tid) * 2;
        o[0] = sa;
        o[1] = sq;
    }
}

// per-(image, channel) affine of the normalisation: y = a * x + b with a = rstd * gamma, b = beta - mean * a
template <typename T>
__device__ __forceinline__ void gn_write_affine(float2* __restrict__ ab, int b, int C, int g, int cpg, int k0, int kstep,
                                                float mean, float rstd, const T* __restrict__ gamma,
                                                const T* __restrict__ beta) {
    for (int k = k0; k < cpg; k += kstep) {
        const int c = g * cpg + k;
        const float a = rstd * to_float(gamma[c]);
        ab[(size_t)b * C + c] = make_float2(a, to_float(beta[c]) - mean * a);
    }
}

template <typename T>
__global__ void gn_finalize_kernel(const float* __restrict__ partial, int splits, float inv_n, float eps,
                                   float2* __restrict__ ab, int C, int cpg, const T* __restrict__ gamma,
                                   const T* __restrict__ beta) {
    const int b = blockIdx.x, g = threadIdx.x >> 5, lane = threadIdx.x & 31;  // block = 32 groups x 32 lanes
    griddep_launch_dependents();
    griddep_wait();
    float sa = 0.f, sq = 0.f;
    for (int k = lane; k < splits; k += 32) {
        const float2 p = *reinterpret_cast<const float2*>(partial + (((size_t)b * splits + k) * 32 + g) * 2);
        sa += p.x;
        sq += p.y;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {  // fixed-order tree: deterministic
        sa += __shfl_xor_sync(0xffffffffu, sa, o);
        sq += __shfl_xor_sync(0xffffffffu, sq, o);
    }
    const float mean = sa * inv_n;  // every lane holds the totals after the butterfly
    const float rstd = rsqrtf(fmaxf(sq * inv_n - mean * mean, 0.f) + eps);
    gn_write_affine(ab, b, C, g, cpg, lane, 32, mean, rstd, gamma, beta);
}

// Apply pass: y = silu?(a[b, c] * x + b[b, c]).  block = (C/8 channel vectors, ry rows), grid = (row chunks, B): a thread
// keeps ONE channel vector for all of its rows, so the affine is loaded once into registers and there is no index
// arithmetic in the loop; four 16 B loads are in flight per thread, a warp's loads are contiguous runs of the row.
template <typename T>
__global__ void gn_apply_kernel(GnSrc<T> s, int HW, int rows_per_cta, int silu, const float2* __restrict__ ab,
                                T* __restrict__ y) {
    griddep_launch_dependents();
    griddep_wait();
    const int C = s.C1 + s.C2;
    const int b = blockIdx.y;
    const int c0 = threadIdx.x * 8;
    float a[8], sft[8];
    {
        const float4* p4 = reinterpret_cast<const float4*>(ab + (size_t)b * C + c0);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float4 v = __ldg(p4 + i);
            a[2 * i] = v.x;
            sft[2 * i] = v.y;
            a[2 * i + 1] = v.z;
            sft[2 * i + 1] = v.w;
        }
    }
    const int r0 = blockIdx.x * rows_per_cta;
    const int r1 = min(r0 + rows_per_cta, HW);
    const int step = blockDim.y;
    auto emit = [&](const uint4& u, int r) {
        const auto* h2 = reinterpret_cast<const typename Pair<T>::type*>(&u);
        float v[8];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float2 f = to_float2(h2[i]);
            v[2 * i] = fmaf(a[2 * i], f.x, sft[2 * i]);
            v[2 * i + 1] = fmaf(a[2 * i + 1], f.y, sft[2 * i + 1]);
        }
        if (silu) {
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] = __fdividef(v[i], 1.0f + __expf(-v[i]));
        }
        const uint4 o = make_uint4(pack2<T>(v[0], v[1]), pack2<T>(v[2], v[3]), pack2<T>(v[4], v[5]), pack2<T>(v[6], v[7]));
        *reinterpret_cast<uint4*>(y + ((size_t)b * HW + r) * C + c0) = o;
    };
    int r = r0 + threadIdx.y;
    for (; r + 3 * step < r1; r += 4 * step) {
        const uint4 u0 = gn_load8(s, (size_t)b * HW + r, c0);
        const uint4 u1 = gn_load8(s, (size_t)b * HW + r + step, c0);
        const uint4 u2 = gn_load8(s, (size_t)b * HW + r + 2 * step, c0);
        const uint4 u3 = gn_load8(s, (size_t)b * HW + r + 3 * step, c0);
        emit(u0, r);
        emit(u1, r + step);
        emit(u2, r + 2 * step);
        emit(u3, r + 3 * step);
    }
    for (; r < r1; r += step) emit(gn_load8(s, (size_t)b * HW + r, c0), r);
}

template <typename T>
static int launch_gn_apply(const GnSrc<T>& s, int B, int HW, int silu, const float2* ab, T* y, cudaStream_t stream) {
    const int C = s.C1 + s.C2;
    const int tx = C / 8;
    int ty = 512 / tx;
    if (ty < 1) ty = 1;
    if (ty > 16) ty = 16;
    // ~2 CTAs per SM slot at batch 4 (the row partition depends on (HW, C) only); at least 4 rows per thread
    int rows_per_cta = (HW + 63) / 64;
    if (rows_per_cta < 4 * ty) rows_per_cta = 4 * ty;
    const int chunks = (HW + rows_per_cta - 1) / rows_per_cta;
    OMG_CUDA(launch_pdl(gn_apply_kernel<T>, dim3(chunks, B), dim3(tx, ty), 0, stream, s, HW, rows_per_cta, silu, ab, y));
    return check_launch("gn_apply_kernel");
}

// ---------------------------------------------------------------------------------------------------------------------
// GroupNorm statistics from per-channel partials.  The producing GEMM / conv writes, per image and per 32-pixel block of
// its output, the per-channel (sum, sum of squares) of the fp16-rounded values (gemm_tc.cu epilogue); omg_colstats
// produces the same layout from a stored tensor.  gn_reduce_kernel turns them into (mean, rstd) per (image, group) for
// ANY grouping of the channel concatenation (x1 | x2) - a decoder GroupNorm's groups straddle the hidden / skip
// boundary - in a fixed summation order (deterministic, independent of the batch position).
struct GnParts {
    const float2* p1;
    const float2* p2;
    int C1, C2, rb1, rb2;
};

__global__ void gn_reduce_kernel(GnParts s, int cpg, float inv_n, float eps, float2* __restrict__ ab,
                                 const __half* __restrict__ gamma, const __half* __restrict__ beta) {
    griddep_launch_dependents();
    griddep_wait();
    const int g = blockIdx.x, b = blockIdx.y;
    const int c_lo = g * cpg, c_hi = c_lo + cpg;
    float sa[4] = {0.f, 0.f, 0.f, 0.f}, sq[4] = {0.f, 0.f, 0.f, 0.f};
    // thread = (channel of the group, slice of the 32-row blocks): four independent loads in flight per thread
    auto accumulate = [&](const float2* __restrict__ base, int n, int rb, int ld) {
        if (n <= 0) return;
        const int lanes = blockDim.x / n;           // row-block slices (>= 3 for cpg <= 80 and 256 threads)
        const int k = threadIdx.x % n, sl = threadIdx.x / n;
        if (sl >= lanes) return;
        int r = sl;
        for (; r + 3 * lanes < rb; r += 4 * lanes) {
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const float2 v = __ldg(base + (size_t)(r + u * lanes) * ld + k);
                sa[u] += v.x;
                sq[u] += v.y;
            }
        }
        for (; r < rb; r += lanes) {
            const float2 v = __ldg(base + (size_t)r * ld + k);
            sa[0] += v.x;
            sq[0] += v.y;
        }
    };
    {
        const int lo = min(c_lo, s.C1), hi = min(c_hi, s.C1);
        accumulate(s.p1 + (size_t)b * s.rb1 * s.C1 + lo, hi - lo, s.rb1, s.C1);
    }
    if (s.C2 > 0) {
        const int lo = max(c_lo, s.C1) - s.C1, hi = max(c_hi, s.C1) - s.C1;
        accumulate(s.p2 + (size_t)b * s.rb2 * s.C2 + lo, hi - lo, s.rb2, s.C2);
    }
    float a = (sa[0] + sa[1]) + (sa[2] + sa[3]), q = (sq[0] + sq[1]) + (sq[2] + sq[3]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        a += __shfl_xor_sync(0xffffffffu, a, o);
        q += __shfl_xor_sync(0xffffffffu, q, o);
    }
    __shared__ float2 red[8];
    __shared__ float2 mr;
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = make_float2(a, q);
    __syncthreads();
    if (threadIdx.x == 0) {
        float ta = 0.f, tq = 0.f;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) {  // fixed order: deterministic
            ta += red[w].x;
            tq += red[w].y;
        }
        const float mean = ta * inv_n;
        mr = make_float2(mean, rsqrtf(fmaxf(tq * inv_n - mean * mean, 0.f) + eps));
    }
    __syncthreads();
    gn_write_affine(ab, b, s.C1 + s.C2, g, cpg, threadIdx.x, blockDim.x, mr.x, mr.y, gamma, beta);
}

// grid = (ceil(ceil(HW/32) / 8), B), block = 256: one warp per 32-row block; lane = channel pair, strided over C
__global__ void colstats_kernel(const __half* __restrict__ x, int C, int HW, float2* __restrict__ out) {
    griddep_launch_dependents();
    griddep_wait();
    const int rbs = (HW + 31) / 32;
    const int rb = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (rb >= rbs) return;
    const int b = blockIdx.y, lane = threadIdx.x & 31;
    const int r0 = rb * 32, r1 = min(r0 + 32, HW);
    const __half* xb = x + ((size_t)b * HW) * C;
    for (int c = 2 * lane; c < C; c += 64) {
        float s0 = 0.f, q0 = 0.f, s1 = 0.f, q1 = 0.f;
        for (int r = r0; r < r1; ++r) {
            const float2 f = __half22float2(*reinterpret_cast<const __half2*>(xb + (size_t)r * C + c));
            s0 += f.x;
            q0 = fmaf(f.x, f.x, q0);
            s1 += f.y;
            q1 = fmaf(f.y, f.y, q1);
        }
        float4* o = reinterpret_cast<float4*>(out + ((size_t)b * rbs + rb) * C + c);
        *o = make_float4(s0, q0, s1, q1);
    }
}

// One warp per token row; exact two-pass variance held in registers (C <= 2560).
template <int MAX_VEC>
__global__ void layernorm_kernel(const __half* __restrict__ x, const __half* __restrict__ gamma,
                                 const __half* __restrict__ beta, __half* __restrict__ y, long long rows, int C,
                                 float eps) {
    griddep_launch_dependents();
    griddep_wait();
    const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= rows) return;
    const int lane = threadIdx.x & 31;
    const int nvec = C / 8;
    const uint4* xr = reinterpret_cast<const uint4*>(x + row * C);
    float v[MAX_VEC][8];
    float sum = 0.f;
#pragma unroll
    for (int k = 0; k < MAX_VEC; ++k) {
        const int vi = lane + k * 32;
        if (vi < nvec) {
            const uint4 u = xr[vi];
            const __half2* h2 = reinterpret_cast<const __half2*>(&u);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const float2 f = __half22float2(h2[i]);
                v[k][2 * i] = f.x;
                v[k][2 * i + 1] = f.y;
                sum += f.x + f.y;
            }
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    const float mean = sum / (float)C;
    float sq = 0.f;
#pragma unroll
    for (int k = 0; k < MAX_VEC; ++k) {
        const int vi = lane + k * 32;
        if (vi < nvec) {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const float d = v[k][i] - mean;
                sq += d * d;
            }
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
    const float rstd = rsqrtf(sq / (float)C + eps);
    uint4* yr = reinterpret_cast<uint4*>(y + row * C);
#pragma unroll
    for (int k = 0; k < MAX_VEC; ++k) {
        const int vi = lane + k * 32;
        if (vi < nvec) {
            const uint4 gw = reinterpret_cast<const uint4*>(gamma)[vi];
            const uint4 bw = reinterpret_cast<const uint4*>(beta)[vi];
            const __half2* g2 = reinterpret_cast<const __half2*>(&gw);
            const __half2* b2 = reinterpret_cast<const __half2*>(&bw);
            uint4 o;
            __half2* oh = reinterpret_cast<__half2*>(&o);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const float2 gf = __half22float2(g2[i]);
                const float2 bf = __half22float2(b2[i]);
                oh[i] = __floats2half2_rn((v[k][2 * i] - mean) * rstd * gf.x + bf.x,
                                          (v[k][2 * i + 1] - mean) * rstd * gf.y + bf.y);
            }
            yr[vi] = o;
        }
    }
}

}  // namespace omg

using namespace omg;

template <typename T>
static int groupnorm_impl(const void* x1, int C1, const void* x2, int C2, int B, int HW, const void* gamma,
                             const void* beta, float eps, int silu, void* stats_ws, void* y, void* stream_) {
    cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
    const int C = C1 + C2;
    const char* fn = std::is_same<T, __half>::value ? "omg_groupnorm" : "omg_groupnorm_bf16";
    OMG_CHECK(x1 && gamma && beta && stats_ws && y, "%s: null pointer", fn);
    OMG_CHECK(C1 > 0 && C1 % 8 == 0 && C2 >= 0 && C2 % 8 == 0 && (C2 == 0 || x2), "%s: bad channel split", fn);
    OMG_CHECK(C % 32 == 0 && C <= 2560, "%s: C=%d must be a multiple of 32 and <= 2560", fn, C);
    OMG_CHECK(B >= 1 && HW >= 1, "%s: empty input", fn);
    const int cpg = C / 32;
    GnSrc<T> s{static_cast<const T*>(x1), static_cast<const T*>(x2), C1, C2};
    const int tx = C / 8;
    int ty = 1024 / tx;
    if (ty > 16) ty = 16;
    if (ty < 1) ty = 1;
    // the row partition depends on (HW, C) only - never on the batch size - so an image's statistics are
    // bit-identical whatever batch it is processed in (grouped multi-stream forwards rely on this)
    int rows_per_cta = (HW + 63) / 64;
    if (rows_per_cta < 4 * ty) rows_per_cta = 4 * ty;
    int splits = (HW + rows_per_cta - 1) / rows_per_cta;
    if (splits > OMG_GN_MAX_SPLITS) {
        splits = OMG_GN_MAX_SPLITS;
        rows_per_cta = (HW + splits - 1) / splits;
        splits = (HW + rows_per_cta - 1) / rows_per_cta;
    }
    float2* ab = static_cast<float2*>(stats_ws);                              // [B][C] (a, b) of y = a x + b
    float* partial = static_cast<float*>(stats_ws) + (size_t)B * 2 * 2560;   // [B][splits][32][2]
    const size_t smem = (size_t)2 * ty * C * sizeof(float);
    static bool configured = false;
    if (!configured) {
        OMG_CUDA(cudaFuncSetAttribute(gn_partial_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * 8192 * 4));  // ty * C <= 1024 * 8
        configured = true;
    }
    OMG_CUDA(launch_pdl(gn_partial_kernel<T>, dim3(splits, B), dim3(tx, ty), smem, stream, s, HW, cpg, rows_per_cta, partial));
    if (check_launch("gn_partial_kernel")) return 1;
    OMG_CUDA(launch_pdl(gn_finalize_kernel<T>, dim3(B), dim3(1024), 0, stream, (const float*)partial, splits,
                        1.0f / ((float)HW * (float)cpg), eps, ab, C, cpg, static_cast<const T*>(gamma),
                        static_cast<const T*>(beta)));
    if (check_launch("gn_finalize_kernel")) return 1;
    return launch_gn_apply(s, B, HW, silu, ab, static_cast<T*>(y), stream);
}

static int colstats_impl(const void* x, int C, int B, int HW, void* out, void* stream_) {
    cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
    OMG_CHECK(x && out, "omg_colstats: null pointer");
    OMG_CHECK(C >= 8 && C % 8 == 0 && B >= 1 && HW >= 1, "omg_colstats: bad shape");
    const int rbs = (HW + 31) / 32;
    OMG_CUDA(launch_pdl(colstats_kernel, dim3((rbs + 7) / 8, B), dim3(256), 0, stream, static_cast<const __half*>(x), C, HW,
                        static_cast<float2*>(out)));
    return check_launch("colstats_kernel");
}

static int groupnorm_apply_impl(const void* x1, int C1, const void* part1, int rb1, const void* x2, int C2,
                                   const void* part2, int rb2, int B, int HW, const void* gamma, const void* beta, float eps,
                                   int silu, void* stats_ws, void* y, void* stream_) {
    cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
    const int C = C1 + C2;
    OMG_CHECK(x1 && part1 && gamma && beta && stats_ws && y, "omg_groupnorm_apply: null pointer");
    OMG_CHECK(C1 > 0 && C1 % 8 == 0 && C2 >= 0 && C2 % 8 == 0 && (C2 == 0 || (x2 && part2)), "omg_groupnorm_apply: bad channel split");
    OMG_CHECK(C % 32 == 0 && C <= 2560, "omg_groupnorm_apply: C=%d must be a multiple of 32 and <= 2560", C);
    OMG_CHECK(B >= 1 && HW >= 1 && rb1 >= 1 && (C2 == 0 || rb2 >= 1), "omg_groupnorm_apply: empty input");
    const int cpg = C / 32;
    GnSrc<> s{static_cast<const __half*>(x1), static_cast<const __half*>(x2), C1, C2};
    GnParts parts{static_cast<const float2*>(part1), static_cast<const float2*>(part2), C1, C2, rb1, rb2};
    float2* ab = static_cast<float2*>(stats_ws);  // [B][C] (a, b) of y = a x + b
    OMG_CUDA(launch_pdl(gn_reduce_kernel, dim3(32, B), dim3(256), 0, stream, parts, cpg, 1.0f / ((float)HW * (float)cpg), eps, ab,
                        static_cast<const __half*>(gamma), static_cast<const __half*>(beta)));
    if (check_launch("gn_reduce_kernel")) return 1;
    return launch_gn_apply(s, B, HW, silu, ab, static_cast<__half*>(y), stream);
}

static int layernorm_impl(const void* x, const void* gamma, const void* beta, void* y, long long rows, int C,
                             float eps, void* stream_) {
    cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
    OMG_CHECK(x && gamma && beta && y, "omg_layernorm: null pointer");
    OMG_CHECK(C % 8 == 0 && C >= 8 && C <= 2560, "omg_layernorm: C=%d unsupported", C);
    OMG_CHECK(rows >= 1, "omg_layernorm: empty input");
    const int warps = 8;
    const unsigned grid = (unsigned)((rows + warps - 1) / warps);
    const int nvec = C / 8;
    const __half* xp = static_cast<const __half*>(x);
    const __half* gp = static_cast<const __half*>(gamma);
    const __half* bp = static_cast<const __half*>(beta);
    __half* yp = static_cast<__half*>(y);
    if (nvec <= 96)
        OMG_CUDA(launch_pdl(layernorm_kernel<3>, dim3(grid), dim3(warps * 32), 0, stream, xp, gp, bp, yp, rows, C, eps));
    else if (nvec <= 160)
        OMG_CUDA(launch_pdl(layernorm_kernel<5>, dim3(grid), dim3(warps * 32), 0, stream, xp, gp, bp, yp, rows, C, eps));
    else
        OMG_CUDA(launch_pdl(layernorm_kernel<10>, dim3(grid), dim3(warps * 32), 0, stream, xp, gp, bp, yp, rows, C, eps));
    return check_launch("layernorm_kernel");
}

// C-ABI entry points: launch, and - while this thread records a launch plan (omg_plan_record_begin) - remember the call
extern "C" int omg_groupnorm(const void* x1, int C1, const void* x2, int C2, int B, int HW, const void* gamma,
                             const void* beta, float eps, int silu, void* stats_ws, void* y, void* stream_) {
    const int rc = groupnorm_impl<__half>(x1, C1, x2, C2, B, HW, gamma, beta, eps, silu, stats_ws, y, stream_);
    if (rc == 0 && ::omg::plan_recording()) ::omg::plan_note([=](void* s) { return groupnorm_impl<__half>(x1, C1, x2, C2, B, HW, gamma, beta, eps, silu, stats_ws, y, s); });
    return rc;
}

extern "C" int omg_groupnorm_bf16(const void* x1, int C1, const void* x2, int C2, int B, int HW, const void* gamma,
                                  const void* beta, float eps, int silu, void* stats_ws, void* y, void* stream_) {
    const int rc = groupnorm_impl<__nv_bfloat16>(x1, C1, x2, C2, B, HW, gamma, beta, eps, silu, stats_ws, y, stream_);
    if (rc == 0 && ::omg::plan_recording()) ::omg::plan_note([=](void* s) { return groupnorm_impl<__nv_bfloat16>(x1, C1, x2, C2, B, HW, gamma, beta, eps, silu, stats_ws, y, s); });
    return rc;
}

extern "C" int omg_colstats(const void* x, int C, int B, int HW, void* out, void* stream_) {
    const int rc = colstats_impl(x, C, B, HW, out, stream_);
    if (rc == 0 && ::omg::plan_recording()) ::omg::plan_note([=](void* s) { return colstats_impl(x, C, B, HW, out, s); });
    return rc;
}

extern "C" int omg_groupnorm_apply(const void* x1, int C1, const void* part1, int rb1, const void* x2, int C2,
                                   const void* part2, int rb2, int B, int HW, const void* gamma, const void* beta, float eps,
                                   int silu, void* stats_ws, void* y, void* stream_) {
    const int rc = groupnorm_apply_impl(x1, C1, part1, rb1, x2, C2, part2, rb2, B, HW, gamma, beta, eps, silu, stats_ws, y, stream_);
    if (rc == 0 && ::omg::plan_recording()) ::omg::plan_note([=](void* s) { return groupnorm_apply_impl(x1, C1, part1, rb1, x2, C2, part2, rb2, B, HW, gamma, beta, eps, silu, stats_ws, y, s); });
    return rc;
}

extern "C" int omg_layernorm(const void* x, const void* gamma, const void* beta, void* y, long long rows, int C,
                             float eps, void* stream_) {
    const int rc = layernorm_impl(x, gamma, beta, y, rows, C, eps, stream_);
    if (rc == 0 && ::omg::plan_recording()) ::omg::plan_note([=](void* s) { return layernorm_impl(x, gamma, beta, y, rows, C, eps, s); });
    return rc;
}
