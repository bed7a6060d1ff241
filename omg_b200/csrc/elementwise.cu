// HBM-bound element-wise kernels of the denoising step.
//
// omg_fuse_step: region noise fusion + classifier-free guidance + Euler step + next-step model inputs in ONE
// launch (reference: src/pipelines/lora_pipeline.py:568-615 does this with ~15 boolean-index kernels, each
// forcing a host sync through nonzero(); src/pipelines/instantid_pipeline.py:618-690 is identical).
// Algorithmic bytes per launch (HW latent pixels, n concepts): read (4 + 2n) * HW*8*2 B noise + n * HW*4 B masks
// + HW*2*4*4 B latents; write HW*2*4*4 B latents + 6 * HW*8*2 B next inputs.
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <type_traits>

#include "../../include/omg_b200.h"
#include "host_common.h"
#include "ptx.cuh"

namespace omg {

struct FuseParams {
    const __half* noise_main;                          // [4, HW, 8]  rows: uncond0, uncond1, cond0, cond1
    const __half* noise_concept[OMG_MAX_CONCEPTS];     // [2, HW, 8]  rows: uncond, cond
    const float* mask[OMG_MAX_CONCEPTS];               // [HW] in {0,1}
    int n_concepts;
    float guidance, sigma, sigma_next;
    float* latents;          // [2, HW, 4] fp32 state (image 0 = layout, image 1 = edited)
    __half* next_main_in;    // [4, HW, 8] = scale_model_input(cat([latents]*2)), channels 4..7 zero
    __half* next_concept_in; // [2, HW, 8] = scaled latent of image 1, twice
    __half* latents_f16;     // optional [2, HW, 4] fp16 copy of the new latents (pipeline output)
    int HW;
};

__device__ __forceinline__ void load4(const __half* p, float (&v)[4]) {
    const uint2 u = *reinterpret_cast<const uint2*>(p);
    const __half2* h = reinterpret_cast<const __half2*>(&u);
    const float2 a = __half22float2(h[0]), b = __half22float2(h[1]);
    v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
}

__global__ void fuse_step_kernel(FuseParams p) {
    griddep_launch_dependents();
    griddep_wait();
    const int pix = blockIdx.x * blockDim.x + threadIdx.x;
    if (pix >= p.HW) return;
    const size_t HW = p.HW;
    float u0[4], u1[4], c0[4], c1[4];
    load4(p.noise_main + (0 * HW + pix) * 8, u0);
    load4(p.noise_main + (1 * HW + pix) * 8, u1);
    load4(p.noise_main + (2 * HW + pix) * 8, c0);
    load4(p.noise_main + (3 * HW + pix) * 8, c1);
    if (p.n_concepts > 0) {
        // union mask zeroes the main prediction of image 1, every concept adds its own prediction inside its mask
        bool any = false;
        float au[4] = {0, 0, 0, 0}, ac[4] = {0, 0, 0, 0};
        for (int k = 0; k < p.n_concepts; ++k) {
            if (p.mask[k] == nullptr) continue;
            if (p.mask[k][pix] == 1.0f) {
                any = true;
                float ku[4], kc[4];
                load4(p.noise_concept[k] + (0 * HW + pix) * 8, ku);
                load4(p.noise_concept[k] + (1 * HW + pix) * 8, kc);
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    au[i] += ku[i];
                    ac[i] += kc[i];
                }
            }
        }
        if (any) {
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                u1[i] = au[i];
                c1[i] = ac[i];
            }
        }
    }
    const float dt = p.sigma_next - p.sigma;
    const float in_scale = rsqrtf(p.sigma_next * p.sigma_next + 1.0f);
    float4 l0 = *reinterpret_cast<float4*>(p.latents + (0 * HW + pix) * 4);
    float4 l1 = *reinterpret_cast<float4*>(p.latents + (1 * HW + pix) * 4);
    float e0[4], e1[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        e0[i] = u0[i] + p.guidance * (c0[i] - u0[i]);
        e1[i] = u1[i] + p.guidance * (c1[i] - u1[i]);
    }
    l0.x += e0[0] * dt; l0.y += e0[1] * dt; l0.z += e0[2] * dt; l0.w += e0[3] * dt;
    l1.x += e1[0] * dt; l1.y += e1[1] * dt; l1.z += e1[2] * dt; l1.w += e1[3] * dt;
    *reinterpret_cast<float4*>(p.latents + (0 * HW + pix) * 4) = l0;
    *reinterpret_cast<float4*>(p.latents + (1 * HW + pix) * 4) = l1;
    if (p.latents_f16) {
        __half2* o0 = reinterpret_cast<__half2*>(p.latents_f16 + (0 * HW + pix) * 4);
        __half2* o1 = reinterpret_cast<__half2*>(p.latents_f16 + (1 * HW + pix) * 4);
        o0[0] = __floats2half2_rn(l0.x, l0.y); o0[1] = __floats2half2_rn(l0.z, l0.w);
        o1[0] = __floats2half2_rn(l1.x, l1.y); o1[1] = __floats2half2_rn(l1.z, l1.w);
    }
    uint4 s0, s1;
    {
        __half2* h = reinterpret_cast<__half2*>(&s0);
        h[0] = __floats2half2_rn(l0.x * in_scale, l0.y * in_scale);
        h[1] = __floats2half2_rn(l0.z * in_scale, l0.w * in_scale);
        h[2] = h[3] = __floats2half2_rn(0.f, 0.f);
        h = reinterpret_cast<__half2*>(&s1);
        h[0] = __floats2half2_rn(l1.x * in_scale, l1.y * in_scale);
        h[1] = __floats2half2_rn(l1.z * in_scale, l1.w * in_scale);
        h[2] = h[3] = __floats2half2_rn(0.f, 0.f);
    }
    if (p.next_main_in) {
        uint4* o = reinterpret_cast<uint4*>(p.next_main_in);
        o[0 * HW + pix] = s0;
        o[1 * HW + pix] = s1;
        o[2 * HW + pix] = s0;
        o[3 * HW + pix] = s1;
    }
    if (p.next_concept_in) {
        uint4* o = reinterpret_cast<uint4*>(p.next_concept_in);
        o[0 * HW + pix] = s1;
        o[1 * HW + pix] = s1;
    }
}

// out[b, w, :] = sum_n coef[w, n] * ctx[b, n, :]   (coef = M diag(alpha) or diag(1 - alpha); L = 77)
__global__ void ctx_mix_kernel(const __half* __restrict__ ctx, const float* __restrict__ coef, __half* __restrict__ out,
                               int L, int C) {
    griddep_launch_dependents();
    griddep_wait();
    const int b = blockIdx.z, w = blockIdx.y;
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    float acc = 0.f;
    for (int n = 0; n < L; ++n) {
        const float a = coef[w * L + n];
        if (a != 0.f) acc += a * __half2float(ctx[((size_t)b * L + n) * C + c]);
    }
    out[((size_t)b * L + w) * C + c] = __float2half_rn(acc);
}

__global__ void axpy_kernel(const uint4* __restrict__ a, const uint4* __restrict__ b, float alpha,
                            uint4* __restrict__ y, long long nvec) {
    griddep_launch_dependents();
    griddep_wait();
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nvec) return;
    const uint4 ua = a[i], ub = b[i];
    const __half2* ha = reinterpret_cast<const __half2*>(&ua);
    const __half2* hb = reinterpret_cast<const __half2*>(&ub);
    uint4 o;
    __half2* ho = reinterpret_cast<__half2*>(&o);
#pragma unroll
    for (int t = 0; t < 4; ++t) {
        const float2 fa = __half22float2(ha[t]), fb = __half22float2(hb[t]);
        ho[t] = __floats2half2_rn(fa.x + alpha * fb.x, fa.y + alpha * fb.y);
    }
    y[i] = o;
}

// In-place softmax(scale * x) over the rows of an fp16 | bf16 matrix, fp32 arithmetic, one CTA per row, the row kept in
// registers (cols <= 256 threads x MAXV vectors x 8).  Used by the VAE decoder's single-head attention (head_dim 512
// is outside the flash kernel's d = 64), whose scores are materialised by omg_gemm.
constexpr int SM_THREADS = 256;
constexpr int SM_MAXV = 16;  // cols <= 32768
template <typename T>
__global__ void __launch_bounds__(SM_THREADS) softmax_rows_kernel(T* __restrict__ x, int cols, long long ld, float scale_log2) {
    using T2 = typename Pair<T>::type;
    griddep_launch_dependents();
    griddep_wait();
    __shared__ float red[SM_THREADS / 32];
    uint4* row = reinterpret_cast<uint4*>(x + (long long)blockIdx.x * ld);
    const int nvec = cols >> 3;
    uint4 v[SM_MAXV];
    float mx = -INFINITY;
#pragma unroll
    for (int i = 0; i < SM_MAXV; ++i) {
        const int j = threadIdx.x + i * SM_THREADS;
        if (j < nvec) {
            v[i] = row[j];
            const T2* h = reinterpret_cast<const T2*>(&v[i]);
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                const float2 f = to_float2(h[t]);
                mx = fmaxf(mx, fmaxf(f.x, f.y));
            }
        }
    }
    auto block_reduce = [&](float val, bool is_max) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float other = __shfl_xor_sync(0xffffffffu, val, o);
            val = is_max ? fmaxf(val, other) : val + other;
        }
        __syncthreads();
        if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = val;
        __syncthreads();
        float r = red[0];
#pragma unroll
        for (int w = 1; w < SM_THREADS / 32; ++w) r = is_max ? fmaxf(r, red[w]) : r + red[w];
        return r;
    };
    // scale > 0 is checked by the host: max(scale * x) = scale * max(x)
    const float m = block_reduce(mx, true) * scale_log2;
    float sum = 0.f;
#pragma unroll
    for (int i = 0; i < SM_MAXV; ++i) {
        const int j = threadIdx.x + i * SM_THREADS;
        if (j < nvec) {
            const T2* h = reinterpret_cast<const T2*>(&v[i]);
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                const float2 f = to_float2(h[t]);
                sum += exp2f(fmaf(f.x, scale_log2, -m)) + exp2f(fmaf(f.y, scale_log2, -m));
            }
        }
    }
    const float inv = 1.0f / block_reduce(sum, false);
    // the exponentials are recomputed rather than kept: the kernel is HBM-bound and the row already fills the registers
#pragma unroll
    for (int i = 0; i < SM_MAXV; ++i) {
        const int j = threadIdx.x + i * SM_THREADS;
        if (j < nvec) {
            const T2* h = reinterpret_cast<const T2*>(&v[i]);
            uint32_t o[4];
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                const float2 f = to_float2(h[t]);
                o[t] = pack2<T>(exp2f(fmaf(f.x, scale_log2, -m)) * inv, exp2f(fmaf(f.y, scale_log2, -m)) * inv);
            }
            row[j] = make_uint4(o[0], o[1], o[2], o[3]);
        }
    }
}

}  // namespace omg

using namespace omg;

template <typename T>
static int softmax_rows_impl(void* x, long long rows, int cols, long long ld, float scale, void* stream_) {
    cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
    const char* fn = std::is_same<T, __half>::value ? "omg_softmax_rows" : "omg_softmax_rows_bf16";
    OMG_CHECK(x && rows >= 1 && rows <= 0x7fffffffLL, "%s: bad arguments", fn);
    OMG_CHECK(cols >= 8 && cols % 8 == 0 && cols <= SM_THREADS * SM_MAXV * 8 && ld % 8 == 0 && ld >= cols,
              "%s: cols=%d must be a multiple of 8 and <= %d, ld a multiple of 8", fn, cols, SM_THREADS * SM_MAXV * 8);
    OMG_CHECK(scale > 0.f, "%s: scale must be positive", fn);
    OMG_CUDA(launch_pdl(softmax_rows_kernel<T>, dim3((unsigned)rows), dim3(SM_THREADS), 0, stream,
                        static_cast<T*>(x), cols, ld, scale * 1.4426950408889634f));
    return check_launch("softmax_rows_kernel");
}

static int axpy_impl(const void* a, const void* b, float alpha, void* y, long long n, void* stream_) {
    cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
    OMG_CHECK(a && b && y && n > 0 && n % 8 == 0, "omg_axpy: bad arguments");
    const long long nvec = n / 8;
    OMG_CUDA(launch_pdl(axpy_kernel, dim3((unsigned)((nvec + 255) / 256)), dim3(256), 0, stream,
                        static_cast<const uint4*>(a), static_cast<const uint4*>(b), alpha, static_cast<uint4*>(y), nvec));
    return check_launch("axpy_kernel");
}

static int fuse_step_impl(const omg_fuse_desc* d, void* stream_) {
    cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
    OMG_CHECK(d && d->noise_main && d->latents, "omg_fuse_step: null pointer");
    OMG_CHECK(d->n_concepts >= 0 && d->n_concepts <= OMG_MAX_CONCEPTS, "omg_fuse_step: n_concepts=%d out of range",
              d->n_concepts);
    OMG_CHECK(d->HW >= 1, "omg_fuse_step: empty latent");
    FuseParams p;
    p.noise_main = static_cast<const __half*>(d->noise_main);
    for (int k = 0; k < OMG_MAX_CONCEPTS; ++k) {
        p.noise_concept[k] = k < d->n_concepts ? static_cast<const __half*>(d->noise_concept[k]) : nullptr;
        p.mask[k] = k < d->n_concepts ? static_cast<const float*>(d->mask[k]) : nullptr;
        OMG_CHECK(k >= d->n_concepts || p.mask[k] == nullptr || p.noise_concept[k] != nullptr,
                  "omg_fuse_step: concept %d has a mask but no noise prediction", k);
    }
    p.n_concepts = d->n_concepts;
    p.guidance = d->guidance;
    p.sigma = d->sigma;
    p.sigma_next = d->sigma_next;
    p.latents = static_cast<float*>(d->latents);
    p.next_main_in = static_cast<__half*>(d->next_main_in);
    p.next_concept_in = static_cast<__half*>(d->next_concept_in);
    p.latents_f16 = static_cast<__half*>(d->latents_f16);
    p.HW = d->HW;
    OMG_CUDA(launch_pdl(fuse_step_kernel, dim3((d->HW + 127) / 128), dim3(128), 0, stream, p));
    return check_launch("fuse_step_kernel");
}

static int ctx_mix_impl(const void* ctx, const void* coef, void* out, int B, int L, int C, void* stream_) {
    cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
    OMG_CHECK(ctx && coef && out && B >= 1 && L >= 1 && C >= 1, "omg_ctx_mix: bad arguments");
    OMG_CUDA(launch_pdl(ctx_mix_kernel, dim3((C + 127) / 128, L, B), dim3(128), 0, stream,
                        static_cast<const __half*>(ctx), static_cast<const float*>(coef), static_cast<__half*>(out), L, C));
    return check_launch("ctx_mix_kernel");
}

// C-ABI entry points: launch, and - while this thread records a launch plan (omg_plan_record_begin) - remember the call
extern "C" int omg_softmax_rows(void* x, long long rows, int cols, long long ld, float scale, void* stream_) {
    const int rc = softmax_rows_impl<__half>(x, rows, cols, ld, scale, stream_);
    if (rc == 0 && ::omg::plan_recording()) ::omg::plan_note([=](void* s) { return softmax_rows_impl<__half>(x, rows, cols, ld, scale, s); });
    return rc;
}

extern "C" int omg_softmax_rows_bf16(void* x, long long rows, int cols, long long ld, float scale, void* stream_) {
    const int rc = softmax_rows_impl<__nv_bfloat16>(x, rows, cols, ld, scale, stream_);
    if (rc == 0 && ::omg::plan_recording()) ::omg::plan_note([=](void* s) { return softmax_rows_impl<__nv_bfloat16>(x, rows, cols, ld, scale, s); });
    return rc;
}

extern "C" int omg_axpy(const void* a, const void* b, float alpha, void* y, long long n, void* stream_) {
    const int rc = axpy_impl(a, b, alpha, y, n, stream_);
    if (rc == 0 && ::omg::plan_recording()) ::omg::plan_note([=](void* s) { return axpy_impl(a, b, alpha, y, n, s); });
    return rc;
}

extern "C" int omg_fuse_step(const omg_fuse_desc* d, void* stream_) {
    const int rc = fuse_step_impl(d, stream_);
    if (rc == 0 && ::omg::plan_recording()) {
        const omg_fuse_desc c = *d;  // by value: a plan outlives the caller's descriptor
        ::omg::plan_note([c](void* s) { return fuse_step_impl(&c, s); });
    }
    return rc;
}

extern "C" int omg_ctx_mix(const void* ctx, const void* coef, void* out, int B, int L, int C, void* stream_) {
    const int rc = ctx_mix_impl(ctx, coef, out, B, L, C, stream_);
    if (rc == 0 && ::omg::plan_recording()) ::omg::plan_note([=](void* s) { return ctx_mix_impl(ctx, coef, out, B, L, C, s); });
    return rc;
}
