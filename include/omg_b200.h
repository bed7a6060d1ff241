/*
 * omg_b200 — C ABI of the B200-native OMG denoising hot path.
 *
 * The reference (kongzhecn/OMG) is pure Python on diffusers and has no FFI of its own; the
 * "interface each entry point replaces" is therefore the torch / diffusers / xformers library call
 * the reference makes at the cited line.  Ownership: the caller owns every buffer; the library only
 * borrows raw device pointers for the duration of the call and keeps no state besides a per-process
 * error string.  Every function returns 0 on success, non-zero on failure (omg_last_error() gives
 * the message); nothing throws across the boundary.  All kernels are launched on the CUstream /
 * cudaStream_t handle passed as `stream` (void*), never synchronise the host, and are CUDA-graph
 * capturable.  fp16 storage, fp32 accumulation.  Activations are channels-last:
 * (B, H, W, C) == (B, H*W tokens, C).
 */
#ifndef OMG_B200_H
#define OMG_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OMG_MAX_A 4
#define OMG_MAX_SEGS 12

/* Strided channels-last view: element (b,h,w,c) lives at ptr + b*sb + h*sh + w*sw + c (in elements). */
typedef struct {
    const void* ptr;
    int32_t C, W, H, B;
    int64_t sw, sh, sb;
} omg_view4;

/* One K-segment of a (implicit) GEMM: A operand = view a[a_idx] shifted by (dx,dy) pixels (out-of-range
 * pixels read as zero = conv padding), channels [a_c0, a_c0+k_len); weight columns [b_k0, b_k0+k_len). */
typedef struct {
    int32_t a_idx, dx, dy, a_c0, k_len, b_k0;
    int32_t b_idx; /* 0: columns of w, 1: columns of w2 (e.g. the LoRA up-projection B, kept un-merged) */
} omg_seg;

enum { OMG_EPI_NONE = 0, OMG_EPI_GEGLU = 1, OMG_EPI_SILU = 2, OMG_EPI_QUICK_GELU = 3, OMG_EPI_GELU = 4, OMG_EPI_GELU_TANH = 5 };

/* Element type of the 16-bit operands of omg_gemm (omg_gemm_desc.dtype).  bf16 has fp32's exponent range: the VAE decoder
 * runs it for weights whose activations overflow fp16 (the original SDXL VAE, which diffusers up-casts to fp32). */
enum { OMG_DTYPE_F16 = 0, OMG_DTYPE_BF16 = 1 };

/*
 * out[pix, n] = epi( sum_seg sum_k A_seg[pix+(dx,dy), k] * W[n, b_k0+k] + bias[n] + rowvec[b, n] ) + residual[pix, n]
 *
 * Replaces: torch.nn.Linear / Conv2d(3x3 | 1x1, stride 1 | 2) / peft LoRA delta / GEGLU inside
 * diffusers UNet2DConditionModel.forward, reference call sites src/pipelines/lora_pipeline.py:546-566,592-599
 * (cuBLAS / cuDNN in the reference).  tcgen05 tensor cores, TMA-staged operands.
 * OMG_EPI_GEGLU: W rows (and bias) are interleaved (value_j, gate_j) pairs; out has N/2 channels,
 * out_j = value_j * gelu_erf(gate_j).   OMG_EPI_SILU: epi(x) = x * sigmoid(x) (time-embedding MLPs).
 * OMG_EPI_QUICK_GELU: x * sigmoid(1.702 x), OMG_EPI_GELU: erf-gelu (the fc1 activations of the two CLIP text towers,
 * transformers CLIPMLP [3P], reached from src/pipelines/lora_pipeline.py:315-347).
 */
typedef struct {
    omg_view4 a[OMG_MAX_A];
    int32_t n_a;
    omg_seg segs[OMG_MAX_SEGS];
    int32_t n_segs;
    const void* w;      /* [N, Ktot] row-major fp16 */
    int32_t N, Ktot;
    const void* w2;     /* optional second weight matrix [N, K2tot] (segments with b_idx == 1) or NULL */
    int32_t K2tot;
    omg_view4 d;        /* output view; d.W/H/B define the pixel grid the tiles walk */
    const void* bias;   /* [N] fp16 or NULL */
    const void* rowvec; /* [B, rowvec_ld] fp16 or NULL: per-image additive vector (time-embedding projection) */
    int32_t rowvec_ld;
    const void* residual; /* contiguous [B*H*W, residual_ld] fp16 or NULL, added after the epilogue */
    int32_t residual_ld;
    int32_t epilogue;
    int32_t block_n;    /* 0 = auto; else 64 | 128 | 160 | 256 */
    /* LayerNorm folded into a GEMM pair (BasicTransformerBlock norm1/2/3 [3P] followed by to_q|k|v / ff.net.0.proj):
     * the GEMM that PRODUCES the hidden state h writes per-row partial (sum, sum of squares) of its output, one
     * partial per n-tile, to row_stats_out [n_tiles][rows][2] fp32; the GEMM that CONSUMES LayerNorm(h) runs on raw h
     * with gamma folded into its weights and finishes  out = rstd * (acc - mean * c1[n]) + c2[n]  in the epilogue,
     * c1 = row sums of the folded fp16 weights, c2 = W beta + bias (fp32 [N]).  No LayerNorm kernel, no normalised
     * copy of h.  ln_dim = channels of h; row_stats_parts = n-tiles of the producer (omg_gemm_plan). */
    void* row_stats_out;
    const void* row_stats_in;
    int32_t row_stats_parts;
    int64_t row_stats_stride; /* rows per partial plane (0 = rows of this GEMM); lets a row-sliced GEMM index the full buffer */
    int32_t ln_dim;
    float ln_eps;
    const void* col_c1;
    const void* col_c2;
    /* multi-stream launches: streams (row groups) with different LoRA sets have different c1/c2; then col_c1/col_c2
     * are [n_col_groups][N] and rows [col_group_end[g-1], col_group_end[g]) use plane g (boundaries % 128 == 0). */
    int32_t n_col_groups;
    int64_t col_group_end[8];
    int32_t w_group_planes; /* 0: one weight matrix for all rows; else == n_col_groups: w is [planes][N][Ktot] and row
                             * group g multiplies with plane g (per-stream weights, e.g. W + s B_g A_g merged per concept) */
    int32_t cta_pair;   /* 0 = auto, 1 = single-CTA tiles, 2 = CTA pairs (cta_group::2, 256 x block_n tiles; block_n 256 | 160),
                         * 3 = tall tiles (one CTA, 256 x 160: two 128-row sub-tiles share each weight tile; block_n 160) */
    /* GroupNorm statistics out of the producing GEMM / conv (ResnetBlock2D norm1/norm2, Transformer2DModel.norm,
     * conv_norm_out [3P]): per image and per 32-pixel block of the output, the per-channel (sum, sum of squares) of the
     * fp16-ROUNDED output values, written as float2 to col_stats_out [B][col_stats_rb_total][N]; this launch fills the
     * blocks [col_stats_rb0, col_stats_rb0 + omg_gemm_colstats_blocks(W, H)) of every image.  The consuming
     * omg_groupnorm_apply reduces them to (mean, rstd) per group - for any grouping, also over the channel
     * concatenation of two producers - so GroupNorm never re-reads its input for statistics.  Not with GEGLU. */
    void* col_stats_out;
    int32_t col_stats_rb0, col_stats_rb_total;
    /* fp32 master copy of the residual trunk (x <- x + f(x) through ~70 transformer blocks and the ResBlocks): the addend
     * is read from residual_f32 [pixels, residual_f32_ld] instead of the fp16 `residual`, and the result is ALSO written as
     * fp32 to out_f32 [pixels, out_f32_ld] (the fp16 output stays what the next GEMM / norm reads), so rounding to fp16
     * no longer accumulates along the chain.  Either may be NULL.  Contiguous output view, N % 32 == 0, not with GEGLU. */
    const void* residual_f32;
    int64_t residual_f32_ld;
    void* out_f32;
    int64_t out_f32_ld;
    /* OMG_DTYPE_F16 (0, what a zeroed descriptor has) or OMG_DTYPE_BF16: the type of every 16-bit operand of the call -
     * A views, w, w2, bias, residual and the output.  bf16 supports OMG_EPI_NONE with bias, residual, K-segments, shifted
     * and strided views and every tile shape; activations / GEGLU, folded LayerNorm (row_stats_*), col_stats_out, rowvec,
     * weight planes / column groups and the fp32 twins are rejected. */
    int32_t dtype;
} omg_gemm_desc;

int omg_gemm(const omg_gemm_desc* desc, void* stream);

/* Tile plan omg_gemm will use for an output grid (W, H, B) with N channels: block_n and the number of row-statistics
 * partial planes this GEMM emits (= row_stats_parts for the consumer; two per n-tile). */
int omg_gemm_plan(int N, int epilogue, int W, int H, int B, int* block_n, int* stats_parts);

/* Number of 32-pixel column-statistics blocks one omg_gemm launch over an output grid (W, H) writes per image. */
int omg_gemm_colstats_blocks(int W, int H);

#define OMG_ATTN_MAX_ITEMS 16

/*
 * Flash attention, head_dim 64, fp32 softmax, probabilities never materialised:
 *   out[out_b[i], :, h] = (accumulate ? out : 0) + out_weight * softmax(scale * Q[q_b[i],:,h] K[k_b[i],:,h]^T) V[v_b[i],:,h]
 * for every item i and head h.  Q/K/V are row-major [batch, tokens, ld] fp16 with the head's 64 columns at
 * col0 + 64*h.
 *
 * Replaces: attn.get_attention_scores + controller(probs) + torch.bmm in RegionControlNet_AttnProcessor
 * (src/pipelines/lora_pipeline.py:114-116) with the prompt-to-prompt edit of src/prompt_attention/p2p_attention.py:
 * 124-138 folded into the (q_b, k_b, v_b) remap; xformers.ops.memory_efficient_attention / F.scaled_dot_product_
 * attention of the concept UNet (src/ip_adapter/attention_processor.py:197-204,383-401); and the decoupled
 * text + scale*ip sum (attention_processor.py:370-409) via accumulate/out_weight.
 */
typedef struct {
    const void* q; int32_t q_ld; int64_t q_bs; int32_t q_col0;
    const void* k; int32_t k_ld; int64_t k_bs; int32_t k_col0;
    const void* v; int32_t v_ld; int64_t v_bs; int32_t v_col0;
    void* out;     int32_t out_ld; int64_t out_bs; int32_t out_col0;
    int32_t n_q, n_kv, heads, head_dim;
    int32_t n_items;
    int32_t out_b[OMG_ATTN_MAX_ITEMS], q_b[OMG_ATTN_MAX_ITEMS], k_b[OMG_ATTN_MAX_ITEMS], v_b[OMG_ATTN_MAX_ITEMS];
    float scale;      /* softmax scale, head_dim^-0.5 */
    float out_weight; /* weight of this term */
    int32_t accumulate;
    int32_t causal;   /* 1: key j attends only to queries i >= j (CLIP text towers); n_kv <= 128 only */
} omg_attn_desc;

int omg_attention(const omg_attn_desc* desc, void* stream);

/*
 * GroupNorm(32 groups) over channels-last fp16, optional SiLU, input = channel-concatenation of (x1 | x2).
 * y[B, HW, C1+C2].  stats_ws: OMG_GN_WS_FLOATS(B) floats of scratch.  Deterministic: no atomics, results do not depend
 * on the batch position of an image.  Replaces torch GroupNorm + SiLU + torch.cat inside diffusers
 * ResnetBlock2D / Transformer2DModel / UNet up-blocks [3P] (call site src/pipelines/lora_pipeline.py:546-566).
 */
#define OMG_GN_MAX_SPLITS 256
#define OMG_GN_WS_FLOATS(B) ((B) * (2 * 2 * 2560 + 64 * OMG_GN_MAX_SPLITS))
int omg_groupnorm(const void* x1, int C1, const void* x2, int C2, int B, int HW, const void* gamma, const void* beta,
                  float eps, int silu, void* stats_ws, void* y, void* stream);
/* omg_groupnorm with bf16 x1, x2, gamma, beta and y (same contract, fp32 statistics). */
int omg_groupnorm_bf16(const void* x1, int C1, const void* x2, int C2, int B, int HW, const void* gamma, const void* beta,
                       float eps, int silu, void* stats_ws, void* y, void* stream);

/* Per-channel (sum, sum of squares) partials of a stored channels-last tensor x [B, HW, C], one float2 per channel per
 * 32-row block: out [B][ceil(HW/32)][C] - the layout omg_gemm's col_stats_out produces (for tensors that were modified
 * after their producing GEMM, e.g. skip connections that received ControlNet residuals). */
int omg_colstats(const void* x, int C, int B, int HW, void* out, void* stream);

/* GroupNorm(32) [+ SiLU] of cat(x1 | x2) from per-channel partials (omg_gemm col_stats_out / omg_colstats): one tiny
 * reduction launch (partials -> mean, rstd per image and group, fixed summation order) and one apply pass.
 * part1 [B][rb1][C1] float2, part2 [B][rb2][C2] float2 (NULL when C2 == 0); stats_ws: OMG_GN_WS_FLOATS(B) floats. */
int omg_groupnorm_apply(const void* x1, int C1, const void* part1, int rb1, const void* x2, int C2, const void* part2,
                        int rb2, int B, int HW, const void* gamma, const void* beta, float eps, int silu, void* stats_ws,
                        void* y, void* stream);

/* LayerNorm over the last dim of [rows, C] fp16 (BasicTransformerBlock norm1/2/3 [3P]). */
int omg_layernorm(const void* x, const void* gamma, const void* beta, void* y, long long rows, int C, float eps,
                  void* stream);

#define OMG_MAX_CONCEPTS 8

/*
 * One denoising-step tail in a single launch: region noise fusion, classifier-free guidance, Euler-discrete step,
 * and the next step's scaled model inputs.  Replaces src/pipelines/lora_pipeline.py:568-615 and :491-492,583-585
 * (src/pipelines/instantid_pipeline.py:618-690).
 *   noise_main [4, HW, 8] fp16 rows (uncond0, uncond1, cond0, cond1), channels 0..3 used;
 *   noise_concept[k] [2, HW, 8] rows (uncond, cond); mask[k] [HW] float {0,1} or NULL (concept skipped);
 *   image-1 rows: eps = (1 - U) * eps_main + sum_k M_k * eps_k with U = OR_k M_k;
 *   eps = eps_u + guidance * (eps_c - eps_u);  latents += eps * (sigma_next - sigma)   (fp32 state [2, HW, 4]);
 *   next_main_in [4, HW, 8] = latents / sqrt(sigma_next^2 + 1) in row order (img0, img1, img0, img1);
 *   next_concept_in [2, HW, 8] = scaled image-1 latent twice; latents_f16 optional fp16 copy [2, HW, 4].
 */
typedef struct {
    const void* noise_main;
    const void* noise_concept[OMG_MAX_CONCEPTS];
    const void* mask[OMG_MAX_CONCEPTS];
    int32_t n_concepts;
    float guidance, sigma, sigma_next;
    void* latents;
    void* next_main_in;
    void* next_concept_in;
    void* latents_f16;
    int32_t HW;
} omg_fuse_desc;

int omg_fuse_step(const omg_fuse_desc* desc, void* stream);

/*
 * out[b, w, :] = sum_n coef[w, n] * ctx[b, n, :]  (fp16 ctx/out [B, L, C], fp32 coef [L, L]).  Builds the
 * prompt-to-prompt edited context  M diag(alpha) ctx  /  diag(1-alpha) ctx  so that the cross-attention edit
 * P0 M * alpha + (1-alpha) P1  (src/prompt_attention/p2p_attention.py:131-134,146-147) becomes two plain attention
 * terms over projected V.
 */
int omg_ctx_mix(const void* ctx, const void* coef, void* out, int B, int L, int C, void* stream);

/* y = a + alpha * b over n fp16 elements (n % 8 == 0): ControlNet residual injection
 * (down_block_additional_residuals / mid_block_additional_residual, src/pipelines/lora_pipeline.py:546-556). */
int omg_axpy(const void* a, const void* b, float alpha, void* y, long long n, void* stream);

/* In-place row softmax: x[r, :cols] = softmax(scale * x[r, :cols]) for an fp16 matrix with row stride ld (elements),
 * fp32 arithmetic; cols % 8 == 0, cols <= 32768, scale > 0.  The VAE decoder's mid-block attention (one head of
 * 512 channels: `Attention(heads=1)` inside diffusers' AutoencoderKL, reached from src/pipelines/lora_pipeline.py:649)
 * materialises its scores with omg_gemm, normalises them here and applies them with a second omg_gemm. */
int omg_softmax_rows(void* x, long long rows, int cols, long long ld, float scale, void* stream);
/* omg_softmax_rows over a bf16 matrix (same contract). */
int omg_softmax_rows_bf16(void* x, long long rows, int cols, long long ld, float scale, void* stream);

/*
 * EfficientViT-SAM image encoder (the segmentation model between the two stages; SURVEY 8f-4), the ops that are not
 * GEMM-shaped.  Channels-last fp16, fp32 arithmetic.  Dense convolutions of the encoder go through omg_gemm (BatchNorm
 * folded into the weights, OMG_EPI_GELU_TANH), LayerNorm2d through omg_layernorm.
 *   omg_dwconv: depthwise k x k (3 | 5) convolution, stride 1 | 2, "same" padding, + bias, act 1 = tanh-GELU; w is
 *     tap-major [k*k, C]; x / y rows of ldx / ldy elements (MBConv.depth_conv, LiteMLA.aggreg[.][0];
 *     src/efficientvit/models/nn/ops.py:196-241,371-392).
 *   omg_group1x1: grouped 1x1 convolution with square groups of 32 channels, w [C, 32] (LiteMLA.aggreg[.][1]).
 *   omg_relu_linear_attention: LiteMLA.relu_linear_att (ops.py:404-440): per head (q | k | v, dim 32)
 *     out = relu(q) (relu(k)^T [v | 1]) normalised by its last column + eps; qkv [B, N, heads*96] -> out [B, N, heads*32].
 *   omg_resize_bicubic: F.interpolate(mode="bicubic", align_corners=False) (SamNeck inputs, sam.py:117-123).
 */
int omg_dwconv(const void* x, const void* w, const void* bias, void* y, int B, int H, int W, int C, int ldx, int ldy, int ksize,
               int stride, int act, void* stream);
int omg_group1x1(const void* x, const void* w, void* y, long long pixels, int C, int ldx, int ldy, int group, void* stream);
int omg_relu_linear_attention(const void* qkv, void* out, int B, int N, int heads, int dim, float eps, void* stream);
int omg_resize_bicubic(const void* x, void* y, int B, int H, int W, int C, int Ho, int Wo, void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Launch plans: a forward as a handle.  The reference drives one UNet forward as a Python call
 * (`self.unet(latent_model_input, t, ...)`, src/pipelines/lora_pipeline.py:558-567, 588-606); a host that is not Python -
 * or does not want ~720 descriptor builds per forward - records that call once and replays it through this handle:
 *
 *   omg_plan* fwd = omg_plan_create();
 *   omg_plan_record_begin(fwd);  ... one eager forward: omg_gemm / omg_attention / omg_groupnorm_apply / ... ;
 *   omg_plan_record_end(fwd);
 *   for every step:  (write the sample and the step's time embedding into their buffers)  omg_plan_run(fwd, stream);
 *
 * While a thread records, every entry point above that launched successfully also appends a copy of its call - the
 * descriptor by value, so every pointer in it must stay valid for as long as the plan is run (the executor's persistent
 * workspace does) - and omg_plan_run re-issues the calls in order on `stream` with no further host work than the launches.
 * Replay validates each descriptor and encodes its tensor maps again (a plan holds descriptors, not encoded launches), so a
 * plan is valid exactly as long as the buffers its descriptors point to.
 * One recording per thread at a time; a plan may be run from any thread once recording has ended.
 */
typedef struct omg_plan omg_plan;
omg_plan* omg_plan_create(void);
void omg_plan_destroy(omg_plan* plan);
int omg_plan_record_begin(omg_plan* plan);
int omg_plan_record_end(omg_plan* plan);
int omg_plan_length(const omg_plan* plan);     /* number of recorded launches; -1 for NULL */
int omg_plan_clear(omg_plan* plan);
int omg_plan_run(const omg_plan* plan, void* stream);

/* Error string of the last failing call on this thread (never NULL). */
const char* omg_last_error(void);
/* Library / build identification: returns e.g. "omg_b200 sm_100a". */
const char* omg_version(void);
/* Number of kernel launches issued by this library since process start (bench.py's gpu_launches). */
uint64_t omg_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif
