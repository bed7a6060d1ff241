"""Host-side launchers: torch tensors (device memory + stream plumbing only) -> C-ABI descriptors.

All activations are channels-last fp16: (B, H, W, C), equivalently (B, H*W tokens, C).  `linear`, `conv3x3`,
`upsample2x_conv3x3`, `groupnorm` and `softmax_rows` also run bf16 (the VAE decoder's path for weights whose activations
overflow fp16): they take the element type from the input tensor and refuse operands of another type.
"""
import ctypes as C

import torch

from . import _lib as L


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _chk16(t: torch.Tensor):
    if not t.is_cuda or t.dtype != torch.float16:
        raise ValueError("expected a CUDA fp16 tensor (there is no CPU path)")


_GEMM_DTYPES = {torch.float16: L.DTYPE_F16, torch.bfloat16: L.DTYPE_BF16}


def _same_dtype(x: torch.Tensor, *others) -> torch.dtype:
    """x.dtype, after checking that x is a CUDA fp16 | bf16 tensor and that every other operand given has its type."""
    if not x.is_cuda or x.dtype not in _GEMM_DTYPES:
        raise ValueError("expected a CUDA fp16 or bf16 tensor (there is no CPU path)")
    for t in others:
        if t is not None and t.dtype != x.dtype:
            raise ValueError(f"mixed operand dtypes: input is {x.dtype}, an operand is {t.dtype}")
    return x.dtype


def view4(t: torch.Tensor, dtype: torch.dtype = torch.float16) -> L.View4:
    """(B,H,W,C) tensor (any pixel strides, unit channel stride) or 2-D [M,K] matrix of `dtype` -> omg_view4."""
    if _same_dtype(t) != dtype:
        raise ValueError(f"expected a CUDA {dtype} tensor, got {t.dtype}")
    if t.dim() == 2:
        assert t.stride(1) == 1
        return L.View4(t.data_ptr(), t.shape[1], t.shape[0], 1, 1, t.stride(0), t.stride(0) * t.shape[0],
                       t.stride(0) * t.shape[0])
    assert t.dim() == 4 and t.stride(3) == 1
    B, H, W, Cc = t.shape
    return L.View4(t.data_ptr(), Cc, W, H, B, t.stride(2), t.stride(1), t.stride(0))


def _ptr(t):
    return None if t is None else t.data_ptr()


class LaunchPlan:
    """omg_plan (include/omg_b200.h): the launches of one forward recorded at the C ABI and replayed from C with no
    descriptor building - what a non-Python host holds instead of the reference's `self.unet(...)` call
    (src/pipelines/lora_pipeline.py:558-567).  Everything a recorded launch points to must outlive the plan (the
    executor's persistent workspace does; tensors allocated inside the recorded region do not)."""

    def __init__(self):
        self._lib = L.load()
        self._h = self._lib.omg_plan_create()
        if not self._h:
            raise RuntimeError("omg_plan_create failed")

    def __enter__(self):
        L.check(self._lib.omg_plan_record_begin(self._h), "omg_plan_record_begin")
        return self

    def __exit__(self, *exc):
        L.check(self._lib.omg_plan_record_end(self._h), "omg_plan_record_end")
        return False

    def __len__(self):
        return int(self._lib.omg_plan_length(self._h))

    def clear(self):
        L.check(self._lib.omg_plan_clear(self._h), "omg_plan_clear")

    def run(self, stream=None):
        L.check(self._lib.omg_plan_run(self._h, _stream() if stream is None else stream), "omg_plan_run")

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h:
            self._lib.omg_plan_destroy(h)


def gemm(a_views, segs, w, N, Ktot, d_view, bias=None, rowvec=None, rowvec_ld=0, residual=None, residual_ld=0,
         epilogue=L.EPI_NONE, block_n=0, w2=None, stats_out=None, ln=None, cta_pair=0, row_groups=None, colstats=None,
         residual_f32=None, out_f32=None, dtype=torch.float16):
    d = L.GemmDesc()
    d.dtype = _GEMM_DTYPES[dtype]
    if residual_f32 is not None:   # [pixels, N] fp32 twins of the residual trunk (see omg_gemm_desc)
        d.residual_f32, d.residual_f32_ld = residual_f32.data_ptr(), residual_f32.stride(-2)
    if out_f32 is not None:
        d.out_f32, d.out_f32_ld = out_f32.data_ptr(), out_f32.stride(-2)
    d.cta_pair = cta_pair
    if colstats is not None:  # (partials [B, rb_total, N, 2] fp32, first block this launch fills)
        part, rb0 = colstats
        d.col_stats_out, d.col_stats_rb0, d.col_stats_rb_total = part.data_ptr(), rb0, part.shape[1]
    if row_groups is not None:  # per-stream weight planes: w is [len(row_groups) * N, Ktot]
        d.w_group_planes = d.n_col_groups = len(row_groups)
        for i, e in enumerate(row_groups):
            d.col_group_end[i] = e
    d.n_a = len(a_views)
    for i, v in enumerate(a_views):
        d.a[i] = v
    d.n_segs = len(segs)
    for i, s in enumerate(segs):
        d.segs[i] = L.Seg(*s) if len(s) == 7 else L.Seg(*s, 0)
    d.w = w.data_ptr()
    d.N, d.Ktot = N, Ktot
    if w2 is not None:
        d.w2, d.K2tot = w2.data_ptr(), w2.shape[1]
    d.d = d_view
    d.bias = _ptr(bias)
    d.rowvec = _ptr(rowvec)
    d.rowvec_ld = rowvec_ld
    d.residual = _ptr(residual)
    d.residual_ld = residual_ld
    d.epilogue = epilogue
    d.block_n = block_n
    if stats_out is not None:
        d.row_stats_out = stats_out.data_ptr()
    if ln is not None:  # folded LayerNorm: (stats [parts, rows, 2] fp32, parts, rows per part, row offset, dim, eps, c1, c2)
        stats, parts, stride, row0, dim, eps, c1, c2, group_ends = ln
        d.row_stats_in = stats.data_ptr() + row0 * 8
        d.row_stats_parts, d.row_stats_stride, d.ln_dim, d.ln_eps = parts, stride, dim, eps
        d.col_c1, d.col_c2 = c1.data_ptr(), c2.data_ptr()
        d.n_col_groups = len(group_ends)
        for i, e in enumerate(group_ends):
            d.col_group_end[i] = e
    L.check(L.load().omg_gemm(C.byref(d), _stream()), "omg_gemm")


def gemm_plan(N, epilogue, W, H=1, B=1):
    """(block_n, n_tiles) omg_gemm will use; n_tiles = number of row-statistics partials a producer emits."""
    bn, nt = C.c_int(0), C.c_int(0)
    L.check(L.load().omg_gemm_plan(N, epilogue, W, H, B, C.byref(bn), C.byref(nt)), "omg_gemm_plan")
    return bn.value, nt.value


def colstats_blocks(W, H=1):
    """32-pixel column-statistics blocks one omg_gemm launch over an output grid (W, H) writes per image."""
    return L.load().omg_gemm_colstats_blocks(W, H)


def linear(x, w, bias=None, residual=None, out=None, epilogue=L.EPI_NONE, extra=None, block_n=0, lora=None,
           stats_out=None, ln=None, cta_pair=0, row_groups=None, colstats=None, residual_f32=None, out_f32=None):
    """out[M, N'] = epi(x[M,K] @ w[N, :K]^T (+ extra K-segments) + bias) + residual.

    `extra` = list of (tensor [M,Ki], column offset into w): further K-segments of the same weight matrix.
    `lora`  = (t [M,R], w2 [N,R]): un-merged LoRA delta  t @ w2^T  with t = A x (scales folded into w2).
    """
    dt = _same_dtype(x, w, bias, residual, out, *[t for t, _ in (extra or [])], *(lora or ()))
    M, K = x.shape
    N, Ktot = w.shape
    if row_groups is not None:
        N //= len(row_groups)
    n_out = N // 2 if epilogue == L.EPI_GEGLU else N
    if out is None:
        out = torch.empty((M, n_out), dtype=dt, device=x.device)
    views = [view4(x, dt)]
    segs = [(0, 0, 0, 0, K, 0)]
    for t, off in (extra or []):
        views.append(view4(t, dt))
        segs.append((len(views) - 1, 0, 0, 0, t.shape[1], off))
    w2 = None
    if lora is not None:
        t, w2 = lora
        views.append(view4(t, dt))
        segs.append((len(views) - 1, 0, 0, 0, t.shape[1], 0, 1))
    # colstats: partials [B, rb, N, 2] of an output of B images x HW tokens; the [M, N] GEMM sees them as one image
    # of M rows, which is the same memory when no 128-row tile straddles two images (HW % 128 == 0, caller's duty)
    cs = None if colstats is None else (colstats.view(1, -1, colstats.shape[2], 2), 0)
    gemm(views, segs, w, N, Ktot, view4(out, dt), bias=bias, residual=residual,
         residual_ld=0 if residual is None else residual.stride(0), epilogue=epilogue, block_n=block_n, w2=w2,
         stats_out=stats_out, ln=ln, cta_pair=cta_pair, row_groups=row_groups, colstats=cs,
         residual_f32=residual_f32, out_f32=out_f32, dtype=dt)
    return out


def _taps3x3(Cin, a_idx=0, c0=0, k0=0):
    return [(a_idx, kx - 1, ky - 1, c0, Cin, k0 + (ky * 3 + kx) * Cin) for ky in range(3) for kx in range(3)]


def conv3x3(x, w, bias=None, rowvec=None, residual=None, out=None, shortcut=None, block_n=0, cta_pair=0, colstats=None,
            residual_f32=None, out_f32=None):
    """3x3 / stride 1 / pad 1 conv over (B,H,W,Cin).  w = [N, 9*Cin (+ shortcut K)] packed (ky, kx, c).

    shortcut = list of (tensor (B,H,W,Ci), weight column offset): 1x1-conv K-segments added to the same accumulator
    (ResnetBlock2D conv_shortcut).  rowvec [B, N] is added per image (time-embedding projection).
    """
    dt = _same_dtype(x, w, bias, rowvec, residual, out, *[t for t, _ in (shortcut or [])])
    B, H, W, Cin = x.shape
    N, Ktot = w.shape
    if out is None:
        out = torch.empty((B, H, W, N), dtype=dt, device=x.device)
    views = [view4(x, dt)]
    segs = _taps3x3(Cin)
    for t, off in (shortcut or []):
        views.append(view4(t, dt))
        segs.append((len(views) - 1, 0, 0, 0, t.shape[3], off))
    gemm(views, segs, w, N, Ktot, view4(out, dt), bias=bias, rowvec=rowvec,
         rowvec_ld=0 if rowvec is None else rowvec.stride(0),
         residual=residual, residual_ld=0 if residual is None else N, block_n=block_n, cta_pair=cta_pair,
         colstats=None if colstats is None else (colstats, 0), residual_f32=residual_f32, out_f32=out_f32, dtype=dt)
    return out


def conv3x3_s2(x, w, bias=None, out=None, block_n=0, colstats=None):
    """3x3 / stride 2 / pad 1 conv (Downsample2D): A operands are the four stride-2 phase views of x."""
    B, H, W, Cin = x.shape
    N, Ktot = w.shape
    assert H % 2 == 0 and W % 2 == 0
    if out is None:
        out = torch.empty((B, H // 2, W // 2, N), dtype=torch.float16, device=x.device)
    views = [view4(x[:, py::2, px::2, :]) for py in range(2) for px in range(2)]
    segs = []
    for ky in range(3):
        for kx in range(3):
            py, oy = (1, -1) if ky == 0 else ((0, 0) if ky == 1 else (1, 0))
            px, ox = (1, -1) if kx == 0 else ((0, 0) if kx == 1 else (1, 0))
            segs.append((py * 2 + px, ox, oy, 0, Cin, (ky * 3 + kx) * Cin))
    gemm(views, segs, w, N, Ktot, view4(out), bias=bias, block_n=block_n,
         colstats=None if colstats is None else (colstats, 0))
    return out


def upsample2x_conv3x3(x, w, bias=None, out=None, block_n=0, colstats=None, cta_pair=0):
    """nearest-2x upsample followed by 3x3 conv (Upsample2D) without materialising the upsampled tensor:
    each output phase (py,px) is a 9-tap conv over x with shifted taps, stored through a strided output view."""
    dt = _same_dtype(x, w, bias, out)
    B, H, W, Cin = x.shape
    N, Ktot = w.shape
    if out is None:
        out = torch.empty((B, 2 * H, 2 * W, N), dtype=dt, device=x.device)
    xv = view4(x, dt)
    off = {0: (-1, 0, 0), 1: (0, 0, 1)}
    for py in range(2):
        for px in range(2):
            segs = [(0, off[px][kx], off[py][ky], 0, Cin, (ky * 3 + kx) * Cin) for ky in range(3) for kx in range(3)]
            cs = None if colstats is None else (colstats, (py * 2 + px) * colstats_blocks(W, H))
            gemm([xv], segs, w, N, Ktot, view4(out[:, py::2, px::2, :], dt), bias=bias, block_n=block_n, colstats=cs, dtype=dt,
                 cta_pair=cta_pair)
    return out


def attention(q, k, v, out, heads, n_q, n_kv, items, q_col0=0, k_col0=0, v_col0=0, out_col0=0, scale=0.125,
              out_weight=1.0, accumulate=False, causal=False):
    """q/k/v/out: [batch, tokens, ld] fp16.  items: list of (out_b, q_b, k_b, v_b)."""
    for t in (q, k, v, out):
        _chk16(t)
        assert t.dim() == 3 and t.stride(2) == 1
    d = L.AttnDesc()
    d.q, d.q_ld, d.q_bs, d.q_col0 = q.data_ptr(), q.stride(1), q.stride(0), q_col0
    d.k, d.k_ld, d.k_bs, d.k_col0 = k.data_ptr(), k.stride(1), k.stride(0), k_col0
    d.v, d.v_ld, d.v_bs, d.v_col0 = v.data_ptr(), v.stride(1), v.stride(0), v_col0
    d.out, d.out_ld, d.out_bs, d.out_col0 = out.data_ptr(), out.stride(1), out.stride(0), out_col0
    d.n_q, d.n_kv, d.heads, d.head_dim = n_q, n_kv, heads, 64
    d.n_items = len(items)
    for i, (ob, qb, kb, vb) in enumerate(items):
        d.out_b[i], d.q_b[i], d.k_b[i], d.v_b[i] = ob, qb, kb, vb
    d.scale, d.out_weight, d.accumulate, d.causal = scale, out_weight, int(accumulate), int(causal)
    L.check(L.load().omg_attention(C.byref(d), _stream()), "omg_attention")
    return out


def groupnorm(x1, gamma, beta, eps, silu, x2=None, out=None, stats_ws=None):
    """GroupNorm(32)(cat([x1, x2], channel)) [+ SiLU]; x: (B, H, W, C) or (B, HW, C), fp16 or bf16 (gamma, beta, x2 and
    out of the same type)."""
    dt = _same_dtype(x1, gamma, beta, x2, out)
    B = x1.shape[0]
    C1 = x1.shape[-1]
    HW = x1.numel() // (B * C1)
    C2 = 0 if x2 is None else x2.shape[-1]
    assert x1.is_contiguous() and (x2 is None or x2.is_contiguous())
    if out is None:
        out = torch.empty((*x1.shape[:-1], C1 + C2), dtype=dt, device=x1.device)
    if stats_ws is None:
        stats_ws = torch.empty(B * (10240 + 64 * 256), dtype=torch.float32, device=x1.device)
    name = "omg_groupnorm" if dt == torch.float16 else "omg_groupnorm_bf16"
    L.check(getattr(L.load(), name)(x1.data_ptr(), C1, _ptr(x2), C2, B, HW, gamma.data_ptr(), beta.data_ptr(),
                                    float(eps), int(silu), stats_ws.data_ptr(), out.data_ptr(), _stream()), name)
    return out


def colstats(x, out=None):
    """Per-channel (sum, sumsq) partials of a stored (B, HW.., C) tensor, one per 32-row block: [B, ceil(HW/32), C, 2]."""
    _chk16(x)
    assert x.is_contiguous()
    B, Cc = x.shape[0], x.shape[-1]
    HW = x.numel() // (B * Cc)
    if out is None:
        out = torch.empty((B, (HW + 31) // 32, Cc, 2), dtype=torch.float32, device=x.device)
    assert out.shape[0] >= B and out.shape[1] == (HW + 31) // 32 and out.shape[2] == Cc
    L.check(L.load().omg_colstats(x.data_ptr(), Cc, B, HW, out.data_ptr(), _stream()), "omg_colstats")
    return out


def groupnorm_apply(x1, part1, gamma, beta, eps, silu, x2=None, part2=None, out=None, stats_ws=None):
    """GroupNorm(32)(cat([x1, x2], channel)) [+ SiLU] with the statistics taken from per-channel partials
    (omg_gemm colstats / ops.colstats): no statistics pass over x."""
    _chk16(x1)
    B, C1 = x1.shape[0], x1.shape[-1]
    HW = x1.numel() // (B * C1)
    C2 = 0 if x2 is None else x2.shape[-1]
    assert x1.is_contiguous() and (x2 is None or x2.is_contiguous())
    assert part1.shape[0] == B and part1.shape[2] == C1 and (x2 is None or (part2.shape[0] == B and part2.shape[2] == C2))
    if out is None:
        out = torch.empty((*x1.shape[:-1], C1 + C2), dtype=torch.float16, device=x1.device)
    if stats_ws is None:
        stats_ws = torch.empty(B * (10240 + 64 * 256), dtype=torch.float32, device=x1.device)
    L.check(L.load().omg_groupnorm_apply(x1.data_ptr(), C1, part1.data_ptr(), part1.shape[1], _ptr(x2), C2, _ptr(part2),
                                         0 if part2 is None else part2.shape[1], B, HW, gamma.data_ptr(), beta.data_ptr(),
                                         float(eps), int(silu), stats_ws.data_ptr(), out.data_ptr(), _stream()),
            "omg_groupnorm_apply")
    return out


def dwconv(x, w, bias=None, out=None, ksize=3, stride=1, act=0):
    """Depthwise k x k conv ("same" padding) over (B, H, W, C) rows that may be strided views along the channel axis
    (x.stride(2) = row stride); w tap-major [k*k, C]; act 1 = tanh-GELU."""
    _chk16(x)
    B, H, W, Cc = x.shape
    assert x.stride(3) == 1 and x.stride(1) == x.stride(2) * W and x.stride(0) == x.stride(1) * H
    Ho, Wo = (H + stride - 1) // stride, (W + stride - 1) // stride
    if out is None:
        out = torch.empty((B, Ho, Wo, Cc), dtype=torch.float16, device=x.device)
    assert out.stride(3) == 1 and out.stride(1) == out.stride(2) * Wo and out.stride(0) == out.stride(1) * Ho
    L.check(L.load().omg_dwconv(x.data_ptr(), w.data_ptr(), _ptr(bias), out.data_ptr(), B, H, W, Cc, x.stride(2), out.stride(2),
                                ksize, stride, int(act), _stream()), "omg_dwconv")
    return out


def group1x1(x, w, out):
    """Grouped 1x1 conv, square groups of 32 channels: x (.., C) rows strided, w [C, 32], out (.., C) rows strided."""
    _chk16(x)
    Cc = x.shape[-1]
    pixels = x.numel() // Cc
    L.check(L.load().omg_group1x1(x.data_ptr(), w.data_ptr(), out.data_ptr(), pixels, Cc, x.stride(-2), out.stride(-2), 32, _stream()),
            "omg_group1x1")
    return out


def relu_linear_attention(qkv, heads, dim=32, eps=1e-15, out=None):
    """LiteMLA core: qkv (B, N, heads*3*dim) contiguous -> (B, N, heads*dim)."""
    _chk16(qkv)
    assert qkv.is_contiguous()
    B, N, _ = qkv.shape
    if out is None:
        out = torch.empty((B, N, heads * dim), dtype=torch.float16, device=qkv.device)
    L.check(L.load().omg_relu_linear_attention(qkv.data_ptr(), out.data_ptr(), B, N, heads, dim, float(eps), _stream()),
            "omg_relu_linear_attention")
    return out


def resize_bicubic(x, Ho, Wo, out=None):
    """F.interpolate(mode='bicubic', align_corners=False) over (B, H, W, C)."""
    _chk16(x)
    assert x.is_contiguous()
    B, H, W, Cc = x.shape
    if out is None:
        out = torch.empty((B, Ho, Wo, Cc), dtype=torch.float16, device=x.device)
    L.check(L.load().omg_resize_bicubic(x.data_ptr(), out.data_ptr(), B, H, W, Cc, Ho, Wo, _stream()), "omg_resize_bicubic")
    return out


def layernorm(x, gamma, beta, eps=1e-5, out=None):
    _chk16(x)
    assert x.is_contiguous()
    Cc = x.shape[-1]
    rows = x.numel() // Cc
    if out is None:
        out = torch.empty_like(x)
    L.check(L.load().omg_layernorm(x.data_ptr(), gamma.data_ptr(), beta.data_ptr(), out.data_ptr(), rows, Cc,
                                   float(eps), _stream()), "omg_layernorm")
    return out


def fuse_step(noise_main, noise_concepts, masks, guidance, sigma, sigma_next, latents, next_main_in=None,
              next_concept_in=None, latents_f16=None):
    d = L.FuseDesc()
    d.noise_main = noise_main.data_ptr()
    d.n_concepts = len(noise_concepts)
    for i, (n, m) in enumerate(zip(noise_concepts, masks)):
        d.noise_concept[i] = _ptr(n)
        d.mask[i] = _ptr(m)
    d.guidance, d.sigma, d.sigma_next = float(guidance), float(sigma), float(sigma_next)
    d.latents = latents.data_ptr()
    d.next_main_in = _ptr(next_main_in)
    d.next_concept_in = _ptr(next_concept_in)
    d.latents_f16 = _ptr(latents_f16)
    d.HW = latents.shape[1] * latents.shape[2] if latents.dim() == 4 else latents.shape[1]
    L.check(L.load().omg_fuse_step(C.byref(d), _stream()), "omg_fuse_step")


def axpy(a, b, alpha=1.0, out=None):
    """out = a + alpha * b (fp16, same shape)."""
    _chk16(a)
    if out is None:
        out = torch.empty_like(a)
    L.check(L.load().omg_axpy(a.data_ptr(), b.data_ptr(), float(alpha), out.data_ptr(), a.numel(), _stream()),
            "omg_axpy")
    return out


def softmax_rows(x, scale=1.0):
    """In-place softmax(scale * x) over the last dimension of a 2-D fp16 | bf16 matrix (rows may be strided)."""
    dt = _same_dtype(x)
    assert x.dim() == 2 and x.stride(1) == 1
    name = "omg_softmax_rows" if dt == torch.float16 else "omg_softmax_rows_bf16"
    L.check(getattr(L.load(), name)(_ptr(x), x.shape[0], x.shape[1], x.stride(0), float(scale), _stream()), name)
    return x


def ctx_mix(ctx, coef, out=None):
    _chk16(ctx)
    B, Lk, Cc = ctx.shape
    if out is None:
        out = torch.empty_like(ctx)
    L.check(L.load().omg_ctx_mix(ctx.data_ptr(), coef.data_ptr(), out.data_ptr(), B, Lk, Cc, _stream()),
            "omg_ctx_mix")
    return out


# ------------------------------------------------------------------ weight packing (host, once per model load)
def pack_conv3x3_weight(w):
    """torch Conv2d weight [N, C, 3, 3] -> [N, 9*C] with K order (ky, kx, c)."""
    N, Cc = w.shape[:2]
    return w.permute(0, 2, 3, 1).reshape(N, 9 * Cc).contiguous()


def pack_geglu_weight(w, b=None):
    """GEGLU proj Linear(c -> 8c): rows [value(4c) ; gate(4c)] -> interleaved (value_j, gate_j)."""
    n2 = w.shape[0] // 2
    wi = torch.stack([w[:n2], w[n2:]], dim=1).reshape(w.shape[0], w.shape[1]).contiguous()
    bi = None if b is None else torch.stack([b[:n2], b[n2:]], dim=1).reshape(-1).contiguous()
    return wi, bi
