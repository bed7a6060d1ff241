"""bf16 activation path of the VAE decoder (weights whose activations overflow fp16, e.g. the original SDXL VAE): the
bf16 GEMM in every tile shape, GroupNorm and row softmax against fp32 torch, the decoder against the fp32 oracle
(oracle/vae.py) and against torch-eager bf16, an overflow fixture that fp16 cannot decode, determinism and launch-plan
replay.  Inputs are rounded to bf16 before the fp32 references see them, so the errors measure the bf16 path's own
arithmetic.  The original SDXL VAE weights are not part of the suite; the overflow fixture stands in for them."""
import json
import os
import subprocess
import sys

import pytest
import torch
import torch.nn.functional as F

from scripts.vae_bench import eager_decode

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BF = torch.bfloat16
# bounds = 1.25 x the largest rel-L2 measured on a B200 (GEMM 1.66e-3 in every tile mode and shape, GroupNorm 1.68e-3,
# decoder 1.10e-2 on the toy widths / 8.7e-3 at SDXL widths, where torch-eager bf16 measured 1.44e-2 / 1.16e-2);
# ceilings of the bf16 path: GEMM 1e-2, decoder 2e-2
GEMM_BOUND = 2.1e-3
GN_BOUND = 2.1e-3
DECODE_BOUND = 1.4e-2


def rel(a, b):
    a, b = a.float().cpu(), b.float().cpu()
    return ((a - b).norm() / b.norm()).item()


def rnd(*shape, seed, scale=1.0):
    return (torch.randn(*shape, generator=torch.Generator().manual_seed(seed)) * scale).to(BF).cuda()


# every tile mode: block_n x cta_pair (1 single, 2 CTA pairs, 3 tall; combinations without such a variant run as
# single tiles), and the 256 x 320 pair tile
MODES = [(bn, cp) for bn in (64, 128, 160, 256) for cp in (1, 2, 3)] + [(320, 0)]


@pytest.mark.parametrize("block_n,cta_pair", MODES)
def test_gemm_bf16_linear_bias_residual(block_n, cta_pair):
    from omg_b200 import ops
    x, w = rnd(1024, 640, seed=1), rnd(640, 640, seed=2, scale=640 ** -0.5)
    b, r = rnd(640, seed=3, scale=0.1), rnd(1024, 640, seed=4)
    got = ops.linear(x, w, bias=b, residual=r, block_n=block_n, cta_pair=cta_pair)
    assert got.dtype == BF
    ref = x.float() @ w.float().t() + b.float() + r.float()
    err = rel(got, ref)
    print("linear", block_n, cta_pair, err)
    assert err < GEMM_BOUND


@pytest.mark.parametrize("block_n,cta_pair", MODES)
def test_gemm_bf16_conv3x3_shortcut_and_k_tail(block_n, cta_pair):
    """3x3 conv over 72 channels (K tail of 8 per tap) + a 1x1 shortcut K-segment over 40 channels, bias."""
    from omg_b200 import ops
    N = 640
    x, t = rnd(2, 16, 16, 72, seed=5), rnd(2, 16, 16, 40, seed=6)
    w3, w1 = rnd(N, 72, 3, 3, seed=7, scale=(9 * 72) ** -0.5), rnd(N, 40, seed=8, scale=40 ** -0.5)
    b = rnd(N, seed=9, scale=0.1)
    w = torch.cat([ops.pack_conv3x3_weight(w3), w1], dim=1).contiguous()
    got = ops.conv3x3(x, w, bias=b, shortcut=[(t, 9 * 72)], block_n=block_n, cta_pair=cta_pair)
    ref = (F.conv2d(x.float().permute(0, 3, 1, 2), w3.float(), b.float(), padding=1)
           + F.conv2d(t.float().permute(0, 3, 1, 2), w1.float()[:, :, None, None])).permute(0, 2, 3, 1)
    err = rel(got, ref)
    print("conv3x3", block_n, cta_pair, err)
    assert err < GEMM_BOUND


@pytest.mark.parametrize("block_n,cta_pair", MODES)
def test_gemm_bf16_upsample2x_conv3x3(block_n, cta_pair):
    """The four phase launches of nearest-2x upsample + 3x3 conv: shifted A views, strided output views."""
    from omg_b200 import ops
    N = 640
    x = rnd(2, 16, 16, 128, seed=10)
    w3, b = rnd(N, 128, 3, 3, seed=11, scale=(9 * 128) ** -0.5), rnd(N, seed=12, scale=0.1)
    got = ops.upsample2x_conv3x3(x, ops.pack_conv3x3_weight(w3), bias=b, block_n=block_n, cta_pair=cta_pair)
    up = F.interpolate(x.float().permute(0, 3, 1, 2), scale_factor=2.0, mode="nearest")
    ref = F.conv2d(up, w3.float(), b.float(), padding=1).permute(0, 2, 3, 1)
    err = rel(got, ref)
    print("upsample2x_conv3x3", block_n, cta_pair, err)
    assert err < GEMM_BOUND


def test_gemm_bf16_with_omg_gemm_320_env():
    """OMG_GEMM_320=1 turns 160-wide choices into 256 x 320 pair tiles; a bf16 launch must take them too."""
    code = ("import sys, torch; sys.path.insert(0, %r)\n"
            "from omg_b200 import ops\n"
            "x = torch.randn(4096, 1280).to(torch.bfloat16).cuda(); w = (torch.randn(1280, 1280) / 36).to(torch.bfloat16).cuda()\n"
            "assert ops.gemm_plan(1280, 0, 4096)[0] == 160\n"
            "y = ops.linear(x, w); ref = x.float() @ w.float().t()\n"
            "print(((y.float() - ref).norm() / ref.norm()).item())\n") % ROOT
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=dict(os.environ, OMG_GEMM_320="1"))
    assert r.returncode == 0, r.stderr
    assert float(r.stdout.split()[-1]) < GEMM_BOUND


def test_bf16_refusals_through_ops():
    from omg_b200 import _lib as L
    from omg_b200 import ops
    x, w = rnd(256, 64, seed=1), rnd(128, 64, seed=2)
    with pytest.raises(ValueError, match="mixed operand dtypes"):
        ops.linear(x, w.half())
    with pytest.raises(ValueError, match="mixed operand dtypes"):
        ops.linear(x, w, bias=torch.zeros(128, dtype=torch.float16, device="cuda"))
    with pytest.raises(ValueError, match="mixed operand dtypes"):
        ops.groupnorm(x.view(1, 256, 64), torch.ones(64, device="cuda").half(), torch.zeros(64, device="cuda", dtype=BF), 1e-6, 0)
    with pytest.raises(ValueError):
        ops.layernorm(x, torch.ones(64, device="cuda", dtype=BF), torch.zeros(64, device="cuda", dtype=BF))  # fp16 only
    with pytest.raises(ValueError):
        ops.conv3x3_s2(rnd(1, 8, 8, 64, seed=3), rnd(64, 9 * 64, seed=4))  # fp16 only
    with pytest.raises(RuntimeError, match="epilogue activation"):
        ops.linear(x, w, epilogue=L.EPI_SILU)
    with pytest.raises(RuntimeError, match="fp32 twins"):
        ops.linear(x, w, out_f32=torch.empty(256, 128, device="cuda"))
    with pytest.raises(RuntimeError, match="folded LayerNorm"):
        ops.linear(x, w, stats_out=torch.empty(4, 256, 2, device="cuda"))


@pytest.mark.parametrize("silu", [0, 1])
@pytest.mark.parametrize("scale", [1.0, 2.5e5])
def test_groupnorm_bf16(silu, scale):
    """cat(x1 | x2) GroupNorm(32) [+ SiLU]; at scale 2.5e5 the inputs reach ~1e6 (beyond fp16), with a mean offset of
    the same order as the spread."""
    from omg_b200 import ops
    x1 = (rnd(2, 256, 96, seed=20) * scale + 0.5 * scale).to(BF)
    x2 = (rnd(2, 256, 32, seed=21) * scale - 0.3 * scale).to(BF)
    g, b = rnd(128, seed=22, scale=0.1) + 1.0, rnd(128, seed=23, scale=0.1)
    g, b = g.to(BF), b.to(BF)
    got = ops.groupnorm(x1, g, b, 1e-6, silu, x2=x2)
    assert got.dtype == BF and got.shape == (2, 256, 128)
    xc = torch.cat([x1, x2], dim=-1).float().permute(0, 2, 1)
    ref = F.group_norm(xc, 32, g.float(), b.float(), eps=1e-6).permute(0, 2, 1)
    if silu:
        ref = F.silu(ref)
    if scale > 1:
        assert float(torch.cat([x1, x2], -1).float().abs().max()) > 8e5
    err = rel(got, ref)
    print("groupnorm bf16", silu, scale, err)
    assert err < GN_BOUND


@pytest.mark.parametrize("rows,cols,scale", [(7, 64, 1.0), (33, 1024, 0.5), (16, 16384, 0.044), (5, 32768, 1.0)])
def test_softmax_rows_bf16(rows, cols, scale):
    from omg_b200 import ops
    x = rnd(rows, cols, seed=rows + cols, scale=4.0)
    ref = torch.softmax(x.float() * scale, dim=-1)
    big = torch.zeros(rows, cols + 8, dtype=BF, device="cuda")  # strided rows
    big[:, :cols] = x
    ops.softmax_rows(big[:, :cols], scale)
    got = big[:, :cols].float()
    assert (got - ref).abs().max().item() < 8e-3 * ref.max().item() + 1e-6
    assert torch.allclose(got.sum(-1), torch.ones(rows, device="cuda"), atol=1e-2)
    assert float(big[:, cols:].abs().max()) == 0.0


def _vae_case(which, h, w, batch, seed=3):
    from omg_b200 import synthetic
    from omg_b200.vae import VaeConfig
    from oracle import vae as ov
    cfg = VaeConfig.tiny() if which == "tiny" else VaeConfig.sdxl()
    ocfg = ov.VaeConfig(block_out_channels=cfg.block_out_channels)
    sd32 = synthetic.make_vae_state_dict(cfg, seed=seed)
    sd = {k: v.to(BF).float() for k, v in sd32.items()}
    lat = (torch.randn(batch, 4, h, w, generator=torch.Generator().manual_seed(5)) * 0.13025 * 3).to(BF).float()
    return cfg, ocfg, sd32, sd, lat


@pytest.mark.parametrize("which,h,w,batch", [("tiny", 16, 16, 2), ("tiny", 8, 24, 1), ("sdxl", 32, 32, 1)])
def test_decode_bf16_matches_oracle(which, h, w, batch):
    from omg_b200.vae import PackedVaeDecoder
    from oracle import vae as ov
    cfg, ocfg, sd32, sd, lat = _vae_case(which, h, w, batch)
    torch.set_num_threads(32)
    ref = ov.decode(sd, lat, ocfg)
    dec = PackedVaeDecoder(sd, cfg, device="cuda", dtype=BF)
    got = dec.decode(lat.cuda())
    assert got.dtype == BF and got.shape == ref.shape == (batch, 3, 8 * h, 8 * w)
    err = rel(got, ref)
    sd_gpu = {k: v.cuda() for k, v in sd.items()}
    eager = eager_decode(sd_gpu, lat.cuda(), ocfg, BF)
    err_eager = rel(eager, ref)
    err_unrounded = rel(got, ov.decode(sd32, lat, ocfg))  # against the fp32 weights before bf16 rounding (for the docs)
    print(which, h, w, "bf16 decode rel-L2", err, "torch-eager bf16", err_eager, "vs unrounded fp32 weights", err_unrounded)
    assert err < DECODE_BOUND
    assert err <= err_eager  # no worse than the library arithmetic of torch in the same type
    img = dec(lat.cuda(), "pt")
    assert torch.allclose(img.cpu(), ov.postprocess(ref), atol=3e-2)


def _overflow_fixture():
    """The tiny synthetic VAE, bf16-rounded, with conv_in scaled by 2^17: its fp32 output leaves the fp16 range while
    the decoded image (every later GroupNorm renormalises) stays finite."""
    cfg, ocfg, _, sd, lat = _vae_case("tiny", 16, 16, 2)
    for k in ("decoder.conv_in.weight", "decoder.conv_in.bias"):
        sd[k] = sd[k] * 2.0 ** 17
    return cfg, ocfg, sd, lat


def test_overflow_fixture_needs_bf16():
    from omg_b200.vae import PackedVaeDecoder
    from oracle import vae as ov
    cfg, ocfg, sd, lat = _overflow_fixture()
    z = F.conv2d(lat / ocfg.scaling_factor, sd["post_quant_conv.weight"], sd["post_quant_conv.bias"])
    conv_in = F.conv2d(z, sd["decoder.conv_in.weight"], sd["decoder.conv_in.bias"], padding=1)
    assert float(conv_in.abs().max()) > 65504
    ref = ov.decode(sd, lat, ocfg)
    assert bool(torch.isfinite(ref).all())
    with pytest.raises(FloatingPointError, match="bf16"):
        PackedVaeDecoder(sd, cfg, device="cuda")(lat.cuda(), "pt")
    got = PackedVaeDecoder(sd, cfg, device="cuda", dtype=BF).decode(lat.cuda())
    assert bool(torch.isfinite(got).all())
    err = rel(got, ref)
    print("overflow fixture bf16 decode rel-L2", err)
    assert err < DECODE_BOUND


@pytest.mark.parametrize("force_upcast,dtype", [(True, torch.bfloat16), (False, torch.float16)])
def test_from_pretrained_picks_the_type_from_force_upcast(tmp_path, force_upcast, dtype):
    from safetensors.torch import save_file
    from omg_b200.vae import PackedVaeDecoder
    from oracle import vae as ov
    cfg, ocfg, sd, lat = _overflow_fixture()
    save_file({k: v.contiguous() for k, v in sd.items()}, str(tmp_path / "diffusion_pytorch_model.safetensors"))
    with open(tmp_path / "config.json", "w") as f:
        json.dump({"_class_name": "AutoencoderKL", "block_out_channels": list(cfg.block_out_channels), "layers_per_block": 2,
                   "latent_channels": 4, "out_channels": 3, "scaling_factor": cfg.scaling_factor,
                   "force_upcast": force_upcast}, f)
    dec = PackedVaeDecoder.from_pretrained(str(tmp_path), device="cuda")
    assert dec.dtype == dtype and dec.cfg == cfg
    if dtype == torch.bfloat16:
        assert rel(dec.decode(lat.cuda()), ov.decode(sd, lat, ocfg)) < DECODE_BOUND
    else:
        with pytest.raises(FloatingPointError):
            dec(lat.cuda(), "pt")


def test_decode_bf16_is_deterministic():
    from omg_b200.vae import PackedVaeDecoder
    cfg, _, _, sd, lat = _vae_case("tiny", 16, 16, 2)
    dec = PackedVaeDecoder(sd, cfg, device="cuda", dtype=BF)
    a, b = dec.decode(lat.cuda()), dec.decode(lat.cuda())
    assert torch.equal(a, b)


def test_launch_plan_replays_bf16_gemm_groupnorm_softmax():
    from omg_b200 import ops
    x, w, bias = rnd(512, 256, seed=30), rnd(256, 256, seed=31, scale=1 / 16), rnd(256, seed=32)
    g, b = rnd(256, seed=33, scale=0.1) + 1, rnd(256, seed=34, scale=0.1)
    g = g.to(BF)
    y, n = torch.empty(512, 256, dtype=BF, device="cuda"), torch.empty(1, 512, 256, dtype=BF, device="cuda")
    ws = torch.empty(10240 + 64 * 256, device="cuda")
    s = rnd(64, 512, seed=35, scale=4.0)
    s0 = s.clone()
    plan = ops.LaunchPlan()
    with plan:
        ops.linear(x, w, bias=bias, out=y)
        ops.groupnorm(y.view(1, 512, 256), g, b, 1e-6, 1, out=n, stats_ws=ws)
        ops.softmax_rows(s, 0.5)
    assert len(plan) == 3
    torch.cuda.synchronize()
    y1, n1, s1 = y.clone(), n.clone(), s.clone()
    y.zero_()
    n.zero_()
    s.copy_(s0)
    plan.run()
    torch.cuda.synchronize()
    assert torch.equal(y, y1) and torch.equal(n, n1) and torch.equal(s, s1)


def test_pipeline_image_output_with_a_bf16_decoder():
    from omg_b200 import factory, synthetic
    from omg_b200.config import UNetConfig
    from omg_b200.vae import PackedVaeDecoder, VaeConfig
    wl = factory.build_lora_workload(UNetConfig.tiny(), 128, 2, 8, 6, 7.5)
    wl.pipe.vae_decoder = PackedVaeDecoder(synthetic.make_vae_state_dict(VaeConfig.tiny(), 1), VaeConfig.tiny(), dtype=BF)
    kw = dict(wl.call_kwargs)
    kw["output_type"] = "pt"
    lat0 = torch.randn(1, 4, 16, 16, generator=torch.Generator().manual_seed(0)).half()
    out = wl.pipe(stage=1, latents=lat0, **kw).images
    assert out.shape == (2, 3, 128, 128) and float(out.min()) >= 0.0 and float(out.max()) <= 1.0
    assert torch.isfinite(out).all()
