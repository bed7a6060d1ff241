"""SDXL VAE decoder on the B200 kernels (SURVEY 8f-1: the step right after the denoising loop,
src/pipelines/lora_pipeline.py:634-661: `image = vae.decode(latents / scaling_factor)` + postprocess).

Everything runs through the same C-ABI kernels as the UNet: channels-last fp16 activations, 3x3 convs as implicit
GEMMs (`omg_gemm`: 9 shifted TMA reads, the 1x1 `conv_shortcut` as an extra K-segment of conv2, residual add in the
epilogue, nearest-2x upsample + conv as four phase convs without the upsampled tensor), GroupNorm(32, eps 1e-6)[+SiLU]
(`omg_groupnorm`).  The mid-block attention is one head of 512 channels - outside the flash kernel's head_dim 64 - and
runs as scores = omg_gemm(Q, K), `omg_softmax_rows`, out = omg_gemm(P, V^T): 512 MB of scores per 1024^2 image, two
550 GFLOP GEMMs.  `post_quant_conv` (1x1, 4 -> 4) carries the 1 / scaling_factor and is padded to the 8-channel
granularity of the TMA path.

Precision: fp16 or bf16 storage, fp32 accumulation.  The reference up-casts this module to fp32 because the original
SDXL VAE weights overflow fp16 activations (the VAE config's `force_upcast`, lora_pipeline.py:635-646).  bf16 has
fp32's exponent range, so `PackedVaeDecoder(..., dtype=torch.bfloat16)` decodes those weights with the same kernels
(bf16 operands on the same tensor-core path; fp32 GroupNorm statistics); fp16 (the default) suits the fp16-safe
re-export of the weights and is a little more accurate.  `PackedVaeDecoder.from_pretrained` picks the type from
`force_upcast`, the signal the reference uses for its fp32 up-cast.
"""
import json
import os
from dataclasses import dataclass
from typing import Dict, Optional, Tuple

import torch

from . import ops


@dataclass(frozen=True)
class VaeConfig:
    block_out_channels: Tuple[int, ...] = (128, 256, 512, 512)
    layers_per_block: int = 2
    latent_channels: int = 4
    out_channels: int = 3
    scaling_factor: float = 0.13025

    @staticmethod
    def sdxl() -> "VaeConfig":
        return VaeConfig()

    @staticmethod
    def tiny() -> "VaeConfig":
        return VaeConfig(block_out_channels=(64, 64, 128, 128))


def vae_config_from(sd: Dict[str, torch.Tensor], config: Optional[dict] = None) -> Tuple[VaeConfig, torch.dtype]:
    """(VaeConfig, activation dtype) of a diffusers AutoencoderKL: from its `config.json` dict when given (widths,
    `scaling_factor`; `force_upcast`, diffusers' default true, selects bf16 and false fp16), else inferred from the
    decoder's parameter shapes, with `VaeConfig`'s scaling factor and bf16 (the type that holds any SDXL VAE)."""
    if config is not None:
        d = VaeConfig()
        cfg = VaeConfig(block_out_channels=tuple(config.get("block_out_channels", d.block_out_channels)),
                        layers_per_block=int(config.get("layers_per_block", d.layers_per_block)),
                        latent_channels=int(config.get("latent_channels", d.latent_channels)),
                        out_channels=int(config.get("out_channels", d.out_channels)),
                        scaling_factor=float(config.get("scaling_factor", d.scaling_factor)))
        return cfg, (torch.bfloat16 if config.get("force_upcast", True) else torch.float16)
    n_up = 1 + max(int(k.split(".")[2]) for k in sd if k.startswith("decoder.up_blocks."))
    # up block i runs at width block_out_channels[n_up - 1 - i]
    rev = [sd[f"decoder.up_blocks.{i}.resnets.0.conv1.weight"].shape[0] for i in range(n_up)]
    n_res = 1 + max(int(k.split(".")[4]) for k in sd if k.startswith("decoder.up_blocks.0.resnets."))
    cfg = VaeConfig(block_out_channels=tuple(reversed(rev)), layers_per_block=n_res - 1,
                    latent_channels=sd["post_quant_conv.weight"].shape[0], out_channels=sd["decoder.conv_out.weight"].shape[0])
    return cfg, torch.bfloat16


def vae_decoder_param_shapes(cfg: VaeConfig) -> Dict[str, Tuple[int, ...]]:
    """Parameter name -> shape of `post_quant_conv` + `decoder.*` in the diffusers AutoencoderKL key layout."""
    S: Dict[str, Tuple[int, ...]] = {}

    def conv(n, i, o, k):
        S[n + ".weight"], S[n + ".bias"] = (o, i, k, k), (o,)

    def norm(n, c):
        S[n + ".weight"], S[n + ".bias"] = (c,), (c,)

    def res(n, i, o):
        norm(n + ".norm1", i)
        conv(n + ".conv1", i, o, 3)
        norm(n + ".norm2", o)
        conv(n + ".conv2", o, o, 3)
        if i != o:
            conv(n + ".conv_shortcut", i, o, 1)

    top = cfg.block_out_channels[-1]
    conv("post_quant_conv", cfg.latent_channels, cfg.latent_channels, 1)
    conv("decoder.conv_in", cfg.latent_channels, top, 3)
    res("decoder.mid_block.resnets.0", top, top)
    a = "decoder.mid_block.attentions.0"
    norm(a + ".group_norm", top)
    for proj in ("to_q", "to_k", "to_v", "to_out.0"):
        S[f"{a}.{proj}.weight"], S[f"{a}.{proj}.bias"] = (top, top), (top,)
    res("decoder.mid_block.resnets.1", top, top)
    prev = top
    rev = tuple(reversed(cfg.block_out_channels))
    for i, ch in enumerate(rev):
        for j in range(cfg.layers_per_block + 1):
            res(f"decoder.up_blocks.{i}.resnets.{j}", prev if j == 0 else ch, ch)
        if i < len(rev) - 1:
            conv(f"decoder.up_blocks.{i}.upsamplers.0.conv", ch, ch, 3)
        prev = ch
    norm("decoder.conv_norm_out", cfg.block_out_channels[0])
    conv("decoder.conv_out", cfg.block_out_channels[0], cfg.out_channels, 3)
    return S


def vae_decoder_flops(cfg: VaeConfig, h: int, w: int) -> float:
    """2*MAC of every conv / linear + 4*N*N*C of the mid attention for one image at latent h x w."""
    total = 0.0
    n_up = len(cfg.block_out_channels)
    for name, shape in vae_decoder_param_shapes(cfg).items():
        if not name.endswith(".weight") or len(shape) < 2:
            continue
        if name.startswith("decoder.up_blocks."):
            scale = 2 ** int(name.split(".")[2]) * (2 if ".upsamplers." in name else 1)
        elif name.startswith("decoder.conv_out"):
            scale = 2 ** (n_up - 1)
        else:
            scale = 1
        k = shape[2] * shape[3] if len(shape) == 4 else 1
        total += 2.0 * (h * scale) * (w * scale) * shape[0] * shape[1] * k
    return total + 4.0 * (h * w) ** 2 * cfg.block_out_channels[-1]


class PackedVaeDecoder:
    """Weights of `post_quant_conv` + `decoder.*` (diffusers AutoencoderKL key layout) repacked once for the kernels.
    `dtype` (fp16 | bf16) is the type the weights are packed in and the activations are decoded in."""

    def __init__(self, state_dict: Dict[str, torch.Tensor], cfg: VaeConfig = VaeConfig(), device="cuda",
                 dtype: torch.dtype = torch.float16):
        self.cfg, self.device, self.dtype = cfg, torch.device(device), dtype
        if self.device.type != "cuda":
            raise RuntimeError("the B200 path needs a CUDA device (there is no CPU fallback)")
        if dtype not in (torch.float16, torch.bfloat16):
            raise ValueError(f"the VAE decoder runs fp16 or bf16, not {dtype}")
        sd = {k: v.float() for k, v in state_dict.items() if k.startswith(("decoder.", "post_quant_conv."))}
        dev, p = self.device, {}
        self.p = p

        def _cast(t, dev):  # packed in the decode type (fp16 | bf16)
            return t.to(device=dev, dtype=dtype).contiguous()

        def conv(name, pad_in=0, pad_out=0):
            w, b = sd[name + ".weight"], sd[name + ".bias"]
            if pad_in:
                w = torch.cat([w, w.new_zeros(w.shape[0], pad_in, 3, 3)], dim=1)
            if pad_out:
                w = torch.cat([w, w.new_zeros(pad_out, *w.shape[1:])], dim=0)
                b = torch.cat([b, b.new_zeros(pad_out)])
            return ops.pack_conv3x3_weight(w), b

        def res(name):
            for i in ("1", "2"):
                p[f"{name}.g{i}"] = _cast(sd[f"{name}.norm{i}.weight"], dev)
                p[f"{name}.b{i}"] = _cast(sd[f"{name}.norm{i}.bias"], dev)
            w1, b1 = conv(name + ".conv1")
            w2, b2 = conv(name + ".conv2")
            if name + ".conv_shortcut.weight" in sd:  # 1x1 shortcut: extra K columns of conv2, biases summed
                w2 = torch.cat([w2, sd[name + ".conv_shortcut.weight"].flatten(1)], dim=1)
                b2 = b2 + sd[name + ".conv_shortcut.bias"]
            p[name + ".w1"], p[name + ".bias1"] = _cast(w1, dev), _cast(b1, dev)
            p[name + ".w2"], p[name + ".bias2"] = _cast(w2, dev), _cast(b2, dev)

        lc = cfg.latent_channels
        pad = (-lc) % 8
        # post_quant_conv with 1 / scaling_factor folded in, padded to 8 x 8 (zero rows / columns)
        wpq = torch.zeros(lc + pad, lc + pad)
        wpq[:lc, :lc] = sd["post_quant_conv.weight"].flatten(1) / cfg.scaling_factor
        bpq = torch.zeros(lc + pad)
        bpq[:lc] = sd["post_quant_conv.bias"]
        p["pq.w"], p["pq.b"] = _cast(wpq, dev), _cast(bpq, dev)
        w, b = conv("decoder.conv_in", pad_in=pad)
        p["conv_in.w"], p["conv_in.b"] = _cast(w, dev), _cast(b, dev)
        top = cfg.block_out_channels[-1]
        res("decoder.mid_block.resnets.0")
        a = "decoder.mid_block.attentions.0"
        p["attn.g"], p["attn.b"] = _cast(sd[a + ".group_norm.weight"], dev), _cast(sd[a + ".group_norm.bias"], dev)
        s = top ** -0.5  # softmax scale folded into the query projection
        p["attn.wqkv"] = _cast(torch.cat([sd[a + ".to_q.weight"] * s, sd[a + ".to_k.weight"], sd[a + ".to_v.weight"]]), dev)
        p["attn.bqkv"] = _cast(torch.cat([sd[a + ".to_q.bias"] * s, sd[a + ".to_k.bias"], sd[a + ".to_v.bias"]]), dev)
        p["attn.wo"], p["attn.bo"] = _cast(sd[a + ".to_out.0.weight"], dev), _cast(sd[a + ".to_out.0.bias"], dev)
        res("decoder.mid_block.resnets.1")
        self.n_up = len(cfg.block_out_channels)
        for i in range(self.n_up):
            for j in range(cfg.layers_per_block + 1):
                res(f"decoder.up_blocks.{i}.resnets.{j}")
            if i < self.n_up - 1:
                w, b = conv(f"decoder.up_blocks.{i}.upsamplers.0.conv")
                p[f"up{i}.w"], p[f"up{i}.b"] = _cast(w, dev), _cast(b, dev)
        p["out.g"], p["out.b"] = _cast(sd["decoder.conv_norm_out.weight"], dev), _cast(sd["decoder.conv_norm_out.bias"], dev)
        w, b = conv("decoder.conv_out", pad_out=(-cfg.out_channels) % 8)
        p["conv_out.w"], p["conv_out.b"] = _cast(w, dev), _cast(b, dev)
        self._ws = None

    @classmethod
    def from_pretrained(cls, path: str, device="cuda") -> "PackedVaeDecoder":
        """A diffusers VAE directory (`config.json` + `diffusion_pytorch_model[.fp16].safetensors`), or a checkpoint root
        with a `vae/` subfolder.  The decode type follows the config's `force_upcast` (see `vae_config_from`)."""
        from .checkpoints import load_unet_weights
        sub = "vae" if os.path.isdir(os.path.join(path, "vae")) else ""
        sd = load_unet_weights(path, subfolder=sub)
        cfg_path = os.path.join(path, sub, "config.json")
        config = None
        if os.path.isfile(cfg_path):
            with open(cfg_path) as f:
                config = json.load(f)
        cfg, dtype = vae_config_from(sd, config)
        return cls(sd, cfg, device=device, dtype=dtype)

    # ------------------------------------------------------------------------------------------------ blocks
    def _stats_ws(self, B):
        n = B * (10240 + 64 * 256)  # OMG_GN_WS_FLOATS(B)
        if self._ws is None or self._ws.numel() < n:
            self._ws = torch.empty(n, dtype=torch.float32, device=self.device)
        return self._ws

    def _res(self, name, x):
        p = self.p
        ws = self._stats_ws(x.shape[0])
        a1 = ops.groupnorm(x, p[name + ".g1"], p[name + ".b1"], 1e-6, 1, stats_ws=ws)
        h = ops.conv3x3(a1, p[name + ".w1"], bias=p[name + ".bias1"])
        del a1
        a2 = ops.groupnorm(h, p[name + ".g2"], p[name + ".b2"], 1e-6, 1, stats_ws=ws, out=h)
        cout = p[name + ".bias1"].shape[0]
        if p[name + ".w2"].shape[1] > 9 * cout:
            return ops.conv3x3(a2, p[name + ".w2"], bias=p[name + ".bias2"], shortcut=[(x, 9 * cout)])
        return ops.conv3x3(a2, p[name + ".w2"], bias=p[name + ".bias2"], residual=x)

    def _attention(self, x):
        p = self.p
        B, H, W, C = x.shape
        N = H * W
        n = ops.groupnorm(x, p["attn.g"], p["attn.b"], 1e-6, 0, stats_ws=self._stats_ws(B))
        qkv = ops.linear(n.view(B * N, C), p["attn.wqkv"], bias=p["attn.bqkv"]).view(B, N, 3 * C)
        o = torch.empty((B, N, C), dtype=x.dtype, device=x.device)
        scores = torch.empty((N, N), dtype=x.dtype, device=x.device)
        for b in range(B):  # one image at a time: the score matrix is N x N (512 MB at 128 x 128 latents)
            q, k, v = qkv[b, :, :C], qkv[b, :, C:2 * C], qkv[b, :, 2 * C:]
            ops.linear(q.contiguous(), k.contiguous(), out=scores)   # (Q / sqrt(C)) K^T
            ops.softmax_rows(scores, 1.0)
            ops.linear(scores, v.t().contiguous(), out=o[b])         # P V
        out = torch.empty_like(x)
        ops.linear(o.view(B * N, C), p["attn.wo"], bias=p["attn.bo"], residual=x.view(B * N, C), out=out.view(B * N, C))
        return out

    # ------------------------------------------------------------------------------------------------ decode
    @torch.no_grad()
    def decode(self, latents: torch.Tensor) -> torch.Tensor:
        """(B, 4, h, w) latents (as the pipelines return them) -> (B, 3, 8h, 8w) image in the decode type, nominally in
        [-1, 1]."""
        cfg, p = self.cfg, self.p
        B, lc, h, w = latents.shape
        pad = (-lc) % 8
        z = torch.zeros((B, h, w, lc + pad), dtype=self.dtype, device=self.device)
        z[..., :lc] = latents.to(self.device).permute(0, 2, 3, 1)
        z = ops.linear(z.view(B * h * w, lc + pad), p["pq.w"], bias=p["pq.b"]).view(B, h, w, lc + pad)
        x = ops.conv3x3(z, p["conv_in.w"], bias=p["conv_in.b"])
        x = self._res("decoder.mid_block.resnets.0", x)
        x = self._attention(x)
        x = self._res("decoder.mid_block.resnets.1", x)
        for i in range(self.n_up):
            for j in range(cfg.layers_per_block + 1):
                x = self._res(f"decoder.up_blocks.{i}.resnets.{j}", x)
            if i < self.n_up - 1:
                x = ops.upsample2x_conv3x3(x, p[f"up{i}.w"], bias=p[f"up{i}.b"])
        x = ops.groupnorm(x, p["out.g"], p["out.b"], 1e-6, 1, stats_ws=self._stats_ws(B), out=x)
        img = ops.conv3x3(x, p["conv_out.w"], bias=p["conv_out.b"])
        return img[..., :cfg.out_channels].permute(0, 3, 1, 2)

    def __call__(self, latents: torch.Tensor, output_type: str = "pt"):
        """The pipelines' `vae_decoder(latents, output_type)`: VaeImageProcessor.postprocess [3P] - denormalise to
        [0, 1]; 'pt' tensor (B,3,H,W), 'np' array (B,H,W,3), 'pil' list of images."""
        dec = self.decode(latents).float()
        if not bool(torch.isfinite(dec).all()):
            # fp16 activations overflow with the original SDXL VAE weights (the reference up-casts this module to
            # fp32 for that reason, lora_pipeline.py:635-646): refuse to hand back NaN / black images
            if self.dtype == torch.float16:
                raise FloatingPointError("VAE decode produced non-finite values in fp16: decode in bf16 "
                                         "(PackedVaeDecoder(..., dtype=torch.bfloat16), or from_pretrained on a VAE whose "
                                         "config has force_upcast), use the fp16-safe SDXL VAE weights (same keys), or "
                                         "output_type='latent'")
            raise FloatingPointError("VAE decode produced non-finite values in bf16")
        img = (dec / 2 + 0.5).clamp(0, 1)
        if output_type == "pt":
            return img
        arr = img.permute(0, 2, 3, 1).cpu().numpy()
        if output_type == "np":
            return arr
        if output_type == "pil":
            from PIL import Image
            return [Image.fromarray((a * 255).round().astype("uint8")) for a in arr]
        raise ValueError(f"unknown output_type {output_type}")
