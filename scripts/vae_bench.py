"""VAE decode timing at the bench workload's size: 2 images, 128x128 latents -> 1024x1024, SDXL widths, synthetic
weights.  Prints one JSON line per decode path: ours in each --dtype (fp16, bf16), and torch eager (oracle/vae.py on
the GPU) in fp32 - the reference's up-cast path, with torch's default TF32 settings, recorded in the line - and in
bf16.  Each line: ms per 2-image decode (median of 5 after 2 warm-ups), algorithmic TFLOP/s, peak memory, rel-L2
against the eager fp32 image, and the GPU name and power limit read in the same run."""
import argparse
import json
import subprocess
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, ".")
from omg_b200 import synthetic  # noqa: E402
from omg_b200.vae import PackedVaeDecoder, VaeConfig, vae_decoder_flops  # noqa: E402
from oracle import vae as ov  # noqa: E402

DTYPES = {"fp16": torch.float16, "bf16": torch.bfloat16}


def eager_decode(sd, latents, ocfg, dtype):
    """torch-eager decode with weights and activations in `dtype`: the sequence of oracle.vae.decode over the same
    restatement's blocks (whose arithmetic follows the tensors' type), every intermediate stored in `dtype` - the
    yardstick for a decoder that stores its activations in that type."""
    g = ocfg.norm_num_groups
    sd = {k: v.to(dtype) for k, v in sd.items()}
    z = latents.to(dtype) / ocfg.scaling_factor
    z = F.conv2d(z, sd["post_quant_conv.weight"], sd["post_quant_conv.bias"])
    x = F.conv2d(z, sd["decoder.conv_in.weight"], sd["decoder.conv_in.bias"], padding=1)
    x = ov._res(x, sd, "decoder.mid_block.resnets.0", g)
    x = ov._attn(x, sd, "decoder.mid_block.attentions.0", g)
    x = ov._res(x, sd, "decoder.mid_block.resnets.1", g)
    n_up = len(ocfg.block_out_channels)
    for i in range(n_up):
        for j in range(ocfg.layers_per_block + 1):
            x = ov._res(x, sd, f"decoder.up_blocks.{i}.resnets.{j}", g)
        if i < n_up - 1:
            x = F.interpolate(x, scale_factor=2.0, mode="nearest")
            x = F.conv2d(x, sd[f"decoder.up_blocks.{i}.upsamplers.0.conv.weight"],
                         sd[f"decoder.up_blocks.{i}.upsamplers.0.conv.bias"], padding=1)
    x = ov._gn(x, sd, "decoder.conv_norm_out", g, True)
    return F.conv2d(x, sd["decoder.conv_out.weight"], sd["decoder.conv_out.bias"], padding=1)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                              str(torch.cuda.current_device())], capture_output=True, text=True, check=True).stdout
        name, power = [s.strip() for s in out.strip().split(",")]
    except (OSError, subprocess.CalledProcessError, ValueError):
        name, power = torch.cuda.get_device_name(), "unknown"
    return {"gpu": name, "power_limit": power}


def timed(fn):
    for _ in range(2):
        img = fn()
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    ts = []
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        img = fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    ts.sort()
    return ts[len(ts) // 2], img


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--dtype", nargs="+", choices=sorted(DTYPES), default=["fp16", "bf16"],
                    help="activation types of our decoder to time (the torch-eager fp32 and bf16 paths always run)")
    args = ap.parse_args()
    cfg = VaeConfig.sdxl()
    ocfg = ov.VaeConfig(block_out_channels=cfg.block_out_channels)
    sd = synthetic.make_vae_state_dict(cfg, 0)
    B, h, w = 2, 128, 128
    lat = (torch.randn(B, 4, h, w, generator=torch.Generator().manual_seed(0)) * 0.4).half().cuda()
    fl = B * vae_decoder_flops(cfg, h, w)
    info = gpu_info()
    tf32 = {"cudnn_allow_tf32": torch.backends.cudnn.allow_tf32, "matmul_allow_tf32": torch.backends.cuda.matmul.allow_tf32}
    sd_gpu = {k: v.cuda() for k, v in sd.items()}
    with torch.no_grad():
        ms_ref, ref = timed(lambda: ov.decode(sd_gpu, lat, ocfg))
        mem_ref = torch.cuda.max_memory_allocated()
        ref = ref.float()
        lines = [("torch_eager", "fp32", ms_ref, ref, mem_ref, tf32)]
        ms, img = timed(lambda: eager_decode(sd_gpu, lat, ocfg, torch.bfloat16))
        lines.append(("torch_eager", "bf16", ms, img, torch.cuda.max_memory_allocated(), tf32))
        del img
        for name in args.dtype:
            dec = PackedVaeDecoder(sd, cfg, dtype=DTYPES[name])
            ms, img = timed(lambda: dec.decode(lat))
            lines.append(("ours", name, ms, img, torch.cuda.max_memory_allocated(), {}))
            del dec
    for impl, dt, ms, img, mem, extra in lines:
        err = ((img.float() - ref).norm() / ref.norm()).item()
        print(json.dumps({"name": "vae_decode_2x1024", "impl": impl, "dtype": dt, "ms": round(ms, 3),
                          "tflops": round(fl / ms / 1e9, 1), "algorithmic_tflop": round(fl / 1e12, 2),
                          "finite": bool(torch.isfinite(img).all()), "rel_l2_vs_eager_fp32": float(f"{err:.3e}"),
                          "peak_mem_gb": round(mem / 2 ** 30, 2), **extra, **info}), flush=True)


if __name__ == "__main__":
    main()
