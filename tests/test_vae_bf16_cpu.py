"""CPU side of the VAE decoder's bf16 path: the `dtype` field of omg_gemm_desc sits where the ctypes mirror puts it, the
C ABI refuses what bf16 mode does not support before touching a GPU, both CLIs parse --vae, and the decoder's config
and decode type come from `config.json` or the parameter shapes."""
import ctypes
import importlib.util
import os
import shutil
import subprocess
import sys
import tempfile

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def test_dtype_field_offset_matches_the_c_layout():
    from omg_b200 import _lib as L
    cc = shutil.which("gcc") or shutil.which("cc")
    if cc is None:
        pytest.skip("no C compiler")
    src = ('#include <stddef.h>\n#include <stdio.h>\n#include "omg_b200.h"\n'
           'int main(void) { printf("%d %d %d %d\\n", (int)offsetof(omg_gemm_desc, dtype), (int)sizeof(omg_gemm_desc), '
           'OMG_DTYPE_F16, OMG_DTYPE_BF16); return 0; }\n')
    with tempfile.TemporaryDirectory() as tmp:
        c, exe = os.path.join(tmp, "probe.c"), os.path.join(tmp, "probe")
        with open(c, "w") as f:
            f.write(src)
        subprocess.run([cc, "-std=c99", "-pedantic", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), c, "-o", exe],
                       check=True)
        off, size, f16, bf16 = [int(v) for v in subprocess.run([exe], capture_output=True, text=True, check=True).stdout.split()]
    assert off == L.GemmDesc.dtype.offset and size == ctypes.sizeof(L.GemmDesc)
    assert (f16, bf16) == (L.DTYPE_F16, L.DTYPE_BF16) == (0, 1)
    assert L.GemmDesc().dtype == L.DTYPE_F16  # a zeroed descriptor keeps the fp16 behaviour


def test_c_abi_refuses_what_bf16_mode_does_not_support():
    """Each refusal names the feature; none of these calls reaches a CUDA API (pointers are never dereferenced)."""
    import ctypes as C
    from omg_b200 import _lib as L
    lib = L.load()

    def err(**fields):
        g = L.GemmDesc()
        g.dtype = L.DTYPE_BF16
        for k, v in fields.items():
            setattr(g, k, v)
        assert lib.omg_gemm(C.byref(g), None) == 1
        return lib.omg_last_error().decode()

    assert "unknown dtype 7" in err(dtype=7)
    for epi in (L.EPI_GEGLU, L.EPI_SILU, L.EPI_QUICK_GELU, L.EPI_GELU, L.EPI_GELU_TANH):
        assert "epilogue activation" in err(epilogue=epi)
    assert "folded LayerNorm (row_stats_*)" in err(row_stats_out=0x1000)
    assert "folded LayerNorm (row_stats_*)" in err(row_stats_in=0x1000)
    assert "col_stats_out" in err(col_stats_out=0x1000)
    assert "rowvec" in err(rowvec=0x1000)
    assert "weight planes or column groups" in err(w_group_planes=2, n_col_groups=2)
    assert "weight planes or column groups" in err(n_col_groups=2)
    assert "fp32 twins" in err(residual_f32=0x1000)
    assert "fp32 twins" in err(out_f32=0x1000)
    fake = C.c_void_p(0x1000)
    assert lib.omg_groupnorm_bf16(fake, 100, None, 0, 1, 16, fake, fake, 1e-6, 0, fake, fake, None) == 1
    assert "omg_groupnorm_bf16: bad channel split" in lib.omg_last_error().decode()
    assert lib.omg_softmax_rows_bf16(fake, 4, 12, 16, 1.0, None) == 1
    assert "omg_softmax_rows_bf16" in lib.omg_last_error().decode()


def _parse(fname, argv):
    spec = importlib.util.spec_from_file_location("cli_" + fname[:-3], os.path.join(ROOT, fname))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    old, sys.argv = sys.argv, [fname, *argv]
    try:
        return vars(mod.parse_args())
    finally:
        sys.argv = old


@pytest.mark.parametrize("fname", ["inference_lora.py", "inference_instantid.py"])
def test_clis_parse_vae(fname):
    assert _parse(fname, [])["vae"] == ""
    assert _parse(fname, ["--vae", "/ckpt/sdxl"])["vae"] == "/ckpt/sdxl"


def test_lora_cli_vae_and_vae_fp16_safe_are_mutually_exclusive():
    assert _parse("inference_lora.py", ["--vae_fp16_safe", "/ckpt/vae-fp16-fix"])["vae_fp16_safe"] == "/ckpt/vae-fp16-fix"
    with pytest.raises(SystemExit):
        _parse("inference_lora.py", ["--vae", "/a", "--vae_fp16_safe", "/b"])


def _meta_state_dict(cfg):
    from omg_b200.vae import vae_decoder_param_shapes
    return {k: torch.empty(s, device="meta") for k, s in vae_decoder_param_shapes(cfg).items()}


@pytest.mark.parametrize("which", ["sdxl", "tiny"])
def test_config_inferred_from_parameter_shapes(which):
    from omg_b200.vae import VaeConfig, vae_config_from
    cfg = VaeConfig.sdxl() if which == "sdxl" else VaeConfig.tiny()
    got, dtype = vae_config_from(_meta_state_dict(cfg))
    assert got == cfg and dtype == torch.bfloat16


def test_config_from_config_json():
    from omg_b200.vae import VaeConfig, vae_config_from
    sd = _meta_state_dict(VaeConfig.tiny())
    conf = {"_class_name": "AutoencoderKL", "block_out_channels": [64, 64, 128, 128], "layers_per_block": 2,
            "latent_channels": 4, "out_channels": 3, "scaling_factor": 0.5, "force_upcast": True}
    cfg, dtype = vae_config_from(sd, conf)
    assert cfg == VaeConfig(block_out_channels=(64, 64, 128, 128), scaling_factor=0.5) and dtype == torch.bfloat16
    assert vae_config_from(sd, dict(conf, force_upcast=False))[1] == torch.float16
    del conf["force_upcast"]  # diffusers' default for AutoencoderKL is force_upcast=True
    assert vae_config_from(sd, conf)[1] == torch.bfloat16


def test_eager_yardstick_follows_the_oracle():
    """scripts/vae_bench.eager_decode, the torch-eager bf16 yardstick of the GPU tests, is the oracle's decode sequence:
    in fp32 it reproduces oracle.vae.decode exactly."""
    from omg_b200 import synthetic
    from omg_b200.vae import VaeConfig
    from oracle import vae as ov
    from scripts.vae_bench import eager_decode
    cfg = VaeConfig.tiny()
    ocfg = ov.VaeConfig(block_out_channels=cfg.block_out_channels)
    sd = synthetic.make_vae_state_dict(cfg, seed=3)
    lat = torch.randn(1, 4, 4, 4, generator=torch.Generator().manual_seed(5)) * 0.4
    assert torch.equal(eager_decode(sd, lat, ocfg, torch.float32), ov.decode(sd, lat, ocfg))
    assert eager_decode(sd, lat, ocfg, torch.bfloat16).dtype == torch.bfloat16
