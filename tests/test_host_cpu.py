"""CPU tests: the C-ABI library loads and exports every declared symbol, host-side logic (prompt-to-prompt tables,
schedule, masks, config arithmetic, LoRA packing) and the 2-rank gloo path of the data-parallel plumbing."""
import ctypes
import math
import os
import re
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
from make_golden import ToyTokenizer  # noqa: E402


def test_library_exports_every_declared_symbol():
    from omg_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "omg_b200.h")).read()
    declared = set(re.findall(r"\b(omg_[a-z0-9_]+)\s*\(", hdr))
    declared = {d for d in declared if not d.endswith("_desc")}
    assert {"omg_gemm", "omg_attention", "omg_groupnorm", "omg_layernorm", "omg_fuse_step", "omg_ctx_mix", "omg_axpy",
            "omg_last_error", "omg_version", "omg_launch_count"} <= declared
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), f"{name} not exported"
    assert set(_lib.SYMBOLS) == declared
    l2 = _lib.load()
    assert l2.omg_version().decode().startswith("omg_b200")
    # the launch counter of a freshly loaded library starts at zero; a new interpreter, because GPU tests earlier in
    # this process may already have launched kernels through the same library
    import subprocess
    code = f"import sys; sys.path.insert(0, {ROOT!r}); from omg_b200 import _lib; print(_lib.load().omg_launch_count())"
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, check=True)
    assert int(r.stdout) == 0


def test_header_is_plain_c99_and_matches_the_ctypes_layout():
    """include/omg_b200.h compiles as C99 (no C++, no CUDA headers: the boundary is plain pointers and sizes) and the
    descriptor sizes the C compiler sees are the ones the ctypes binding uses."""
    import shutil
    import subprocess
    import tempfile
    from omg_b200 import _lib as L
    cc = shutil.which("gcc") or shutil.which("cc")
    if cc is None:
        pytest.skip("no C compiler")
    with tempfile.TemporaryDirectory() as tmp:
        exe = os.path.join(tmp, "abi_check")
        subprocess.run([cc, "-std=c99", "-pedantic", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"),
                        os.path.join(ROOT, "tests", "c_host", "abi_check.c"), "-o", exe], check=True)
        sizes = [int(v) for v in subprocess.run([exe], capture_output=True, text=True, check=True).stdout.split()]
    assert sizes == [ctypes.sizeof(t) for t in (L.View4, L.Seg, L.GemmDesc, L.AttnDesc, L.FuseDesc)]


def test_launch_plan_handle_protocol():
    """omg_plan_* (the forward-as-a-handle boundary): create / record / run / destroy and their error strings; no launch
    entry point is called, so nothing here needs a GPU."""
    from omg_b200 import _lib as L
    from omg_b200 import ops
    lib = L.load()
    plan = ops.LaunchPlan()
    assert len(plan) == 0
    plan.run(0)                                              # an empty plan runs (no CUDA call behind it)
    with plan:
        with pytest.raises(RuntimeError, match="already recording"):
            ops.LaunchPlan().__enter__()                     # one recording per thread
        assert lib.omg_plan_run(plan._h, None) == 1 and b"still being recorded" in lib.omg_last_error()
        assert lib.omg_plan_clear(plan._h) == 1
        # a call that fails validation is not recorded
        assert lib.omg_gemm(None, None) == 1
    assert len(plan) == 0
    assert lib.omg_plan_record_end(plan._h) == 1 and b"not being recorded" in lib.omg_last_error()
    assert lib.omg_plan_length(None) == -1
    assert lib.omg_plan_run(None, None) == 1 and b"null plan" in lib.omg_last_error()
    plan.clear()


def test_struct_sizes_match_c_layout():
    """ctypes mirrors of the descriptors must have the C sizes (checked against a compile-time table)."""
    from omg_b200 import _lib
    assert ctypes.sizeof(_lib.View4) == 48
    assert ctypes.sizeof(_lib.Seg) == 28
    assert ctypes.sizeof(_lib.GemmDesc) % 8 == 0
    assert ctypes.sizeof(_lib.AttnDesc) % 8 == 0


def test_no_cpu_fallback():
    from omg_b200 import ops
    with pytest.raises(ValueError):
        ops.linear(torch.zeros(8, 8), torch.zeros(8, 8))


def test_p2p_tables_match_reference_golden():
    from omg_b200.prompt_attention import AttentionReplace
    G = os.path.join(ROOT, "tests", "golden")
    d = torch.load(os.path.join(G, "p2p_same.pt"))
    c = AttentionReplace(d["prompts"], 50, {"default_": 1.0}, 0.4, 4, 4, tokenizer=ToyTokenizer())
    assert torch.equal(c.cross_replace_alpha, d["alpha"]) and torch.equal(c.mapper, d["mapper"])
    assert c.num_self_replace == (0, 20)
    d = torch.load(os.path.join(G, "p2p_edit.pt"))
    c = AttentionReplace(d["prompts"], d["num_steps"], dict(d["cross"]), d["self"], 4, 4, tokenizer=ToyTokenizer())
    assert torch.equal(c.cross_replace_alpha, d["alpha"]) and torch.equal(c.mapper, d["mapper"])
    with pytest.raises(ValueError):
        AttentionReplace(["a b c", "a b"], 10, 1.0, 0.4, 4, 4, tokenizer=ToyTokenizer())


def test_p2p_counters_and_edit_spec():
    from omg_b200.prompt_attention import AttentionReplace
    c = AttentionReplace(["x y"] * 2, 50, {"default_": 1.0}, 0.4, 32, 32)
    c.num_att_layers = 140
    assert c.self_replace_active(1024) and not c.self_replace_active(4096)
    c.advance(139)
    assert (c.cur_step, c.cur_att_layer) == (0, 139)
    c.advance(1)
    assert (c.cur_step, c.cur_att_layer) == (1, 0)
    c.advance(140 * 19)
    assert c.cur_step == 20 and not c.self_replace_active(1024)
    base, keep = c.cross_edit()
    assert torch.equal(base, torch.eye(77)) and keep is None
    c.reset()
    assert (c.cur_step, c.cur_att_layer) == (0, 0)
    with pytest.raises(RuntimeError):
        c(torch.zeros(4, 2, 2), True, "mid")
    c.cur_step = 51
    with pytest.raises(IndexError):
        c.cross_edit()


def test_cross_edit_equals_probability_edit():
    """P0 (M diag(a) V) + P1 (diag(1-a) V) == ((P0 M) * a + (1-a) * P1) V for the reference's edit."""
    from omg_b200.prompt_attention import AttentionReplace
    c = AttentionReplace(["a photo of a man", "a photo of a dog"], 10, {"default_": 0.6, "dog": (0.2, 0.9)}, 0.3, 4, 4,
                         tokenizer=ToyTokenizer())
    g = torch.Generator().manual_seed(0)
    for step in (0, 2, 7, 9):
        c.cur_step = step
        base, keep = c.cross_edit()
        P0 = torch.softmax(torch.randn(5, 77, generator=g), -1)
        P1 = torch.softmax(torch.randn(5, 77, generator=g), -1)
        V = torch.randn(77, 16, generator=g)
        alpha = c.cross_replace_alpha[step, 0, 0, 0]
        ref = ((P0 @ c.mapper[0]) * alpha + (1 - alpha) * P1) @ V
        mine = P0 @ (base @ V) + (P1 @ (keep @ V) if keep is not None else 0)
        assert torch.allclose(mine, ref, atol=1e-5)


def test_schedule_matches_published_sdxl_values():
    from omg_b200.scheduler import EulerDiscreteSchedule
    s = EulerDiscreteSchedule()
    ts = s.set_timesteps(30)
    assert ts[0] == 958.0 and ts[-1] == 1.0 and s.sigmas[-1] == 0.0
    sig_max = math.sqrt((1 - s.alphas_cumprod[-1]) / s.alphas_cumprod[-1])
    assert abs(sig_max - 14.6146) < 1e-3
    assert abs(s.init_noise_sigma - math.sqrt(s.sigmas[0] ** 2 + 1)) < 1e-6
    assert np.all(np.diff(s.sigmas) < 0)


def test_config_arithmetic():
    from omg_b200.config import UNetConfig, lora_target_names, param_shapes, unet_flops
    cfg = UNetConfig.sdxl()
    assert sum(math.prod(v) for v in param_shapes(cfg).values()) == 2_567_463_684
    assert abs(unet_flops(cfg, 128, 128) / 1e12 - 6.761) < 2e-3
    assert len(lora_target_names(cfg)) == 722


def test_latent_mask_is_nearest_and_binary():
    from omg_b200.pipelines import _binary_latent_mask
    m = torch.zeros(64, 64)
    m[8:24, 16:40] = 1
    m[40, 40] = 0.5
    out = _binary_latent_mask(m, 8, 8, "cpu").reshape(8, 8)
    ref = (torch.nn.functional.interpolate(m[None, None], size=(8, 8), mode="nearest")[0, 0] == 1).float()
    assert torch.equal(out, ref) and out.sum() == 6
    assert _binary_latent_mask(None, 8, 8, "cpu") is None


def _dp_worker(rank, world, port, q):
    import torch.distributed as dist
    from omg_b200.distributed import broadcast_state_dict, gather_latents, shard_indices
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    sd = {"b": torch.full((3,), float(rank)), "a": torch.arange(4.0) * (rank + 1)}
    broadcast_state_dict(sd, 0)
    # the form bench.py uses: rank 0 packs its weights into ONE flat buffer, the others receive into an empty one
    from omg_b200.distributed import broadcast_flat, empty_flat_state_dict, flat_layout, flatten_state_dict
    shapes = {"w": (5, 3), "v": (7,), "u": (2, 2, 2)}
    if rank == 0:
        src = {k: torch.arange(float(torch.tensor(shp).prod())).reshape(shp) + i for i, (k, shp) in enumerate(shapes.items())}
        flat, views = flatten_state_dict(src, dtype=torch.float32)
    else:
        flat, views = empty_flat_state_dict(shapes, "cpu", dtype=torch.float32)
    broadcast_flat(flat, 0)
    layout, total = flat_layout(shapes)
    assert flat.numel() == total and all(off % 128 == 0 for off, _ in layout.values())
    for i, (k, shp) in enumerate(shapes.items()):
        assert torch.equal(views[k], torch.arange(float(torch.tensor(shp).prod())).reshape(shp) + i)
    n = 5
    idx = shard_indices(n, rank, world)
    local = torch.stack([torch.full((2, 2), float(j)) for j in idx])
    allv = gather_latents(local, n)
    q.put((rank, sd["a"].tolist(), sd["b"].tolist(), allv[:, 0, 0].tolist(), idx))
    dist.barrier()
    dist.destroy_process_group()


def test_data_parallel_plumbing_gloo_world2():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() % 1000)
    procs = [ctx.Process(target=_dp_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=120) for _ in range(2))
    for p in procs:
        p.join(timeout=60)
    for rank, a, b, allv, idx in res:
        assert a == [0.0, 1.0, 2.0, 3.0] and b == [0.0, 0.0, 0.0]      # rank 0's weights everywhere
        assert allv == [0.0, 1.0, 2.0, 3.0, 4.0]                       # image order restored
    assert res[0][4] == [0, 2, 4] and res[1][4] == [1, 3]


def test_gemm_plan_tile_choice_is_host_logic_and_stable():
    """omg_gemm_plan runs without a GPU: the wave-quantisation cost model behind the tile shape, and the number of
    LayerNorm-statistics partials (2 per n-tile) every producer of one consumer must agree on.  N = 1280 / 640 / 320
    (the narrow UNet widths) take 160-wide tiles (tall 256 x 160 at launch), the wide QKV / GEGLU GEMMs 256 (CTA pairs)."""
    from omg_b200 import _lib as L
    from omg_b200 import ops
    assert ops.gemm_plan(1280, L.EPI_NONE, 4096) == (160, 16)      # main rows, c = 1280
    assert ops.gemm_plan(1280, L.EPI_NONE, 8192) == (160, 16)      # grouped fusion step: same plan, so same partials
    assert ops.gemm_plan(640, L.EPI_NONE, 16384) == (160, 8)
    assert ops.gemm_plan(320, L.EPI_NONE, 65536) == (160, 4)
    assert ops.gemm_plan(3840, L.EPI_NONE, 4096) == (256, 30)
    assert ops.gemm_plan(10240, L.EPI_GEGLU, 4096) == (256, 80)
    assert ops.gemm_plan(8, L.EPI_NONE, 65536)[0] == 64            # conv_out: 8 padded channels
    with pytest.raises(RuntimeError):
        ops.gemm_plan(4, L.EPI_NONE, 128)                          # N < 8 is rejected with an error string


def test_c_abi_rejects_bad_arguments_before_touching_the_gpu():
    """Every entry point validates its descriptor first and reports through the status code + omg_last_error(); none of
    these calls reaches a CUDA API, so they run on a machine without a GPU (pointers are never dereferenced)."""
    import ctypes as C
    from omg_b200 import _lib as L
    lib = L.load()
    fake = C.c_void_p(0x1000)

    def err(rc):
        assert rc == 1
        return lib.omg_last_error().decode()

    assert "multiple of 8" in err(lib.omg_softmax_rows(fake, 4, 12, 16, 1.0, None))
    assert "scale must be positive" in err(lib.omg_softmax_rows(fake, 4, 16, 16, -1.0, None))
    d = L.AttnDesc()
    d.head_dim, d.n_items = 32, 1
    assert "head_dim 32 unsupported" in err(lib.omg_attention(C.byref(d), None))
    d.head_dim, d.n_items = 64, 99
    assert "n_items=99 out of range" in err(lib.omg_attention(C.byref(d), None))
    assert "null descriptor" in err(lib.omg_gemm(None, None))
    g = L.GemmDesc()
    g.n_a = 0
    assert "n_a=0 out of range" in err(lib.omg_gemm(C.byref(g), None))
    g.n_a, g.n_segs = 1, 99
    assert "n_segs=99 out of range" in err(lib.omg_gemm(C.byref(g), None))
    f = L.FuseDesc()
    f.n_concepts, f.noise_main, f.latents = 9, 0x1000, 0x1000
    assert "n_concepts=9 out of range" in err(lib.omg_fuse_step(C.byref(f), None))
    assert "bad channel split" in err(lib.omg_groupnorm(fake, 100, None, 0, 1, 16, fake, fake, 1e-5, 0, fake, fake, None))


def test_cli_flags_match_the_reference_parse_args():
    """Every flag of the reference CLIs (inference_lora.py:203-222, inference_instantid.py:259-286; names, defaults and
    types extracted from the reference files by tests/golden/make_golden.py) exists here with the same default;
    extra flags are additive."""
    import importlib.util
    import json
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    gold = json.load(open(os.path.join(root, "tests", "golden", "cli_flags.json")))
    for fname, flags in gold.items():
        spec = importlib.util.spec_from_file_location("cli_" + fname[:-3], os.path.join(root, fname))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        argv, sys.argv = sys.argv, [fname]
        try:
            ns = vars(mod.parse_args())
        finally:
            sys.argv = argv
        for name, (default, tname) in flags.items():
            assert name in ns, f"{fname}: flag --{name} of the reference is missing"
            assert ns[name] == default and type(ns[name]).__name__ == tname, (fname, name, ns[name], default)


def test_product_resampler_matches_reference_golden():
    """omg_b200.resampler.resampler_forward (the function ConceptModels._encode_prompt_image_emb runs, SURVEY A13)
    against the output of the reference's own Resampler module (tests/golden/resampler.pt, src/ip_adapter/
    resampler.py:109-120)."""
    import os
    from omg_b200.resampler import resampler_forward
    d = torch.load(os.path.join(os.path.dirname(__file__), "golden", "resampler.pt"))
    y = resampler_forward(d["sd"], d["x"], d["heads"], d["dim_head"])
    assert y.shape == d["y"].shape and torch.allclose(y, d["y"], atol=2e-6)


def test_latent_init_follows_the_reference_generator_call():
    """A15 (lora_pipeline.py:397-409): latents = randn((1,4,h,w), generator, fp16) * init_noise_sigma, duplicated.  The
    product's prepare_latents must draw the SAME numbers from the same seeded generator (one randn call of that shape
    and dtype) - checked here on the host generator the CLIs use when CUDA is absent, and on cuda in the GPU test."""
    from omg_b200.pipelines import _BasePipeline
    from omg_b200.scheduler import EulerDiscreteSchedule

    class P(_BasePipeline):
        def __init__(self):
            self.scheduler = EulerDiscreteSchedule()
            self.scheduler.set_timesteps(30)

        _execution_device = torch.device("cpu")

    pipe = P()
    g = torch.Generator().manual_seed(14)
    lat = pipe.prepare_latents(16, 24, g, None)
    ref = torch.randn((1, 4, 16, 24), generator=torch.Generator().manual_seed(14), dtype=torch.float16)
    ref = ref.float() * pipe.scheduler.init_noise_sigma
    assert lat.shape == (2, 16, 24, 4) and lat.dtype == torch.float32
    assert torch.equal(lat[0], ref[0].permute(1, 2, 0)) and torch.equal(lat[1], lat[0])
    # the generator state advanced by exactly that one call
    assert torch.equal(torch.randn(3, generator=g),
                       (lambda h: (torch.randn((1, 4, 16, 24), generator=h, dtype=torch.float16), torch.randn(3, generator=h))[1])(
                           torch.Generator().manual_seed(14)))
