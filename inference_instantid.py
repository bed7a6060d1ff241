#!/usr/bin/env python
"""OMG + InstantID multi-identity generation on the B200 path.  The reference CLI's flags (names, defaults, types:
inference_instantid.py:259-286, pinned by tests/golden/cli_flags.json), prompt mini-DSL, two-stage flow and output
files; additions (non-breaking): --synthetic, --tiny, --num_inference_steps, --image_size, --dedup, --mask_boxes,
--face_embeds, --face_kps, --vae.

Face analysis (insightface antelopev2), segmentation and the VAE sit outside the accelerated hot path (SURVEY section
8): when `insightface` is not importable the identities come from --face_embeds (one 512-d .pt / .npy per region) and
the stage-2 key-points from --face_kps; regions come from --mask_boxes.  In --synthetic mode identities are unit-norm
random 512-d embeddings (seeds 1, 2), the IdentityNet condition is the reference's `draw_kps_multi` rendering of fixed
key-points and the masks are the config rectangles.
"""
import argparse
import math
import os

import numpy as np
import torch


def draw_kps_multi(image_size, kps_list, color_list=((255, 0, 0), (0, 255, 0), (0, 0, 255), (255, 255, 0),
                                                     (255, 0, 255))):
    """Key-point condition image of the IdentityNet: limbs as filled rotated ellipses towards the nose point, then
    the five points as discs (inference_instantid.py:127-156).  image_size = (w, h); returns an HxWx3 uint8 array."""
    import cv2
    stick_width, limb_seq = 4, np.array([[0, 2], [1, 2], [3, 2], [4, 2]])
    w, h = image_size
    canvas = np.zeros([h, w, 3])
    for kps in kps_list:
        kps = np.array(kps)
        for a, b in limb_seq:
            color = color_list[a]
            xs, ys = kps[[a, b]][:, 0], kps[[a, b]][:, 1]
            length = ((xs[0] - xs[1]) ** 2 + (ys[0] - ys[1]) ** 2) ** 0.5
            angle = math.degrees(math.atan2(ys[0] - ys[1], xs[0] - xs[1]))
            poly = cv2.ellipse2Poly((int(np.mean(xs)), int(np.mean(ys))), (int(length / 2), stick_width), int(angle),
                                    0, 360, 1)
            canvas = cv2.fillConvexPoly(canvas.copy(), poly, color)
        canvas = (canvas * 0.6).astype(np.uint8)  # truncation per face, as the reference does (:148)
        for idx, (x, y) in enumerate(kps):
            canvas = cv2.circle(canvas.copy(), (int(x), int(y)), 10, color_list[idx], -1)
    return canvas.astype(np.uint8)


def prepare_text(prompt, region_prompts):
    """'[prompt]-*-[negative]-*-ref_image|...' -> [(region, negative, ref_image), ...]
    (inference_instantid.py:233-254)."""
    out = []
    for region in region_prompts.split("|"):
        if region == "":
            break
        pos, neg, ref = region.split("-*-")
        out.append((pos.replace("[", "").replace("]", ""), neg.replace("[", "").replace("]", ""), ref))
    return prompt, out


def parse_args():
    """Flags of the reference (inference_instantid.py:259-286), then the additive ones."""
    p = argparse.ArgumentParser("", add_help=True)
    p.add_argument("--pretrained_model", default="./checkpoint/YamerMIX_v8", type=str)
    p.add_argument("--controlnet_path", default="./checkpoint/InstantID/ControlNetModel", type=str)
    p.add_argument("--spatial_condition", default="", type=str)
    p.add_argument("--t2i_controlnet_path", default="", type=str)
    p.add_argument("--face_adapter_path", default="./checkpoint/InstantID/ip-adapter.bin", type=str)
    p.add_argument("--efficientViT_checkpoint", default="./checkpoint/sam/xl1.pt", type=str)
    p.add_argument("--dino_checkpoint", default="./checkpoint/GroundingDINO", type=str)
    p.add_argument("--sam_checkpoint", default="./checkpoint/sam/sam_vit_h_4b8939.pth", type=str)
    p.add_argument("--antelopev2_path", default="./checkpoint/antelopev2", type=str)
    p.add_argument("--save_dir", default="results/instantID", type=str)
    p.add_argument("--prompt", default="Close-up photo of the cool man and beautiful woman as they accidentally discover "
                   "a mysterious island while on vacation by the sea, facing the camera smiling, 35mm photograph, film, "
                   "professional, 4k, highly detailed.", type=str)
    p.add_argument("--negative_prompt", default="noisy, blurry, soft, deformed, ugly", type=str)
    p.add_argument("--prompt_rewrite", type=str,
                   default="[Close-up photo of the a man, 35mm photograph, professional, 4k, highly detailed.]-*"
                           "-[noisy, blurry, soft, deformed, ugly]-*-"
                           "./example/chris-evans.jpg|"
                           "[Close-up photo of the a woman, 35mm photograph, professional, 4k, highly detailed.]-"
                           "*-[noisy, blurry, soft, deformed, ugly]-*-"
                           "./example/TaylorSwift.png")
    p.add_argument("--seed", default=53, type=int)
    p.add_argument("--suffix", default="", type=str)
    p.add_argument("--segment_type", default="yoloworld", help="GroundingDINO or yoloworld", type=str)
    p.add_argument("--style_lora", default="", type=str)
    p.add_argument("--cfg_scale", default=3.0, type=float)
    p.add_argument("--IdentityNet_rate", default=0.8, type=float)
    p.add_argument("--adapter_ratio", default=0.8, type=float)
    p.add_argument("--controlNet_ratio", default=0.8, type=float)
    # additions
    p.add_argument("--dedup", action="store_true", help="skip work that repeats identical work (same outputs): twin "
                   "rows before the first fusion step, stage-2 steps 0..15")
    p.add_argument("--synthetic", action="store_true", help="random-init SDXL-shaped weights, synthetic identities")
    p.add_argument("--tiny", action="store_true", help="with --synthetic: toy widths (plumbing check)")
    p.add_argument("--num_inference_steps", default=50, type=int)
    p.add_argument("--image_size", default=1024, type=int)
    p.add_argument("--mask_boxes", default="", type=str, help="x0,y0,x1,y1|x0,y0,x1,y1 (pixels), replaces segmentation")
    p.add_argument("--face_embeds", default="", type=str, help="a.pt|b.pt: 512-d identity embeddings, one per region "
                   "(replaces insightface on the reference images)")
    p.add_argument("--face_kps", default="", type=str, help="JSON file: list of five (x, y) key-points per face for "
                   "the stage-2 IdentityNet condition (replaces insightface on the stage-1 image)")
    p.add_argument("--vae", default="", type=str, help="diffusers VAE directory, or a checkpoint root with vae/: decode "
                   "both stages to PNG on the GPU, in bf16 when its config.json has force_upcast (the original SDXL VAE), "
                   "else fp16 (without it the latents are saved)")
    return p.parse_args()


def build_model_sd(pretrained_model, controlnet_path, face_adapter, device, prompts, antelopev2_path, width, height,
                   style_lora, condition_checkpoint, adapter_ratio):
    """inference_instantid.py:195-230 on the packed executors: IdentityNet + base UNet + CLIP towers from the diffusers
    checkouts, InstantID's ip-adapter.bin (Resampler + to_k_ip / to_v_ip) through omg_b200.checkpoints, the optional
    t2i ControlNet as `pipe.controlnet2`, the style LoRA on both pipelines.  The concept pipeline shares the packed
    base weights (the reference loads the same checkpoint a second time, :205-210)."""
    from omg_b200.pipelines import (ConceptModels, InstantidMultiConceptPipeline, load_controlnet,
                                    revise_regionally_controlnet_forward)
    from omg_b200.prompt_attention import AttentionReplace
    controlnet = load_controlnet(controlnet_path, device)
    pipe = InstantidMultiConceptPipeline.from_pretrained(pretrained_model, controlnet=controlnet,
                                                         torch_dtype=torch.float16, variant="fp16", device=device)
    controller = AttentionReplace(prompts, 50, cross_replace_steps={"default_": 1.}, self_replace_steps=0.4,
                                  tokenizer=pipe.tokenizer, width=width, height=height)
    revise_regionally_controlnet_forward(pipe, controller)
    pipe_concept = ConceptModels.from_pretrained(pretrained_model, unet=pipe.unet, prompt_encoder=pipe.prompt_encoder,
                                                 device=device)
    pipe_concept.load_ip_adapter_instantid(face_adapter)
    pipe_concept.set_ip_adapter_scale(adapter_ratio)
    if condition_checkpoint is not None and os.path.exists(condition_checkpoint):
        pipe.controlnet2 = load_controlnet(condition_checkpoint, device)
    if style_lora is not None and os.path.exists(style_lora):
        pipe.load_lora_weights(style_lora, weight_name="pytorch_lora_weights.safetensors", adapter_name="style")
        pipe_concept.load_lora_weights(style_lora, weight_name="pytorch_lora_weights.safetensors", adapter_name="style")
    app = None
    try:  # insightface is outside the path; identities can come from --face_embeds instead
        from insightface.app import FaceAnalysis
        app = FaceAnalysis(name="antelopev2", root=antelopev2_path,
                           providers=["CUDAExecutionProvider", "CPUExecutionProvider"])
        app.prepare(ctx_id=0, det_size=(640, 640))
    except ImportError:
        print("insightface not importable: identities from --face_embeds, key-points from --face_kps")
    return pipe, controller, pipe_concept, app


def _load_vec(path):
    if path.endswith(".npy"):
        return torch.from_numpy(np.load(path)).float().reshape(-1)
    return torch.as_tensor(torch.load(path, map_location="cpu", weights_only=True)).float().reshape(-1)


def sample_image(pipe, input_prompt, input_neg_prompt=None, generator=None, concept_models=None,
                 num_inference_steps=50, guidance_scale=3, controller=None, face_app=None, image=None, stage=None,
                 region_masks=None, controlnet_conditioning_scale=None, **extra_kargs):
    """inference_instantid.py:72-109."""
    image_condition = [image] if image is not None else None
    return pipe(prompt=input_prompt, concept_models=concept_models, negative_prompt=input_neg_prompt,
                generator=generator, guidance_scale=guidance_scale, num_inference_steps=num_inference_steps,
                cross_attention_kwargs={"scale": 0.8}, controller=controller, image=image_condition, face_app=face_app,
                stage=stage, controlnet_conditioning_scale=controlnet_conditioning_scale, region_masks=region_masks,
                **extra_kargs).images


def build_synthetic(args, device):
    from omg_b200 import synthetic
    from omg_b200.config import UNetConfig
    from omg_b200.pipelines import ConceptModels, InstantidMultiConceptPipeline, revise_regionally_controlnet_forward
    from omg_b200.prompt_attention import AttentionReplace
    from omg_b200.unet import PackedUNet
    cfg = UNetConfig.tiny() if args.tiny else UNetConfig.sdxl()
    sd = synthetic.make_state_dict(cfg, seed=0, device=device, dtype=torch.float16)
    unet = PackedUNet(cfg, sd, device=device)
    idnet = PackedUNet(cfg, synthetic.make_state_dict(cfg, seed=1, controlnet=True, device=device,
                                                      dtype=torch.float16), device=device, controlnet=True)
    pipe = InstantidMultiConceptPipeline(unet, controlnet=idnet)
    controller = AttentionReplace([args.prompt] * 2, 50, cross_replace_steps={"default_": 1.0}, self_replace_steps=0.4,
                                  width=args.image_size // 32, height=args.image_size // 32)
    revise_regionally_controlnet_forward(pipe, controller)
    cm = ConceptModels(unet)
    # perceiver Resampler of InstantID (dim 1280, depth 4, heads 20, 16 queries, 512 -> cross_attention_dim)
    dim, depth, heads = (1280, 4, 20) if not args.tiny else (128, 2, 4)
    g = torch.Generator().manual_seed(7)
    D = cfg.cross_attention_dim

    def rn(*s, fan=None):
        return torch.randn(*s, generator=g) * ((fan or s[-1]) ** -0.5)

    rs = {"latents": rn(1, 16, dim), "proj_in.weight": rn(dim, 512), "proj_in.bias": torch.zeros(dim),
          "proj_out.weight": rn(D, dim), "proj_out.bias": torch.zeros(D), "norm_out.weight": torch.ones(D),
          "norm_out.bias": torch.zeros(D)}
    for i in range(depth):
        a, f = f"layers.{i}.0", f"layers.{i}.1"
        for n in ("norm1", "norm2"):
            rs[f"{a}.{n}.weight"], rs[f"{a}.{n}.bias"] = torch.ones(dim), torch.zeros(dim)
        rs[f"{a}.to_q.weight"], rs[f"{a}.to_kv.weight"], rs[f"{a}.to_out.weight"] = rn(dim, dim), rn(2 * dim, dim), rn(dim, dim)
        rs[f"{f}.0.weight"], rs[f"{f}.0.bias"] = torch.ones(dim), torch.zeros(dim)
        rs[f"{f}.1.weight"], rs[f"{f}.3.weight"] = rn(4 * dim, dim), rn(dim, 4 * dim)
    cm.load_ip_adapter_instantid(rs, synthetic.make_ip_adapter(cfg, 31, device=device), heads=heads,
                                 dim_head=dim // heads, num_tokens=16)
    return pipe, controller, cm


if __name__ == "__main__":
    args = parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("the B200 path needs a CUDA device (there is no CPU fallback)")
    device = torch.device("cuda")
    from omg_b200 import synthetic
    size = args.image_size
    width = height = size
    prompts = [args.prompt] * 2
    regions = prepare_text(args.prompt, args.prompt_rewrite)[1]
    spatial_condition = None
    if args.spatial_condition:
        if not os.path.exists(args.spatial_condition):
            raise SystemExit(f"--spatial_condition {args.spatial_condition}: no such file")
        from PIL import Image
        spatial_condition = Image.open(args.spatial_condition).convert("RGB").resize((width, height))
        print("use pose condition")
    kwargs = {"height": height, "width": width, "t2i_image": spatial_condition,
              "t2i_controlnet_conditioning_scale": args.controlNet_ratio, "output_type": "latent",
              "num_inference_steps": args.num_inference_steps}
    face_app = None
    if args.synthetic:
        pipe, controller, cm = build_synthetic(args, device)
        cm.set_ip_adapter_scale(args.adapter_ratio)
        g = torch.Generator().manual_seed(1)
        faces = [torch.nn.functional.normalize(torch.randn(512, generator=g), dim=0) for _ in regions]
        s = size / 1024.0
        kps = [[[300 * s + dx * s, 380 * s], [400 * s + dx * s, 380 * s], [350 * s + dx * s, 440 * s],
                [310 * s + dx * s, 500 * s], [390 * s + dx * s, 500 * s]] for dx in (0, 380)][: len(regions)]
        masks = synthetic.rect_masks(len(regions), (size, size))
    else:
        pipe, controller, cm, face_app = build_model_sd(args.pretrained_model, args.controlnet_path,
                                                        args.face_adapter_path, device, list(prompts), args.antelopev2_path,
                                                        width // 32, height // 32, args.style_lora,
                                                        args.t2i_controlnet_path, args.adapter_ratio)
        faces = [_load_vec(f) for f in args.face_embeds.split("|") if f] or None
        if faces is None and face_app is None:
            raise SystemExit("no identities: install insightface or pass --face_embeds a.pt|b.pt")
        kps = None
        if args.face_kps:
            import json
            kps = json.load(open(args.face_kps))
        masks = []
        for box in [b for b in args.mask_boxes.split("|") if b]:
            x0, y0, x1, y1 = [int(v) for v in box.split(",")]
            m = torch.zeros(height, width)
            m[y0:y1, x0:x1] = 1
            masks.append(m)
        masks = masks or [None] * len(regions)
    pipe.dedup = args.dedup
    if args.vae:
        from omg_b200.vae import PackedVaeDecoder
        pipe.vae_decoder = PackedVaeDecoder.from_pretrained(args.vae, device=device)
        kwargs["output_type"] = "pil"  # VAE decode + postprocess
    input_prompt = [prompts, regions]
    common = dict(input_prompt=input_prompt, concept_models=cm, input_neg_prompt=[args.negative_prompt] * len(input_prompt),
                  controller=controller, face_app=face_app, controlnet_conditioning_scale=args.IdentityNet_rate,
                  guidance_scale=args.cfg_scale, face_embeds=faces, **kwargs)
    image = sample_image(pipe, generator=torch.Generator(device).manual_seed(args.seed), stage=1, **common)
    controller.reset()
    if any(m is not None for m in masks):
        if kps is None:
            raise SystemExit("stage 2 needs the faces' key-points: --face_kps (insightface on the decoded stage-1 image "
                             "is outside the path)")
        face_kps = torch.from_numpy(draw_kps_multi((width, height), kps)).permute(2, 0, 1).float() / 255.0
        image = sample_image(pipe, generator=torch.Generator(device).manual_seed(args.seed), stage=2, image=face_kps,
                             region_masks=masks, **common)
    import hashlib
    configs = [f"pretrained_model: {args.pretrained_model}\n", f"context_prompt: {args.prompt}\n",
               f"neg_context_prompt: {args.negative_prompt}\n", f"prompt_rewrite: {args.prompt_rewrite}\n"]
    hash_code = hashlib.sha256("".join(configs).encode("utf-8")).hexdigest()[:8]
    save_dir = os.path.join(args.save_dir, f"seed_{args.seed}")
    os.makedirs(save_dir, exist_ok=True)
    print(f"save to: {save_dir}")
    for idx, name in ((0, "stage-1"), (1, "stage-2")):
        if args.vae:
            image[idx].save(os.path.join(save_dir, name + ".png"))
        else:
            torch.save(image[idx].cpu(), os.path.join(save_dir, name + ".pt"))
    with open(os.path.join(save_dir, f"**---{args.suffix}---{hash_code}.txt"), "w") as fw:
        fw.writelines(configs)
