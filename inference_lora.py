#!/usr/bin/env python
"""OMG + LoRA multi-concept generation on the B200 path.  Same flags, prompt mini-DSL, two-stage flow and output
files as the reference CLI (inference_lora.py:201-323); additions (non-breaking): --synthetic, --num_inference_steps,
--image_size, --mask_boxes, --vae_fp16_safe, --vae.

The segmentation models between the stages (YOLO-World / GroundingDINO + SAM) and the VAE / text encoders are outside
the accelerated hot path (SURVEY section 8): masks come from --mask_boxes (x0,y0,x1,y1 per concept, '|' separated) or,
in --synthetic mode, from the fixed config-2 rectangles; without a VAE the latents are saved (stage-{1,2}.pt) next to
a PNG visualisation of their first three channels.
"""
import argparse
import hashlib
import os

import torch


def prepare_text(prompt, region_prompts):
    """'[prompt]-*-[negative]|[prompt]-*-[negative]' -> (prompt, [(region, region_negative), ...])
    (inference_lora.py:128-149)."""
    regions = []
    for region in region_prompts.split("|"):
        if region == "":
            break
        pos, neg = region.split("-*-")
        regions.append((pos.replace("[", "").replace("]", ""), neg.replace("[", "").replace("]", "")))
    return prompt, regions


def sample_image(pipe, input_prompt, input_neg_prompt=None, generator=None, concept_models=None,
                 num_inference_steps=50, guidance_scale=7.5, controller=None, stage=None, region_masks=None,
                 lora_list=None, styleL=None, **extra_kargs):
    """inference_lora.py:37-73."""
    spatial_condition = extra_kargs.pop("spatial_condition")
    spatial_condition_input = [spatial_condition] * len(input_prompt) if spatial_condition is not None else None
    return pipe(prompt=input_prompt, concept_models=concept_models, negative_prompt=input_neg_prompt,
                generator=generator, guidance_scale=guidance_scale, num_inference_steps=num_inference_steps,
                cross_attention_kwargs={"scale": 0.8}, controller=controller, stage=stage, region_masks=region_masks,
                lora_list=lora_list, styleL=styleL, image=spatial_condition_input, **extra_kargs).images


def parse_args():
    p = argparse.ArgumentParser("", add_help=True)
    p.add_argument("--pretrained_sdxl_model", default="./checkpoint/stable-diffusion-xl-base-1.0", type=str)
    p.add_argument("--controlnet_checkpoint", default="./checkpoint/controlnet-openpose-sdxl-1.0", type=str)
    p.add_argument("--spatial_condition", default="", type=str)
    p.add_argument("--efficientViT_checkpoint", default="./checkpoint/sam/xl1.pt", type=str)
    p.add_argument("--dino_checkpoint", default="./checkpoint/GroundingDINO", type=str)
    p.add_argument("--sam_checkpoint", default="./checkpoint/sam/sam_vit_h_4b8939.pth", type=str)
    p.add_argument("--save_dir", default="results/lora", type=str)
    p.add_argument("--prompt", type=str, default="Close-up photo of the cool man and beautiful woman as they "
                   "accidentally discover a mysterious island while on vacation by the sea, facing the camera smiling, "
                   "35mm photograph, film, professional, 4k, highly detailed.")
    p.add_argument("--negative_prompt", default="noisy, blurry, soft, deformed, ugly", type=str)
    p.add_argument("--prompt_rewrite", type=str,
                   default="[Close-up photo of the Chris Evans in surprised expressions, 35mm photograph, film, "
                           "professional, 4k, highly detailed.]-*-[noisy, blurry, soft, deformed, ugly]|"
                           "[Close-up photo of the TaylorSwift in surprised expressions, 35mm photograph, film, "
                           "professional, 4k, highly detailed.]-*-[noisy, blurry, soft, deformed, ugly]")
    p.add_argument("--lora_path", type=str,
                   default="./checkpoint/lora/chris-evans.safetensors|./checkpoint/lora/TaylorSwiftSDXL.safetensors")
    p.add_argument("--style_lora", default="", type=str)
    p.add_argument("--segment_type", default="yoloworld", help="GroundingDINO or yoloworld", type=str)
    p.add_argument("--seed", default=14, type=int)
    p.add_argument("--suffix", default="", type=str)
    # additions
    p.add_argument("--dedup", action="store_true", help="skip work that repeats identical work (same outputs): twin "
                   "rows before the first fusion step, stage-2 steps 0..15")
    p.add_argument("--synthetic", action="store_true", help="random-init SDXL-shaped weights, synthetic encoders/masks")
    p.add_argument("--num_inference_steps", default=50, type=int)
    p.add_argument("--image_size", default=1024, type=int)
    p.add_argument("--tiny", action="store_true", help="with --synthetic: toy widths (plumbing check)")
    p.add_argument("--decode", action="store_true", help="with --synthetic: decode with a random-init VAE decoder")
    p.add_argument("--mask_boxes", default="", type=str, help="x0,y0,x1,y1|x0,y0,x1,y1 (pixels), replaces segmentation")
    vae = p.add_mutually_exclusive_group()
    vae.add_argument("--vae_fp16_safe", default="", type=str, help="directory of fp16-safe SDXL VAE weights: decode to "
                     "PNG on the GPU (without it the latents are saved)")
    vae.add_argument("--vae", default="", type=str, help="diffusers VAE directory, or a checkpoint root with vae/: decode "
                     "both stages to PNG on the GPU, in bf16 when its config.json has force_upcast (the original SDXL VAE), "
                     "else fp16")
    return p.parse_args()


def _latents_png(lat, path):
    from PIL import Image
    x = lat[:3].float()
    x = (x - x.amin()) / (x.amax() - x.amin() + 1e-8)
    Image.fromarray((x.permute(1, 2, 0).cpu().numpy() * 255).astype("uint8")).resize((512, 512)).save(path)


def build_model_synthetic(args, prompts, device):
    from omg_b200 import factory
    from omg_b200.config import UNetConfig
    cfg = UNetConfig.tiny() if args.tiny else UNetConfig.sdxl()
    n = len([r for r in args.prompt_rewrite.split("|") if r])
    wl = factory.build_lora_workload(cfg, args.image_size, n, 32, args.num_inference_steps, 7.5, device=device)
    return wl.pipe, wl.controller, wl.concept_models, wl.call_kwargs["lora_list"], wl.masks


def build_model_sd(args, prompts, device):
    """Real checkpoints, mirroring the reference's build_model_sd (inference_lora.py:150-171): the diffusers-layout
    UNet / ControlNet safetensors load straight into PackedUNet, the LoRA files (kohya / SGM / diffusers layouts) through
    omg_b200.checkpoints, the prompts through the two CLIP towers (omg_b200.text).  Segmentation and the VAE are
    outside the path: regions come from --mask_boxes and the outputs are latents."""
    from omg_b200 import checkpoints as ck
    from omg_b200.config import UNetConfig
    from omg_b200.pipelines import ConceptModels, LoraMultiConceptPipeline, revise_regionally_controlnet_forward
    from omg_b200.prompt_attention import AttentionReplace
    from omg_b200.text import ClipPromptEncoder
    from omg_b200.unet import PackedUNet
    cfg = UNetConfig.sdxl()
    unet = PackedUNet(cfg, ck.load_unet_weights(args.pretrained_sdxl_model, "unet"), device=device)
    controlnet = None
    if args.spatial_condition and os.path.exists(args.spatial_condition):
        controlnet = PackedUNet(cfg, ck.load_unet_weights(args.controlnet_checkpoint, "", None), device=device,
                                controlnet=True)
    enc = ClipPromptEncoder.from_pretrained(args.pretrained_sdxl_model, device)
    vae = None
    if args.vae_fp16_safe:
        # opt-in: the decoder runs fp16 activations, which the ORIGINAL SDXL VAE weights overflow (the reference
        # up-casts the VAE to fp32, lora_pipeline.py:635-646); point this at the fp16-safe re-export (same keys).
        # The decoder raises on non-finite output instead of writing black PNGs.  Default output: latents.
        from omg_b200.vae import PackedVaeDecoder
        vae_dir = args.vae_fp16_safe
        sub = "vae" if os.path.isdir(os.path.join(vae_dir, "vae")) else ""
        vae = PackedVaeDecoder(ck.load_unet_weights(vae_dir, sub, None), device=device)
    pipe = LoraMultiConceptPipeline(unet, controlnet=controlnet, prompt_encoder=enc, vae_decoder=vae)
    controller = AttentionReplace(prompts, 50, cross_replace_steps={"default_": 1.}, self_replace_steps=0.4,
                                  tokenizer=enc.tokenizer, width=args.image_size // 32, height=args.image_size // 32)
    revise_regionally_controlnet_forward(pipe, controller)
    pipe_concept = ConceptModels(unet, prompt_encoder=enc)
    if args.style_lora and os.path.exists(args.style_lora):
        pipe.load_lora_weights(args.style_lora, weight_name="pytorch_lora_weights.safetensors", adapter_name="style")
        pipe_concept.load_lora_weights(args.style_lora, weight_name="pytorch_lora_weights.safetensors", adapter_name="style")
    pipe_list = []
    for lora_path in args.lora_path.split("|"):
        adapter_name = lora_path.split("/")[-1].split(".")[0]
        pipe_concept.load_lora_weights(lora_path, weight_name="pytorch_lora_weights.safetensors", adapter_name=adapter_name)
        pipe_list.append(adapter_name)
    if not args.mask_boxes:
        print("no --mask_boxes given: only stage 1 (the layout pass) will run")
    return pipe, controller, pipe_concept, pipe_list, [None] * len(pipe_list)


if __name__ == "__main__":
    args = parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("the B200 path needs a CUDA device (there is no CPU fallback)")
    device = torch.device("cuda")
    prompts = [args.prompt] * 2
    width = height = args.image_size
    # pose condition (inference_lora.py:241-246): opened, RGB, resized to the image size, passed as `image=`
    spatial_condition = None
    if args.spatial_condition:
        if os.path.exists(args.spatial_condition):
            from PIL import Image
            spatial_condition = Image.open(args.spatial_condition).convert("RGB").resize((width, height))
            print("use pose condition")
        else:
            raise SystemExit(f"--spatial_condition {args.spatial_condition}: no such file")
        if args.synthetic:
            raise SystemExit("--spatial_condition needs the real ControlNet checkpoint (not available with --synthetic)")
    kwargs = {"height": height, "width": width, "spatial_condition": spatial_condition, "output_type": "latent"}
    build = build_model_synthetic if args.synthetic else build_model_sd
    pipe, controller, pipe_concepts, pipe_list, synth_masks = build(args, prompts, device)
    pipe.dedup = args.dedup
    if args.synthetic and args.decode:
        from omg_b200 import synthetic
        from omg_b200.vae import PackedVaeDecoder, VaeConfig
        vcfg = VaeConfig.tiny() if args.tiny else VaeConfig.sdxl()
        pipe.vae_decoder = PackedVaeDecoder(synthetic.make_vae_state_dict(vcfg, 0), vcfg, device=device)
    if args.vae:
        from omg_b200.vae import PackedVaeDecoder
        pipe.vae_decoder = PackedVaeDecoder.from_pretrained(args.vae, device=device)
    decoded = pipe.vae_decoder is not None
    if decoded:
        kwargs["output_type"] = "pil"  # lora_pipeline.py:634-661: VAE decode + postprocess
    styleL = bool(args.style_lora) and os.path.exists(args.style_lora)
    input_prompt = [prompts, prepare_text(args.prompt, args.prompt_rewrite)[1]]
    common = dict(input_prompt=input_prompt, concept_models=pipe_concepts,
                  input_neg_prompt=[args.negative_prompt] * len(input_prompt), controller=controller,
                  lora_list=pipe_list, styleL=styleL, num_inference_steps=args.num_inference_steps, **kwargs)
    image = sample_image(pipe, generator=torch.Generator(device).manual_seed(args.seed), stage=1, **common)
    controller.reset()
    if args.mask_boxes:
        masks = []
        for box in args.mask_boxes.split("|"):
            x0, y0, x1, y1 = [int(v) for v in box.split(",")]
            m = torch.zeros(height, width)
            m[y0:y1, x0:x1] = 1
            masks.append(m)
    else:
        masks = synth_masks
    if any(m is not None for m in masks):
        image = sample_image(pipe, generator=torch.Generator(device).manual_seed(args.seed), stage=2,
                             region_masks=masks, **common)
    configs = [f"pretrained_model: {args.pretrained_sdxl_model}\n", f"context_prompt: {args.prompt}\n",
               f"neg_context_prompt: {args.negative_prompt}\n", f"prompt_rewrite: {args.prompt_rewrite}\n"]
    hash_code = hashlib.sha256("".join(configs).encode("utf-8")).hexdigest()[:8]
    save_dir = os.path.join(args.save_dir, f"seed_{args.seed}")
    os.makedirs(save_dir, exist_ok=True)
    print(f"save to: {save_dir}")
    for idx, name in ((0, "stage-1"), (1, "stage-2")):
        if decoded:
            image[idx].save(os.path.join(save_dir, name + ".png"))
        else:
            torch.save(image[idx].cpu(), os.path.join(save_dir, name + ".pt"))
            _latents_png(image[idx], os.path.join(save_dir, name + ".png"))
    with open(os.path.join(save_dir, f"**---{args.suffix}---{hash_code}.txt"), "w") as fw:
        fw.writelines(configs)
