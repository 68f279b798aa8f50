"""Edit one image (same flags and flow as the reference ``run_single_image.py:18-192``) on the B200-native engine.

    python run_single_image.py --image path/to/image.jpg --prompt "a rusty bicycle"

Additions over the reference: ``--strength`` (documented by the reference, ``IMPLEMENTATION.md:119``, but never wired to a
flag; default 0.8 = the code default ``src/pipeline.py:217``).  matplotlib is imported only when a plot is requested.
"""
import argparse
import os
import time
from datetime import datetime

from PIL import Image

from run_batch import checkpoints_from_args, vae_dtype_from_args
from src.pipeline import FastEditor


def build_parser():
    p = argparse.ArgumentParser(description="Fast image editing on a single image")
    p.add_argument("--image", type=str, required=True, help="Path to input image")
    p.add_argument("--prompt", type=str, required=True, help="Editing prompt")
    p.add_argument("--model", type=str, default="sdxl", choices=["sdxl", "ssd-1b"])
    p.add_argument("--negative_prompt", type=str, default="")
    p.add_argument("--steps", type=int, default=4)
    p.add_argument("--guidance", type=float, default=1.5)
    p.add_argument("--control_scale", type=float, default=0.5)
    p.add_argument("--canny_low", type=int, default=100)
    p.add_argument("--canny_high", type=int, default=200)
    p.add_argument("--seed", type=int, default=None)
    p.add_argument("--strength", type=float, default=0.80, help="img2img strength (extension; reference default 0.8)")
    p.add_argument("--output_dir", type=str, default="outputs")
    p.add_argument("--no_cpu_offload", action="store_true")
    p.add_argument("--quality_mode", action="store_true")
    p.add_argument("--full_precision", action="store_true")
    p.add_argument("--full_controlnet", action="store_true")
    p.add_argument("--compute_metrics", action="store_true")
    p.add_argument("--show_plot", action="store_true")
    from run_batch import add_checkpoint_args, add_size_arg
    add_checkpoint_args(p)
    add_size_arg(p)
    return p


def _save_plot(source_img, edited_img, title, path):
    import matplotlib
    matplotlib.use("Agg")
    import matplotlib.pyplot as plt
    fig, axes = plt.subplots(1, 2, figsize=(12, 6))
    axes[0].imshow(source_img); axes[0].set_title("Source Image"); axes[0].axis("off")
    axes[1].imshow(edited_img); axes[1].set_title(title); axes[1].axis("off")
    plt.tight_layout(); plt.savefig(path, dpi=150, bbox_inches="tight"); plt.close()


def main(argv=None):
    args = build_parser().parse_args(argv)
    if args.quality_mode:
        args.full_precision = args.full_controlnet = args.no_cpu_offload = True
        print("[Quality Mode] Enabled: fp32 + full ControlNet + no CPU offload")
    if not os.path.exists(args.image):
        print(f"Error: Image not found at {args.image}")
        return
    model_suffix = f"{args.model}_{'fp32' if args.full_precision else 'fp16'}"
    edited_dir = os.path.join(args.output_dir, "single", "edited", model_suffix)
    comparisons_dir = os.path.join(args.output_dir, "single", "comparisons", model_suffix)
    os.makedirs(edited_dir, exist_ok=True)
    os.makedirs(comparisons_dir, exist_ok=True)
    print(f"\n[1/4] Loading image from {args.image}")
    source_img = Image.open(args.image).convert("RGB")
    print(f"      Image size: {source_img.size}")
    print("\n[2/4] Initializing FastEditor...")
    editor = FastEditor(model_name=args.model, device="cuda", enable_cpu_offload=not args.no_cpu_offload,
                        use_full_precision=args.full_precision, use_full_controlnet=args.full_controlnet,
                        checkpoints=checkpoints_from_args(args), vae_dtype=vae_dtype_from_args(args))
    mem = editor.get_memory_usage()
    print(f"      GPU Memory: {mem['allocated_gb']:.2f}GB allocated, {mem['reserved_gb']:.2f}GB reserved")
    print("\n[3/4] Running image editing...")
    print(f"      Prompt: {args.prompt}")
    print(f"      Steps: {args.steps}, Guidance: {args.guidance}, Control Scale: {args.control_scale}")
    t0 = time.time()
    edited_img = editor.edit(image=source_img, prompt=args.prompt, negative_prompt=args.negative_prompt, strength=args.strength,
                             num_inference_steps=args.steps, guidance_scale=args.guidance, controlnet_conditioning_scale=args.control_scale,
                             canny_low_threshold=args.canny_low, canny_high_threshold=args.canny_high, seed=args.seed, size=args.size)
    elapsed = time.time() - t0
    print(f"      Editing completed in {elapsed:.2f} seconds")
    mem = editor.get_memory_usage()
    print(f"      GPU Memory: {mem['allocated_gb']:.2f}GB allocated, {mem['reserved_gb']:.2f}GB reserved")
    ts = datetime.now().strftime("%Y%m%d_%H%M%S")
    output_path = os.path.join(edited_dir, f"edited_{ts}.jpg")
    edited_img.save(output_path)
    print(f"\n      Saved edited image to: {output_path}")
    title = f"Edited Image ({args.model.upper()})\n\"{args.prompt}\""
    if args.compute_metrics:
        from src.metrics import MetricsCalculator
        print("\n[4/4] Computing metrics...")
        calc = MetricsCalculator(device="cuda")
        m = calc.calculate_all_metrics(source_img=source_img, edited_img=edited_img, prompt=args.prompt)
        for k, label in (("ssim", "SSIM"), ("lpips", "LPIPS"), ("psnr", "PSNR"), ("mse", "MSE"), ("clip_score", "CLIP Score")):
            print(f"        {label}: {m[k]:.4f}")
        with open(os.path.join(edited_dir, f"metrics_{ts}.txt"), "w") as f:
            f.write(f"Image: {args.image}\nPrompt: {args.prompt}\nModel: {args.model}\nTime: {elapsed:.2f}s\n\nMetrics:\n")
            for k in ("ssim", "lpips", "psnr", "mse", "clip_score"):
                f.write(f"  {k}: {m[k]:.6f}\n")
        _save_plot(source_img, edited_img, title, os.path.join(comparisons_dir, f"comparison_{ts}.png"))
        calc.clear_memory()
    elif args.show_plot:
        _save_plot(source_img, edited_img, title, os.path.join(comparisons_dir, f"comparison_{ts}.png"))
    editor.clear_memory()
    print("\nDone!")


if __name__ == "__main__":
    main()
