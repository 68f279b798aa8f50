"""Batch editing over a PIE-Bench-style mapping file — same flags and per-image semantics as the reference
``run_batch.py:44-290`` (filters, ``--skip_existing``, per-image try/except that counts failures and continues),
on the B200-native engine.

    python run_batch.py --num_images 50 --editing_types 0 1 2
    torchrun --nproc-per-node 8 run_batch.py ...        # sharded sweep: rank r edits entries[r::world]

Additions over the reference: ``--strength`` and multi-GPU sharding via the torchrun environment.
"""
import argparse
import json
import os
import time

from PIL import Image

from fast_image_editing_with_generative_models_b200 import sweep
from src.pipeline import FastEditor


def load_mapping_file(mapping_path):
    with open(mapping_path, "r") as f:
        return json.load(f)


def safe_join(base_dir, user_path):
    """Join paths refusing absolute paths and directory traversal (ValueError), as the reference does."""
    user_path = os.path.normpath(user_path)
    if os.path.isabs(user_path) or user_path.startswith(".."):
        raise ValueError(f"Invalid path: {user_path}")
    full_path = os.path.abspath(os.path.join(base_dir, user_path))
    if not full_path.startswith(os.path.abspath(base_dir)):
        raise ValueError(f"Path traversal detected: {user_path}")
    return full_path


def build_parser():
    p = argparse.ArgumentParser(description="Batch image editing on PIE-Bench")
    p.add_argument("--mapping_file", type=str, default="data/PIE-Bench_v1/mapping_file.json")
    p.add_argument("--source_dir", type=str, default="data/PIE-Bench_v1/annotation_images")
    p.add_argument("--output_dir", type=str, default="outputs")
    p.add_argument("--model", type=str, default="sdxl", choices=["sdxl", "ssd-1b"])
    p.add_argument("--num_images", type=int, default=None)
    p.add_argument("--editing_types", nargs="+", type=str, default=None)
    p.add_argument("--image_ids", nargs="+", type=str, default=None)
    p.add_argument("--steps", type=int, default=4)
    p.add_argument("--guidance", type=float, default=1.5)
    p.add_argument("--control_scale", type=float, default=0.5)
    p.add_argument("--canny_low", type=int, default=100)
    p.add_argument("--canny_high", type=int, default=200)
    p.add_argument("--seed", type=int, default=None)
    p.add_argument("--strength", type=float, default=0.80, help="img2img strength (extension; reference default 0.8)")
    p.add_argument("--negative_prompt", type=str, default="")
    p.add_argument("--no_cpu_offload", action="store_true")
    p.add_argument("--quality_mode", action="store_true")
    p.add_argument("--full_precision", action="store_true")
    p.add_argument("--full_controlnet", action="store_true")
    p.add_argument("--skip_existing", action="store_true")
    p.add_argument("--save_comparisons", action="store_true")
    # extensions of the B200 build
    p.add_argument("--micro_batch", type=int, default=8, help="images per GPU per engine call (FastEditor.edit_many)")
    p.add_argument("--io_threads", type=int, default=4, help="host threads for JPEG decode / encode")
    p.add_argument("--summary_json", type=str, default=None, help="rank 0 writes the run's counters and timings here (sweep benchmarks)")
    p.add_argument("--no_gpu_jpeg", action="store_true", help="encode *.jpg outputs with PIL on the host instead of the GPU encoder "
                   "(the files are byte-identical either way)")
    add_checkpoint_args(p)
    add_size_arg(p)
    add_lora_arg(p)
    return p


def add_size_arg(p):
    p.add_argument("--size", type=parse_size, default=(1024, 1024), metavar="{WxH|auto}",
                   help="output size: WIDTHxHEIGHT (multiples of 64 in [256, 2048], at most 1024x1024 pixels) or auto = the SDXL "
                        "aspect-ratio bucket closest to each input (default 1024x1024)")


def parse_size(text):
    """--size value -> FastEditor(size=...): 'auto' or (width, height)."""
    import argparse
    from fast_image_editing_with_generative_models_b200.editor import resolve_size
    if text == "auto":
        return "auto"
    try:
        w, h = (int(v) for v in text.lower().split("x"))
        return resolve_size((w, h), (w, h))
    except ValueError as e:
        raise argparse.ArgumentTypeError(f"--size {text!r}: expected WIDTHxHEIGHT or auto ({e})") from None


def add_checkpoint_args(p):
    """Real-weight folders (extension; the reference downloads from the HF hub, src/pipeline.py:89-154).  Defaults come from the
    FIE_CHECKPOINTS / FIE_CONTROLNET / FIE_VAE / FIE_LCM_LORA environment variables; without any, synthetic weights + a warning."""
    p.add_argument("--checkpoints", type=str, default=None, help="diffusers SDXL / SSD-1B pipeline folder (unet/ vae/ text_encoder*/ tokenizer*/)")
    p.add_argument("--controlnet_dir", type=str, default=None, help="ControlNet-Canny folder (config.json + safetensors)")
    p.add_argument("--vae_dir", type=str, default=None, help="VAE folder (e.g. sdxl-vae-fp16-fix); default <checkpoints>/vae")
    p.add_argument("--unet_dir", type=str, default=None, help="UNet folder override (SSD-1B: the lcm-ssd-1b UNet)")
    p.add_argument("--lcm_lora", type=str, default=None, help="LCM-LoRA safetensors file (SDXL)")
    p.add_argument("--vae_dtype", choices=("auto", "fp16", "bf16"), default="auto",
                   help="VAE storage type: auto = bf16 if the VAE config.json says force_upcast: true (e.g. stabilityai/sdxl-vae), else fp16")


def parse_lora(text: str):
    """--lora PATH[=WEIGHT] -> (path, weight); the weight defaults to 1.0."""
    path, sep, w = text.rpartition("=")
    if sep:
        try:
            return path, float(w)
        except ValueError:
            pass
    return text, 1.0


def add_lora_arg(p):
    p.add_argument("--lora", type=parse_lora, action="append", default=[], metavar="PATH[=WEIGHT]",
                   help="style LoRA (.safetensors file or folder), repeatable: loaded after the editor is built and active next to the "
                        "LCM-LoRA at WEIGHT (default 1.0); editor.pipe.load_lora_weights / set_adapters")


def apply_lora_args(editor, args):
    """Loads every --lora adapter and activates them, at their weights, next to the adapters the editor was built with."""
    if not args.lora:
        return
    names = editor.pipe.get_active_adapters()
    weights = [1.0] * len(names)
    for i, (path, w) in enumerate(args.lora):
        name = f"lora_{i}"
        editor.pipe.load_lora_weights(path, adapter_name=name)
        names.append(name)
        weights.append(w)
    editor.pipe.set_adapters(names, weights)


def vae_dtype_from_args(args):
    """--vae_dtype -> FastEditor(vae_dtype=...): None (auto), torch.float16 or torch.bfloat16."""
    import torch
    return {"auto": None, "fp16": torch.float16, "bf16": torch.bfloat16}[args.vae_dtype]


def checkpoints_from_args(args):
    from fast_image_editing_with_generative_models_b200.editor import expand_checkpoints
    if not args.checkpoints:
        return None           # FastEditor then consults the environment variables
    return expand_checkpoints(args.checkpoints, args.controlnet_dir, args.vae_dir, args.lcm_lora, args.unet_dir)


def micro_batches(work, mb, size):
    """Work items -> groups of at most ``mb`` for edit_many.  With ``size="auto"`` the items are first grouped by their bucket (first-seen
    order; only the image header is read), so that each group holds one size: full micro-batches and one CUDA graph per bucket,
    instead of small padded chunks of every bucket in each group.  An unreadable image goes to a group of its own kind; loading it
    reports the error."""
    if size != "auto":
        return [work[i:i + mb] for i in range(0, len(work), mb)]
    from fast_image_editing_with_generative_models_b200.editor import resolve_size
    by_bucket = {}
    for it in work:
        try:
            with Image.open(it[2]) as im:
                key = resolve_size("auto", im.size)
        except Exception:
            key = None
        by_bucket.setdefault(key, []).append(it)
    return [items[i:i + mb] for items in by_bucket.values() for i in range(0, len(items), mb)]


def select_entries(mapping, args):
    """The reference's filtering rules (``run_batch.py:117-140``)."""
    if args.image_ids:
        return [(i, mapping[i]) for i in args.image_ids if i in mapping]
    if args.editing_types:
        sel = [(i, e) for i, e in mapping.items() if e.get("editing_type_id") in args.editing_types]
    else:
        sel = list(mapping.items())
    if args.num_images and args.num_images < len(sel):
        sel = sel[: args.num_images]
    return sel


def main(argv=None):
    args = build_parser().parse_args(argv)
    if args.quality_mode:
        args.full_precision = args.full_controlnet = args.no_cpu_offload = True
    rank, world, local = sweep.init_distributed()
    say = print if rank == 0 else (lambda *a, **k: None)
    model_suffix = f"{args.model}_{'fp32' if args.full_precision else 'fp16'}"
    edited_dir = os.path.join(args.output_dir, "batch", "edited", model_suffix)
    comparisons_dir = os.path.join(args.output_dir, "batch", "comparisons", model_suffix)
    os.makedirs(edited_dir, exist_ok=True)
    say(f"\n[1/3] Loading mapping file from {args.mapping_file}")
    mapping = load_mapping_file(args.mapping_file)
    selected = select_entries(mapping, args)
    say(f"[2/3] Selected {len(selected)} images; world size {world}")
    if not selected:
        say("\n      No images selected. Exiting.")
        return
    mine = sweep.shard(selected, rank, world)
    say(f"\n[3/3] Initializing FastEditor ({model_suffix})...")
    device = f"cuda:{local}" if world > 1 else "cuda"
    editor = FastEditor(model_name=args.model, device=device, enable_cpu_offload=not args.no_cpu_offload,
                        use_full_precision=args.full_precision, use_full_controlnet=args.full_controlnet, verbose=rank == 0,
                        checkpoints=checkpoints_from_args(args), vae_dtype=vae_dtype_from_args(args))
    if hasattr(editor, "pipe"):
        editor.pipe.set_progress_bar_config(disable=True)
    apply_lora_args(editor, args)
    processed = skipped = failed = 0
    total_time = 0.0
    # ---- per-entry admission (the reference's checks, run_batch.py:185-207), then micro-batches of --micro_batch images ----
    work = []
    for image_id, entry in mine:
        try:
            source_filename = entry["image_path"]
            source_path = safe_join(args.source_dir, source_filename)
            output_path = os.path.join(edited_dir, source_filename)
            if args.skip_existing and os.path.exists(output_path):
                skipped += 1
                continue
            if not os.path.exists(source_path):
                failed += 1
                continue
            if not entry.get("editing_prompt", ""):
                failed += 1
                continue
            work.append((image_id, entry, source_path, output_path))
        except ValueError as e:
            print(f"\n      Invalid path for {image_id}: {e}")
            failed += 1
        except Exception as e:
            print(f"\n      Error processing {image_id} ({type(e).__name__}): {e}")
            failed += 1
    mb = max(int(args.micro_batch), 1)
    groups = micro_batches(work, mb, args.size)
    edit_kw = dict(negative_prompt=args.negative_prompt, strength=args.strength, num_inference_steps=args.steps, guidance_scale=args.guidance,
                   controlnet_conditioning_scale=args.control_scale, canny_low_threshold=args.canny_low, canny_high_threshold=args.canny_high,
                   size=args.size)

    def load(item):
        return Image.open(item[2]).convert("RGB")

    def save(img, item, source_img):
        os.makedirs(os.path.dirname(item[3]), exist_ok=True)
        if isinstance(img, (bytes, bytearray)):        # already a JPEG file, encoded on the GPU (byte-identical to PIL's encoder)
            with open(item[3], "wb") as f:
                f.write(img)
            if args.save_comparisons:
                import io
                img = Image.open(io.BytesIO(img)).convert("RGB")
        else:
            img.save(item[3])
        if args.save_comparisons:
            from run_single_image import _save_plot
            cp = os.path.join(comparisons_dir, item[1]["image_path"].replace(".jpg", ".png"))
            os.makedirs(os.path.dirname(cp), exist_ok=True)
            _save_plot(source_img, img, f"Edited ({args.model.upper()})\n\"{item[1]['editing_prompt'][:60]}\"", cp)

    t_warm = 0.0
    if groups and hasattr(editor, "warm_up"):          # capture the CUDA graph of this schedule as part of initialisation, not of image 1
        as_jpeg0 = (not args.no_gpu_jpeg) and all(it[3].lower().endswith((".jpg", ".jpeg")) for it in groups[0])
        t_warm = editor.warm_up(mb, **({"output": "jpeg"} if as_jpeg0 else {}), **edit_kw)
    # JPEG decode of the next group and JPEG encode of the previous one run on host threads (PIL releases the GIL in its codecs)
    # while the GPU edits the current group.
    from concurrent.futures import ThreadPoolExecutor
    pool = ThreadPoolExecutor(max_workers=max(int(args.io_threads), 1))
    saves = []
    loads = [pool.submit(load, it) for it in groups[0]] if groups else []
    for gi, group in enumerate(groups):
        nxt = [pool.submit(load, it) for it in groups[gi + 1]] if gi + 1 < len(groups) else []
        items, imgs = [], []
        for it, fut in zip(group, loads):
            try:
                imgs.append(fut.result())
                items.append(it)
            except FileNotFoundError as e:
                print(f"\n      File not found for {it[0]}: {e}")
                failed += 1
            except Exception as e:
                print(f"\n      Error processing {it[0]} ({type(e).__name__}): {e}")
                failed += 1
        loads = nxt
        if not items:
            continue
        t0 = time.time()
        try:
            as_jpeg = (not args.no_gpu_jpeg) and all(it[3].lower().endswith((".jpg", ".jpeg")) for it in items)
            outs = editor.edit_many(imgs, [it[1]["editing_prompt"] for it in items], seed=args.seed, micro_batch=mb,
                                    **({"output": "jpeg"} if as_jpeg else {}), **edit_kw)
        except Exception as e:   # per-image isolation, as the reference (run_batch.py:250-261): retry the group image by image
            print(f"\n      Batch of {len(items)} failed ({type(e).__name__}: {e}); retrying per image")
            outs = []
            for it, im in zip(items, imgs):
                try:
                    outs.append(editor.edit(image=im, prompt=it[1]["editing_prompt"], seed=args.seed, **edit_kw))
                except Exception as e1:
                    print(f"\n      Error processing {it[0]} ({type(e1).__name__}): {e1}")
                    outs.append(None)
        total_time += time.time() - t0
        for it, im, out in zip(items, imgs, outs):
            if out is None:
                failed += 1
                continue
            saves.append((it, pool.submit(save, out, it, im)))
        done_before = processed + len(items)
        if done_before // 10 != processed // 10:
            editor.clear_memory()
        processed += sum(o is not None for o in outs)
        if rank == 0:
            print(f"\r      Editing[{rank}]: {sum(len(g) for g in groups[:gi + 1])}/{len(work)}", end="", flush=True)
    for it, fut in saves:
        try:
            fut.result()
        except Exception as e:
            print(f"\n      Error saving {it[0]} ({type(e).__name__}): {e}")
            processed -= 1
            failed += 1
    pool.shutdown()
    import torch
    dev = torch.device(device)
    processed_all = int(sweep.sum_over_ranks(processed, dev))
    skipped_all = int(sweep.sum_over_ranks(skipped, dev))
    failed_all = int(sweep.sum_over_ranks(failed, dev))
    time_all = sweep.sum_over_ranks(total_time, dev)
    wall = sweep.max_over_ranks(total_time, dev)
    say("\n" + "=" * 60 + "\nBATCH PROCESSING SUMMARY\n" + "=" * 60)
    say(f"\nProcessed:  {processed_all} images\nSkipped:    {skipped_all} images\nFailed:     {failed_all} images")
    if processed_all > 0:
        say(f"\nAverage time per image: {time_all / processed_all:.2f}s")
        say(f"Total time: {wall:.2f}s ({wall / 60:.1f} minutes) on {world} GPU(s)")
    else:
        say("\nWARNING: No images were successfully processed!")
    if args.summary_json and rank == 0:
        with open(args.summary_json, "w") as f:
            json.dump({"model": args.model, "world": world, "processed": processed_all, "skipped": skipped_all, "failed": failed_all,
                       "seconds_edit_max_over_ranks": wall, "seconds_edit_sum_over_ranks": time_all, "seconds_warmup_rank0": t_warm,
                       "images_per_s": processed_all / wall if wall > 0 else None, "micro_batch": mb, "gpu_jpeg": not args.no_gpu_jpeg,
                       "strength": args.strength, "steps": args.steps, "guidance": args.guidance}, f)
    say(f"\nOutputs saved to:\n  - Edited images: {edited_dir}")
    editor.clear_memory()
    say("\nDone!")


if __name__ == "__main__":
    main()
