"""bf16 VAE vs fp16 VAE on one B200 (DESIGN.md 3.11).

1. VAE encode and decode of 8 x 1024^2 (SDXL VAE topology, seeded synthetic weights), CUDA events after warm-up, for three modes:
   fp16 with fp16 attention scores (synthetic-weight default), fp16 with fp32 scores (what real checkpoints use) and bf16.  The modes
   alternate within each repetition, so drift of the shared machine hits all three alike; the median per mode is reported.
2. The per-kernel-family split of ops.PROFILE (one profiled encode + decode per mode, in a separate pass).
3. FastEditor.edit_many (SDXL, 8 images per call, strength 0.5) with vae_dtype fp16 and bf16, alternating in one process.

Writes one JSON file (--out) that records the card name and power limit next to the numbers."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from fast_image_editing_with_generative_models_b200 import configs as C  # noqa: E402
from fast_image_editing_with_generative_models_b200 import ops  # noqa: E402
from fast_image_editing_with_generative_models_b200 import synthetic as S  # noqa: E402
from fast_image_editing_with_generative_models_b200.engine import VAE  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    name, power, clk = [s.strip() for s in q.stdout.splitlines()[0].split(",")]
    return dict(name=name, power_limit=power, max_sm_clock=clk)


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--edit_reps", type=int, default=5)
    ap.add_argument("--out", type=str, default="vae_bf16_bench.json", help="JSON result file (profiles/vae_bf16_bench.json is one such run)")
    ap.add_argument("--skip_edit", action="store_true")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a B200"
    dev = torch.device("cuda:0")
    res = dict(card=card(), batch=args.batch, resolution=1024, reps=args.reps)
    B = args.batch
    vcfg = C.VAEConfig()
    vp = S.make_vae_params(vcfg)
    modes = {"fp16_scores_f16": dict(dtype=torch.float16, attention_scores_f32=False),
             "fp16_scores_f32": dict(dtype=torch.float16, attention_scores_f32=True),
             "bf16": dict(dtype=torch.bfloat16)}
    vaes = {k: VAE(vp, vcfg, dev, **kw) for k, kw in modes.items()}
    img = torch.from_numpy(np.stack([S.synthetic_image(s, 1024, 1024) for s in range(B)])).to(dev)
    xp = ops.preprocess_pad8(img, True)
    z = (torch.randn((B, 128, 128, 4), generator=torch.Generator().manual_seed(0)) * vcfg.scaling_factor).half().to(dev)
    with torch.no_grad():
        for v in vaes.values():                      # warm-up: module loads, attribute setup, allocator
            v.encode_moments(xp); v.decode(z)
        torch.cuda.synchronize()
        t = {k: dict(encode=[], decode=[]) for k in modes}
        for _ in range(args.reps):
            for k, v in vaes.items():
                t[k]["encode"].append(timed(lambda: v.encode_moments(xp)))
                t[k]["decode"].append(timed(lambda: v.decode(z)))
        res["vae_ms"] = {k: {s: dict(median=float(np.median(x)), min=float(np.min(x)), max=float(np.max(x))) for s, x in d.items()} for k, d in t.items()}
        for k in modes:
            m = res["vae_ms"][k]
            m["step_median"] = m["encode"]["median"] + m["decode"]["median"]
        # per-family split (profiled pass: events around every call, so the totals exceed the unprofiled times)
        res["profile_ms"] = {}
        for k, v in vaes.items():
            fam = {}
            for stage, fn in (("encode", lambda: v.encode_moments(xp)), ("decode", lambda: v.decode(z))):
                ops.PROFILE = []
                fn()
                summ = ops.profile_summary()
                ops.PROFILE = None
                fam[stage] = {f: dict(calls=d["calls"], ms=round(d["ms"], 3)) for f, d in sorted(summ.items(), key=lambda kv: -kv[1]["ms"])}
            res["profile_ms"][k] = fam
    print(json.dumps(res["vae_ms"], indent=1))
    del vaes
    torch.cuda.empty_cache()
    if not args.skip_edit:
        from PIL import Image
        from fast_image_editing_with_generative_models_b200 import model_zoo
        from fast_image_editing_with_generative_models_b200.editor import FastEditor
        state = model_zoo.synthetic_state("sdxl")
        eds = {"fp16": FastEditor("sdxl", device="cuda:0", state=state, verbose=False, vae_dtype=torch.float16),
               "bf16": FastEditor("sdxl", device="cuda:0", state=state, verbose=False, vae_dtype=torch.bfloat16)}
        ims = [Image.fromarray(S.synthetic_image(s, 1024, 1024)) for s in range(B)]
        prompts = ["a watercolor painting"] * B
        for ed in eds.values():                      # warm-up + CUDA-graph capture
            ed.edit_many(ims, prompts, strength=0.5, seed=0)
        te = {k: [] for k in eds}
        for _ in range(args.edit_reps):
            for k, ed in eds.items():
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                ed.edit_many(ims, prompts, strength=0.5, seed=0)
                torch.cuda.synchronize()
                te[k].append((time.perf_counter() - t0) * 1e3)
        res["edit_many_ms"] = {k: dict(median=float(np.median(x)), min=float(np.min(x)), max=float(np.max(x)), images=B) for k, x in te.items()}
        print(json.dumps(res["edit_many_ms"], indent=1))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
