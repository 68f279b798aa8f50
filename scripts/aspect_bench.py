"""Edits at the SDXL aspect-ratio buckets on one B200 (DESIGN.md 3.12).

1. Per bucket: FastEditor.edit_many (SDXL, seeded synthetic weights, 8 images per call, strength 0.5) at the bucket's size, alternating
   with 1024 x 1024 in the same process so that drift of the shared machine hits both alike.  Reports the median ms per call (one
   step of bench.py), ms per megapixel and its ratio to 1024^2, and the per-stage / per-kernel-family split of one profiled eager edit
   of each size (profiled separately: events around every call, so its totals exceed the graph-replay times).
2. Per convolution: TFLOP/s of the implicit-GEMM convolution on the VAE and UNet layer shapes at 1152 x 896 and 1216 x 832 (the form
   the library picks, and the im2col form forced), next to the same layer at 1024 x 1024 (box / halo form, and im2col forced).
   CUDA events over windows of 20 launches after warm-up, the four variants alternating window by window (median and range of
   --conv_rounds windows); the inputs rotate over enough copies to exceed the 126 MB L2.

Writes one JSON file (--out) that records the card name and power limit next to the numbers."""
import argparse
import json
import math
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from fast_image_editing_with_generative_models_b200 import _lib, ops  # noqa: E402
from fast_image_editing_with_generative_models_b200 import synthetic as S  # noqa: E402
from fast_image_editing_with_generative_models_b200.weights import pack_conv3x3, pack_conv_up2x  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    name, power, clk = [s.strip() for s in q.stdout.splitlines()[0].split(",")]
    return dict(name=name, power_limit=power, max_sm_clock=clk)


def conv_layers(width, height):
    """(name, kind, batch, h, w, cin, cout, stride, pad_mode): the VAE (batch 8) and SDXL UNet (batch 16 = 8 x CFG) conv shapes."""
    L = []
    for c, f in ((128, 1), (256, 2), (512, 4), (512, 8)):
        L.append((f"vae conv {c} @1/{f}", "conv", 8, height // f, width // f, c, c, 1, 0))
    L.append(("vae down 128 @1 s2", "conv", 8, height, width, 128, 128, 2, 1))
    for c, f in ((512, 8), (512, 4), (256, 2)):
        L.append((f"vae up2x {c} from 1/{f}", "up2x", 8, height // f, width // f, c, c, 1, 0))
    for c, f in ((320, 8), (640, 16), (1280, 32)):
        L.append((f"unet conv {c} @1/{f}", "conv", 16, height // f, width // f, c, c, 1, 0))
    L.append(("unet down 320 @1/8 s2", "conv", 16, height // 8, width // 8, 320, 320, 2, 0))
    return L


def make_conv(layer, dev):
    """-> (launch(x), inputs, FLOP per launch) for one layer; the inputs rotate over > 2 x L2 of distinct data."""
    name, kind, n, h, w, cin, cout, stride, pad_mode = layer
    g = torch.Generator().manual_seed(0)
    wt = (torch.randn((cout, cin, 3, 3), generator=g) / math.sqrt(9 * cin)).half()
    wp = (pack_conv_up2x(wt) if kind == "up2x" else pack_conv3x3(wt)).to(dev)
    bias = torch.randn((cout,), generator=g).to(dev)
    in_bytes = n * h * w * cin * 2
    copies = max(1, -(-256 * 2 ** 20 // in_bytes))
    gd = torch.Generator(device=dev).manual_seed(1)
    xs = [torch.randn((n, h, w, cin), generator=gd, device=dev, dtype=torch.float16) for _ in range(min(copies, 8))]
    while len(xs) * in_bytes < 256 * 2 ** 20:
        xs.append(xs[-1].clone())
    if kind == "up2x":
        return (lambda x: ops.conv_up2x(x, wp, col_bias=bias)), xs, 2.0 * n * 4 * h * w * cout * 4 * cin
    return (lambda x: ops.conv3x3(x, wp, stride=stride, pad_mode=pad_mode, col_bias=bias)), xs, 2.0 * n * (h // stride) * (w // stride) * cout * 9 * cin


def window_ms(fn, xs, force_im2col, reps):
    """Mean ms per launch over one window of ``reps`` launches (CUDA events), after three warm-up launches in the same form."""
    L = _lib.lib()
    L.fie_tune_conv_im2col(1 if force_im2col else 0)
    try:
        for x in xs[:3]:
            fn(x)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(reps):
            fn(xs[i % len(xs)])
        e1.record()
        torch.cuda.synchronize()
    finally:
        L.fie_tune_conv_im2col(0)
    return e0.elapsed_time(e1) / reps


def time_layer(lay, lay1024, dev, rounds, reps=20):
    """The four variants of one layer, alternating window by window (``rounds`` windows each) so that drift of the shared machine hits
    all four alike; median and range of the windows.  Where the library already picks im2col at the bucket shape, bucket_auto and
    bucket_im2col run the same code: their difference is the measurement noise."""
    at_b, at_1024 = make_conv(lay, dev), make_conv(lay1024, dev)
    variants = {"bucket_auto": (at_b, False), "bucket_im2col": (at_b, True), "at_1024_auto": (at_1024, False), "at_1024_im2col": (at_1024, True)}
    t = {k: [] for k in variants}
    for _ in range(rounds):
        for k, ((fn, xs, _), force) in variants.items():
            t[k].append(window_ms(fn, xs, force, reps))
    out = {}
    for k, ((_, _, flop), _) in variants.items():
        ms = float(np.median(t[k]))
        out[k] = dict(ms=round(ms, 4), tflops=round(flop / ms / 1e9, 1), ms_range=[round(min(t[k]), 4), round(max(t[k]), 4)])
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--reps", type=int, default=5, help="alternating edit_many pairs per bucket")
    ap.add_argument("--buckets", type=str, default="all", help="'all' or a comma list like 1152x896,1216x832")
    ap.add_argument("--out", type=str, default="aspect_bench.json", help="JSON result file (profiles/aspect_bench.json is one such run)")
    ap.add_argument("--conv_rounds", type=int, default=7, help="alternating timing windows per convolution variant")
    ap.add_argument("--skip_edit", action="store_true")
    ap.add_argument("--skip_conv", action="store_true")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a B200"
    dev = torch.device("cuda:0")
    from PIL import Image
    from fast_image_editing_with_generative_models_b200 import model_zoo
    from fast_image_editing_with_generative_models_b200.editor import FastEditor
    res = dict(card=card(), batch=args.batch, strength=0.5, model="sdxl (synthetic weights)")
    buckets = [b for b in FastEditor.SDXL_BUCKETS if b != (1024, 1024)]
    if args.buckets != "all":
        buckets = [tuple(int(v) for v in s.split("x")) for s in args.buckets.split(",")]
    B = args.batch
    if not args.skip_conv:
        res["conv"] = []
        for bucket in ((1152, 896), (1216, 832)):
            for lay, lay1024 in zip(conv_layers(*bucket), conv_layers(1024, 1024)):
                row = dict(layer=lay[0], bucket=f"{bucket[0]}x{bucket[1]}", shape=list(lay[2:]), **time_layer(lay, lay1024, dev, args.conv_rounds))
                print(json.dumps(row))
                res["conv"].append(row)
                torch.cuda.empty_cache()
    if not args.skip_edit:
        state = model_zoo.synthetic_state("sdxl")
        ed = FastEditor("sdxl", device="cuda:0", state=state, verbose=False)
        ed._engine.max_graphs = 2
        prompts = ["a watercolor painting"] * B
        sq = [Image.fromarray(S.synthetic_image(s, 1024, 1024)) for s in range(B)]

        def one(ims, wh):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            ed.edit_many(ims, prompts, strength=0.5, seed=0, size=wh)
            torch.cuda.synchronize()
            return (time.perf_counter() - t0) * 1e3

        def profiled(ims, wh):
            d_img = torch.from_numpy(np.stack([np.array(i) for i in ims])).to(dev)
            pe, pl = ed._encode_prompts(prompts, [""] * B)
            noises = [torch.cat(z, 0) for z in zip(*[ed._draw_noises(0, 2, wh) for _ in range(B)])]
            ops.PROFILE, ops.STAGES[:] = [], []
            ed._engine.edit_batch(d_img, pe, pl, noises, strength=0.5, use_graph=False)
            fam, st = ops.profile_summary(), ops.stage_summary()
            ops.PROFILE = None
            ops.STAGES[:] = []
            return dict(stages_ms={k: round(v, 2) for k, v in st.items()},
                        families_ms={f: dict(calls=d["calls"], ms=round(d["ms"], 2)) for f, d in sorted(fam.items(), key=lambda kv: -kv[1]["ms"])})

        res["edit_many"] = []
        for wh in buckets:
            ims = [Image.fromarray(S.synthetic_image(s, wh[1], wh[0])) for s in range(B)]
            one(ims, wh); one(sq, None)                     # warm-up + CUDA-graph capture of both sizes
            tb, ts = [], []
            for _ in range(args.reps):
                tb.append(one(ims, wh))
                ts.append(one(sq, None))
            mb, ms = float(np.median(tb)), float(np.median(ts))
            mp_b, mp_s = B * wh[0] * wh[1] / 1e6, B * 1024 * 1024 / 1e6
            row = dict(bucket=f"{wh[0]}x{wh[1]}", ms_per_step=round(mb, 2), ms_per_step_1024=round(ms, 2),
                       ms_per_mp=round(mb / mp_b, 3), ms_per_mp_1024=round(ms / mp_s, 3), per_mp_ratio=round((mb / mp_b) / (ms / mp_s), 4),
                       min_max=[round(min(tb), 2), round(max(tb), 2)], min_max_1024=[round(min(ts), 2), round(max(ts), 2)])
            print(json.dumps(row))
            row["profile"] = profiled(ims, wh)
            row["profile_1024"] = profiled(sq, (1024, 1024))
            res["edit_many"].append(row)
            ed._engine.release_graphs()
            torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
