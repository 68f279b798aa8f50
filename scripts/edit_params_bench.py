"""Per-image edit settings on the B200: what a changed setting costs (profiles/edit_params_bench.json).

(a) slider: SDXL 1024^2, warm_up, then FastEditor.edit calls, each with a new (controlnet_conditioning_scale, guidance_scale) pair
    (guidance > 1): per-call latency (first and median), graph captures and torch.cuda.memory_reserved.  Only the scalar edit() API is
    used, so ``--repo`` may point at an older checkout of the project for the before numbers.
(b) mixed micro-batch: edit_many of 8 images with 8 distinct settings against the same images with one setting, alternated, and against
    one edit_many call per setting (the only way to mix settings before they were device data).

Times: a host clock around work that ends in a device synchronise (edit / edit_many return host images); medians of alternating
repetitions.  The card's name, power limit and max SM clock are read in the same run.

    python scripts/edit_params_bench.py --out DIR/edit_params_bench.json [--repo PATH] [--parts ab] [--calls 12] [--reps 5]
"""
import argparse
import json
import os
import subprocess
import sys
import time

HERE = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    name, power, clock = [v.strip() for v in q.stdout.strip().splitlines()[0].split(",")]
    return dict(card=name, power_limit=power, max_sm_clock=clock)


def median(v):
    v = sorted(v)
    return v[len(v) // 2] if len(v) % 2 else 0.5 * (v[len(v) // 2 - 1] + v[len(v) // 2])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--repo", default=HERE, help="checkout whose package is measured")
    ap.add_argument("--parts", default="ab")
    ap.add_argument("--calls", type=int, default=12)
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    sys.path.insert(0, os.path.abspath(a.repo))
    import torch
    from PIL import Image
    from fast_image_editing_with_generative_models_b200.editor import FastEditor
    from fast_image_editing_with_generative_models_b200.synthetic import synthetic_image
    assert torch.cuda.is_available(), "edit_params_bench measures on the GPU"
    dev = torch.device("cuda:0")
    res = dict(gpu_info(), repo=os.path.abspath(a.repo), torch=torch.__version__)
    ed = FastEditor("sdxl", verbose=False)
    eng = ed._engine
    captures = [0]
    orig = eng._capture

    def counted(*args, **kw):
        captures[0] += 1
        return orig(*args, **kw)
    eng._capture = counted
    ims = [Image.fromarray(synthetic_image(s, 1024, 1024)) for s in range(8)]
    if "a" in a.parts:
        t0 = time.perf_counter()
        ed.warm_up(micro_batch=1, strength=0.5, guidance_scale=1.5)
        warm = time.perf_counter() - t0
        c0 = captures[0]
        lat = []
        for i in range(a.calls):
            cs, gs = 0.3 + 0.5 * i / max(a.calls - 1, 1), 1.5 + 2.5 * ((7 * i) % a.calls) / max(a.calls - 1, 1)
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
            ed.edit(ims[i % 8], "a watercolor painting", strength=0.5, guidance_scale=gs, controlnet_conditioning_scale=cs, seed=i)
            torch.cuda.synchronize(dev)
            lat.append(time.perf_counter() - t0)
        res["slider"] = dict(calls=a.calls, warm_up_s=round(warm, 3), first_call_ms=round(1e3 * lat[0], 2), median_call_ms=round(1e3 * median(lat), 2),
                             max_call_ms=round(1e3 * max(lat), 2), captures_during_calls=captures[0] - c0,
                             graphs_cached=len(eng._graphs), memory_reserved_gb=round(torch.cuda.memory_reserved(dev) / 2 ** 30, 2))
        print(json.dumps(res["slider"]), flush=True)
    if "b" in a.parts:
        gs = [1.5 + i / 7 for i in range(8)]
        cs = [0.3 + 0.5 * i / 7 for i in range(8)]
        lo, hi = [80 + 5 * i for i in range(8)], [180 + 10 * i for i in range(8)]
        mixed = lambda: ed.edit_many(ims, "a watercolor painting", strength=0.5, guidance_scale=gs, controlnet_conditioning_scale=cs,
                                     canny_low_threshold=lo, canny_high_threshold=hi, seeds=list(range(8)))
        uniform = lambda: ed.edit_many(ims, "a watercolor painting", strength=0.5, guidance_scale=2.0, controlnet_conditioning_scale=0.5,
                                       seeds=list(range(8)))
        per_setting = lambda: [ed.edit_many([ims[i]], "a watercolor painting", strength=0.5, guidance_scale=gs[i], controlnet_conditioning_scale=cs[i],
                                            canny_low_threshold=lo[i], canny_high_threshold=hi[i], seeds=[i]) for i in range(8)]
        for f in (mixed, uniform, per_setting):
            f()
        c0 = captures[0]
        t = {"mixed": [], "uniform": [], "per_setting": []}
        for _ in range(a.reps):
            for name, f in (("mixed", mixed), ("uniform", uniform), ("per_setting", per_setting)):
                torch.cuda.synchronize(dev)
                t0 = time.perf_counter()
                f()
                torch.cuda.synchronize(dev)
                t[name].append(time.perf_counter() - t0)
        res["mixed_micro_batch"] = dict(images=8, reps=a.reps, captures_during_reps=captures[0] - c0,
                                        **{f"{k}_ms": round(1e3 * median(v), 2) for k, v in t.items()},
                                        **{f"{k}_all_ms": [round(1e3 * x, 2) for x in v] for k, v in t.items()})
        print(json.dumps(res["mixed_micro_batch"]), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
