"""What a LoRA adapter change costs on the B200 (profiles/lora_swap_bench.json).

SDXL with synthetic weights (the LCM-LoRA fused at build, adapter "default_0") and one synthetic rank-64 style adapter on every LoRA
target of the UNet:

* ``set_adapters``: CUDA events around each call, alternating between two weight sets of the style adapter (0.5 and 1.0); the median,
  and the bytes the update moves (pristine read + live write of every adapted module, fp16 factor operands, fp32 device factors) over
  that time against the measured HBM copy peak DESIGN.md cites (6441.6 GB/s), and its GEMM FLOP;
* the alternative: building a new FastEditor with the adapter fused at load, plus its warm_up (graph capture);
* ``edit_many`` of one 1024^2 image with and without the adapter active, alternated in one process (same kernels: equal within noise);
* the device memory the pristine copies add.

    python scripts/lora_swap_bench.py --out DIR/lora_swap_bench.json [--switches 20] [--reps 7]
"""
import argparse
import json
import os
import subprocess
import sys
import time

HERE = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, HERE)
COPY_PEAK_GBS = 6441.6          # DESIGN.md section 3: measured device-to-device copy rate of the B200


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    name, power, clock = [v.strip() for v in q.stdout.strip().splitlines()[0].split(",")]
    return dict(card=name, power_limit=power, max_sm_clock=clock)


def median(v):
    v = sorted(v)
    return v[len(v) // 2] if len(v) % 2 else 0.5 * (v[len(v) // 2 - 1] + v[len(v) // 2])


def update_work(adapters):
    """Bytes and FLOP of one recompute of every module the active deltas touch (the arithmetic of lora._write)."""
    targets = adapters._all_targets()["unet"]
    nbytes = flop = 0
    for part, mod in adapters._written:
        t = targets[mod]
        r = sum(a.shape[0] for (n, p, m), (a, _) in adapters._dev_factors.items() if p == part and m == mod)
        kp = (3 * r + 63) // 64 * 64                             # factors as fp16 hi + lo pairs: K = 3 R
        phases = 4 if t.kind == "up2x" else 1
        n = t.weight[0].shape[1] if t.kind == "up2x" else t.weight.shape[1]
        w_bytes = phases * t.out * n * 2
        nbytes += 2 * w_bytes                                   # pristine read + live write
        nbytes += 2 * phases * (t.out + n) * kp * 2              # fp16 operands of the GEMM (written, then read)
        nbytes += (t.out + n * (9 if t.kind != "rows" else 1)) * r * 4     # fp32 factors on the device
        flop += phases * 2 * t.out * n * kp
    return nbytes, flop


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--switches", type=int, default=20)
    ap.add_argument("--reps", type=int, default=7)
    a = ap.parse_args()
    import torch
    from PIL import Image
    from fast_image_editing_with_generative_models_b200 import model_zoo
    from fast_image_editing_with_generative_models_b200 import synthetic as S
    from fast_image_editing_with_generative_models_b200.editor import FastEditor
    assert torch.cuda.is_available(), "lora_swap_bench measures on the GPU"
    dev = torch.device("cuda:0")
    res = dict(gpu_info(), torch=torch.__version__, model="sdxl (synthetic weights)", style_rank=64)
    state = model_zoo.synthetic_state("sdxl")
    style = S.make_lora_params(state["unet"], rank=64, seed=60)
    img = [Image.fromarray(S.synthetic_image(3, 1024, 1024))]
    ed = FastEditor("sdxl", verbose=False, state=state)
    ed.warm_up(1)
    torch.cuda.synchronize(dev)
    mem0 = torch.cuda.memory_allocated(dev)
    t0 = time.perf_counter()
    ed.pipe.load_lora_weights(style, adapter_name="style")
    torch.cuda.synchronize(dev)
    res["load_lora_weights_s"] = time.perf_counter() - t0
    res["memory_increase_gb"] = (torch.cuda.memory_allocated(dev) - mem0) / 1024 ** 3
    res["pristine_copies_gb"] = ed.pipe.adapters.pristine_bytes() / 1024 ** 3
    # set_adapters between two weight sets, CUDA events around each call
    times = []
    for i in range(a.switches + 2):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        ed.pipe.set_adapters(["default_0", "style"], [1.0, 0.5 if i % 2 else 1.0])
        e.record()
        e.synchronize()
        if i >= 2:
            times.append(s.elapsed_time(e))
    nbytes, flop = update_work(ed.pipe.adapters)
    ms = median(times)
    res["set_adapters_ms"] = dict(median=ms, min=min(times), max=max(times), n=len(times))
    res["set_adapters_bytes_gb"] = nbytes / 1e9
    res["set_adapters_tflop"] = flop / 1e12
    res["set_adapters_gbs"] = nbytes / 1e9 / (ms / 1e3)
    res["set_adapters_share_of_copy_peak"] = res["set_adapters_gbs"] / COPY_PEAK_GBS
    res["modules_written"] = len(ed.pipe.adapters._written)
    # edit_many with and without the adapter, alternated
    step = {"off": [], "on": []}
    for i in range(2 * a.reps + 2):
        key = "on" if i % 2 else "off"
        ed.pipe.set_adapters(["default_0", "style"], [1.0, 1.0 if key == "on" else 0.0])
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        ed.edit_many(img, "a watercolor", seed=1, micro_batch=1)
        torch.cuda.synchronize(dev)
        if i >= 2:
            step[key].append(time.perf_counter() - t0)
    res["edit_many_1x1024_s"] = {k: dict(median=median(v), min=min(v), max=max(v), n=len(v)) for k, v in step.items()}
    # the alternative: a new editor with the adapter fused at load (+ its graph capture)
    comb = {}
    for k in state["lora"]:
        if k.endswith(".lora_A.weight"):
            m = k[: -len(".lora_A.weight")]
            comb[k] = torch.cat([state["lora"][k], style[k]], 0)
            comb[m + ".lora_B.weight"] = torch.cat([state["lora"][m + ".lora_B.weight"], style[m + ".lora_B.weight"]], 1)
    del ed
    torch.cuda.empty_cache()
    t0 = time.perf_counter()
    ed2 = FastEditor("sdxl", verbose=False, state=dict(state, lora=comb))
    torch.cuda.synchronize(dev)
    t1 = time.perf_counter()
    ed2.warm_up(1)
    res["rebuild_fused_s"] = dict(build=t1 - t0, build_and_warm_up=time.perf_counter() - t0)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
