#!/usr/bin/env python
"""Headline benchmark: 1024x1024 4-step guided edits per second (BASELINE.json metric) on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W]            # N=1 directly; N>1 under torchrun (or self-spawned)
    python bench.py --impl reference ...                           # the reference's CPU path (oracle port) on host cores
    python bench.py --config {0,1,2,3}                             # the other BASELINE.json configurations
    python bench.py --dump-outputs DIR ...                         # also save the last timed step's outputs as DIR/*.npy

Default workload = BASELINE.json configs[3] (the configuration the images/s metric is quoted on): SDXL UNet (LCM-LoRA fused) +
ControlNet-Canny small + fp16-fix VAE topology, fp16, 8 synthetic 1024x1024 images per GPU per step, 4 LCM steps at strength 0.5
(2 executed UNet+ControlNet evaluations), CFG 1.5, ControlNet scale 0.5, Canny 100/200.  A "step" is one engine pass over the
per-GPU batch.  Images are sharded over ranks (weak scaling, no hot-path collective); the uint8 outputs are all-gathered over
NCCL after every step.

  value  device-resident inputs, ``EditEngine.edit_batch`` (CUDA-graph replay of the whole edit)
  e2e    the plugin call: host PIL images + prompt strings -> ``FastEditor.edit_many`` -> host PIL images; PIL->numpy->pinned->H2D,
         both CLIP text towers, per-image ``torch.Generator`` noise, the edit, D2H and ``Image.fromarray`` are all inside the timed region
  --config 0  the reference's own CPU case (configs[0]: SSD-1B, one image, fp32, host cores) == ``--impl reference --model ssd-1b``
  --config 1  Canny + VAE encode/decode only, batch 32 (memory-bound kernels)
  --config 2  SSD-1B full edit, batch 1 (latency)
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

TFLOP_PER_IMAGE = {"sdxl": 44.45, "ssd-1b": 34.22}      # BASELINE.md section 3 (CN-small, 2 executed steps)
VAE_TFLOP_PER_IMAGE = 4.887 + 10.486                     # encode + decode
_budget = os.environ.get("FIE_REF_BUDGET_S")
REF_BUDGET_S = float(_budget) if _budget else None       # optional wall budget of the timed CPU edits; unset: exactly --steps edits


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=int, default=3, choices=[0, 1, 2, 3], help="BASELINE.json configs[] index (default 3: the headline)")
    ap.add_argument("--model", default=None, choices=["sdxl", "ssd-1b"])
    ap.add_argument("--batch", type=int, default=None, help="images per GPU per step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--metrics-eval", action="store_true", help="time the evaluation metrics (MetricsCalculator, DESIGN 3.10) instead of the edit; a step = 4 image pairs")
    ap.add_argument("--no-graph", action="store_true", help="launch the ~2000 kernels of an edit eagerly instead of replaying one CUDA graph")
    ap.add_argument("--profile-out", default=None, help="write the per-kernel-family breakdown JSON here")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned as DIR/<name>.npy (float32 or float64)")
    a = ap.parse_args()
    if a.config == 0:
        a.impl = "reference"
    if a.model is None:
        a.model = "ssd-1b" if a.config in (0, 2) else "sdxl"
    if a.batch is None:
        a.batch = {0: 1, 1: 32, 2: 1, 3: 8}[a.config]
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs needs a B200 path (the reference arm returns no outputs)")
    return a


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons every 200 ms while the timed region runs."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) >= 7 and r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# The reference's CPU path: the fp32 oracle restatement of the diffusers pipeline on all host cores
# ------------------------------------------------------------------------------------------------

def cpu_reference_edit(state, size: int, threads: int):
    """ONE full edit of ONE image on the CPU — the reference's path as ``FastEditor(device="cpu", use_full_precision=True)`` would
    run it: Canny (plain-C oracle of cv2.Canny), VAE encode, 2 executed ControlNet + UNet CFG-pair evaluations with the LoRA
    applied unfused, LCM steps, VAE decode, fp32 torch CPU ops on ``threads`` threads.  -> (seconds, {stage: seconds})."""
    import numpy as np
    import torch
    from oracle import c_oracle
    from oracle import diffusion_oracle as O
    from fast_image_editing_with_generative_models_b200 import synthetic as S
    torch.set_num_threads(threads)
    img = S.synthetic_image(0, size, size)
    ucfg = state["unet_cfg"]
    pe, pl = S.synthetic_prompt(0, ucfg.cross_attention_dim, ucfg.projection_class_embeddings_input_dim - 6 * ucfg.addition_time_embed_dim)
    noises = S.synthetic_noises(0, 1, size // 8, size // 8)
    m = O.EditModels(ucfg, state["unet"], state["cn_cfg"], state["cn"], state["vae_cfg"], state["vae"], state.get("lora"), state.get("lora_scale", 1.0))
    marks = []
    t0 = time.perf_counter()
    marks.append(("canny", t0))
    with torch.no_grad():
        edges = c_oracle.canny_u8(img[None], 100, 200, replicate3=True)
        O.edit_pipeline(m, torch.from_numpy(img[None]), torch.from_numpy(edges), pe.float(), pl.float(), noises, strength=0.5,
                        num_inference_steps=4, guidance_scale=1.5, controlnet_conditioning_scale=0.5, dtype=torch.float32,
                        on_stage=lambda name: marks.append((name, time.perf_counter())))
    t1 = time.perf_counter()
    stages = {}
    for (n0, a), (_, b) in zip(marks[:-1], marks[1:]):
        stages[n0] = stages.get(n0, 0.0) + (b - a)
    return t1 - t0, stages


def cpu_model_name():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def timed_cpu_edits(state, edits: int, threads: int):
    """One untimed 64x64 warm-up (thread pools, oneDNN primitive caches), then ``edits`` full 1024x1024 edits; only when the
    FIE_REF_BUDGET_S wall budget is set, fewer (at least one) once another edit would overrun it.
    -> (list of seconds, stage split of the first)."""
    cpu_reference_edit(state, 64, threads)
    times, stages0 = [], None
    t_begin = time.perf_counter()
    while len(times) < edits:
        t, st = cpu_reference_edit(state, 1024, threads)
        times.append(t)
        stages0 = stages0 or st
        if REF_BUDGET_S is not None and (time.perf_counter() - t_begin) + t > REF_BUDGET_S:
            break
    return times, stages0


def run_reference(a):
    """--impl reference: the reference's own CPU implementation of the path, MEASURED at full size.  diffusers is not installable
    here (DESIGN.md section 4), so this is the oracle port (kind "port"); rank 0 only.  A step of this arm is a bounded sample of
    the GPU arm's step: ONE of its 1024x1024 images (the images of a step are independent)."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    from fast_image_editing_with_generative_models_b200 import model_zoo
    threads = os.cpu_count() or 1
    state = model_zoo.synthetic_state(a.model)
    times, stages = timed_cpu_edits(state, a.steps, threads)
    t = sum(times) / len(times)
    value = 1.0 / t
    bound = "" if REF_BUDGET_S is None else f", bounded by a {REF_BUDGET_S:.0f} s wall budget (FIE_REF_BUDGET_S)"
    sample = (f"{len(times)} timed full fp32 oracle edit(s) of ONE 1024x1024 image each (Canny + VAE encode + 2 x (ControlNet + UNet CFG pair) + "
              f"VAE decode, {a.model} + ControlNet-small widths, LoRA unfused as in the reference) on {threads} host threads "
              f"({cpu_model_name()}), after one untimed 64x64 warm-up; {a.steps} steps requested{bound}; "
              f"nothing is extrapolated")
    line = {"impl": "reference", "metric": "1024x1024 4-step edit images/sec", "value": value, "unit": "images/s", "n_gpus": a.gpus,
            "steps": len(times), "steps_requested": a.steps, "warmup": 1, "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            # the GPU arm's config, key for key (same workload); what a step of THIS arm is (one of its independent images) is stated in
            # cpu_baseline.sample and reference_step
            "config": arm_config(a, max(a.gpus, 1), launch="torch CPU ops (fp32 oracle port of the diffusers pipeline), all host threads"),
            "reference_step": "one timed step = ONE full 1024x1024 edit of one image of the workload's per-GPU batch (the images are independent)",
            "cpu_baseline": {"value": value, "unit": "images/s", "cores": threads, "kind": "port", "sample": sample,
                             "seconds_per_edit": [round(x, 2) for x in times], "stages_s": {k: round(v, 2) for k, v in (stages or {}).items()}},
            "e2e": {"value": value, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def workload_name(a):
    if a.config == 1:
        return f"Canny + VAE encode/decode only, fp16, {a.batch} x 1024x1024 images (BASELINE configs[1])"
    tag = {0: "configs[0], the reference's CPU case", 2: "configs[2], latency", 3: "configs[3]"}[a.config]
    return (f"{a.model.upper()} + LCM + ControlNet-Canny(small) + VAE full edit, {'fp32' if a.config == 0 else 'fp16'}, {a.batch} x 1024x1024 "
            f"images/GPU (BASELINE {tag}), 4 LCM steps @ strength 0.5 (2 executed), CFG 1.5")


def arm_config(a, world, launch):
    """The `config` object of the JSON line — identical keys and workload for the B200 arm and the reference arm."""
    return {"workload": workload_name(a), "images_per_gpu": a.batch, "global_batch": a.batch * world, "strength": 0.5, "executed_steps": 2,
            "cfg": 1.5, "parallelism": f"dp{world} (independent images, NCCL all-gather of uint8 outputs)",
            "weights": "seeded random-init of the named architectures", "launch": launch,
            "l2": "inputs larger than L2 (5 GB weights + GB-scale activations per step)"}


def load_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


DUMP_MAX_ELEMENTS = 4 << 20      # per array: 16 MB of float32, so the few arrays of a dump stay far below 64 MB


def dump_outputs(out_dir, arrays):
    """Writes each array of ``arrays`` (name -> numpy array) as ``out_dir/<name>.npy``: float64 stays float64, everything else
    becomes float32 (exact for the uint8 and fp16 outputs).  An array of more than DUMP_MAX_ELEMENTS elements is replaced by
    the flattened values at DUMP_MAX_ELEMENTS sorted positions drawn by a generator seeded with 0, so two runs with the same
    arguments sample the same positions and their files compare element for element."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, x in arrays.items():
        x = np.asarray(x)
        x = x.astype(np.float64 if x.dtype == np.float64 else np.float32)
        if x.size > DUMP_MAX_ELEMENTS:
            pick = np.sort(np.random.default_rng(0).choice(x.size, DUMP_MAX_ELEMENTS, replace=False))
            x = x.reshape(-1)[pick]
        np.save(os.path.join(out_dir, f"{name}.npy"), x)


def latest_profile_json(pattern):
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", pattern)))
    return json.load(open(files[-1])) if files else None


def _metrics_img(seed, h=512, w=512):
    import numpy as np
    rng = np.random.RandomState(seed)
    x = rng.rand(h, w, 3)
    for _ in range(3):
        x = (x + np.roll(x, 1, 0) + np.roll(x, 1, 1) + np.roll(x, -1, 0)) / 4
    x = (x - x.min()) / (x.max() - x.min())
    return (x * 255).astype(np.uint8)


def run_metrics_eval(a):
    """``--metrics-eval``: the evaluation metrics next to the path (SURVEY 8(f)-4, DESIGN 3.10) — ``MetricsCalculator.calculate_all_metrics``
    per image pair on the GPU (host PIL images in, Python floats out: the reference's call, src/metrics.py:338-381) with the per-metric split,
    and as ``cpu_baseline`` the CPU restatement (oracle/metrics_oracle.py: torch fp32 on all host cores, transformers' CLIP, torchvision's
    SqueezeNet) on the same pair.  One JSON line."""
    import time
    import warnings
    import numpy as np
    import torch
    pairs = a.steps * 4                 # one step = one pass over the 4 image pairs
    from PIL import Image
    from fast_image_editing_with_generative_models_b200 import ops
    from fast_image_editing_with_generative_models_b200.metrics import MetricsCalculator
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        calc = MetricsCalculator(device="cuda")
    src = [Image.fromarray(_metrics_img(i)) for i in range(4)]
    edited = [Image.fromarray(_metrics_img(100 + i, 1024, 1024)) for i in range(4)]        # the editor's 1024^2 outputs; metrics run on 512^2 Lanczos copies
    prompt = "a watercolor painting of a fox in the snow"
    for i in range(3):
        calc.calculate_all_metrics(src[i % 4], edited[i % 4], prompt)
    torch.cuda.synchronize()
    launches0 = ops.LAUNCHES
    t0 = time.perf_counter()
    for _ in range(a.steps):
        metrics = [calc.calculate_all_metrics(src[i], edited[i], prompt) for i in range(4)]
    torch.cuda.synchronize()
    per_pair = (time.perf_counter() - t0) / pairs
    launches = (ops.LAUNCHES - launches0) / pairs
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, {k: np.array([m[k] for m in metrics], np.float64) for k in metrics[0]})   # [4] per metric
    split = {}
    for name, fn in (("ssim", lambda: calc.calculate_ssim(src[0], edited[0])), ("lpips", lambda: calc.calculate_lpips(src[0], edited[0])),
                     ("clip_score", lambda: calc.calculate_clip_score(edited[0], prompt)), ("psnr", lambda: calc.calculate_psnr(src[0], edited[0])),
                     ("mse", lambda: calc.calculate_mse(src[0], edited[0])), ("dino_distance", lambda: calc.dino_metric.calculate_distance(src[0], edited[0]))):
        fn()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(10):
            fn()
        torch.cuda.synchronize()
        split[name] = round((time.perf_counter() - t0) / 10 * 1e3, 3)
    out = {"metric": "evaluated image pairs per second (all six metrics, PIL in -> floats out)", "value": round(1.0 / per_pair, 2), "unit": "pairs/s", "n_gpus": 1,
           "higher_is_better": True, "ms_per_pair": round(per_pair * 1e3, 2),
           "gpu_launches_per_pair": launches, "ms_per_metric": split, "weights": "synthetic (seeded random init)", "steps": a.steps, "pairs": pairs,
           "device": torch.cuda.get_device_name(0)}
    if not a.no_cpu_baseline:
        from oracle import metrics_oracle as MO
        from fast_image_editing_with_generative_models_b200 import lpips as L
        from fast_image_editing_with_generative_models_b200 import vit
        from fast_image_editing_with_generative_models_b200.metrics import clip_b16_text_config
        from fast_image_editing_with_generative_models_b200.text_encoder import make_clip_params, pseudo_token_ids
        from transformers import CLIPConfig, CLIPModel
        a = np.asarray(src[0])
        b = np.asarray(edited[0].resize((512, 512), Image.LANCZOS))
        cpu = {}

        def timed(name, fn, reps=2):
            fn()
            t0 = time.perf_counter()
            for _ in range(reps):
                fn()
            cpu[name] = round((time.perf_counter() - t0) / reps * 1e3, 1)
        timed("resize_lanczos", lambda: edited[0].resize((512, 512), Image.LANCZOS))
        timed("ssim", lambda: MO.ssim(a, b))
        timed("mse+psnr", lambda: (MO.mse(a, b), MO.psnr(a, b)))
        lp = L.make_lpips_params()
        feats, lins = MO.squeezenet_features(lp), [lp[f"lin{k}.model.1.weight"].reshape(-1) for k in range(7)]
        timed("lpips", lambda: MO.lpips_squeeze(feats, lins, a, b))
        vcfg, tcfg = vit.clip_b16_vision_config(), clip_b16_text_config()
        params = dict(vit.make_vit_params(vcfg)); params.update(make_clip_params(tcfg))
        hc = CLIPConfig(text_config=dict(vocab_size=tcfg.vocab_size, hidden_size=tcfg.hidden_size, intermediate_size=tcfg.intermediate_size, num_hidden_layers=tcfg.num_layers,
                                         num_attention_heads=tcfg.num_heads, eos_token_id=2, bos_token_id=0, pad_token_id=1),
                        vision_config=dict(hidden_size=vcfg.hidden_size, intermediate_size=vcfg.intermediate_size, num_hidden_layers=vcfg.num_layers,
                                           num_attention_heads=vcfg.num_heads, image_size=224, patch_size=16), projection_dim=512)
        hf = CLIPModel(hc).eval()
        hf.load_state_dict(params, strict=False)
        ids = pseudo_token_ids(prompt, tcfg.vocab_size).unsqueeze(0)
        timed("clip_score", lambda: MO.clip_score(hf, b, ids))
        dcfg = vit.dino_vitb8_config()
        dino = MO.DinoViT(vit.make_vit_params(dcfg), 8, 12)
        timed("dino_distance", lambda: MO.dino_distance(dino, a, b), reps=1)
        cpu["total"] = round(sum(cpu.values()), 1)
        out["cpu_baseline"] = {"kind": "port", "cores": torch.get_num_threads(), "ms_per_metric": cpu, "value": round(1e3 / cpu["total"], 3),
                               "unit": "pairs/s", "sample": "one 512^2 / 1024^2 pair, torch fp32 on the host cores"}
    print(json.dumps(out))


def main():
    a = parse()
    if a.impl == "reference":
        return run_reference(a)
    if a.metrics_eval:
        return run_metrics_eval(a)
    world_env = int(os.environ.get("WORLD_SIZE", "1"))
    if a.gpus > 1 and world_env == 1:
        # convenience: `python bench.py --gpus N` spawns the torchrun launch the driver would use
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={a.gpus}", "--master-addr", "127.0.0.1",
               "--master-port", os.environ.get("MASTER_PORT", "29511"), os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))

    import warnings
    import numpy as np
    import torch
    import torch.distributed as dist
    from PIL import Image
    from fast_image_editing_with_generative_models_b200 import _lib, model_zoo, ops, sweep
    from fast_image_editing_with_generative_models_b200 import synthetic as S
    from fast_image_editing_with_generative_models_b200.editor import FastEditor

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (B200); the product path has no CPU fallback")
    _lib.lib()   # fail loudly if the CUDA extension is missing
    rank, world, local = sweep.init_distributed()
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    B, H = a.batch, 1024
    peaks = load_peaks()
    peak_tf = float(peaks.get("bf16_tflops_sustained", 1400.0))
    peak_hbm = float(peaks.get("hbm_gbs", 6400.0))
    peak_src = "measured (MEASURED_PEAKS.json bf16_tflops_sustained; kernel timed inside a long step)" if peaks else "fallback (B200_PROFILING.md sustained ~1400)"

    state = model_zoo.synthetic_state(a.model)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")          # synthetic weights are the point here ("data": "synthetic")
        editor = FastEditor(model_name=a.model, device=f"cuda:{local}", enable_cpu_offload=False, state=state, text_encoders=True, verbose=False)
    eng = editor.pipe.engine
    eng.use_graphs = not a.no_graph      # one CUDA graph per edit (the product default of FastEditor); --no-graph = eager launches
    ucfg = eng.unet.cfg
    pooled_dim = ucfg.projection_class_embeddings_input_dim - 6 * ucfg.addition_time_embed_dim
    idx0 = rank * B
    imgs_np = np.stack([S.synthetic_image(idx0 + i, H, H) for i in range(B)])
    pe, pl = S.synthetic_prompt(0, ucfg.cross_attention_dim, pooled_dim)
    noises = S.synthetic_noises(idx0, B, H // 8, H // 8)
    imgs = torch.from_numpy(imgs_np).to(dev)
    pe_d, pl_d = pe.to(dev), pl.to(dev)
    nz_d = [n.to(dev, torch.float16) for n in noises]
    EDIT = dict(strength=0.5, num_inference_steps=4, guidance_scale=1.5, controlnet_conditioning_scale=0.5)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        return sweep.max_over_ranks(e0.elapsed_time(e1), dev)

    if a.config == 1:
        return run_config1(a, eng, imgs, dev, rank, world, peak_tf, peak_hbm, peak_src, timed, ClockSampler(local))

    last = {}

    def step():
        out = eng.edit_batch(imgs, pe_d, pl_d, nz_d, **EDIT)
        last["images"] = sweep.gather_outputs(out.images) if world > 1 else out.images
        last["edges"] = out.edges              # gathered after the timed region, for --dump-outputs only
        return last["images"]

    W = max(a.warmup, 3)
    for _ in range(W):
        step()
    # ---- timed region: device-resident inputs ----
    sampler = ClockSampler(local)
    sampler.start()
    l0 = ops.LAUNCHES
    ms = timed(step, a.steps, 0)
    launches = ops.LAUNCHES - l0
    clocks = sampler.stop()
    value = world * B * a.steps / (ms * 1e-3)
    if a.dump_outputs:
        # before any further edit: with graph replay the outputs are the graph's static buffers, which the next call overwrites.
        # With several ranks rank 0 writes every rank's images and edges (the gather is collective, so every rank takes part).
        edges = sweep.gather_outputs(last["edges"])         # the local tensor itself with one rank
        if rank == 0:
            dump_outputs(a.dump_outputs, {"images": last["images"].cpu().numpy(), "edges": edges.cpu().numpy()})

    # ---- end-to-end through the plugin API: FastEditor.edit_many on host PIL images and prompt strings -> host PIL images ----
    pil = [Image.fromarray(imgs_np[i]) for i in range(B)]
    call = [0]

    def e2e_call(n_batches):
        """One public-API call over n_batches x B images (the way run_batch.py drives a sweep): new prompts every call, so both CLIP
        towers run for every image; per-image generators; outputs come back as PIL images."""
        call[0] += 1
        images = pil * n_batches
        prompts = [f"edit {call[0]}: make image {j} look like a watercolour painting" for j in range(len(images))]
        outs = editor.edit_many(images, prompts, negative_prompt="", seeds=list(range(len(images))), micro_batch=B, **EDIT)
        assert len(outs) == len(images) and outs[-1].size == (H, H)
        return outs

    e2e_call(1)
    ms_e2e = timed(lambda: e2e_call(a.steps), 1, 0)                 # ONE call over steps x B images: host work pipelined under the GPU
    ms_e2e_1 = timed(lambda: e2e_call(1), max(min(a.steps, 3), 1), 0) / max(min(a.steps, 3), 1)   # one B-image call at a time: nothing overlaps
    tok = 2 * 77 * 4                                                 # int32 token ids of the two towers (neg + pos)
    h2d = B * H * H * 3 + B * tok
    d2h = B * H * H * 3
    e2e = {"value": world * B * a.steps / (ms_e2e * 1e-3), "unit": "images/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
           "api": f"FastEditor.edit_many({a.steps * B} PIL images, {a.steps * B} prompt strings, seeds) -> PIL images, micro-batches of {B}; "
                  "PIL->numpy->pinned->H2D, CLIP text towers, per-image torch.Generator noise, D2H and Image.fromarray inside the timed region",
           "ms_per_step": ms_e2e / a.steps,
           "single_call": {"images_per_call": B, "ms_per_call": ms_e2e_1, "value": world * B / (ms_e2e_1 * 1e-3),
                           "note": "one edit_many call per step: host staging and PIL conversion are not overlapped with GPU work"}}
    # the same call returning JPEG files encoded on the GPU (what run_batch.py writes for *.jpg targets): D2H shrinks to the file bytes
    def e2e_jpeg(n_batches):
        call[0] += 1
        images = pil * n_batches
        prompts = [f"edit {call[0]}: make image {j} look like a watercolour painting" for j in range(len(images))]
        files = editor.edit_many(images, prompts, negative_prompt="", seeds=list(range(len(images))), micro_batch=B, output="jpeg", **EDIT)
        assert len(files) == len(images) and files[0][:2] == b"\xff\xd8" and files[0][-2:] == b"\xff\xd9"
        return files
    jf = e2e_jpeg(1)
    ms_jpeg = timed(lambda: e2e_jpeg(a.steps), 1, 0)
    e2e["jpeg_output"] = {"value": world * B * a.steps / (ms_jpeg * 1e-3), "ms_per_step": ms_jpeg / a.steps,
                          "file_bytes_per_step": int(sum(len(f) for f in jf)), "d2h_prefix_bytes_per_image": int(getattr(editor, "_jpeg_prefix", 0)),
                          "api": "FastEditor.edit_many(..., output='jpeg') -> bytes of the *.jpg files (GPU baseline JPEG encoder, byte-identical to Pillow)"}
    # batch-1 latency of the reference's own call, FastEditor.edit (host PIL in -> host PIL out)
    lat = None
    if world == 1:
        editor.edit(image=pil[0], prompt="warm-up", seed=0, **EDIT)
        ms1 = timed(lambda: editor.edit(image=pil[0], prompt=f"latency probe {call[0]}", seed=0, **EDIT), 5, 1) / 5
        lat = {"api": "FastEditor.edit (1 PIL image -> 1 PIL image)", "model": a.model, "ms_per_edit": ms1}

    # ---- per-kernel-family attribution (one instrumented step, after the timed regions) ----
    eng.edit_batch(imgs, pe_d, pl_d, nz_d, strength=0.5, use_graph=False)      # untimed eager step: fills the caching allocator outside the graph pool
    torch.cuda.synchronize()
    ops.PROFILE = []
    ops.STAGES.clear()
    eng.edit_batch(imgs, pe_d, pl_d, nz_d, strength=0.5, use_graph=False)
    fam = ops.profile_summary()
    stages = ops.stage_summary()
    ops.PROFILE = None
    TC = ("gemm", "conv3x3", "conv_up2x")        # every launch of k_gemm_conv with a FLOP count (conv_up2x = 4 phase launches per call)
    tc_ms = sum(fam[k]["ms"] for k in TC if k in fam)
    tc_flop = sum(fam[k]["work"] for k in TC if k in fam)
    tc_calls = sum(fam[k]["calls"] * (4 if k == "conv_up2x" else 1) for k in TC if k in fam)
    total_ms = sum(d["ms"] for d in fam.values())
    achieved = tc_flop / (tc_ms * 1e-3) / 1e12 if tc_ms > 0 else 0.0
    traffic, traffic_src = None, None
    tj = latest_profile_json("r*_gemm_traffic.json")          # DRAM bytes per launch from the committed ncu --set full capture
    if tj:
        traffic, traffic_src = tj.get("dram_bytes_per_launch_avg"), tj.get("source")
    tp = latest_profile_json("r*_tensor_pipe_step.json")     # whole-step ncu pass: time-weighted sm__pipe_tensor_cycles_active over ALL launches
    roofline = {"kernel": "k_gemm_conv (tcgen05 GEMM / implicit-GEMM conv3x3)", "bound": "tensor", "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s",
                "frac": achieved / peak_tf, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src, "launches_per_step": tc_calls,
                "share_of_step": tc_ms / total_ms if total_ms else None,
                "flop_per_launch_avg": tc_flop / max(tc_calls, 1), "ms_per_launch_avg": tc_ms / max(tc_calls, 1)}
    breakdown = {k: {"calls": d["calls"], "ms": round(d["ms"], 3), "rate": (d["work"] / (d["ms"] * 1e-3) / (1e12 if d["unit"] == "FLOP" else 1e9)) if d["ms"] > 0 else 0.0,
                     "rate_unit": "TFLOP/s" if d["unit"] == "FLOP" else "GB/s"} for k, d in sorted(fam.items(), key=lambda kv: -kv[1]["ms"])}
    if a.profile_out and rank == 0:
        json.dump(breakdown, open(a.profile_out, "w"), indent=1)

    # ---- CPU baseline (rank 0, single-GPU run only): ONE measured full-size fp32 edit of one image of this workload ----
    cpu_baseline = None
    if world == 1 and not a.no_cpu_baseline:
        threads = os.cpu_count() or 1
        times, st = timed_cpu_edits(state, 1, threads)
        cpu_baseline = {"value": 1.0 / times[0], "unit": "images/s", "cores": threads, "kind": "port", "cpu": cpu_model_name(),
                        "sample": f"one full fp32 oracle edit of ONE 1024x1024 image of this workload ({a.model}, {times[0]:.1f} s measured, not extrapolated) "
                                  f"on {threads} host threads after a 64x64 warm-up",
                        "stages_s": {k: round(v, 2) for k, v in st.items()}}

    if rank == 0:
        upe = stages.get("unet_step", 0.0) / 2.0 if stages else None
        line = {"metric": "1024x1024 4-step edit images/sec", "value": value, "unit": "images/s", "n_gpus": world, "steps": a.steps,
                "warmup": W, "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f16", "data": "synthetic",
                "config": arm_config(a, world, launch="eager" if a.no_graph else "cuda-graph replay of the whole edit"),
                "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu_baseline,
                "image_roofline": {"tflop_per_image": TFLOP_PER_IMAGE[a.model], "achieved_tflops_per_gpu": value / world * TFLOP_PER_IMAGE[a.model],
                                   "frac_of_peak": value / world * TFLOP_PER_IMAGE[a.model] / peak_tf},
                # the other two quantities BASELINE.json's metric names: UNet step time and tensor-pipe utilisation
                "unet_step_ms": upe,          # per executed step, CFG batch of 2 x images_per_gpu rows
                "stages_ms": {k: round(v, 3) for k, v in stages.items()},
                "tensor_pipe": {"achieved_over_measured_peak": achieved / peak_tf,
                                "ncu_sm__pipe_tensor_cycles_active_pct": tp.get("tensor_pipe_active_pct_time_weighted") if tp else None,
                                "ncu_unet_step_pct": tp.get("unet_step_tensor_pipe_active_pct") if tp else None,
                                "ncu_source": tp.get("source") if tp else None},
                "latency_batch1": lat,
                "breakdown": breakdown}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_config1(a, eng, imgs, dev, rank, world, peak_tf, peak_hbm, peak_src, timed, sampler):
    """BASELINE configs[1]: Canny + VAE encode + VAE decode only, batch 32 of 1024x1024 images — the memory-bound kernels (Canny,
    GroupNorm) beside the VAE convolutions.  The batch is processed in chunks of 8 images (activation memory), a step = all 32."""
    import torch
    from fast_image_editing_with_generative_models_b200 import ops
    B = imgs.shape[0]
    CH = 8
    vae = eng.vae
    lat = [torch.randn((CH, 128, 128, 4), device=dev, generator=torch.Generator(dev).manual_seed(i)).half() for i in range(B // CH)]
    last = {}

    def step():
        edges = ops.canny(imgs, 100, 200, out_channels=3)
        outs = []
        for c in range(B // CH):
            vae.encode_moments(ops.preprocess_pad8(imgs[c * CH:(c + 1) * CH], True))
            outs.append(ops.postprocess(vae.decode(lat[c])))
        last["edges"], last["images"] = edges, outs
        return edges, outs

    W = max(a.warmup, 3)
    for _ in range(W):
        step()
    sampler.start()
    l0 = ops.LAUNCHES
    ms = timed(step, a.steps, 0)
    launches = ops.LAUNCHES - l0
    clocks = sampler.stop()
    if a.dump_outputs:
        from fast_image_editing_with_generative_models_b200 import sweep
        got = {"edges": last["edges"], "images": torch.cat(last["images"])}
        got = {k: sweep.gather_outputs(v) for k, v in got.items()}      # collective (every rank takes part); local with one rank
        if rank == 0:
            dump_outputs(a.dump_outputs, {k: v.cpu().numpy() for k, v in got.items()})
    ops.PROFILE = []
    step()
    fam = ops.profile_summary()
    ops.PROFILE = None
    TC = ("gemm", "conv3x3", "conv_up2x")
    tc_ms = sum(fam[k]["ms"] for k in TC if k in fam)
    tc_flop = sum(fam[k]["work"] for k in TC if k in fam)
    tc_calls = sum(fam[k]["calls"] * (4 if k == "conv_up2x" else 1) for k in TC if k in fam)
    achieved = tc_flop / (tc_ms * 1e-3) / 1e12 if tc_ms else 0.0
    hbm = {}
    for k in ("canny", "groupnorm"):
        if k in fam and fam[k]["ms"] > 0:
            gbs = fam[k]["work"] / (fam[k]["ms"] * 1e-3) / 1e9
            hbm[k] = {"bound": "hbm", "achieved": gbs, "peak": peak_hbm, "unit": "GB/s", "frac": gbs / peak_hbm, "ms": round(fam[k]["ms"], 3), "calls": fam[k]["calls"]}
    value = world * B * a.steps / (ms * 1e-3)
    if rank == 0:
        line = {"metric": "1024x1024 Canny + VAE encode/decode images/sec", "value": value, "unit": "images/s", "n_gpus": world, "steps": a.steps, "warmup": W,
                "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
                "config": {"workload": workload_name(a), "images_per_gpu": B, "chunk": CH, "l2": "inputs larger than L2"},
                "clocks": clocks, "e2e": None, "gpu_launches": int(launches),
                "roofline": {"kernel": "k_gemm_conv (VAE convolutions)", "bound": "tensor", "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s",
                             "frac": achieved / peak_tf, "traffic": None, "peak_source": peak_src, "launches_per_step": tc_calls},
                "hbm_rooflines": hbm, "cpu_baseline": None,
                "image_roofline": {"tflop_per_image": VAE_TFLOP_PER_IMAGE, "achieved_tflops_per_gpu": value / world * VAE_TFLOP_PER_IMAGE,
                                   "frac_of_peak": value / world * VAE_TFLOP_PER_IMAGE / peak_tf},
                "breakdown": {k: {"calls": d["calls"], "ms": round(d["ms"], 3)} for k, d in sorted(fam.items(), key=lambda kv: -kv[1]["ms"])}}
        print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
