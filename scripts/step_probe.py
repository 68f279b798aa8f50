#!/usr/bin/env python
"""One eager SDXL batch-8 edit (or one UNet step of it) inside a cudaProfilerStart/Stop range — the target of the whole-step ncu
pass that measures the time-weighted tensor-pipe utilisation over ALL launches (VERDICT r1 weak #6):

    ncu --profile-from-start off --clock-control none --csv --log-file gpurun_out/tp_edit.csv \
        --metrics sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_elapsed,gpu__time_duration.sum python scripts/step_probe.py edit
    ... python scripts/step_probe.py unet          # only one ControlNet + UNet evaluation (CFG batch of 16 rows)
    python scripts/ncu_tensor_pipe.py gpurun_out/tp_edit.csv gpurun_out/tp_unet.csv > profiles/r2_tensor_pipe_step.json
"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from fast_image_editing_with_generative_models_b200 import model_zoo, ops
from fast_image_editing_with_generative_models_b200 import synthetic as S

mode = sys.argv[1] if len(sys.argv) > 1 else "edit"
model = sys.argv[2] if len(sys.argv) > 2 else "sdxl"
B = int(sys.argv[3]) if len(sys.argv) > 3 else 8
dev = torch.device("cuda:0")
state = model_zoo.synthetic_state(model)
eng = model_zoo.build_engine(state, dev)
ucfg = eng.unet.cfg
imgs = torch.from_numpy(np.stack([S.synthetic_image(i, 1024, 1024) for i in range(B)])).to(dev)
pe, pl = S.synthetic_prompt(0, ucfg.cross_attention_dim, ucfg.projection_class_embeddings_input_dim - 6 * ucfg.addition_time_embed_dim)
pe, pl = pe.to(dev), pl.to(dev)
nz = [n.to(dev, torch.float16) for n in S.synthetic_noises(0, B, 128, 128)]
for _ in range(2):
    eng.edit_batch(imgs, pe, pl, nz, strength=0.5, use_graph=False)
torch.cuda.synchronize()
if mode == "edit":
    torch.cuda.profiler.start()
    eng.edit_batch(imgs, pe, pl, nz, strength=0.5, use_graph=False)
    torch.cuda.synchronize()
    torch.cuda.profiler.stop()
else:
    ctx = torch.cat([pe[0:1].expand(B, -1, -1), pe[1:2].expand(B, -1, -1)], 0).contiguous()
    te = torch.cat([pl[0:1].expand(B, -1), pl[1:2].expand(B, -1)], 0).contiguous()
    tid = [1024.0, 1024.0, 0.0, 0.0, 1024.0, 1024.0]
    ps_cn, ps_un = eng.cn.prepare_prompt(ctx, te, tid), eng.unet.prepare_prompt(ctx, te, tid)
    cond = eng.cn.cond_embedding(ops.preprocess_pad8(ops.canny(imgs, 100, 200, out_channels=3), normalize=False))
    cond = torch.cat([cond, cond], 0)
    x2 = torch.randn((2 * B, 128, 128, 4), device=dev).half()
    t = torch.full((2 * B,), 499.0, dtype=torch.float32, device=dev)          # per-row timesteps and ControlNet scales, as the edit
    scale = torch.full((2 * B,), 0.5, dtype=torch.float32, device=dev)        # reads them from its parameter block
    for it in range(2):
        if it == 1:
            torch.cuda.synchronize()
            torch.cuda.profiler.start()
        feats = eng.cn.encode(x2, t, ps_cn, cond, 77)
        eps = eng.unet.forward(x2, t, ps_un, nctx=77, merge=eng.cn.merge_into(feats, scale))
    torch.cuda.synchronize()
    torch.cuda.profiler.stop()
print("probe done", mode, ops.LAUNCHES)
