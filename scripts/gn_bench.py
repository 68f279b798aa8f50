#!/usr/bin/env python
"""GroupNorm timing per shape under both slab policies (fie_tune_groupnorm_slab 0: always the two-kernel path, 1: the default):
the UNet / ControlNet / VAE shapes of an SDXL batch-8 edit."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from fast_image_editing_with_generative_models_b200 import _lib, ops

dev = torch.device("cuda:0")
SHAPES = [(16, 1024, 1280, 0), (16, 1024, 1280, 1280), (16, 1024, 1280, 640), (16, 4096, 640, 0), (16, 4096, 1280, 640), (16, 4096, 640, 640), (16, 4096, 640, 320),
          (16, 16384, 320, 0), (16, 16384, 640, 320), (16, 16384, 320, 320), (8, 16384, 512, 0), (8, 65536, 512, 0), (8, 262144, 256, 0), (8, 1048576, 128, 0)]
for slab in (0, 1):
    _lib.lib().fie_tune_groupnorm_slab(slab)
    tot = 0.0
    for n, hw, c0, c1 in SHAPES:
        x0 = torch.randn((n, hw, c0), device=dev).half()
        x1 = torch.randn((n, hw, c1), device=dev).half() if c1 else None
        g, b = torch.ones(c0 + c1, device=dev), torch.zeros(c0 + c1, device=dev)
        for _ in range(3):
            ops.groupnorm(x0, g, b, 1e-5, True, 32, x1)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        it = 20
        e0.record()
        for _ in range(it):
            ops.groupnorm(x0, g, b, 1e-5, True, 32, x1)
        e1.record(); torch.cuda.synchronize()
        us = e0.elapsed_time(e1) / it * 1e3
        gb = 4.0 * n * hw * (c0 + c1) / 1e9
        tot += us
        print(f"slab {slab} [{n},{hw},{c0}+{c1}]  {us:8.1f} us  {gb / (us * 1e-6):8.0f} GB/s (algorithmic read+write)", flush=True)
    print("slab", slab, " total", round(tot, 1), "us")
_lib.lib().fie_tune_groupnorm_slab(1)
