"""Host-side LCMScheduler logic (timestep table and per-image coefficient tables); the arithmetic on latents runs in
``fie_cfg_lcm_step_batched`` / ``fie_vae_sample_add_noise_batched``.  Mirrors diffusers ``LCMScheduler`` as configured by the
reference (``LCMScheduler.from_config(..., timestep_spacing="trailing")``, ``src/pipeline.py:138-141,158-161``):
scaled_linear betas 0.00085..0.012 over 1000 steps, epsilon prediction, original_inference_steps 50,
timestep_scaling 10, sigma_data 0.5."""
from __future__ import annotations

from typing import Dict, List, Sequence, Tuple

import numpy as np


class LCMSchedule:
    def __init__(self, num_train_timesteps: int = 1000, beta_start: float = 0.00085, beta_end: float = 0.012,
                 original_inference_steps: int = 50, timestep_scaling: float = 10.0):
        betas = np.linspace(np.float32(beta_start) ** 0.5, np.float32(beta_end) ** 0.5, num_train_timesteps, dtype=np.float32) ** 2
        self.alphas_cumprod = np.cumprod((1.0 - betas).astype(np.float32), dtype=np.float32)
        self.num_train_timesteps = num_train_timesteps
        self.original_inference_steps = original_inference_steps
        self.timestep_scaling = timestep_scaling
        self.sigma_data = 0.5
        self.timesteps: List[int] = []

    def set_timesteps(self, n: int) -> List[int]:
        k = self.num_train_timesteps // self.original_inference_steps
        origin = (np.arange(1, self.original_inference_steps + 1) * k - 1)[::-1]
        idx = np.floor(np.linspace(0, len(origin), num=n, endpoint=False)).astype(np.int64)
        self.timesteps = [int(v) for v in origin[idx]]
        return self.timesteps

    def img2img_timesteps(self, n: int, strength: float) -> Tuple[List[int], int]:
        """diffusers img2img ``get_timesteps``: keeps the last int(n*strength) steps; returns (timesteps, begin_index)."""
        self.set_timesteps(n)
        init = min(int(n * strength), n)
        t_start = max(n - init, 0)
        return self.timesteps[t_start:], t_start

    def add_noise_coeffs(self, t: int) -> Tuple[float, float]:
        a = float(self.alphas_cumprod[t])
        return a ** 0.5, (1.0 - a) ** 0.5

    STEP_COLUMNS = ("guidance", "sqrt_a", "sqrt_1ma", "c_skip", "c_out", "sqrt_a_prev", "sqrt_1ma_prev")

    def batch_tables(self, steps: Sequence[int], strengths: Sequence[float], guidance: Sequence[float]):
        """Per-image schedules of one batch, every image with its own ``(num_inference_steps, strength)`` and guidance (pass 1.0 for a
        batch without CFG) -> (timesteps [B][n_exec], add-noise coefficients fp32 [B, 2] = (sqrt_a, sqrt_1ma) at each image's first
        timestep, step table fp32 [n_exec, B, 7] in the columns of ``STEP_COLUMNS``), the values of :meth:`add_noise_coeffs` and
        :meth:`step_coeffs` rounded to fp32.  Every image must execute the same number of steps (one launch sequence)."""
        ts, add, rows = [], [], []
        for i, (n, st) in enumerate(zip(steps, strengths)):
            t, begin = self.img2img_timesteps(int(n), float(st))
            if ts and len(t) != len(ts[0]):
                raise ValueError(f"image {i}: {n} steps at strength {st} execute {len(t)} steps, image 0 executes {len(ts[0])}; "
                                 "the images of one batch must execute the same number of steps")
            ts.append(t)
            add.append(self.add_noise_coeffs(t[0]))
            cs = [self.step_coeffs(begin + k) for k in range(len(t))]
            rows.append([[float(guidance[i])] + [c[name] for name in self.STEP_COLUMNS[1:]] for c in cs])
        table = np.asarray(rows, dtype=np.float32).transpose(1, 0, 2) if rows else np.zeros((0, 0, 7), np.float32)
        return ts, np.asarray(add, dtype=np.float32).reshape(-1, 2), np.ascontiguousarray(table)

    def step_coeffs(self, step_index: int) -> Dict[str, float]:
        t = self.timesteps[step_index]
        last = step_index == len(self.timesteps) - 1
        prev_t = t if last else self.timesteps[step_index + 1]
        a_t, a_prev = float(self.alphas_cumprod[t]), float(self.alphas_cumprod[prev_t])
        s = t * self.timestep_scaling
        return dict(t=t, last=last, sqrt_a=a_t ** 0.5, sqrt_1ma=(1 - a_t) ** 0.5,
                    c_skip=self.sigma_data ** 2 / (s ** 2 + self.sigma_data ** 2), c_out=s / (s ** 2 + self.sigma_data ** 2) ** 0.5,
                    sqrt_a_prev=a_prev ** 0.5, sqrt_1ma_prev=(1 - a_prev) ** 0.5)
