"""CPU: host side of per-image edit settings -- broadcasting and validation, edit_many's grouping by (size, executed steps, CFG),
the per-image scheduler tables, the parameter block layout, the Canny threshold normalisation (against cv2) and the graph key."""
import math

import cv2
import numpy as np
import pytest
import torch

from fast_image_editing_with_generative_models_b200 import ops
from fast_image_editing_with_generative_models_b200.editor import micro_batches
from fast_image_editing_with_generative_models_b200.pipeline import EditParams, graph_key, per_image, per_image_settings
from fast_image_editing_with_generative_models_b200.scheduler import LCMSchedule


def test_per_image_broadcasts_scalars_and_checks_sequences():
    assert per_image("guidance_scale", 1.5, 3) == [1.5, 1.5, 1.5]
    assert per_image("guidance_scale", [1.5, 2, np.float32(3.0)], 3) == [1.5, 2, 3.0]
    assert per_image("canny_low", np.array([1, 2]), 2) == [1, 2]
    with pytest.raises(ValueError, match="2 values for 3 images"):
        per_image("guidance_scale", [1.5, 2.0], 3)
    with pytest.raises(ValueError, match="image 1 must be a finite number"):
        per_image("controlnet_conditioning_scale", [0.5, float("nan")], 2)
    with pytest.raises(ValueError, match="image 0 must be a finite number"):
        per_image("strength", float("inf"), 2)
    with pytest.raises(ValueError, match="must be a number"):
        per_image("strength", "0.5", 2)


def test_per_image_settings_validation_names_the_image():
    st = per_image_settings(3, [0.5, 0.25, 1.0], [4, 8, 2], 1.5, [0.3, 0.4, 0.5], 100, [200, 150, 250])
    assert st["n_exec"] == [2, 2, 2]
    assert st["controlnet_conditioning_scale"] == [0.3, 0.4, 0.5] and st["canny_low_threshold"] == [100] * 3
    with pytest.raises(ValueError, match=r"image 1: The value of strength should in \[0.0, 1.0\] but is 1.5"):
        per_image_settings(2, [0.5, 1.5], 4, 1.5, 0.5, 100, 200)
    with pytest.raises(ValueError, match="image 2: `num_inference_steps` has to be a positive integer"):
        per_image_settings(3, 0.5, [4, 4, 2.5], 1.5, 0.5, 100, 200)
    with pytest.raises(ValueError, match="image 0: After adjusting the num_inference_steps by strength parameter: 0.1"):
        per_image_settings(2, [0.1, 0.5], 4, 1.5, 0.5, 100, 200)
    with pytest.raises(ValueError, match="1 values for 2 images"):
        per_image_settings(2, 0.5, [4], 1.5, 0.5, 100, 200)
    with pytest.raises(ValueError, match="canny_high_threshold of image 1"):
        per_image_settings(2, 0.5, 4, 1.5, 0.5, 100, [200, float("nan")])


def test_micro_batches_group_by_size_steps_and_cfg_in_input_order():
    sizes = [(1024, 1024)] * 6 + [(1152, 896)] * 2
    n_exec = [2, 2, 4, 2, 2, 2, 2, 2]
    guidance = [1.5, 1.0, 2.0, 2.5, 1.5, 0.5, 1.5, 1.5]
    plan = micro_batches(sizes, n_exec, guidance, 2)
    assert plan == [(((1024, 1024), 2, True), [0, 3]), (((1024, 1024), 2, True), [4]), (((1024, 1024), 2, False), [1, 5]),
                    (((1024, 1024), 4, True), [2]), (((1152, 896), 2, True), [6, 7])]
    # every image exactly once; results are written back by index, so they come back in input order
    assert sorted(i for _, idx in plan for i in idx) == list(range(8))
    for (wh, n, cfg), idx in plan:
        assert all(sizes[i] == wh and n_exec[i] == n and (guidance[i] > 1) == cfg for i in idx)


def test_batch_tables_equal_the_scalar_schedule_per_image():
    sched = LCMSchedule()
    steps, strengths, guidance = [4, 8, 5, 3], [0.5, 0.25, 0.4, 0.7], [1.5, 2.25, 1.75, 3.0]
    ts, add, table = sched.batch_tables(steps, strengths, guidance)
    assert add.dtype == np.float32 and table.dtype == np.float32 and table.shape == (2, 4, 7)
    for i in range(4):
        ref = LCMSchedule()
        t, begin = ref.img2img_timesteps(steps[i], strengths[i])
        assert ts[i] == t
        assert add[i].tolist() == np.float32(ref.add_noise_coeffs(t[0])).tolist()
        for k in range(len(t)):
            c = ref.step_coeffs(begin + k)
            want = np.array([guidance[i]] + [c[n] for n in LCMSchedule.STEP_COLUMNS[1:]], dtype=np.float32)
            assert table[k, i].tobytes() == want.tobytes()
    assert ts[0] == [499, 259] and ts[1] == [259, 139]          # same step count, different timesteps
    with pytest.raises(ValueError, match="image 1"):
        sched.batch_tables([4, 4], [0.5, 0.75], [1.5, 1.5])


def test_parameter_block_layout():
    sched = LCMSchedule()
    p = EditParams.pack(sched, 3, strength=[0.5, 0.25, 0.5], num_inference_steps=[4, 8, 4], guidance_scale=[1.5, 2.0, 2.5],
                        controlnet_conditioning_scale=[0.3, 0.6, 0.9], canny_low=[100, 250.7, -3], canny_high=[200, 120, 5000])
    assert (p.n_images, p.n_exec, p.cfg) == (3, 2, True) and p.block.dtype == np.float32
    v = p.views(torch.from_numpy(p.block.copy()))
    assert v["thr"].tolist() == [[100, 200], [120, 250], [0, 2040]]
    assert v["scale"].tolist() == pytest.approx([0.3, 0.6, 0.9] * 2)
    assert v["t"].tolist() == [[499, 259, 499] * 2, [259, 139, 259] * 2]
    ts, add, table = LCMSchedule().batch_tables([4, 8, 4], [0.5, 0.25, 0.5], [1.5, 2.0, 2.5])
    assert v["add"].numpy().tobytes() == add.tobytes() and v["step"].numpy().tobytes() == table.tobytes()
    # no CFG: one row per image and guidance 1 in the step table
    q = EditParams.pack(sched, 2, guidance_scale=[1.0, 0.5])
    w = q.views(torch.from_numpy(q.block.copy()))
    assert not q.cfg and w["scale"].numel() == 2 and w["t"].shape == (2, 2) and w["step"][:, :, 0].eq(1.0).all()
    with pytest.raises(ValueError, match="all be > 1"):
        EditParams.pack(sched, 2, guidance_scale=[1.5, 1.0])
    with pytest.raises(ValueError, match="image 1 executes 3 denoising steps, image 0 executes 2"):
        EditParams.pack(sched, 2, strength=[0.5, 0.75])
    with pytest.raises(ValueError, match=r"image 0: The value of strength should in \[0.0, 1.0\] but is -0.5"):
        EditParams.pack(sched, 1, strength=-0.5)


def test_graph_key_keeps_only_what_changes_the_launch_sequence():
    sched = LCMSchedule()
    shapes = ((4, 256, 256, 3), (2, 77, 2048), (2, 1280), 3)
    a = EditParams.pack(sched, 4, guidance_scale=1.5, controlnet_conditioning_scale=0.5, canny_low=100, canny_high=200)
    b = EditParams.pack(sched, 4, strength=[0.5, 0.25, 0.5, 0.5], num_inference_steps=[4, 8, 4, 4], guidance_scale=[1.5, 2.0, 3.0, 7.5],
                        controlnet_conditioning_scale=[0.1, 0.2, 0.3, 0.9], canny_low=[10, 20, 30, 40], canny_high=[50, 60, 70, 80])
    assert graph_key(*shapes, a, False) == graph_key(*shapes, b, False)
    assert graph_key(*shapes, a, False) != graph_key(*shapes, a, True)                                         # blur
    assert graph_key(*shapes, a, False) != graph_key(*shapes, EditParams.pack(sched, 4, guidance_scale=1.0), False)   # CFG
    assert graph_key(*shapes, a, False) != graph_key(*shapes, EditParams.pack(sched, 4, strength=0.75), False)        # n_exec
    assert graph_key(*shapes, a, False) != graph_key((4, 512, 512, 3), *shapes[1:], a, False)                  # size


@pytest.mark.parametrize("low,high", [(100, 200), (200, 100), (-5, 5000), (-100, -50), (3000, 4000), (-1, 30), (99.7, 200.2),
                                      (2040.5, 2100), (0, 0), (50.5, 50.2), (2039, 2041)])
def test_canny_threshold_normalisation_matches_cv2(low, high):
    lo, hi = ops.canny_thresholds(low, high)
    assert 0 <= lo <= hi <= 2040 and isinstance(lo, int) and isinstance(hi, int)
    rng = np.random.default_rng(int(abs(low) * 7 + abs(high)) % 1000)
    imgs = [rng.integers(0, 256, (61, 83), dtype=np.uint8),                                     # random
            cv2.GaussianBlur(rng.integers(0, 256, (64, 96), dtype=np.uint8), (9, 9), 3),        # smooth
            np.tile(np.arange(0, 256, 4, dtype=np.uint8), (40, 2)),                             # ramp
            (np.indices((48, 48)).sum(0) % 2 * 255).astype(np.uint8)]                           # checkerboard: maximal magnitudes
    for g in imgs:
        assert np.array_equal(cv2.Canny(g, low, high), cv2.Canny(g, lo, hi)), (low, high, lo, hi)
    assert math.floor(min(low, high)) <= 0 or lo == min(2040, math.floor(min(low, high)))
