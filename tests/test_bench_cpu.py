"""CPU: the host-side pieces of bench.py — the measured CPU reference leg (the fp32 oracle, stage split) and the argument handling
that maps BASELINE.json configs[] to workloads.  The GPU legs are exercised by the driver's bench run."""
import sys

import pytest


def test_cpu_reference_edit_runs_the_whole_path_and_splits_stages():
    import bench
    from fast_image_editing_with_generative_models_b200 import model_zoo
    state = model_zoo.synthetic_state("sdxl", tiny=True)
    t, stages = bench.cpu_reference_edit(state, 64, 2)
    assert t > 0 and {"canny", "vae_encode", "controlnet_step", "unet_step", "vae_decode"} <= set(stages)
    assert abs(sum(stages.values()) - t) < 0.05 * t + 0.05                      # the split accounts for the measured time


@pytest.mark.parametrize("argv,model,batch,impl", [([], "sdxl", 8, "b200"), (["--config", "2"], "ssd-1b", 1, "b200"), (["--config", "1"], "sdxl", 32, "b200"),
                                                  (["--config", "0"], "ssd-1b", 1, "reference"), (["--impl", "reference"], "sdxl", 8, "reference"),
                                                  (["--model", "ssd-1b", "--batch", "4"], "ssd-1b", 4, "b200")])
def test_config_switch(monkeypatch, argv, model, batch, impl):
    import bench
    monkeypatch.setattr(sys, "argv", ["bench.py"] + argv)
    a = bench.parse()
    assert (a.model, a.batch, a.impl) == (model, batch, impl)
    assert "1024x1024" in bench.workload_name(a)


@pytest.mark.parametrize("steps,budget,timed", [(5, None, 5), (3, None, 3), (5, 100.0, 1)])
def test_reference_arm_times_the_requested_steps(monkeypatch, capsys, steps, budget, timed):
    """--impl reference --steps K times exactly K full-size edits, however long each takes; only an explicit FIE_REF_BUDGET_S cuts
    the count short.  The edit is replaced by a stub that reports 200 s per 1024x1024 edit."""
    import json
    import bench
    from fast_image_editing_with_generative_models_b200 import model_zoo
    sizes = []

    def fake_edit(state, size, threads):
        sizes.append(size)
        return 200.0, {"unet_step": 200.0}
    monkeypatch.setattr(bench, "cpu_reference_edit", fake_edit)
    monkeypatch.setattr(bench, "REF_BUDGET_S", budget)
    monkeypatch.setattr(model_zoo, "synthetic_state", lambda name: {})
    monkeypatch.setattr(sys, "argv", ["bench.py", "--impl", "reference", "--steps", str(steps)])
    bench.run_reference(bench.parse())
    line = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    assert sizes == [64] + [1024] * timed
    assert line["steps"] == timed and line["steps_requested"] == steps and len(line["cpu_baseline"]["seconds_per_edit"]) == timed


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "d"], ["--config", "0", "--dump-outputs", "d"]])
def test_rejected_arguments(monkeypatch, argv):
    import bench
    monkeypatch.setattr(sys, "argv", ["bench.py"] + argv)
    with pytest.raises(SystemExit):
        bench.parse()


def test_dump_outputs_types_and_seeded_sample(tmp_path):
    """Small arrays are written whole as float32 (float64 kept); a large one becomes the same seeded sample on every call."""
    import numpy as np
    import bench
    big = np.random.default_rng(1).integers(0, 256, bench.DUMP_MAX_ELEMENTS + 1000, dtype=np.uint8)
    small = np.arange(12, dtype=np.float16).reshape(3, 4)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"images": big, "edges": small, "psnr": np.float64(31.25)})
    got = {p.stem: np.load(p) for p in (tmp_path / "a").glob("*.npy")}
    assert set(got) == {"images", "edges", "psnr"}
    assert got["edges"].dtype == np.float32 and np.array_equal(got["edges"], small.astype(np.float32))
    assert got["psnr"].dtype == np.float64 and float(got["psnr"]) == 31.25
    assert got["images"].dtype == np.float32 and got["images"].shape == (bench.DUMP_MAX_ELEMENTS,)
    assert np.array_equal(got["images"], np.load(tmp_path / "b" / "images.npy"))
    assert set(np.unique(got["images"]).tolist()) <= set(range(256))
    assert sum(p.stat().st_size for p in (tmp_path / "a").iterdir()) <= 64 << 20
