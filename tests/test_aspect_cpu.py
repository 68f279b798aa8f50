"""CPU: the ``size`` argument of FastEditor (bucket choice, validation), the CLIs' ``--size``, the per-image noise shapes and the
SDXL micro-conditioning at non-square sizes."""
import pytest
import torch

from fast_image_editing_with_generative_models_b200.editor import FastEditor, resolve_size


@pytest.mark.parametrize("image_size,bucket", [((640, 480), (1152, 896)), ((4000, 3000), (1152, 896)), ((480, 640), (896, 1152)),
                                               ((900, 1600), (768, 1344)), ((1080, 1920), (768, 1344)), ((1920, 1080), (1344, 768)),
                                               ((512, 512), (1024, 1024)), ((3000, 1000), (1536, 640)), ((1000, 3000), (640, 1536)),
                                               ((1216, 832), (1216, 832)), ((832, 1216), (832, 1216))])
def test_auto_picks_the_closest_bucket_in_log_aspect(image_size, bucket):
    assert resolve_size("auto", image_size) == bucket


def test_auto_tie_goes_to_the_earlier_bucket(monkeypatch):
    # a square input is exactly as far (in log aspect ratio) from a bucket as from its transpose
    monkeypatch.setattr(FastEditor, "SDXL_BUCKETS", ((1152, 896), (896, 1152)))
    assert resolve_size("auto", (700, 700)) == (1152, 896)
    monkeypatch.setattr(FastEditor, "SDXL_BUCKETS", ((896, 1152), (1152, 896)))
    assert resolve_size("auto", (700, 700)) == (896, 1152)


def test_buckets_are_valid_sizes():
    assert FastEditor.SDXL_BUCKETS[0] == (1024, 1024) and len(FastEditor.SDXL_BUCKETS) == 9
    for b in FastEditor.SDXL_BUCKETS:
        assert resolve_size(b, (1, 1)) == b


def test_explicit_and_default_sizes():
    assert resolve_size(None, (640, 480)) == (1024, 1024)
    assert resolve_size((1152, 896), (10, 10)) == (1152, 896)
    assert resolve_size((256, 2048), (10, 10)) == (256, 2048)
    assert resolve_size([768, 768], (10, 10)) == (768, 768)


@pytest.mark.parametrize("size", [(1000, 1000), (1024, 1000), (1152, 900), (192, 1024), (1024, 192), (2112, 256), (256, 2112),
                                  (1088, 1024), (2048, 1024), (1536, 768), "square", "1024x1024", (1024,), (1024, 1024, 3), 1024,
                                  (1024.0, 1024.0), (True, 1024)])
def test_invalid_sizes_raise_value_error(size):
    with pytest.raises(ValueError):
        resolve_size(size, (640, 480))


def test_cli_size_flag():
    import run_batch
    import run_single_image
    pb = run_batch.build_parser()
    ps = run_single_image.build_parser()
    base = ["--image", "x.png", "--prompt", "p"]
    assert pb.parse_args([]).size == (1024, 1024) and ps.parse_args(base).size == (1024, 1024)
    assert pb.parse_args(["--size", "1216x832"]).size == (1216, 832) and ps.parse_args(base + ["--size", "832x1216"]).size == (832, 1216)
    assert pb.parse_args(["--size", "auto"]).size == "auto" and ps.parse_args(base + ["--size", "auto"]).size == "auto"
    for bad in ("1000x1000", "2048x1024", "big", "1024", "1024x1024x3"):
        with pytest.raises(SystemExit):
            pb.parse_args(["--size", bad])
        with pytest.raises(SystemExit):
            ps.parse_args(base + ["--size", bad])


@pytest.mark.parametrize("size", [(1024, 1024), (1216, 832), (640, 1536)])
def test_noise_shapes_follow_the_size(size):
    ed = FastEditor.__new__(FastEditor)            # no engine: only the host-side RNG draw
    ed._dev = torch.device("cpu")
    w, h = size
    noises = ed._draw_noises(7, 2, size)
    assert len(noises) == 3 and all(n.shape == (1, 4, h // 8, w // 8) and n.dtype == torch.float16 for n in noises)
    # the reference's RNG order: one generator per image, draws in sequence
    g = torch.Generator().manual_seed(7)
    ref = [torch.randn((1, 4, h // 8, w // 8), generator=g, dtype=torch.float16) for _ in range(3)]
    assert all(torch.equal(a, b) for a, b in zip(noises, ref))
    assert ed._draw_noises(7, 2)[0].shape == (1, 4, 128, 128)


@pytest.mark.parametrize("height,width", [(1024, 1024), (832, 1216), (1216, 832), (640, 1536)])
def test_time_ids_are_height_width_as_diffusers(height, width):
    from fast_image_editing_with_generative_models_b200.pipeline import sdxl_time_ids
    # diffusers StableDiffusionXL*Pipeline._get_add_time_ids: list(original_size + crops_coords_top_left + target_size), where
    # original_size = target_size = (height, width) and crops_coords_top_left = (0, 0)
    original_size, crop, target_size = (height, width), (0, 0), (height, width)
    assert sdxl_time_ids(height, width) == [float(v) for v in original_size + crop + target_size]


def test_gn_stats_rows_must_divide_the_rows():
    """Producer-side GroupNorm statistics key each warp's rows to an image: the image count must be exact (M = images x rows per
    image), else rows of a partial last image would land past the statistics buffer.  Rejected before any CUDA work."""
    import ctypes
    from fast_image_editing_with_generative_models_b200 import _lib
    L = _lib.lib()
    buf = (ctypes.c_ubyte * 256)()
    p = ctypes.addressof(buf)
    ep = _lib.Epilogue(scale=1.0, gn_stats=p, gn_groups=2, gn_rows_per_image=64)
    # M = 96 rows is not a whole number of 64-row images
    assert L.fie_gemm_f16(p, 64, None, 0, 0, p, p, 64, 96, 64, 64, ctypes.byref(ep), None) != 0
    assert b"divides the rows" in L.fie_last_error()


def test_run_batch_groups_auto_micro_batches_by_bucket(tmp_path):
    from PIL import Image
    import run_batch
    sizes = [(640, 480), (480, 640), (800, 600), (512, 512), (1600, 1200), (600, 800), (1024, 1024), (640, 480)]
    work = []
    for i, sz in enumerate(sizes):
        path = tmp_path / f"{i}.png"
        Image.new("RGB", sz).save(path)
        work.append((str(i), {}, str(path), str(tmp_path / f"o{i}.png")))
    work.append(("missing", {}, str(tmp_path / "missing.png"), str(tmp_path / "om.png")))
    groups = run_batch.micro_batches(work, 2, "auto")
    assert [[it[0] for it in g] for g in groups] == [["0", "2"], ["4", "7"], ["1", "5"], ["3", "6"], ["missing"]]
    assert run_batch.micro_batches(work, 4, (1024, 1024)) == [work[0:4], work[4:8], work[8:]]
