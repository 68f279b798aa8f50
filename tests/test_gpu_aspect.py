"""GPU: edits at the SDXL aspect-ratio buckets.

Kernels: the im2col form of the implicit-GEMM convolution (output widths that are neither a multiple nor a divisor of 128)
against fp32 F.conv2d on the same rounded inputs, for every convolution form the VAE, UNet and ControlNet use.
Pipeline: tiny same-topology edits at all nine buckets against the fp32 oracle, and the drop-in ``size`` argument."""
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from tests.util import rel_err

pytestmark = pytest.mark.gpu

BF = torch.bfloat16


def _ops():
    from fast_image_editing_with_generative_models_b200 import ops
    return ops


def _rand(shape, dev, seed, scale=1.0):
    g = torch.Generator("cpu").manual_seed(seed)
    return (torch.randn(shape, generator=g) * scale).to(dev)


def _conv_ref(x, w, b, stride=1, pad_mode=0):
    xc = x.float().permute(0, 3, 1, 2)
    if stride == 2 and pad_mode == 1:
        y = F.conv2d(F.pad(xc, (0, 1, 0, 1)), w.float(), b, stride=2)
    else:
        y = F.conv2d(xc, w.float(), b, stride=stride, padding=1)
    return y.permute(0, 2, 3, 1)


class _forced_im2col:
    """Forces the im2col form on shapes the rectangular box also tiles (test hook)."""

    def __enter__(self):
        from fast_image_editing_with_generative_models_b200 import _lib
        _lib.lib().fie_tune_conv_im2col(1)

    def __exit__(self, *a):
        from fast_image_editing_with_generative_models_b200 import _lib
        _lib.lib().fie_tune_conv_im2col(0)


# ------------------------------------------------------------------ kernels

@pytest.mark.parametrize("dtype", [torch.float16, BF])
@pytest.mark.parametrize("n,h,w,cin,cout,stride,pad_mode", [
    (2, 104, 152, 64, 320, 1, 0),       # UNet / ControlNet level 0 at 1216 x 832
    (2, 52, 76, 128, 640, 1, 0),        # level 1
    (2, 26, 38, 192, 128, 1, 0),        # level 2 (cin 192: odd K-block count, padded K block)
    (1, 12, 576, 128, 128, 1, 0),       # VAE widths at 1152 x 896
    (1, 12, 288, 256, 256, 1, 0),
    (1, 12, 144, 512, 96, 1, 0),
    (3, 26, 38, 64, 64, 1, 0),          # 988 pixels per image: tiles cross image boundaries
    (2, 104, 152, 320, 320, 2, 0),      # UNet Downsample2D 152 -> 76
    (2, 52, 76, 64, 96, 2, 0),          # 76 -> 38
    (1, 16, 1216, 128, 128, 2, 1),      # VAE encoder Downsample2D 1216 -> 608
    (1, 16, 304, 64, 64, 2, 1),         # 304 -> 152
])
def test_conv3x3_im2col(cuda_dev, n, h, w, cin, cout, stride, pad_mode, dtype):
    ops = _ops()
    from fast_image_editing_with_generative_models_b200.weights import pack_conv3x3
    x = _rand((n, h, w, cin), cuda_dev, 40).to(dtype)
    wt = (_rand((cout, cin, 3, 3), cuda_dev, 41) / math.sqrt(9 * cin)).to(dtype)
    bias = _rand((cout,), cuda_dev, 42)
    out = torch.empty((n, h // stride, w // stride, cout), dtype=torch.float16, device=cuda_dev)   # fp16 output: 2^-11 rounding
    ops.conv3x3(x, pack_conv3x3(wt.float(), dtype=dtype), stride=stride, pad_mode=pad_mode, col_bias=bias, out=out)
    ref = _conv_ref(x, wt, bias, stride, pad_mode)
    assert out.shape == ref.shape
    assert rel_err(out, ref) < 2e-3, rel_err(out, ref)


@pytest.mark.parametrize("dtype", [torch.float16, BF])
@pytest.mark.parametrize("n,h,w,cin,cout", [(2, 13, 72, 128, 128), (1, 8, 144, 256, 64), (2, 26, 38, 64, 96)])
def test_conv_up2x_im2col(cuda_dev, n, h, w, cin, cout, dtype):
    """Fused nearest-2x upsample + conv at input widths the box cannot tile (VAE decoder at 1152 x 896: 72 -> 144 -> 288)."""
    ops = _ops()
    from fast_image_editing_with_generative_models_b200.weights import pack_conv_up2x
    x = _rand((n, h, w, cin), cuda_dev, 70).to(dtype)
    wt = (_rand((cout, cin, 3, 3), cuda_dev, 71) / math.sqrt(9 * cin)).to(dtype)
    bias = _rand((cout,), cuda_dev, 72)
    out = ops.conv_up2x(x, pack_conv_up2x(wt.float(), dtype=dtype), col_bias=bias)
    xu = F.interpolate(x.float().permute(0, 3, 1, 2), scale_factor=2.0, mode="nearest").permute(0, 2, 3, 1)
    ref = _conv_ref(xu, wt, bias)
    # phase weights are fp32 sums of up to four taps rounded once to the operand type (as test_conv_up2x / the bf16 VAE tests)
    tol = 3e-3 if dtype == torch.float16 else 1.5e-2
    assert out.shape == ref.shape and rel_err(out, ref) < tol, rel_err(out, ref)


@pytest.mark.parametrize("out_dtype", [torch.float16, BF])
@pytest.mark.parametrize("n,h,w,cout,silu", [(1, 832, 1216, 128, False), (2, 40, 152, 96, True)])
def test_conv3x3_c8_image_input_im2col(cuda_dev, n, h, w, cout, silu, out_dtype):
    """conv_in on the zero-padded 8-channel image (overlapping 16-byte pixel view) at 1216 x 832."""
    ops = _ops()
    from fast_image_editing_with_generative_models_b200.weights import pack_conv3x3_c8
    img = torch.randint(0, 256, (n, h, w, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(53)).to(cuda_dev)
    xp = ops.preprocess_pad8(img, True)
    x = (2.0 * (img.float() / 255.0) - 1.0).half()
    wt = _rand((cout, 3, 3, 3), cuda_dev, 54) / 5
    bias = _rand((cout,), cuda_dev, 55)
    out = ops.conv3x3_c8(xp, pack_conv3x3_c8(wt), col_bias=bias, act=ops.ACT_SILU if silu else ops.ACT_NONE, out_dtype=out_dtype)
    ref = F.conv2d(x.permute(0, 3, 1, 2).float(), wt, bias, padding=1)
    ref = (F.silu(ref) if silu else ref).permute(0, 2, 3, 1)
    assert out.dtype == out_dtype
    assert rel_err(out, ref) < (1e-3 if out_dtype == torch.float16 else 4e-3), rel_err(out, ref)


@pytest.mark.parametrize("n,h,w,cout,res", [(2, 104, 152, 320, True), (3, 26, 38, 64, False), (1, 112, 144, 32, False)])
def test_conv3x3_c8_latent_input_im2col(cuda_dev, n, h, w, cout, res):
    """Latent conv_in (4 channels padded to 8) with the ControlNet's fused residual, at latent widths 152 / 38 / 144."""
    ops = _ops()
    from fast_image_editing_with_generative_models_b200.weights import pack_conv3x3_c8
    x = (_rand((n, h, w, 4), cuda_dev, 56) * 3).half()
    xp = ops.pad8(x)
    wt = _rand((cout, 4, 3, 3), cuda_dev, 57) / 6
    bias = _rand((cout,), cuda_dev, 58)
    r = _rand((n, h, w, cout), cuda_dev, 59).half() if res else None
    out = ops.conv3x3_c8(xp, pack_conv3x3_c8(wt), col_bias=bias, residual=r)
    ref = F.conv2d(x.permute(0, 3, 1, 2).float(), wt, bias, padding=1).permute(0, 2, 3, 1)
    if res:
        ref = ref + r.float()
    assert rel_err(out, ref) < 1e-3, rel_err(out, ref)


@pytest.mark.parametrize("dtype", [torch.float16, BF])
def test_conv_im2col_epilogues(cuda_dev, dtype):
    """Residual + SiLU, time-embedding row bias, and bf16 / fp32 outputs at width 152."""
    ops = _ops()
    from fast_image_editing_with_generative_models_b200.weights import pack_conv3x3
    n, h, w, cin, cout = 2, 20, 152, 128, 192
    x = _rand((n, h, w, cin), cuda_dev, 80).to(dtype)
    wt = (_rand((cout, cin, 3, 3), cuda_dev, 81) / math.sqrt(9 * cin)).to(dtype)
    wp = pack_conv3x3(wt.float(), dtype=dtype)
    bias = _rand((cout,), cuda_dev, 82)
    temb = _rand((n, cout), cuda_dev, 83)
    base = _conv_ref(x, wt, None)
    out_dtypes = [torch.float16] if dtype == torch.float16 else [torch.float16, BF]
    for od in out_dtypes:
        res = _rand((n, h, w, cout), cuda_dev, 84).to(od)
        out = torch.empty((n, h, w, cout), dtype=od, device=cuda_dev)
        ops.conv3x3(x, wp, col_bias=bias, residual=res, out=out)
        tol = 2e-3 if od == torch.float16 else 4e-3
        assert rel_err(out, base + bias + res.float()) < tol, (od, rel_err(out, base + bias + res.float()))
        ops.conv3x3(x, wp, col_bias=bias, act=ops.ACT_SILU, out=out)
        assert rel_err(out, F.silu(base + bias)) < tol
        ops.conv3x3(x, wp, row_bias=temb, rows_per_group=h * w, out=out)
        assert rel_err(out, base + temb[:, None, None, :]) < tol
    out32 = torch.empty((n, h, w, cout), dtype=torch.float32, device=cuda_dev)
    if dtype == BF:
        ops.conv3x3(x, wp, col_bias=bias, out=out32)
        assert rel_err(out32, base + bias) < 1e-4


@pytest.mark.parametrize("n,h,w,cin,cout,groups", [(2, 16, 152, 128, 512, 32), (2, 32, 144, 64, 256, 32), (1, 64, 76, 128, 128, 32),
                                                   (2, 104, 152, 128, 512, 32), (3, 8, 76, 64, 512, 32)])
def test_conv_im2col_groupnorm_statistics(cuda_dev, n, h, w, cin, cout, groups):
    """Producer-side GroupNorm statistics (rows per image a multiple of 32) on the im2col form equal a float64 reduction.
    2 x 104 x 152 (the latent level of 1216 x 832: 15808 rows per image) and 3 x 8 x 76 (608) have 128-row tiles that straddle two images
    and a last tile that ends past M."""
    ops = _ops()
    from fast_image_editing_with_generative_models_b200.weights import pack_conv3x3
    monkey_cpg, ops.GN_FUSE_CPG = ops.GN_FUSE_CPG, (4, 8, 16, 32)
    try:
        x = _rand((n, h, w, cin), cuda_dev, 90).half()
        wt = (_rand((cout, cin, 3, 3), cuda_dev, 91) / math.sqrt(9 * cin)).half()
        bias = _rand((cout,), cuda_dev, 92)
        res = _rand((n, h, w, cout), cuda_dev, 93).half()
        wp = pack_conv3x3(wt)
        y = ops.conv3x3(x, wp, col_bias=bias, residual=res, gn_groups=groups)
        assert hasattr(y, "_gn_stats")
        st = y._gn_stats[0].clone()
        y2 = ops.conv3x3(x, wp, col_bias=bias, residual=res)
        assert torch.equal(y, y2)
        yg = y.double().view(n, h * w, groups, cout // groups)
        s_ref, q_ref = yg.sum(dim=(1, 3)), (yg * yg).sum(dim=(1, 3))
        s_got, q_got = st[..., 0].double() / 2 ** 20, st[..., 1].double() / 2 ** 20
        assert float(((s_got - s_ref).abs() / (q_ref.sqrt() + 1)).max()) < 5e-2 and float(((q_got - q_ref).abs() / q_ref).max()) < 2e-3
        gamma = _rand((cout,), cuda_dev, 94) * 0.1 + 1
        beta = _rand((cout,), cuda_dev, 95) * 0.1
        out = ops.groupnorm(y, gamma, beta, 1e-6, True, groups)
        ref = F.silu(F.group_norm(y.float().permute(0, 3, 1, 2), groups, gamma, beta, 1e-6)).permute(0, 2, 3, 1)
        assert float((out.float() - ref).abs().max()) < 8e-3
    finally:
        ops.GN_FUSE_CPG = monkey_cpg


@pytest.mark.parametrize("n,h,w,cin,cout,stride,pad_mode", [
    (2, 32, 32, 128, 320, 1, 0), (2, 8, 8, 256, 256, 1, 0), (2, 64, 64, 320, 320, 2, 0), (1, 64, 64, 128, 128, 2, 1), (1, 16, 256, 64, 96, 1, 0)])
def test_im2col_forced_on_box_shapes(cuda_dev, n, h, w, cin, cout, stride, pad_mode):
    """The forced im2col form on shapes the box path tiles: the same pixels and K order as the per-tap box form (bit-identical),
    and within accumulation order of the halo form (1 x 16 x 256)."""
    ops = _ops()
    from fast_image_editing_with_generative_models_b200.weights import pack_conv3x3
    x = _rand((n, h, w, cin), cuda_dev, 60).half()
    wt = (_rand((cout, cin, 3, 3), cuda_dev, 61) / math.sqrt(9 * cin)).half()
    bias = _rand((cout,), cuda_dev, 62)
    wp = pack_conv3x3(wt)
    out_box = ops.conv3x3(x, wp, stride=stride, pad_mode=pad_mode, col_bias=bias)
    with _forced_im2col():
        out_i2c = ops.conv3x3(x, wp, stride=stride, pad_mode=pad_mode, col_bias=bias)
    ref = _conv_ref(x, wt, bias, stride, pad_mode)
    assert rel_err(out_i2c, ref) < 2e-3, rel_err(out_i2c, ref)
    if w // stride < 128:
        assert torch.equal(out_i2c, out_box)
    else:
        # only the fp32 accumulation order differs: at most about one fp16 step of the largest output apart
        assert float((out_i2c.float() - out_box.float()).abs().max()) <= 2e-3 * float(ref.abs().max())


def test_im2col_forced_up2x_and_c8(cuda_dev):
    ops = _ops()
    from fast_image_editing_with_generative_models_b200.weights import pack_conv3x3_c8, pack_conv_up2x
    x = _rand((2, 16, 32, 64), cuda_dev, 63).half()
    w4 = pack_conv_up2x((_rand((64, 64, 3, 3), cuda_dev, 64) / 24).half())
    xp = ops.pad8((_rand((2, 32, 64, 4), cuda_dev, 65) * 3).half())
    w8 = pack_conv3x3_c8(_rand((96, 4, 3, 3), cuda_dev, 66) / 6)
    up_box, c8_box = ops.conv_up2x(x, w4), ops.conv3x3_c8(xp, w8)
    with _forced_im2col():
        up_i2c, c8_i2c = ops.conv_up2x(x, w4), ops.conv3x3_c8(xp, w8)
    assert torch.equal(up_i2c, up_box) and torch.equal(c8_i2c, c8_box)


def test_im2col_conv_writes_only_its_output(cuda_dev):
    """Outputs carved out of one sentinel-filled arena: the last partial tile (rows past M) must not be stored."""
    ops = _ops()
    from fast_image_editing_with_generative_models_b200.weights import pack_conv3x3, pack_conv3x3_c8, pack_conv_up2x
    n, h, w_, cin, cout = 3, 26, 38, 64, 96           # M = 2964: not a multiple of 128 or 256
    x = _rand((n, h, w_, cin), cuda_dev, 77).half()
    wt = (_rand((cout, cin, 3, 3), cuda_dev, 78) / math.sqrt(9 * cin)).half()

    def arena(shape):
        k = int(np.prod(shape))
        buf = torch.full((64 + k + 64,), 1234.0, dtype=torch.float16, device=cuda_dev)
        return buf, buf[64:64 + k].view(*shape)

    def guards_ok(buf):
        return bool((buf[:64] == 1234.0).all()) and bool((buf[-64:] == 1234.0).all())

    buf, out = arena((n, h, w_, cout))
    ops.conv3x3(x, pack_conv3x3(wt), out=out)
    buf2, out2 = arena((n, 2 * h, 2 * w_, cout))
    ops.conv_up2x(x, pack_conv_up2x(wt), out=out2)
    buf3, out3 = arena((n, h // 2, w_ // 2, cout))
    ops.conv3x3(x, pack_conv3x3(wt), stride=2, out=out3)
    torch.cuda.synchronize()
    assert guards_ok(buf) and guards_ok(buf2) and guards_ok(buf3)
    assert rel_err(out, _conv_ref(x, wt, None)) < 2e-3
    assert rel_err(out3, _conv_ref(x, wt, None, 2, 0)) < 2e-3


# ------------------------------------------------------------------ pipeline at the buckets

BUCKETS = ((1024, 1024), (1152, 896), (896, 1152), (1216, 832), (832, 1216), (1344, 768), (768, 1344), (1536, 640), (640, 1536))


@pytest.fixture(scope="module")
def tiny_engine(cuda_dev):
    from fast_image_editing_with_generative_models_b200 import synthetic as S
    from fast_image_editing_with_generative_models_b200.pipeline import EditEngine
    from oracle import diffusion_oracle as O
    ucfg, ccfg, vcfg = O.tiny_unet_config(), O.tiny_controlnet_config(), O.tiny_vae_config()
    up, cp, vp = S.make_unet_params(ucfg), S.make_controlnet_params(ccfg), S.make_vae_params(vcfg)
    lp = S.make_lora_params(up, rank=8)
    eng = EditEngine(up, ucfg, cp, ccfg, vp, vcfg, cuda_dev, lp, 1.0)
    f32 = lambda p: O.to_dtype(p, torch.float32, cuda_dev)
    return eng, O.EditModels(ucfg, f32(up), ccfg, f32(cp), vcfg, f32(vp), f32(lp), 1.0)


def test_bucket_list_matches_the_editor():
    from fast_image_editing_with_generative_models_b200.editor import FastEditor
    assert tuple(FastEditor.SDXL_BUCKETS) == BUCKETS


@pytest.mark.parametrize("width,height", BUCKETS)
def test_edit_tiny_at_bucket(cuda_dev, tiny_engine, width, height):
    """Same-topology tiny models at every bucket against the fp32 oracle: Canny bit-exact, final latents <= 2e-2, SSIM >= 0.99."""
    from fast_image_editing_with_generative_models_b200.synthetic import synthetic_image, synthetic_noises
    from oracle import c_oracle
    from oracle import diffusion_oracle as O
    eng, m = tiny_engine
    ucfg = m.unet_cfg
    imgs = np.stack([synthetic_image(5, height, width)])
    g = torch.Generator().manual_seed(9)
    pe = torch.randn((2, 77, ucfg.cross_attention_dim), generator=g).half()
    pl = torch.randn((2, 64), generator=g).half()
    noises = synthetic_noises(0, 1, height // 8, width // 8)
    d_img = torch.from_numpy(imgs).to(cuda_dev)
    out = eng.edit_batch(d_img, pe, pl, noises, strength=0.5, return_latents=True)
    assert out.images.shape == (1, height, width, 3) and out.latents.shape == (1, height // 8, width // 8, 4)
    edges_ref = c_oracle.canny_u8(imgs, 100, 200, replicate3=True)
    assert np.array_equal(out.edges.cpu().numpy(), edges_ref)
    with torch.no_grad():
        ref = O.edit_pipeline(m, d_img, torch.from_numpy(edges_ref).to(cuda_dev), pe.float().to(cuda_dev), pl.float().to(cuda_dev), noises,
                              strength=0.5, dtype=torch.float32, return_all=True)
    lat_err = float((out.latents.permute(0, 3, 1, 2).float() - ref["latents"]).abs().max())
    s = O.ssim(out.images.permute(0, 3, 1, 2).float() / 255.0, ref["image_u8"].permute(0, 3, 1, 2).float() / 255.0)
    print(f"\n[tiny {width}x{height}] latents max-abs {lat_err:.4g}; SSIM {s:.5f}")
    assert lat_err <= 2e-2 and s >= 0.99


@pytest.mark.parametrize("width,height", [(1216, 832), (832, 1216)])
def test_full_size_ssd1b_at_bucket(cuda_dev, width, height):
    """SSD-1B + ControlNet-small, one image, strength 0.5, against the fp32 oracle; torch-fp16's own error is reported as the floor."""
    from fast_image_editing_with_generative_models_b200 import model_zoo
    from fast_image_editing_with_generative_models_b200 import synthetic as S
    from oracle import c_oracle
    from oracle import diffusion_oracle as O
    from tests.test_gpu_fullsize import _compare, _oracle, _state
    state = _state("ssd-1b")
    ucfg = state["unet_cfg"]
    imgs = np.stack([S.synthetic_image(0, height, width)])
    pe, pl = S.synthetic_prompt(0, ucfg.cross_attention_dim, ucfg.projection_class_embeddings_input_dim - 6 * ucfg.addition_time_embed_dim)
    noises = S.synthetic_noises(0, 1, height // 8, width // 8)
    d_img = torch.from_numpy(imgs).to(cuda_dev)
    eng = model_zoo.build_engine(state, cuda_dev)
    out = eng.edit_batch(d_img, pe, pl, noises, strength=0.5, return_latents=True)
    edges_ref = c_oracle.canny_u8(imgs, 100, 200, replicate3=True)
    assert np.array_equal(out.edges.cpu().numpy(), edges_ref), "Canny control image not bit-exact"
    latents, images = out.latents.clone(), out.images.clone()
    del eng, out
    torch.cuda.empty_cache()
    ref = _oracle(state, cuda_dev, torch.float32, d_img, edges_ref, pe, pl, noises, 0.5)
    lat_err, s, _ = _compare(f"ssd-1b {width}x{height}", latents, images, ref)
    ref16 = _oracle(state, cuda_dev, torch.float16, d_img, edges_ref, pe, pl, noises, 0.5)
    floor = float((ref16["latents"].float() - ref["latents"]).abs().max())
    print(f"[ssd-1b {width}x{height}] torch-fp16 oracle vs fp32 oracle: latents max-abs {floor:.4g}")
    assert lat_err <= max(2e-2, floor), (lat_err, floor)
    assert s >= 0.99, s


def test_full_size_sdxl_b8_graph_replay_at_1152x896(cuda_dev):
    """SDXL, 8 images of 1152 x 896: the CUDA-graph replay equals the eager launch sequence bit for bit, and so does a second replay."""
    from fast_image_editing_with_generative_models_b200 import model_zoo
    from fast_image_editing_with_generative_models_b200 import synthetic as S
    from tests.test_gpu_fullsize import _state
    state = _state("sdxl")
    ucfg = state["unet_cfg"]
    W, H, B = 1152, 896, 8
    imgs = np.stack([S.synthetic_image(s, H, W) for s in range(B)])
    pe, pl = S.synthetic_prompt(0, ucfg.cross_attention_dim, ucfg.projection_class_embeddings_input_dim - 6 * ucfg.addition_time_embed_dim)
    noises = S.synthetic_noises(0, B, H // 8, W // 8)
    d_img = torch.from_numpy(imgs).to(cuda_dev)
    eng = model_zoo.build_engine(state, cuda_dev)
    eager = eng.edit_batch(d_img, pe, pl, noises, strength=0.5, return_latents=True, use_graph=False)
    e_lat, e_img = eager.latents.clone(), eager.images.clone()
    assert e_img.shape == (B, H, W, 3) and bool(torch.isfinite(e_lat.float()).all())
    g1 = eng.edit_batch(d_img, pe, pl, noises, strength=0.5, return_latents=True, use_graph=True)
    g1_lat, g1_img = g1.latents.clone(), g1.images.clone()
    g2 = eng.edit_batch(d_img, pe, pl, noises, strength=0.5, return_latents=True, use_graph=True)
    assert torch.equal(g1_lat, e_lat) and torch.equal(g1_img, e_img), "graph replay differs from eager"
    assert torch.equal(g2.latents, g1_lat) and torch.equal(g2.images, g1_img), "two replays differ"


# ------------------------------------------------------------------ drop-in: FastEditor(size=...)

@pytest.fixture(scope="module")
def editor(cuda_dev):
    from src.pipeline import FastEditor
    return FastEditor(model_name="ssd-1b", device="cuda", enable_cpu_offload=False, tiny=True, verbose=False)


def _image(seed, size):
    from PIL import Image
    from fast_image_editing_with_generative_models_b200.synthetic import synthetic_image
    return Image.fromarray(synthetic_image(seed, 1024, 1024)).resize(size)


def test_edit_auto_size_is_the_pillow_resized_edit(editor):
    from PIL import Image
    img = _image(1, (640, 480))
    a = editor.edit(img, "a rusty bicycle", seed=42, size="auto")
    assert a.size == (1152, 896) and a.mode == "RGB"
    b = editor.edit(img.resize((1152, 896), Image.LANCZOS), "a rusty bicycle", seed=42, size="auto")
    assert np.array_equal(np.array(a), np.array(b))
    c = editor.edit(img, "a rusty bicycle", seed=42, size=(1152, 896))
    assert np.array_equal(np.array(a), np.array(c))
    d = editor.edit(img, "a rusty bicycle", seed=42, size=(832, 1216))
    assert d.size == (832, 1216)
    with pytest.raises(ValueError):
        editor.edit(img, "a rusty bicycle", seed=42, size=(1000, 1000))


def test_size_none_is_the_default(editor):
    img = _image(2, (640, 480))
    a = editor.edit(img, "a rusty bicycle", seed=3)
    b = editor.edit(img, "a rusty bicycle", seed=3, size=None)
    assert a.size == (1024, 1024) and a.tobytes() == b.tobytes()
    m1 = editor.edit_many([img, _image(3, (1024, 1024))], "x", seed=3, micro_batch=2)
    m2 = editor.edit_many([img, _image(3, (1024, 1024))], "x", seed=3, micro_batch=2, size=None)
    assert all(p.tobytes() == q.tobytes() for p, q in zip(m1, m2))


def test_edit_many_auto_groups_by_bucket(editor):
    import io
    imgs = [_image(10, (640, 480)), _image(11, (480, 640)), _image(12, (700, 700)), _image(13, (800, 600)), _image(14, (1152, 896)),
            _image(15, (1920, 1080))]
    prompts = [f"prompt {i}" for i in range(len(imgs))]
    seeds = [1, 2, 3, 4, 5, 6]
    many = editor.edit_many(imgs, prompts, seeds=seeds, micro_batch=2, size="auto")
    want = [(1152, 896), (896, 1152), (1024, 1024), (1152, 896), (1152, 896), (1344, 768)]
    assert [m.size for m in many] == want
    for bucket in set(want):
        sub = [i for i, w in enumerate(want) if w == bucket]
        alone = editor.edit_many([imgs[i] for i in sub], [prompts[i] for i in sub], seeds=[seeds[i] for i in sub], micro_batch=2, size="auto")
        for i, a in zip(sub, alone):
            assert np.array_equal(np.array(many[i]), np.array(a)), (bucket, i)
    jpgs = editor.edit_many(imgs, prompts, seeds=seeds, micro_batch=2, size="auto", output="jpeg")
    for p, j in zip(many, jpgs):
        b = io.BytesIO()
        p.save(b, "JPEG")
        assert b.getvalue() == j
    t = editor.warm_up(2, size=(1216, 832))
    assert t > 0
    # clear_memory keeps only the staging buffers of the most recently used size
    assert len([k for k in editor._pinned if isinstance(k[0], int)]) > 1
    editor.clear_memory()
    assert [k for k in editor._pinned if isinstance(k[0], int)] == [(2, 832, 1216)]
