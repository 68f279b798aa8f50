"""GPU: the bf16 VAE (DESIGN.md 3.11).  Kernel parity of every bf16 entry point against fp32 torch on the same bf16-rounded inputs,
device packing == host packing, range-safe deterministic GroupNorm, VAE parity against the fp32 oracle (tiny and the SDXL VAE topology at
1024^2), a synthetic VAE whose decoder leaves the fp16 range, and the end-to-end edit with ``vae_dtype=torch.bfloat16``."""
import ctypes
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import c_oracle
from oracle import diffusion_oracle as O

pytestmark = pytest.mark.gpu

BF = torch.bfloat16


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    return torch.device("cuda:0")


def _g(seed):
    return torch.Generator().manual_seed(seed)


def _randn(shape, seed, dev, scale=1.0):
    return (torch.randn(shape, generator=_g(seed)) * scale).to(dev)


def _close(got, ref, rel, what):
    err = float((got.float() - ref.float()).abs().max())
    lim = rel * max(1.0, float(ref.abs().max()))
    print(f"{what}: max-abs {err:.4g} (limit {lim:.4g})")
    assert math.isfinite(err) and err <= lim, (what, err, lim)


# ---------------------------------------------------------------- GEMM


@pytest.mark.parametrize("cg", [1, 2])
@pytest.mark.parametrize("out_dtype", [BF, torch.float16, torch.float32])
def test_gemm_bf16_forms(dev, cg, out_dtype):
    from fast_image_editing_with_generative_models_b200 import _lib, ops
    L = _lib.lib()
    M = 128 if cg == 1 else 1000
    N, K = 192, 320
    a = _randn((M, K), 1, dev).to(BF)
    w = _randn((N, K), 2, dev, 0.05).to(BF)
    bias = _randn((N,), 3, dev)
    L.fie_tune_gemm(cg, 0)
    try:
        ref = a.float() @ w.float().t()
        _close(ops.gemm(a, w, out_dtype=out_dtype), ref, 8e-3, f"gemm cg{cg} -> {out_dtype}")
        if out_dtype != torch.float32:
            res = _randn((M, N), 4, dev).to(out_dtype)
            got = ops.gemm(a, w, col_bias=bias, act=ops.ACT_SILU, scale=0.5, residual=res, out_dtype=out_dtype)
            _close(got, F.silu(ref + bias) * 0.5 + res.float(), 8e-3, f"gemm cg{cg} bias+silu+scale+residual -> {out_dtype}")
            mb = _randn((M,), 5, dev)                                      # V^T projection: per-row bias
            _close(ops.gemm(a, w, m_bias=mb, out_dtype=out_dtype), ref + mb[:, None], 8e-3, f"gemm cg{cg} m_bias -> {out_dtype}")
            rs = torch.rand((M,), generator=_g(6)).to(dev) + 0.5           # P V: 1 / rowsum
            _close(ops.gemm(a, w, row_scale=rs, out_dtype=out_dtype), ref * rs[:, None], 8e-3, f"gemm cg{cg} row_scale -> {out_dtype}")
            # slow epilogue path: N not a multiple of 32 (partial chunks), residual read element-wise in the output type
            w2 = w[:72].contiguous()
            res2 = _randn((M, 72), 7, dev).to(out_dtype)
            _close(ops.gemm(a, w2, residual=res2, out_dtype=out_dtype), a.float() @ w2.float().t() + res2.float(), 8e-3,
                   f"gemm cg{cg} N=72 slow path -> {out_dtype}")
    finally:
        L.fie_tune_gemm(0, 0)


def test_gemm_bf16_rejects_gn_stats_without_cuda_work(dev):
    from fast_image_editing_with_generative_models_b200 import _lib, ops
    L = _lib.lib()
    a = torch.zeros((128, 64), dtype=BF, device=dev)
    w = torch.zeros((64, 64), dtype=BF, device=dev)
    out = torch.empty((128, 64), dtype=BF, device=dev)
    st = torch.zeros((1, 2, 2), dtype=torch.int64, device=dev)
    ep = ops._epilogue(gn=(st, 2, 128))
    rc = L.fie_gemm_bf16(a.data_ptr(), 64, None, 0, 0, w.data_ptr(), out.data_ptr(), 64, 128, 64, 64, ctypes.byref(ep), _lib.DT_BF16, None)
    assert rc == -1 and b"gn_stats" in L.fie_last_error()


# ---------------------------------------------------------------- convolutions


def _conv_ref(x, w, b, stride=1, pad_mode=0):
    xc = x.float().permute(0, 3, 1, 2)
    if stride == 2 and pad_mode == 1:
        xc = F.pad(xc, (0, 1, 0, 1))
        y = F.conv2d(xc, w.float(), b, stride=2)
    else:
        y = F.conv2d(xc, w.float(), b, stride=stride, padding=1)
    return y.permute(0, 2, 3, 1)


@pytest.mark.parametrize("halo", [1, 0])
def test_conv3x3_bf16_halo_and_per_tap(dev, halo):
    from fast_image_editing_with_generative_models_b200 import _lib, ops
    from fast_image_editing_with_generative_models_b200.weights import pack_conv3x3
    x = _randn((2, 128, 16, 128), 10, dev).to(BF).permute(0, 2, 3, 1).contiguous()         # NHWC [2, 16, 128, 128]
    w = _randn((96, 128, 3, 3), 11, dev, 0.03).to(BF).float()
    b = _randn((96,), 12, dev)
    res = _randn((2, 16, 128, 96), 13, dev).to(BF)
    _lib.lib().fie_tune_conv_halo(halo, 0)
    try:
        got = ops.conv3x3(x, pack_conv3x3(w, dtype=BF), col_bias=b, residual=res)
    finally:
        _lib.lib().fie_tune_conv_halo(1, 0)
    assert got.dtype == BF
    _close(got, _conv_ref(x, w, b) + res.float(), 8e-3, f"conv3x3 bf16 halo={halo}")
    out16 = torch.empty((2, 16, 128, 96), dtype=torch.float16, device=dev)     # fp16 output of bf16 operands (decoder conv_out)
    ops.conv3x3(x, pack_conv3x3(w, dtype=BF), col_bias=b, out=out16)
    _close(out16, _conv_ref(x, w, b), 8e-3, "conv3x3 bf16 -> fp16")


def test_conv3x3_bf16_stride2_pad_mode1_and_up2x(dev):
    from fast_image_editing_with_generative_models_b200 import ops
    from fast_image_editing_with_generative_models_b200.weights import pack_conv3x3, pack_conv_up2x
    x = _randn((2, 64, 32, 32), 20, dev).to(BF).permute(0, 2, 3, 1).contiguous()
    w = _randn((64, 64, 3, 3), 21, dev, 0.05).to(BF).float()
    b = _randn((64,), 22, dev)
    got = ops.conv3x3(x, pack_conv3x3(w, dtype=BF), stride=2, pad_mode=1, col_bias=b)
    _close(got, _conv_ref(x, w, b, 2, 1), 8e-3, "conv3x3 bf16 stride 2 pad_mode 1")
    up = ops.conv_up2x(x, pack_conv_up2x(w, dtype=BF), col_bias=b)
    xu = F.interpolate(x.float().permute(0, 3, 1, 2), scale_factor=2.0, mode="nearest").permute(0, 2, 3, 1)
    # the phase weights sum up to three taps of w before the bf16 rounding: compare against the fp32 conv of the fp32 sums' rounding budget
    _close(up, _conv_ref(xu, w, b), 1.5e-2, "conv_up2x bf16")


def test_conv3x3_c8_bf16_output(dev):
    from fast_image_editing_with_generative_models_b200 import ops
    from fast_image_editing_with_generative_models_b200.synthetic import synthetic_image
    from fast_image_editing_with_generative_models_b200.weights import pack_conv3x3_c8
    img = torch.from_numpy(np.stack([synthetic_image(s, 128, 128) for s in range(2)])).to(dev)
    xp = ops.preprocess_pad8(img, True)
    w = _randn((128, 3, 3, 3), 30, dev, 0.2)
    b = _randn((128,), 31, dev)
    got = ops.conv3x3_c8(xp, pack_conv3x3_c8(w), col_bias=b, out_dtype=BF)
    assert got.dtype == BF
    ref = F.conv2d(O.preprocess_image(img, torch.float32), w, b, padding=1).permute(0, 2, 3, 1)
    _close(got, ref, 8e-3, "conv3x3_c8 -> bf16")


def test_device_packing_equals_host_packing(dev):
    from fast_image_editing_with_generative_models_b200.weights import cast_f16, pack_conv3x3, pack_conv_up2x
    w = torch.randn((40, 24, 3, 3), generator=_g(40))
    for pad in ((None, None), (64, 32)):
        assert torch.equal(pack_conv3x3(w.to(dev), *pad, dtype=BF).cpu(), pack_conv3x3(w, *pad, dtype=BF))
    assert torch.equal(pack_conv_up2x(w.to(dev), dtype=BF).cpu(), pack_conv_up2x(w, dtype=BF))
    lin = torch.randn((48, 40), generator=_g(41))
    assert torch.equal(cast_f16(lin.to(dev), BF).cpu(), cast_f16(lin, BF))


# ---------------------------------------------------------------- GroupNorm


@pytest.mark.parametrize("n,hw,c,groups,silu,scale,offset", [
    (2, 1024, 128, 32, True, 1.0, 0.0),            # slab path (one CTA per (image, group))
    (2, 4096, 512, 32, False, 1.0, 0.5),           # slab path, 16 channels per group
    (2, 65536, 128, 32, True, 3.0, -1.0),          # two-kernel path (chunk partials)
    (1, 16384, 512, 32, True, 1.0, 0.0),           # two-kernel path, 16 channels per group
    (2, 65536, 128, 32, False, 1e6 / 300.0, 1e6),  # |x| ~ 1e6 with mean = 300 sigma: the int64 fixed point would overflow
    (1, 16384, 256, 32, True, 1e3, -3e5),
])
def test_groupnorm_bf16(dev, n, hw, c, groups, silu, scale, offset):
    from fast_image_editing_with_generative_models_b200 import ops
    x = (_randn((n, hw, c), 50 + c, dev, scale) + offset).to(BF)
    gamma = _randn((c,), 51, dev) * 0.5 + 1.0
    beta = _randn((c,), 52, dev) * 0.1
    got = ops.groupnorm(x, gamma, beta, 1e-6, silu, groups)
    again = ops.groupnorm(x, gamma, beta, 1e-6, silu, groups)
    assert torch.equal(got, again), "bf16 GroupNorm is not bit-reproducible"
    ref = F.group_norm(x.double().permute(0, 2, 1), groups, gamma.double(), beta.double(), 1e-6).permute(0, 2, 1)
    if silu:
        ref = F.silu(ref)
    assert torch.isfinite(got.float()).all()
    err = (got.double() - ref).abs()
    lim = ref.abs() * 2.0 ** -8 + 2e-3                  # bf16 output rounding (half an ulp is 2^-9 relative) plus fp32 arithmetic
    print(f"groupnorm bf16 [{n},{hw},{c}] x~{offset:g}+-{scale:g}: max-abs {float(err.max()):.4g}")
    assert bool((err <= lim).all()), float((err - lim).max())


def test_groupnorm_bf16_concatenated_source(dev):
    from fast_image_editing_with_generative_models_b200 import ops
    x0 = _randn((2, 65536, 64), 60, dev).to(BF)
    x1 = _randn((2, 65536, 64), 61, dev, 2.0).to(BF)
    gamma, beta = torch.ones(128, device=dev), torch.zeros(128, device=dev)
    got = ops.groupnorm(x0, gamma, beta, 1e-6, True, 32, x1=x1)
    ref = F.silu(F.group_norm(torch.cat([x0, x1], -1).double().permute(0, 2, 1), 32, eps=1e-6)).permute(0, 2, 1)
    assert bool(((got.double() - ref).abs() <= ref.abs() * 2.0 ** -8 + 2e-3).all())


# ---------------------------------------------------------------- attention


@pytest.mark.parametrize("profile", [False, True])
def test_attention_vae_bf16(dev, profile):
    from fast_image_editing_with_generative_models_b200 import ops
    from fast_image_editing_with_generative_models_b200.engine import _VAEAttention
    ntok, d = 1024, 512
    q = _randn((ntok, d), 70, dev, 3.0).to(BF)
    k = _randn((ntok, d), 71, dev, 3.0).to(BF)
    v = _randn((ntok, d), 72, dev).to(BF)
    vt = v.t().contiguous()
    scale = 1.0 / math.sqrt(d)
    if profile:
        got = _VAEAttention._attention_unfused(q, k, vt, ntok, d, scale, ntok, True)
    else:
        got = ops.attention_vae(q, k, vt, scale)
    assert got.dtype == BF
    ref = F.scaled_dot_product_attention(q.float()[None, None], k.float()[None, None], v.float()[None, None])[0, 0]
    _close(got, ref, 1e-2, f"attention_vae bf16 (unfused={profile})")


# ---------------------------------------------------------------- VAE parity


def _vae_errs(vae, vp, vcfg, img, z, dev):
    """(engine, torch-bf16 oracle) max-abs errors against the fp32 oracle for encode moments and decode, and the engine's decoded SSIM."""
    from fast_image_editing_with_generative_models_b200 import ops
    mom = vae.encode_moments(ops.preprocess_pad8(img, True)).permute(0, 3, 1, 2).float()
    dec = vae.decode(z.permute(0, 2, 3, 1).contiguous().half() * vcfg.scaling_factor).permute(0, 3, 1, 2)[:, :3].float()
    with torch.no_grad():
        p32 = O.to_dtype(vp, torch.float32, dev)
        m32 = O.vae_encode_moments(p32, vcfg, O.preprocess_image(img, torch.float32))
        d32 = O.vae_decode(p32, vcfg, z.half().float())
        del p32
        pbf = O.to_dtype(vp, BF, dev)
        mbf = O.vae_encode_moments(pbf, vcfg, O.preprocess_image(img, BF)).float()
        dbf = O.vae_decode(pbf, vcfg, z.half().to(BF)).float()
        del pbf
    e = dict(mom=float((mom - m32).abs().max()), mom_torch_bf16=float((mbf - m32).abs().max()),
             dec=float((dec - d32).abs().max()), dec_torch_bf16=float((dbf - d32).abs().max()),
             ssim=O.ssim(((dec + 1) / 2).clamp(0, 1), ((d32 + 1) / 2).clamp(0, 1)))
    print("bf16 VAE vs fp32 oracle:", {k: round(v, 6) for k, v in e.items()})
    return e, dec


def _check(e):
    assert e["mom"] <= e["mom_torch_bf16"], e
    assert e["dec"] <= e["dec_torch_bf16"], e
    assert e["ssim"] >= 0.99, e


def test_vae_bf16_tiny(dev):
    from fast_image_editing_with_generative_models_b200 import synthetic as S
    from fast_image_editing_with_generative_models_b200.engine import VAE
    vcfg = O.tiny_vae_config()
    vp = S.make_vae_params(vcfg)
    img = torch.from_numpy(np.stack([S.synthetic_image(s, 256, 256) for s in range(2)])).to(dev)
    z = torch.randn((2, 4, 32, 32), generator=_g(3)).to(dev)
    e, _ = _vae_errs(VAE(vp, vcfg, dev, dtype=BF), vp, vcfg, img, z, dev)
    _check(e)


def test_vae_bf16_sdxl_topology_1024(dev):
    from fast_image_editing_with_generative_models_b200 import configs as C
    from fast_image_editing_with_generative_models_b200 import synthetic as S
    from fast_image_editing_with_generative_models_b200.engine import VAE
    vcfg = C.VAEConfig()
    vp = S.make_vae_params(vcfg)
    img = torch.from_numpy(S.synthetic_image(0, 1024, 1024)[None]).to(dev)
    z = torch.randn((1, 4, 128, 128), generator=_g(4)).to(dev)
    e, _ = _vae_errs(VAE(vp, vcfg, dev, dtype=BF), vp, vcfg, img, z, dev)
    _check(e)


def test_vae_bf16_decodes_a_decoder_beyond_fp16(dev):
    """The case the bf16 VAE exists for: a decoder whose residual stream leaves the fp16 range (scaled from the mid block on, normalised
    away by conv_norm_out).  torch's fp16 execution of the oracle overflows; the engine's bf16 decode stays finite and accurate.  On the
    tiny VAE a factor of 2^14 leaves the stream at ~2.8e4, so the factor is 2^16; the test asserts that the case is out of range."""
    from fast_image_editing_with_generative_models_b200 import synthetic as S
    from fast_image_editing_with_generative_models_b200.engine import VAE
    vcfg = O.tiny_vae_config()
    vp = dict(S.make_vae_params(vcfg))
    for k in ("weight", "bias"):
        vp[f"decoder.mid_block.resnets.1.conv2.{k}"] = vp[f"decoder.mid_block.resnets.1.conv2.{k}"] * 2.0 ** 16
    z = torch.randn((2, 4, 32, 32), generator=_g(5)).to(dev)
    g, eps = vcfg.norm_groups, vcfg.norm_eps
    with torch.no_grad():
        p32 = O.to_dtype(vp, torch.float32, dev)
        h = O._conv(p32, "decoder.conv_in", O._conv(p32, "post_quant_conv", z.half().float(), padding=0))
        h = O.resnet_block(p32, "decoder.mid_block.resnets.0", h, None, g, eps)
        h = O._vae_attn(p32, "decoder.mid_block.attentions.0", h, g, eps)
        h = O.resnet_block(p32, "decoder.mid_block.resnets.1", h, None, g, eps)
        stream_max = float(h.abs().max())
        d16 = O.vae_decode(O.to_dtype(vp, torch.float16, dev), vcfg, z.half())
    print(f"fp32 oracle residual stream max-abs {stream_max:.4g}; torch-fp16 decode finite: {bool(torch.isfinite(d16).all())}")
    assert stream_max > 65504.0
    assert not bool(torch.isfinite(d16).all())
    img = torch.from_numpy(np.stack([S.synthetic_image(s, 256, 256) for s in range(2)])).to(dev)
    e, dec = _vae_errs(VAE(vp, vcfg, dev, dtype=BF), vp, vcfg, img, z, dev)
    assert bool(torch.isfinite(dec).all())
    _check(e)


# ---------------------------------------------------------------- end to end


def _edit(state, dev, B, H, strength, graph, floor=False):
    from fast_image_editing_with_generative_models_b200 import model_zoo
    from fast_image_editing_with_generative_models_b200 import synthetic as S
    eng = model_zoo.build_engine(dict(state, vae_dtype=BF), dev)
    assert eng.vae.dtype == BF
    ucfg = state["unet_cfg"]
    imgs = np.stack([S.synthetic_image(s, H, H) for s in range(B)])
    pe, pl = S.synthetic_prompt(0, ucfg.cross_attention_dim, ucfg.projection_class_embeddings_input_dim - 6 * ucfg.addition_time_embed_dim)
    noises = S.synthetic_noises(0, B, H // 8, H // 8)
    d_img = torch.from_numpy(imgs).to(dev)
    eager = eng.edit_batch(d_img, pe, pl, noises, strength=strength, return_latents=True, use_graph=False)
    e_lat, e_img = eager.latents.clone(), eager.images.clone()
    eager2 = eng.edit_batch(d_img, pe, pl, noises, strength=strength, return_latents=True, use_graph=False)
    assert torch.equal(eager2.latents, e_lat) and torch.equal(eager2.images, e_img), "two eager runs differ"
    if graph:
        g1 = eng.edit_batch(d_img, pe, pl, noises, strength=strength, return_latents=True, use_graph=True)
        g1_lat = g1.latents.clone()
        g2 = eng.edit_batch(d_img, pe, pl, noises, strength=strength, return_latents=True, use_graph=True)
        assert torch.equal(g1_lat, e_lat) and torch.equal(g2.latents, e_lat) and torch.equal(g2.images, e_img), "graph replay differs from eager"
    edges = eager2.edges.cpu().numpy()
    edges_ref = c_oracle.canny_u8(imgs, 100, 200, replicate3=True)
    assert np.array_equal(edges, edges_ref)
    del eng, eager, eager2
    torch.cuda.empty_cache()
    cast = lambda p: None if p is None else O.to_dtype(p, torch.float32, dev)
    m = O.EditModels(ucfg, cast(state["unet"]), state["cn_cfg"], cast(state["cn"]), state["vae_cfg"], cast(state["vae"]), cast(state.get("lora")), 1.0)
    with torch.no_grad():
        ref = O.edit_pipeline(m, d_img, torch.from_numpy(edges_ref).to(dev), pe.to(dev), pl.to(dev), noises, strength=strength, dtype=torch.float32,
                              return_all=True)
    lat_err = float((e_lat.permute(0, 3, 1, 2).float() - ref["latents"]).abs().max())
    s = O.ssim(e_img.permute(0, 3, 1, 2).float() / 255.0, ref["image_u8"].permute(0, 3, 1, 2).float() / 255.0)
    fl = None
    if floor:
        # the torch-bf16 floor: the same fp32 oracle pipeline with only its VAE executed by torch in bf16
        enc, dec = O.vae_encode_moments, O.vae_decode
        O.vae_encode_moments = lambda p, cfg, x: enc(O.to_dtype(p, BF, dev), cfg, x.to(BF)).float()
        O.vae_decode = lambda p, cfg, z: dec(O.to_dtype(p, BF, dev), cfg, z.to(BF)).float()
        try:
            with torch.no_grad():
                ref_bf = O.edit_pipeline(m, d_img, torch.from_numpy(edges_ref).to(dev), pe.to(dev), pl.to(dev), noises, strength=strength,
                                         dtype=torch.float32, return_all=True)
        finally:
            O.vae_encode_moments, O.vae_decode = enc, dec
        fl = float((ref_bf["latents"] - ref["latents"]).abs().max())
    print(f"bf16-VAE edit {state['unet_cfg'].name} b{B} {H}^2: latents max-abs {lat_err:.4g} (torch-bf16-VAE floor {fl}); SSIM {s:.5f}")
    assert lat_err <= 2e-2 or (fl is not None and lat_err <= fl), (lat_err, fl)
    assert s >= 0.99, s


def test_edit_bf16_vae_tiny(dev):
    from fast_image_editing_with_generative_models_b200 import model_zoo
    _edit(model_zoo.synthetic_state("sdxl", tiny=True), dev, 2, 256, 0.5, graph=True)


def test_edit_bf16_vae_ssd1b_1024(dev):
    from fast_image_editing_with_generative_models_b200 import model_zoo
    _edit(model_zoo.synthetic_state("ssd-1b"), dev, 1, 1024, 0.5, graph=True, floor=True)


def test_force_upcast_checkpoint_selects_bf16(dev, tmp_path):
    from fast_image_editing_with_generative_models_b200 import checkpoints as K
    from fast_image_editing_with_generative_models_b200 import configs as C
    from fast_image_editing_with_generative_models_b200 import synthetic as S
    from fast_image_editing_with_generative_models_b200.editor import FastEditor
    ucfg, ccfg, vcfg = C.tiny_unet_config(), C.tiny_controlnet_config(False), C.tiny_vae_config()
    K.save_model_dir(tmp_path / "unet", K.unet_config_to_json(ucfg), S.make_unet_params(ucfg))
    K.save_model_dir(tmp_path / "controlnet", {**K.unet_config_to_json(ccfg.unet), "conditioning_embedding_out_channels": list(ccfg.cond_channels)},
                     S.make_controlnet_params(ccfg))
    K.save_model_dir(tmp_path / "vae", {"block_out_channels": list(vcfg.block_out_channels), "layers_per_block": vcfg.layers_per_block,
                                        "latent_channels": vcfg.latent_channels, "scaling_factor": vcfg.scaling_factor, "force_upcast": True},
                     S.make_vae_params(vcfg))
    ck = {"unet": str(tmp_path / "unet"), "controlnet": str(tmp_path / "controlnet"), "vae": str(tmp_path / "vae")}
    ed = FastEditor("sdxl", device="cuda:0", checkpoints=ck, verbose=False)
    assert ed.vae_dtype == BF and ed._engine.vae.dtype == BF
    from PIL import Image
    out = ed.edit(Image.fromarray(S.synthetic_image(0, 256, 256)), "a photo", strength=0.5)
    a = np.asarray(out)
    assert a.shape == (1024, 1024, 3) and a.std() > 0
