"""GPU: each hand-written kernel (through the C-ABI) against the torch op it replaces, fp32 math on the same
fp16-rounded inputs.  Tolerances are written next to each check."""
import math

import pytest
import torch
import torch.nn.functional as F

from tests.util import rel_err

pytestmark = pytest.mark.gpu


def _ops():
    from fast_image_editing_with_generative_models_b200 import ops
    return ops


def _rand(shape, dev, seed, scale=1.0):
    g = torch.Generator("cpu").manual_seed(seed)
    return (torch.randn(shape, generator=g) * scale).to(dev)


# ------------------------------------------------------------------ elementwise / norms
def test_pre_post_process_pad8(cuda_dev):
    ops = _ops()
    img = torch.randint(0, 256, (2, 64, 96, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(0)).to(cuda_dev)
    x = ops.preprocess_pad8(img, True)[:, 1:-1, 1:97]
    ref = (2.0 * (img.float() / 255.0) - 1.0).half()
    assert torch.equal(x[..., :3], ref) and float(x[..., 3:].abs().max()) == 0.0
    c = ops.preprocess_pad8(img, False)[:, 1:-1, 1:97]
    assert torch.equal(c[..., :3], (img.float() / 255.0).half())
    y = _rand((2, 64, 96, 4), cuda_dev, 1).half()
    out = ops.postprocess(y)
    ref = ((y[..., :3] / 2 + 0.5).clamp(0, 1).float() * 255).round().to(torch.uint8)
    assert torch.equal(out, ref)


def test_silu(cuda_dev):
    ops = _ops()
    a = _rand((2, 16, 16, 64), cuda_dev, 2).half()
    assert rel_err(ops.silu(a), F.silu(a.float())) < 2e-3


def test_sincos(cuda_dev):
    ops = _ops()
    from oracle.diffusion_oracle import sincos_embedding
    vals = [499.0, 259.0, 1024.0, 0.0]
    out = ops.sincos_embedding(vals, 320, cuda_dev)
    ref = sincos_embedding(torch.tensor(vals), 320).to(cuda_dev)
    assert float((out.float() - ref).abs().max()) < 2e-3   # fp16 output of values in [-1,1]


@pytest.mark.parametrize("n,hw,c0,c1,silu,eps", [(2, 256, 64, 0, True, 1e-5), (2, 1024, 320, 0, True, 1e-5), (1, 4096, 128, 0, False, 1e-6),
                                                 (2, 64, 1280, 640, True, 1e-5), (2, 256, 640, 320, True, 1e-5), (1, 300, 512, 0, True, 1e-6)])
def test_groupnorm(cuda_dev, n, hw, c0, c1, silu, eps):
    ops = _ops()
    x0 = (_rand((n, hw, c0), cuda_dev, 4) * 1.5 + 0.3).half()
    x1 = (_rand((n, hw, c1), cuda_dev, 5) * 0.7 - 0.2).half() if c1 else None
    c = c0 + c1
    gamma = _rand((c,), cuda_dev, 6) * 0.1 + 1
    beta = _rand((c,), cuda_dev, 7) * 0.1
    out = ops.groupnorm(x0, gamma, beta, eps, silu, 32, x1)
    xc = torch.cat([x0, x1], dim=-1) if c1 else x0
    ref = F.group_norm(xc.float().permute(0, 2, 1), 32, gamma, beta, eps)
    ref = (F.silu(ref) if silu else ref).permute(0, 2, 1)
    assert float((out.float() - ref).abs().max()) < 8e-3     # fp16 output rounding of O(1..4) values


@pytest.mark.parametrize("rows,c", [(300, 128), (1024, 640), (2048, 1280), (77, 256)])
def test_layernorm(cuda_dev, rows, c):
    ops = _ops()
    x = (_rand((rows, c), cuda_dev, 8) * 2 + 0.5).half()
    gamma = _rand((c,), cuda_dev, 9) * 0.1 + 1
    beta = _rand((c,), cuda_dev, 10) * 0.1
    out = ops.layernorm(x, gamma, beta)
    ref = F.layer_norm(x.float(), (c,), gamma, beta, 1e-5)
    assert float((out.float() - ref).abs().max()) < 6e-3


@pytest.mark.parametrize("rows,cols", [(100, 1000), (64, 16384), (7, 20000), (33, 1020)])
def test_softmax_rows(cuda_dev, rows, cols):
    ops = _ops()
    s = _rand((rows, cols), cuda_dev, 11) * 5
    out = ops.softmax_rows(s, 0.3)
    ref = torch.softmax(s * 0.3, dim=-1)
    assert float((out.float() - ref).abs().max()) < 1e-3 and float((out.float().sum(-1) - 1).abs().max()) < 2e-2
    # fp16 scores (pre-scaled by the producing GEMM), softmax in place
    h = (s * 0.3).half()
    ref16 = torch.softmax(h.float(), dim=-1)
    out16 = ops.softmax_rows(h, 1.0, out=h)
    assert out16.data_ptr() == h.data_ptr() and float((out16.float() - ref16).abs().max()) < 1e-3


def test_scheduler_kernels_per_image_tables(cuda_dev):
    ops = _ops()
    from fast_image_editing_with_generative_models_b200.scheduler import LCMSchedule as Tables
    from oracle.diffusion_oracle import LCMSchedule, vae_sample
    sched = LCMSchedule()
    ts, begin = sched.img2img_timesteps(4, 0.5)
    _, add, table = Tables().batch_tables([4, 4], [0.5, 0.5], [1.5, 1.5])             # per-image coefficient tables, fp32
    add, table = torch.from_numpy(add).to(cuda_dev), torch.from_numpy(table).to(cuda_dev)
    mom = _rand((2, 16, 16, 8), cuda_dev, 12).half()
    xi = _rand((2, 16, 16, 4), cuda_dev, 13).half()
    nz = _rand((2, 16, 16, 4), cuda_dev, 14).half()
    sa, s1 = sched.add_noise_coeffs(ts[0])
    out, out16 = ops.vae_sample_add_noise(mom, xi, nz, 0.13025, add)
    assert out.dtype == torch.float32 and torch.equal(out16, out.half())
    z0 = vae_sample(mom.permute(0, 3, 1, 2).float(), xi.permute(0, 3, 1, 2).float(), 0.13025)
    ref = (sa * z0 + s1 * nz.permute(0, 3, 1, 2).float()).permute(0, 2, 3, 1)
    assert float((out.float() - ref).abs().max()) < 1e-5
    eps = _rand((4, 16, 16, 32), cuda_dev, 15).half()
    x = _rand((2, 16, 16, 4), cuda_dev, 16)
    for k in (0, 1):
        c = sched.step_coeffs(begin + k)
        got, got16 = ops.cfg_lcm_step(eps[:2], eps[2:], x, None if c["last"] else nz, table[k], c["last"])
        e = eps[:2, ..., :4].float() + 1.5 * (eps[2:, ..., :4].float() - eps[:2, ..., :4].float())
        ref = sched.step(e, begin + k, x, nz.float())
        assert float((got - ref).abs().max()) < 2e-5 and torch.equal(got16, got.half())


# ------------------------------------------------------------------ tensor-core GEMM (epilogue and tile forms: test_gpu_gemm.py) / conv
@pytest.mark.parametrize("m,c,n", [(16384, 1280, 3840), (4096, 640, 640), (100, 64, 192), (45000, 320, 352), (128, 128, 128)])
def test_gemm_folded_layernorm(cuda_dev, m, c, n):
    """x = A W0^T + b0 + res (producer writes LayerNorm row statistics) ; y = LN(x) W^T + b without a normalisation pass
    (BasicTransformerBlock: norm -> Linear), vs F.layer_norm + F.linear in fp32 on the same fp16 x."""
    ops = _ops()
    from fast_image_editing_with_generative_models_b200.weights import fold_layernorm
    a = _rand((m, 64), cuda_dev, 90).half()
    w0 = (_rand((c, 64), cuda_dev, 91) / 8).half()
    b0 = _rand((c,), cuda_dev, 92) * 0.5 + 0.7                    # rows with a non-zero mean
    res = (_rand((m, c), cuda_dev, 93) * 2).half()
    st = ops.zeros_i64((m, 2), cuda_dev)
    x = ops.gemm(a, w0, col_bias=b0, residual=res, ln_out=st)
    xf = x.float()
    s_ref, q_ref = xf.double().sum(1), (xf.double() ** 2).sum(1)
    got = st.double() / 2 ** 20
    assert float((got[:, 0] - s_ref).abs().max()) < 2e-3 * max(1.0, float(s_ref.abs().max())), "row sums"
    assert float(((got[:, 1] - q_ref).abs() / q_ref).max()) < 1e-4, "row sums of squares"
    gamma = 1.0 + 0.3 * _rand((c,), cuda_dev, 94)
    beta = 0.2 * _rand((c,), cuda_dev, 95)
    w = _rand((n, c), cuda_dev, 96) / math.sqrt(c)
    b = _rand((n,), cuda_dev, 97)
    ref = F.linear(F.layer_norm(xf, (c,), gamma, beta, 1e-5), w, b)
    wf, bf = fold_layernorm(w, b, gamma, beta)
    y = ops.gemm(x, wf, col_bias=bf, ln_in=(st, 1e-5))
    assert rel_err(y, ref) < 2e-3, rel_err(y, ref)
    y2 = ops.gemm(ops.layernorm(x, gamma, beta), w.half(), col_bias=b)           # the unfused path it replaces
    assert rel_err(y, ref) <= 1.5 * rel_err(y2, ref) + 1e-4, (rel_err(y, ref), rel_err(y2, ref))


@pytest.mark.parametrize("m,c", [(1024, 640), (16384, 1280), (200, 64)])
def test_gemm_folded_layernorm_geglu(cuda_dev, m, c):
    """LN -> GEGLU projection (FeedForward of BasicTransformerBlock) folded into one GEMM."""
    ops = _ops()
    from fast_image_editing_with_generative_models_b200.weights import fold_layernorm, pack_geglu
    x = (_rand((m, c), cuda_dev, 80) * 1.5 + 0.3).half()
    eye = torch.eye(c, device=cuda_dev).half()
    st = ops.zeros_i64((m, 2), cuda_dev)
    x2 = ops.gemm(x, eye, ln_out=st)                                 # copy through the GEMM to obtain the statistics
    assert torch.equal(x2, x)
    gamma = 1.0 + 0.3 * _rand((c,), cuda_dev, 81)
    beta = 0.2 * _rand((c,), cuda_dev, 82)
    w = _rand((8 * c, c), cuda_dev, 83) / math.sqrt(c)
    b = _rand((8 * c,), cuda_dev, 84)
    h = F.linear(F.layer_norm(x.float(), (c,), gamma, beta, 1e-5), w, b)
    ref = h[:, :4 * c] * F.gelu(h[:, 4 * c:])
    wg, bg = pack_geglu(*fold_layernorm(w, b, gamma, beta))
    y = ops.gemm(x, wg, col_bias=bg, act=ops.ACT_GEGLU, ln_in=(st, 1e-5))
    assert rel_err(y, ref) < 3e-3, rel_err(y, ref)


@pytest.mark.parametrize("n,h,w,cin,cout,stride,pad_mode", [
    (2, 16, 16, 64, 64, 1, 0), (2, 32, 32, 128, 320, 1, 0), (1, 128, 128, 64, 128, 1, 0), (2, 8, 8, 256, 256, 1, 0),
    (1, 256, 128, 64, 96, 1, 0), (2, 64, 64, 320, 320, 2, 0), (1, 64, 64, 128, 128, 2, 1), (2, 16, 16, 64, 64, 2, 0), (1, 256, 256, 64, 64, 2, 1)])
def test_conv3x3(cuda_dev, n, h, w, cin, cout, stride, pad_mode):
    ops = _ops()
    from fast_image_editing_with_generative_models_b200.weights import pack_conv3x3
    x = _rand((n, h, w, cin), cuda_dev, 40).half()
    wt = (_rand((cout, cin, 3, 3), cuda_dev, 41) / math.sqrt(9 * cin)).half()
    bias = _rand((cout,), cuda_dev, 42)
    out = ops.conv3x3(x, pack_conv3x3(wt), stride=stride, pad_mode=pad_mode, col_bias=bias)
    xn = x.permute(0, 3, 1, 2).float()
    if stride == 2 and pad_mode == 1:
        ref = F.conv2d(F.pad(xn, (0, 1, 0, 1)), wt.float(), bias, stride=2, padding=0)
    else:
        ref = F.conv2d(xn, wt.float(), bias, stride=stride, padding=1)
    ref = ref.permute(0, 2, 3, 1)
    assert out.shape == ref.shape
    assert rel_err(out, ref) < 2e-3, rel_err(out, ref)


@pytest.mark.parametrize("n,h,w,cin,cout", [(2, 40, 256, 192, 160), (1, 128, 128, 320, 320), (3, 17, 384, 64, 32), (1, 512, 512, 128, 128)])
def test_conv3x3_halo_vs_per_tap(cuda_dev, n, h, w, cin, cout):
    """Stride-1 convs with >= 128-pixel rows use the halo form (input rows loaded once, taps read through shifted smem
    descriptors); it must agree with the per-tap form bit-for-bit up to accumulation order, and with F.conv2d."""
    ops = _ops()
    from fast_image_editing_with_generative_models_b200 import _lib
    from fast_image_editing_with_generative_models_b200.weights import pack_conv3x3
    x = _rand((n, h, w, cin), cuda_dev, 56).half()
    wt = (_rand((cout, cin, 3, 3), cuda_dev, 57) / math.sqrt(9 * cin)).half()
    bias = _rand((cout,), cuda_dev, 58)
    res = _rand((n, h, w, cout), cuda_dev, 59).half()
    wp = pack_conv3x3(wt)
    L = _lib.lib()
    try:
        L.fie_tune_conv_halo(1, 4096)
        out_h = ops.conv3x3(x, wp, col_bias=bias, residual=res)
        L.fie_tune_conv_halo(0, 0)
        out_t = ops.conv3x3(x, wp, col_bias=bias, residual=res)
    finally:
        L.fie_tune_conv_halo(1, 640)
    ref = F.conv2d(x.permute(0, 3, 1, 2).float(), wt.float(), bias, padding=1).permute(0, 2, 3, 1) + res.float()
    assert rel_err(out_t, ref) < 2e-3, rel_err(out_t, ref)
    assert rel_err(out_h, ref) < 2e-3, rel_err(out_h, ref)
    assert float((out_h.float() - out_t.float()).abs().max()) <= 2e-2 * float(ref.abs().max())


@pytest.mark.parametrize("n,h,w,cin,cout,groups", [(2, 64, 64, 128, 128, 32), (1, 128, 128, 64, 256, 32), (3, 32, 32, 128, 512, 32), (2, 16, 16, 64, 64, 16)])
def test_conv_epilogue_groupnorm_statistics(cuda_dev, n, h, w, cin, cout, groups):
    """GroupNorm statistics accumulated by the producing convolution's epilogue (fixed-point integer atomics) equal the
    statistics kernel's, and the GroupNorm that consumes them matches F.group_norm; both are bit-reproducible."""
    ops = _ops()
    from fast_image_editing_with_generative_models_b200.weights import pack_conv3x3
    monkey_cpg, ops.GN_FUSE_CPG = ops.GN_FUSE_CPG, (4, 8, 16, 32)        # exercise every supported group width
    try:
        _check_conv_gn_stats(ops, pack_conv3x3, cuda_dev, n, h, w, cin, cout, groups)
    finally:
        ops.GN_FUSE_CPG = monkey_cpg


def _check_conv_gn_stats(ops, pack_conv3x3, cuda_dev, n, h, w, cin, cout, groups):
    x = _rand((n, h, w, cin), cuda_dev, 70).half()
    wt = (_rand((cout, cin, 3, 3), cuda_dev, 71) / math.sqrt(9 * cin)).half()
    bias = _rand((cout,), cuda_dev, 72)
    res = _rand((n, h, w, cout), cuda_dev, 73).half()
    gamma = _rand((cout,), cuda_dev, 74) * 0.1 + 1
    beta = _rand((cout,), cuda_dev, 75) * 0.1
    wp = pack_conv3x3(wt)
    y = ops.conv3x3(x, wp, col_bias=bias, residual=res, gn_groups=groups)
    assert hasattr(y, "_gn_stats")
    st = y._gn_stats[0].clone()
    out_fused = ops.groupnorm(y, gamma, beta, 1e-6, True, groups)
    y2 = ops.conv3x3(x, wp, col_bias=bias, residual=res)                       # same values, no producer statistics
    assert torch.equal(y, y2) and not hasattr(y2, "_gn_stats")
    out_plain = ops.groupnorm(y2, gamma, beta, 1e-6, True, groups)
    ref = F.silu(F.group_norm(y.float().permute(0, 3, 1, 2), groups, gamma, beta, 1e-6)).permute(0, 2, 3, 1)
    assert float((out_fused.float() - ref).abs().max()) < 8e-3
    assert float((out_fused.float() - out_plain.float()).abs().max()) < 4e-3       # fp32 (pre-rounding) vs fp16 inputs of the statistics
    # statistics against a float64 reduction of the fp16 output
    yg = y.double().view(n, h * w, groups, cout // groups)
    s_ref, q_ref = yg.sum(dim=(1, 3)), (yg * yg).sum(dim=(1, 3))
    s_got, q_got = st[..., 0].double() / 2 ** 20, st[..., 1].double() / 2 ** 20
    assert float(((s_got - s_ref).abs() / (q_ref.sqrt() + 1)).max()) < 5e-2 and float(((q_got - q_ref).abs() / q_ref).max()) < 2e-3
    # reproducible: integer accumulation does not depend on the order in which tiles finish
    y3 = ops.conv3x3(x, wp, col_bias=bias, residual=res, gn_groups=groups)
    assert torch.equal(y3._gn_stats[0], st)
    assert torch.equal(ops.groupnorm(y2, gamma, beta, 1e-6, True, groups), out_plain)


def test_conv3x3_small_cout_and_epilogue(cuda_dev):
    ops = _ops()
    from fast_image_editing_with_generative_models_b200.weights import pack_conv3x3
    n, h, w, cin, cout = 2, 32, 32, 128, 4
    x = _rand((n, h, w, cin), cuda_dev, 43).half()
    wt = (_rand((cout, cin, 3, 3), cuda_dev, 44) / math.sqrt(9 * cin)).half()
    bias = _rand((cout,), cuda_dev, 45)
    wp = pack_conv3x3(wt, pad_cout_to=32)
    bp = torch.zeros(32, device=cuda_dev); bp[:cout] = bias
    out = ops.conv3x3(x, wp, cout_valid=cout, col_bias=bp)
    ref = F.conv2d(x.permute(0, 3, 1, 2).float(), wt.float(), bias, padding=1).permute(0, 2, 3, 1)
    assert out.shape == (n, h, w, cout) and rel_err(out, ref) < 2e-3
    # time-embedding broadcast + residual
    cout = 128
    wt = (_rand((cout, cin, 3, 3), cuda_dev, 46) / math.sqrt(9 * cin)).half()
    temb = _rand((n, cout), cuda_dev, 47)
    res = _rand((n, h, w, cout), cuda_dev, 48).half()
    out = ops.conv3x3(x, pack_conv3x3(wt), row_bias=temb, rows_per_group=h * w, residual=res)
    ref = F.conv2d(x.permute(0, 3, 1, 2).float(), wt.float(), None, padding=1).permute(0, 2, 3, 1) + temb[:, None, None, :] + res.float()
    assert rel_err(out, ref) < 2e-3


@pytest.mark.parametrize("n,h,w,cin,cout", [(2, 16, 16, 64, 64), (2, 32, 32, 128, 320), (1, 128, 128, 64, 128), (2, 8, 8, 256, 256), (1, 64, 256, 64, 96)])
def test_conv_up2x(cuda_dev, n, h, w, cin, cout):
    """Fused nearest-2x upsample + conv3x3 (Upsample2D) vs F.interpolate + F.conv2d."""
    ops = _ops()
    from fast_image_editing_with_generative_models_b200.weights import pack_conv_up2x
    x = _rand((n, h, w, cin), cuda_dev, 70).half()
    wt = (_rand((cout, cin, 3, 3), cuda_dev, 71) / math.sqrt(9 * cin)).half()
    bias = _rand((cout,), cuda_dev, 72)
    out = ops.conv_up2x(x, pack_conv_up2x(wt), col_bias=bias)
    ref = F.conv2d(F.interpolate(x.permute(0, 3, 1, 2).float(), scale_factor=2.0, mode="nearest"), wt.float(), bias, padding=1).permute(0, 2, 3, 1)
    assert out.shape == ref.shape
    assert rel_err(out, ref) < 3e-3, rel_err(out, ref)     # phase weights are fp32 sums rounded once to fp16


def test_conv3x3_cin4(cuda_dev):
    ops = _ops()
    n, h, w, cout = 2, 40, 56, 320
    x = _rand((n, h, w, 4), cuda_dev, 50).half()
    wt = _rand((cout, 4, 3, 3), cuda_dev, 51) / 6
    bias = _rand((cout,), cuda_dev, 52)
    out = ops.conv3x3_cin4(x, wt.permute(0, 2, 3, 1).contiguous(), bias, cout)
    ref = F.conv2d(x.permute(0, 3, 1, 2).float(), wt, bias, padding=1).permute(0, 2, 3, 1)
    assert rel_err(out, ref) < 2e-3
    out = ops.conv3x3_cin4(x, wt[:16].permute(0, 2, 3, 1).contiguous(), bias[:16], 16, ld_out=64, act=ops.ACT_SILU)
    ref = F.silu(F.conv2d(x.permute(0, 3, 1, 2).float(), wt[:16], bias[:16], padding=1)).permute(0, 2, 3, 1)
    assert rel_err(out[..., :16], ref) < 2e-3 and float(out[..., 16:].abs().max()) == 0.0


@pytest.mark.parametrize("n,h,w,cout,silu", [(2, 128, 128, 128, False), (1, 256, 256, 64, True), (2, 64, 32, 96, False), (1, 1024, 1024, 128, False)])
def test_conv3x3_c8_image_input(cuda_dev, n, h, w, cout, silu):
    """Tensor-core conv_in on the zero-padded 8-channel image layout (overlapping TMA view) vs F.conv2d on the u8->fp16 image."""
    ops = _ops()
    from fast_image_editing_with_generative_models_b200.weights import pack_conv3x3_c8
    img = torch.randint(0, 256, (n, h, w, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(53)).to(cuda_dev)
    xp = ops.preprocess_pad8(img, True)
    x = (2.0 * (img.float() / 255.0) - 1.0).half()
    assert xp.shape == (n, h + 2, w + 8, 8)
    assert torch.equal(xp[:, 1:h + 1, 1:w + 1, :3], x) and float(xp[..., 3:].abs().max()) == 0.0
    assert float(xp[:, 0].abs().max()) == 0.0 and float(xp[:, -1].abs().max()) == 0.0 and float(xp[:, :, 0].abs().max()) == 0.0 and float(xp[:, :, w + 1:].abs().max()) == 0.0
    wt = _rand((cout, 3, 3, 3), cuda_dev, 54) / 5
    bias = _rand((cout,), cuda_dev, 55)
    out = ops.conv3x3_c8(xp, pack_conv3x3_c8(wt), col_bias=bias, act=ops.ACT_SILU if silu else ops.ACT_NONE)
    ref = F.conv2d(x.permute(0, 3, 1, 2).float(), wt, bias, padding=1)        # fp32 weights: the kernel carries them as hi + lo fp16
    ref = (F.silu(ref) if silu else ref).permute(0, 2, 3, 1)
    assert rel_err(out, ref) < 1e-3, rel_err(out, ref)


@pytest.mark.parametrize("n,h,w,cout,res", [(2, 128, 128, 320, True), (1, 16, 16, 64, False), (3, 32, 32, 512, True), (2, 8, 8, 32, False)])
def test_conv3x3_c8_latent_input(cuda_dev, n, h, w, cout, res):
    """Latent-resolution conv_in (4 channels padded to 8) with the ControlNet's fused `+ cond_emb` residual, vs F.conv2d."""
    ops = _ops()
    from fast_image_editing_with_generative_models_b200.weights import pack_conv3x3_c8
    x = (_rand((n, h, w, 4), cuda_dev, 56) * 3).half()
    xp = ops.pad8(x)
    assert xp.shape == (n, h + 2, w + 8, 8)
    assert torch.equal(xp[:, 1:h + 1, 1:w + 1, :4], x) and float(xp[..., 4:].abs().max()) == 0.0
    assert float(xp[:, 0].abs().max()) == 0.0 and float(xp[:, -1].abs().max()) == 0.0 and float(xp[:, :, 0].abs().max()) == 0.0 and float(xp[:, :, w + 1:].abs().max()) == 0.0
    wt = _rand((cout, 4, 3, 3), cuda_dev, 57) / 6
    bias = _rand((cout,), cuda_dev, 58)
    r = _rand((n, h, w, cout), cuda_dev, 59).half() if res else None
    out = ops.conv3x3_c8(xp, pack_conv3x3_c8(wt), col_bias=bias, residual=r)
    ref = F.conv2d(x.permute(0, 3, 1, 2).float(), wt, bias, padding=1).permute(0, 2, 3, 1)
    if res:
        ref = ref + r.float()
    assert rel_err(out, ref) < 1e-3, rel_err(out, ref)


# ------------------------------------------------------------------ softmax (the d=64 attention kernels: test_gpu_attention.py)
@pytest.mark.parametrize("rows,cols,d", [(300, 1016, 64), (512, 16384, 512), (100, 4096, 128)])
def test_softmax_exp_with_row_scale_in_the_pv_gemm(cuda_dev, rows, cols, d):
    """VAE mid-block attention path: exp-only softmax (unnormalised fp16 P', 1 / rowsum on the side) + P V GEMM with the row scale in
    its epilogue == softmax(S) @ V."""
    ops = _ops()
    s = (_rand((rows, cols), cuda_dev, 85) * 3).half()
    v = _rand((cols, d), cuda_dev, 86).half()
    vt = v.t().contiguous()
    p, inv = ops.softmax_rows_exp(s.clone(), 1.0)
    assert float(p.float().max()) <= 1.0 and float(p.float().max(1).values.min()) == 1.0      # the row maximum maps to exactly 1
    assert torch.allclose(inv, 1.0 / p.float().sum(1), rtol=1e-5)
    out = ops.gemm(p, vt, row_scale=inv)
    ref = torch.softmax(s.float(), dim=1) @ v.float()
    assert rel_err(out, ref) < 2e-3, rel_err(out, ref)
    s2 = s.clone()
    p2, inv2 = ops.softmax_rows_exp(s2, 1.0, out=s2)                                           # in place
    assert torch.equal(p2, p) and torch.equal(inv2, inv)
    old = ops.gemm(ops.softmax_rows(s.clone(), 1.0), vt)                                       # the normalising form it replaces
    assert rel_err(out, ref) <= rel_err(old, ref) + 1e-4


# ------------------------------------------------------------------ guard bands (compute-sanitizer is not available on the GPU pool)
def test_conv_and_groupnorm_write_only_their_output(cuda_dev):
    """Outputs carved out of one sentinel-filled arena, back to back: a kernel that overruns its tensor corrupts the neighbour's guard."""
    ops = _ops()
    from fast_image_editing_with_generative_models_b200.weights import pack_conv3x3
    n, h, w_, cin, cout = 2, 24, 32, 64, 96
    x = _rand((n, h, w_, cin), cuda_dev, 77).half()
    wt = pack_conv3x3((_rand((cout, cin, 3, 3), cuda_dev, 78) / math.sqrt(9 * cin)).half())
    arena = torch.full((64 + n * h * w_ * cout + 64,), 1234.0, dtype=torch.float16, device=cuda_dev)
    out = arena[64:64 + n * h * w_ * cout].view(n, h, w_, cout)
    ops.conv3x3(x, wt, out=out)
    torch.cuda.synchronize()
    assert bool((arena[:64] == 1234.0).all()) and bool((arena[-64:] == 1234.0).all())
    ref = F.conv2d(x.permute(0, 3, 1, 2).float(), wt.view(cout, 3, 3, cin).permute(0, 3, 1, 2).float(), padding=1).permute(0, 2, 3, 1)
    assert rel_err(out, ref) < 2e-3


@pytest.mark.parametrize("ntok,chunk", [(16384, 0), (16384, 4096), (4096, 0), (1000, 384)])
def test_attn_vae_d512_matches_fp32_sdpa(cuda_dev, ntok, chunk):
    """fie_attn_vae_d512_f16 (SURVEY 8(b)): softmax(q k^T / sqrt(512)) v for the VAE mid-block attention vs fp32
    F.scaled_dot_product_attention, at the path's size (16 384 tokens) and ragged ones, fp16 and fp32 scores."""
    import torch.nn.functional as F
    from fast_image_editing_with_generative_models_b200 import ops
    d = 512
    g = torch.Generator("cpu").manual_seed(ntok + chunk)
    q, k, v = (torch.randn((ntok, d), generator=g).to(cuda_dev).half() for _ in range(3))
    ref = F.scaled_dot_product_attention(q.float()[None, None], k.float()[None, None], v.float()[None, None])[0, 0]
    vt = v.t().contiguous()
    for f32 in (False, True):
        out = ops.attention_vae(q, k, vt, d ** -0.5, f32_scores=f32, chunk_rows=chunk).float()
        err = float((out - ref).abs().max())
        assert err < 2e-3 * max(1.0, float(ref.abs().max())), (f32, err)


def test_attn_vae_large_logits_need_fp32_scores(cuda_dev):
    """Logits in the hundreds (what real SDXL-VAE checkpoints produce, ADVICE r1): fp16 scores quantise them to 0.125-0.25 before the
    exponential; the fp32-score mode (the default when real checkpoints are loaded) stays at fp16-output accuracy."""
    import torch.nn.functional as F
    from fast_image_editing_with_generative_models_b200 import ops
    ntok, d = 2048, 512
    g = torch.Generator("cpu").manual_seed(5)
    q = (torch.randn((ntok, d), generator=g) * 4.0).to(cuda_dev).half()
    k = (torch.randn((ntok, d), generator=g) * 4.0).to(cuda_dev).half()
    v = torch.randn((ntok, d), generator=g).to(cuda_dev).half()
    ref = F.scaled_dot_product_attention(q.float()[None, None], k.float()[None, None], v.float()[None, None])[0, 0]
    assert float((q.float() @ k.float().t() * d ** -0.5).abs().max()) > 60           # the regime in question
    vt = v.t().contiguous()
    e32 = float((ops.attention_vae(q, k, vt, d ** -0.5, f32_scores=True).float() - ref).abs().max())
    e16 = float((ops.attention_vae(q, k, vt, d ** -0.5, f32_scores=False).float() - ref).abs().max())
    print("large-logit VAE attention: max-abs error fp32 scores", e32, "fp16 scores", e16)
    assert e32 < 5e-3 and e32 <= e16


@pytest.mark.parametrize("n,hw,c0,c1,silu", [(2, 1024, 1280, 0, True), (2, 1024, 1280, 1280, True), (2, 4096, 640, 0, False), (2, 4096, 1280, 640, True),
                                             (2, 16384, 320, 0, True), (1, 16384, 640, 320, True), (2, 16384, 320, 320, True), (3, 1000, 320, 0, True),
                                             (2, 16384, 512, 0, False)])
def test_groupnorm_single_pass_cluster_kernel(cuda_dev, n, hw, c0, c1, silu, monkeypatch):
    """k_gn_slab: the UNet / ControlNet norms (10..80 channels per group; concatenated skip sources whose boundary falls INSIDE a
    group; clusters of 1, 2, 4 and 8 CTAs; a row count that does not divide by the cluster size) against fp32 torch, and against the
    two-kernel path it replaces.  A large common offset checks the two-pass variance (no E[x^2] - mean^2 cancellation)."""
    ops = _ops()
    from fast_image_editing_with_generative_models_b200 import _lib
    _lib.lib().fie_tune_groupnorm_slab(8)              # allow clusters (the default policy only takes single-CTA slabs)
    x0 = (_rand((n, hw, c0), cuda_dev, 40) * 1.5 + 0.3).half()
    x1 = (_rand((n, hw, c1), cuda_dev, 41) * 0.7 - 0.2).half() if c1 else None
    c = c0 + c1
    gamma = _rand((c,), cuda_dev, 42) * 0.1 + 1
    beta = _rand((c,), cuda_dev, 43) * 0.1
    out = ops.groupnorm(x0, gamma, beta, 1e-5, silu, 32, x1)
    xc = torch.cat([x0, x1], dim=-1) if c1 else x0
    ref = F.group_norm(xc.float().permute(0, 2, 1), 32, gamma, beta, 1e-5)
    ref = (F.silu(ref) if silu else ref).permute(0, 2, 1)
    assert float((out.float() - ref).abs().max()) < 8e-3
    assert torch.equal(out, ops.groupnorm(x0, gamma, beta, 1e-5, silu, 32, x1)), "must be deterministic"
    # large mean, small spread: fp32 E[x^2] - mean^2 would lose the variance; the two-pass form does not
    xo = (x0.float() * 0.05 + 60.0).half()
    out_o = ops.groupnorm(xo, gamma[:c0], beta[:c0], 1e-5, False, 32)
    ref_o = F.group_norm(xo.float().permute(0, 2, 1), 32, gamma[:c0], beta[:c0], 1e-5).permute(0, 2, 1)
    _lib.lib().fie_tune_groupnorm_slab(0)
    two = ops.groupnorm(x0, gamma, beta, 1e-5, silu, 32, x1)                   # the two-kernel path on the same input
    _lib.lib().fie_tune_groupnorm_slab(1)              # back to the default policy
    assert float((out_o.float() - ref_o).abs().max()) < 2e-2
    assert float((two.float() - out.float()).abs().max()) < 8e-3


def test_native_weight_packing_matches_the_torch_transforms(cuda_dev):
    """csrc/pack.cu (SURVEY 8(b) fie_pack_weights_*): the load-time transforms as CUDA kernels against weights.py's torch
    implementations on CPU tensors — layouts bit-exact, the fp32 reductions (LayerNorm fold, LoRA fuse) to fp32 rounding."""
    from fast_image_editing_with_generative_models_b200 import weights as Wt
    g = torch.Generator("cpu").manual_seed(7)
    rn = lambda *s: torch.randn(s, generator=g)
    w = rn(70, 24, 3, 3)
    for pads in ((None, None), (96, 64)):
        assert torch.equal(Wt.pack_conv3x3(w.to(cuda_dev), *pads).cpu(), Wt.pack_conv3x3(w, *pads))
    w8 = rn(40, 3, 3, 3) / 5
    assert torch.equal(Wt.pack_conv3x3_c8(w8.to(cuda_dev), 64).cpu(), Wt.pack_conv3x3_c8(w8, 64))
    w4 = rn(33, 4, 3, 3)
    assert torch.equal(Wt.pack_conv3x3_c8(w4.to(cuda_dev)).cpu(), Wt.pack_conv3x3_c8(w4))
    wu = rn(48, 64, 3, 3)
    assert torch.equal(Wt.pack_conv_up2x(wu.to(cuda_dev)).cpu(), Wt.pack_conv_up2x(wu))
    wl = rn(130, 96)
    assert torch.equal(Wt.cast_f16(wl.to(cuda_dev)).cpu(), wl.half())
    # LayerNorm fold: rows centred after the gamma product; bias = b + W beta
    wf, bf, ga, be = rn(200, 640) / 25, rn(200), 1 + 0.3 * rn(640), 0.2 * rn(640)
    for b_, be_ in ((bf, be), (None, be), (bf, None), (None, None)):
        w16, bias = Wt.fold_layernorm(wf.to(cuda_dev), None if b_ is None else b_.to(cuda_dev), ga.to(cuda_dev), None if be_ is None else be_.to(cuda_dev))
        r16, rb = Wt.fold_layernorm(wf, b_, ga, be_)
        assert w16.dtype == torch.float16 and bias.dtype == torch.float32
        assert float((w16.cpu().float() - r16.float()).abs().max()) <= 2 ** -11 * float(r16.float().abs().max())      # at most one fp16 ulp (fp32 mean order)
        assert float((bias.cpu() - rb).abs().max()) < 1e-5 * max(1.0, float(rb.abs().max()))
    # LoRA fuse: linear and convolution (A [r,in,k,k], B [out,r,1,1]), ragged sizes
    for shape_w, shape_a, shape_b in (((100, 70), (8, 70), (100, 8)), ((45, 20, 3, 3), (64, 20, 3, 3), (45, 64, 1, 1)), ((33, 17, 1, 1), (4, 17, 1, 1), (33, 4, 1, 1))):
        w0, a0, b0 = rn(*shape_w), rn(*shape_a), rn(*shape_b)
        got = Wt.fuse_lora(w0.to(cuda_dev), a0.to(cuda_dev), b0.to(cuda_dev), 0.75).cpu()
        ref = Wt.fuse_lora(w0, a0, b0, 0.75)
        assert got.shape == ref.shape and float((got - ref).abs().max()) < 1e-5 * float(ref.abs().max()) * 8


@pytest.mark.parametrize("mean_over_sigma", [1.0, 8.0, 30.0])
def test_gemm_folded_layernorm_activation_scale_stress(cuda_dev, mean_over_sigma):
    """ADVICE r1: the folded LayerNorm rounds the CENTRED weights to fp16, so its error grows with |mean(x)| / sigma(x) of the residual
    stream (real checkpoints carry rows with large common offsets).  The error is measured against fp32 LN + Linear and bounded by what the
    algebra predicts — mean/sigma * 2^-11 * ||w_n||_2 per output, i.e. a few 1e-3 of the output scale even at mean = 30 sigma — and must
    not exceed the unfused fp16 path (LayerNorm output rounded to fp16) by more than that term."""
    ops = _ops()
    from fast_image_editing_with_generative_models_b200.weights import fold_layernorm
    m, c, n = 2048, 1280, 640
    x = (_rand((m, c), cuda_dev, 110) * 1.0 + mean_over_sigma).half()
    eye = torch.eye(c, device=cuda_dev).half()
    st = ops.zeros_i64((m, 2), cuda_dev)
    assert torch.equal(ops.gemm(x, eye, ln_out=st), x)
    gamma = 1.0 + 0.3 * _rand((c,), cuda_dev, 111)
    beta = 0.2 * _rand((c,), cuda_dev, 112)
    w = _rand((n, c), cuda_dev, 113) / math.sqrt(c)
    b = _rand((n,), cuda_dev, 114)
    ref = F.linear(F.layer_norm(x.float(), (c,), gamma, beta, 1e-5), w, b)
    wf, bf = fold_layernorm(w, b, gamma, beta)
    y = ops.gemm(x, wf, col_bias=bf, ln_in=(st, 1e-5))
    y2 = ops.gemm(ops.layernorm(x, gamma, beta), w.half(), col_bias=b)
    e, e2 = rel_err(y, ref), rel_err(y2, ref)
    predicted = mean_over_sigma * 2 ** -11 * 1.3 / float(ref.abs().max()) * 3      # ||gamma * w_n|| ~ 1.3, three-sigma over 640 x 2048 outputs... loose by design
    print(f"mean/sigma {mean_over_sigma}: folded rel err {e:.3g}, unfused fp16 path {e2:.3g}, predicted fold term {predicted:.3g}")
    assert e < 2e-3 + 2 * predicted, (e, predicted)
    assert e <= e2 + 2 * predicted + 1e-4
