"""GPU: the tensor-core GEMM (k_gemm_conv, csrc/gemm_conv.cu) against the float64 epilogue contract of tests/gemm_cases.py.  Every
check holds each output element to the per-element bound written out there and prints the worst err/tol of the case.  The tile
forms (CTA group, K blocks per stage, M sub-tiles, accumulator width) are forced one by one through fie_tune_gemm; the fast and the
slow (epi_slow_chunk) epilogue paths are each run with every activation; the fused LayerNorm / GroupNorm statistics are checked
against a float64 sum of the kernel's own fp16 output."""
import math

import pytest
import torch

from tests import gemm_cases as G
from tests.util import guarded

pytestmark = pytest.mark.gpu

ACTS = (G.NONE, G.SILU, G.GELU, G.QUICKGELU, G.RELU)


def _ops():
    from fast_image_editing_with_generative_models_b200 import ops
    return ops


def _lib():
    from fast_image_editing_with_generative_models_b200 import _lib
    return _lib


@pytest.fixture(scope="module")
def sms(cuda_dev):
    return torch.cuda.get_device_properties(cuda_dev).multi_processor_count


def _dev(dev, a, w, ep):
    return a.to(dev), w.to(dev), ep.to(dev)


def _gemm(a, w, ep, a1=None, out=None, **kw):
    return _ops().gemm(a, w, a1=a1, out=out, **ep.kwargs(), **kw)


def _check(label, out, ref, tol):
    r = G.err_ratio(out, ref, tol)
    print(f"{label}: worst err/tol {r:.3f}")
    assert r <= 1.0, (label, r)
    return r


def _out(m, n, ld, dev, dtype=torch.float16):
    return guarded(m, n, ld, dev, dtype=dtype)


def _ld(n, fast):
    """Output row stride: 32-byte aligned (fast epilogue path) or 16-byte aligned only (slow path)."""
    return (n + 15) // 16 * 16 + (16 if fast else 8)


def _run_forms(label, a, w, ep, dev, forms, a1=None, out_dtype=torch.float16, ld=None):
    """Every form in forms on one problem: each output within the bound and inside its guard bands.  Returns {form: output}."""
    lib = _lib().lib()
    m, n_out = a.shape[0], (w.shape[0] // 2 if ep.act == G.GEGLU else w.shape[0])
    ref, tol = G.expected(a, w, ep, out_dtype, a1)
    ld = ld or _ld(n_out, True)
    outs, worst = {}, 0.0
    for f in forms:
        out, ok = _out(m, n_out, ld, dev, out_dtype)
        with G.forced_form(lib, *f):
            _gemm(a, w, ep, a1=a1, out=out)
        torch.cuda.synchronize()
        assert ok(), (label, f)
        r = G.err_ratio(out, ref, tol)
        assert r <= 1.0, (label, f, r)
        worst = max(worst, r)
        outs[f] = out.clone()
    print(f"{label}: {len(forms)} forms, worst err/tol {worst:.3f}")
    return outs


def _assert_bit_identical(label, outs):
    forms = list(outs)
    diff = [f for f in forms[1:] if not torch.equal(outs[f], outs[forms[0]])]
    print(f"{label}: {len(forms) - len(diff)} of {len(forms)} forms bit-identical to {forms[0]}" + (f"; differ: {diff}" if diff else ""))
    assert not diff, (label, diff)


# ------------------------------------------------------------------ every tile form, full epilogue
FORM_SHAPES = {
    "partial last tile column, odd num_kb": (1000, 352, 320),
    "N % 32 = 8, K tail of 8": (300, 200, 72),
    "add-embedding M=2": (2, 1280, 2816),
    "add-embedding M=16": (16, 1280, 1280),
    "persistent ragged": (45000, 624, 256),
}


@pytest.mark.parametrize("name", list(FORM_SHAPES))
def test_gemm_forms(cuda_dev, name):
    """Col + row bias, m_bias, scale 0.5 and a residual in every (cg, kps, mt, block_n); all forms give the same bits: the K order of
    an element does not depend on the form, and the 32-column chunks that pick the fast or the slow epilogue are the same in all."""
    m, n, k = FORM_SHAPES[name]
    a, w, ep = _dev(cuda_dev, *G.generic(m, n, k, 100 + m % 97, rows_per_group=64))
    _assert_bit_identical(name, _run_forms(name, a, w, ep, cuda_dev, G.forms()))


def test_gemm_forms_two_source(cuda_dev):
    """A = [A0 | A1] along K (k_split = 384) with a ragged second source of 200 columns, both row-strided views."""
    m, n = 700, 288
    a, w, ep = _dev(cuda_dev, *G.generic(m, n, 584, 110))
    big0 = torch.zeros((m, 448), dtype=torch.float16, device=cuda_dev)
    big1 = torch.zeros((m, 216), dtype=torch.float16, device=cuda_dev)
    a0, a1 = big0[:, :384], big1[:, 8:208]
    a0.copy_(a[:, :384]); a1.copy_(a[:, 384:])
    _assert_bit_identical("two-source", _run_forms("two-source", a0, w, ep, cuda_dev, G.forms(), a1=a1))


@pytest.mark.parametrize("cg", [1, 2])
@pytest.mark.parametrize("extra", [-1, 0, 1])
def test_gemm_tile_counts_around_the_slot_count(cuda_dev, sms, cg, extra):
    """sms / cg - 1, sms / cg and sms / cg + 1 tiles: the last CTA runs a second tile (TMEM double-buffer parity, cross-tile residual
    and bias prefetch) or none; K = 320 gives an odd number of K blocks under KPS = 2.  The last tile is ragged in M."""
    slots = sms // cg
    n, k = 64, 320
    for f in [(cg, kps, mt, 64) for kps in (1, 2) for mt in (1, 2)]:
        m = 128 * cg * f[2] * (slots + extra) - 40
        a, w, ep = _dev(cuda_dev, *G.generic(m, n, k, 120 + cg, rows_per_group=32))
        _run_forms(f"{slots + extra} tiles {f}", a, w, ep, cuda_dev, [f])


# ------------------------------------------------------------------ the epilogue contract on both paths
PATH_SHAPES = {"fast": (1000, 320, 136, 256), "slow": (1000, 200, 136, 1000)}        # (M, N, K, rows_per_group)
SWEEP_N = {"fast": 896, "slow": 872}


def _path_case(gen, act, path, seed):
    m, n, k, rpg = PATH_SHAPES[path]
    if gen == "generic":
        return G.generic(m, n, k, seed, act=act, rows_per_group=rpg)
    if gen == "activation_sweep":
        return G.activation_sweep(256, SWEEP_N[path], 64, seed, act=act)
    if gen == "cancelling_acc":
        return G.cancelling_acc(m, n, 320, seed, act=act)
    return G.cancelling_residual(m, n, 320, seed, act=act)


@pytest.mark.parametrize("path", ["fast", "slow"])
@pytest.mark.parametrize("act", ACTS, ids=[G.ACT_NAMES[a] for a in ACTS])
@pytest.mark.parametrize("gen", ["generic", "activation_sweep", "cancelling_acc", "cancelling_residual"])
def test_gemm_epilogue_contract(cuda_dev, gen, act, path):
    """v = act(acc + col + row + m_bias) * scale + residual on the fast path (ldd % 16 == 0, rows_per_group % 32 == 0, full
    chunks) and on epi_slow_chunk (ldd = N + 8, rows_per_group = 1000, N % 32 != 0): generic inputs, pre swept over [-90, 20],
    an accumulator that cancels against the bias, and a residual that cancels v."""
    a, w, ep = _dev(cuda_dev, *_path_case(gen, act, path, 200 + act))
    m, n = a.shape[0], w.shape[0]
    out, ok = _out(m, n, _ld(n, path == "fast"), cuda_dev)
    _gemm(a, w, ep, out=out)
    torch.cuda.synchronize()
    assert ok()
    _check(f"{gen} {G.ACT_NAMES[act]} {path}", out, *G.expected(a, w, ep))


@pytest.mark.parametrize("act", ACTS, ids=[G.ACT_NAMES[a] for a in ACTS])
def test_gemm_row_scale(cuda_dev, act):
    """row_scale[m] * acc + biases (the softmax normalisation of the VAE attention) with each activation."""
    a, w, ep = _dev(cuda_dev, *G.generic(1000, 320, 136, 210 + act, act=act, m_bias=False, residual=False, scale=1.0, row_scale=True))
    out, ok = _out(1000, 320, _ld(320, True), cuda_dev)
    _gemm(a, w, ep, out=out)
    torch.cuda.synchronize()
    assert ok()
    _check(f"row_scale {G.ACT_NAMES[act]}", out, *G.expected(a, w, ep))


@pytest.mark.parametrize("path", ["fast", "slow"])
@pytest.mark.parametrize("n", [512, 640, 320])
def test_gemm_geglu_epilogue(cuda_dev, n, path):
    """GEGLU with col + row bias, scale 0.5 and a residual, block_n = 256, 128, 64, in each of its forms; on the slow path the
    GEGLU value and gate both come from epi_slow_chunk.  Then a residual that cancels v."""
    m, k = 300, 192
    rpg = 256 if path == "fast" else 1000
    a, w, ep = G.generic(m, n, k, 220 + n, act=G.GEGLU, m_bias=False, residual=False, rows_per_group=rpg)
    ep = G.replace(ep, residual=torch.randn((m, n // 2), generator=torch.Generator().manual_seed(n)).half())
    a, w, ep = _dev(cuda_dev, a, w, ep)
    label = f"geglu N={n} {path}"
    _assert_bit_identical(label, _run_forms(label, a, w, ep, cuda_dev, G.forms(n), ld=_ld(n // 2, path == "fast")))
    a, w, ep = _dev(cuda_dev, *G.cancelling_residual(m, n, k, 230 + n, act=G.GEGLU))
    out, ok = _out(m, n // 2, _ld(n // 2, path == "fast"), cuda_dev)
    _gemm(a, w, ep, out=out)
    torch.cuda.synchronize()
    assert ok()
    _check(f"cancelling_residual {label}", out, *G.expected(a, w, ep))


@pytest.mark.parametrize("act", [G.NONE, G.GELU])
def test_gemm_fp32_output_with_residual(cuda_dev, act):
    """fp32 output with an fp16 residual always takes the slow path; also with m_bias and an activation."""
    a, w, ep = _dev(cuda_dev, *G.generic(600, 320, 136, 240 + act, act=act))
    out = _gemm(a, w, ep, out_f32=True)
    assert out.dtype == torch.float32
    _check(f"fp32 out + residual {G.ACT_NAMES[act]}", out, *G.expected(a, w, ep, torch.float32))


@pytest.mark.parametrize("out_dtype", [torch.bfloat16, torch.float16, torch.float32], ids=["bf16", "fp16", "fp32"])
def test_gemm_bf16_operands_forms(cuda_dev, out_dtype):
    """bf16 A and W (the bf16 VAE) with bf16, fp16 or fp32 output in every form; the 16-bit residual is in the output's type."""
    a, w, ep = G.generic(1000, 352, 320, 250, dtype=torch.bfloat16, act=G.SILU, residual=out_dtype != torch.float32)
    if ep.residual is not None:
        ep = G.replace(ep, residual=ep.residual.to(out_dtype))
    a, w, ep = _dev(cuda_dev, a, w, ep)
    label = f"bf16 -> {str(out_dtype)[6:]}"
    _assert_bit_identical(label, _run_forms(label, a, w, ep, cuda_dev, G.forms(), out_dtype=out_dtype))


# ------------------------------------------------------------------ fused LayerNorm / GroupNorm statistics
def _stats_inputs(kind, m, n, seed, dev):
    if kind == "generic":
        return _dev(dev, *G.generic(m, n, 64, seed, m_bias=False, rows_per_group=1024))
    # every output is 1 + (2^-13 .. 3 2^-13), which fp16 rounds down to exactly 1: a sum of the unrounded values is off by ~2^-12 each
    g = torch.Generator().manual_seed(seed)
    a = (torch.randn((m, 64), generator=g) * 2.0 ** -6).half()
    w = (torch.randn((n, 64), generator=g) * 2.0 ** -12).half()
    return _dev(dev, a, w, G.Epi(col_bias=torch.full((n,), 1.0 + 2.0 ** -12)))


@pytest.mark.parametrize("kind", ["generic", "rounds_down"])
@pytest.mark.parametrize("n,groups", [(512, 32), (320, 10)])
def test_gemm_statistics(cuda_dev, sms, kind, n, groups):
    """ln_out (row sums) and gn_stats (per image and group) equal a float64 sum of the kernel's own fp16 output, in every form, with
    many tiles per CTA and images of 16 row tiles (gn_flush merges sums across tiles); bound: fp32 partial sums plus 2^-21 per
    fixed-point atomic.  A fixed form gives bit-identical statistics twice."""
    ops, lib = _ops(), _lib().lib()
    m, rows = 32768, 4096
    a, w, ep = _stats_inputs(kind, m, n, 260 + n, cuda_dev)
    cpg = n // groups
    worst = 0.0
    for f in G.forms():
        cg, _, mt, bn = f
        runs = []
        for _ in range(2 if f == (2, 2, 1, 128) else 1):
            st = ops.zeros_i64((m, 2), cuda_dev)
            with G.forced_form(lib, *f):
                out = _gemm(a, w, ep, ln_out=st, gn_groups=groups, gn_rows=rows)
            gst = out._gn_stats[0]
            runs.append((out, st, gst))
        if len(runs) == 2:
            assert all(torch.equal(x, y) for x, y in zip(runs[0], runs[1])), "statistics differ between two runs of one form"
        out, st, gst = runs[0]
        x = out.double()
        nb = math.ceil(n / bn)
        # ln_out: per row, 2 nb atomics of fp32 partial sums over <= bn / 2 values
        for j, (exact, absum) in enumerate(((x.sum(1), x.abs().sum(1)), ((x * x).sum(1), (x * x).sum(1)))):
            tol = (bn + 2) * 2.0 ** -24 * absum + 2 * nb * 2.0 ** -21
            worst = max(worst, float(((st[:, j].double() / 2 ** 20 - exact).abs() / tol).max()))
        # gn_stats: per image and group, partial sums over cpg values, a 5-step butterfly and up to T tiles, one atomic per 32 rows
        tiles = math.ceil(m / (128 * cg * mt)) * nb
        t_max = math.ceil(tiles / (sms // cg)) * mt
        xg = x.view(m // rows, rows, groups, cpg)
        for j, (exact, absum) in enumerate(((xg.sum((1, 3)), xg.abs().sum((1, 3))), ((xg * xg).sum((1, 3)), (xg * xg).sum((1, 3))))):
            tol = (cpg + 8 + t_max) * 2.0 ** -24 * absum + rows // 32 * 2.0 ** -21
            worst = max(worst, float(((gst[..., j].double() / 2 ** 20 - exact).abs() / tol).max()))
        assert worst <= 1.0, (kind, n, f, worst)
    print(f"statistics {kind} N={n}: {len(G.forms())} forms, worst err/tol {worst:.3f}")


# ------------------------------------------------------------------ forcing a form that has no legal tile
@pytest.mark.parametrize("code,block_n,n,act", [(G.form_code(0, 0, 2), 160, 320, G.NONE), (G.form_code(0, 0, 2), 0, 512, G.GEGLU),
                                                (3, 0, 320, G.NONE), (G.form_code(0, 3, 0), 0, 320, G.NONE)],
                         ids=["mt2 block_n 160", "mt2 geglu N=512", "cg3", "kps3"])
def test_forced_form_without_a_legal_tile_is_an_error(cuda_dev, code, block_n, n, act):
    """A forced (cg, kps, mt, block_n) that no tile matches raises instead of silently running the default form."""
    lib = _lib().lib()
    a, w, ep = _dev(cuda_dev, *G.generic(256, n, 64, 270, act=act, m_bias=False, residual=False))
    lib.fie_tune_gemm(code, block_n)
    try:
        with pytest.raises(_lib().FieError, match="forced"):
            _gemm(a, w, ep)
    finally:
        lib.fie_tune_gemm(0, 0)
    _gemm(a, w, ep)                                   # the default again


# ------------------------------------------------------------------ former test_gpu_kernels.py GEMM tests, held to the bound
def _rand(shape, dev, seed, scale=1.0):
    g = torch.Generator("cpu").manual_seed(seed)
    return (torch.randn(shape, generator=g) * scale).to(dev)


@pytest.mark.parametrize("m,n,k", [(128, 64, 64), (256, 160, 320), (300, 320, 640), (2048, 1280, 1280), (77, 640, 2048), (4096, 1920, 640), (2, 1280, 320), (512, 8, 8), (16384, 512, 512)])
def test_gemm_plain(cuda_dev, m, n, k):
    a = _rand((m, k), cuda_dev, 20).half()
    w = (_rand((n, k), cuda_dev, 21) / math.sqrt(k)).half()
    ep = G.Epi(col_bias=_rand((n,), cuda_dev, 22))
    _check(f"plain {m}x{n}x{k}", _gemm(a, w, ep), *G.expected(a, w, ep))


def test_gemm_epilogues(cuda_dev):
    m, n, k = 512, 640, 640
    a = _rand((m, k), cuda_dev, 23).half()
    w = (_rand((n, k), cuda_dev, 24) / math.sqrt(k)).half()
    bias = _rand((n,), cuda_dev, 25)
    res = _rand((m, n), cuda_dev, 26).half()
    rowb = _rand((2, n), cuda_dev, 27)
    for label, ep in (("bias residual scale", G.Epi(col_bias=bias, residual=res, scale=0.5)),
                      ("row bias silu", G.Epi(row_bias=rowb, rows_per_group=256, act=G.SILU)),
                      ("m_bias", G.Epi(m_bias=_rand((m,), cuda_dev, 28)))):
        _check(label, _gemm(a, w, ep), *G.expected(a, w, ep))
    ep = G.Epi()
    out = _gemm(a, w, ep, out_f32=True)
    assert out.dtype == torch.float32
    _check("fp32 out", out, *G.expected(a, w, ep, torch.float32))
    # two-source K (virtual concat)
    a0, a1 = a[:, :384].contiguous(), a[:, 384:].contiguous()
    _check("two-source", _gemm(a0, w, ep, a1=a1), *G.expected(a0, w, ep, a1=a1))
    # strided A view (row stride > K)
    big = _rand((m, 3 * k), cuda_dev, 29).half()
    _check("strided A", _gemm(big[:, k:2 * k], w, ep), *G.expected(big[:, k:2 * k], w, ep))


@pytest.mark.parametrize("force_bn", [0, 224, 160, 96])
def test_gemm_epilogue_persistent_ragged(cuda_dev, force_bn):
    """Many tiles per CTA, ragged M, N that leaves empty / partial accumulator chunks in the last tile column, bias + residual:
    exercises the epilogue's cross-item prefetch queues (residual, staged biases) across fast and slow chunks."""
    m, n, k = 45000, 624, 256
    a = _rand((m, k), cuda_dev, 33).half()
    w = (_rand((n, k), cuda_dev, 34) / math.sqrt(k)).half()
    bias = _rand((n,), cuda_dev, 35)
    res = _rand((m, n), cuda_dev, 36).half()
    rowb = _rand((m // 1000, n), cuda_dev, 37)
    eps = (G.Epi(col_bias=bias, residual=res), G.Epi(col_bias=bias, row_bias=rowb, rows_per_group=1000),
           G.Epi(col_bias=bias, row_bias=rowb, rows_per_group=1024, residual=res, scale=0.25))
    with G.forced_form(_lib().lib(), block_n=force_bn):
        outs = [_gemm(a, w, ep) for ep in eps]
    for i, (out, ep) in enumerate(zip(outs, eps)):
        _check(f"persistent ragged bn={force_bn} #{i}", out, *G.expected(a, w, ep))


@pytest.mark.parametrize("m,c", [(256, 64), (1024, 640), (300, 128)])
def test_gemm_geglu(cuda_dev, m, c):
    from fast_image_editing_with_generative_models_b200.weights import pack_geglu
    a = _rand((m, c), cuda_dev, 30).half()
    w = (_rand((8 * c, c), cuda_dev, 31) / math.sqrt(c)).half()
    b = _rand((8 * c,), cuda_dev, 32) * 0.5
    wp, bp = pack_geglu(w, b)
    ep = G.Epi(col_bias=bp, act=G.GEGLU)
    out = _gemm(a, wp, ep)
    assert out.shape == (m, 4 * c)
    _check(f"geglu {m}x{c}", out, *G.expected(a, wp, ep))


@pytest.mark.parametrize("m,n,k", [(300, 96, 128), (1000, 352, 64), (257, 640, 320), (128, 1280, 1280)])
def test_gemm_writes_only_its_output(cuda_dev, m, n, k):
    """Ragged M / N with a strided output inside a sentinel-filled buffer: rows >= M, columns >= N and the row padding stay intact
    (fast and slow epilogue paths, residual prefetch queue, LayerNorm statistics)."""
    a = _rand((m, k), cuda_dev, 70).half()
    w = (_rand((n, k), cuda_dev, 71) / math.sqrt(k)).half()
    ep = G.Epi(col_bias=_rand((n,), cuda_dev, 72), residual=_rand((m, n), cuda_dev, 73).half())
    ref, tol = G.expected(a, w, ep)
    for ld in (n + 16, n + 8):
        out, ok = guarded(m, n, ld, cuda_dev)
        st = torch.zeros((m + 8, 2), dtype=torch.int64, device=cuda_dev)
        use_ln = n % 32 == 0 and ld % 16 == 0
        _gemm(a, w, ep, out=out, ln_out=st[:m] if use_ln else None)
        torch.cuda.synchronize()
        assert ok(), (m, n, k, ld)
        _check(f"guarded {m}x{n}x{k} ld={ld}", out, ref, tol)
        assert int(st[m:].abs().sum()) == 0                              # statistics rows beyond M untouched
        if use_ln:
            assert float((st[:m, 0].double() / 2 ** 20 - out.float().double().sum(1)).abs().max()) < 1e-2
