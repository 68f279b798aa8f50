"""GPU: the head_dim-64 attention kernels of csrc/attention.cu -- k_attention_d64_p (self-attention, nkv > 128: lazy reference max,
persistent grid) and k_attention_d64_kv1 (cross-attention and causal, nkv <= 128) -- against softmax(scale q k^T) v in float64 on
the same fp16 inputs.  Every check holds each output element to the bound of tests/attention_cases.py and prints the worst
err/tol of the case; tests/test_attention_cases_cpu.py shows on the CPU which kernel paths the inputs reach."""
import pytest
import torch
import torch.nn.functional as F

from tests import attention_cases as A
from tests.util import guarded

pytestmark = pytest.mark.gpu


def _ops():
    from fast_image_editing_with_generative_models_b200 import ops
    return ops


@pytest.fixture(scope="module")
def sms(cuda_dev):
    return torch.cuda.get_device_properties(cuda_dev).multi_processor_count


def _inputs(gen, b, heads, nq, nkv, seed, dev, scale=0.125):
    return tuple(t.to(dev) for t in A.GENERATORS[gen](b, heads, nq, nkv, seed, scale))


def _check(label, out, q, k, v, b, heads, nq, nkv, scale=0.125, causal=False):
    o64, pv = A.reference(q, k, v, b, heads, nq, nkv, scale, causal)
    r = A.err_ratio(out, o64, pv)
    print(f"{label}: worst err/tol {r:.3f}")
    assert r <= 1.0, (label, r)
    return o64


def _run(gen, b, heads, nq, nkv, seed, dev, scale=0.125, causal=False):
    q, k, v = _inputs(gen, b, heads, nq, nkv, seed, dev, scale)
    out = _ops().attention_d64(q, k, v, b, heads, nq, nkv, scale=scale, causal=causal)
    _check(f"{gen} b{b} h{heads} nq{nq} nkv{nkv} scale {scale}{' causal' if causal else ''}", out, q, k, v, b, heads, nq, nkv, scale, causal)
    return q, k, v, out


def _rand(shape, dev, seed):
    return torch.randn(shape, generator=torch.Generator("cpu").manual_seed(seed)).to(dev)


# ------------------------------------------------------------------ N(0, 1) inputs over both kernels
@pytest.mark.parametrize("b,heads,nq,nkv", [(1, 1, 128, 128), (2, 2, 256, 256), (2, 10, 1024, 1024), (2, 4, 256, 77), (1, 2, 64, 64), (2, 2, 4096, 4096), (1, 3, 200, 333),
                                            (16, 20, 1024, 77), (3, 5, 1000, 77), (2, 10, 4096, 77), (1, 1, 300, 1), (4, 7, 520, 128)])
def test_attention_d64(cuda_dev, b, heads, nq, nkv):
    c = heads * 64
    q = _rand((b * nq, c), cuda_dev, 60).half()
    k = _rand((b * nkv, c), cuda_dev, 61).half()
    v = _rand((b * nkv, c), cuda_dev, 62).half()
    out = _ops().attention_d64(q, k, v, b, heads, nq, nkv)
    _check(f"N(0,1) b{b} h{heads} nq{nq} nkv{nkv}", out, q, k, v, b, heads, nq, nkv)


# ------------------------------------------------------------------ A. the lazy reference max of k_attention_d64_p
@pytest.mark.parametrize("gen", ["late_max", "all_negative"])
@pytest.mark.parametrize("nkv", A.P_NKV)
def test_attention_rescale_path(cuda_dev, gen, nkv):
    """late_max: row maxima that grow by 0.37 to 300 (log2) per K/V tile, so the reference moves after the first tile in mixed
    warps, with stale first halves past 2^127 and the max in either half and in the ragged last tile.  all_negative: a zero-filled
    key past nkv taken into the max would flush every P to zero."""
    _run(gen, A.P_B, A.P_HEADS, A.P_NQ, nkv, nkv, cuda_dev)


# ------------------------------------------------------------------ B. persistent grid: several items per CTA
@pytest.mark.parametrize("case", ["sms+1 items, 2 tiles, empty 2nd Q tile", "2sms+1 items, 3 tiles, partial 2nd Q tile", "200 items, 4 tiles",
                                  "312 items, 7 tiles", "b16 h10 4096^2", "b16 h20 1024^2"])
def test_attention_persistent_grid(cuda_dev, sms, case):
    """Items (batch, head, 256 query rows) beyond the grid: each CTA switches Q buffers, wraps the 3-stage K/V ring across items,
    issues the next item's first S early and resets the row max and sum per item.  Both UNet self-attention shapes included."""
    b, heads, nq, nkv, gen = {
        "sms+1 items, 2 tiles, empty 2nd Q tile": (sms + 1, 1, 100, 256, "late_max"),
        "2sms+1 items, 3 tiles, partial 2nd Q tile": (1, 2 * sms + 1, 200, 384, "late_max"),
        "200 items, 4 tiles": (2, 50, 300, 512, "all_negative"),
        "312 items, 7 tiles": (8, 13, 600, 800, "late_max"),
        "b16 h10 4096^2": (16, 10, 4096, 4096, "late_max"),
        "b16 h20 1024^2": (16, 20, 1024, 1024, "normal"),
    }[case]
    _run(gen, b, heads, nq, nkv, 7, cuda_dev)


# ------------------------------------------------------------------ C. items do not depend on where or when they run
@pytest.mark.parametrize("nq,nkv,causal", [(600, 785, False), (1000, 77, False), (77, 77, True)])
def test_attention_items_are_independent(cuda_dev, nq, nkv, causal):
    """An item's arithmetic does not depend on the CTA that runs it or on the items before it, so a multi-item call equals, bit for
    bit, per-image and per-head calls (one item per CTA) and itself on a second run: state carried across items would show here."""
    ops = _ops()
    b, heads = 8, 20 if causal else 10
    q, k, v = _inputs("late_max" if nkv > 128 else "normal", b, heads, nq, nkv, 11, cuda_dev)
    out = ops.attention_d64(q, k, v, b, heads, nq, nkv, causal=causal)
    _check(f"items b{b} h{heads} nq{nq} nkv{nkv}{' causal' if causal else ''}", out, q, k, v, b, heads, nq, nkv, causal=causal)
    assert torch.equal(ops.attention_d64(q, k, v, b, heads, nq, nkv, causal=causal), out)
    for i in range(b):
        one = ops.attention_d64(q[i * nq:(i + 1) * nq], k[i * nkv:(i + 1) * nkv], v[i * nkv:(i + 1) * nkv], 1, heads, nq, nkv, causal=causal)
        assert torch.equal(one, out[i * nq:(i + 1) * nq]), ("image", i)
    for h in range(heads):
        cols = slice(h * 64, (h + 1) * 64)
        one = ops.attention_d64(q[:, cols], k[:, cols], v[:, cols], b, 1, nq, nkv, causal=causal)
        assert torch.equal(one, out[:, cols]), ("head", h)


# ------------------------------------------------------------------ D. cross-attention, k_attention_d64_kv1
@pytest.mark.parametrize("gen,scale", [("all_negative", 0.125), ("normal", 1.0)])
@pytest.mark.parametrize("nkv", A.KV1_NKV)
def test_cross_attention(cuda_dev, gen, scale, nkv):
    """Ragged key counts (masked columns of the 128-key tile; 16-column P V blocks cut at nkv) with all-negative logits, where a
    masked zero score in the max flushes P, and with peaked scale-1 rows."""
    _run(gen, A.KV1_B, A.KV1_HEADS, A.KV1_NQ, nkv, 100 + nkv, cuda_dev, scale)


@pytest.mark.parametrize("b,heads,nq", [(16, 10, 4096), (16, 20, 1024)])
def test_cross_attention_ctx_kv_views(cuda_dev, b, heads, nq):
    """The UNet's cross-attention shapes as the engine calls them: K and V are column views of one wide buffer holding the prompt
    K/V of every transformer block."""
    c, nkv = heads * 64, 77
    q = _rand((b * nq, c), cuda_dev, 80).half()
    ctx_kv = _rand((b * nkv, 24 * c), cuda_dev, 81).half()
    off = 9 * c
    k, v = ctx_kv[:, off:off + c], ctx_kv[:, off + c:off + 2 * c]
    out = _ops().attention_d64(q, k, v, b, heads, nq, nkv)
    _check(f"ctx_kv views b{b} h{heads} nq{nq} ldkv {ctx_kv.shape[1]}", out, q, k, v, b, heads, nq, nkv)


# ------------------------------------------------------------------ E. causal (CLIP text towers)
@pytest.mark.parametrize("scale", [0.125, 1.0])
@pytest.mark.parametrize("n", [1, 16, 64, 77, 128])
def test_causal_attention(cuda_dev, sms, n, scale):
    """Key j visible to query i iff j <= i, against float64 SDPA is_causal=True; more (batch, head) items than SMs.  Row 0 sees
    only key 0, so its output is V's row 0 exactly."""
    b, heads = 3, sms // 3 + 1
    q, k, v, out = _run("normal", b, heads, n, n, 200 + n, cuda_dev, scale, causal=True)
    qh, kh, vh = (t.double().view(b, n, heads, 64).transpose(1, 2) for t in (q, k, v))
    sdpa = F.scaled_dot_product_attention(qh, kh, vh, is_causal=True, scale=scale).transpose(1, 2).reshape(b * n, heads * 64)
    o64, _ = A.reference(q, k, v, b, heads, n, n, scale, causal=True)
    assert float((o64 - sdpa).abs().max()) < 1e-12
    assert torch.equal(out.view(b, n, heads * 64)[:, 0], v.view(b, n, heads * 64)[:, 0])


# ------------------------------------------------------------------ F. scale, strides, output store forms
@pytest.mark.parametrize("scale", [0.125, 1.0, 0.05])
@pytest.mark.parametrize("nkv", [77, 333])
def test_attention_scale(cuda_dev, scale, nkv):
    _run("normal", 2, 3, 300, nkv, 300 + nkv, cuda_dev, scale)


def test_attention_fused_qkv_views(cuda_dev):
    """q, k, v as column views of one fused qkv projection (leading dimension 3c), as the UNet self-attention passes them."""
    _check_fused_qkv(cuda_dev, 2, 5, 256)


@pytest.mark.parametrize("b,heads,n", [(2, 3, 785), (3, 4, 77)])
def test_attention_fused_qkv_views_ragged(cuda_dev, b, heads, n):
    """The same with a ragged last K/V tile (k_attention_d64_p) and with 77 tokens (k_attention_d64_kv1)."""
    _check_fused_qkv(cuda_dev, b, heads, n)


def _check_fused_qkv(cuda_dev, b, heads, n):
    c = heads * 64
    qkv = _rand((b * n, 3 * c), cuda_dev, 63).half()
    q, k, v = qkv[:, :c], qkv[:, c:2 * c], qkv[:, 2 * c:]
    out = _ops().attention_d64(q, k, v, b, heads, n, n)
    _check(f"fused qkv b{b} h{heads} n{n}", out, q, k, v, b, heads, n, n)


@pytest.mark.parametrize("nkv", [77, 333])
def test_attention_separate_leading_dims(cuda_dev, nkv):
    b, heads, nq = 2, 3, 300
    c = heads * 64
    q = _rand((b * nq, c + 64), cuda_dev, 64).half()[:, :c]
    k = _rand((b * nkv, 2 * c + 8), cuda_dev, 65).half()[:, c + 8:]
    v = _rand((b * nkv, c + 136), cuda_dev, 66).half()[:, 72:72 + c]
    assert len({q.stride(0), k.stride(0), v.stride(0)}) == 3
    out = _ops().attention_d64(q, k, v, b, heads, nq, nkv)
    _check(f"ldq {q.stride(0)} ldk {k.stride(0)} ldv {v.stride(0)} nkv {nkv}", out, q, k, v, b, heads, nq, nkv)


@pytest.mark.parametrize("nkv,causal", [(77, False), (333, False), (77, True)])
def test_attention_narrow_store(cuda_dev, nkv, causal):
    """Output rows that are not 32-byte aligned take the 16-byte store form: a row stride of c + 8, and an output that starts
    8 halves into its buffer.  Both must equal the aligned output bit for bit."""
    ops = _ops()
    b, heads = 2, 3
    nq = nkv if causal else 300
    c = heads * 64
    q, k, v = _inputs("normal", b, heads, nq, nkv, 400 + nkv, cuda_dev)
    wide = ops.attention_d64(q, k, v, b, heads, nq, nkv, causal=causal)
    _check(f"narrow store nkv{nkv}{' causal' if causal else ''}", wide, q, k, v, b, heads, nq, nkv, causal=causal)
    strided = torch.empty((b * nq, c + 8), dtype=torch.float16, device=cuda_dev)[:, :c]
    shifted = torch.empty((b * nq * c + 8,), dtype=torch.float16, device=cuda_dev)[8:].view(b * nq, c)
    for out in (strided, shifted):
        ops.attention_d64(q, k, v, b, heads, nq, nkv, out=out, causal=causal)
        assert torch.equal(out, wide)


# ------------------------------------------------------------------ G. guard bands
@pytest.mark.parametrize("b,heads,nq,nkv,pad,lead,causal", [(2, 3, 200, 333, 64, 64, False), (1, 2, 130, 77, 64, 64, False), (2, 2, 256, 256, 64, 64, False),
                                                            (2, 3, 200, 333, 8, 72, False), (1, 2, 130, 77, 8, 72, False), (3, 4, 77, 77, 8, 64, True),
                                                            (8, 10, 600, 785, 64, 64, False)])
def test_attention_writes_only_its_output(cuda_dev, b, heads, nq, nkv, pad, lead, causal):
    """The output inside a sentinel-filled buffer, with row padding pad and lead halves in front (pad 8 / lead 72: the 16-byte store
    form): rows past nq of the last Q tile and the padding stay intact."""
    ops = _ops()
    c = heads * 64
    q = _rand((b * nq, c), cuda_dev, 74).half(); k = _rand((b * nkv, c), cuda_dev, 75).half(); v = _rand((b * nkv, c), cuda_dev, 76).half()
    out, ok = guarded(b * nq, c, c + pad, cuda_dev, lead=lead)
    ops.attention_d64(q, k, v, b, heads, nq, nkv, out=out, causal=causal)
    torch.cuda.synchronize()
    assert ok()
    ref = ops.attention_d64(q, k, v, b, heads, nq, nkv, causal=causal)
    assert torch.equal(out, ref)
