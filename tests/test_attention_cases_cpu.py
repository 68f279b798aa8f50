"""CPU: the inputs of tests/test_gpu_attention.py reach the kernel paths they are meant to, and the error bound they are held to is
tight enough to catch a skipped rescale yet holds for the kernels' own rounding.  Uses the replay of k_attention_d64_p's lazy
reference-max rule and a torch emulation of its arithmetic (tests/attention_cases.py)."""
import math

import pytest
import torch
import torch.nn.functional as F

from tests import attention_cases as A

SL2 = A.scale_log2(0.125)


def _replay(gen, b, heads, nq, nkv, seed):
    q, k, v = A.GENERATORS[gen](b, heads, nq, nkv, seed)
    ov, moved = A.replay(A.scores32(q, k, b, heads, nq, nkv), SL2)
    return ov[..., 1:], moved[..., 1:]


@pytest.mark.parametrize("nkv", A.P_NKV)
def test_late_max_drives_the_rescale(nkv):
    """The rescale at tile j > 0 runs in many rows, in warps that also hold rows that do not move, with overshoots just below the
    threshold (P up to 2^7.9 without a move), just above it, and past 127 (first half recomputed)."""
    b, heads, nq = A.P_B, A.P_HEADS, A.P_NQ
    ov, moved = _replay("late_max", b, heads, nq, nkv, nkv)
    assert int(moved.any(-1).sum()) >= b * heads * nq // 2
    warps = moved[:, :, :nq // 32 * 32].reshape(b, heads, nq // 32, 32, -1)
    assert int((warps.any(3) & ~warps.all(3)).sum()) >= b * heads * (nq // 32)
    assert int(((ov > 7) & (ov < 8)).sum()) > 0 and int(((ov > 8) & (ov < 9)).sum()) > 0 and int((ov > 127).sum()) > 0
    # the fp32 scores of the CPU and the tensor cores may differ in the last bits: only STRADDLE rows come near the threshold
    straddle = torch.tensor([[c == A.STRADDLE for c in A.late_max_classes(nq, bi * heads + h)] for bi in range(b) for h in range(heads)])
    clear = ~straddle.view(b, heads, nq, 1).expand_as(ov)
    assert float((ov[clear] - A.THRESHOLD).abs().min()) >= 0.05


@pytest.mark.parametrize("nkv", A.P_NKV)
def test_late_max_peak_positions(nkv):
    """The tile maxima sit in the first half of even tiles, the second half of odd ones, and on the last key of the ragged last tile."""
    q, k, _ = A.late_max(1, 1, 64, nkv, nkv)
    k0 = k[:, 0].float()
    nt = (nkv + A.TILE - 1) // A.TILE
    for j in range(nt):
        pos = int(k0[j * A.TILE:(j + 1) * A.TILE].argmax())
        if j == nt - 1:
            assert j * A.TILE + pos == nkv - 1
        else:
            assert pos // 64 == j % 2
        assert float(k0[j * A.TILE:(j + 1) * A.TILE].max()) == j


@pytest.mark.parametrize("nkv", A.P_NKV + A.KV1_NKV)
def test_all_negative_rows_are_far_below_zero(nkv):
    """Every row max is below -30 in scaled log2 units, so P against a reference of 0 underflows fp16; last tiles of more than 64
    keys (197, 333) and key counts that are not multiples of 16 (kv1) are among the shapes."""
    b, heads, nq = (A.P_B, A.P_HEADS, A.P_NQ) if nkv > 128 else (A.KV1_B, A.KV1_HEADS, A.KV1_NQ)
    q, k, _ = A.all_negative(b, heads, nq, nkv, nkv if nkv > 128 else 100 + nkv)
    assert float(A.scores32(q, k, b, heads, nq, nkv).amax() * SL2) < -30
    assert float(torch.tensor(2.0 ** -30).half()) == 0.0


@pytest.mark.parametrize("b,heads,nq,nkv", [(2, 2, 256, 256), (2, 10, 1024, 1024), (2, 2, 4096, 4096), (1, 3, 200, 333)])
def test_normal_inputs_never_rescale(b, heads, nq, nkv):
    """The N(0, 1) inputs of test_attention_d64 (the only self-attention inputs the suite had before the rescale tests) never move
    the reference max after the first tile: on their own they leave the O rescale unchecked."""
    g = lambda seed, n: torch.randn((b * n, heads * 64), generator=torch.Generator("cpu").manual_seed(seed)).half()
    q, k = g(60, nq), g(61, nkv)
    ov, moved = A.replay(A.scores32(q, k, b, heads, nq, nkv), SL2)
    assert not bool(moved[..., 1:].any()) and float(ov[..., 1:].max()) < A.THRESHOLD - 2


@pytest.mark.parametrize("gen,nkv,scale", [("late_max", 197, 0.125), ("late_max", 1024, 0.125), ("all_negative", 333, 0.125),
                                           ("constant", 333, 0.125), ("normal", 785, 1.0), ("normal", 257, 0.05)])
def test_bound_holds_for_the_kernel_arithmetic(gen, nkv, scale):
    """The emulated kernel stays within half the bound; without the O rescale, the late-max rows exceed it."""
    b, heads, nq = 1, 2, 300
    q, k, v = A.GENERATORS[gen](b, heads, nq, nkv, 5, scale)
    o64, pv = A.reference(q, k, v, b, heads, nq, nkv, scale)
    r = A.err_ratio(A.emulate_p(q, k, v, b, heads, nq, nkv, scale), o64, pv)
    print(f"{gen} nkv {nkv} scale {scale}: emulated err/tol {r:.3f}")
    assert r <= 0.5
    if gen == "late_max":
        assert A.err_ratio(A.emulate_p(q, k, v, b, heads, nq, nkv, scale, rescale_o=False), o64, pv) > 1


def test_cubic_exp2_error():
    """The cubic exp2 of the kernel is within 8.8e-5 of 2^x (the figure in the error model)."""
    x = torch.linspace(-20, 8, 200001, dtype=torch.float64).float()
    rel = (A.ex2_cubic(x).double() / torch.exp2(x.double()) - 1).abs().max()
    assert float(rel) <= 8.8e-5


def test_reference_matches_sdpa():
    """The chunked float64 reference equals SDPA, plain and causal (top-left: key j visible to query i iff j <= i)."""
    b, heads, nq, nkv = 2, 3, 40, 40
    q, k, v = A.normal(b, heads, nq, nkv, 9)
    for causal in (False, True):
        o64, pv = A.reference(q, k, v, b, heads, nq, nkv, 0.3, causal, max_elems=nq * nkv * 2)
        qh, kh, vh = (t.double().view(b, -1, heads, 64).transpose(1, 2) for t in (q, k, v))
        ref = F.scaled_dot_product_attention(qh, kh, vh, is_causal=causal, scale=0.3).transpose(1, 2).reshape(b * nq, heads * 64)
        assert float((o64 - ref).abs().max()) < 1e-12
        assert bool((pv >= o64.abs() - 1e-12).all())


def test_constant_rows_give_the_mean_of_v():
    b, heads, nq, nkv = 1, 2, 64, 333
    q, k, v = A.constant_rows(b, heads, nq, nkv, 3)
    o64, _ = A.reference(q, k, v, b, heads, nq, nkv, 0.125)
    assert float((o64 - v.double().mean(0)).abs().max()) < 1e-12
    assert math.isfinite(float(o64.abs().max()))
