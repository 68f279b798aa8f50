"""CPU: the error bound of tests/gemm_cases.py holds for the GEMM's own arithmetic, emulated in fp32, with a margin of two, yet is
tight enough that each emulated epilogue defect exceeds it on at least one generator; the cancelling generators cancel."""
import pytest
import torch

from tests import gemm_cases as G

ACTS = (G.NONE, G.SILU, G.GELU, G.QUICKGELU, G.RELU)


def _cases():
    """(label, a, w, Epi, out_dtype): every generator, every activation, row_scale, bf16 operands and outputs, GEGLU."""
    cases = []
    for act in ACTS:
        n = G.ACT_NAMES[act]
        cases.append((f"generic {n}", *G.generic(300, 200, 136, 1 + act, act=act), torch.float16))
        cases.append((f"row_scale {n}", *G.generic(256, 96, 64, 11 + act, act=act, m_bias=False, residual=False, scale=1.0, row_scale=True), torch.float16))
        cases.append((f"sweep {n}", *G.activation_sweep(64, 880, 64, 21 + act, act=act), torch.float16))
        cases.append((f"cancelling_acc {n}", *G.cancelling_acc(128, 96, 320, 31 + act, act=act), torch.float16))
        cases.append((f"cancelling_residual {n}", *G.cancelling_residual(128, 96, 320, 41 + act, act=act), torch.float16))
    cases.append(("generic f32 out", *G.generic(128, 72, 200, 51, residual=False), torch.float32))
    for odt in (torch.bfloat16, torch.float16, torch.float32):
        a, w, ep = G.generic(192, 160, 128, 52, dtype=torch.bfloat16, residual=odt != torch.float32)
        if ep.residual is not None:
            ep = G.replace(ep, residual=ep.residual.to(odt))
        cases.append((f"bf16 -> {odt}", a, w, ep, odt))
    for n in (512, 640, 320):
        a, w, ep = G.generic(160, n, 128, 60 + n, act=G.GEGLU, m_bias=False, residual=False)
        ep = G.replace(ep, residual=torch.randn((160, n // 2), generator=torch.Generator().manual_seed(n)).half())
        cases.append((f"geglu N={n}", a, w, ep, torch.float16))
        cases.append((f"cancelling_residual geglu N={n}", *G.cancelling_residual(128, n, 128, 70 + n, act=G.GEGLU), torch.float16))
    return cases


CASES = _cases()


def _ratio(a, w, ep, odt, mutant=None):
    ref, tol = G.expected(a, w, ep, odt)
    return G.err_ratio(G.emulate(a, w, ep, odt, mutant=mutant), ref, tol)


@pytest.mark.parametrize("i", range(len(CASES)), ids=[c[0] for c in CASES])
def test_emulated_kernel_within_half_the_bound(i):
    label, a, w, ep, odt = CASES[i]
    r = _ratio(a, w, ep, odt)
    print(f"{label}: emulated err/tol {r:.3f}")
    assert r <= 0.5, (label, r)


@pytest.mark.parametrize("mutant", G.MUTANTS)
def test_each_emulated_defect_exceeds_the_bound(mutant):
    worst = max(((_ratio(a, w, ep, odt, mutant), label) for label, a, w, ep, odt in CASES), key=lambda t: t[0])
    print(f"{mutant}: worst err/tol {worst[0]:.3g} ({worst[1]})")
    assert worst[0] > 1.0, (mutant, worst)


def test_cancelling_accumulator_is_hundreds_of_times_pre():
    for act in ACTS:
        a, w, ep = G.cancelling_acc(128, 96, 320, 31 + act, act=act)
        d = G.reference(a, w, ep)
        ratio = d["acc"].abs() / d["pre"].abs().clamp_min(1e-30)
        assert float(ratio.median()) > 100, float(ratio.median())


def test_cancelling_residual_leaves_the_rounding_residue():
    for act in ACTS:
        a, w, ep = G.cancelling_residual(128, 96, 320, 41 + act, act=act)
        d = G.reference(a, w, ep)
        res = ep.residual.double()
        assert float(d["out"].abs().max()) <= 2.0 ** -11 * float(res.abs().max())      # |v - fp16(v)| <= 2^-11 |v|
        live = d["act"] != 0                                                         # (ReLU: half of the outputs are 0)
        assert float((d["out"][live] != 0).double().mean()) > 0.9                    # yet almost never exactly 0


@pytest.mark.parametrize("act", (G.SILU, G.GELU, G.QUICKGELU, G.RELU))
def test_activation_sweep_covers_the_tails(act):
    a, w, ep = G.activation_sweep(64, 880, 64, 21 + act, act=act)
    pre = G.reference(a, w, ep)["pre"]
    assert float(pre.min()) < -89 and float(pre.max()) > 19.8
    hist = torch.histc(pre.float(), bins=110, min=-90, max=20)
    assert int((hist == 0).sum()) == 0                                               # every unit interval of [-90, 20] is hit
    assert float(G.reference(a, w, ep)["acc"].abs().max()) < 0.5


def test_tanh_gelu_differs_by_ten_percent_in_the_tail():
    x = torch.tensor([-3.0], dtype=torch.float64)
    assert abs(float(G.gelu_tanh32(x.float()) / G.gelu64(x)) - 1) > 0.09
    assert abs(float(G.gelu_as32(x.float()) / G.gelu64(x)) - 1) < 1e-4


def test_forms():
    f = G.forms()
    assert len(f) == 2 * 2 * (8 + 4) and len(set(f)) == len(f)
    assert all(bn % 32 == 0 and mt * bn <= 256 for _, _, mt, bn in f)
    assert G.forms(512) == [(cg, kps, 1, 256) for cg in (1, 2) for kps in (1, 2)]
    assert len(G.forms(640)) == 8 and {bn for *_, bn in G.forms(640)} == {128}
    assert {bn for *_, bn in G.forms(320)} == {64} and len(G.forms(320)) == 8
    assert G.form_code(2, 1, 2) == 2 | 4 | 512
