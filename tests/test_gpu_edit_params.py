"""GPU: per-image edit settings read from device memory -- the kernels' batched calls against one-image calls, cv2 and a
float64 reference, and the engine: per-image results independent of the other images' settings, one CUDA graph for every setting of
one (size, executed steps, CFG), edit_many's grouping and staging."""
import cv2
import numpy as np
import pytest
import torch

from oracle import diffusion_oracle as O
from tests import gemm_cases as G

pytestmark = pytest.mark.gpu


# ------------------------------------------------------------------ kernels
def test_sincos_from_device_equals_host_form(cuda_dev):
    from fast_image_editing_with_generative_models_b200 import ops
    vals = [999.0, 759.0, 499.0, 259.0, 139.0, 19.0, 0.0, 1.5, 1024.0, 123.456]
    dev = torch.tensor(vals * 20, dtype=torch.float32, device=cuda_dev)            # 200 rows: beyond the host form's 64
    for dim in (320, 256):
        got = ops.sincos_embedding(dev, dim, cuda_dev)
        for r0 in range(0, 200, 50):
            ref = ops.sincos_embedding(dev[r0:r0 + 50].tolist(), dim, cuda_dev)
            assert torch.equal(got[r0:r0 + 50].view(torch.int16), ref.view(torch.int16))


def test_cfg_lcm_and_vae_sample_per_image_equal_one_image_calls(cuda_dev):
    from fast_image_editing_with_generative_models_b200 import ops
    from fast_image_editing_with_generative_models_b200.scheduler import LCMSchedule
    g = torch.Generator().manual_seed(5)
    B, h, w = 4, 16, 24
    mom = torch.randn((B, h, w, 8), generator=g).half().to(cuda_dev)
    xi, nz = (torch.randn((B, h, w, 4), generator=g).half().to(cuda_dev) for _ in range(2))
    steps, strengths, guidance = [4, 8, 5, 4], [0.5, 0.25, 0.4, 0.5], [1.5, 2.25, 1.0, 7.5]
    ts, add, table = LCMSchedule().batch_tables(steps, strengths, guidance)
    add = torch.from_numpy(add).to(cuda_dev)
    x32, x16 = ops.vae_sample_add_noise(mom, xi, nz, 0.13025, add)
    for i in range(B):
        r32, r16 = ops.vae_sample_add_noise(mom[i:i + 1], xi[i:i + 1], nz[i:i + 1], 0.13025, add[i:i + 1])
        assert torch.equal(x32[i:i + 1], r32) and torch.equal(x16[i:i + 1].view(torch.int16), r16.view(torch.int16))
    eps = torch.randn((2 * B, h, w, 8), generator=g).half().to(cuda_dev)[..., :4]
    tab = torch.from_numpy(table).to(cuda_dev)
    for k in range(table.shape[0]):
        last = k == table.shape[0] - 1
        y32, y16 = ops.cfg_lcm_step(eps[:B], eps[B:], x32, None if last else nz, tab[k], last)
        for i in range(B):
            r32, r16 = ops.cfg_lcm_step(eps[i:i + 1], eps[B + i:B + i + 1], x32[i:i + 1].contiguous(), None if last else nz[i:i + 1],
                                        tab[k, i:i + 1], last)
            assert torch.equal(y32[i:i + 1], r32) and torch.equal(y16[i:i + 1].view(torch.int16), r16.view(torch.int16))
        x32 = y32


@pytest.mark.parametrize("h,w", [(256, 256), (200, 264)])           # the four-pixel fast tile kernel, and the generic k_nms<3>
def test_canny_per_image_thresholds_equal_cv2(cuda_dev, h, w):
    from fast_image_editing_with_generative_models_b200 import ops
    from fast_image_editing_with_generative_models_b200.synthetic import synthetic_image
    pairs = [(100, 200), (200, 100), (-5, 5000), (-1, 30), (3000, 4000), (50.7, 120.2)]
    imgs = np.stack([synthetic_image(s, h, w, kind="noise" if s % 2 else "shapes") for s in range(len(pairs))])
    thr = torch.tensor([ops.canny_thresholds(*p) for p in pairs], dtype=torch.int32, device=cuda_dev)
    got = ops.canny(torch.from_numpy(imgs).to(cuda_dev), out_channels=1, thresholds=thr).cpu().numpy()
    for i, (lo, hi) in enumerate(pairs):
        ref = cv2.Canny(cv2.cvtColor(imgs[i], cv2.COLOR_RGB2GRAY), lo, hi)
        assert np.array_equal(got[i], ref), (i, lo, hi)


@pytest.mark.parametrize("m,n,k,out_dtype", [(1000, 320, 320, torch.float16), (1000, 320, 320, torch.float32), (1000, 80, 192, torch.float16),
                                             (768, 256, 128, torch.bfloat16), (768, 80, 128, torch.bfloat16)])
def test_gemm_group_scale_against_float64(cuda_dev, m, n, k, out_dtype):
    """group_scale replaces the scale per group of rows_per_group rows, before the residual add; fast epilogue path (fp16 / bf16 output,
    N % 32 == 0, aligned) and the out-of-line one (fp32 output with a residual, or the partial last chunk of N = 80)."""
    from fast_image_editing_with_generative_models_b200 import ops
    dtype = torch.bfloat16 if out_dtype == torch.bfloat16 else torch.float16
    rpg = 100
    a, w, ep = G.generic(m, n, k, seed=m + n, dtype=dtype, m_bias=False, residual=True, rows_per_group=rpg)
    ep = ep.to(cuda_dev)
    ep.row_bias = None
    gs = torch.linspace(0.1, 1.3, -(-m // rpg), dtype=torch.float32)
    a, w = a.to(cuda_dev), w.to(cuda_dev)
    kw = ep.kwargs()
    kw.pop("scale")
    out = ops.gemm(a, w, out_f32=out_dtype == torch.float32, out_dtype=out_dtype if dtype == torch.bfloat16 else None, group_scale=gs.to(cuda_dev), **kw)
    ref_ep = G.replace(ep, scale=1.0, residual=None)
    ref, tol = G.expected(a, w, ref_ep, out_dtype)
    srow = gs.double().to(cuda_dev)[torch.arange(m, device=cuda_dev) // rpg][:, None]
    ref, tol = ref * srow, tol * srow
    if ep.residual is not None:
        ref = ref + ep.residual.double()
        tol = tol + G.U_OUT[out_dtype] * ref.abs()
    assert G.err_ratio(out, ref, tol) <= 1.0
    # equal values: bit-identical to the scalar scale
    same = ops.gemm(a, w, out_f32=out_dtype == torch.float32, out_dtype=out_dtype if dtype == torch.bfloat16 else None,
                    group_scale=torch.full_like(gs, 0.75).to(cuda_dev), **kw)
    scalar = ops.gemm(a, w, out_f32=out_dtype == torch.float32, out_dtype=out_dtype if dtype == torch.bfloat16 else None, scale=0.75, **kw)
    assert torch.equal(same.view(torch.int16) if same.element_size() == 2 else same, scalar.view(torch.int16) if scalar.element_size() == 2 else scalar)


# ------------------------------------------------------------------ engine (tiny SDXL)
_TINY = {}


def _tiny(dev):
    from fast_image_editing_with_generative_models_b200 import model_zoo
    if "eng" not in _TINY:
        _TINY["state"] = model_zoo.synthetic_state("sdxl", tiny=True)
        _TINY["eng"] = model_zoo.build_engine(_TINY["state"], dev)
    return _TINY["state"], _TINY["eng"]


def _tiny_inputs(state, B, H=256, n_noise=4, seed=0):
    from fast_image_editing_with_generative_models_b200 import synthetic as S
    ucfg = state["unet_cfg"]
    imgs = torch.from_numpy(np.stack([S.synthetic_image(seed + s, H, H) for s in range(B)]))
    pe, pl = S.synthetic_prompt(seed, ucfg.cross_attention_dim, ucfg.projection_class_embeddings_input_dim - 6 * ucfg.addition_time_embed_dim)
    return imgs, pe, pl, S.synthetic_noises(seed, B, H // 8, H // 8, n_noise)


SETTINGS = [dict(guidance_scale=1.5, controlnet_conditioning_scale=0.5, canny_low=100, canny_high=200),
            dict(guidance_scale=2.5, controlnet_conditioning_scale=0.8, canny_low=50, canny_high=150),
            dict(guidance_scale=1.2, controlnet_conditioning_scale=0.3, canny_low=150, canny_high=80),
            dict(guidance_scale=4.0, controlnet_conditioning_scale=1.0, canny_low=20.5, canny_high=300)]


def _mixed(settings):
    return {k: [s[k] for s in settings] for k in settings[0]}


@pytest.mark.parametrize("use_graph", [False, True])
def test_engine_per_image_settings_equal_uniform_batches(cuda_dev, use_graph):
    """Image i of a batch with four distinct settings equals image i of a uniform batch (same images, same shape) run with image i's
    settings, bit for bit: per-image results depend only on that image's data at a fixed batch shape."""
    state, eng = _tiny(cuda_dev)
    imgs, pe, pl, noises = _tiny_inputs(state, 4)
    d = imgs.to(cuda_dev)
    mixed = eng.edit_batch(d, pe, pl, noises, strength=0.5, return_latents=True, use_graph=use_graph, **_mixed(SETTINGS))
    m_img, m_lat, m_edge = mixed.images.clone(), mixed.latents.clone(), mixed.edges.clone()
    for i, s in enumerate(SETTINGS):
        u = eng.edit_batch(d, pe, pl, noises, strength=0.5, return_latents=True, use_graph=use_graph, **s)
        assert torch.equal(u.edges[i], m_edge[i]), i
        assert torch.equal(u.latents[i], m_lat[i]), (i, float((u.latents[i] - m_lat[i]).abs().max()))
        assert torch.equal(u.images[i], m_img[i]), i


def test_engine_scalars_equal_lists_and_one_graph_for_every_setting(cuda_dev):
    from fast_image_editing_with_generative_models_b200 import ops
    state, eng = _tiny(cuda_dev)
    eng.release_graphs()
    imgs, pe, pl, noises = _tiny_inputs(state, 4, seed=3)
    d = imgs.to(cuda_dev)
    s = SETTINGS[1]
    a = eng.edit_batch(d, pe, pl, noises, strength=0.5, return_latents=True, use_graph=False, **s)
    a_lat, a_img = a.latents.clone(), a.images.clone()
    b = eng.edit_batch(d, pe, pl, noises, strength=[0.5] * 4, num_inference_steps=[4] * 4, return_latents=True, use_graph=False,
                       **{k: [v] * 4 for k, v in s.items()})
    assert torch.equal(a_lat, b.latents) and torch.equal(a_img, b.images)
    # >= 6 distinct scalar settings at one (size, n_exec, CFG): one capture; graph equals eager
    for j, (gs, cs, lo, hi) in enumerate([(1.5, 0.5, 100, 200), (2.0, 0.3, 80, 160), (2.5, 0.8, 120, 240), (3.0, 0.6, 60, 90),
                                         (1.8, 1.0, 100, 100), (4.0, 0.4, 10, 400)]):
        kw = dict(guidance_scale=gs, controlnet_conditioning_scale=cs, canny_low=lo, canny_high=hi)
        e = eng.edit_batch(d, pe, pl, noises, strength=0.5, return_latents=True, use_graph=False, **kw)
        e_lat, e_img = e.latents.clone(), e.images.clone()
        l0 = ops.LAUNCHES
        g = eng.edit_batch(d, pe, pl, noises, strength=0.5, return_latents=True, use_graph=True, **kw)
        assert ops.LAUNCHES - l0 > 100
        assert torch.equal(g.latents, e_lat) and torch.equal(g.images, e_img), j
    assert len(eng._graphs) == 1
    # a new executed step count, CFG off or another size: a new key
    eng.edit_batch(d, pe, pl, _tiny_inputs(state, 4, n_noise=5, seed=3)[3], strength=0.75, use_graph=True)
    assert len(eng._graphs) == 2
    eng.edit_batch(d, pe, pl, noises, strength=0.5, guidance_scale=1.0, use_graph=True)
    assert len(eng._graphs) == 3
    imgs2, _, _, noises2 = _tiny_inputs(state, 4, H=320, seed=3)
    eng.edit_batch(imgs2.to(cuda_dev), pe, pl, noises2, strength=0.5, use_graph=True)
    assert len(eng._graphs) == 4
    eng.release_graphs()


def test_engine_mixed_step_counts_against_oracle(cuda_dev):
    """(4 steps, strength 0.5) and (8 steps, strength 0.25) both execute 2 steps, at different timesteps: one batch, each image within
    2e-2 of the fp32 oracle run with its own arguments."""
    from oracle.canny_oracle import preprocess_image as canny_ref
    state, eng = _tiny(cuda_dev)
    imgs, pe, pl, noises = _tiny_inputs(state, 2, seed=5)
    args = [dict(strength=0.5, num_inference_steps=4), dict(strength=0.25, num_inference_steps=8)]
    out = eng.edit_batch(imgs.to(cuda_dev), pe, pl, noises, strength=[a["strength"] for a in args],
                         num_inference_steps=[a["num_inference_steps"] for a in args], return_latents=True, use_graph=False)
    f32 = lambda p: None if p is None else O.to_dtype(p, torch.float32, cuda_dev)
    m = O.EditModels(state["unet_cfg"], f32(state["unet"]), state["cn_cfg"], f32(state["cn"]), state["vae_cfg"], f32(state["vae"]), f32(state["lora"]), 1.0)
    for i, a in enumerate(args):
        edges = torch.from_numpy(canny_ref(imgs[i].numpy())[None]).to(cuda_dev)
        with torch.no_grad():
            ref = O.edit_pipeline(m, imgs[i:i + 1].to(cuda_dev), edges, pe.float().to(cuda_dev), pl.float().to(cuda_dev),
                                  [n[i:i + 1] for n in noises], dtype=torch.float32, return_all=True, **a)
        err = float((out.latents[i:i + 1].permute(0, 3, 1, 2).float() - ref["latents"]).abs().max())
        ssim = O.ssim(out.images[i:i + 1].permute(0, 3, 1, 2).float() / 255, ref["image_u8"].permute(0, 3, 1, 2).float() / 255)
        print(f"image {i} {a}: latents max-abs {err:.4g}, SSIM {ssim:.5f}")
        assert err <= 2e-2 and ssim >= 0.99


# ------------------------------------------------------------------ FastEditor.edit_many
def test_edit_many_per_image_settings_equal_per_setting_calls(cuda_dev):
    """Three micro-batches with distinct settings per image equal one call per setting (catches a parameter block overwritten while
    its copy is in flight), and guidance <= 1 / > 1 images are grouped apart."""
    from PIL import Image
    from fast_image_editing_with_generative_models_b200.editor import FastEditor
    from fast_image_editing_with_generative_models_b200.synthetic import synthetic_image
    ed = FastEditor("sdxl", tiny=True, verbose=False)
    n = 12
    ims = [Image.fromarray(synthetic_image(s, 256, 256)) for s in range(n)]
    gs = [1.5, 2.0, 0.8, 2.5, 1.0, 3.0, 0.9, 1.75, 0.5, 2.25, 1.0, 0.7]                 # six with CFG, six without: four micro-batches of 3
    cs = [0.3 + 0.07 * i for i in range(n)]
    lo = [60 + 10 * i for i in range(n)]
    hi = [150 + 15 * i for i in range(n)]
    kw = dict(strength=0.5, micro_batch=3, size=(256, 256))
    many = ed.edit_many(ims, "a prompt", guidance_scale=gs, controlnet_conditioning_scale=cs, canny_low_threshold=lo,
                        canny_high_threshold=hi, seeds=list(range(n)), **kw)
    assert len(ed._engine._graphs) == 2                                                  # (CFG on) and (CFG off)
    for i in range(n):
        solo = ed.edit_many([ims[i]] * 3, "a prompt", guidance_scale=gs[i], controlnet_conditioning_scale=cs[i], canny_low_threshold=lo[i],
                            canny_high_threshold=hi[i], seeds=[i] * 3, **kw)
        assert np.array_equal(np.array(many[i]), np.array(solo[0])), i
    assert len(ed._engine._graphs) == 2


# ------------------------------------------------------------------ full size
def test_sdxl_b8_distinct_settings_one_graph(cuda_dev):
    """SDXL 8 x 1024^2, eight distinct settings as one graph: graph equals eager; two images closer to the fp32 oracle run with their
    own arguments than torch's fp16 run of the oracle is (the noise floor of test_gpu_fullsize), and the one nearest BASELINE's guidance
    of 1.5 within its 2e-2.  (The CFG combine eps_u + g (eps_c - eps_u) amplifies eps differences by about 2g - 1: at g = 2.36 both the
    engine, 2.1e-2, and torch's fp16 run, 3.5e-2, exceed 2e-2.)"""
    from fast_image_editing_with_generative_models_b200 import model_zoo
    from fast_image_editing_with_generative_models_b200 import synthetic as S
    from oracle import c_oracle
    state = model_zoo.synthetic_state("sdxl")
    eng = model_zoo.build_engine(state, cuda_dev)
    B, H = 8, 1024
    imgs = np.stack([S.synthetic_image(s, H, H) for s in range(B)])
    ucfg = state["unet_cfg"]
    pe, pl = S.synthetic_prompt(0, ucfg.cross_attention_dim, ucfg.projection_class_embeddings_input_dim - 6 * ucfg.addition_time_embed_dim)
    noises = S.synthetic_noises(0, B, H // 8, H // 8, 4)
    gs = [1.5 + i / 7 for i in range(B)]
    cs = [0.3 + 0.5 * i / 7 for i in range(B)]
    lo = [80 + 5 * i for i in range(B)]
    hi = [180 + 10 * i for i in range(B)]
    kw = dict(strength=0.5, num_inference_steps=4, guidance_scale=gs, controlnet_conditioning_scale=cs, canny_low=lo, canny_high=hi,
              return_latents=True)
    d = torch.from_numpy(imgs).to(cuda_dev)
    eager = eng.edit_batch(d, pe, pl, noises, use_graph=False, **kw)
    e_lat, e_img = eager.latents.clone(), eager.images.clone()
    g = eng.edit_batch(d, pe, pl, noises, use_graph=True, **kw)
    assert len(eng._graphs) == 1
    assert torch.equal(g.latents, e_lat) and torch.equal(g.images, e_img)
    cast = lambda p, dt: None if p is None else O.to_dtype(p, dt, cuda_dev)
    for i in (1, 6):
        edges = torch.from_numpy(c_oracle.canny_u8(imgs[i:i + 1], lo[i], hi[i], replicate3=True)).to(cuda_dev)
        errs = {}
        for dt in (torch.float32, torch.float16):
            m = O.EditModels(ucfg, cast(state["unet"], dt), state["cn_cfg"], cast(state["cn"], dt), state["vae_cfg"], cast(state["vae"], dt),
                             cast(state["lora"], dt), 1.0)
            with torch.no_grad():
                ref = O.edit_pipeline(m, d[i:i + 1], edges, pe.to(cuda_dev, dt), pl.to(cuda_dev, dt), [n[i:i + 1] for n in noises], strength=0.5,
                                      guidance_scale=gs[i], controlnet_conditioning_scale=cs[i], dtype=dt, return_all=True)
            if dt == torch.float32:
                ref32 = ref["latents"]
                errs["engine"] = float((g.latents[i:i + 1].permute(0, 3, 1, 2).float() - ref32).abs().max())
                errs["ref_absmax"] = float(ref32.abs().max())
            else:
                errs["torch_fp16"] = float((ref["latents"].float() - ref32).abs().max())
            del m
        print(f"image {i}: latents max-abs vs fp32 oracle {errs}")
        assert errs["engine"] < errs["torch_fp16"]
        if gs[i] < 2.0:
            assert errs["engine"] <= 2e-2
