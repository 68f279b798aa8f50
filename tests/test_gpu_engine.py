"""GPU: module-level and end-to-end parity of the engine against the oracle (fp32 torch restatement of diffusers)
with identical seeded weights and inputs.  Tiny same-topology configs keep the fp32 oracle cheap; the full-size
SSD-1B / SDXL checks run the oracle in fp32 on the GPU (torch is the checker, never the product path)."""
import math

import numpy as np
import pytest
import torch

from oracle import diffusion_oracle as O
from tests.util import rel_err

pytestmark = pytest.mark.gpu


def _nhwc(x):
    return x.permute(0, 2, 3, 1).contiguous()


def _nchw(x):
    return x.permute(0, 3, 1, 2).contiguous()


def _models(dev, lora=False, full_cn=False, mid_depth=1):
    from fast_image_editing_with_generative_models_b200 import synthetic as S
    ucfg = O.tiny_unet_config(mid_depth=mid_depth)
    ccfg = O.tiny_controlnet_config(full=full_cn)
    vcfg = O.tiny_vae_config()
    up, cp, vp = S.make_unet_params(ucfg), S.make_controlnet_params(ccfg), S.make_vae_params(vcfg)
    lp = S.make_lora_params(up, rank=8) if lora else None
    return ucfg, up, ccfg, cp, vcfg, vp, lp


def test_vae_encode_decode_tiny(cuda_dev):
    from fast_image_editing_with_generative_models_b200 import ops
    from fast_image_editing_with_generative_models_b200.engine import VAE
    from fast_image_editing_with_generative_models_b200.synthetic import synthetic_image
    ucfg, up, ccfg, cp, vcfg, vp, _ = _models(cuda_dev)
    vae = VAE(vp, vcfg, cuda_dev)
    img = torch.from_numpy(np.stack([synthetic_image(s, 256, 256) for s in range(2)])).to(cuda_dev)
    mom = vae.encode_moments(ops.preprocess_pad8(img, True))
    vp32 = O.to_dtype(vp, torch.float32, cuda_dev)
    ref = O.vae_encode_moments(vp32, vcfg, O.preprocess_image(img, torch.float32))
    err = float((_nchw(mom).float() - ref).abs().max())
    print("vae moments max-abs", err, "ref absmax", float(ref.abs().max()))
    assert err < 2e-2 * max(1.0, float(ref.abs().max()))
    z = torch.randn((2, 4, 32, 32), generator=torch.Generator().manual_seed(3)).to(cuda_dev)
    dec = vae.decode(_nhwc(z).half() * vcfg.scaling_factor)
    refd = O.vae_decode(vp32, vcfg, z.half().float())
    err = float((_nchw(dec)[:, :3].float() - refd).abs().max())
    print("vae decode max-abs", err, "ref absmax", float(refd.abs().max()))
    assert err < 3e-2 * max(1.0, float(refd.abs().max()))


@pytest.mark.parametrize("mid_depth,lora", [(1, False), (None, True)])
def test_unet_controlnet_merge_tiny(cuda_dev, mid_depth, lora):
    """The ControlNet residuals (its zero convolutions at scale 0.5) against the oracle's, and the UNet eps with those residuals merged
    by the zero-convolution GEMM epilogues (ControlNet.merge_into, the edit's path) against the oracle's UNet given the oracle's."""
    from fast_image_editing_with_generative_models_b200 import ops
    from fast_image_editing_with_generative_models_b200.engine import ControlNet, UNet
    ucfg, up, ccfg, cp, vcfg, vp, lp = _models(cuda_dev, lora=lora, full_cn=lora, mid_depth=mid_depth)
    unet = UNet(up, ucfg, cuda_dev, lp, 1.0)
    cn = ControlNet(cp, ccfg, cuda_dev)
    B, h = 2, 32
    g = torch.Generator().manual_seed(5)
    x = torch.randn((B, 4, h, h), generator=g).half().to(cuda_dev)
    ctx = torch.randn((B, 77, ucfg.cross_attention_dim), generator=g).half().to(cuda_dev)
    te = torch.randn((B, 64), generator=g).half().to(cuda_dev)
    cond = (torch.rand((B, 3, 8 * h, 8 * h), generator=g) > 0.9).half().to(cuda_dev)
    tids = [256.0, 256.0, 0.0, 0.0, 256.0, 256.0]
    t = 499.0
    ps_cn = cn.prepare_prompt(ctx, te, tids)
    ps_un = unet.prepare_prompt(ctx, te, tids)
    cond_p8 = torch.zeros((B, 8 * h + 2, 8 * h + 8, 8), dtype=torch.float16, device=cuda_dev)   # layout of ops.preprocess_pad8
    cond_p8[:, 1:-1, 1:8 * h + 1, :3] = _nhwc(cond)
    cemb = cn.cond_embedding(cond_p8)
    t_rows = torch.full((B,), t, dtype=torch.float32, device=cuda_dev)
    feats = cn.encode(_nhwc(x), t_rows, ps_cn, cemb)
    fh, fskips = feats
    down = [ops.gemm(f, w, col_bias=b, scale=0.5) for f, (w, b) in zip(fskips, cn.zero)]
    mid = ops.gemm(fh, cn.zero_mid[0], col_bias=cn.zero_mid[1], scale=0.5)
    eps = unet.forward(_nhwc(x), t_rows, ps_un, merge=cn.merge_into(feats, torch.full((B,), 0.5, dtype=torch.float32, device=cuda_dev)))
    # oracle, fp32 on the GPU
    up32, cp32 = O.to_dtype(up, torch.float32, cuda_dev), O.to_dtype(cp, torch.float32, cuda_dev)
    lora32 = O._LoRA(O.to_dtype(lp, torch.float32, cuda_dev), 1.0) if lp else None
    tid_t = torch.tensor(tids, device=cuda_dev)[None].expand(B, -1)
    tt = torch.tensor([t], device=cuda_dev)
    rcemb = O.controlnet_cond_embedding(cp32, ccfg, cond.float())
    print("cond-emb rel", rel_err(_nchw(cemb), rcemb))
    assert rel_err(_nchw(cemb), rcemb) < 1e-2
    rdown, rmid = O.controlnet_forward(cp32, ccfg, x.float(), tt, ctx.float(), te.float(), tid_t, cond.float(), 0.5)
    for i, (a, b) in enumerate(zip(down, rdown)):
        e = rel_err(_nchw(a), b)
        print("cn down", i, e)
        assert e < 2e-2
    assert rel_err(_nchw(mid), rmid) < 2e-2
    reps = O.unet_forward(up32, ucfg, x.float(), tt, ctx.float(), te.float(), tid_t, rdown, rmid, lora32)
    e = rel_err(_nchw(eps), reps)
    print("unet eps rel", e, "abs", float((_nchw(eps).float() - reps).abs().max()), "ref absmax", float(reps.abs().max()))
    assert e < 2e-2


def test_edit_pipeline_tiny(cuda_dev):
    """End-to-end: Canny bit-exact, final latents max-abs <= 2e-2, decoded SSIM >= 0.99 (BASELINE.json criteria)."""
    from fast_image_editing_with_generative_models_b200.pipeline import EditEngine
    from fast_image_editing_with_generative_models_b200.synthetic import synthetic_image, synthetic_noises
    from oracle.canny_oracle import preprocess_image as canny_ref
    ucfg, up, ccfg, cp, vcfg, vp, lp = _models(cuda_dev, lora=True)
    eng = EditEngine(up, ucfg, cp, ccfg, vp, vcfg, cuda_dev, lp, 1.0)
    B, H = 2, 256
    imgs = np.stack([synthetic_image(s, H, H) for s in range(B)])
    g = torch.Generator().manual_seed(9)
    pe = torch.randn((2, 77, ucfg.cross_attention_dim), generator=g).half()
    pl = torch.randn((2, 64), generator=g).half()
    noises = synthetic_noises(0, B, H // 8, H // 8)
    out = eng.edit_batch(torch.from_numpy(imgs).to(cuda_dev), pe, pl, noises, strength=0.5, return_extras=True)
    edges_ref = np.stack([canny_ref(i) for i in imgs])
    assert np.array_equal(out.edges.cpu().numpy(), edges_ref)
    m = O.EditModels(ucfg, O.to_dtype(up, torch.float32, cuda_dev), ccfg, O.to_dtype(cp, torch.float32, cuda_dev), vcfg,
                     O.to_dtype(vp, torch.float32, cuda_dev), O.to_dtype(lp, torch.float32, cuda_dev), 1.0)
    ref = O.edit_pipeline(m, torch.from_numpy(imgs).to(cuda_dev), torch.from_numpy(edges_ref).to(cuda_dev), pe.float().to(cuda_dev),
                          pl.float().to(cuda_dev), noises, strength=0.5, dtype=torch.float32, return_all=True)
    lat_err = float((_nchw(out.latents).float() - ref["latents"]).abs().max())
    print("latents max-abs", lat_err, "ref absmax", float(ref["latents"].abs().max()))
    assert lat_err <= 2e-2
    a = out.images.permute(0, 3, 1, 2).float() / 255.0
    b = ref["image_u8"].permute(0, 3, 1, 2).float() / 255.0
    s = O.ssim(a, b)
    print("ssim", s, "img std", float(b.std()))
    assert s >= 0.99
    # strength 0.8 executes 3 steps and consumes one more noise tensor
    out3 = eng.edit_batch(torch.from_numpy(imgs).to(cuda_dev), pe, pl, noises, strength=0.8, return_latents=True)
    ref3 = O.edit_pipeline(m, torch.from_numpy(imgs).to(cuda_dev), torch.from_numpy(edges_ref).to(cuda_dev), pe.float().to(cuda_dev),
                           pl.float().to(cuda_dev), noises, strength=0.8, dtype=torch.float32, return_all=True)
    assert float((_nchw(out3.latents).float() - ref3["latents"]).abs().max()) <= 2e-2


@pytest.mark.parametrize("strength,steps,guidance", [(1.0, 4, 1.5), (0.5, 4, 1.0), (0.6, 5, 2.0)])
def test_edit_pipeline_tiny_schedules(cuda_dev, strength, steps, guidance):
    """Other corners of the reference's `edit()` arguments: every step executed (strength 1.0: 4 steps, 5 noise tensors), no
    classifier-free guidance (guidance_scale <= 1: one UNet row per image, the pipeline's `do_cfg` gate), another step count."""
    from fast_image_editing_with_generative_models_b200.pipeline import EditEngine
    from fast_image_editing_with_generative_models_b200.synthetic import synthetic_image, synthetic_noises
    from oracle.canny_oracle import preprocess_image as canny_ref
    ucfg, up, ccfg, cp, vcfg, vp, lp = _models(cuda_dev, lora=False)
    eng = EditEngine(up, ucfg, cp, ccfg, vp, vcfg, cuda_dev, None, 1.0)
    B, H = 1, 256
    imgs = np.stack([synthetic_image(s + 3, H, H) for s in range(B)])
    g = torch.Generator().manual_seed(19)
    pe = torch.randn((2, 77, ucfg.cross_attention_dim), generator=g).half()
    pl = torch.randn((2, 64), generator=g).half()
    noises = synthetic_noises(1, B, H // 8, H // 8, count=2 + steps)
    out = eng.edit_batch(torch.from_numpy(imgs).to(cuda_dev), pe, pl, noises, strength=strength, num_inference_steps=steps,
                         guidance_scale=guidance, return_latents=True)
    edges_ref = np.stack([canny_ref(i) for i in imgs])
    m = O.EditModels(ucfg, O.to_dtype(up, torch.float32, cuda_dev), ccfg, O.to_dtype(cp, torch.float32, cuda_dev), vcfg,
                     O.to_dtype(vp, torch.float32, cuda_dev), None, 1.0)
    ref = O.edit_pipeline(m, torch.from_numpy(imgs).to(cuda_dev), torch.from_numpy(edges_ref).to(cuda_dev), pe.float().to(cuda_dev),
                          pl.float().to(cuda_dev), noises, strength=strength, num_inference_steps=steps, guidance_scale=guidance,
                          dtype=torch.float32, return_all=True)
    err = float((_nchw(out.latents).float() - ref["latents"]).abs().max())
    # noise floor: torch's own fp16 execution of the same modules against the fp32 oracle.  At strength 1.0 the first step runs at
    # t = 999 where x0 = (x - sqrt(1 - abar) eps) / sqrt(abar) divides by 0.068, so ANY fp16 evaluation of eps is amplified ~15x;
    # the 2e-2 criterion of BASELINE.json is stated for strength 0.5, beyond it the engine must stay at or below the fp16 floor.
    m16 = O.EditModels(ucfg, O.to_dtype(up, torch.float16, cuda_dev), ccfg, O.to_dtype(cp, torch.float16, cuda_dev), vcfg,
                       O.to_dtype(vp, torch.float16, cuda_dev), None, 1.0)
    ref16 = O.edit_pipeline(m16, torch.from_numpy(imgs).to(cuda_dev), torch.from_numpy(edges_ref).to(cuda_dev), pe.to(cuda_dev),
                            pl.to(cuda_dev), noises, strength=strength, num_inference_steps=steps, guidance_scale=guidance,
                            dtype=torch.float16, return_all=True)
    floor = float((ref16["latents"].float() - ref["latents"]).abs().max())
    print("strength", strength, "steps", steps, "guidance", guidance, "latents max-abs", err, "torch-fp16 floor", floor)
    assert err <= max(2e-2, 1.25 * floor)
    assert O.ssim(out.images.permute(0, 3, 1, 2).float() / 255.0, ref["image_u8"].permute(0, 3, 1, 2).float() / 255.0) >= 0.99


def test_edit_graph_replay_matches_eager(cuda_dev):
    """The whole edit replayed as one CUDA graph gives the eager result (up to the fp32 atomics of the GroupNorm statistics),
    for fresh inputs copied into the graph's static buffers, and keeps counting its kernel launches."""
    from fast_image_editing_with_generative_models_b200 import model_zoo, ops
    from fast_image_editing_with_generative_models_b200 import synthetic as S
    state = model_zoo.synthetic_state("sdxl", tiny=True)
    eng = model_zoo.build_engine(state, cuda_dev)
    ucfg = state["unet_cfg"]
    B, H = 2, 256
    pe, pl = S.synthetic_prompt(0, ucfg.cross_attention_dim, ucfg.projection_class_embeddings_input_dim - 6 * ucfg.addition_time_embed_dim)
    outs = []
    for seed in (0, 7):
        imgs = torch.from_numpy(np.stack([S.synthetic_image(seed + s, H, H) for s in range(B)])).to(cuda_dev)
        noises = S.synthetic_noises(seed, B, H // 8, H // 8)
        eager = eng.edit_batch(imgs, pe, pl, noises, strength=0.5, return_latents=True, use_graph=False)
        l0 = ops.LAUNCHES
        graphed = eng.edit_batch(imgs, pe, pl, noises, strength=0.5, return_latents=True, use_graph=True)
        assert ops.LAUNCHES - l0 > 100
        assert torch.equal(graphed.edges, eager.edges)
        assert float((graphed.latents.float() - eager.latents.float()).abs().max()) <= 2e-2   # run-to-run spread of the atomics alone is ~8e-3
        assert int((graphed.images.int() - eager.images.int()).abs().max()) <= 3
        outs.append(graphed.images.clone())
    assert len(eng._graphs) == 1 and not torch.equal(outs[0], outs[1])
