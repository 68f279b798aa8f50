"""GPU: LoRA adapters on a built editor (``editor.pipe.load_lora_weights`` / ``set_adapters`` / ``unload_lora_weights``, lora.py) —
exact restore, agreement with a load-time fuse and with the fp32 oracle, CUDA-graph validity, untouched buffers, the text encoders
and the CLIs."""
import math

import numpy as np
import pytest
import torch
from PIL import Image

from oracle import diffusion_oracle as O
from tests.util import rel_err

pytestmark = pytest.mark.gpu

H = 256


def _tensors(obj, path="", out=None, seen=None):
    """Every tensor reachable from an engine object -> {path: tensor}."""
    out = {} if out is None else out
    seen = set() if seen is None else seen
    if isinstance(obj, torch.Tensor):
        out.setdefault(path, obj)
    elif isinstance(obj, (list, tuple)):
        for i, v in enumerate(obj):
            _tensors(v, f"{path}[{i}]", out, seen)
    elif isinstance(obj, dict):
        for k, v in obj.items():
            _tensors(v, f"{path}.{k}", out, seen)
    elif hasattr(obj, "__dict__") and type(obj).__module__.startswith("fast_image_editing") and id(obj) not in seen:
        seen.add(id(obj))
        for k, v in vars(obj).items():
            _tensors(v, f"{path}.{k}", out, seen)
    return out


def _snapshot(eng):
    return {k: t.clone() for k, t in _tensors({"unet": eng.unet, "cn": eng.cn, "vae": eng.vae}).items()}


def _bytes(t):
    return t.contiguous().reshape(-1).view(torch.uint8)


def _changed(eng, snap):
    """Paths of the tensors whose bytes differ from the snapshot."""
    now = _tensors({"unet": eng.unet, "cn": eng.cn, "vae": eng.vae})
    return {k for k, t in now.items() if not torch.equal(_bytes(t), _bytes(snap[k]))}


def _style(unet_params, rank=4, seed=40, conv_in=True, conv_out=True):
    """A synthetic style adapter on every LoRA target (and on conv_in and conv_out: the hi/lo and row-padded layouts; the oracle's
    _LoRA adapts neither)."""
    from fast_image_editing_with_generative_models_b200 import synthetic as S
    sd = S.make_lora_params(unet_params, rank=rank, seed=seed, b_scale=0.05)
    g = torch.Generator().manual_seed(seed + 1)
    for name in (["conv_in"] if conv_in else []) + (["conv_out"] if conv_out else []):
        w = unet_params[name + ".weight"]
        sd[name + ".lora_A.weight"] = torch.randn((rank, w.shape[1], 3, 3), generator=g) / math.sqrt(9 * w.shape[1])
        sd[name + ".lora_B.weight"] = torch.randn((w.shape[0], rank, 1, 1), generator=g) * 0.02
    return sd


def _combined(base, style, w_base=1.0, w_style=1.0):
    """Two peft dicts as one of rank r1 + r2 (B columns scaled by the weights): what a load-time fuse of both gives."""
    out = {}
    for k in set(base or {}) | set(style):
        if not k.endswith(".lora_A.weight"):
            continue
        m = k[: -len(".lora_A.weight")]
        parts = [(w, d[m + ".lora_A.weight"], d[m + ".lora_B.weight"]) for w, d in ((w_base, base or {}), (w_style, style)) if m + ".lora_A.weight" in d]
        out[k] = torch.cat([a for _, a, _ in parts], 0)
        out[m + ".lora_B.weight"] = torch.cat([w * b for w, _, b in parts], 1)
    return out


def _editor(model="sdxl", state=None):
    from src.pipeline import FastEditor
    return FastEditor(model_name=model, device="cuda", tiny=True, verbose=False, state=state)


def _images(n=2):
    from fast_image_editing_with_generative_models_b200.synthetic import synthetic_image
    return [Image.fromarray(synthetic_image(s + 11, H, H)) for s in range(n)]


def _edit(ed, seeds=(1, 2)):
    out = ed.edit_many(_images(len(seeds)), "a watercolor", seeds=list(seeds), size=(H, H), micro_batch=len(seeds))
    return np.stack([np.array(o) for o in out])


@pytest.fixture(scope="module")
def sdxl_state():
    from fast_image_editing_with_generative_models_b200 import model_zoo
    return model_zoo.synthetic_state("sdxl", tiny=True)


def test_exact_restore_and_only_adapted_buffers_change(cuda_dev, sdxl_state):
    ed = _editor(state=sdxl_state)
    eng = ed._engine
    snap = _snapshot(eng)
    before = _edit(ed)
    style = {k: v for k, v in _style(sdxl_state["unet"], conv_in=False).items() if ".attentions." in k}
    ed.pipe.load_lora_weights(style, adapter_name="style")
    assert ed.get_active_adapters() == ["default_0", "style"] and ed.get_memory_usage()["lora_pristine_gb"] > 0
    # only the packed buffers of the adapted modules changed: no resnet, no ControlNet, no VAE tensor
    changed = _changed(eng, snap)
    targets = eng.unet.lora_targets()
    adapted = {id(t) for m, tg in targets.items() if m + ".lora_A.weight" in style for t in (tg.weight, tg.bias) if t is not None}
    paths = _tensors({"unet": eng.unet, "cn": eng.cn, "vae": eng.vae})
    assert changed and all(id(paths[k]) in adapted for k in changed), sorted(changed)[:5]
    assert not any(k.startswith((".cn", ".vae")) for k in changed)
    with_style = _edit(ed)
    assert not np.array_equal(with_style, before)
    for ws in ([1.0, 0.5], [0.3, 2.0], [0.0, 1.0]):
        ed.pipe.set_adapters(["default_0", "style"], ws)
    ed.pipe.set_adapters(["default_0", "style"], [1.0, 0.0])                 # the set the editor was built with
    assert not _changed(eng, snap) and ed.get_memory_usage()["lora_pristine_gb"] == 0
    assert np.array_equal(_edit(ed), before)
    ed.pipe.set_adapters(["style"], [0.7])
    ed.pipe.unload_lora_weights()
    assert not _changed(eng, snap) and ed.get_active_adapters() == ["default_0"]
    assert np.array_equal(_edit(ed), before)


def _module_rows(t, buf):
    if t.kind in ("up2x", "c8") or t.perm is not None:
        return buf
    return buf[t.row0:t.row0 + t.out]


def _ulp16(x):
    a = x.float().abs().clamp_min(2.0 ** -14)
    return torch.exp2(torch.floor(torch.log2(a)) - 10)


def test_matches_a_load_time_fuse(cuda_dev, sdxl_state):
    """LCM-LoRA + style fused at load vs loaded on the built engine: packed weights within 1 fp16 ulp of the larger magnitude of the
    weight before and after the change (the built weight is already rounded once, so where the delta cancels it the result can differ
    by half an ulp of the built weight), latents within 2e-2."""
    from fast_image_editing_with_generative_models_b200 import model_zoo
    from fast_image_editing_with_generative_models_b200 import synthetic as S
    from fast_image_editing_with_generative_models_b200.weights import unpack_conv3x3_c8
    style = _style(sdxl_state["unet"])
    ref = model_zoo.build_engine(dict(sdxl_state, lora=_combined(sdxl_state["lora"], style, 1.0, 0.6)), cuda_dev)
    ed = _editor(state=sdxl_state)
    ed.pipe.load_lora_weights({"unet." + k: v for k, v in style.items()}, adapter_name="style")
    ed.pipe.set_adapters(["default_0", "style"], [1.0, 0.6])
    got_t, ref_t = ed._engine.unet.lora_targets(), ref.unet.lora_targets()
    for m, t in got_t.items():
        r = ref_t[m]
        if t.kind == "c8":
            a, b = unpack_conv3x3_c8(t.weight, t.out, t.inp), unpack_conv3x3_c8(r.weight, r.out, r.inp)
            assert float((a - b).abs().max()) <= 2.0 ** -18 * float(b.abs().max()), m
            continue
        a, b = _module_rows(t, t.weight).float(), _module_rows(r, r.weight).float()
        if t.weight.data_ptr() not in ed.pipe.adapters._pristine:            # not adapted (the embeddings' linears): as built
            assert torch.equal(a, b), m
            continue
        p = _module_rows(t, ed.pipe.adapters._pristine[t.weight.data_ptr()]).float()
        err = (a - b).abs() / _ulp16(torch.maximum(torch.maximum(a.abs(), b.abs()), p.abs()))
        assert float(err.max()) <= 1.0, (m, float(err.max()))
        if t.bias is not None:
            assert rel_err(_module_rows(t, t.bias), _module_rows(r, r.bias)) < 1e-5, m
    ucfg = sdxl_state["unet_cfg"]
    pe, pl = S.synthetic_prompt(0, ucfg.cross_attention_dim, ucfg.projection_class_embeddings_input_dim - 6 * ucfg.addition_time_embed_dim)
    imgs = torch.from_numpy(np.stack([np.array(i) for i in _images()])).to(cuda_dev)
    noises = S.synthetic_noises(0, 2, H // 8, H // 8)
    a = ed._engine.edit_batch(imgs, pe, pl, noises, strength=0.5, return_latents=True, use_graph=False)
    b = ref.edit_batch(imgs, pe, pl, noises, strength=0.5, return_latents=True, use_graph=False)
    err = float((a.latents.float() - b.latents.float()).abs().max())
    print("load-time fuse vs adapter: latents max-abs", err)
    assert err <= 2e-2


def _oracle_case(dev, ed, state, style_lora, w_style, strength=0.5, n=1, size=H):
    """Engine with the adapter loaded vs the unfused fp32 oracle (_LoRA) with the combined dict; also torch fp16 on the same modules."""
    from fast_image_editing_with_generative_models_b200 import synthetic as S
    from oracle.canny_oracle import preprocess_image as canny_ref
    ucfg = state["unet_cfg"]
    comb = _combined(state["lora"], style_lora, 1.0, w_style)
    imgs = np.stack([S.synthetic_image(s + 5, size, size) for s in range(n)])
    pe, pl = S.synthetic_prompt(3, ucfg.cross_attention_dim, ucfg.projection_class_embeddings_input_dim - 6 * ucfg.addition_time_embed_dim)
    noises = S.synthetic_noises(4, n, size // 8, size // 8)
    out = ed._engine.edit_batch(torch.from_numpy(imgs).to(dev), pe, pl, noises, strength=strength, return_latents=True, use_graph=False)
    edges = torch.from_numpy(np.stack([canny_ref(i) for i in imgs])).to(dev)
    res = {}
    for dt in (torch.float32, torch.float16):
        m = O.EditModels(ucfg, O.to_dtype(state["unet"], dt, dev), state["cn_cfg"], O.to_dtype(state["cn"], dt, dev), state["vae_cfg"],
                         O.to_dtype(state["vae"], dt, dev), O.to_dtype(comb, dt, dev), 1.0)
        with torch.no_grad():
            res[dt] = O.edit_pipeline(m, torch.from_numpy(imgs).to(dev), edges, pe.to(dev, dt), pl.to(dev, dt), noises, strength=strength,
                                      dtype=dt, return_all=True)
    ref = res[torch.float32]
    err = float((out.latents.permute(0, 3, 1, 2).float() - ref["latents"]).abs().max())
    floor = float((res[torch.float16]["latents"].float() - ref["latents"]).abs().max())
    ssim = O.ssim(out.images.permute(0, 3, 1, 2).float() / 255.0, ref["image_u8"].permute(0, 3, 1, 2).float() / 255.0)
    print("latents max-abs", err, "torch-fp16 floor", floor, "ssim", ssim)
    assert err <= 2e-2 and err <= floor and ssim >= 0.99                    # BASELINE's bound, and no worse than torch fp16


@pytest.mark.parametrize("model", ["sdxl", "ssd-1b"])
def test_matches_the_fp32_oracle_tiny(cuda_dev, model):
    from fast_image_editing_with_generative_models_b200 import model_zoo
    state = model_zoo.synthetic_state(model, tiny=True)
    ed = _editor(model, state=state)
    assert ed.get_active_adapters() == (["default_0"] if model == "sdxl" else [])
    style = _style(state["unet"], rank=8, conv_in=False, conv_out=False)
    ed.pipe.load_lora_weights(style, adapter_name="style")
    ed.pipe.set_adapters((["default_0"] if model == "sdxl" else []) + ["style"], ([1.0] if model == "sdxl" else []) + [0.5])
    _oracle_case(cuda_dev, ed, state, style, 0.5)


def test_matches_the_fp32_oracle_sdxl_1024(cuda_dev):
    """Full-size SDXL, one 1024^2 image, a synthetic rank-64 style adapter at strength 0.5."""
    from fast_image_editing_with_generative_models_b200 import model_zoo
    from src.pipeline import FastEditor
    state = model_zoo.synthetic_state("sdxl")
    ed = FastEditor(model_name="sdxl", device="cuda", verbose=False, state=state)
    style = _style(state["unet"], rank=64, seed=60, conv_in=False, conv_out=False)
    ed.pipe.load_lora_weights(style, adapter_name="style")
    ed.pipe.set_adapters(["default_0", "style"], [1.0, 0.5])
    _oracle_case(cuda_dev, ed, state, style, 0.5, size=1024)


def test_graphs_stay_valid_across_adapter_changes(cuda_dev, sdxl_state):
    ed = _editor(state=sdxl_state)
    ed.warm_up(2, size=(H, H))
    graphs = {k: id(v["graph"]) for k, v in ed._engine._graphs.items()}
    assert graphs
    a0 = _edit(ed)
    ed.pipe.load_lora_weights(_style(sdxl_state["unet"]), adapter_name="style")
    ed.pipe.load_lora_weights(_style(sdxl_state["unet"], seed=77), adapter_name="other")
    ed.pipe.set_adapters(["default_0", "style"], [1.0, 0.8])
    a1 = _edit(ed)
    assert {k: id(v["graph"]) for k, v in ed._engine._graphs.items()} == graphs     # no new capture, the same graph objects
    ed._engine.use_graphs = False
    assert np.array_equal(_edit(ed), a1)                                     # replay == eager with the same adapters
    ed._engine.use_graphs = True
    ed.pipe.set_adapters(["default_0", "other"], [0.5, 1.0])
    a2 = _edit(ed)
    ed.pipe.set_adapters(["default_0", "style"], [1.0, 0.8])
    assert np.array_equal(_edit(ed), a1) and not np.array_equal(a1, a2) and not np.array_equal(a1, a0)
    ed.pipe.set_adapters(["default_0", "other"], [0.5, 1.0])
    assert np.array_equal(_edit(ed), a2)
    assert {k: id(v["graph"]) for k, v in ed._engine._graphs.items()} == graphs


def _tiny_towers(dev):
    from fast_image_editing_with_generative_models_b200 import text_encoder as T
    c1 = T.CLIPTextConfig(name="t1", vocab_size=1000, hidden_size=64, num_layers=2, num_heads=1, intermediate_size=128, seed=41)
    c2 = T.CLIPTextConfig(name="t2", vocab_size=1000, hidden_size=64, num_layers=2, num_heads=1, intermediate_size=128, hidden_act="gelu",
                          projection_dim=64, seed=42)
    return c1, T.make_clip_params(c1), c2, T.make_clip_params(c2)


def test_text_encoder_adapters_and_prompt_cache(cuda_dev, sdxl_state):
    from fast_image_editing_with_generative_models_b200 import text_encoder as T
    c1, p1, c2, p2 = _tiny_towers(cuda_dev)
    ed = _editor(state=sdxl_state)
    ed._text, ed._text_vocab = T.SDXLTextEncoders(p1, c1, p2, c2, cuda_dev), 1000      # the GPU towers, as a checkpoint folder gives them
    e0 = [t.clone() for t in ed._encode_prompt("a red fox", "")]
    g = torch.Generator().manual_seed(90)
    sd, fused = {}, ({k: v.clone() for k, v in p1.items()}, {k: v.clone() for k, v in p2.items()})
    for te, params, p in (("lora_te1_", fused[0], p1), ("lora_te2_", fused[1], p2)):
        for m in ("text_model.encoder.layers.0.self_attn.q_proj", "text_model.encoder.layers.1.self_attn.v_proj", "text_model.encoder.layers.1.mlp.fc1",
                  "text_model.encoder.layers.0.mlp.fc2") + (("text_projection",) if te == "lora_te2_" else ()):
            w = p[m + ".weight"]
            down = torch.randn((4, w.shape[1]), generator=g) / math.sqrt(w.shape[1])
            up = torch.randn((w.shape[0], 4), generator=g) * 0.05
            flat = te + m.replace(".", "_")
            sd[flat + ".lora_down.weight"], sd[flat + ".lora_up.weight"], sd[flat + ".alpha"] = down, up, torch.tensor(2.0)
            params[m + ".weight"] = w + 0.5 * up @ down
    ed.pipe.load_lora_weights(sd, adapter_name="te_style")
    assert ed.get_list_adapters() == {"unet": ["default_0"], "text_encoder": ["te_style"], "text_encoder_2": ["te_style"]}
    e1 = ed._encode_prompt("a red fox", "")                                   # same string: the cache was cleared
    ref = T.SDXLTextEncoders(fused[0], c1, fused[1], c2, cuda_dev)
    ids = torch.stack([T.pseudo_token_ids("", 1000), T.pseudo_token_ids("a red fox", 1000)])
    r = ref.encode(ids, ids)
    for got, want, old in zip(e1, r, e0):
        print("text-encoder adapter: rel err", rel_err(got, want), "change", rel_err(old, want))
        assert rel_err(got, want) < 5e-3 and not torch.equal(got, old)
    ed.pipe.unload_lora_weights()
    assert all(torch.equal(a, b) for a, b in zip(ed._encode_prompt("a red fox", ""), e0))


def test_clis_take_lora(cuda_dev, tmp_path, monkeypatch, sdxl_state):
    import json

    from safetensors.torch import save_file
    monkeypatch.setenv("FIE_TINY", "1")
    import run_batch
    import run_single_image
    lora = tmp_path / "style.safetensors"
    save_file({"unet." + k: v.contiguous() for k, v in _style(sdxl_state["unet"], rank=8).items()}, str(lora))
    src = tmp_path / "src" / "0_random"
    src.mkdir(parents=True)
    _images(1)[0].save(src / "000000000000.jpg")
    mf = tmp_path / "mapping_file.json"
    mf.write_text(json.dumps({"000000000000": {"image_path": "0_random/000000000000.jpg", "original_prompt": "a photo", "editing_prompt": "a painting", "editing_type_id": "0"}}))
    outs = {}
    for tag, extra in (("plain", []), ("lora", ["--lora", f"{lora}=0.7"])):
        out = tmp_path / tag
        run_single_image.main(["--image", str(src / "000000000000.jpg"), "--prompt", "a painting", "--seed", "7", "--output_dir", str(out),
                               "--no_cpu_offload"] + extra)
        run_batch.main(["--mapping_file", str(mf), "--source_dir", str(tmp_path / "src"), "--output_dir", str(out), "--seed", "7",
                        "--no_cpu_offload", "--size", "256x256"] + extra)
        single = next((out / "single" / "edited").rglob("edited_*.jpg"))
        batch = next(p for p in out.rglob("0_random/*.jpg") if "single" not in str(p))
        outs[tag] = (np.array(Image.open(single)), np.array(Image.open(batch)))
    for a, b in zip(outs["plain"], outs["lora"]):
        assert a.shape == b.shape and not np.array_equal(a, b)
