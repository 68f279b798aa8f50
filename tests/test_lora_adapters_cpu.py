"""CPU: runtime LoRA adapters (lora.py) — the factor algebra of every packed layout in float64, the key splitting of LoRA files into
UNet / text-encoder parts, and the adapter bookkeeping and its errors (no GPU: the device writes are recorded, not run)."""
import math

import pytest
import torch

from fast_image_editing_with_generative_models_b200 import checkpoints as K
from fast_image_editing_with_generative_models_b200 import configs as C
from fast_image_editing_with_generative_models_b200 import synthetic as S
from fast_image_editing_with_generative_models_b200 import text_encoder as T
from fast_image_editing_with_generative_models_b200 import weights as Wt
from fast_image_editing_with_generative_models_b200.lora import LoraAdapters

D = torch.float64


def _rand(*shape, seed=0):
    return torch.randn(shape, generator=torch.Generator().manual_seed(seed), dtype=D)


def _adapters(out, inp, taps=None):
    """Two adapters of ranks 3 and 5 with weights 0.7 and -1.3 -> (delta sum w_i B_i A_i, B' [out, 8], stacked A [8, inp(, 3, 3)])."""
    shp = (inp,) if taps is None else (inp, 3, 3)
    fs = [(0.7, _rand(3, *shp, seed=1), _rand(out, 3, seed=2)), (-1.3, _rand(5, *shp, seed=3), _rand(out, 5, seed=4))]
    delta = sum(w * (b @ a.reshape(a.shape[0], -1)) for w, a, b in fs).reshape(out, *shp)
    return delta, torch.cat([w * b for w, _, b in fs], 1), torch.cat([a for _, a, _ in fs], 0)


def _close(a, b):
    assert torch.allclose(a, b, rtol=1e-12, atol=1e-12), float((a - b).abs().max())


def test_fused_rows_take_the_delta_at_their_row_offsets():
    """Fused q/k/v, the concatenated cross-attention K/V and time_emb_proj matrices: each module's delta lands at its own rows."""
    ws = [_rand(6, 16, seed=10 + i) for i in range(3)]
    packed = torch.cat(ws, 0)
    delta, bp, a = _adapters(6, 16)
    ref = torch.cat([ws[0], ws[1] + delta, ws[2]], 0)
    got = packed.clone()
    got[6:12] += bp @ a
    _close(got, ref)


def test_layernorm_fold_factor_and_bias_delta():
    w, g, beta, b = _rand(12, 32, seed=5), 1 + 0.1 * _rand(32, seed=6), _rand(32, seed=7), _rand(12, seed=8)
    delta, bp, a = _adapters(12, 32)

    def fold(w_):                     # weights.fold_layernorm's CPU arithmetic, kept in float64
        return Wt._centre_rows(w_ * g[None, :]), b + w_ @ beta
    (w0, b0), (w1, b1) = fold(w), fold(w + delta)
    a2, ab = Wt.fold_layernorm_lora(a, g, beta)
    _close(w1, w0 + bp @ a2)
    _close(b1, b0 + bp @ ab)
    assert Wt.fold_layernorm_lora(a, g, None)[1] is None


def test_geglu_interleave_permutes_the_rows_of_b():
    c = 64
    w, g, beta = _rand(8 * c, c, seed=9), 1 + 0.1 * _rand(c, seed=10), _rand(c, seed=11)
    delta, bp, a = _adapters(8 * c, c)
    perm = Wt.geglu_rows(8 * c)
    a2, ab = Wt.fold_layernorm_lora(a, g, beta)
    fold = lambda w_: Wt._centre_rows(w_ * g[None, :])
    _close(fold(w + delta)[perm], fold(w)[perm] + bp[perm] @ a2)
    _close(((w + delta) @ beta)[perm], (w @ beta)[perm] + bp[perm] @ ab)
    # the packer uses the same order
    w16, _ = Wt.pack_geglu(w.float(), None)
    assert torch.equal(w16, w.float()[perm])


@pytest.mark.parametrize("pad", [(None, None), (32, 24)])
def test_conv3x3_layout_factor(pad):
    w = _rand(20, 16, 3, 3, seed=12)
    delta, bp, a = _adapters(20, 16, taps=True)
    got = Wt.conv3x3_layout(w, *pad)
    got[:20] += bp @ Wt.conv3x3_layout(a, pad_cin_to=pad[1])
    _close(got, Wt.conv3x3_layout(w + delta, *pad))
    assert torch.equal(Wt.pack_conv3x3(w.float(), *pad), Wt.conv3x3_layout(w.float(), *pad).half())


def test_upsample_phase_filters_factor():
    w = _rand(12, 8, 3, 3, seed=13)
    delta, bp, a = _adapters(12, 8, taps=True)
    base, a4, ref = Wt.conv_up2x_layout(w), Wt.conv_up2x_layout(a), Wt.conv_up2x_layout(w + delta)
    assert a4.shape == (4, 8, 32)
    for p in range(4):
        _close(base[p] + bp @ a4[p], ref[p])
    assert torch.equal(Wt.pack_conv_up2x(w.float()), Wt.conv_up2x_layout(w.float()).half())


def test_conv_in_hi_lo_pair_unpacks_to_the_fp32_weight():
    w = _rand(64, 4, 3, 3, seed=14).float() * 0.3
    packed = Wt.pack_conv3x3_c8(w)
    back = Wt.unpack_conv3x3_c8(packed, 64, 4)
    assert float((back - w).abs().max()) <= 2.0 ** -20 * float(w.abs().max())
    delta, bp, a = _adapters(64, 4, taps=True)
    again = Wt.unpack_conv3x3_c8(Wt.pack_conv3x3_c8(back + delta.float()), 64, 4)      # what a delta on conv_in does
    assert float((again - (w + delta.float())).abs().max()) <= 2.0 ** -19 * float((w + delta.float()).abs().max())


# ---- key splitting ------------------------------------------------------------------------------------------------------------

def _tiny_clip(proj):
    return T.tiny_clip_config(proj, "gelu" if proj else "quick_gelu")


def test_lora_file_splits_into_unet_and_text_encoder_parts():
    unet = S.make_unet_params(C.tiny_unet_config())
    p1, p2 = T.make_clip_params(_tiny_clip(False)), T.make_clip_params(_tiny_clip(True))
    um = "down_blocks.1.attentions.0.proj_in"
    tm = "text_model.encoder.layers.1.self_attn.k_proj"
    a, b = _rand(4, 128).float(), _rand(128, 4).float()
    sd = {}
    for kohya, peft, m in (("lora_unet_", "unet.", um), ("lora_te1_", "text_encoder.", tm), ("lora_te2_", "text_encoder_2.", tm)):
        flat = kohya + m.replace(".", "_")
        sd[flat + ".lora_down.weight"], sd[flat + ".lora_up.weight"], sd[flat + ".alpha"] = a, b, torch.tensor(2.0)
        mp = m.replace("proj_in", "proj_out").replace("k_proj", "v_proj")
        sd[peft + mp + ".lora_A.weight"], sd[peft + mp + ".lora_B.weight"] = a, b
    parts = K.split_lora(sd)
    assert sorted(parts) == ["text_encoder", "text_encoder_2", "unet"] and all(len(p) == 5 for p in parts.values())
    for part, names in (("unet", list(unet)), ("text_encoder", list(p1)), ("text_encoder_2", list(p2))):
        got = K.lora_to_peft(parts[part], names, part)
        m = um if part == "unet" else tm
        mp = m.replace("proj_in", "proj_out").replace("k_proj", "v_proj")
        assert sorted(got) == sorted([m + ".lora_A.weight", m + ".lora_B.weight", mp + ".lora_A.weight", mp + ".lora_B.weight"])
        assert torch.equal(got[m + ".lora_B.weight"], b * 0.5) and torch.equal(got[mp + ".lora_B.weight"], b)
    # keys with no part prefix stay UNet keys (a peft file saved from a bare UNet)
    assert list(K.split_lora({um + ".lora_A.weight": a, um + ".lora_B.weight": b})) == ["unet"]


@pytest.mark.parametrize("key", ["unet.conv_in.dora_scale", "lora_unet_conv_in.hada_w1_a", "lora_unet_conv_in.lokr_w1"])
def test_unsupported_lora_formats_are_refused(key):
    with pytest.raises(ValueError, match="unsupported format"):
        K.split_lora({key: torch.zeros(2)})


@pytest.mark.parametrize("key", ["lora_te_text_model_encoder_layers_0_mlp_fc1.lora_down.weight",     # SD 1.x text encoder
                                 "unet.down_blocks.1.attentions.0.proj_in.alpha",                     # an alpha lora_to_peft would not apply
                                 "lora_unet_down_blocks_1_attentions_0_proj_in.lora_up.weight",       # no lora_down
                                 "unet.down_blocks.1.attentions.0.proj_in.lora_B.weight",             # no lora_A
                                 "lora_unet_conv_in.weight"])
def test_lora_keys_that_would_be_skipped_are_refused(key):
    with pytest.raises(ValueError, match="known layout"):
        K.split_lora({key: torch.zeros(2, 2)})


def test_read_lora_sources(tmp_path):
    from safetensors.torch import save_file
    sd = {"unet.conv_in.lora_A.weight": torch.zeros(2, 4, 3, 3)}
    save_file(sd, str(tmp_path / "pytorch_lora_weights.safetensors"))
    save_file(sd, str(tmp_path / "style.safetensors"))
    assert list(K.read_lora(tmp_path)) == list(sd)
    assert list(K.read_lora(str(tmp_path), weight_name="style.safetensors")) == list(sd)
    assert list(K.read_lora(str(tmp_path / "style.safetensors"))) == list(sd)
    assert K.read_lora(sd) == sd
    for bad in ("latent-consistency/lcm-lora-sdxl", str(tmp_path / "missing.safetensors"), 3):
        with pytest.raises(ValueError):
            K.read_lora(bad)


# ---- bookkeeping --------------------------------------------------------------------------------------------------------------

class _Engine:
    """The two things LoraAdapters needs from an engine: the UNet (packed on the CPU) and the device."""

    def __init__(self):
        from fast_image_editing_with_generative_models_b200.engine import UNet
        cfg = C.tiny_unet_config()
        self.params = S.make_unet_params(cfg)
        self.unet = UNet(self.params, cfg, torch.device("cpu"))
        self.dev = torch.device("cpu")


@pytest.fixture(scope="module")
def engine():
    return _Engine()


def _make(engine, base=True):
    """LoraAdapters whose device update is recorded: calls[-2] is the last {(part, module): [(relative weight, adapter object)]}."""
    calls = []
    base_lora = {"default_0": (S.make_lora_params(engine.params, rank=4), 1.0)} if base else None
    ad = LoraAdapters(engine, base_lora, on_change=lambda: calls.append("changed"))
    ad._apply = lambda deltas: calls.append({k: list(v) for k, v in deltas.items()})
    return ad, calls


def _named(ad, deltas):
    """Adapter objects -> names; a build-time adapter reads "built:<name>" (its name may since belong to another adapter)."""
    names = {id(o): n for n, o in ad._adapters.items()}
    names.update({id(o): "built:" + n for n, o in ad._built.items()})
    return {k: [(w, names[id(o)]) for w, o in v] for k, v in deltas.items()}


def _style(engine, rank=4, seed=30):
    return S.make_lora_params({k: v for k, v in engine.params.items() if "attentions" in k}, rank=rank, seed=seed)


def _state(ad):
    return ad.get_active_adapters(), ad.get_list_adapters(), dict(ad._weights)


def test_naming_activation_and_relative_weights(engine):
    ad, calls = _make(engine)
    assert _state(ad)[:2] == (["default_0"], {"unet": ["default_0"]})
    ad.load_lora_weights(_style(engine))
    assert ad.get_active_adapters() == ["default_0", "default_1"] and ad._weights["default_1"] == 1.0
    assert calls[-1] == "changed" and all(ws == [(1.0, "default_1")] for ws in _named(ad, calls[-2]).values())
    ad.load_lora_weights(_style(engine, seed=31), adapter_name="pixel")
    ad.set_adapters(["default_0", "pixel"], [0.5, 0.8])
    d = _named(ad, calls[-2])
    assert ad.get_active_adapters() == ["default_0", "pixel"]
    # default_0 is fused at 1.0: its delta is (0.5 - 1.0); default_1 is inactive
    assert all(n != "default_1" for ws in d.values() for _, n in ws)
    assert any((0.8, "pixel") in ws and (-0.5, "built:default_0") in ws for ws in d.values())
    # the active set as built: no delta at all (every written module is restored)
    ad.set_adapters(["default_0", "pixel"], [1.0, 0.0])
    assert calls[-2] == {}
    ad.delete_adapters("default_0")
    assert ad.get_active_adapters() == ["pixel"] and "default_0" not in ad.get_list_adapters()["unet"]
    assert all(ws == [(-1.0, "built:default_0")] for ws in _named(ad, calls[-2]).values())
    ad.unload_lora_weights()
    assert calls[-2] == {} and _state(ad)[:2] == (["default_0"], {"unet": ["default_0"]})
    nxt, _ = _make(engine, base=False)
    nxt.load_lora_weights(_style(engine))
    assert nxt.get_active_adapters() == ["default_0"]                   # SSD-1B: no load-time adapter, the first unnamed one is default_0


@pytest.mark.parametrize("explicit", [False, True])
def test_a_deleted_build_time_name_given_to_a_new_adapter(engine, explicit):
    """Deleting the fused LCM-LoRA and loading another adapter under its name (the next unnamed name is default_0 again) subtracts the
    LCM-LoRA and adds the new adapter: deltas belong to adapters, not to names."""
    ad, calls = _make(engine)
    lcm_modules = {("unet", k[: -len(".lora_A.weight")]) for k in ad._built["default_0"].parts["unet"] if k.endswith(".lora_A.weight")}
    ad.delete_adapters("default_0")
    style = _style(engine)
    ad.load_lora_weights(style, **({"adapter_name": "default_0"} if explicit else {}))
    assert ad.get_active_adapters() == ["default_0"] and ad._adapters["default_0"] is not ad._built["default_0"]
    d = _named(ad, calls[-2])
    style_modules = {("unet", k[: -len(".lora_A.weight")]) for k in style if k.endswith(".lora_A.weight")}
    assert set(d) == lcm_modules | style_modules
    for key, ws in d.items():
        assert ((-1.0, "built:default_0") in ws) == (key in lcm_modules) and ((1.0, "default_0") in ws) == (key in style_modules)
    ad.set_adapters(["default_0"], 0.5)
    d = _named(ad, calls[-2])
    assert all(sorted(ws) == [(-1.0, "built:default_0"), (0.5, "default_0")] for k, ws in d.items() if k in style_modules)
    ad.unload_lora_weights()
    assert calls[-2] == {} and ad._adapters["default_0"] is ad._built["default_0"] and ad.get_active_adapters() == ["default_0"]


def test_a_failed_device_update_is_undone(engine, monkeypatch):
    """A device update that stops part way (here a write that raises on the 5th module) writes the previous state back: every module
    it touched is restored and the adapters are unchanged."""
    import contextlib

    monkeypatch.setattr(torch.cuda, "device", lambda d: contextlib.nullcontext())
    ad = LoraAdapters(engine, {"default_0": (S.make_lora_params(engine.params, rank=4), 1.0)})
    targets = ad._all_targets()["unet"]
    before = {m: t.weight.clone() for m, t in targets.items()}
    n = [0]

    def write(t, fs):
        n[0] += 1
        if n[0] == 5:
            raise RuntimeError("device error")
        ad._rows(t, t.weight).fill_(7.0)
    ad._write = write
    with pytest.raises(RuntimeError, match="device error"):
        ad.load_lora_weights(_style(engine), adapter_name="s")
    assert all(torch.equal(t.weight, before[m]) for m, t in targets.items())
    assert ad.get_active_adapters() == ["default_0"] and not ad._written and ad.pristine_bytes() == 0


def test_set_adapters_weight_forms(engine):
    ad, calls = _make(engine)
    ad.load_lora_weights(_style(engine), adapter_name="s")
    ad.set_adapters("s")
    assert ad._weights == {"s": 1.0}
    ad.set_adapters(["default_0", "s"], 0.25)
    assert ad._weights == {"default_0": 0.25, "s": 0.25}


def _bad_calls(engine):
    a = torch.zeros(4, 64)
    return [
        ("duplicate", lambda ad: ad.load_lora_weights(_style(engine), adapter_name="default_0")),
        ("unknown set", lambda ad: ad.set_adapters(["default_0", "nope"])),
        ("unknown delete", lambda ad: ad.delete_adapters(["nope"])),
        ("weight count", lambda ad: ad.set_adapters(["default_0"], [1.0, 2.0])),
        ("nan weight", lambda ad: ad.set_adapters(["default_0"], [math.nan])),
        ("inf weight", lambda ad: ad.set_adapters(["default_0"], math.inf)),
        ("text weight", lambda ad: ad.set_adapters(["default_0"], ["x"])),
        ("unmatched", lambda ad: ad.load_lora_weights({"lora_unet_no_such_layer.lora_down.weight": a, "lora_unet_no_such_layer.lora_up.weight": a.t()})),
        ("dora", lambda ad: ad.load_lora_weights({"unet.conv_in.lora_A.weight": a, "unet.conv_in.dora_scale": a})),
        ("loha", lambda ad: ad.load_lora_weights({"lora_unet_conv_in.hada_w1_a": a})),
        ("no packed form", lambda ad: ad.load_lora_weights({"unet.down_blocks.1.attentions.0.norm.lora_A.weight": a,
                                                             "unet.down_blocks.1.attentions.0.norm.lora_B.weight": torch.zeros(128, 4)})),
        ("factor shape", lambda ad: ad.load_lora_weights({"unet.down_blocks.1.attentions.0.proj_in.lora_A.weight": a,
                                                           "unet.down_blocks.1.attentions.0.proj_in.lora_B.weight": torch.zeros(128, 4)})),
        ("hub id", lambda ad: ad.load_lora_weights("latent-consistency/lcm-lora-sdxl")),
        ("empty", lambda ad: ad.load_lora_weights({})),
    ]


@pytest.mark.parametrize("case", range(14))
def test_errors_leave_the_adapters_unchanged(engine, case):
    what, call = _bad_calls(engine)[case]
    ad, calls = _make(engine)
    ad.load_lora_weights(_style(engine), adapter_name="s")
    before, n = _state(ad), len(calls)
    with pytest.raises(ValueError):
        call(ad)
    assert _state(ad) == before and len(calls) == n, what
    ad.set_adapters(["default_0", "s"], [1.0, 0.5])                      # still usable
    assert ad._weights == {"default_0": 1.0, "s": 0.5}


def test_text_encoder_part_without_gpu_towers_is_ignored_with_a_warning(engine):
    ad, calls = _make(engine)
    sd = {"unet." + k: v for k, v in _style(engine).items()}
    sd["lora_te1_text_model_encoder_layers_0_mlp_fc1.lora_down.weight"] = torch.zeros(4, 128)
    sd["lora_te1_text_model_encoder_layers_0_mlp_fc1.lora_up.weight"] = torch.zeros(256, 4)
    with pytest.warns(RuntimeWarning, match="text_encoder part"):
        ad.load_lora_weights(sd, adapter_name="s")
    assert ad.get_list_adapters() == {"unet": ["default_0", "s"]}
