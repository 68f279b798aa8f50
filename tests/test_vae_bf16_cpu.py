"""CPU: host side of the bf16 VAE — ``force_upcast`` parsing, the ``vae_dtype`` resolution and its warning, the CLI flag, the bf16 host
packing (a torch restatement), and argument validation of the new C-ABI entry points (rejected before any CUDA call)."""
import ctypes
import json

import pytest
import torch

from fast_image_editing_with_generative_models_b200 import _lib
from fast_image_editing_with_generative_models_b200 import checkpoints as K
from fast_image_editing_with_generative_models_b200 import editor as E
from fast_image_editing_with_generative_models_b200 import weights as W

BF = torch.bfloat16
VAE_JSON = {"block_out_channels": [128, 256, 512, 512], "layers_per_block": 2, "latent_channels": 4, "scaling_factor": 0.13025}


@pytest.mark.parametrize("value,expected", [(True, True), (False, False), (None, None)])
def test_force_upcast_is_parsed(value, expected):
    d = dict(VAE_JSON) if value is None else {**VAE_JSON, "force_upcast": value}
    assert K.vae_config_from_json(json.loads(json.dumps(d))).force_upcast is expected


@pytest.mark.parametrize("force_upcast", [True, False, None])
def test_vae_dtype_resolution(force_upcast):
    assert E.resolve_vae_dtype(None, force_upcast) == (BF if force_upcast else torch.float16)
    assert E.resolve_vae_dtype(torch.float16, force_upcast) == torch.float16
    assert E.resolve_vae_dtype(BF, force_upcast) == BF
    with pytest.raises(ValueError):
        E.resolve_vae_dtype(torch.float32, force_upcast)


def test_fp16_vae_warning_only_for_real_weights_without_force_upcast_false():
    for real in (True, False):
        for dt in (torch.float16, BF):
            for fu in (True, False, None):
                msg = E.vae_fp16_warning(real, dt, fu)
                assert (msg is not None) == (real and dt == torch.float16 and fu is not False), (real, dt, fu)
    msg = E.vae_fp16_warning(True, torch.float16, None)
    assert "sdxl-vae-fp16-fix" in msg and "vae_dtype=torch.bfloat16" in msg


@pytest.mark.parametrize("flag,expected", [([], None), (["--vae_dtype", "auto"], None), (["--vae_dtype", "fp16"], torch.float16),
                                           (["--vae_dtype", "bf16"], BF)])
def test_cli_flag_reaches_the_editor(tmp_path, monkeypatch, flag, expected):
    import run_batch
    import run_single_image
    seen = []

    class Stop(Exception):
        pass

    class Fake:
        def __init__(self, **kw):
            seen.append(kw)
            raise Stop

    img = tmp_path / "x.png"
    from PIL import Image
    Image.new("RGB", (16, 16)).save(img)
    mp = tmp_path / "m.json"
    mp.write_text(json.dumps({"0": {"image_path": "x.png", "editing_prompt": "p", "editing_type_id": "0"}}))
    monkeypatch.setattr(run_batch, "FastEditor", Fake)
    monkeypatch.setattr(run_single_image, "FastEditor", Fake)
    with pytest.raises(Stop):
        run_batch.main(["--mapping_file", str(mp), "--source_dir", str(tmp_path), "--output_dir", str(tmp_path / "o")] + flag)
    with pytest.raises(Stop):
        run_single_image.main(["--image", str(img), "--prompt", "p", "--output_dir", str(tmp_path / "o")] + flag)
    assert [kw["vae_dtype"] for kw in seen] == [expected, expected]


def test_bf16_host_packing_equals_a_torch_restatement():
    g = torch.Generator().manual_seed(0)
    w = torch.randn((40, 24, 3, 3), generator=g)
    p = W.pack_conv3x3(w, 64, 32, dtype=BF)
    ref = torch.zeros((64, 3, 3, 32), dtype=BF)
    ref[:40, :, :, :24] = w.permute(0, 2, 3, 1).to(BF)
    assert p.dtype == BF and torch.equal(p, ref.reshape(64, 288))
    up = W.pack_conv_up2x(w, dtype=BF)
    assert torch.equal(up, _up2x_ref(w).to(BF))
    lin = torch.randn((48, 40), generator=g)
    assert torch.equal(W.cast_f16(lin, BF), lin.to(BF))
    with pytest.raises(ValueError):
        W.cast_f16(lin, torch.float32)


def _up2x_ref(w):
    """Phase (a, b), tap (ty, tx) of nearest-2x upsample + conv3x3 = the sum of the 3x3 taps landing on that input pixel, rows first."""
    sets = ([[0], [1, 2]], [[0, 1], [2]])              # [phase bit][tap] -> kernel indices
    out = torch.empty((4, w.shape[0], 2, 2, w.shape[1]))
    for a in (0, 1):
        for b in (0, 1):
            for ty in (0, 1):
                for tx in (0, 1):
                    rows = [sum(w[:, :, kh, kw] for kh in sets[a][ty]) for kw in range(3)]
                    out[2 * a + b, :, ty, tx] = sum(rows[kw] for kw in sets[b][tx])
    return out.reshape(4, w.shape[0], 4 * w.shape[1])


def test_new_entry_points_reject_bad_arguments_without_a_gpu():
    L = _lib.lib()
    buf = (ctypes.c_ubyte * 256)()
    p = ctypes.addressof(buf)
    ep = _lib.Epilogue()
    ep.scale = 1.0
    ep.rows_per_group = 1
    # out_dtype outside FIE_DT_*
    for rc in (L.fie_gemm_bf16(p, 64, None, 0, 0, p, p, 64, 128, 64, 64, ctypes.byref(ep), 7, None),
               L.fie_conv3x3_bf16(p, p, p, 64, 1, 8, 128, 64, 64, 64, 1, 0, ctypes.byref(ep), -1, None),
               L.fie_conv_up2x_bf16(p, p, p, 64, 1, 8, 128, 64, 64, ctypes.byref(ep), 3, None),
               L.fie_conv3x3_c8_bf16(p, p, p, 64, 1, 8, 128, 64, 64, ctypes.byref(ep), 9, None)):
        assert rc == -1 and b"bad out_dtype" in L.fie_last_error()
    # out_f32 set but a 16-bit output requested
    ep.out_f32 = 1
    assert L.fie_gemm_bf16(p, 64, None, 0, 0, p, p, 64, 128, 64, 64, ctypes.byref(ep), _lib.DT_BF16, None) == -1
    assert b"out_f32" in L.fie_last_error()
    ep.out_f32 = 0
    # producer-side GroupNorm statistics with bf16 output
    ep.gn_stats, ep.gn_groups, ep.gn_rows_per_image = p, 2, 128
    assert L.fie_gemm_bf16(p, 64, None, 0, 0, p, p, 64, 128, 64, 64, ctypes.byref(ep), _lib.DT_BF16, None) == -1
    assert b"gn_stats" in L.fie_last_error()
    assert L.fie_conv3x3_bf16(p, p, p, 64, 1, 8, 128, 64, 64, 64, 1, 0, ctypes.byref(ep), _lib.DT_BF16, None) == -1
    assert b"gn_stats" in L.fie_last_error()
    # GroupNorm: workspace size, channel multiples; attention: d % 64; softmax / packers: bad shapes
    need = L.fie_groupnorm_bf16_workspace_bytes(8, 1 << 20, 128, 32)
    assert need >= 8 * 32 * 3 * 4 and need % 256 == 0
    assert L.fie_groupnorm_bf16(p, 128, None, 0, p, 8, 1 << 20, 32, p, p, 1e-6, 1, p, need - 1, None) == -1
    assert b"workspace too small" in L.fie_last_error()
    assert L.fie_groupnorm_bf16(p, 12, None, 0, p, 1, 64, 4, p, p, 1e-6, 1, p, 1 << 30, None) == -1
    assert b"multiples of 8" in L.fie_last_error()
    assert L.fie_attn_vae_d512_bf16(p, 512, p, 512, p, p, 512, 100, 500, 0.1, 0, p, 1 << 30, None) == -1
    assert b"d % 64" in L.fie_last_error()
    assert L.fie_softmax_rows_f32_to_bf16(p, 3, p, 4, 1, 4, 1.0, None) == -1
    assert L.fie_pack_conv3x3_bf16(p, p, 8, 8, 4, 8, None) == -1
    assert L.fie_pack_conv_up2x_bf16(p, p, 0, 8, None) == -1
    assert L.fie_pack_rows_bf16(p, p, None, p, None, 4, 4, None) == -1
