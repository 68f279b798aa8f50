"""CPU: the C-ABI library builds, loads, and exports every symbol include/fie_b200.h declares (no compute calls)."""
import ctypes
import os
import re

from fast_image_editing_with_generative_models_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    names = set()
    for fn in os.listdir(os.path.join(ROOT, "include")):
        if fn.endswith(".h"):
            src = open(os.path.join(ROOT, "include", fn)).read()
            src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
            names |= set(re.findall(r"\b(fie_[a-z0-9_]+)\s*\(", src))
    return names


def test_library_exports_every_declared_symbol():
    if not os.path.exists(_lib.LIB_PATH):
        _lib.build()
    L = ctypes.CDLL(_lib.LIB_PATH)
    declared = _declared_symbols()
    assert len(declared) >= 20
    for name in declared:
        assert hasattr(L, name), f"{name} declared in include/ but not exported"
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)


def test_no_gpu_calls_needed_for_queries():
    L = _lib.lib()
    assert L.fie_version() >= 100
    assert L.fie_geglu_block_n(10240) == 256 and L.fie_geglu_block_n(512) == 256 and L.fie_geglu_block_n(384) == 128
    assert L.fie_canny_workspace_bytes(1, 1024, 1024) >= 6 * 1024 * 1024


def test_epilogue_struct_layout():
    # fie_epilogue: 7 x 8-byte fields + float + 2 ints = 68 -> 72; + gn_stats pointer, gn_groups int (+4 pad), gn_rows_per_image = 96;
    # + ln_stats_out, ln_stats_in pointers, ln_eps float, ln_dim int = 120; + row_scale pointer = 128
    assert ctypes.sizeof(_lib.Epilogue) == 128


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, "fast_image_editing_with_generative_models_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in src and "from oracle" not in src, f


def test_only_tests_smoke_and_bench_touch_the_oracle():
    """oracle/ is test infrastructure: besides tests/, only __graft_entry__.smoke() and bench.py (cpu_baseline / --impl reference legs)
    may import it — not the CLIs, not the drop-in modules, not the helper scripts."""
    offenders = []
    for rel in ("scripts", "src"):
        for dirpath, _, files in os.walk(os.path.join(ROOT, rel)):
            offenders += [os.path.join(dirpath, f) for f in files if f.endswith((".py", ".sh"))]
    offenders += [os.path.join(ROOT, f) for f in ("run_batch.py", "run_single_image.py", "evaluate.py")]
    for path in offenders:
        src = open(path).read()
        assert "import oracle" not in src and "from oracle" not in src, path


def test_argument_validation_reports_errors_without_a_gpu():
    """Every entry point validates its arguments before touching CUDA and reports through the return code + fie_last_error(): the
    reference's callers rely on ordinary exceptions per image (run_batch.py:250-261), never on a process abort."""
    L = _lib.lib()
    buf = (ctypes.c_ubyte * 64)()
    p = ctypes.addressof(buf)
    cases = [
        (L.fie_canny_u8(p, p, 1, 8, 8, 2, 1, 100, 200, p, 1 << 20, None), "in_channels"),
        (L.fie_gaussian_blur5_u8(p, p, 1, 8, 8, 1, None), "in-place"),
        (L.fie_gaussian_blur5_u8(p, p + 16, 1, 8, 8, 2, None), "channels"),
        (L.fie_jpeg_encode_u8(p, 1, 16, 16, 75, p, 16, p, p, 1 << 30, None), "out_stride"),
        (L.fie_attn_vae_d512_f16(p, 512, p, 512, p, p, 512, 100, 500, 0.1, 0, 0, p, 1 << 30, None), "d % 64"),
        (L.fie_fuse_lora_f32(p, p, p, 1.0, 0, 4, 8, None), "bad arguments"),
        (L.fie_pack_conv3x3_c8_f16(p, p, 8, 9, 8, None), "cin <= 8"),
        (L.fie_ssim_u8(p, p, 1, 8, 8, 3, 11, 1.5, 0.01, 0.03, p, None), "smaller than the window"),
        (L.fie_ssim_u8(p, p, 1, 32, 32, 3, 10, 1.5, 0.01, 0.03, p, None), "odd"),
        (L.fie_patchify_f16(p, 1, p, 1, 30, 32, 16, None, None, None), "multiples of the patch"),
        (L.fie_vit_assemble_f16(p, p, p, p, 1, 4, 12, None), "multiple of 8"),
        (L.fie_im2col3x3_f16(p, 0, 16, p, 1, 8, 8, 16, 1, 1, 100, None, None, None), "kpad"),
        (L.fie_maxpool3s2_ceil_f16(p, p, 1, 8, 8, 12, None), "multiple of 8"),
        (L.fie_resample_f32(p, 1, p, None, 1, 8, 8, 8, 4, None, None, 0, None, None, 0, None, None, None), "tables missing"),
    ]
    for rc, needle in cases:
        assert rc != 0
    assert L.fie_canny_u8(p, p, 1, 8, 8, 2, 1, 100, 200, p, 1 << 20, None) != 0 and b"in_channels" in L.fie_last_error()
    assert L.fie_attn_vae_d512_f16(p, 512, p, 512, p, p, 512, 100, 500, 0.1, 0, 0, p, 1 << 30, None) != 0 and b"d % 64" in L.fie_last_error()
    assert L.fie_ssim_u8(p, p, 1, 8, 8, 3, 11, 1.5, 0.01, 0.03, p, None) != 0 and b"smaller than the window" in L.fie_last_error()
    assert L.fie_patchify_f16(p, 1, p, 1, 30, 32, 16, None, None, None) != 0 and b"patch size" in L.fie_last_error()
    # the GEGLU epilogue takes no per-row bias (the fast and slow epilogue paths would apply it to different operands)
    ep = _lib.Epilogue(m_bias=p, scale=1.0, act=2)
    assert L.fie_gemm_f16(p, 64, None, 0, 0, p, p, 32, 128, 64, 64, ctypes.byref(ep), None) != 0 and b"m_bias" in L.fie_last_error()
    # pure host queries
    assert L.fie_jpeg_header_bytes() == 623 and L.fie_jpeg_max_bytes(1024, 1024) > 3 * 1024 * 1024
    assert L.fie_jpeg_workspace_bytes(8, 1024, 1024) > 8 * 4096 * 384 * 2
    assert L.fie_attn_vae_workspace_bytes(16384, 0, 0) >= 16384 * 16384 * 2 and L.fie_attn_vae_workspace_bytes(16384, 4096, 1) >= 4096 * 16384 * 6
