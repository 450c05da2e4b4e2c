"""CPU-side checks of the drop-in boundary: the C-ABI library loads and exports every symbol that
include/xqb200.h declares; argument validation returns error codes (no GPU work is launched)."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "xqb200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(xq_[a-z0-9_]+)\s*\(", text)))


def test_header_symbols_are_exported():
    from imagefolder_b200 import _capi
    L = _capi.lib()
    syms = declared_symbols()
    assert len(syms) >= 16
    for s in syms:
        assert hasattr(L, s), f"{s} declared in include/xqb200.h but not exported by libxqb200.so"
    assert sorted(_capi.EXPORTED_SYMBOLS) == syms
    assert L.xq_abi_version() == 1
    assert L.xq_strerror(0) == b"ok"


def test_desc_struct_layout_matches_header():
    from imagefolder_b200 import _capi
    # 8 ints + 3 arrays of 32 4-byte values + 2 floats + 2 ints + 3 floats
    assert ctypes.sizeof(_capi.XqMsDesc) == 4 * (8 + 3 * 32 + 2 + 2 + 3)


def test_argument_validation_without_gpu():
    from imagefolder_b200 import _capi
    L = _capi.lib()
    assert L.xq_vq_workspace_bytes(0, 32, 256, 8192) == 0
    assert L.xq_vq_workspace_bytes(256, 32, 256, 8192) >= 4 * 8192 * 32
    assert L.xq_vq_forward(None, None, 1, 1, 1, 1, 1, 1, 0.25, None, None, None, None, None, 0, None) == -1
    d = _capi.make_ms_desc(2, 8, 5, 5, 64, 4, [1, 2, 5], [0, 1, 3], _capi.XQ_MS_VQ_ZNORM)
    assert L.xq_ms_total_tokens(d) == 2 * (1 + 4 + 25)
    assert L.xq_ms_workspace_bytes(d) > 0 and L.xq_ms_saved_bytes(d) == 4 * 2 * 8 * 25
    bad = _capi.make_ms_desc(2, 8, 5, 5, 64, 4, [1, 2, 4], [0, 1, 3], _capi.XQ_MS_VQ_ZNORM)  # last scale != H
    assert L.xq_ms_total_tokens(bad) == -1
    bsq = _capi.make_ms_desc(2, 6, 3, 3, 100, 0, [1, 3], [0, 0], _capi.XQ_MS_BSQ)  # V != 2**C
    assert L.xq_ms_workspace_bytes(bsq) == 0
    with pytest.raises(ValueError):
        _capi.check(-1, "x")
    with pytest.raises(_capi.XqError):
        _capi.check(-2, "x")


def test_cpu_tensors_are_rejected_loudly():
    """no CPU fallback: the product refuses host tensors instead of silently computing elsewhere."""
    import torch
    from imagefolder_b200 import VectorQuantizer, _capi
    q = VectorQuantizer(64, 8)
    with pytest.raises(_capi.XqError):
        q(torch.randn(1, 8, 2, 2))


def test_state_dict_keys_match_reference():
    from imagefolder_b200 import LFQ, VectorQuantizer, VectorQuantizer2
    pn = [1, 2, 3]
    assert set(VectorQuantizer(64, 8).state_dict()) == {"embedding.weight", "ema_vocab_hit_SV"}
    k2 = set(VectorQuantizer2(64, 8, v_patch_nums=pn).state_dict())
    assert k2 == {"ema_vocab_hit_SV", "embedding.weight"} | {f"quant_resi.qresi_ls.{i}.{n}" for i in range(4)
                                                              for n in ("weight", "bias")}
    kl = set(LFQ(64, 6, v_patch_nums=pn).state_dict())
    assert kl == {"ema_vocab_hit_SV", "scaler"} | {f"quant_resi.qresi_ls.{i}.{n}" for i in range(4)
                                                    for n in ("weight", "bias")}
    q = VectorQuantizer2(64, 8, v_patch_nums=[1, 1, 2, 3, 3, 4, 5, 6, 8, 11])
    assert q._phi_map(10) == [0, 0, 1, 1, 1, 2, 2, 3, 3, 3]        # SURVEY.md 8a / quant.py:285-288
    assert VectorQuantizer2(8, 4, v_patch_nums=pn, share_quant_resi=1)._phi_map(3) == [0, 0, 0]
    assert VectorQuantizer2(8, 4, v_patch_nums=pn, share_quant_resi=0)._phi_map(3) == [0, 1, 2]


def test_bench_helpers_are_total():
    """bench.py's explanatory extras must never cost the JSON line (no GPU needed for these helpers)."""
    import importlib.util, os
    spec = importlib.util.spec_from_file_location("_bench", os.path.join(os.path.dirname(os.path.dirname(__file__)), "bench.py"))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    rows = [{"entry": "xq_vit_residual_ln_bwd", "calls_per_step": 50.0, "ms_per_step": 16.7, "ms_per_call": 0.334, "alg_GBps": 5350.0,
             "alg_TFps": None, "alg_bytes_per_call": 1.787e9, "alg_flops_per_call": 0.0},
            {"entry": "xq_vq_forward", "calls_per_step": 1.0, "ms_per_step": 0.2, "ms_per_call": 0.2, "alg_GBps": None,
             "alg_TFps": None, "alg_bytes_per_call": 0, "alg_flops_per_call": 0.0}]
    r = b.top_kernel_roofline(rows, 6385.8, 1678.2, 211.0, {"xq_vit_residual_ln_bwd": 1.788e9})
    assert r["kernel"] == "xq_vit_residual_ln_bwd" and r["bound"] == "hbm" and abs(r["frac"] - 5350.0 / 6385.8) < 1e-12
    assert r["traffic"] == 1.788e9 and abs(r["share_of_step"] - 16.7 / 211.0) < 1e-12
    # an entry with tensor FLOPs is reported against the roof it sits closer to
    attn = {"entry": "xq_vit_attn_bwd", "calls_per_step": 24.0, "ms_per_step": 32.0, "ms_per_call": 1.33, "alg_GBps": 1100.0,
            "alg_TFps": 390.0, "alg_bytes_per_call": 1.46e9, "alg_flops_per_call": 5.17e11}
    r = b.top_kernel_roofline(rows + [attn], 6385.8, 1678.2, 211.0)
    assert r["kernel"] == "xq_vit_attn_bwd" and r["bound"] == "tensor" and abs(r["frac"] - 390.0 / 1678.2) < 1e-12
    assert r["traffic"] is None and abs(r["hbm_frac"] - 1100.0 / 6385.8) < 1e-12
    assert b.top_kernel_roofline([], 6385.8, 1678.2, 1.0) is None
    assert b.top_kernel_roofline(rows[1:], 6385.8, 1678.2, 1.0) is None
    assert "error" in b._safe(lambda: 1 / 0) and b._safe(lambda: 3) == 3
    hbm, tf, src = b.peaks()
    assert hbm > 1000 and tf > 100 and src.split()[0] in ("measured", "fallback")


def test_argument_validation_of_the_newer_entry_points_without_gpu():
    """every check below fails BEFORE any CUDA call, so it runs without a device"""
    import ctypes as C
    from imagefolder_b200 import _capi
    L = _capi.lib()
    one = C.c_void_p(16)                     # a non-null dummy pointer; never dereferenced on these paths
    d = _capi.make_ms_desc(2, 8, 5, 5, 64, 4, [1, 2, 5], [0, 1, 3], _capi.XQ_MS_VQ_ZNORM)
    f = C.cast(one, C.POINTER(C.c_float))
    assert L.xq_ms_embed(d, 0, 4, f, f, f, None, f, None, None, None) == -1           # si1 > SN
    assert L.xq_ms_embed(d, 2, 2, f, f, f, None, f, None, None, None) == -1           # empty range
    assert L.xq_ms_embed(d, 0, 3, None, f, f, None, f, None, None, None) == -1        # no feature maps
    assert L.xq_lpips_workspace_bytes(4, 64 * 64) >= 8 * 4 * 16
    assert L.xq_lpips_layer_forward(None, one, 0, f, 1, 8, 16, 1e-10, 0, f, one, 1 << 20, None) == -1
    assert L.xq_lpips_layer_forward(one, one, 0, f, 2, 8, 4096, 1e-10, 0, f, one, 8, None) == -2     # workspace too small
    assert L.xq_lpips_layer_forward(one, one, 1, f, 1, 8, 15, 1e-10, 0, f, one, 1 << 20, None) == -4  # bf16 needs even H*W
    assert L.xq_lpips_layer_backward(one, one, 0, f, 0, 8, 16, 1e-10, f, one, None) == -1
    assert L.xq_diffaug_forward(f, f, 2, 9, 8, 8, 7, 2, 2, f, f, None) == -4          # more than 8 channels
    assert L.xq_diffaug_forward(f, None, 2, 3, 8, 8, 1, 2, 2, f, f, None) == -1       # flags set but no random numbers
    assert L.xq_diffaug_backward(f, f, 2, 3, 8, 8, 8, 2, 2, f, f, None) == -1         # unknown flag bit
    assert L.xq_vit_pack_workspace_bytes() >= 4
    assert L.xq_vit_pack_qkv(one, one, one, one, None, 16, 768, one, 2, None) == -2    # workspace too small
    assert L.xq_vit_pack_qkv(one, one, one, one, None, 16, 4096, one, 256, None) == -4  # 3C/8 chunks beyond the kernel's range
    assert L.xq_vit_pack_qkv(one, one, one, one, None, 16, 12, one, 256, None) == -1   # C % 8 != 0
    assert L.xq_vit_assemble_fwd(one, 1, f, 2, 4, 6, 16, 3, f, None) == -1            # t0 + Ls > T
    assert L.xq_vit_assemble_fwd(one, 1, f, 2, 4, 8, 18, 1, f, None) == -1            # D % 4 != 0
    assert L.xq_vit_assemble_bwd(f, 2, 4, 8, 16, 1, None, 0, None, None) == -1        # nothing to compute
    assert L.xq_vit_patchify(f, one, 2, 3, 64, 64, 6, None) == -4                      # patch % 4 != 0
    assert L.xq_vit_patchify(f, one, 2, 3, 60, 64, 16, None) == -4                     # H % patch != 0
    assert L.xq_vit_residual_ln_bwd(None, None, None, None, None, None, None, None, None, None, 1, 8, 768, None, None, None,
                                    None, None, None, None, 0, None) == -1


def test_attention_entry_points_validate_arguments_without_gpu():
    """xq_vit_attn_fwd / bwd (csrc/attn_kernel.cu): NULL pointers, unsupported head dims, misaligned buffers and short
    workspaces are refused with error codes before anything is launched."""
    from imagefolder_b200 import _capi
    L = _capi.lib()
    assert L.xq_vit_attn_fwd(None, None, None, 1, 16, 1, 64, 0.125, None) == -1
    assert L.xq_vit_attn_fwd(4096, 8192, 12288, 1, 16, 1, 32, 0.125, None) == -4      # head_dim != 64: unsupported
    assert L.xq_vit_attn_fwd(4097, 8192, 12288, 1, 16, 1, 64, 0.125, None) == -1      # qkv not 16-byte aligned
    assert L.xq_vit_attn_fwd(4096, 8192, 12288, 0, 16, 1, 64, 0.125, None) == -1
    assert L.xq_vit_attn_bwd_workspace_bytes(0, 16, 1) == 0
    need = L.xq_vit_attn_bwd_workspace_bytes(2, 513, 12)
    assert need >= 2 * 12 * 513 * 64 * 4 + 2 * 2 * 12 * 640 * 4
    assert L.xq_vit_attn_bwd(None, None, None, None, None, None, 1, 16, 1, 64, 0.125, None, 0, None) == -1
    assert L.xq_vit_attn_bwd(4096, 4096, 4096, 4096, 4096, None, 2, 513, 12, 64, 0.125, 4096, need - 1, None) == -2   # workspace
    assert L.xq_vit_attn_bwd(4096, 4096, 4096, 4096, 4096, None, 2, 513, 12, 128, 0.125, 4096, need, None) == -4


def test_fused_mlp_gemm_entry_points_validate_arguments_without_gpu():
    """xq_vit_fc1_gelu_fwd / xq_vit_fc2_dgelu_bwd (csrc/gemm_kernel.cu): NULL pointers, misaligned buffers and widths the CTA-pair
    tile does not cover are refused before anything is launched (the host then keeps library GEMM + the stand-alone kernel)."""
    import ctypes as C
    from imagefolder_b200 import _capi
    L = _capi.lib()
    f = C.cast(C.c_void_p(4096), C.POINTER(C.c_float))
    assert L.xq_vit_fc1_gelu_fwd(None, 4096, f, 4096, 4096, 128, 3072, 768, None) == -1
    assert L.xq_vit_fc1_gelu_fwd(4096, 4096, f, 4096, 4096, 0, 3072, 768, None) == -1            # M = 0
    assert L.xq_vit_fc1_gelu_fwd(4096, 4096, f, 4096, 4096, 128, 3000, 768, None) == -4          # N % 256 != 0: unsupported
    assert L.xq_vit_fc1_gelu_fwd(4096, 4096, f, 4096, 4096, 128, 3072, 100, None) == -4          # K % 64 != 0: unsupported
    assert L.xq_vit_fc1_gelu_fwd(4100, 4096, f, 4096, 4096, 128, 3072, 768, None) == -1          # x not 16-byte aligned
    assert L.xq_vit_fc2_dgelu_bwd(4096, 4096, 4096, f, 4096, None, 128, 3072, 768, None) == -1   # no bias-gradient buffer
    assert L.xq_vit_fc2_dgelu_bwd(4096, None, 4096, f, 4096, f, 128, 3072, 768, None) == -1
    assert L.xq_vit_fc2_dgelu_bwd(4096, 4096, 4096, f, 4096, f, 128, 1000, 768, None) == -4


def test_fused_mlp_dispatch_conditions():
    """vit_ops.mlp_tc_ok: the fused GEMMs take bf16 CUDA tokens with hidden % 256 == 0 and in- / out-features % 64 == 0 (the
    out-features are the K of the fused backward GEMM, which refuses K % 64 != 0); everything else stays on library GEMM +
    stand-alone bias / GELU kernel (same results, tests/test_gpu_vit_ops.py)."""
    import torch
    from imagefolder_b200 import vit_ops

    class CudaBf16Tokens:            # the only attributes mlp_tc_ok reads from the tokens
        is_cuda = True
        dtype = torch.bfloat16

    fc1, fc2 = torch.nn.Linear(768, 3072), torch.nn.Linear(3072, 768)
    y = torch.zeros(4, 768, dtype=torch.bfloat16)
    assert not vit_ops.mlp_tc_ok(y, fc1, fc2)                          # CPU tensor: never
    tok = CudaBf16Tokens()
    assert vit_ops.mlp_tc_ok(tok, fc1, fc2)
    assert vit_ops.mlp_tc_ok(tok, fc1, torch.nn.Linear(3072, 192))     # out-features != in-features, still % 64
    for out_features in (200, 8, 96, 776):                              # % 8 == 0 but not % 64: the backward would be refused
        assert not vit_ops.mlp_tc_ok(tok, fc1, torch.nn.Linear(3072, out_features)), out_features
    assert not vit_ops.mlp_tc_ok(tok, torch.nn.Linear(768, 3000), torch.nn.Linear(3000, 768))   # hidden % 256 != 0
    assert not vit_ops.mlp_tc_ok(tok, torch.nn.Linear(200, 3072), fc2)                           # in-features % 64 != 0
    assert not vit_ops.mlp_tc_ok(tok, torch.nn.Linear(768, 3072, bias=False), fc2)               # no fc1 bias
    f32 = CudaBf16Tokens()
    f32.dtype = torch.float32
    assert not vit_ops.mlp_tc_ok(f32, fc1, fc2)
    assert vit_ops.MLP_TC_ENABLED[0] is True
