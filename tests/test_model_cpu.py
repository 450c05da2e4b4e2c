"""CPU tests of the host logic: config contract, VQModel wiring, and the product's ViT
encoder/decoder against the oracle's independent restatement (same weights, fp32)."""
import json
import os

import numpy as np
import pytest
import torch
import yaml

from imagefolder_b200 import config as xcfg
from imagefolder_b200.xqgan_model import ModelArgs, VQModel, VQ_models
from oracle import vit_ref


def small_model(name="VQ-8192", **over):
    c = dict(xcfg.SHIPPED_CONFIGS[name])
    c.update(encoder_model="vit_small_patch14_dinov2.lvd142m", decoder_model="vit_small_patch14_dinov2.lvd142m",
             semantic_guide="none", detail_guide="none")
    c.update(over)
    args = xcfg.parse_args([])
    for k, v in c.items():
        setattr(args, k, v)
    torch.manual_seed(0)
    return xcfg.build_vq_model(args), args


@pytest.mark.parametrize("name", ["VQ-8192", "VP2-16384", "MSVR10P2-4096", "MSBR10P2-16384"])
def test_encode_decode_match_oracle(name):
    model, args = small_model(name)
    model.eval()
    cfg = vit_ref.cfg_from_model_args(model.config, num_heads=6)
    ref = vit_ref.RefTokenizer(model.state_dict(), cfg)
    x = torch.rand(2, 3, 256, 256) * 2 - 1
    with torch.no_grad():
        h = model.encode(x)
        h_ref = ref.encode(x)
        assert h.shape == h_ref.shape
        np.testing.assert_allclose(h.numpy(), h_ref.numpy(), rtol=1e-4, atol=1e-5)
        C = model.Cvae
        s = int(np.sqrt(model.config.num_latent_tokens // model.product_quant))
        q = torch.randn(2, C, s, s)
        d, d_ref = model.decode(q), ref.decode(q)
        assert d.shape == (2, 3, 256, 256)
        np.testing.assert_allclose(d.numpy(), d_ref.numpy(), rtol=1e-4, atol=1e-5)


def test_checkpoint_keys_follow_reference_names():
    model, _ = small_model("MSVR10P2-4096")
    keys = set(model.state_dict())
    for k in ["encoder.model.patch_embed.proj.weight", "encoder.model.cls_token", "encoder.model.pos_embed",
              "encoder.model.blocks.0.attn.qkv.weight", "encoder.model.blocks.11.ls2.gamma", "encoder.model.norm.bias",
              "encoder.latent_tokens", "encoder.lvl_embed.weight", "encoder.lvl1LC", "decoder.mask_token",
              "decoder.lvl_embed.weight", "decoder.to_pixel.model.weight", "decoder.model.blocks.3.mlp.fc1.bias",
              "quant_conv.weight", "post_quant_conv.bias", "quantizes.0.embedding.weight",
              "quantizes.1.quant_resi.qresi_ls.3.bias", "quantizes.0.ema_vocab_hit_SV"]:
        assert k in keys, k
    assert not any(k.startswith("decoder.model.patch_embed.proj") for k in keys)   # deleted, dinov2.py:309-310
    assert model.encoder.lvl1LC.shape == (1, 257 + 242) and model.decoder.lvl1LC.shape == (1, 257 + 122)
    assert model.decoder.last_layer is model.decoder.to_pixel.model.weight


def test_yaml_contract(tmp_path):
    """flat YAML -> argparse defaults, CLI wins, unknown keys accepted (xqgan_train.py:168-175)."""
    for name, cfg in xcfg.SHIPPED_CONFIGS.items():
        p = tmp_path / f"{name}.yaml"
        p.write_text(yaml.safe_dump(dict(cfg, data_path="/x", cloud_save_path="y", lr="3e-5")))
        args = xcfg.parse_args(["--config", str(p)])
        assert args.codebook_size == cfg["codebook_size"] and args.lr == 3e-5
        assert list(args.v_patch_nums) == cfg["v_patch_nums"]
        kw = xcfg.model_kwargs(args)
        assert "codebook_l2_norm" not in kw and "scale" not in kw      # parsed but never forwarded
        args2 = xcfg.parse_args(["--config", str(p), "--codebook-size", "77", "--guide_type_2", "patch"])
        assert args2.codebook_size == 77 and args2.guide_type_2 == "patch"
    a = xcfg.parse_args(["--config", str(tmp_path / "RobustTok.yaml")])
    assert xcfg.perturbation_schedule(a, 0) == (1.0, 0.1, 100)
    assert xcfg.perturbation_schedule(a, 200) == (0.5, 0.1, 50)
    al, be, de = xcfg.perturbation_schedule(a, 80)
    assert abs(al - 0.75) < 1e-12 and de == 75


def test_shipped_config_table_matches_reference_yamls(golden_dir):
    """golden = the reference's configs/*.yaml, one object per file holding the keys the table mirrors
    (tests/golden/make_golden.py --configs-only)."""
    with open(os.path.join(golden_dir, "reference_configs.json")) as f:
        yamls = json.load(f)
    assert set(yamls) == set(xcfg.SHIPPED_CONFIGS)
    for name, y in yamls.items():
        for k, v in xcfg.SHIPPED_CONFIGS[name].items():
            ref = float(y[k]) if k == "lr" else y[k]
            assert ref == v, (name, k)


def test_model_variants_build():
    m, _ = small_model("VP2-4096")
    assert len(m.quantizes) == 2 and type(m.quantizes[0]).__name__ == "VectorQuantizer"
    m, _ = small_model("MSBR10P2-4096")
    assert type(m.quantizes[1]).__name__ == "LFQ" and m.quantizes[0].vocab_size == 4096
    assert m.post_quant_conv.in_channels == 24
    m, _ = small_model("RobustTok")
    assert type(m.quantize).__name__ == "VectorQuantizer" and m.quantize.z_channels == 64
    cnn = VQ_models["VQ-16"](semantic_guide="none", detail_guide="none", v_patch_nums=[16], z_channels=32,
                             codebook_embed_dim=8, codebook_size=64)     # ModelArgs default enc/dec type 'cnn'
    keys = set(cnn.state_dict())
    for k in ["encoder.conv_in.weight", "encoder.conv_blocks.0.res.1.conv2.bias", "encoder.conv_blocks.1.res.0.norm1.weight",
              "encoder.conv_blocks.2.res.0.nin_shortcut.weight", "encoder.conv_blocks.3.downsample.conv.weight",
              "encoder.conv_blocks.4.attn.1.proj_out.bias", "encoder.mid.1.q.weight", "encoder.norm_out.weight",
              "decoder.conv_blocks.0.attn.2.k.weight", "decoder.conv_blocks.3.upsample.conv.bias", "decoder.conv_out.weight"]:
        assert k in keys, k
    with torch.no_grad():
        h = cnn.eval().encode(torch.randn(1, 3, 64, 64))
        assert h.shape == (1, 8, 4, 4)
        assert cnn.decode(torch.randn(1, 8, 4, 4)).shape == (1, 3, 64, 64)
    assert cnn.decoder.last_layer is cnn.decoder.conv_out.weight
    m, _ = small_model("VQ-4096", semantic_guide="dinov2")
    assert not any(p.requires_grad for p in m.semantic_model.parameters())
    m.train()
    assert not m.semantic_model.training


def test_cnn_encoder_decoder_match_reference_golden():
    """row a13: same state_dict -> same outputs as the reference's conv Encoder / Decoder (fp32, CPU)."""
    from conftest import load_golden
    from imagefolder_b200.cnn import Decoder, Encoder
    g = load_golden("cnn_small")
    enc = Encoder(ch=32, ch_mult=(1, 2), num_res_blocks=1, z_channels=8).eval()
    dec = Decoder(ch=32, ch_mult=(1, 2), num_res_blocks=1, z_channels=8).eval()
    enc.load_state_dict({k[4:]: torch.tensor(v) for k, v in g.items() if k.startswith("enc.")}, strict=True)
    dec.load_state_dict({k[4:]: torch.tensor(v) for k, v in g.items() if k.startswith("dec.")}, strict=True)
    with torch.no_grad():
        np.testing.assert_allclose(enc(torch.tensor(g["x"])).numpy(), g["h"], rtol=1e-4, atol=1e-5)
        np.testing.assert_allclose(dec(torch.tensor(g["z"])).numpy(), g["y"], rtol=1e-4, atol=1e-5)
