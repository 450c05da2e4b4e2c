"""Config contract of the tokenizer trainer: flat YAML = argparse defaults.

Mirrors tokenizer/tokenizer_image/xqgan_train.py:71-176 (argument names, types, defaults; YAML keys
override defaults, CLI overrides YAML, unknown YAML keys are accepted silently) and :285-313 (which
arguments reach the model -- note codebook_l2_norm / soft_entropy / scale do NOT, SURVEY.md section 0),
plus the latent-perturbation anneal schedule (:62-68, :429-432).
"""
from __future__ import annotations

import argparse
from typing import Dict, Optional, Sequence

import yaml

# name -> (type, default); store_true flags have type bool
_ARGS = {
    "vq_model": (str, "VQ-16"), "ema": ("flag", False), "finetune": ("flag", False),
    "codebook_size": (int, 16384), "codebook_embed_dim": (int, 8), "codebook_l2_norm": ("flag", True),
    "codebook_weight": (float, 1.0), "entropy_loss_ratio": (float, 0.0), "commit_loss_beta": (float, 0.25),
    "reconstruction_weight": (float, 1.0), "perceptual_weight": (float, 1.0), "disc_weight": (float, 0.5),
    "dropout_p": (float, 0.0), "image_size": (int, 256), "epochs": (int, 40), "lr": (float, 1e-4),
    "lr_scheduler": (str, "none"), "weight_decay": (float, 0.0), "beta1": (float, 0.9), "beta2": (float, 0.95),
    "max_grad_norm": (float, 1.0), "global_batch_size": (int, 128), "global_seed": (int, 0),
    "mixed_precision": (str, "bf16"), "enc_type": (str, "cnn"), "dec_type": (str, "cnn"),
    "semantic_guide": (str, "none"), "detail_guide": (str, "none"), "num_latent_tokens": (int, 256),
    "encoder_model": (str, "vit_small_patch14_dinov2.lvd142m"),
    "decoder_model": (str, "vit_small_patch14_dinov2.lvd142m"), "abs_pos_embed": (bool, False),
    "product_quant": (int, 1), "share_quant_resi": (int, 4), "codebook_drop": (float, 0.0), "half_sem": (bool, False),
    "start_drop": (int, 1), "sem_loss_weight": (float, 0.1), "detail_loss_weight": (float, 0.1),
    "enc_tuning_method": (str, "full"), "dec_tuning_method": (str, "full"), "clip_norm": (bool, False),
    "sem_loss_scale": (float, 1.0), "detail_loss_scale": (float, 1.0), "guide_type_1": (str, "class"),
    "guide_type_2": (str, "class"), "lfq": ("flag", False), "end_ratio": (float, 0.5), "anneal_start": (int, 200),
    "anneal_end": (int, 200), "alpha": (float, 0.0), "beta": (float, 0.0), "delta": (int, 100),
}


def make_parser() -> argparse.ArgumentParser:
    p = argparse.ArgumentParser(add_help=False)
    for name, (typ, default) in _ARGS.items():
        flags = ["--" + name, "--" + name.replace("_", "-")] if "_" in name else ["--" + name]
        if typ == "flag":
            p.add_argument(*flags, dest=name, action="store_true", default=default)
        else:
            p.add_argument(*flags, dest=name, type=typ, default=default)
    p.add_argument("--v-patch-nums", "--v_patch_nums", dest="v_patch_nums", type=int, nargs="+",
                   default=[1, 2, 3, 4, 5, 6, 8, 10, 13, 16])
    p.add_argument("--config", type=str, default=None)
    return p


def parse_args(argv: Optional[Sequence[str]] = None, config: Optional[str] = None) -> argparse.Namespace:
    """xqgan_train.py:168-175: YAML -> set_defaults, then re-parse so the CLI wins."""
    argv = list(argv or [])
    parser = make_parser()
    args, _ = parser.parse_known_args(argv)
    path = config or args.config
    if path is not None:
        with open(path, "r", encoding="utf-8") as f:
            file_yaml = yaml.safe_load(f)
        parser.set_defaults(**file_yaml)
        args, _ = parser.parse_known_args(argv)
    return args


def model_kwargs(args) -> Dict:
    """the subset of arguments forwarded to VQ_models[...](...)  (xqgan_train.py:285-313)."""
    names = ["codebook_size", "codebook_embed_dim", "commit_loss_beta", "entropy_loss_ratio", "dropout_p",
             "v_patch_nums", "enc_type", "encoder_model", "dec_type", "decoder_model", "semantic_guide",
             "detail_guide", "num_latent_tokens", "abs_pos_embed", "share_quant_resi", "product_quant",
             "codebook_drop", "half_sem", "start_drop", "sem_loss_weight", "detail_loss_weight", "clip_norm",
             "sem_loss_scale", "detail_loss_scale", "guide_type_1", "guide_type_2", "lfq"]
    return {n: getattr(args, n) for n in names}


def build_vq_model(args, **overrides):
    from .xqgan_model import VQ_models
    kw = model_kwargs(args)
    kw.update(overrides)
    kw["v_patch_nums"] = list(kw["v_patch_nums"])
    return VQ_models[args.vq_model](**kw)


def get_random_ratio(randomness_anneal_start, randomness_anneal_end, end_ratio, cur_step):
    """xqgan_train.py:62-68."""
    if cur_step < randomness_anneal_start:
        return 1.0
    elif cur_step > randomness_anneal_end:
        return end_ratio
    return 1.0 - (cur_step - randomness_anneal_start) / (randomness_anneal_end - randomness_anneal_start) * end_ratio


def perturbation_schedule(args, epoch: int):
    """(alpha, beta, delta) for this epoch  (xqgan_train.py:429-432)."""
    ratio = get_random_ratio(args.anneal_start, args.anneal_end, args.end_ratio, epoch)
    return ratio * args.alpha, args.beta, int(ratio * args.delta)


# model-relevant keys of the reference's configs/*.yaml (kept as data so tests can materialise the
# YAMLs without the reference tree; tests/test_model_cpu.py checks them against tests/golden/reference_configs.json)
_COMMON = dict(image_size=256, vq_model="VQ-16", enc_type="dinov2", dec_type="dinov2", semantic_guide="dinov2",
               global_batch_size=1024, epochs=200, lr_scheduler="cosine", lr=3e-5, abs_pos_embed=True, ema=True,
               encoder_model="vit_base_patch14_dinov2.lvd142m", decoder_model="vit_base_patch14_dinov2.lvd142m",
               start_drop=3, sem_loss_weight=0.1, enc_tuning_method="full")
_MS = dict(product_quant=2, codebook_drop=0.1, num_latent_tokens=121, v_patch_nums=[1, 1, 2, 3, 3, 4, 5, 6, 8, 11],
           half_sem=True)
_BSQ = dict(detail_guide="sam", entropy_loss_ratio=0.1, clip_norm=True, codebook_l2_norm=True, soft_entropy=True,
            scale=1.0, lfq=True)
SHIPPED_CONFIGS = {
    "VQ-4096": dict(_COMMON, codebook_embed_dim=64, codebook_size=4096, product_quant=1, codebook_drop=0.0,
                    num_latent_tokens=256, v_patch_nums=[16], half_sem=False, guide_type_1="class"),
    "VQ-8192": dict(_COMMON, codebook_embed_dim=32, codebook_size=8192, product_quant=1, codebook_drop=0.0,
                    num_latent_tokens=256, v_patch_nums=[16], half_sem=False, guide_type_1="class"),
    "RobustTok": dict(_COMMON, codebook_embed_dim=64, codebook_size=4096, product_quant=1, codebook_drop=0.0,
                      num_latent_tokens=256, v_patch_nums=[16], half_sem=False, guide_type_1="class",
                      anneal_start=40, anneal_end=120, alpha=1.0, beta=0.1, delta=100),
    "VP2-4096": dict(_COMMON, codebook_embed_dim=32, codebook_size=4096, product_quant=2, codebook_drop=0.1,
                     num_latent_tokens=256, v_patch_nums=[16], half_sem=True),
    "VP2-16384": dict(_COMMON, codebook_embed_dim=32, codebook_size=16384, product_quant=2, codebook_drop=0.1,
                      num_latent_tokens=256, v_patch_nums=[16], half_sem=True),
    "MSVR10P2-4096": dict(**_COMMON, **_MS, codebook_embed_dim=32, codebook_size=4096),
    "MSVR10P2-8192": dict(**_COMMON, **_MS, codebook_embed_dim=32, codebook_size=8192),
    "MSVR10P2-16384": dict(**_COMMON, **_MS, codebook_embed_dim=32, codebook_size=16384),
    "MSBR10P2-4096": dict(**_COMMON, **_MS, **_BSQ, codebook_embed_dim=12, codebook_size=4096),
    "MSBR10P2-16384": dict(**_COMMON, **_MS, **_BSQ, codebook_embed_dim=14, codebook_size=16384),
}
