#!/usr/bin/env python
"""bench.py -- tokenizer training throughput (images/sec at 256x256) + VQ-argmin roofline.

    python bench.py --gpus 1 --steps 8 --warmup 3                    # our arm (CUDA path)
    python bench.py --impl reference --gpus 1 --steps 2 --warmup 1   # CPU arm: the oracle port
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N ... # one rank per GPU (NCCL)
    python bench.py --gpus 1 --steps 8 --warmup 3 --dump-outputs DIR # + the last timed step's outputs as DIR/*.npy

Workload (BASELINE.json configs[1]): VQ-8192 tokenizer training, bf16 autocast, per-GPU batch 256,
256x256 synthetic images, random-init ViT-B encoder/decoder.  One step = VQModel forward
(encode -> quantize -> latent perturbation -> decode) + L2 reconstruction/vq/commit losses + backward
+ AdamW (+ DDP gradient all-reduce for N > 1): the body of xqgan_train.py:448-462 restricted to the
in-scope path (no LPIPS / discriminator / frozen teacher, whose weights cannot be downloaded here --
BASELINE.md section 3).  Weak scaling: per-GPU batch is fixed.

Prints ONE JSON line (rank 0).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOAD = "VQ-8192"
METRIC = "tokenizer_train_images_per_sec_256x256"


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=6)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", type=str, default="ours", choices=["ours", "reference", "eager"],
                   help="ours: libxqb200 path; reference: CPU oracle port (the contract's reference arm); eager: the "
                        "reference's way of computing the path in plain PyTorch on the SAME GPU (extra, informative)")
    p.add_argument("--workload", type=str, default=WORKLOAD)
    p.add_argument("--batch", type=int, default=256, help="per-GPU batch")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-extra", action="store_true", help="skip the MSVR10P2-4096 ours-vs-eager extra measurement")
    p.add_argument("--fp32-grads", action="store_true", help="multi-GPU: all-reduce fp32 gradient buckets (stock DDP) instead of bf16")
    p.add_argument("--cpu-sample", type=int, default=0, help="images per CPU-baseline step (0 = auto)")
    p.add_argument("--dump-outputs", type=str, default=None, metavar="DIR",
                   help="write what the last timed step computed (losses, reconstruction, tokens, gradients, updated "
                        "weights; fixed seeded samples of the large ones) as DIR/<name>.npy, to compare two builds")
    a = p.parse_args()
    if a.steps < 1 or a.warmup < 0:
        p.error("--steps must be >= 1 and --warmup >= 0")
    if a.dump_outputs is not None and a.impl == "reference":
        p.error("--dump-outputs writes what a GPU arm computed: use it with --impl ours or eager")
    return a


# ----------------------------------------------------------------------------------------------
def build_model(workload: str, device):
    from imagefolder_b200 import config as xcfg
    cfg = dict(xcfg.SHIPPED_CONFIGS[workload])
    cfg.update(semantic_guide="none", detail_guide="none")  # teachers need downloaded weights (out of scope)
    args = xcfg.parse_args([])
    for k, v in cfg.items():
        setattr(args, k, v)
    torch.manual_seed(0)
    model = xcfg.build_vq_model(args)
    return model.to(device), args


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "200"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# C-ABI entry point -> the kernel that dominates it (the name ncu reports; key of profiles/ncu_traffic.json)
ENTRY_MAIN_KERNEL = {"xq_vit_attn_bwd": "attn_bwd_kernel", "xq_vit_attn_fwd": "attn_fwd_kernel",
                     "xq_vit_residual_ln_bwd": "residual_ln_bwd_kernel", "xq_vit_residual_ln_fwd": "residual_ln_fwd_kernel",
                     "xq_vit_gelu_fwd": "gelu_fwd_kernel", "xq_vit_gelu_bwd": "gelu_bwd_kernel",
                     "xq_vit_fc1_gelu_fwd": "mlp_gemm_kernel_fwd", "xq_vit_fc2_dgelu_bwd": "mlp_gemm_kernel_bwd"}


def top_kernel_roofline(kern_table, hbm_peak, tf_peak, step_ms, ncu_traffic=None, src="measured"):
    """Roofline of the libxqb200 entry point that takes the most time per step -- the dominant kernel of ours (the VQ search
    kernel that BASELINE's metric names is two orders of magnitude smaller than the attention / ViT glue kernels).  An entry
    with tensor FLOPs is placed against both roofs and reported against the one it sits closer to (the binding one)."""
    rows = [r for r in kern_table if r.get("alg_GBps")]
    if not rows:
        return None
    top = max(rows, key=lambda r: r["ms_per_step"])
    hbm_frac = top["alg_GBps"] / hbm_peak
    out = {"kernel": top["entry"], "ms_per_call": top["ms_per_call"], "calls_per_step": top["calls_per_step"],
           "share_of_step": top["ms_per_step"] / step_ms if step_ms else None,
           "traffic": (ncu_traffic or {}).get(ENTRY_MAIN_KERNEL.get(top["entry"], top["entry"]), (ncu_traffic or {}).get(top["entry"])),
           "main_kernel": ENTRY_MAIN_KERNEL.get(top["entry"]), "peak_source": src,
           "algorithmic_bytes": top["alg_bytes_per_call"], "hbm_gbs": top["alg_GBps"], "hbm_frac": hbm_frac}
    if top.get("alg_TFps") and top["alg_TFps"] / tf_peak >= hbm_frac:
        out.update({"bound": "tensor", "achieved": top["alg_TFps"], "peak": tf_peak, "unit": "TFLOP/s",
                    "frac": top["alg_TFps"] / tf_peak, "algorithmic_flops": top["alg_flops_per_call"]})
    else:
        out.update({"bound": "hbm", "achieved": top["alg_GBps"], "peak": hbm_peak, "unit": "GB/s", "frac": hbm_frac})
        if top.get("alg_TFps"):
            out.update({"tensor_tfs": top["alg_TFps"], "tensor_frac": top["alg_TFps"] / tf_peak})
    out["note"] = ("algorithmic bytes / FLOPs (each call's operands once; attention: 4 B H N^2 d forward, 10 B H N^2 d backward) / "
                   "CUDA-event time of the C-ABI call inside the timed steps, helper launches of the call (pre-pass, accumulator "
                   "conversion, memsets) included; traffic = dram bytes of the call's main kernel from the ncu capture keyed by "
                   "entry + workload in profiles/ncu_traffic.json (null when that shape was not captured)")
    return out


def _safe(fn):
    try:
        return fn()
    except Exception as e:          # an explanatory extra must never cost the bench line
        return {"error": repr(e)[:200]}


def peaks():
    """(HBM GB/s, dense bf16 TFLOP/s, source).  Every kernel bench.py times sits inside a long training step, so the tensor
    roof is the SUSTAINED cuBLAS figure of MEASURED_PEAKS.json (the burst one is for a kernel timed alone)."""
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        if "bf16_tflops_sustained" in d:
            return d.get("hbm_gbs", 6650.0), d["bf16_tflops_sustained"], "measured (MEASURED_PEAKS.json: hbm_gbs, bf16_tflops_sustained)"
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops", 1590.0), "measured (MEASURED_PEAKS.json: hbm_gbs, bf16_tflops)"
    return 6650.0, 1590.0, "fallback (B200_PROFILING.md)"


# ----------------------------------------------------------------------------------------------
class Ctx:
    """process-wide state shared by every measurement of this run (one process per GPU)."""

    def __init__(self):
        import torch.distributed as dist
        self.dist = dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py (impl=ours) needs a CUDA device: there is no CPU fallback")
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        torch.backends.cuda.matmul.allow_tf32 = True   # xqgan_train.py:5-6
        torch.backends.cudnn.allow_tf32 = True

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(self, *vals):
        t = torch.tensor(list(vals), device=self.dev, dtype=torch.float64)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(x) for x in t]


def make_step(ctx, workload, B, impl, keep_last=False):
    """model + optimizer + the training-step closure of one workload (the body of xqgan_train.py:448-462 restricted to
    the in-scope path).  impl 'eager' = the reference's way of computing the path in plain PyTorch on the same GPU.
    keep_last: the closure keeps the forward outputs of its latest call in `step.last` (for --dump-outputs)."""
    import torch.nn.functional as F
    from imagefolder_b200 import config as xcfg
    model, margs = build_model(workload, ctx.dev)
    model.train()
    fwd_module = model
    if impl == "eager":
        from oracle.eager_ref import EagerTokenizer   # baseline leg only: reference-style eager ops, no libxqb200
        fwd_module = EagerTokenizer(model)
    net = fwd_module
    if ctx.world > 1:
        # gradients are the only collective on the critical path (SURVEY.md section 8e).  bf16 buckets halve the bytes NCCL moves
        # through the HBM the glue kernels are streaming from (the master weights / AdamW state stay fp32); `--fp32-grads`
        # restores stock DDP.  The eager arm keeps stock DDP: it is the reference's configuration (xqgan_train.py:412).
        net = torch.nn.parallel.DistributedDataParallel(fwd_module, device_ids=[ctx.local], gradient_as_bucket_view=True,
                                                        bucket_cap_mb=100)
        if impl == "ours" and not getattr(ctx, "fp32_grads", False):
            from torch.distributed.algorithms.ddp_comm_hooks import default_hooks
            net.register_comm_hook(None, default_hooks.bf16_compress_hook)
    opt = torch.optim.AdamW(model.parameters(), lr=3e-5, betas=(0.9, 0.95), weight_decay=0.0, fused=True)
    alpha, beta, delta = xcfg.perturbation_schedule(margs, 0)

    def step(x):
        with torch.autocast("cuda", dtype=torch.bfloat16):
            dec, (vq, commit, ent, usages), _, _, _ = net(x, 0, alpha, beta, delta)
            loss = F.mse_loss(dec.float(), x) + vq + commit + ent
        opt.zero_grad(set_to_none=True)
        loss.backward()
        opt.step()
        if keep_last:
            step.last = {"loss": loss, "vq_loss": vq, "commit_loss": commit, "entropy_loss": ent,
                         "codebook_usage": usages, "reconstruction": dec}
        return loss

    g = torch.Generator(device=ctx.dev).manual_seed(1234 * ctx.world + ctx.rank)
    imgs_dev = torch.rand(B, 3, 256, 256, device=ctx.dev, generator=g) * 2 - 1
    return model, margs, step, imgs_dev


def time_resident(ctx, step, imgs_dev, steps, warmup, collect_kernels=False):
    """W warm-up steps, then exactly K steps bracketed by barrier + synchronize, CUDA events on the launching stream."""
    from imagefolder_b200 import _capi
    for _ in range(warmup):
        step(imgs_dev)
    ctx.barrier()
    if collect_kernels:
        _capi.TIMING = {}
    _capi.LAUNCHES[0] = 0
    ctx.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step(imgs_dev)
    e1.record()
    ctx.barrier()
    ms = e0.elapsed_time(e1)
    timing, _capi.TIMING = _capi.TIMING, None
    return ms, _capi.LAUNCHES[0], (timing or {})


def kernel_table(timing, steps):
    rows = []
    for name, evs in timing.items():
        tot = sum(t[0].elapsed_time(t[1]) for t in evs)
        nb = sum(t[2] for t in evs)
        nf = sum(t[3] for t in evs)
        rows.append({"entry": name, "calls_per_step": len(evs) / steps, "ms_per_step": tot / steps,
                     "ms_per_call": tot / len(evs), "alg_GBps": (nb / (tot * 1e-3) / 1e9) if nb else None,
                     "alg_TFps": (nf / (tot * 1e-3) / 1e12) if nf else None,
                     "alg_bytes_per_call": nb / len(evs), "alg_flops_per_call": nf / len(evs)})
    rows.sort(key=lambda r: -r["ms_per_step"])
    return rows


def dump_outputs(out_dir, model, last):
    """--dump-outputs: what the last timed step handed its caller, as DIR/<name>.npy -- the losses and codebook usages
    (float64), the reconstruction (float32), every quantizer's token indices (float64, exact), and the gradients and
    AdamW-updated weights of all parameters in model.parameters() order (float32).  The reconstruction, gradients and
    weights are samples at fixed seeded positions (about 33 MB in all at batch 256), the same for every run."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)

    def save(name, t, dtype):
        arr = t.detach().cpu().numpy() if torch.is_tensor(t) else np.asarray(t)
        np.save(os.path.join(out_dir, name + ".npy"), arr.astype(dtype))

    def sample(flat, n):
        if flat.numel() <= n:
            return flat
        pos = np.sort(np.random.default_rng(0).choice(flat.numel(), n, replace=False))
        return flat[torch.from_numpy(pos).to(flat.device)]

    for k in ("loss", "vq_loss", "commit_loss", "entropy_loss"):
        save(k, torch.as_tensor(last[k]), np.float64)
    save("codebook_usage", [float(u) for u in last["codebook_usage"]], np.float64)
    dec = last["reconstruction"]
    save("reconstruction", sample(dec.float().reshape(-1), 1 << 22), np.float32)
    tokens = []
    for q in model._quantizers():
        if hasattr(q, "last_idx_Bl"):
            tokens.append(torch.cat([t.reshape(dec.shape[0], -1) for t in q.last_idx_Bl], 1))
        elif hasattr(q, "last_idx"):
            tokens.append(q.last_idx.reshape(dec.shape[0], -1))
    if tokens:
        save("tokens", torch.cat(tokens, 1), np.float64)
    params = list(model.parameters())
    grads = torch.cat([(p.grad if p.grad is not None else torch.zeros_like(p)).float().reshape(-1) for p in params])
    save("grads", sample(grads, 1 << 21), np.float32)
    del grads
    save("params", sample(torch.cat([p.detach().float().reshape(-1) for p in params]), 1 << 21), np.float32)


def ncu_traffic_table():
    """dram bytes per launch keyed by kernel name, read from the committed ncu summaries (profiles/ncu_traffic.json,
    written by tools/ncu_summarize.py from the .ncu-rep captures); None when a kernel / shape has no capture."""
    path = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    try:
        return json.load(open(path))
    except Exception:
        return {}


def quantizer_roofline(workload, margs, B, kern_ms, entry, hbm, tf, src):
    """Roofline object of the quantizer kernel the metric names, per workload (SURVEY.md section 8d):
       VQ / VP2  -> tensor roof of the contraction 2*rows*V*C   (vq_search_tc_kernel)
       MSVR      -> same contraction summed over the 10 scales, plus the 10-step dependent-chain note (ms_forward_kernel)
       MSBR      -> HBM roof of the streaming BSQ kernels (no contraction: a sign test)."""
    if not kern_ms:
        return None
    C, V = margs.codebook_embed_dim, margs.codebook_size
    pq = margs.product_quant
    multi = len(margs.v_patch_nums) > 1
    rows_branch = B * (sum(p * p for p in margs.v_patch_nums) if multi else margs.num_latent_tokens // pq)
    hw = margs.v_patch_nums[-1] ** 2 if multi else margs.num_latent_tokens // pq
    traffic = ncu_traffic_table()
    if getattr(margs, "lfq", False):
        # per branch: read f, write f_hat (fp32 [B,C,H,W]) + int64 indices + Phi weights
        bytes_alg = 2 * B * C * hw * 4 + rows_branch * 8 + 4 * (C * C * 9 + C) * 4
        gbs = bytes_alg / (kern_ms * 1e-3) / 1e9
        return {"bound": "hbm", "kernel": "ms_forward_kernel (BSQ mode) + bsq_entropy kernels; timed = one xq_ms_forward call (one PQ branch)",
                "achieved": gbs, "peak": hbm, "unit": "GB/s", "frac": gbs / hbm,
                "traffic": traffic.get(f"ms_forward_kernel/{workload}/B{B}"), "peak_source": src, "kernel_ms": kern_ms,
                "algorithmic_bytes": bytes_alg,
                "note": "implicit codebook (sign test): no contraction, pure streaming; the kernel is a 10-step dependent chain "
                        "per image, so latency x 10 bounds it before HBM does"}
    bytes_alg = rows_branch * C * 4 + V * C * 4 + rows_branch * 8 + rows_branch * C * 4
    if multi:
        bytes_alg = 2 * B * C * hw * 4 + rows_branch * 8 + V * C * 4 + 4 * (C * C * 9 + C) * 4
    flops_alg = 2.0 * rows_branch * V * C
    gbs = bytes_alg / (kern_ms * 1e-3) / 1e9
    tfs = flops_alg / (kern_ms * 1e-3) / 1e12
    if multi:
        name = "ms_forward_kernel (fused 10-scale residual loop in shared memory, FP32 search); timed = one xq_ms_forward call (one PQ branch)"
        note = ("10 DEPENDENT scales per image: latency x 10 bounds the kernel; the per-scale searches are CUDA-core FP32 "
                "(DESIGN.md section 9), so the tensor fraction is reported against the contraction's roof, not achieved on tensor cores")
        tkey = f"ms_forward_kernel/{workload}/B{B}"
    else:
        tc = (C in (32, 64)) and os.environ.get("XQ_VQ_ALGO", "auto")[0] != "e"
        name = ("vq_search_tc_kernel (tcgen05 TF32 screening + exact fp32 rescoring)" if tc else
                "vq_search_kernel (exact fp32 CUDA-core)") + "; timed = the xq_vq_forward call (codebook prep + search + loss finalize)"
        note = "contraction-bound, not HBM-bound (arithmetic intensity ~1900 FLOP/B, DESIGN.md section 5)"
        tkey = f"vq_search_tc_kernel/N{rows_branch}/V{V}/C{C}"
    out = {"bound": "tensor", "kernel": name, "achieved": tfs, "peak": tf, "unit": "TFLOP/s", "frac": tfs / tf,
           "traffic": traffic.get(tkey), "peak_source": src + " (dense bf16 cuBLAS; no TF32 peak is measured on this pool)",
           "kernel_ms": kern_ms, "algorithmic_flops": flops_alg, "algorithmic_bytes": bytes_alg, "hbm_gbs": gbs,
           "hbm_frac": gbs / hbm, "note": note + "; traffic = dram bytes/launch from the committed ncu capture of this "
           "kernel + shape (profiles/ncu_traffic.json), null when that shape was not captured"}
    if not multi:
        # TMEM -> register read floor of the tcgen05 path: every approximate score (N*V fp32) crosses the tcgen05.ld port once
        out["tmem_read_floor_ms"] = rows_branch * V * 4 / (125.0 * 148 * 1.9e9) * 1e3
    return out


def extra_msvr(ctx, a):
    """The north star's second target, made driver-visible: MSVR10P2-4096 at per-GPU batch 128, this framework vs the
    reference's own way of computing the path in PyTorch eager, on the SAME ranks, back to back."""
    import gc
    res = {}
    for impl, steps, warm in (("ours", 3, 2), ("eager", 2, 1)):
        model, margs, step, imgs = make_step(ctx, "MSVR10P2-4096", 128, impl)
        ms, launches, timing = time_resident(ctx, step, imgs, steps, warm, collect_kernels=(impl == "ours"))
        (ms,) = ctx.max_over_ranks(ms)
        res[impl] = {"img_s": ctx.world * 128 * steps / (ms * 1e-3), "ms_per_step": ms / steps, "steps": steps, "warmup": warm}
        if impl == "ours":
            res["ours"]["gpu_launches"] = launches
            if "xq_ms_forward" in timing:
                ts = [t[0].elapsed_time(t[1]) for t in timing["xq_ms_forward"]]
                hbm, tf, src = peaks()
                res["roofline"] = quantizer_roofline("MSVR10P2-4096", margs, 128, sum(ts) / len(ts), "xq_ms_forward", hbm, tf, src)
        del model, step, imgs, timing
        gc.collect()
        torch.cuda.empty_cache()
    return {"workload": "MSVR10P2-4096 tokenizer training step, per-GPU batch 128, 256x256, ViT-B enc/dec (same step "
                        "definition as the headline)",
            "msvr_img_s": res["ours"]["img_s"], "msvr_eager_img_s": res["eager"]["img_s"],
            "msvr_speedup": res["ours"]["img_s"] / res["eager"]["img_s"], "ours": res["ours"], "eager": res["eager"],
            "roofline": res.get("roofline"),
            "note": "eager = oracle/eager_ref.EagerTokenizer: the reference's op sequence (materialised N x V distances, per-scale "
                    "Python loop, .item() usage syncs, SDPA + unfused ViT glue) in PyTorch eager with bf16 autocast"}


def run_ours(a):
    import gc
    from imagefolder_b200 import _capi, vit_ops
    ctx = Ctx()
    ctx.fp32_grads = a.fp32_grads
    world, rank, local, dev = ctx.world, ctx.rank, ctx.local, ctx.dev
    model, margs, step, imgs_dev = make_step(ctx, a.workload, a.batch, a.impl, keep_last=a.dump_outputs is not None)
    B = a.batch
    imgs_host = imgs_dev.cpu().pin_memory()
    barrier = ctx.barrier

    for _ in range(a.warmup):
        step(imgs_dev)
    barrier()
    torch.cuda.reset_peak_memory_stats()
    # a generation-2 Python GC pass over the module / autograd heap takes hundreds of ms and, when it lands inside a
    # timed region, drains the launch queue: collect now and keep the collector off until both regions are done
    gc.collect()
    gc.disable()

    # ---- timed region 1: inputs resident in HBM
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    ms, launches, timing = time_resident(ctx, step, imgs_dev, a.steps, 0, collect_kernels=True)
    kern_ms, kern_entry = None, None
    for entry in ("xq_vq_forward", "xq_ms_forward"):
        if entry in timing:
            ts = [t[0].elapsed_time(t[1]) for t in timing[entry]]
            kern_ms, kern_entry = sum(ts) / len(ts), entry
            break
    kern_table = kernel_table(timing, a.steps)
    timing.clear()          # release the CUDA events before the next region
    if a.impl == "ours" and vit_ops.ATTN_TC_ENABLED[0]:
        # the fused path must be the one that ran (a silent library fallback would hide behind the step time)
        names = {r["entry"] for r in kern_table}
        want = {"xq_vit_attn_fwd", "xq_vit_attn_bwd", "xq_vit_residual_ln_fwd"}
        want |= {"xq_vit_fc1_gelu_fwd", "xq_vit_fc2_dgelu_bwd"} if vit_ops.MLP_TC_ENABLED[0] else {"xq_vit_gelu_fwd"}
        assert want <= names, names

    # ---- timed region 2: end to end through the public API with HOST buffers
    # one-off setup outside the clock (a data loader allocates its pinned buffers and copy stream once; cudaHostAlloc
    # under a loaded GPU was measured to stall 150-700 ms here)
    copy_stream = torch.cuda.Stream(device=dev)
    loss_pinned = torch.empty(a.steps, dtype=torch.float32).pin_memory()
    # every step: H2D of ITS inputs from pinned memory (prefetched on a copy stream while the previous step computes,
    # as a data loader does) and a D2H read of ITS loss (async into pinned memory; synchronised before the clock stops)

    def prefetch():
        with torch.cuda.stream(copy_stream):
            xb = imgs_host.to(dev, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(copy_stream)
        return xb, ev

    # one untimed pass through this path (the first use of the copy stream / the first pinned->device DMA of a process was
    # measured at ~100 ms on a 2-GPU box; it is a warm-up cost like the W compute steps above)
    xw, evw = prefetch()
    torch.cuda.current_stream().wait_event(evw)
    xw.record_stream(torch.cuda.current_stream())
    loss_pinned[0:1].copy_(step(xw).detach().float().reshape(1), non_blocking=True)
    del xw
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    nxt = prefetch()
    marks = [torch.cuda.Event(enable_timing=True) for _ in range(a.steps)]
    for i in range(a.steps):
        x, ev = nxt
        torch.cuda.current_stream().wait_event(ev)
        x.record_stream(torch.cuda.current_stream())
        if i + 1 < a.steps:
            nxt = prefetch()
        loss = step(x)
        loss_pinned[i:i + 1].copy_(loss.detach().float().reshape(1), non_blocking=True)
        marks[i].record()
    f1.record()
    barrier()
    loss_host = float(loss_pinned[-1])
    ms_e2e = f0.elapsed_time(f1)
    e2e_steps = [round(([f0] + marks)[i].elapsed_time(marks[i]), 2) for i in range(a.steps)]
    gc.enable()
    clk = clocks.stop() if rank == 0 else None
    if a.dump_outputs is not None and rank == 0:
        dump_outputs(a.dump_outputs, model, step.last)

    ms, ms_e2e = ctx.max_over_ranks(ms, ms_e2e)
    peak_mem = torch.cuda.max_memory_allocated() / 2 ** 30

    extra = None
    if a.impl == "ours" and not a.no_extra:
        # free the headline model before the second workload (all ranks take part: DDP collectives inside)
        state_for_cpu = {k: v.detach().cpu() for k, v in model.state_dict().items()} if (rank == 0 and world == 1 and not a.no_cpu_baseline) else None
        cfg_for_cpu = model.config
        del step, imgs_dev
        model = None
        gc.collect()
        torch.cuda.empty_cache()
        extra = _safe(lambda: extra_msvr(ctx, a))
    else:
        state_for_cpu, cfg_for_cpu = (model.state_dict(), model.config)
    if rank != 0:
        if world > 1:
            ctx.dist.destroy_process_group()
        return
    hbm, tf, src = peaks()
    qroof = quantizer_roofline(a.workload, margs, B, kern_ms, kern_entry, hbm, tf, src)
    # headline roofline = the dominant kernel of ours inside the timed steps; the quantizer kernel BASELINE's metric names
    # keeps its own object (`roofline_quantizer`) -- it is ~0.1 % of the step
    roof = _safe(lambda: top_kernel_roofline(
        kern_table, hbm, tf, ms / a.steps,
        {k.split("/")[0]: v for k, v in ncu_traffic_table().items() if k.endswith(f"/{a.workload}/B{B}")}, src)) or qroof
    if a.impl == "eager":
        roof = qroof = None
    out = {
        "impl": "ours" if a.impl == "ours" else "eager_gpu",
        "metric": METRIC, "value": world * B * a.steps / (ms * 1e-3), "unit": "images/s", "n_gpus": world,
        "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms / a.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": workload_config(a, world),
        "e2e": {"value": world * B * a.steps / (ms_e2e * 1e-3), "unit": "images/s",
                "h2d_bytes_per_step": imgs_host.numel() * 4, "d2h_bytes_per_step": 4, "ms_per_step": ms_e2e / a.steps,
                "step_ms": e2e_steps},
        "gpu_launches": launches, "clocks": clk, "roofline": roof, "peak_mem_gib": peak_mem,
        "our_kernels": [dict(r, hbm_frac=(r["alg_GBps"] / hbm if r["alg_GBps"] else None)) for r in kern_table],
        "our_kernels_ms_per_step": sum(r["ms_per_step"] for r in kern_table),
        "roofline_quantizer": qroof,
        "last_loss": loss_host, "extra": extra,
        "parity_note": "token indices are bit-exact against the reference's CPU fp32 path except on provable near-ties "
                       "(top-2 margin < 1e-5; counted in tests/test_gpu_quantizers.py::test_msvr_unscreened_seed_counts_mismatches_on_gpu)",
    }
    if not a.no_cpu_baseline and world == 1 and a.impl == "ours":
        out["cpu_baseline"] = cpu_arm(a, steps=1, warmup=0, state=state_for_cpu, margs=cfg_for_cpu)
    print(json.dumps(out), flush=True)
    if world > 1:
        ctx.dist.destroy_process_group()


# ----------------------------------------------------------------------------------------------
def cpu_arm(a, steps, warmup, state=None, margs=None, budget_s=14.0):
    """the oracle port of the same training step on the host cores (bounded sample: about `budget_s` seconds of
    CPU work per timed step, so the whole arm ends within minutes whatever --steps is)."""
    from oracle import vit_ref, xq_oracle as xo
    import torch.nn.functional as F  # noqa: F401
    # measured on the B200 host (128-core Xeon 8562Y+, tools/cpu_probe.py): 16 threads 1.10 img/s, 32 -> 1.05,
    # 64 -> 0.53, 128 -> pathological (> 90 s/step): the step's small GEMMs do not scale past ~16-32 threads
    cores = min(os.cpu_count() or 1, 16)
    torch.set_num_threads(cores)
    xo.set_num_threads(cores)
    if state is None:
        model, _ = build_model(a.workload, "cpu")
        state, margs = model.state_dict(), model.config
    cfg = vit_ref.cfg_from_model_args(margs)
    ref = vit_ref.RefTokenizer(state, cfg, requires_grad=True)
    opt = torch.optim.AdamW(ref.parameters(), lr=3e-5, betas=(0.9, 0.95), weight_decay=0.0)
    n = a.cpu_sample
    g = torch.Generator().manual_seed(7)
    SN = len(cfg["v_patch_nums"])
    if n <= 0:  # size the sample for ~10-20 s per step
        x = torch.rand(2, 3, 256, 256, generator=g) * 2 - 1
        t0 = time.time()
        ref.train_step(x, opt, dropout=torch.randint(3, SN + 1, (2,)).numpy() if SN > 1 else None)
        per_img = (time.time() - t0) / 2
        n = int(max(2, min(32, budget_s / max(per_img, 1e-3))))
    x = torch.rand(n, 3, 256, 256, generator=g) * 2 - 1
    dr = torch.randint(3, SN + 1, (n,)).numpy() if SN > 1 else None
    for _ in range(warmup):
        ref.train_step(x, opt, dr)
    t0 = time.time()
    for _ in range(steps):
        ref.train_step(x, opt, dr)
    dt = time.time() - t0
    return {"value": n * steps / dt, "unit": "images/s", "cores": cores, "kind": "port",
            "sample": f"{n} images/step x {steps} step(s) of the {a.workload} training step (fp32, torch CPU ViT + "
                      f"C oracle quantizer), {dt:.1f} s", "ms_per_step": dt / steps * 1e3}


def workload_config(a, world):
    """the `config` object of a bench line: both arms print the SAME object for the same command line (the reference arm times a
    bounded sample of this workload on the host cores and says so in its `cpu_baseline.sample` / `note`)"""
    B = a.batch
    return {"workload": f"{a.workload} tokenizer training step, per-GPU batch {B}, 256x256, ViT-B enc/dec, "
                        "fwd+bwd+AdamW, L2+vq+commit loss (no LPIPS/GAN/teacher)",
            "global_batch": world * B, "parallelism": f"dp{world}",
            "grad_allreduce": ("none (1 GPU)" if world == 1 else ("fp32 buckets" if a.fp32_grads else "bf16-compressed buckets (fp32 master weights)")),
            "l2_policy": "inputs (201 MB/step) + activations exceed the 126 MB L2"}


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    total = max(1, a.steps) + min(a.warmup, 1)
    base = cpu_arm(a, steps=max(1, a.steps), warmup=min(a.warmup, 1), budget_s=max(2.0, 150.0 / total))
    out = {"impl": "reference", "metric": METRIC, "value": base["value"], "unit": "images/s",
           "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": base["ms_per_step"],
           "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": workload_config(a, max(1, a.gpus)),
           "note": "host-core arm: the oracle port of the reference path (torch-CPU ViT + C oracle quantizer, fp32) on a bounded "
                   "sample of the workload above; the reference itself is Python + un-vendored timm and cannot travel.  Rank 0 "
                   "only; the GPU-specific config keys describe the arm it is compared with",
           "cpu_baseline": base,
           "e2e": {"value": base["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    args = parse()
    os.environ.setdefault("OMP_WAIT_POLICY", "PASSIVE")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)
