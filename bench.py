#!/usr/bin/env python
"""bench.py — headline benchmark of the B200-native SimpleTuner training step.

Workload (BASELINE.json configs[1]): Flux.1-dev (19 double + 38 single MMDiT blocks, D=3072, 24x128 heads,
guidance-distilled) LoRA rank 16 on all attention projections, bf16, 1024x1024 images as cached latents
[B,16,128,128] + cached T5 embeds [B,512,4096] + pooled CLIP [B,768], batch 4 per GPU.  Weights are
random-init of that architecture and data is synthetic (no network): said in `data`.

One "step" = prepare_batch (noise + sigma sampling + noisy latents + patchify) -> model_predict
(transformer forward) -> loss -> backward (dgrad through all 57 blocks + LoRA wgrad) -> value clip ->
AdamW step on the LoRA parameters.  `value` is measured with the batch already resident in HBM; `e2e`
runs the same public API (`TrainStep.__call__`) from PINNED HOST buffers, with the host->device copy
of the batch and a device->host read of the loss inside the timed region every step.

`--impl reference` times the reference path's CPU restatement (oracle/flux_oracle.py, "port": the
reference itself needs diffusers/accelerate/peft which are not installable here) on the host cores.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

import torch  # noqa: E402

METRIC = "images/sec Flux.1-dev LoRA bf16 1024^2"
UNIT = "images/s"

# Flux.1-dev geometry and the algorithmic work of one training sample (BASELINE.md §3, SURVEY.md §8d)
FLUX_DEV = dict(in_channels=64, num_layers=19, num_single_layers=38, attention_head_dim=128, num_attention_heads=24,
                joint_attention_dim=4096, pooled_projection_dim=768, guidance_embeds=True, axes_dims_rope=(16, 56, 56))
S_IMG, S_TXT, D_MODEL = 4096, 512, 3072
TF_FWD_LINEAR = 57 * (S_IMG + S_TXT) * 24 * D_MODEL ** 2 * 1e-12 * 1.0   # 59.5 TF  (2*M*N*K summed = tokens * 24 D^2)
TF_FWD_ATTN = 57 * 4 * (S_IMG + S_TXT) ** 2 * D_MODEL * 1e-12            # 14.9 TF
TF_STEP_SAMPLE = (TF_FWD_LINEAR + TF_FWD_ATTN) + TF_FWD_LINEAR + 2 * TF_FWD_ATTN  # 163.6 TF (LoRA: fwd + dgrad + attn bwd)


def measured_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return d, "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.rows = []
        self._stop = threading.Event()
        self._t = None

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.idx)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self._stop.wait(0.2)

    def start(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()

    def stop(self):
        self._stop.set()
        if self._t:
            self._t.join(timeout=3)
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            for i, n in enumerate(names):
                if len(r) > 3 + i and r[3 + i].lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ model
def build_model(device, cfg_over=None, rank=16, seed=0, target="all", dropout=0.0):
    from simpletuner_b200.flux.model import Flux, default_config
    from simpletuner_b200.flux.transformer import FluxTransformer2DModel

    kw = dict(FLUX_DEV)
    kw.update(cfg_over or {})
    with torch.device(device):
        m = FluxTransformer2DModel(**kw)
    g = torch.Generator(device=device).manual_seed(seed)
    with torch.no_grad():
        for name, p in m.named_parameters():
            if name.endswith("norm_q.weight") or name.endswith("norm_k.weight") or "norm_added" in name:
                p.fill_(1.0)
            elif name.endswith(".bias"):
                p.normal_(0.0, 0.01, generator=g)
            else:
                p.normal_(0.0, 0.02, generator=g)
    w = Flux(default_config(lora_rank=rank, flux_lora_target=target, lora_dropout=dropout), transformer=m, device=device)
    w.add_lora_adapter()
    with torch.no_grad():  # non-zero B so every LoRA gradient path does real work
        for lin in m.lora_linears().values():
            lin.lora_B["default"].weight.normal_(0.0, 0.02, generator=g)
    return w


LYCORIS_DEFAULT = {"algo": "lokr", "multiplier": 1.0, "linear_dim": 10000, "linear_alpha": 1, "factor": 10,
                   "apply_preset": {"target_module": ["Attention", "FeedForward"],
                                    "module_algo_map": {"Attention": {"factor": 10}, "FeedForward": {"factor": 4}}}}
"""The reference's documented LyCORIS config (documentation/LYCORIS.md:24-47)."""


def build_flux_lokr(device, cfg_over=None, seed=0):
    """BASELINE configs[3]: Flux.1-dev + LyCORIS LoKr, latents encoded on the fly by the (random-init) Flux AutoencoderKL."""
    from simpletuner_b200.flux.model import Flux, default_config
    from simpletuner_b200.flux.transformer import FluxTransformer2DModel
    from simpletuner_b200.vae.autoencoder import AutoencoderKL

    kw = dict(FLUX_DEV)
    kw.update(cfg_over or {})
    with torch.device(device):
        m = FluxTransformer2DModel(**kw)
        vae = AutoencoderKL()
    g = torch.Generator(device=device).manual_seed(seed)
    with torch.no_grad():
        for name, p in m.named_parameters():
            if name.endswith("norm_q.weight") or name.endswith("norm_k.weight") or "norm_added" in name:
                p.fill_(1.0)
            elif name.endswith(".bias"):
                p.normal_(0.0, 0.01, generator=g)
            else:
                p.normal_(0.0, 0.02, generator=g)
        for n, p in vae.named_parameters():
            p.normal_(0.0, 0.02, generator=g) if p.dim() > 1 else (p.fill_(1.0) if "norm" in n and n.endswith("weight") else p.zero_())
    w = Flux(default_config(lora_type="lycoris"), transformer=m, device=device)
    net = w.add_lycoris_adapter(json.loads(json.dumps(LYCORIS_DEFAULT)))
    net.to(device)
    with torch.no_grad():   # non-zero w2 so the w1 gradient path does real work (LyCORIS initialises w2 = 0)
        for lora in net.loras:
            lora.lokr_w2.normal_(0.0, 0.01, generator=g)
    m.invalidate_plans()
    return w, net, vae


def lokr_extra_tf_per_sample():
    """One more weight-gradient GEMM (2 * tokens * N * K) per LoKr-adapted Linear, per image."""
    D = 3072
    dbl = 2 * (S_IMG * (4 * D * D + 2 * 4 * D * D) + S_TXT * (4 * D * D + 2 * 4 * D * D))   # q,k,v,out + fc1,fc2 per stream
    sgl = 2 * (S_IMG + S_TXT) * 3 * D * D
    return (19 * dbl + 38 * sgl) * 1e-12


def synth_batch(B, device, pinned=False, seed=0, hw=128, s_txt=S_TXT, joint=4096, pooled=768):
    g = torch.Generator().manual_seed(seed)
    b = {"latent_batch": torch.randn(B, 16, hw, hw, generator=g).bfloat16(),
         "prompt_embeds": torch.randn(B, s_txt, joint, generator=g).bfloat16(),
         "add_text_embeds": torch.randn(B, pooled, generator=g).bfloat16()}
    if pinned:
        return {k: v.pin_memory() for k, v in b.items()}
    return {k: v.to(device) for k, v in b.items()}


# SD3.5-medium geometry (BASELINE configs[2]: "SD3-medium MMDiT full fine-tune bf16, 512^2 aspect buckets, batch=8, 8xB200 DDP")
SD35_MEDIUM = dict(sample_size=128, patch_size=2, in_channels=16, num_layers=24, attention_head_dim=64, num_attention_heads=24,
                   joint_attention_dim=4096, caption_projection_dim=1536, pooled_projection_dim=2048, out_channels=16,
                   pos_embed_max_size=384, dual_attention_layers=tuple(range(13)), qk_norm="rms_norm")
SD3_BUCKETS = [(64, 64), (56, 72), (72, 56), (48, 80), (80, 48)]    # latent (h, w) of the 64-px aligned 512^2-area buckets (SURVEY 8d)
SD3_S_TXT = 231       # 77 CLIP + 154 T5 tokens (sd3/model.py)


def sd3_tf_per_sample(hw=(64, 64), s_txt=SD3_S_TXT, full_ft=True):
    """Algorithmic TFLOP of one SD3.5-medium training sample (SURVEY.md 8d: GEMM 2MNK, attention 4 S^2 D fwd / 8 S^2 D bwd)."""
    D, L, n_dual = 1536, 24, 13
    s_img = (hw[0] // 2) * (hw[1] // 2)
    S = s_img + s_txt
    lin = 0.0
    for i in range(L):
        pre_only = i == L - 1
        lin += 2 * s_img * (3 * D * D + D * D + 8 * D * D)                              # img: qkv, out, mlp
        lin += 2 * s_txt * (3 * D * D + (0 if pre_only else D * D + 8 * D * D))         # txt
        if i < n_dual:
            lin += 2 * s_img * (4 * D * D)                                              # attn2 qkv + out
    attn = sum(4 * S * S * D + (4 * s_img * s_img * D if i < n_dual else 0) for i in range(L))
    fwd = (lin + attn) * 1e-12
    return fwd * 3 if full_ft else fwd + lin * 1e-12 + 2 * attn * 1e-12


def build_sd3_fullft(device, seed=0, tiny=False):
    from simpletuner_b200.flux.model import default_config
    from simpletuner_b200.sd3.model import SD3
    from simpletuner_b200.sd3.transformer import SD3Transformer2DModel

    kw = dict(SD35_MEDIUM)
    if tiny:
        kw.update(num_layers=3, attention_head_dim=64, num_attention_heads=4, joint_attention_dim=256, caption_projection_dim=256,
                  pooled_projection_dim=64, pos_embed_max_size=96, dual_attention_layers=(0,))
    with torch.device(device):
        m = SD3Transformer2DModel(**kw)
    g = torch.Generator(device=device).manual_seed(seed)
    with torch.no_grad():
        for name, p in m.named_parameters():
            if "norm_q" in name or "norm_k" in name or "norm_added" in name:
                p.fill_(1.0)
            elif name.endswith(".bias"):
                p.normal_(0.0, 0.01, generator=g)
            else:
                p.normal_(0.0, 0.02, generator=g)
        m.pos_embed.pos_embed.normal_(0.0, 0.02, generator=g)
    m.enable_full_finetune()
    return SD3(default_config(model_type="full"), transformer=m, device=device)


def synth_batch_sd3(B, device, hw, pinned=False, seed=0, s_txt=SD3_S_TXT, joint=4096, pooled=2048):
    g = torch.Generator().manual_seed(seed)
    b = {"latent_batch": torch.randn(B, 16, hw[0], hw[1], generator=g).bfloat16(),
         "prompt_embeds": torch.randn(B, s_txt, joint, generator=g).bfloat16(),
         "add_text_embeds": torch.randn(B, pooled, generator=g).bfloat16()}
    if pinned:
        return {k: v.pin_memory() for k, v in b.items()}
    return {k: v.to(device) for k, v in b.items()}


# PixArt-Sigma XL (BASELINE configs[4]: "PixArt-Sigma DiT LoRA rank=32, mixed aspect buckets 512-1536, grad-accum=4, 8xB200")
PIXART_SIGMA = dict(num_attention_heads=16, attention_head_dim=72, in_channels=4, out_channels=8, num_layers=28, cross_attention_dim=1152,
                    sample_size=128, caption_channels=4096)
PIXART_BUCKETS = [(64, 64), (96, 128), (128, 128), (112, 144), (160, 160), (192, 192), (128, 96), (144, 112)]   # latent (h, w): 512^2 .. 1536^2 px
PIXART_S_TXT = 300
PIXART_GRAD_ACCUM = 4   # BASELINE configs[4]: a "step" of the PixArt line is one optimizer step = 4 micro-batches


def pixart_tf_per_sample(hw, s_txt=PIXART_S_TXT):
    """LoRA step (fwd + dgrad + attention backward) of one PixArt-Sigma sample, SURVEY.md 8d counting."""
    D, L = 1152, 28
    S = (hw[0] // 2) * (hw[1] // 2)
    lin = L * (2 * S * (4 * D * D + 2 * D * D + 8 * D * D) + 2 * s_txt * 2 * D * D)
    attn = L * (4 * S * S * D + 4 * S * s_txt * D)
    return (2 * lin + 3 * attn) * 1e-12


def build_pixart_lora(device, rank=32, seed=0, tiny=False):
    from simpletuner_b200.pixart.model import PixartSigma, default_config
    from simpletuner_b200.pixart.transformer import PixArtTransformer2DModel

    kw = dict(PIXART_SIGMA)
    if tiny:
        kw.update(num_attention_heads=4, num_layers=2, cross_attention_dim=288, caption_channels=96)
    with torch.device(device):
        m = PixArtTransformer2DModel(**kw)
    g = torch.Generator(device=device).manual_seed(seed)
    with torch.no_grad():
        for name, p in m.named_parameters():
            if name.endswith(".bias"):
                p.normal_(0.0, 0.01, generator=g)
            else:
                p.normal_(0.0, 0.02, generator=g)
    w = PixartSigma(default_config(lora_rank=rank), transformer=m, device=device)
    w.add_lora_adapter()
    with torch.no_grad():
        for lin in m.lora_linears().values():
            lin.lora_B["default"].weight.normal_(0.0, 0.02, generator=g)
    return w


def synth_batch_pixart(B, device, hw, pinned=False, seed=0, s_txt=PIXART_S_TXT, caption=4096):
    g = torch.Generator().manual_seed(seed)
    mask = torch.ones(B, s_txt)
    for b in range(B):   # tokenizer padding on the right, a different length per sample
        mask[b, 40 + int(torch.randint(0, s_txt - 40, (1,), generator=g)):] = 0
    b_ = {"latent_batch": torch.randn(B, 4, hw[0], hw[1], generator=g).bfloat16(),
          "prompt_embeds": torch.randn(B, s_txt, caption, generator=g).bfloat16(), "encoder_attention_mask": mask}
    if pinned:
        return {k: v.pin_memory() for k, v in b_.items()}
    return {k: v.to(device) for k, v in b_.items()}


def vae_conv_flops(block_out=(128, 256, 512, 512), layers=2, latent=16, H=1024, W=1024):
    """Algorithmic FLOPs of one AutoencoderKL encode (SURVEY.md 8d: ~4.9 TF per 1024^2 image)."""
    ch = block_out
    fl = 2 * 27 * ch[0] * H * W
    prev, h, w = ch[0], H, W
    for i, c in enumerate(ch):
        for l in range(layers):
            cin = prev if l == 0 else c
            fl += 2 * 9 * cin * c * h * w + 2 * 9 * c * c * h * w + (2 * cin * c * h * w if cin != c else 0)
        prev = c
        if i != len(ch) - 1:
            h, w = h // 2, w // 2
            fl += 2 * 9 * c * c * h * w
    c, S = ch[-1], h * w
    fl += 4 * (2 * 9 * c * c * S) + 4 * 2 * c * c * S + 2 * 2 * S * S * c
    fl += 2 * 9 * c * 2 * latent * S
    return fl


def run_vae(args):
    """`--config vae_encode` (SURVEY 8 rows a29-a31, the path BASELINE configs[3] runs on the fly): Flux AutoencoderKL encode ->
    latent_dist.sample() -> scale_vae_latents_for_cache of B x 1024^2 images per step; e2e from pinned host pixels with the
    cached latents read back to the host."""
    from simpletuner_b200 import ops
    from simpletuner_b200.vae.autoencoder import AutoencoderKL

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=device)
    B = args.batch or 4
    res = 256 if args.tiny else 1024
    with torch.device(device):
        vae = AutoencoderKL()
    g = torch.Generator(device=device).manual_seed(0)
    with torch.no_grad():
        for n, p in vae.named_parameters():
            p.normal_(0.0, 0.02, generator=g) if p.dim() > 1 else (p.fill_(1.0) if "norm" in n and n.endswith("weight") else p.zero_())
    px_dev = [(torch.rand(B, 3, res, res, device=device, generator=g) * 2 - 1).bfloat16() for _ in range(2)]
    px_host = [(torch.rand(B, 3, res, res) * 2 - 1).bfloat16().pin_memory() for _ in range(2)]
    out_host = torch.empty(B, 16, res // 8, res // 8, dtype=torch.bfloat16).pin_memory()

    def region(fn, n):
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n):
            fn(i)
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=device)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    last = {}

    def dev_step(i):
        last["latents"] = vae.encode_scaled(px_dev[i % 2])

    e2e_step = lambda i: out_host.copy_(vae.encode_scaled(px_host[i % 2].to(device, non_blocking=True)))
    for i in range(args.warmup):
        dev_step(i)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ops.reset_launch_count()
    ms = region(dev_step, args.steps)
    launches = ops.launch_count()
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last)
    e2e_step(0)
    ms_e2e = region(e2e_step, args.steps)
    if rank == 0:
        peaks, peak_src = measured_peaks()
        peak_tf = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops")))
        tf_img = vae_conv_flops(H=res, W=res) * 1e-12
        ach = tf_img * B / (ms / args.steps * 1e-3)
        line = {"metric": "images/sec AutoencoderKL latent encode 1024^2 (VAE cache path)", "value": B * world * args.steps / (ms * 1e-3), "unit": UNIT,
                "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic (random-init Flux AutoencoderKL, U(-1,1) pixels)",
                "config": {"workload": f"Flux AutoencoderKL encode -> latent_dist.sample() -> scale_vae_latents_for_cache, {B} x {res}^2 images per step (caching/vae.py:1293-1355)",
                           "config_name": "vae_encode", "global_batch": B * world, "per_gpu_batch": B, "parallelism": f"dp{world}",
                           "l2_policy": "inputs larger than L2 (activations of one 1024^2 image: 0.27 GB at 128 channels)"},
                "e2e": {"value": B * world * args.steps / (ms_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": B * 3 * res * res * 2,
                        "d2h_bytes_per_step": out_host.numel() * 2, "ms_per_step": ms_e2e / args.steps},
                "gpu_launches": int(launches), "clocks": clocks,
                "roofline": {"bound": "tensor", "kernel": "whole encode (implicit-GEMM 3x3 convs dominate)", "achieved": round(ach, 1), "peak": peak_tf,
                             "unit": "TFLOP/s", "frac": round(ach / peak_tf, 4), "peak_source": f"MEASURED_PEAKS.json bf16_tflops_sustained ({peak_src})",
                             "traffic": None},
                "model_tflops": {"algorithmic_tf_per_image": round(tf_img, 2), "achieved_tflops_per_gpu": round(ach, 1)},
                "peak_mem_gb": round(torch.cuda.max_memory_allocated() / 2 ** 30, 1)}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def run_text(args):
    """`--config text_encode` (SURVEY 8f rank 4): the embed path of `FluxPipeline.encode_prompt` — T5-XXL encoder (24 layers,
    d_model 4096, 64 heads, d_ff 10240, 512 tokens) + CLIP-L text model (12 layers, 768, 77 tokens) — on token ids; a step
    encodes B prompts.  e2e: pinned host token ids in, embeddings read back to the host (what the text-embed cache stores)."""
    from simpletuner_b200 import ops
    from simpletuner_b200.text import CLIPTextModel, T5EncoderModel, encode_token_ids

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=device)
    B = args.batch or 16
    kw5 = dict(vocab_size=512, d_model=256, d_kv=64, d_ff=512, num_layers=2, num_heads=4) if args.tiny else {}
    kwc = dict(vocab_size=512, hidden_size=128, intermediate_size=256, num_hidden_layers=2, num_attention_heads=2) if args.tiny else {}
    with torch.device(device):
        t5, clip = T5EncoderModel(**kw5), CLIPTextModel(**kwc)
    g = torch.Generator(device=device).manual_seed(0)
    with torch.no_grad():
        for m in (t5, clip):
            for n, p in m.named_parameters():
                if "layer_norm" in n and n.endswith("weight"):
                    p.fill_(1.0)
                elif n.endswith("bias"):
                    p.zero_()
                else:
                    p.normal_(0.0, 0.02, generator=g)
    c5, cc = t5.config, clip.config
    S5, Sc = 512, 77
    gh = torch.Generator().manual_seed(1 + rank)
    host = [(torch.randint(3, cc.vocab_size - 1, (B, Sc), generator=gh).pin_memory(), torch.randint(0, c5.vocab_size, (B, S5), generator=gh).pin_memory())
            for _ in range(2)]
    for ci, _ in host:
        ci[:, -1] = cc.vocab_size - 1
    dev = [(a.to(device), b.to(device)) for a, b in host]
    out_e = torch.empty(B, S5, c5.d_model, dtype=torch.bfloat16).pin_memory()
    out_p = torch.empty(B, cc.hidden_size, dtype=torch.bfloat16).pin_memory()

    def region(fn, n):
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n):
            fn(i)
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=device)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    last = {}

    def dev_step(i):
        last["prompt_embeds"], last["pooled_prompt_embeds"], _, _ = encode_token_ids(clip, t5, *dev[i % 2])

    def e2e_step(i):
        ci, ti = host[i % 2]
        e, p_, _, _ = encode_token_ids(clip, t5, ci.to(device, non_blocking=True), ti.to(device, non_blocking=True))
        out_e.copy_(e, non_blocking=True)
        out_p.copy_(p_)

    for i in range(args.warmup):
        dev_step(i)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ops.reset_launch_count()
    ms = region(dev_step, args.steps)
    launches = ops.launch_count()
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last)
    e2e_step(0)
    ms_e2e = region(e2e_step, args.steps)
    if rank == 0:
        peaks, peak_src = measured_peaks()
        peak_tf = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops")))
        inner5 = c5.num_heads * c5.d_kv
        tf_prompt = (c5.num_layers * (2 * S5 * (4 * c5.d_model * inner5 + 3 * c5.d_model * c5.d_ff) + 4 * S5 * S5 * inner5)
                     + cc.num_hidden_layers * (2 * Sc * (4 * cc.hidden_size ** 2 + 2 * cc.hidden_size * cc.intermediate_size) + 4 * Sc * Sc * cc.hidden_size)) * 1e-12
        ach = tf_prompt * B / (ms / args.steps * 1e-3)
        line = {"metric": "prompts/sec Flux text-embed path (T5-XXL encoder 512 tokens + CLIP-L pooled)", "value": B * world * args.steps / (ms * 1e-3),
                "unit": "prompts/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
                "data": "synthetic (random-init T5 v1.1 XXL / CLIP-L architectures, random token ids)",
                "config": {"workload": f"FluxPipeline.encode_prompt compute (flux/pipeline.py:1085, 1127): {B} prompts per step, T5 encoder "
                                       f"{c5.num_layers} x d{c5.d_model} on {S5} tokens + CLIP text {cc.num_hidden_layers} x d{cc.hidden_size} on {Sc} tokens",
                           "config_name": "text_encode", "global_batch": B * world, "per_gpu_batch": B, "parallelism": f"dp{world}",
                           "l2_policy": "inputs larger than L2 (9.5 GB of T5 weights streamed every step)", "tiny": bool(args.tiny)},
                "e2e": {"value": B * world * args.steps / (ms_e2e * 1e-3), "unit": "prompts/s", "h2d_bytes_per_step": B * (S5 + Sc) * 8,
                        "d2h_bytes_per_step": (out_e.numel() + out_p.numel()) * 2, "ms_per_step": ms_e2e / args.steps},
                "gpu_launches": int(launches), "clocks": clocks,
                "roofline": {"bound": "tensor", "kernel": "whole encode (T5 projections / feed-forward GEMMs dominate)", "achieved": round(ach, 1),
                             "peak": peak_tf, "unit": "TFLOP/s", "frac": round(ach / peak_tf, 4),
                             "peak_source": f"MEASURED_PEAKS.json bf16_tflops_sustained ({peak_src})", "traffic": None},
                "model_tflops": {"algorithmic_tf_per_prompt": round(tf_prompt, 3), "achieved_tflops_per_gpu": round(ach, 1)},
                "peak_mem_gb": round(torch.cuda.max_memory_allocated() / 2 ** 30, 1)}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def batch_bytes(b):
    return int(sum(v.numel() * v.element_size() for v in b.values()))


# ------------------------------------------------------------------------------------------------ --dump-outputs
DUMP_MAX_ELEMS = 1 << 22   # 16 MB of float32 per output; no arm writes more than three outputs


def flat_sample(tensors, n=DUMP_MAX_ELEMS, seed=0):
    """The tensors flattened and concatenated in order, as float32 on the host.  When that is more than `n` elements, a
    fixed seeded sample of `n` of them (the same positions on every run), gathered tensor by tensor so that the whole
    concatenation (5 GB for the SD3.5 full fine-tune) is never materialised."""
    sizes = [t.numel() for t in tensors]
    total = sum(sizes)
    if total <= n:
        return torch.cat([t.detach().reshape(-1).float().cpu() for t in tensors])
    idx = torch.randint(0, total, (n,), generator=torch.Generator().manual_seed(seed)).sort().values
    parts, start = [], 0
    for t, size in zip(tensors, sizes):
        lo, hi = torch.searchsorted(idx, torch.tensor([start, start + size])).tolist()
        if hi > lo:
            parts.append(t.detach().reshape(-1)[(idx[lo:hi] - start).to(t.device)].float().cpu())
        start += size
    return torch.cat(parts)


def dump_outputs(out_dir, outputs):
    """Write each output as `<out_dir>/<name>.npy` in float32: a tensor that fits DUMP_MAX_ELEMS keeps its shape, a larger
    tensor or a list of tensors (e.g. the trainable parameters) is stored as `flat_sample` of it."""
    import numpy as np

    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    for name, x in outputs.items():
        if torch.is_tensor(x) and x.numel() <= DUMP_MAX_ELEMS:
            arr = x.detach().float().cpu()
        else:
            arr = flat_sample(list(x) if not torch.is_tensor(x) else [x], n=DUMP_MAX_ELEMS)
        np.save(d / f"{name}.npy", arr.numpy())


# ------------------------------------------------------------------------------------------------ per-kernel timing pass
def profile_kernels(step_fn, batch):
    """One extra (untimed-for-the-headline) step with CUDA events around every GEMM / attention launch on the
    launching stream: gives the live average duration and algorithmic FLOPs of the dominant kernels."""
    from simpletuner_b200 import ops
    import simpletuner_b200.flux.blocks as blocks
    import simpletuner_b200.flux.transformer as tr

    recs = []
    og, oaf, oab = ops.gemm, ops.attn_fwd, ops.attn_bwd

    def timed(kind, flops_fn, fn):
        def wrapper(*a, **k):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out = fn(*a, **k)
            e1.record()
            recs.append((kind, flops_fn(*a, **k), e0, e1))
            return out
        return wrapper

    def gemm_flops(a_list, w_list, *a, **k):
        a0 = a_list[0]
        M = a0.shape[0] * a0.shape[1] if a0.dim() == 3 else a0.shape[0]
        N = w_list[0].shape[0]
        return 2.0 * M * N * sum(x.shape[-1] for x in a_list)

    def attn_f(q, k_, v, *a, **kw):
        B, S, H, HD = q.shape
        return 4.0 * B * H * S * k_.shape[1] * HD

    def attn_b(q, k_, v, *a, **kw):
        return 2.5 * attn_f(q, k_, v)

    ops.gemm = timed("gemm", gemm_flops, og)
    ops.attn_fwd = timed("attn_fwd", attn_f, oaf)
    ops.attn_bwd = timed("attn_bwd", attn_b, oab)
    try:
        step_fn(batch)
        torch.cuda.synchronize()
    finally:
        ops.gemm, ops.attn_fwd, ops.attn_bwd = og, oaf, oab
    agg = {}
    for kind, fl, e0, e1 in recs:
        ms = e0.elapsed_time(e1)
        a = agg.setdefault(kind, {"launches": 0, "ms": 0.0, "tflop": 0.0})
        a["launches"] += 1
        a["ms"] += ms
        a["tflop"] += fl * 1e-12
    # "big" GEMMs only for the roofline of the dominant kernel (>= 1 GFLOP; excludes M=4 conditioning GEMMs)
    big = [(fl, e0.elapsed_time(e1)) for kind, fl, e0, e1 in recs if kind == "gemm" and fl >= 1e11]
    out = {k: {"launches": v["launches"], "ms": round(v["ms"], 3), "tflops": round(v["tflop"] / (v["ms"] * 1e-3), 1) if v["ms"] > 0 else None}
           for k, v in agg.items()}
    if big:
        out["gemm_big"] = {"launches": len(big), "ms": round(sum(m for _, m in big), 3),
                           "avg_ms": round(sum(m for _, m in big) / len(big), 4),
                           "tflops": round(sum(f for f, _ in big) * 1e-12 / (sum(m for _, m in big) * 1e-3), 1),
                           "tflop_per_launch": round(sum(f for f, _ in big) * 1e-12 / len(big), 4)}
    return out


# ------------------------------------------------------------------------------------------------ CPU baseline (oracle port)
class CpuBaseline:
    """Depth-reduced Flux LoRA train step through the fp32 CPU oracle (BASELINE.md 4): full width (D = 3072), full
    4096 + 512-token sequence, B = 1.  One `step(kind)` = forward + LoRA backward of ONE block of that kind ("double" or
    "single") inside the whole step pipeline (noisy latents, embedders, norm_out / proj_out, loss); the block kinds are
    timed separately because a double block costs ~1.5x a single one, and a full-depth sample step is
    19 * t_double + 38 * t_single (embedders / head / loss are < 0.1 % and are counted once per timed block, i.e. over-
    counted)."""

    def __init__(self, threads=None, seq=(S_IMG, S_TXT)):
        from oracle import flux_oracle as O

        self.O = O
        self.threads = threads or os.cpu_count() or 1
        torch.set_num_threads(self.threads)
        self.models = {}
        for kind, blocks in (("double", (1, 0)), ("single", (0, 1))):
            cfg = O.FluxConfig(num_layers=blocks[0], num_single_layers=blocks[1], guidance_embeds=True)
            P = O.init_flux_params(cfg, seed=0)
            L = {k: v.requires_grad_(True) for k, v in O.init_lora_params(cfg, 16, seed=1).items()}
            self.models[kind] = (cfg, P, L)
        hw = int((seq[0] * 4) ** 0.5)
        g = torch.Generator().manual_seed(0)
        self.b = {"latents": torch.randn(1, 16, hw, hw, generator=g), "noise": torch.randn(1, 16, hw, hw, generator=g),
                  "sigmas": torch.tensor([0.6]), "prompt_embeds": torch.randn(1, seq[1], 4096, generator=g),
                  "pooled": torch.randn(1, 768, generator=g)}
        self.loss = None
        self.times = {"double": [], "single": []}

    def step(self, kind: str, record: bool = True) -> float:
        cfg, P, L = self.models[kind]
        t0 = time.perf_counter()
        loss, _ = self.O.flux_train_step_loss(P, cfg, self.b, lora=L)
        loss.backward()
        dt = time.perf_counter() - t0
        for v in L.values():
            v.grad = None
        self.loss = float(loss.item())
        if record:
            self.times[kind].append(dt)
        return dt

    def summary(self):
        td = statistics.median(self.times["double"]) if self.times["double"] else None
        ts = statistics.median(self.times["single"]) if self.times["single"] else None
        if td is None:       # only singles were timed: a double block does the same attention + 1.5x the linear work
            td = 1.5 * ts
        if ts is None:
            ts = td / 1.5
        full = 19 * td + 38 * ts
        return {"t_double_s": td, "t_single_s": ts, "n_double": len(self.times["double"]), "n_single": len(self.times["single"]),
                "spread": {k: [round(min(v), 2), round(max(v), 2)] for k, v in self.times.items() if v},
                "threads": self.threads, "extrapolated_full_depth_sec": full, "images_per_sec": 1.0 / full, "loss": self.loss}


PATTERN = ("double", "single", "single", "double", "single", "single")   # 2 double + 4 single per 6 steps (BASELINE.md 4)


def cpu_baseline_sample(threads=None):
    """Bounded sample for the b200 arm's `cpu_baseline` key: one double + one single block (~40 s of CPU work)."""
    cb = CpuBaseline(threads)
    cb.step("double")
    cb.step("single")
    return cb.summary()


# ------------------------------------------------------------------------------------------------ main arms
WORKLOAD = ("Flux.1-dev LoRA rank16 (flux_lora_target=all, 266 targets, 26.1M trainable) bf16, 1024^2 cached latents [B,16,128,128] + "
            "T5 [B,512,4096], train step = prepare_batch+fwd+loss+bwd+value-clip+optimizer")


def run_reference(args):
    """The reference path's CPU restatement on the host cores.  One "step" = one BLOCK-SAMPLE: forward + LoRA backward of
    one Flux block (kinds cycle double, single, single, ... = 2 : 4) at full width and full sequence, B = 1, i.e. a
    bounded 1/57-of-an-image piece of the workload; `ms_per_step` is the measured time of such a step and `value` is the
    full-depth throughput 1 / (19 * median(t_double) + 38 * median(t_single))."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    cb = CpuBaseline(threads)
    t_all = []
    for i in range(args.warmup + args.steps):
        dt = cb.step(PATTERN[i % len(PATTERN)], record=(i >= args.warmup))
        if i >= args.warmup:
            t_all.append(dt)
    sm = cb.summary()
    value = sm["images_per_sec"]
    sample = (f"fp32 CPU oracle port (reference needs diffusers/accelerate/peft: not installable), B=1, full width D=3072, full "
              f"4096+512-token sequence; each step = fwd + LoRA bwd of ONE block, kinds cycling 2 double : 4 single; "
              f"median t_double={sm['t_double_s']:.1f}s (n={sm['n_double']}), median t_single={sm['t_single_s']:.1f}s (n={sm['n_single']}), "
              f"min/max {sm['spread']}; value = 1/(19 t_double + 38 t_single) (linear-in-depth extrapolation)")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": statistics.mean(t_all) * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32",
        "data": "synthetic (random-init Flux.1-dev architecture; seeded N(0,1) cached latents + T5/CLIP embeds)",
        "config": {"workload": WORKLOAD, "global_batch": 1, "per_gpu_batch": 1, "seq_len": S_IMG + S_TXT, "parallelism": "cpu",
                   "step_is": "one block-sample = 1/57 of one image's train step (see cpu_baseline.sample)",
                   "extrapolated_ms_per_image": sm["extrapolated_full_depth_sec"] * 1e3},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------ eager torch baseline on the GPU
def eager_gpu_step_fn(wrapper, device):
    """What the reference's DEFAULT path costs on this box (informational): the dtype-agnostic oracle restatement of the
    diffusers modules run as eager bf16 torch ops on the GPU, attention through `F.scaled_dot_product_attention`
    (attention_mechanism="diffusers"), PEFT-style un-fused LoRA matmuls, every block under torch.utils.checkpoint
    (gradient_checkpointing=true is the reference default), sharing the B200 model's own parameter tensors."""
    import torch.nn.functional as F
    from torch.utils.checkpoint import checkpoint

    from oracle import flux_oracle as O

    den = wrapper._denoiser()
    P = {k: v.detach() for k, v in den.state_dict().items() if "lora_" not in k}
    lora = {}
    for name, lin in den.lora_linears().items():
        lora[name + ".lora_A.weight"] = lin.lora_A["default"].weight
        lora[name + ".lora_B.weight"] = lin.lora_B["default"].weight
    cfg = O.FluxConfig(**{k: getattr(den.config, k) for k in ("in_channels", "num_layers", "num_single_layers", "attention_head_dim",
                                                               "num_attention_heads", "joint_attention_dim", "pooled_projection_dim",
                                                               "guidance_embeds", "axes_dims_rope")})
    rope_cache = {}
    o_rope, o_dbl, o_sgl = O.rope_tables, O.flux_double_block, O.flux_single_block

    def rope_dev(ids, *a):
        key = (tuple(ids.shape), float(ids.sum()))
        if key not in rope_cache:
            rope_cache[key] = tuple(t.to(device) for t in o_rope(ids.cpu(), *a))
        return rope_cache[key]

    def step(batch):
        O.sdpa = lambda q, k, v: F.scaled_dot_product_attention(q, k, v)
        O.rope_tables = rope_dev
        O.flux_double_block = lambda P_, c, i, x, enc, temb, rope, lo, ls: checkpoint(
            lambda x_, e_, t_: o_dbl(P_, c, i, x_, e_, t_, rope, lo, ls), x, enc, temb, use_reentrant=False)
        O.flux_single_block = lambda P_, c, i, x, temb, rope, lo, ls: checkpoint(
            lambda x_, t_: o_sgl(P_, c, i, x_, t_, rope, lo, ls), x, temb, use_reentrant=False)
        try:
            lat = batch["latent_batch"]
            B, Cc, Hh, Ww = lat.shape
            noise = torch.randn_like(lat)
            sig = torch.sigmoid(torch.randn((B,), device=device))
            sig = (3.0 * sig) / (1 + 2.0 * sig)
            s4 = sig.view(-1, 1, 1, 1).to(lat.dtype)
            noisy = (1 - s4) * lat + s4 * noise
            packed = O.pack_latents(noisy, B, Cc, Hh, Ww)
            img_ids = O.prepare_latent_image_ids(Hh, Ww).to(device)
            txt_ids = torch.zeros(batch["prompt_embeds"].shape[1], 3, device=device)
            g = torch.full((B,), 1.0, device=device)
            out = O.flux_forward(P, cfg, packed, batch["prompt_embeds"], batch["add_text_embeds"], sig, img_ids, txt_ids, g, lora, 1.0)
            pred = O.unpack_latents(out, Hh * 8, Ww * 8, 16)
            loss = F.mse_loss(pred.float(), (noise - lat).float(), reduction="none").mean(dim=(1, 2, 3)).mean()
            loss.backward()
            return loss.detach()
        finally:
            O.sdpa, O.rope_tables, O.flux_double_block, O.flux_single_block = o_sdpa, o_rope, o_dbl, o_sgl

    o_sdpa = O.sdpa
    return step


def time_eager_gpu(wrapper, device, batches, opt, steps=3, warmup=2):
    fn = eager_gpu_step_fn(wrapper, device)

    def one(i):
        fn(batches[i % len(batches)])
        opt.step()
        opt.zero_grad(set_to_none=True)

    for i in range(warmup):
        one(i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        one(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def run_b200(args):
    import torch.distributed as dist

    from simpletuner_b200 import ops
    from simpletuner_b200.training.step import TrainStep, wrap_ddp

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    sd3 = args.config == "sd3_fullft"
    pix = args.config == "pixart_lora"
    lokr = args.config == "flux_lokr"
    B = args.batch if args.batch else (8 if sd3 else (2 if lokr else 4))
    cfg_over = None
    hw, s_txt = 128, S_TXT
    if args.tiny:  # plumbing check only (never a bench value)
        cfg_over = dict(num_layers=1, num_single_layers=2, num_attention_heads=4, joint_attention_dim=256, pooled_projection_dim=64)
        hw, s_txt = 32, 64
    if sd3:
        wrapper = build_sd3_fullft(device, seed=0, tiny=args.tiny)
        if args.dp == "auto":
            args.dp = "flat"     # CUDA-graph replay of fwd + bwd, then one flat 5 GB all-reduce; `--dp ddp` = torch DDP buckets (eager)
    elif pix:
        wrapper = build_pixart_lora(device, rank=32, seed=0, tiny=args.tiny)
    elif lokr:
        wrapper, lokr_net, vae = build_flux_lokr(device, cfg_over, seed=0)
    else:
        wrapper = build_model(device, cfg_over, rank=16, seed=0, target=args.lora_target, dropout=args.lora_dropout)
    if args.gradient_checkpointing:   # non-default: the reference's --gradient_checkpointing memory / time trade-off
        wrapper._denoiser().enable_gradient_checkpointing()
    if world > 1 and args.dp == "ddp":
        wrap_ddp(wrapper, device_ids=[local_rank])
    params = [p for p in wrapper._denoiser().parameters() if p.requires_grad]
    if lokr:
        params = list(lokr_net.parameters())
    if args.optimizer == "adamw_bf16":   # the reference's default optimizer, one libstb200 launch per step
        from simpletuner_b200.training.optim import AdamWBF16
        opt = AdamWBF16(params, lr=1e-4, weight_decay=1e-2, eps=1e-6, seed=1234 + rank)
    else:
        opt = torch.optim.AdamW(params, lr=1e-4, weight_decay=1e-2, fused=True)
    grad_sync = None
    if world > 1 and args.dp == "flat":
        from simpletuner_b200.training.dist import FlatGradSync
        # full fine-tune (5 GB of gradients): 8 chunks, the optimizer of chunk i overlaps the all-reduce of chunk i + 1
        grad_sync = FlatGradSync(params, pipeline_chunks=(int(os.environ.get("STB_GRAD_CHUNKS", "8")) if sd3 else 0))
    accum = PIXART_GRAD_ACCUM if pix else 1
    step = TrainStep(wrapper, opt, max_grad_norm=(0.01 if pix else 2.0), grad_clip_method="value", grad_sync=grad_sync,
                     gradient_accumulation_steps=accum)
    # auto: the two configs whose step is made of many short kernels (SD3.5-medium at 512^2, PixArt-Sigma) replay CUDA graphs
    use_graph = args.graph == "on" or (args.graph == "auto" and (sd3 or pix) and args.dp != "ddp")
    if use_graph:
        from simpletuner_b200.training.step import GraphedTrainStep
        # PixArt (epsilon family): the reference draws timesteps on the host -> prepare_batch stays eager, the rest is replayed
        step = GraphedTrainStep(step, capture_prepare=not pix)
    torch.manual_seed(42 + rank)  # seed_for_each_device=True (trainer.py:2554-2556)
    joint = cfg_over["joint_attention_dim"] if cfg_over else 4096
    pooled = cfg_over["pooled_projection_dim"] if cfg_over else 768
    if sd3:
        # aspect buckets: every rank walks the five 512^2-area buckets round-robin (ranks start at different buckets, as the
        # reference's per-rank samplers do), one uniform shape inside a micro-batch
        kw3 = dict(s_txt=64, joint=256, pooled=64) if args.tiny else {}
        bks = [(16, 16), (12, 20)] if args.tiny else SD3_BUCKETS
        nb = len(bks)
        dev_batches = [synth_batch_sd3(B, device, bks[(i + rank) % nb], seed=100 + rank * 10 + i, **kw3) for i in range(nb)]
        host_batches = [synth_batch_sd3(B, device, bks[(i + rank) % nb], pinned=True, seed=200 + rank * 10 + i, **kw3) for i in range(nb)]
    elif pix:
        kwp = dict(s_txt=40, caption=96) if args.tiny else {}
        bks = [(16, 16), (24, 16), (16, 24), (32, 32)] if args.tiny else PIXART_BUCKETS
        nb = len(bks)
        dev_batches = [synth_batch_pixart(B, device, bks[(i + 3 * rank) % nb], seed=100 + rank * 10 + i, **kwp) for i in range(nb)]
        host_batches = [synth_batch_pixart(B, device, bks[(i + 3 * rank) % nb], pinned=True, seed=200 + rank * 10 + i, **kwp) for i in range(nb)]
    else:
        dev_batches = [synth_batch(B, device, seed=100 + rank * 10 + i, hw=hw, s_txt=s_txt, joint=joint, pooled=pooled) for i in range(2)]
        host_batches = [synth_batch(B, device, pinned=True, seed=200 + rank * 10 + i, hw=hw, s_txt=s_txt, joint=joint, pooled=pooled) for i in range(2)]
    if lokr:
        # on-the-fly VAE encode (BASELINE configs[3]): the batch carries PIXELS; every step encodes them to latents first
        # (vae.encode -> latent_dist.sample() -> scale_vae_latents_for_cache, caching/vae.py:1293-1355) inside the timed region
        res = hw * 8
        gpx = torch.Generator().manual_seed(300 + rank)
        for bl, pin in ((dev_batches, False), (host_batches, True)):
            for b in bl:
                px = (torch.rand(B, 3, res, res, generator=gpx) * 2 - 1).bfloat16()
                b.pop("latent_batch")
                b["pixels"] = px.pin_memory() if pin else px.to(device)
        inner_step = step

        def step(batch):      # noqa: F811 — the user-facing call of this config: pixels in, loss out
            batch = dict(batch)
            batch["latent_batch"] = vae.encode_scaled(batch.pop("pixels"))
            return inner_step(batch)
        step.check_finite = inner_step.check_finite
    nbat = len(dev_batches)
    if use_graph:      # every bucket shape must be captured BEFORE the timed region
        args.warmup = max(args.warmup, nbat)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed_region(fn, n):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n):
            fn(i)
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=device)
        if world > 1:
            every = [torch.zeros_like(ms) for _ in range(world)]
            dist.all_gather(every, ms)
            per_rank_ms.append([round(float(t.item()) / n, 2) for t in every])   # evidence: which rank is the slow one
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    per_rank_ms = []
    last = {}
    # ---- device-resident arm
    def dev_step(i):
        last["loss"] = [step({k: v for k, v in dev_batches[(i * accum + a_) % nbat].items()}) for a_ in range(accum)]

    for i in range(args.warmup):
        dev_step(i)
    if os.environ.get("STB_NCU_RANGE"):
        # `ncu --profile-from-start off ...`: exactly ONE device-resident step inside the profiler range (launch list for
        # profiles/); numbers printed under a profiler are never bench values, so nothing is printed
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        dev_step(args.warmup)
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        return
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ops.reset_launch_count()
    ms_total = timed_region(dev_step, args.steps)
    launches = ops.launch_count()
    clocks = sampler.stop() if rank == 0 else None
    step.check_finite()
    if args.dump_outputs and rank == 0:
        # what a caller of the train step ends up with: the loss of each micro-batch of the last step and the trainable
        # parameters that step's optimizer update left behind
        dump_outputs(args.dump_outputs, {"loss": torch.stack(last["loss"]), "trainable_params": params})

    # ---- end-to-end arm: pinned host batch -> H2D -> step -> D2H loss, every step
    loss_host = torch.empty((), dtype=torch.float32).pin_memory()

    def e2e_step(i):
        for a_ in range(accum):
            hb = host_batches[(i * accum + a_) % nbat]
            ld = step({k: v.to(device, non_blocking=True) for k, v in hb.items()})
        loss_host.copy_(ld, non_blocking=False)  # device->host read of the step's result (synchronises)

    for i in range(max(1, args.warmup // 2)):
        e2e_step(i)
    ms_e2e = timed_region(e2e_step, args.steps)

    # ---- per-kernel pass (extra step, outside both timed regions)
    # (every rank runs it: the step contains the DDP gradient all-reduce)
    eager_step = step.step if use_graph else step
    kern = profile_kernels(lambda b: eager_step(b), dict(dev_batches[0])) if not (sd3 or pix) else None
    barrier()
    mem_gb = torch.cuda.max_memory_allocated() / 2 ** 30

    if rank == 0:
        peaks, peak_src = measured_peaks()
        imgs = B * world * args.steps * accum
        value = imgs / (ms_total * 1e-3)
        e2e_v = imgs / (ms_e2e * 1e-3)
        ms_step = ms_total / args.steps
        peak_tf = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops")))
        roof = None
        if kern and "gemm_big" in kern:
            gb = kern["gemm_big"]
            traffic = None
            tp = ROOT / "profiles" / "r01" / "gemm_traffic.json"
            if tp.exists():  # dram__bytes_read+write of one ncu --set full capture of this kernel (committed summary)
                tj = json.loads(tp.read_text())
                traffic = {"dram_bytes_per_launch": tj["dram_bytes_total"], "algorithmic_bytes": tj["algorithmic_bytes"],
                           "shape": tj["shape"], "source": tj["source"]}
            roof = {"bound": "tensor", "kernel": "gemm_bf16_tn_kernel (tcgen05, all >=0.1 TFLOP launches of one step)",
                    "achieved": gb["tflops"], "peak": peak_tf, "unit": "TFLOP/s", "frac": round(gb["tflops"] / peak_tf, 4),
                    "peak_source": f"MEASURED_PEAKS.json bf16_tflops_sustained ({peak_src}): cuBLAS bf16 back to back for 4 s, "
                                   "the right denominator for a kernel timed inside a long power-capped step",
                    "peak_burst": float(peaks.get("bf16_tflops", 0.0)),
                    "frac_of_burst": round(gb["tflops"] / float(peaks.get("bf16_tflops", peak_tf)), 4), "traffic": traffic,
                    "avg_launch_ms": gb["avg_ms"], "tflop_per_launch": gb["tflop_per_launch"], "launches_per_step": gb["launches"]}
        tf_sample = TF_STEP_SAMPLE
        metric, workload = METRIC, WORKLOAD
        if not (pix or sd3) and (args.lora_target != "all" or args.lora_dropout):
            n_t = len(wrapper._denoiser().lora_linears())
            n_p = sum(p.numel() for p in wrapper._denoiser().parameters() if p.requires_grad)
            workload = workload.replace("flux_lora_target=all, 266 targets, 26.1M trainable",
                                        f"flux_lora_target={args.lora_target}, {n_t} targets, {n_p / 1e6:.1f}M trainable, lora_dropout={args.lora_dropout}")
        if pix:
            tf_sample = sum(pixart_tf_per_sample(hw_) for hw_ in PIXART_BUCKETS) / len(PIXART_BUCKETS)
            metric = "images/sec PixArt-Sigma LoRA r32 bf16, mixed aspect buckets 512-1536, grad-accum 4"
            workload = ("PixArt-Sigma XL (28 blocks, D=1152, 16x72 heads) LoRA rank 32 on attention projections, bf16, mixed aspect buckets "
                        "512^2..1536^2 (latents 64x64 .. 192x192) + 300 caption tokens with random-length masks, epsilon prediction, "
                        "one step = 4 micro-batches (grad-accum 4) + value-clip (0.01) + adamw_bf16")
        if lokr:
            n_t = len(lokr_net.loras)
            n_p = sum(p.numel() for p in lokr_net.parameters())
            metric = "images/sec Flux.1-dev LyCORIS LoKr bf16 1024^2, on-the-fly VAE encode"
            workload = (f"Flux.1-dev LyCORIS LoKr (documentation/LYCORIS.md default: linear_dim 10000 = full-matrix w2, factor 10 on Attention / "
                        f"4 on FeedForward; {n_t} adapted Linears, {n_p / 1e6:.1f}M trainable) bf16, 1024^2 PIXELS [B,3,1024,1024] + T5 [B,512,4096]; "
                        "train step = AutoencoderKL encode + sample + scale (on the fly) + prepare_batch + fwd + loss + bwd (full weight "
                        "gradient of every adapted Linear, contracted to the Kronecker factors) + value-clip + adamw_bf16 + per-step "
                        "rebuild of W + kron(w1, w2)")
            # fwd 1x + dgrad 1x as LoRA-free model, + one more weight-gradient GEMM per adapted Linear (attention + FF of the double
            # blocks, q/k/v of the single blocks) + the VAE encode
            tf_sample = TF_STEP_SAMPLE + lokr_extra_tf_per_sample() + vae_conv_flops(H=1024, W=1024) * 1e-12
        if sd3:
            tf_sample = sum(sd3_tf_per_sample(hw_) for hw_ in SD3_BUCKETS) / len(SD3_BUCKETS)
            metric = "images/sec SD3.5-medium full fine-tune bf16 512^2 buckets"
            workload = ("SD3.5-medium (24 joint blocks, D=1536, 13 dual-attention layers, QK-RMSNorm) FULL fine-tune bf16, 512^2-area aspect "
                        "buckets (64x64, 56x72, 72x56, 48x80, 80x48 latents) + 231 text tokens, train step = prepare_batch+fwd+loss+bwd "
                        "(every weight gradient)+value-clip+adamw_bf16 on all 2.5 B parameters")
        line = {
            "metric": metric, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic (random-init Flux.1-dev architecture; seeded N(0,1) cached latents + T5/CLIP embeds)",
            "config": {
                "workload": workload, "config_name": args.config,
                "global_batch": B * world * accum, "per_gpu_batch": B, "grad_accum": accum,
                "seq_len": (S_IMG + S_TXT) if not (sd3 or pix) else (1024 + SD3_S_TXT if sd3 else "1024..9216 (+300 cross)"),
                "parallelism": f"dp{world}", "grad_exchange": (None if world == 1 else (args.dp + ("+pipelined-optimizer" if (sd3 and args.dp == "flat" and int(os.environ.get("STB_GRAD_CHUNKS", "8")) > 0) else ""))), "cuda_graph": bool(use_graph),
                "activation_recompute": ("every block re-run in backward (--gradient-checkpointing)" if args.gradient_checkpointing else
                                         "none (block-native minimal saves; reference default would recompute every block)"),
                "host_syncs_in_step": 0, "l2_policy": "inputs larger than L2 (24 GB of weights + 16 MB fresh batch streamed every step)",
                "lora_dropout": float(args.lora_dropout) if not (pix or sd3) else 0.0, "optimizer": ("adamw_bf16 (reference default; stochastic-rounding AdamW, one stb_adamw_bf16_multi launch)" if args.optimizer == "adamw_bf16"
                              else "torch.optim.AdamW(fused) on bf16 LoRA params"),
                "tiny": bool(args.tiny),
            },
            "e2e": {"value": e2e_v, "unit": UNIT, "h2d_bytes_per_step": batch_bytes(host_batches[0]), "d2h_bytes_per_step": 4,
                    "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": roof,
            "model_tflops": {"algorithmic_tf_per_image": round(tf_sample, 2),
                             "achieved_tflops_per_gpu": round(tf_sample * B * accum / (ms_step * 1e-3), 1),
                             "frac_of_peak": round(tf_sample * B * accum / (ms_step * 1e-3) / peak_tf, 4)} if not args.tiny else None,
            "kernels": kern, "peak_mem_gb": round(mem_gb, 1),
            # ms/step of every rank for the device-resident region (the reported time is the max): independent replicas with
            # no collective inside backward, so the spread is the GPUs' own power-capped clocks, not communication
            "per_rank_ms_per_step": per_rank_ms[0] if per_rank_ms else None,
        }
        if (sd3 or pix) and roof is None:
            ach = tf_sample * B * accum / (ms_step * 1e-3)
            roof = {"bound": "tensor", "kernel": "whole step, algorithmic FLOPs (SURVEY 8d counting)", "achieved": round(ach, 1),
                    "peak": peak_tf, "unit": "TFLOP/s", "frac": round(ach / peak_tf, 4), "peak_source": f"MEASURED_PEAKS.json bf16_tflops_sustained ({peak_src})",
                    "traffic": None}
            line["roofline"] = roof
        if world == 1 and not args.no_eager_baseline and not args.tiny and not (sd3 or pix):
            try:   # informational: the reference's default eager path (SDPA + per-block checkpointing) on this GPU, same batch
                torch.cuda.empty_cache()
                ms_eager = time_eager_gpu(wrapper, device, dev_batches, opt)
                line["gpu_eager_baseline"] = {
                    "value": B / (ms_eager * 1e-3), "unit": UNIT, "ms_per_step": ms_eager,
                    "what": "eager bf16 torch ops (oracle restatement of the diffusers modules) on this GPU, F.scaled_dot_product_attention, "
                            "un-fused PEFT-style LoRA, torch.utils.checkpoint around every block (reference default "
                            "gradient_checkpointing=true), same parameters / batch / optimizer; 3 timed steps after 2 warm-up"}
            except Exception as e:  # noqa
                line["gpu_eager_baseline"] = {"error": str(e)[:300]}
        if world == 1 and not args.no_cpu_baseline and not (sd3 or pix):
            try:
                cb = cpu_baseline_sample()
                line["cpu_baseline"] = {"value": cb["images_per_sec"], "unit": UNIT, "cores": cb["threads"], "kind": "port",
                                        "sample": "fp32 CPU oracle, B=1, full width / full 4608-token sequence, fwd + LoRA bwd of one double "
                                                  f"block ({cb['t_double_s']:.1f} s) and one single block ({cb['t_single_s']:.1f} s), "
                                                  "extrapolated as 19 t_double + 38 t_single; `--impl reference` times the 2:4 pattern with medians"}
            except Exception as e:  # noqa
                line["cpu_baseline"] = {"error": str(e)[:200]}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch (default: 4 for flux_lora, 8 for sd3_fullft)")
    ap.add_argument("--config", default="flux_lora", choices=["flux_lora", "sd3_fullft", "pixart_lora", "vae_encode", "flux_lokr", "text_encode"],
                    help="flux_lora = BASELINE configs[1] (the headline metric); sd3_fullft = configs[2] (SD3.5-medium full fine-tune); "
                         "pixart_lora = configs[4] (PixArt-Sigma LoRA r32, mixed buckets, grad-accum 4); vae_encode = the VAE cache path")
    ap.add_argument("--tiny", action="store_true", help="plumbing check on a toy config (not a benchmark value)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-eager-baseline", action="store_true", help="skip the informational eager-torch GPU baseline (N=1 only)")
    ap.add_argument("--optimizer", default="adamw_bf16", choices=["adamw", "adamw_bf16"],
                    help="adamw_bf16 = the reference's default optimizer (one libstb200 launch); adamw = torch.optim.AdamW(fused)")
    ap.add_argument("--graph", default="auto", choices=["auto", "on", "off"],
                    help="capture prepare_batch+fwd+loss+bwd in a CUDA graph per batch shape (auto: on for sd3_fullft, whose step is launch-bound)")
    ap.add_argument("--dp", default="auto", choices=["auto", "flat", "ddp"],
                    help="gradient exchange for N > 1: flat = one NCCL all-reduce of all LoRA gradients after backward "
                         "(training.dist.FlatGradSync); ddp = torch DDP buckets overlapped with backward (the reference's mechanism)")
    ap.add_argument("--lora-target", default="all", help="flux_lora_target preset (flux_lora only; headline = all)")
    ap.add_argument("--lora-dropout", type=float, default=0.0, help="PEFT lora_dropout (flux_lora only; headline = 0.0)")
    ap.add_argument("--gradient-checkpointing", action="store_true",
                    help="re-run every block in backward like the reference's --gradient_checkpointing (not the headline config)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed device-resident steps, write what the last of them computed as DIR/<name>.npy "
                         "(float32; outputs above 4 Mi elements as a fixed seeded sample) to compare two builds output for output")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs --impl b200")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "b200" and args.config in ("sd3_fullft", "pixart_lora") and world > 1 and not args.tiny:
        # every rank must time the SAME multiset of aspect buckets (ranks only start at different offsets in the bucket list),
        # so the timed micro-batches must be whole cycles of it
        nb, accum = (len(SD3_BUCKETS), 1) if args.config == "sd3_fullft" else (len(PIXART_BUCKETS), PIXART_GRAD_ACCUM)
        cyc = nb // math.gcd(nb, accum)
        if args.steps % cyc:
            ap.error(f"--config {args.config} on {world} GPUs times whole bucket cycles: --steps must be a multiple of {cyc}")
    sys.dont_write_bytecode = True   # the benchmark writes nothing into the tree, not even bytecode of modules build() did not import
    # torch seeds its global generators randomly per process; LoRA A init (kaiming_uniform_) and the VAE's sampling noise
    # draw from them, so without this two runs with the same arguments would start from different inputs
    torch.manual_seed(0)
    if args.dp == "auto" and args.config != "sd3_fullft":
        args.dp = "flat"
    if args.warmup < 3 and args.impl == "b200" and not args.tiny:
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    elif args.config == "vae_encode":
        run_vae(args)
    elif args.config == "text_encode":
        run_text(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
