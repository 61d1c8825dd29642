#!/usr/bin/env python
"""bench.py — images/sec of IMAGDressing-v1 garment-conditioned sampling (512x512, 50 DDIM steps, CFG) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 bench.py --gpus N ...

A "step" is one pass of the hot path over one batch of synthetic inputs: garment-UNet pass + 50 x (CFG-batched
denoising UNet + fused CFG/DDIM). Workload at N=1 = BASELINE.json configs[1]: batch-1 512x512 50-step sampling,
random-init SD1.5 + garment UNet (no checkpoints offline). `value` = images/s with inputs resident in HBM (device
events, max over ranks); `e2e` = the same through the public pipeline call (dressing_sd.pipelines ... IMAGDressing_v1)
with pinned HOST inputs, H2D and D2H copies inside the timed region. `roofline` = the dominant kernel timed in
isolation with CUDA events against MEASURED_PEAKS.json; `cpu_baseline` = the fp32 oracle on the host cores on a
bounded sample. `--impl reference` times the reference's CPU PyTorch path (oracle port) only.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

HW = 64  # 512 / 8
STEPS_DDIM = int(os.environ.get("IMAGD_DDIM_STEPS", "50"))  # 50 is the metric; the env knob only shortens ncu runs
GUIDANCE = 7.5
# analytic work model (BASELINE.md §2): TFLOP per 512x512 image = 50 x (0.951 + 0.803) + 0.803
TFLOP_PER_IMAGE = 50 * (0.951 + 0.803) + 0.803


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=1, help="images per GPU per step")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the batch-8/16/32 and configs[2]/[3] sub-records")
    # non-default workloads (BASELINE.json configs[2] / configs[3]); the driver's contract run never passes these
    ap.add_argument("--workload", default="base", choices=["base", "ipa_controlnet", "inpaint", "train"],
                    help="base = configs[1] (the metric); ipa_controlnet = configs[2]; inpaint = configs[3]")
    ap.add_argument("--height", type=int, default=512)
    ap.add_argument("--width", type=int, default=512)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned as DIR/<name>.npy (float32), to compare two builds")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs needs --impl b200: the reference arm times a sample of UNet forwards, not whole steps")
    return a


DUMP_BUDGET_BYTES = 63_000_000  # all files together stay under 64 MB (10^6 bytes) with room for the .npy headers


def dump_outputs(d, **arrays):
    """Write each output as d/<name>.npy in float32. An output past its share of the budget keeps a fixed, seeded sample
    of its elements (d/<name>.npy, flattened) and their flat indices (d/<name>.index.npy)."""
    import numpy as np

    os.makedirs(d, exist_ok=True)
    share = DUMP_BUDGET_BYTES // len(arrays)
    for name, t in arrays.items():
        a = t.detach().float().cpu().numpy()
        if a.nbytes > share:  # 4-byte value + 8-byte index per kept element
            g = torch.Generator().manual_seed(0)
            idx = torch.randperm(a.size, generator=g)[:share // 12].sort().values.numpy()
            np.save(os.path.join(d, f"{name}.index.npy"), idx)
            a = a.reshape(-1)[idx]
        np.save(os.path.join(d, f"{name}.npy"), a)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops", 1590.0), d.get("bf16_tflops_sustained", 1400.0), "measured"
    return 6650.0, 1590.0, 1400.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=lambda: self.lines.extend(self.proc.stdout), daemon=True).start()
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------ model builders
class _no_default_init:
    """Skip torch's default Linear / Conv2d initialisation while the 860 M-parameter models are constructed (tens of
    seconds of CPU); every parameter is overwritten right after."""

    def __enter__(self):
        nn = torch.nn
        self.saved = (nn.Linear.reset_parameters, nn.Conv2d.reset_parameters)
        nn.Linear.reset_parameters = lambda m: None
        nn.Conv2d.reset_parameters = lambda m: None

    def __exit__(self, *exc):
        torch.nn.Linear.reset_parameters, torch.nn.Conv2d.reset_parameters = self.saved


def build_product(dev, workload="base"):
    from adapter.attention_processor import (CacheAttnProcessor2_0, CAttnProcessor2_0, LoraRefSAttnProcessor2_0,
                                             LoRAIPAttnProcessor2_0, RefSAttnProcessor2_0)
    from imagdressing_b200 import modeling
    from imagdressing_b200.scheduler import DDIMScheduler
    if workload == "base":
        from dressing_sd.pipelines.IMAGDressing_v1_pipeline import IMAGDressing_v1
    elif workload == "ipa_controlnet":
        from dressing_sd.pipelines.IMAGDressing_v1_pipeline_ipa_controlnet import IMAGDressing_v1
    else:
        from dressing_sd.pipelines.IMAGDressing_v1_pipeline_controlnet_inpainting import IMAGDressing_v1

    with _no_default_init():  # every parameter is overwritten by init_synthetic_fast_ below
        unet = modeling.UNet2DConditionModel().to(dev, torch.bfloat16)
        ref = modeling.UNet2DConditionModel().to(dev, torch.bfloat16)
        cn = modeling.ControlNetModel().to(dev, torch.bfloat16) if workload != "base" else None
    procs = {}
    for name in unet.attn_processors.keys():  # inference_IMAGdressing.py:70-85
        if name.startswith("mid_block"):
            hidden = unet.config.block_out_channels[-1]
        elif name.startswith("up_blocks"):
            hidden = list(reversed(unet.config.block_out_channels))[int(name[len("up_blocks.")])]
        else:
            hidden = unet.config.block_out_channels[int(name[len("down_blocks.")])]
        if workload == "ipa_controlnet":  # inference_IMAGdressing_ipa_controlnetpose.py:80-99 (rank-128 LoRA, 4 face tokens)
            procs[name] = (LoraRefSAttnProcessor2_0(name, hidden) if name.endswith("attn1.processor")
                           else LoRAIPAttnProcessor2_0(hidden, unet.config.cross_attention_dim, rank=128, num_tokens=4))
        else:
            procs[name] = (RefSAttnProcessor2_0(name, hidden) if name.endswith("attn1.processor")
                           else CAttnProcessor2_0(name, hidden, unet.config.cross_attention_dim))
    unet.set_attn_processor(procs)
    unet.to(dev, torch.bfloat16)
    ref.set_attn_processor({n: CacheAttnProcessor2_0() for n in ref.attn_processors.keys()})  # :90-94
    modeling.init_synthetic_fast_(unet, 0)
    modeling.init_synthetic_fast_(ref, 1)
    sched = DDIMScheduler(num_train_timesteps=1000, beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear",
                          clip_sample=False, set_alpha_to_one=False, steps_offset=1)  # :119-127
    extra = {}
    if workload != "base":
        modeling.init_synthetic_fast_(cn, 2)
        extra["controlnet"] = cn
        if workload == "ipa_controlnet":
            extra["ip_ckpt"] = None
            unet.invalidate_packed()
    pipe = IMAGDressing_v1(vae=None, reference_unet=ref, unet=unet, tokenizer=None, text_encoder=None,
                           image_encoder=None, ImgProj=None, scheduler=sched, safety_checker=None, feature_extractor=None,
                           **extra)
    if os.environ.get("IMAGD_NO_GRAPH"):  # profiling aid: every kernel launched eagerly so ncu lists them
        pipe._engine.use_cuda_graph = False
    return pipe


def synth_inputs(B, dev, rank=0, pinned=False, workload="base", lh=HW, lw=HW):
    """SURVEY.md §8d synthetic inputs; per-rank seeds derive from the global sample index."""
    g = torch.Generator().manual_seed(42 + 1000 * rank)
    t = dict(latents=torch.randn(B, 4, lh, lw, generator=g), garment=torch.randn(B, 4, lh, lw, generator=g) * 0.18215 * 5,
             prompt=torch.randn(B, 77, 768, generator=g), negative=torch.randn(B, 77, 768, generator=g),
             gtok=torch.randn(B, 16, 768, generator=g))
    if workload != "base":
        t["pose"] = torch.rand(B, 3, lh * 8, lw * 8, generator=g)
    if workload == "ipa_controlnet":
        t["face"] = torch.randn(B, 4, 768, generator=g)
        t["face_null"] = torch.randn(B, 4, 768, generator=g) * 0.1
    if workload == "inpaint":
        t["image_latents"] = torch.randn(B, 4, lh, lw, generator=g)
        m = torch.zeros(B, 1, lh, lw)
        m[:, :, lh // 4: 3 * lh // 4, lw // 4: 3 * lw // 4] = 1.0
        t["mask"] = m
    if pinned:
        return {k: v.pin_memory() for k, v in t.items()}
    return {k: v.to(dev) for k, v in t.items()}


def run_pipe(pipe, x, workload="base"):
    lh, lw = x["latents"].shape[-2:]
    kw = dict(prompt=None, null_prompt=None, negative_prompt=None, ref_image=None, width=lw * 8, height=lh * 8,
              num_inference_steps=STEPS_DDIM, guidance_scale=GUIDANCE, output_type="latent",
              prompt_embeds=x["prompt"], negative_prompt_embeds=x["negative"], latents=x["latents"],
              garment_tokens=x["gtok"], ref_image_latents=x["garment"])
    if workload == "base":
        return pipe(image_scale=1.0, **kw).images
    if workload == "ipa_controlnet":
        return pipe(pose_image=x["pose"], image_scale=1.0, ipa_scale=0.9, s_lora_scale=0.2, c_lora_scale=0.2,
                    face_tokens=x["face"], face_null_tokens=x["face_null"], **kw).images
    return pipe(control_image=x["pose"], strength=1.0, controlnet_conditioning_scale=1.0, image_latents=x["image_latents"],
                mask_latents=x["mask"], **kw).images


# ------------------------------------------------------------------------------------------------ training step (configs[4])
TRAIN_TFLOP_PER_SAMPLE_640x512 = 5.7  # SURVEY.md 8 row a13: 2 x 1.265 (frozen hybrid UNet fwd + dgrad) + 3 x 1.042 (garment UNet)


def build_train(dev):
    """SDModel of reference train.py:244-281 on the product modules: frozen denoising UNet with RefS / C processors, trainable
    garment UNet (cache processors), Resampler and adapter modules; FlatAdamW over the trainable set (train.py:368-398)."""
    from adapter.resampler import Resampler
    from imagdressing_b200 import modeling, train

    pipe = build_product(dev, "base")
    unet, ref = pipe.unet, pipe.reference_unet
    proj = Resampler(dim=768, depth=4, dim_head=64, heads=12, num_queries=16, embedding_dim=1280, output_dim=768, ff_mult=4)
    proj = proj.to(dev, torch.bfloat16)
    modeling.init_synthetic_fast_(proj, 3)
    adapters = torch.nn.ModuleList(unet.attn_processors.values())
    params = train.set_trainable(unet, ref, proj, adapters)
    sd = train.SDModel(unet, ref, proj, adapters)
    opt = train.FlatAdamW(params, lr=1e-5, weight_decay=1e-2)
    return sd, opt, pipe.scheduler


def synth_train_batch(B, dev, rank, pinned, lh, lw):
    g = torch.Generator().manual_seed(4242 + 1000 * rank)
    t = dict(latents=torch.randn(B, 4, lh, lw, generator=g) * 0.18215 * 5, ref_latents=torch.randn(B, 4, lh, lw, generator=g) * 0.18215 * 5,
             clip_image_embeddings=torch.randn(B, 257, 1280, generator=g), encoder_hidden_states=torch.randn(B, 77, 768, generator=g),
             noise=torch.randn(B, 4, lh, lw, generator=g), timesteps=torch.randint(0, 1000, (B,), generator=g))
    if pinned:
        return {k: v.pin_memory() for k, v in t.items()}
    return {k: v.to(dev) for k, v in t.items()}


def train_record(a, dev, rank, local, world, B, h, w, steps, warm, dump_dir=None):
    """Training micro-step measured like the sampling workloads: forward + backward of SDModel on the kernels, bucketed NCCL
    gradient all-reduce overlapped with the backward, AdamW; device events, barrier + synchronize, max over ranks.
    `dump_dir`: write the loss of the last timed step there (dump_outputs)."""
    import torch.distributed as dist

    from imagdressing_b200 import _lib, train

    sd, opt, sched = build_train(dev)
    lh, lw = h // 8, w // 8
    xd = synth_train_batch(B, dev, rank, False, lh, lw)
    xh = synth_train_batch(B, dev, rank, True, lh, lw)

    # The eager step is bound by host time (~5 000 launches of Python + ctypes per step); the captured graph is the product
    # path. IMAGD_TRAIN_GRAPH=0 measures the eager sequence; data parallel the graph contains the bucket all-reduces.
    graphed = None
    mode = "eager"
    if os.environ.get("IMAGD_TRAIN_GRAPH", "1") == "1":
        try:
            graphed = train.GraphedTrainStep(sd, sched, opt, xd)
            mode = "cuda-graph"
        except Exception as e:  # noqa: BLE001
            mode = f"eager (graph capture failed: {type(e).__name__}: {e})"[:200]

    def step(x):
        if graphed is not None:
            return graphed(**x)
        return train.train_step(sd, sched, optimizer=opt, **x)

    def step_e2e():
        x = {k: v.to(dev, non_blocking=True) for k, v in xh.items()}
        return float(step(x).cpu())

    def timed(fn, K):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(K):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms)

    losses = [float(step(xd)) for _ in range(max(warm, 1))]
    c = ClockSampler(local)
    if rank == 0:
        c.start()
    l0 = _lib.launch_count
    last = [None]

    def timed_step():
        last[0] = step(xd)

    ms = timed(timed_step, steps)
    launches = _lib.launch_count - l0
    ck = c.stop() if rank == 0 else None
    if dump_dir and rank == 0:
        dump_outputs(dump_dir, loss=last[0])
    del last
    ms_e2e = timed(step_e2e, steps)
    _, tf_burst, tf_sus, _ = peaks()
    sps = world * B * steps / (ms * 1e-3)
    rec = {"workload": "train", "step_mode": mode, "micro_batch_per_gpu": B, "global_batch": world * B, "height": h, "width": w,
           "samples_per_s": round(sps, 4), "ms_per_step": round(ms / steps, 2), "steps": steps, "warmup": max(warm, 1),
           "e2e_samples_per_s": round(world * B * steps / (ms_e2e * 1e-3), 4),
           "h2d_bytes_per_step": sum(v.numel() * v.element_size() for v in xh.values()), "d2h_bytes_per_step": 4,
           "gpu_launches_per_step": launches // steps, "loss_first_steps": [round(v, 5) for v in losses], "clocks": ck,
           "what": "SDModel.forward (Resampler -> garment UNet taps -> hybrid denoising UNet) + MSE + backward + bucketed "
                   "gradient all-reduce + AdamW, bf16, random-init SD1.5 weights (reference train.py:517-609)"}
    if (h, w) == (640, 512):
        rec["model_tflops"] = round(sps / world * TRAIN_TFLOP_PER_SAMPLE_640x512, 1)
        rec["model_frac_of_sustained_bf16"] = round(sps / world * TRAIN_TFLOP_PER_SAMPLE_640x512 / tf_sus, 4)
    del sd, opt
    from imagdressing_b200 import autograd as _ag

    _ag.clear_cache()  # derived operands / fp32 shadows of the deleted modules
    torch.cuda.empty_cache()
    return rec


# ------------------------------------------------------------------------------------------------ roofline legs
def ncu_traffic_table():
    """DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum) of the roofline kernels, extracted from the
    committed `ncu --set full` captures by tools/ncu_summary.py into profiles/ncu_traffic.json ({kernel: {"bytes": ...,
    "source": "<profiles/ file>"}}); a kernel without a capture reports null."""
    path = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    try:
        return json.load(open(path))
    except Exception:
        return {}


def kernel_roofline(dev, B):
    """Time the step's main kernels alone (CUDA events on the launching stream, L2 flushed between launches) at the
    CFG-batch shapes of batch B: level-0 hybrid attention (B cond samples with garment stream + B uncond), level-0 3x3
    conv, level-0 GEGLU GEMM (LayerNorm folded), level-0 GroupNorm+SiLU. Algorithmic work (SURVEY.md §8d): attention
    4*L*Lkv*C per stream per sample; conv 2*pixels*9*Cin*Cout; GEMM 2*M*N*K; GroupNorm 2 * bytes(x)."""
    from imagdressing_b200 import ops

    hbm, tf_burst, tf_sus, src = peaks()
    flush = torch.empty(160 * 1024 * 1024, device=dev, dtype=torch.int32)  # 640 MB > 126 MB L2

    def timeit(fn, iters=10):
        fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(iters):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        return sum(ts) / len(ts)

    L, C, heads, hd, NB = HW * HW, 320, 8, 40, 2 * B
    qkv = torch.randn(NB, L, 3 * C, device=dev).bfloat16()
    kvr = torch.randn(B, L, 2 * C, device=dev).bfloat16()
    flat = lambda t: t.as_strided((t.shape[0] * t.shape[1], t.shape[2]), (t.stride(1), 1), t.storage_offset())
    s0 = ops.kv_stream(flat(qkv[..., C:2 * C]), flat(qkv[..., 2 * C:]), L)
    s1 = ops.kv_stream(flat(kvr[..., :C]), flat(kvr[..., C:]), L, n_query_samples=B, out_scale=1.0)
    out = torch.empty(NB * L, C, device=dev, dtype=torch.bfloat16)
    ms_attn = timeit(lambda: ops.attention(flat(qkv[..., :C]), NB, L, heads, hd, s0, s1, out=out))
    flops_attn = 4.0 * L * L * C * (NB + B)  # NB self streams + B garment streams
    x = torch.randn(NB, HW, HW, C, device=dev).bfloat16()
    w = (torch.randn(C, 9 * C, device=dev) * 0.02).bfloat16()
    y = torch.empty(NB, HW, HW, C, device=dev, dtype=torch.bfloat16)
    ms_conv = timeit(lambda: ops.conv3x3(x, w, out=y))
    flops_conv = 2.0 * NB * L * 9 * C * C
    tok = torch.randn(NB * L, C, device=dev).bfloat16()
    wg = (torch.randn(8 * C, C, device=dev) * 0.05).bfloat16()
    bg = torch.randn(8 * C, device=dev)
    hg = torch.empty(NB * L, 4 * C, device=dev, dtype=torch.bfloat16)
    ms_geglu = timeit(lambda: ops.gemm(tok, wg, bias=bg, act=ops.ACT_GEGLU, out=hg))
    flops_geglu = 2.0 * NB * L * 8 * C * C
    gam, bet = torch.ones(C, device=dev), torch.zeros(C, device=dev)
    ms_gn = timeit(lambda: ops.groupnorm(x, gam, bet, 32, 1e-5, silu=True, out=y))
    bytes_gn = 2.0 * x.numel() * 2
    traffic = ncu_traffic_table() if B == 1 else {}
    res = {}
    for name, ms, fl in (("hybrid_attention_l0", ms_attn, flops_attn), ("conv3x3_l0", ms_conv, flops_conv),
                         ("geglu_gemm_l0", ms_geglu, flops_geglu)):
        ach = fl / (ms * 1e-3) / 1e12
        t = traffic.get(name, {})
        res[name] = {"bound": "tensor", "achieved": round(ach, 2), "peak": tf_burst, "unit": "TFLOP/s",
                     "frac": round(ach / tf_burst, 4), "traffic": t.get("bytes"), "traffic_source": t.get("source"),
                     "ms": round(ms, 4), "peak_source": src, "algorithmic_gflop_per_launch": round(fl / 1e9, 2)}
    ach = bytes_gn / (ms_gn * 1e-3) / 1e9
    t = traffic.get("groupnorm_silu_l0", {})
    res["groupnorm_silu_l0"] = {"bound": "hbm", "achieved": round(ach, 1), "peak": hbm, "unit": "GB/s",
                                "frac": round(ach / hbm, 4), "traffic": t.get("bytes"), "traffic_source": t.get("source"),
                                "ms": round(ms_gn, 4), "peak_source": src,
                                "algorithmic_mbytes_per_launch": round(bytes_gn / 1e6, 2)}
    return res


FAMILIES = (  # (family, predicate on the profiled launch key) — keys are "symbol(int args...)", see _lib.profile_launches
    ("hybrid_attention_l0", lambda k: k.startswith("imagd_attention_bf16(") and f",{HW * HW},8,40" in k),
    ("attention_other", lambda k: k.startswith("imagd_attention_bf16(")),
    ("conv3x3", lambda k: k.startswith(("imagd_conv3x3_bf16(", "imagd_upconv3x3_bf16("))),
    ("gemm", lambda k: k.startswith("imagd_gemm_bf16(")),
    ("groupnorm", lambda k: k.startswith("imagd_groupnorm_bf16(")),
    ("layernorm", lambda k: k.startswith("imagd_layernorm_bf16(")),
)


def step_shares(pipe):
    """Where one denoising step goes, MEASURED live: the step is launched eagerly once with every C-ABI call bracketed
    by CUDA events on the launching stream; launches are grouped by kernel family. Returns (shares, per_key)."""
    from imagdressing_b200 import _lib

    eng = pipe._engine
    st = next(iter(eng._states.values()))
    st["step_ptr"].zero_()
    eng._step(st)  # warm (eager)
    st["step_ptr"].zero_()
    with _lib.profile_launches() as rec:
        eng._step(st)
    by_key = rec.by_key()
    st["step_ptr"].zero_()
    total = sum(ms for _, ms in by_key.values())
    fam = {}
    for key, (n, ms) in by_key.items():
        name = next((f for f, pred in FAMILIES if pred(key)), "other")
        c, t = fam.get(name, (0, 0.0))
        fam[name] = (c + n, t + ms)
    shares = {k: {"launches": c, "ms": round(t, 4), "share": round(t / total, 4)} for k, (c, t) in
              sorted(fam.items(), key=lambda kv: -kv[1][1])}
    top = sorted(by_key.items(), key=lambda kv: -kv[1][1])[:6]
    return shares, {k: {"launches": n, "ms": round(ms, 4)} for k, (n, ms) in top}, round(total, 4)


def pick_cpu_threads():
    """torch with one thread per logical CPU thrashes on big hosts: probe a few counts on a conv and keep the best."""
    import torch.nn.functional as F

    avail = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    x, w = torch.randn(1, 320, 64, 64), torch.randn(320, 320, 3, 3)
    best, best_t = 1, 1e9
    for n in sorted({min(avail, c) for c in (8, 16, 32, 64, 128)}):
        torch.set_num_threads(n)
        F.conv2d(x, w, padding=1)
        t0 = time.perf_counter()
        for _ in range(3):
            F.conv2d(x, w, padding=1)
        dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = n, dt
    return best


class CpuOracle:
    """The fp32 oracle (reference processors restated; oracle/unet.py) on the host cores, built once."""

    def __init__(self, threads=None):
        from oracle import processors as op
        from oracle import unet as ou

        avail = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
        # a FIXED count, the same in the product line's cpu_baseline and in the --impl reference arm (VERDICT r1 weak #7:
        # the probing pick_cpu_threads chose 32 or 64 from run to run); 32 threads is where the fp32 convs stop scaling
        self.threads = threads or min(32, avail)
        torch.set_num_threads(self.threads)
        with torch.no_grad(), _no_default_init():
            o = ou.UNet2DConditionModel()
            po = {}
            for name in o.attn_processors:
                hidden = {"mid": 1280, "up_blocks.1": 1280, "up_blocks.2": 640, "up_blocks.3": 320, "down_blocks.0": 320,
                          "down_blocks.1": 640, "down_blocks.2": 1280}[next(k for k in (
                              "mid", "up_blocks.1", "up_blocks.2", "up_blocks.3", "down_blocks.0", "down_blocks.1",
                              "down_blocks.2") if name.startswith(k))]
                po[name] = op.RefSAttnProcessor(name, hidden) if "attn1" in name else op.CAttnProcessor(name, hidden, 768)
            o.set_attn_processor(po)
            g = torch.Generator().manual_seed(0)
            for p in o.parameters():
                p.copy_(torch.randn(p.shape, generator=g) * 0.02)
            self.lat, self.txt = torch.randn(1, 4, HW, HW, generator=g), torch.randn(1, 77, 768, generator=g)
            Ls = {320: HW * HW, 640: HW * HW // 4, 1280: HW * HW // 16}
            self.sa = {}
            for name, p in po.items():
                if "attn1" in name:
                    C = p.to_k_ref.weight.shape[0]
                    Lr = HW * HW // 64 if name.startswith("mid") else Ls[C]
                    self.sa[name] = torch.randn(1, Lr, C, generator=g)
            self.t = torch.tensor(981)
            self.o = o
            o(self.lat, self.t, self.txt)  # warm

    def run(self, sample_forwards=10):
        """`sample_forwards` UNet forwards of the B=1 512x512 workload (alternating hybrid / plain), scaled to the
        101 forwards of one image (50 x 2 + 1 garment pass)."""
        with torch.no_grad():
            t0 = time.perf_counter()
            for i in range(sample_forwards):
                if i % 2 == 0:
                    self.o(self.lat, self.t, self.txt, cross_attention_kwargs={"sa_hidden_states": self.sa})
                else:
                    self.o(self.lat, self.t, self.txt)
            dt = time.perf_counter() - t0
        per_fwd = dt / sample_forwards
        img_s = 1.0 / (per_fwd * (2 * STEPS_DDIM + 1))
        return {"value": round(img_s, 6), "unit": "images/s", "cores": self.threads, "kind": "port",
                "sample": f"{sample_forwards} fp32 UNet forwards (B=1, 512x512; alternating hybrid/plain) = {dt:.1f} s, "
                          f"scaled to {2 * STEPS_DDIM + 1} forwards/image", "s_per_forward": round(per_fwd, 3)}


def cpu_train_baseline(h=640, w=512, threads=None):
    """The reference's training step on the host cores: the fp32 oracle (oracle/train_step.py: SDModel forward through both
    UNets + Resampler, MSE, torch-autograd backward; reference train.py:255-281,573-605) for ONE micro-batch-1 sample at
    h x w — a bounded sample of configs[4]'s micro-batch-4 step (samples/s is per sample either way)."""
    from oracle import processors as op
    from oracle import train_step as ts
    from oracle import unet as ou
    from oracle.ddim import DDIMOracle

    avail = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    threads = threads or min(32, avail)
    torch.set_num_threads(threads)
    g = torch.Generator().manual_seed(0)
    with _no_default_init():
        unet, ref = ou.UNet2DConditionModel(), ou.UNet2DConditionModel()
    proj = op.Resampler(dim=768, depth=4, dim_head=64, heads=12, num_queries=16, embedding_dim=1280, output_dim=768, ff_mult=4)
    with torch.no_grad():
        for m in (unet, ref, proj):
            for p in m.parameters():
                p.copy_(torch.randn(p.shape, generator=g) * 0.02)
    adapters = ts.install_training_processors(unet, ref)
    ts.set_trainable(unet, ref, proj, adapters)
    lh, lw = h // 8, w // 8
    r = lambda *sh: torch.randn(*sh, generator=g)
    b = dict(latents=r(1, 4, lh, lw), ref_latents=r(1, 4, lh, lw), clip_image_embeddings=r(1, 257, 1280),
             encoder_hidden_states=r(1, 77, 768), noise=r(1, 4, lh, lw), timesteps=torch.tensor([500]))
    t0 = time.perf_counter()
    loss = float(ts.train_step(unet, ref, proj, DDIMOracle(), **b))
    dt = time.perf_counter() - t0
    return {"value": round(1.0 / dt, 6), "unit": "samples/s", "cores": threads, "kind": "port",
            "sample": f"one fp32 micro-batch-1 training step (forward + backward, {h}x{w}) of the oracle port = {dt:.1f} s; "
                      f"loss {loss:.4f}"}


CPU_SAMPLE_FORWARDS = 10  # per step, in both CPU legs (~15-30 s of CPU work on the GPU box's host)


def cpu_baseline(sample_forwards=CPU_SAMPLE_FORWARDS, threads=None):
    return CpuOracle(threads).run(sample_forwards)


# ------------------------------------------------------------------------------------------------ main
def main():
    a = parse()
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if a.impl == "reference" and a.workload == "train":
        if rank != 0:
            return
        h, w = (640, 512) if (a.height, a.width) == (512, 512) else (a.height, a.width)
        vals = []
        cb = None
        for i in range(min(a.warmup, 1) + max(1, min(a.steps, 3))):  # ~30-60 s each: bounded
            cb = cpu_train_baseline(h, w)
            if i >= min(a.warmup, 1):
                vals.append(cb["value"])
        v = sum(vals) / len(vals)
        cb["value"] = round(v, 6)
        print(json.dumps({"impl": "reference", "metric": f"training samples/sec, {h}x{w} forward+backward", "value": round(v, 6),
                          "unit": "samples/s", "n_gpus": 0, "steps": len(vals), "warmup": min(a.warmup, 1),
                          "ms_per_step": round(1000.0 / v, 1), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                          "dtype": "f32", "data": "synthetic",
                          "config": {"workload": "train.py step (BASELINE.json configs[4]) on the host cores: fp32 oracle port, "
                                                 "micro-batch 1 per step", "global_batch": 1},
                          "cpu_baseline": cb,
                          "e2e": {"value": round(v, 6), "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return
    if a.impl == "reference":
        if rank != 0:
            return
        ms = []
        cb = None
        oracle = CpuOracle()
        for i in range(a.warmup + a.steps):
            cb = oracle.run(sample_forwards=CPU_SAMPLE_FORWARDS)
            if i >= a.warmup:
                ms.append(1000.0 / cb["value"])
        v = 1000.0 / (sum(ms) / len(ms))
        cb["value"] = round(v, 6)
        print(json.dumps({"impl": "reference", "metric": "images/sec, 512x512 50-step DDIM garment-conditioned (CFG)",
                          "value": round(v, 6), "unit": "images/s", "n_gpus": 0, "steps": a.steps, "warmup": a.warmup,
                          "ms_per_step": round(sum(ms) / len(ms), 1), "higher_is_better": True, "scaling": "weak",
                          "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                          "config": {"workload": "batch-1 512x512 50-step DDIM, CFG 7.5, random-init SD1.5 + garment UNet "
                                     "(reference CPU PyTorch path: fp32 oracle port, each step = "
                                     f"{CPU_SAMPLE_FORWARDS} UNet forwards scaled to 101/image)", "global_batch": 1},
                          "cpu_baseline": cb,
                          "e2e": {"value": round(v, 6), "unit": "images/s", "h2d_bytes_per_step": 0,
                                  "d2h_bytes_per_step": 0}}))
        return

    # NCCL_DEBUG is left as the launcher set it (round 1 forced WARN, which hid the communicator's rank count from the
    # driver); the result is still exactly ONE line starting with '{' on stdout, NCCL's own lines start with the host name
    import torch.distributed as dist

    from imagdressing_b200 import _lib

    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    _lib.require_b200()
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B = a.batch
    lh, lw = a.height // 8, a.width // 8
    if a.workload == "train":  # BASELINE.json configs[4]: micro-batch 4 per GPU at 640 x 512 unless overridden
        Bt = a.batch if a.batch != 1 else 4
        h, w = (640, 512) if (a.height, a.width) == (512, 512) else (a.height, a.width)
        rec = train_record(a, dev, rank, local, world, Bt, h, w, a.steps, max(a.warmup, 5), a.dump_outputs)
        cb = None
        if rank == 0 and world == 1 and not a.no_cpu_baseline:
            try:
                cb = cpu_train_baseline(h, w)
            except Exception as e:  # noqa: BLE001
                cb = {"error": f"{type(e).__name__}: {e}"[:200]}
        if rank == 0:
            if cb is not None:
                rec["cpu_baseline"] = cb
            print(json.dumps({
                "metric": f"training samples/sec, {h}x{w} bf16 forward+backward+AdamW, micro-batch {Bt}/GPU", "value": rec["samples_per_s"],
                "unit": "samples/s", "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 3), "ms_per_step": rec["ms_per_step"],
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                "config": {"workload": f"train.py step (BASELINE.json configs[4]): garment UNet + Resampler + adapters trainable, "
                                       f"denoising UNet frozen, micro-batch {Bt}/GPU, {h}x{w}", "global_batch": world * Bt,
                           "parallelism": f"dp{world}"},
                "e2e": {"value": rec["e2e_samples_per_s"], "unit": "samples/s", "h2d_bytes_per_step": rec["h2d_bytes_per_step"],
                        "d2h_bytes_per_step": 4},
                "gpu_launches": rec["gpu_launches_per_step"] * a.steps, "clocks": rec["clocks"], "train": rec}))
        if world > 1:
            dist.destroy_process_group()
        return
    pipe = build_product(dev, a.workload)
    x_dev = synth_inputs(B, dev, rank, False, a.workload, lh, lw)
    x_host = synth_inputs(B, dev, rank, True, a.workload, lh, lw)
    from imagdressing_b200.parallel import gather_latents

    def one_step(x):
        out = run_pipe(pipe, x, a.workload)
        # the single collective of the path: all-gather of the output latents (NCCL over NVLink); no-op at N=1
        return gather_latents(out.contiguous(), world * B)

    def one_step_e2e():
        x = {k: v.to(dev, non_blocking=True) for k, v in x_host.items()}
        return one_step(x).to("cpu", non_blocking=False)

    def timed(fn, K):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(K):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms)

    for _ in range(max(a.warmup, 3)):
        one_step(x_dev)
    clk = ClockSampler(local)
    if rank == 0:
        clk.start()
    l0 = _lib.launch_count
    last = [None]

    def timed_step():
        last[0] = one_step(x_dev)

    ms_total = timed(timed_step, a.steps)
    launches = _lib.launch_count - l0
    clocks = clk.stop() if rank == 0 else None
    if a.dump_outputs and rank == 0:  # before any later call can reuse the output buffer
        dump_outputs(a.dump_outputs, latents=last[0])
    del last
    one_step_e2e()
    ms_e2e = timed(one_step_e2e, a.steps)

    shares = None
    if rank == 0:
        shares, top_keys, eager_ms = step_shares(pipe)

    def extra(workload, Bx, h, w, the_pipe, warm=1, steps=1):
        """One more configuration measured the same way (device events, barrier + synchronize on both sides, max over
        ranks, clocks sampled during the timed region): per-GPU batch Bx of `workload` at h x w pixels."""
        xd = synth_inputs(Bx, dev, rank, False, workload, h // 8, w // 8)
        fn = lambda: gather_latents(run_pipe(the_pipe, xd, workload).contiguous(), world * Bx)
        for _ in range(warm):
            fn()
        c = ClockSampler(local)
        if rank == 0:
            c.start()
        ms = timed(fn, steps)
        ck = c.stop() if rank == 0 else None
        return {"workload": workload, "batch_per_gpu": Bx, "global_batch": world * Bx, "height": h, "width": w,
                "images_per_s": round(world * Bx * steps / (ms * 1e-3), 4), "ms_per_step": round(ms / steps, 2),
                "steps": steps, "warmup": warm, "clocks": ck}

    # north_star: batch 1 / 8 / 16 / 32 at every GPU count — the headline above is the --batch value (1 by default), the
    # others ride along in `batches` (few steps each so the whole run stays within minutes)
    batches, other_configs = [], []
    if standard_run(a) and not a.no_extras:
        for Bx in (8, 16, 32):
            if Bx != B:
                batches.append(extra("base", Bx, a.height, a.width, pipe))
        del pipe
        torch.cuda.empty_cache()
        # BASELINE.json configs[2] (batch-32 IP-Adapter face tokens + ControlNet-pose, 512x512) and configs[3]
        # (768x576 ControlNet-inpainting, 8 per GPU -> global batch 64 at 8 GPUs), through their own pipeline classes
        for workload, Bx, h, w in (("ipa_controlnet", 32, 512, 512), ("inpaint", 8, 768, 576)):
            p2 = build_product(dev, workload)
            other_configs.append(extra(workload, Bx, h, w, p2))
            del p2
            torch.cuda.empty_cache()

    if standard_run(a) and not a.no_extras:
        # BASELINE.json configs[4]: the training step (micro-batch 4 per GPU, 640 x 512), data-parallel over the ranks.
        # A failure here must not cost the headline line: it is reported in the record instead.
        try:
            other_configs.append(train_record(a, dev, rank, local, world, 4, 640, 512, 3, 2))
        except Exception as e:  # noqa: BLE001
            other_configs.append({"workload": "train", "error": f"{type(e).__name__}: {e}"[:300]})

    edges = None
    if rank == 0 and standard_run(a) and not a.no_extras:
        edges = edge_models(dev)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    images = world * B * a.steps
    value = images / (ms_total * 1e-3)
    e2e_v = images / (ms_e2e * 1e-3)
    hbm, tf_burst, tf_sus, src = peaks()
    roofs = kernel_roofline(dev, B)
    # the roofline headline is the kernel with the largest MEASURED share of the step among those timed in isolation
    # (round 1 hard-coded the conv; the level-0 hybrid attention is the largest single kernel)
    fam_of = {"hybrid_attention_l0": "hybrid_attention_l0", "conv3x3_l0": "conv3x3", "geglu_gemm_l0": "gemm",
              "groupnorm_silu_l0": "groupnorm"}
    by_launch = {k: (shares.get(f, {}).get("ms", 0.0) / max(1, shares.get(f, {}).get("launches", 1))) for k, f in
                 fam_of.items()}
    single = {k: shares.get(f, {}).get("share", 0.0) for k, f in fam_of.items()}
    dominant = "hybrid_attention_l0" if single["hybrid_attention_l0"] >= 0.10 else max(single, key=single.get)
    roofline = dict(roofs[dominant])
    roofline["kernel"] = dominant
    roofline["step_share"] = single[dominant]
    roofline["why"] = ("largest single kernel of the step by measured time (family shares in `step_shares`; conv3x3 / gemm "
                       "are families of many shapes, the level-0 hybrid attention is one kernel at one shape)")
    h2d = sum(v.numel() * v.element_size() for v in x_host.values())
    d2h = world * B * 4 * lh * lw * 4
    standard = a.workload == "base" and (lh, lw) == (HW, HW)
    wl = {"base": "garment-conditioned sampling (BASELINE.json configs[1])",
          "ipa_controlnet": "IP-Adapter face tokens (4, rank-128 LoRA processors) + ControlNet-pose residuals "
                            "(BASELINE.json configs[2])",
          "inpaint": "ControlNet inpainting path with the fused per-step latent blend (BASELINE.json configs[3])"}[a.workload]
    line = {
        "metric": f"images/sec, {a.height}x{a.width} 50-step DDIM garment-conditioned (CFG)",
        "value": round(value, 4), "unit": "images/s", "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 3),
        "ms_per_step": round(ms_total / a.steps, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic",
        "config": {"workload": f"batch-{B}/GPU {a.height}x{a.width} (HxW) 50-step DDIM, CFG {GUIDANCE}: {wl}; random-init "
                               "SD1.5 denoising UNet + garment UNet; timed region = garment pass + 50 steps "
                               "(VAE/CLIP excluded)",
                   "global_batch": world * B, "latent": [lh, lw], "ddim_steps": STEPS_DDIM, "parallelism": f"dp{world}",
                   "l2": "activations+weights (3.4 GB bf16) exceed the 126 MB L2; no explicit flush between steps"},
        "e2e": {"value": round(e2e_v, 4), "unit": "images/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
        "gpu_launches": launches, "clocks": clocks,
        "roofline": roofline, "kernels": roofs,
        "step_shares": {"how": "one eager denoising step, every C-ABI launch bracketed by CUDA events on the launching "
                               "stream, grouped by kernel family", "eager_step_kernel_ms": eager_ms, "families": shares,
                        "top_launch_keys": top_keys, "ms_per_launch_of_roofline_kernels": {k: round(v, 4) for k, v in
                                                                                          by_launch.items()}},
    }
    if edges:
        line["edges"] = edges
    if batches:
        line["batches"] = batches
    if other_configs:
        line["other_configs"] = other_configs
    if standard:  # the analytic work model is for the base 512x512 workload only
        line["model_tflops"] = round(value / world * TFLOP_PER_IMAGE, 1)
        line["model_frac_of_sustained_bf16"] = round(value / world * TFLOP_PER_IMAGE / tf_sus, 4)
        for rec in batches:
            rec["model_frac_of_sustained_bf16"] = round(rec["images_per_s"] / world * TFLOP_PER_IMAGE / tf_sus, 4)
    if not a.no_cpu_baseline and world == 1 and standard:
        line["cpu_baseline"] = cpu_baseline()
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def edge_models(dev):
    """The steps either side of the loop, on the same kernels (SURVEY.md 8f rows 1 and 3; excluded from the headline's timed
    region exactly as the metric defines): VAE decode of 32 512x512 images, VAE encode of 1, CLIP ViT-H/14 image encoder
    (hidden_states[-2]) and the SD1.5 text encoder, random-init at the real widths. CUDA events, 1 warm-up + 2 timed calls."""
    from transformers import CLIPTextConfig, CLIPTextModel, CLIPVisionConfig, CLIPVisionModelWithProjection

    from imagdressing_b200 import clip, modeling, vae

    def ev(fn, n=2):
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    out = {}
    with _no_default_init():
        v = vae.AutoencoderKL().to(dev, torch.bfloat16)
    modeling.init_synthetic_fast_(v, 5)
    z = torch.randn(32, 4, HW, HW, device=dev)
    img = torch.rand(1, 3, HW * 8, HW * 8, device=dev) * 2 - 1
    ms = ev(lambda: v.decode(z, return_dict=False))
    out["vae_decode_b32_512x512"] = {"ms": round(ms, 2), "images_per_s": round(32e3 / ms, 2)}
    ms = ev(lambda: v.encode(img))
    out["vae_encode_b1_512x512"] = {"ms": round(ms, 2)}
    del v, z
    torch.cuda.empty_cache()
    torch.manual_seed(0)
    vis = CLIPVisionModelWithProjection(CLIPVisionConfig(hidden_size=1280, intermediate_size=5120, num_hidden_layers=32,
                                                         num_attention_heads=16, image_size=224, patch_size=14,
                                                         projection_dim=1024, hidden_act="gelu")).to(dev, torch.bfloat16).eval()
    enc = clip.accelerate(vis)
    px = torch.randn(2, 3, 224, 224, device=dev)
    out["clip_vit_h14_b2_hidden_states_m2"] = {"ms": round(ev(lambda: enc(px, output_hidden_states=True)), 2)}
    del vis, enc
    txt = CLIPTextModel(CLIPTextConfig(vocab_size=49408, hidden_size=768, intermediate_size=3072, num_hidden_layers=12,
                                       num_attention_heads=12, max_position_embeddings=77, hidden_act="quick_gelu")
                        ).to(dev, torch.bfloat16).eval()
    tenc = clip.accelerate(txt)
    ids = torch.randint(0, 49000, (2, 77), device=dev)
    out["clip_text_b2"] = {"ms": round(ev(lambda: tenc(ids)), 2)}
    torch.cuda.empty_cache()
    return out


def standard_run(a):
    return a.workload == "base" and (a.height, a.width) == (512, 512)


if __name__ == "__main__":
    main()
