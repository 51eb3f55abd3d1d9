#!/usr/bin/env python
"""bench.py — training images/sec of the fused LoRA step (BASELINE.json metric; default = configs[1], Qwen-Image-Edit).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--config NAME] [--dump-outputs DIR]

--config  qwen_edit (default, BASELINE configs[1]) : Qwen-Image-Edit LoRA r=16 bf16, 512x512, cached embeds, batch 4 / GPU
          flux_kontext       (configs[2]) : FLUX-Kontext LoRA r=32 with the YAML target regex, 19+38 blocks, T=512, batch 2 / GPU
          qwen_plus_sharded  (configs[3]) : Qwen-Image-Edit-2509, target + 2 controls (3 x 1024 image tokens, frame offsets 0,1,2), T=448,
                                            batch 4 / GPU, frozen block weights sharded 1/N per rank when N > 1
          qwen_multires      (configs[4]) : Qwen-Image-Edit LoRA r=16, every batch mixes {320^2, 512^2, 640^2} samples (pad-to-max layout, block GEMMs on ragged row bands,
                                            AttentionMaskMseLoss), batch 4 / GPU

b200 arm     : one "step" = noisy-input -> fused MMDiT forward -> flow-matching loss -> fused backward -> NCCL all-reduce of the flat
               LoRA gradient -> clip -> AdamW step; synthetic cached embeddings, random-init weights.  `value` = device-timed (inputs
               resident in HBM), `e2e` = through the public `train_step` with pinned HOST inputs (H2D inside the timed region, loss read
               back every step).  Extras on the same line: `roofline` (the step's dominant GEMM with the epilogue the step really runs,
               plus the attention kernels, each timed live with CUDA events), `cpu_baseline`, `library_baseline` (the eager-PyTorch
               restatement of the reference on the same GPU: cuBLASLt + SDPA, what the reference itself would run here), per-rank times.
reference arm: the reference's eager PyTorch path restated in oracle/mmdit_oracle.py (diffusers/peft are not installable offline —
               DESIGN.md; the restatement is pinned to the reference's own code by tests/test_reference_goldens.py), on the host cores;
               a step is a bounded sample (full-width depth-1 and depth-2 models at B=1, fwd+loss+bwd) fitted linearly in depth.
Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "qwen-image-finetune_b200"))

METRIC = "training images/sec (Qwen-Image-Edit LoRA r=16 bf16, 512x512, cached embeds)"
CFG = dict(layers=60, heads=24, joint=3584, T=352, hw=32, B=4, r=16)  # configs[1] (kept for tools/ that import it)

# algorithmic train FLOPs per image (SURVEY.md §8d): N_blocks * (2 * F_gemm + 3.5 * F_attn), F_gemm = S * 226.49 MF, F_attn = 4 S^2 D
def flop_per_image(n_blocks, S):
    return n_blocks * (2 * S * 226.49e6 + 3.5 * 4 * S ** 2 * 3072)


S_TOK = CFG["T"] + 2 * CFG["hw"] ** 2
FLOP_PER_IMAGE = flop_per_image(CFG["layers"], S_TOK)

CONFIGS = {
    "qwen_edit": dict(model="qwen", blocks=60, T=352, imgs=[(1, 32, 32)] * 2, B=4, r=16, metric=METRIC,
                      workload="Qwen-Image-Edit LoRA r=16 bf16 512x512 cached embeds, 60 blocks D=3072 H=24, S=352 txt + 2x1024 img tokens"),
    "flux_kontext": dict(model="flux", blocks=57, T=512, imgs=[(1, 32, 32)] * 2, B=2, r=32,
                         metric="training images/sec (FLUX-Kontext LoRA r=32 bf16, 512x512, cached embeds)",
                         workload="FLUX-Kontext LoRA r=32 (YAML target regex: every block Linear, AdaLN linears, x_embedder) bf16 512x512, "
                                  "19 double + 38 single blocks, S=512 txt + 2x1024 img tokens"),
    "qwen_plus_sharded": dict(model="qwen", blocks=60, T=448, imgs=[(1, 32, 32)] * 3, B=4, r=16,
                              metric="training images/sec (Qwen-Image-Edit-2509 LoRA r=16 bf16, target + 2 controls 512x512, cached embeds)",
                              workload="Qwen-Image-Edit-2509 (Plus) LoRA r=16 bf16, 3 images/sample with frame offsets 0,1,2, 60 blocks, "
                                       "S=448 txt + 3x1024 img tokens"),
    "qwen_multires": dict(model="qwen", blocks=60, T=352, imgs=None, B=4, r=16,
                          metric="training images/sec (Qwen-Image-Edit LoRA r=16 bf16, multi-resolution {320,512,640}^2, cached embeds)",
                          workload="Qwen-Image-Edit LoRA r=16 bf16, every batch = one 640^2 + one 320^2 + two 512^2 samples (target+control, "
                                   "pad-to-max: 3200 image tokens), AttentionMaskMseLoss, 60 blocks"),
}
MULTIRES_HW = [40, 20, 32, 32]  # latent-patch side of the four samples of a batch (640, 320, 512, 512 px)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops", 1590.0), d.get("bf16_tflops_sustained", 1400.0), "measured"
    return 1590.0, 1400.0, "fallback"


class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.rows, self.proc, self.index, self.first = [], None, index, 0

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def mark(self):
        """Rows sampled before this point (the sampler is started ahead of the barrier: spawning nvidia-smi takes tens of ms, which
        would otherwise delay rank 0's first step and be charged to every rank through the all-reduce) are not part of the result."""
        self.first = len(self.rows)

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        self.rows = self.rows[self.first:] or self.rows[-1:]
        sm = [int(r[0]) for r in self.rows if r and r[0].isdigit()]
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons}


# ====================================================================================================== reference arm
class CpuReference:
    """The reference's eager path (oracle restatement, pinned to the reference's own code by tests/test_reference_goldens.py) on the host
    cores: full-width (D=3072, H=24) models of depth 1 and depth 2 at B=1, bf16 weights, fwd + loss + bwd through the real embedders and
    output head.  step(depth=N) = t1 + (N - 1) * (t2 - t1): linear in depth, the embed / head share counted once.  Thread count: the
    faster of {all cpus the process may use, 32}, chosen AFTER a warm-up pass of each candidate (cold first calls once made 128
    oversubscribed threads look faster than 32)."""

    def __init__(self, cfg, threads=None):
        import torch
        from oracle import mmdit_oracle as mo
        self.mo, self.torch, self.cfg = mo, torch, cfg
        ncpu = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else os.cpu_count()
        g = torch.Generator().manual_seed(1234)
        T = cfg["T"]
        imgs = cfg["imgs"] or [(1, 32, 32)] * 2
        L, Lc = imgs[0][1] * imgs[0][2], sum(f * h * w for f, h, w in imgs[1:])
        rn = lambda *s: torch.randn(*s, generator=g).bfloat16()
        if cfg["model"] == "qwen":
            self.x = dict(image_latents=rn(1, L, 64), control_latents=rn(1, Lc, 64), prompt_embeds=rn(1, T, 3584) * 3,
                          prompt_embeds_mask=torch.ones(1, T, dtype=torch.int64), img_shapes=[list(imgs)], noise=rn(1, L, 64), u=torch.tensor([0.5]))
            mk = lambda d: mo.QwenImageOracle(mo.QwenConfig(num_layers=d))
        else:
            hw = imgs[0][1]
            self.x = dict(image_latents=rn(1, L, 64), control_latents=rn(1, Lc, 64), pooled=rn(1, 768), prompt_embeds=rn(1, T, 4096),
                          text_ids=torch.zeros(T, 3), image_ids=mo.flux_latent_image_ids(hw, hw, 0.0), control_ids=mo.flux_latent_image_ids(hw, hw, 1.0),
                          noise=rn(1, L, 64), t=torch.tensor([0.5]))
            mk = lambda d: mo.FluxOracle(mo.FluxConfig(num_layers=d, num_single_layers=0, guidance_embeds=True))
        self.models = {}
        for d in (1, 2):
            m = mo.init_synthetic_(mk(d))
            mo.add_lora_adapter(m, r=cfg["r"], alpha=cfg["r"], b_std=0.02)
            self.models[d] = m.bfloat16()
        if threads is None:
            cands = sorted({ncpu, min(32, ncpu)})
            best = None
            for n in cands:
                torch.set_num_threads(n)
                self._once(1)  # warm-up of this candidate (allocator, thread pool) — not timed
                t = self._once(1)
                if best is None or t < best[0]:
                    best = (t, n)
            threads = best[1]
        self.threads = threads
        torch.set_num_threads(threads)

    def _once(self, depth):
        m, x = self.models[depth], self.x
        t0 = time.perf_counter()
        if self.cfg["model"] == "qwen":
            loss, _ = self.mo.qwen_compute_loss(m, **x)
        else:
            loss, _ = self.mo.flux_compute_loss_shared(m, x["image_latents"], x["control_latents"], x["pooled"], x["prompt_embeds"], x["text_ids"],
                                                       x["image_ids"], x["control_ids"], noise=x["noise"], t=x["t"])
        loss.backward()
        dt = time.perf_counter() - t0
        m.zero_grad()
        return dt

    def step(self):
        t1, t2 = self._once(1), self._once(2)
        per_block = max(t2 - t1, 0.25 * t1)  # guard against noise making the fit degenerate
        full = t1 + (self.cfg["blocks"] - 1) * per_block
        return dict(t1=t1, t2=t2, per_block_s=per_block, full_step_s=full, images_per_s=1.0 / full, cores=self.threads)

    def sample_text(self, r):
        return (f"B=1, full-width depth-1 ({r['t1']:.2f}s) and depth-2 ({r['t2']:.2f}s) models fwd+loss+bwd, bf16 weights; "
                f"step = t1 + ({self.cfg['blocks']} - 1) x (t2 - t1)")


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = CONFIGS[args.config]
    ref = CpuReference(cfg)
    vals = []
    for i in range(args.warmup + args.steps):
        r = ref.step()
        if i >= args.warmup:
            vals.append(r)
    v = statistics.median([r["images_per_s"] for r in vals])
    line = {"impl": "reference", "metric": cfg["metric"], "value": v, "unit": "images/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 / v, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic",
            "config": {"workload": cfg["workload"] + " (CPU path, fitted in depth)", "name": args.config, "global_batch": 1},
            "cpu_baseline": {"value": v, "unit": "images/s", "cores": vals[-1]["cores"], "kind": "port", "sample": ref.sample_text(vals[-1])},
            "e2e": {"value": v, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    _emit(line)


# ====================================================================================================== B200 arm
def _init_weights(m, dev):
    import torch
    g = torch.Generator(device=dev).manual_seed(1234)
    for k, t in m.w.items():  # N(0, 0.02^2) weights, zero biases, unit norm weights (SURVEY.md §8d cfg 2)
        if k.endswith("_w") and t.ndim >= 2 and "norm" not in k or k in ("norm_out_w",):
            t.normal_(0.0, 0.02, generator=g)


def build_model(dev, layers, cfg=None):
    """Qwen-Image model of `layers` blocks with the configs[1] adapter (also used by tools/profile_step.py)."""
    from qflux_b200.qwen_model import QwenB200Config, QwenImageB200
    cfg = cfg or CONFIGS["qwen_edit"]
    m = QwenImageB200(QwenB200Config(num_layers=layers, num_attention_heads=CFG["heads"], joint_attention_dim=CFG["joint"]), device=dev)
    _init_weights(m, dev)
    m.add_adapter(cfg["r"], cfg["r"], b_std=0.02)
    return m


def build_flux(dev, cfg, scale):
    from qflux_b200.flux_model import FLUX_KONTEXT_YAML_TARGETS as FLUX_YAML_TARGETS, FluxB200, FluxB200Config
    nd, ns = max(1, round(19 * scale)), max(1, round(38 * scale))
    m = FluxB200(FluxB200Config(num_layers=nd, num_single_layers=ns, guidance_embeds=True), device=dev)
    _init_weights(m, dev)
    m.add_adapter(cfg["r"], cfg["r"], target_modules=FLUX_YAML_TARGETS, b_std=0.02)
    return m


def make_batch(cfg, name, host: bool):
    """Synthetic cached embeddings of one step (fp16 latents like the reference's cache, bf16 prompt embeddings)."""
    import torch
    B, T = cfg["B"], cfg["T"]
    pin = (lambda t: t.pin_memory()) if host else (lambda t: t)
    if name == "qwen_multires":
        shapes = [[(1, h, h), (1, h, h)] for h in MULTIRES_HW]
        Lmax = max(h * h for h in MULTIRES_HW)
        x0, ct = torch.zeros(B, Lmax, 64), torch.zeros(B, Lmax, 64)
        for b, h in enumerate(MULTIRES_HW):
            x0[b, : h * h], ct[b, : h * h] = torch.randn(h * h, 64), torch.randn(h * h, 64)
        return dict(image_latents=pin(x0.half()), control_latents=pin(ct.half()), prompt_embeds=pin((torch.randn(B, T, 3584) * 3).bfloat16()),
                    prompt_embeds_mask=torch.ones(B, T, dtype=torch.int64), img_shapes=shapes)
    imgs = cfg["imgs"]
    L, Lc = imgs[0][1] * imgs[0][2], sum(f * h * w for f, h, w in imgs[1:])
    if cfg["model"] == "qwen":
        return dict(image_latents=pin(torch.randn(B, L, 64).half()), control_latents=pin(torch.randn(B, Lc, 64).half()),
                    prompt_embeds=pin((torch.randn(B, T, 3584) * 3).bfloat16()), img_shapes=[list(imgs)] * B)
    from qflux_b200.train_step import FluxKontextStep
    hw = imgs[0][1]
    return dict(image_latents=pin(torch.randn(B, L, 64).half()), control_latents=pin(torch.randn(B, Lc, 64).half()),
                pooled_prompt_embeds=pin(torch.randn(B, 768).bfloat16()), prompt_embeds=pin(torch.randn(B, T, 4096).bfloat16()),
                text_ids=torch.zeros(T, 3), image_ids=FluxKontextStep.latent_image_ids(hw, hw, "cpu", 0.0),
                control_ids=FluxKontextStep.latent_image_ids(hw, hw, "cpu", 1.0))


def _time_kernel(fn, dev, iters=10):
    import torch
    flush = torch.empty(256 << 20, device=dev, dtype=torch.uint8)
    for _ in range(3):
        fn()
    ts = []
    for _ in range(iters):
        flush.zero_()  # L2 flush between timed launches
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return statistics.median(ts)


def kernel_rooflines(dev, B, T, Limg):
    """The step's dominant kernels, each timed stand-alone with CUDA events on the launching stream (L2 flushed between launches):
    the grouped MLP-up projection WITH the epilogue the step runs (GELU + pre-activation: two [M, 4D] outputs), and the attention
    forward / backward at the step's shape.  FLOPs are algorithmic (2 M N K; 4 / 10 x B H S^2 d)."""
    import torch
    from qflux_b200 import lib
    D, H = 3072, 24
    Mi, Mt, N, K = B * Limg, B * T, 4 * D, D
    A0, A1 = torch.randn(Mi, K, device=dev).bfloat16(), torch.randn(Mt, K, device=dev).bfloat16()
    W0, W1 = torch.randn(N, K, device=dev).bfloat16() * 0.02, torch.randn(N, K, device=dev).bfloat16() * 0.02
    b0 = torch.zeros(N, device=dev, dtype=torch.bfloat16)
    o0, o1 = torch.empty(Mi, N, device=dev, dtype=torch.bfloat16), torch.empty(Mt, N, device=dev, dtype=torch.bfloat16)
    u0, u1 = torch.empty_like(o0), torch.empty_like(o1)
    probs = [lib.gemm_problem(A0, W0, o0, bias=b0, out2=u0), lib.gemm_problem(A1, W1, o1, bias=b0, out2=u1)]
    g_ms = _time_kernel(lambda: lib.gemm(probs, N, K, epilogue=lib.EPI_GELU), dev)
    del A0, A1, W0, W1, o0, o1, u0, u1
    S = T + Limg
    mk = lambda: torch.randn(B, H, S, 128, device=dev).bfloat16()
    Q, Kt, V, dO = mk(), mk(), mk(), mk()
    ot, oi = torch.empty(B * T, H * 128, device=dev, dtype=torch.bfloat16), torch.empty(B * Limg, H * 128, device=dev, dtype=torch.bfloat16)
    lse, delta = torch.empty(B, H, S, device=dev), torch.zeros(B, H, S, device=dev)
    f_ms = _time_kernel(lambda: lib.attn_fwd(Q, Kt, V, ot, oi, T, lse), dev)
    dQ, dK, dV = torch.zeros(B, H, S, 128, device=dev), torch.empty_like(Kt), torch.empty_like(V)
    b_ms = _time_kernel(lambda: lib.attn_bwd(Q, Kt, V, dO, lse, delta, dQ, dK, dV, split=T), dev)
    gf, ff, bf_ = 2.0 * (Mi + Mt) * N * K, 4.0 * B * H * S * S * 128, 10.0 * B * H * S * S * 128
    return dict(gemm=(gf / g_ms / 1e9, g_ms, gf), attn_fwd=(ff / f_ms / 1e9, f_ms, ff), attn_bwd=(bf_ / b_ms / 1e9, b_ms, bf_))


def library_baseline(dev, cfg, budget_s=150.0):
    """What the reference itself would run on this GPU: its eager PyTorch step (oracle restatement: cuBLASLt bf16 GEMMs + SDPA, autograd,
    clip, torch AdamW) at the same config, with gradient checkpointing (the reference's shipped setting) and without.  The B200 model
    must have been freed by the caller.  Baseline being measured — never part of the product path."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import library_bar as lb
    out = {}
    t0 = time.time()
    for key, ck in (("grad_checkpointing", True), ("no_checkpointing", False)):
        if time.time() - t0 > budget_s:
            break
        try:
            r = lb._eager_step(cfg["blocks"], cfg["B"], ck, steps=3, warmup=1, T=cfg["T"], imgs=cfg["imgs"])
            out[key] = dict(images_per_s=r["images_per_s"], ms_per_step=r["ms_per_step"], peak_mem_gb=r["peak_mem_gb"])
        except torch.OutOfMemoryError:
            torch.cuda.empty_cache()
            out[key] = dict(error="out of memory on 180 GB")
    return out


DUMP_SAMPLE = 1 << 21  # elements kept of each flat LoRA array (fixed seeded positions): ~8 MB per array in float32


def _step_outputs(m, loss, B):
    """Host copies of what the last train_step handed its caller: the loss, the model's prediction over all image tokens, the summed
    LoRA gradient and the LoRA parameters after the optimizer step.  The flat LoRA arrays (tens of millions of elements at full size)
    are sampled at the same seeded positions every run, so two builds can be compared element for element."""
    import torch

    def sample(flat):
        idx = torch.randperm(flat.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_SAMPLE].sort().values
        return flat[idx.to(flat.device)].float().cpu()
    params = torch.cat([p.detach().reshape(-1) for _, p in sorted(m._lora_params.items())])
    return {"loss": loss.detach().float().reshape(1).cpu(), "pred": m._ws["pred"].view(B, -1, m._ws["pred"].shape[-1]).float().cpu(),
            "lora_grad_sample": sample(m.G32), "lora_params_sample": sample(params)}


def _dump_outputs(out_dir, outputs):
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in outputs.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.numpy())


def run_b200(args):
    import torch
    import torch.distributed as dist
    from qflux_b200 import lib
    from qflux_b200.optim import FusedLoraAdamW
    from qflux_b200.train_step import FluxKontextStep, QwenImageEditStep
    rank, world, local = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    torch.manual_seed(1234 + rank)
    name, cfg = args.config, CONFIGS[args.config]
    scale = args.layers / 60.0 if args.layers else 1.0
    shard = args.shard_weights or (name == "qwen_plus_sharded" and world > 1)
    if cfg["model"] == "qwen":
        m = build_model(dev, args.layers or cfg["blocks"], cfg)
        if shard:
            m.shard_frozen_weights(gather=args.shard_gather)
            shard_gather = m._sharded.gather
        step = QwenImageEditStep(m, "attention_mask" if name == "qwen_multires" else "mse", max_grad_norm=1.0)
    else:
        m = build_flux(dev, cfg, scale)
        if shard:
            m.shard_frozen_weights(gather=args.shard_gather)
            shard_gather = m._sharded.gather
        step = FluxKontextStep(m, "mse", max_grad_norm=1.0)
    n_blocks = (args.layers or cfg["blocks"]) if cfg["model"] == "qwen" else (m.L + m.Ls)
    opt = FusedLoraAdamW(m, lr=1e-4)  # clip + AdamW fused over the flat fp32 LoRA gradient (torch AdamW semantics, fp32 moments)
    B, T = cfg["B"], cfg["T"]
    host = make_batch(cfg, name, host=True)
    bf_keys = ("image_latents", "control_latents", "prompt_embeds", "pooled_prompt_embeds")
    devd = {k: (v.to(dev, torch.bfloat16) if k in bf_keys else (v.to(dev) if torch.is_tensor(v) else v)) for k, v in host.items()}
    h2d = sum(v.numel() * v.element_size() for v in host.values() if torch.is_tensor(v)) + 4 * B
    if name == "qwen_multires":
        toks = [T + 2 * h * h for h in MULTIRES_HW]
        flops_step = sum(flop_per_image(n_blocks, s) for s in toks)  # un-padded algorithmic FLOPs of the batch
        Limg_launch = 2 * max(h * h for h in MULTIRES_HW)
    else:
        Limg_launch = sum(f * h * w for f, h, w in cfg["imgs"])
        flops_step = B * flop_per_image(n_blocks, T + Limg_launch)

    def sync():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # ---------------- device-resident arm
    for _ in range(args.warmup):
        step.train_step(devd, opt)
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    sync()
    clocks.mark()
    n0 = lib.LAUNCHES
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        loss = step.train_step(devd, opt)
    e1.record()
    sync()
    launches = lib.LAUNCHES - n0
    # snapshot of the last timed step, taken before the host-issue and e2e arms below run further optimizer steps
    outputs = _step_outputs(m, loss, B) if args.dump_outputs and rank == 0 else None
    my_ms = e0.elapsed_time(e1) / args.steps
    ms = torch.tensor([my_ms], device=dev)
    per_rank = [my_ms]
    if world > 1:
        allms = [torch.zeros(1, device=dev) for _ in range(world)]
        dist.all_gather(allms, ms)
        per_rank = [float(t.item()) for t in allms]
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_step = ms.item()
    clk = clocks.stop() if rank == 0 else None
    loss_val = float(loss.item())
    # host-side issue time of one step (no synchronisation inside): must stay below the device time, else the GPU starves
    torch.cuda.synchronize()
    th0 = time.perf_counter()
    step.train_step(devd, opt)
    host_issue_ms = (time.perf_counter() - th0) * 1e3
    torch.cuda.synchronize()
    # ---------------- end-to-end arm: pinned host inputs, loss read back every step
    step.train_step(host, opt)
    sync()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step.train_step(host, opt).item()
    torch.cuda.synchronize()
    dt = torch.tensor([time.perf_counter() - t0], device=dev)
    if world > 1:
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    e2e_ips = B * world * args.steps / dt.item()
    # the step's only data-path collective, timed alone: all-reduce(sum) of the flat fp32 LoRA gradient (train_step._sync_and_step)
    allreduce = None
    if world > 1:
        g = torch.zeros_like(m.G32)
        for _ in range(3):
            dist.all_reduce(g)
        sync()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        for _ in range(10):
            dist.all_reduce(g)
        a1.record()
        torch.cuda.synchronize()
        ar = torch.tensor([a0.elapsed_time(a1) / 10], device=dev)
        dist.all_reduce(ar, op=dist.ReduceOp.MAX)
        allreduce = {"bytes": g.numel() * 4, "ms": round(ar.item(), 4), "share_of_step": round(ar.item() / ms_step, 5),
                     "note": "one NCCL all-reduce of the flat fp32 LoRA gradient per optimizer step, after the backward"}
        del g
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    value = B * world / (ms_step / 1e3)
    burst, sustained, which = peaks()
    step_tf = flops_step / (ms_step / 1e3) / 1e12  # per GPU (weak scaling: every rank runs the same per-GPU batch)
    # free the model before the stand-alone kernel timings and the baselines
    del step, opt, m
    torch.cuda.empty_cache()
    kr = kernel_rooflines(dev, B, T, Limg_launch)
    traffic = None
    tp = os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")
    if os.path.exists(tp):
        traffic = json.load(open(tp))
    g_tf, g_ms, g_fl = kr["gemm"]
    roof = {"bound": "tensor",
            "kernel": f"gemm2_kernel<256,false,GELU> (CTA pair, cta_group::2): grouped img+txt MLP-up [{B * Limg_launch}+{B * T},3072]x[12288,3072] "
                      "with the step's epilogue (GELU output + pre-activation, two [M,4D] bf16 stores)",
            "achieved": g_tf, "peak": burst, "unit": "TFLOP/s", "frac": g_tf / burst, "kernel_ms": g_ms, "flop_per_launch": g_fl,
            "traffic": (traffic or {}).get("gemm2_mlp_up_gelu", {}).get("dram_bytes") if name == "qwen_edit" else None,  # measured at that shape only
            "traffic_source": "dram__bytes_read.sum + dram__bytes_write.sum per launch from the ncu --set full capture listed in "
                              "profiles/r02_ncu_traffic.json" if traffic else None,
            "peak_source": f"{which} MEASURED_PEAKS.json bf16_tflops (burst; kernels timed alone, L2 flushed between launches)",
            "other_kernels": {
                "attn_bwd (attention_bwd3.cu, pipelined transposed)": {"achieved": kr["attn_bwd"][0], "frac": kr["attn_bwd"][0] / burst, "kernel_ms": kr["attn_bwd"][1]},
                "attn_fwd (attn_fwd64_kernel)": {"achieved": kr["attn_fwd"][0], "frac": kr["attn_fwd"][0] / burst, "kernel_ms": kr["attn_fwd"][1]}},
            "step_algorithmic_tflops_per_gpu": step_tf, "step_frac_of_sustained": step_tf / sustained, "step_frac_of_burst": step_tf / burst}
    cpu = lib_base = None
    if world == 1 and not args.no_cpu:
        ref = CpuReference(cfg)
        c = ref.step()
        cpu = {"value": c["images_per_s"], "unit": "images/s", "cores": c["cores"], "kind": "port", "sample": ref.sample_text(c)}
        del ref
    if world == 1 and not args.no_library and cfg["model"] == "qwen" and name != "qwen_multires" and not args.layers:
        lib_base = library_baseline(dev, cfg)
    line = {"metric": cfg["metric"], "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic",
            "config": {"workload": cfg["workload"], "name": name, "blocks": n_blocks, "global_batch": B * world, "batch_per_gpu": B,
                       "parallelism": f"dp{world}" + (f"+sharded-frozen-weights({shard_gather}-gather)" if shard else ""),
                       "l2": "inputs > L2: tens of GB of weights + activations stream through 126 MB L2",
                       "optimizer": "qfx_fused_adamw: global-norm clip 1.0 + AdamW on the LoRA params, one kernel over the flat fp32 gradient",
                       "loss": loss_val},
            "clocks": clk, "gpu_launches": launches, "host_issue_ms_per_step": host_issue_ms, "ms_per_step_per_rank": per_rank, "allreduce": allreduce,
            "e2e": {"value": e2e_ips, "unit": "images/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4},
            "roofline": roof, "cpu_baseline": cpu, "library_baseline": lib_base}
    if outputs is not None:
        _dump_outputs(args.dump_outputs, outputs)
    _emit(line)
    if world > 1:
        dist.destroy_process_group()


_JSON_OUT = None


def _emit(line: dict):
    """The ONE JSON line goes to the process's original stdout; everything else (NCCL's version banner, library chatter) was
    re-routed to stderr in main() so that stdout carries nothing but this line."""
    out = _JSON_OUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    global _JSON_OUT
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)  # fd 1 -> stderr for the rest of the run (C libraries print to it directly)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="qwen_edit", choices=list(CONFIGS))
    ap.add_argument("--layers", type=int, default=0, help="debug only: fewer blocks (INVALID as a bench value)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-library", action="store_true", help="skip the library_baseline leg (eager PyTorch on the same GPU)")
    ap.add_argument("--shard-gather", default="auto", choices=["auto", "peer", "nccl"],
                    help="how a sharded block is assembled: copy-engine pulls from IPC-mapped peer shards (one node) or NCCL all-gather")
    ap.add_argument("--shard-weights", action="store_true",
                    help="frozen block weights sharded 1/N per rank, all-gathered per block (default for --config qwen_plus_sharded at N > 1)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (loss, prediction, sampled LoRA gradient and parameters) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs applies to --impl b200")
    if args.impl == "reference":
        run_reference(args)
    else:
        # step 1 of a shape runs eagerly (allocations, kernel attributes), step 2 captures the CUDA graph, step 3 is the first replay:
        # fewer than three warm-up steps would put the capture inside the timed region (the reported "warmup" is what was really done)
        args.warmup = max(args.warmup, 3)
        run_b200(args)


if __name__ == "__main__":
    main()
