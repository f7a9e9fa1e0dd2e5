#!/usr/bin/env python
"""bench.py — images/sec end-to-end (c2i, 16x16 tokens) on N B200s, plus roofline and CPU baseline.

    python bench.py --gpus N --steps K --warmup W            (N>1: launched by torchrun, one rank per GPU)
    python bench.py --impl reference --gpus N --steps K --warmup W

Workload (BASELINE.json configs[1]): LlamaGen-L c2i 256px (16x16 = 256 tokens), cfg_scale 4.0, top_k 2000,
temperature 1.0, bf16 GPT + VQ-16 decode, batch 64 per GPU, random-init weights (non-zero head, SURVEY G1),
synthetic class labels.  One "step" = generate() + decode_code() for one batch of 64 images.
Scaling is weak: every rank samples its own 64 images per step (replica data-parallel, SURVEY §8e); NCCL is used
only for the initial weight broadcast and the barriers.

Prints ONE JSON line (see the task contract): value = whole-job images/s with labels resident in HBM;
e2e = same through the public API with pinned-host labels (H2D) and uint8 pixels copied back (D2H) every step.
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
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "images/sec end-to-end (c2i, 16x16 tokens)"
UNIT = "images/s"


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=5)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", choices=["ours", "reference", "gpu-reference"], default="ours")
    p.add_argument("--gpt-model", default="GPT-L")
    p.add_argument("--image-size", type=int, default=256)
    p.add_argument("--batch", type=int, default=64, help="images per GPU per step")
    p.add_argument("--cfg-scale", type=float, default=4.0)
    p.add_argument("--top-k", type=int, default=2000)
    p.add_argument("--t2i", action="store_true",
                   help="text-conditioned workload (BASELINE configs[4]): T=120 synthetic T5 features with ragged left-padded masks, "
                        "caption-MLP prefill + S tokens; use with --gpt-model GPT-XL --image-size 512 --batch 8 --cfg-scale 7.5 --top-k 1000")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-roofline", action="store_true")
    p.add_argument("--no-gpu-reference", action="store_true",
                   help="skip the leg that times the reference's PyTorch-GPU path (oracle port, bf16, eager + torch.compile) on this GPU")
    p.add_argument("--gpu-reference-batches", default="64,32", help="per-GPU batch sizes of the gpu_reference leg (first = --batch)")
    p.add_argument("--no-operating-points", action="store_true", help="skip the extra B=32 (north_star B=256 / 8 GPUs) timing of our arm")
    p.add_argument("--seed", type=int, default=0)
    p.add_argument("--latency", action="store_true", help="accepted for compatibility: the batch-1 latency leg now always runs")
    p.add_argument("--no-latency", action="store_true",
                   help="skip the per-token decode latency leg at batch 1 (R=2 rows under CFG, AR sampling only, < 2 s)")
    p.add_argument("--dump-outputs", metavar="DIR",
                   help="after the timed steps, write the fp32 pixels the last timed step returned (rank 0) as DIR/pixels.npy, so that "
                        "two builds can be compared output for output; the inputs depend only on the arguments")
    args = p.parse_args()
    if args.steps < 1:
        p.error("--steps must be at least 1")
    return args


def log(msg):
    print(f"[bench {time.strftime('%H:%M:%S')}] {msg}", file=sys.stderr, flush=True)


DUMP_BYTES = 64 << 20


def dump_outputs(dirname, pixels):
    """Write pixels [B, 3, H, W] as dirname/pixels.npy (float32). A batch over DUMP_BYTES keeps every k-th image (0, k, 2k, ...)
    with the smallest k that fits."""
    import numpy as np
    arr = pixels.detach().float().cpu().numpy()
    stride = -(-arr.nbytes // DUMP_BYTES)
    os.makedirs(dirname, exist_ok=True)
    np.save(os.path.join(dirname, "pixels.npy"), np.ascontiguousarray(arr[::stride]))
    log(f"wrote {dirname}/pixels.npy: images 0::{stride} of {arr.shape[0]}, shape {list(arr[::stride].shape)}")


def host_cores():
    """Cores this process may actually use: affinity mask capped by the cgroup CPU quota (a container can
    show 128 logical CPUs while being throttled to a few; oversubscribing OpenMP there is catastrophic)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = max(1, min(n, int(int(quota) / int(period))))
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                n = max(1, min(n, q // per))
        except Exception:
            pass
    return n


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return dict(hbm_gbs=d["hbm_gbs"], bf16_tflops=d["bf16_tflops"], bf16_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_sustained=1400.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------- model shapes
def model_dims(name):
    from llamagen_b200.gpt import _SHAPES, ModelArgs
    L, H, D = _SHAPES[name]
    F = ModelArgs(n_layer=L, n_head=H, dim=D).ffn_dim
    return L, H, D, F


def algorithmic(name, R, S, T=1, V=16384):
    """SURVEY §8(d): algorithmic bytes / flops of one decode step averaged over the S steps (bf16)."""
    L, H, D, F = model_dims(name)
    cbar = T + (S - 1) / 2.0
    w_bytes = 2 * (L * (4 * D * D + 3 * D * F) + D * V)
    kv_read = 4 * L * R * D * cbar
    kv_write = 4 * L * R * D
    step_bytes = w_bytes + kv_read + kv_write + 4 * R * V
    step_flops = 2 * R * (L * (4 * D * D + 3 * D * F) + D * V) + 4 * L * R * D * cbar
    per_launch = {   # SURVEY §8(d) algorithmic bytes one launch must move: weights (+ fp32 logits once); activations and
        # split-K partials live in L2 and are NOT counted (VERDICT r1: the r1 line counted them and over-stated frac)
        "attention": 4 * R * D * cbar + 4 * R * D,
        "gemm_qkv": 2 * 3 * D * D,
        "gemm_wo": 2 * D * D,
        "gemm_w13": 2 * 2 * F * D,
        "gemm_w2": 2 * D * F,
        "gemm_head": 2 * V * D + 4 * R * V,
    }
    per_launch_flops = {"gemm_qkv": 2 * R * 3 * D * D, "gemm_wo": 2 * R * D * D, "gemm_w13": 2 * R * 2 * F * D,
                        "gemm_w2": 2 * R * D * F, "gemm_head": 2 * R * V * D, "attention": 4 * R * D * cbar}
    return dict(step_bytes=step_bytes, step_flops=step_flops, per_launch=per_launch, per_launch_flops=per_launch_flops)


def kernel_class(name: str) -> str:
    n = name.replace("(anonymous namespace)::", "")
    if "attn_tma" in n or "attention_kernel" in n:
        return "attention"
    if "ConvA" in n or "conv_tc_kernel" in n or "conv_tcw_kernel" in n:
        return "vq_conv_gemm"
    if "EpiVq" in n or "softmax_rows" in n:
        return "vq_attn"
    if "gemm_tc" in n or "gemm_dx" in n or "gemm_skinny" in n or "gemm_mma_kernel" in n or "gemv_small" in n:
        return "dense_gemm"
    if "decode_small" in n:
        return "persistent_decode"
    for key, cls in (("residual_norm", "residual_rmsnorm"), ("qkv_epilogue", "qkv_rope_kvwrite"), ("silu_mul", "silu_mul"),
                     ("sample_kernel", "sample"), ("gn_stats", "vq_gn_stats"), ("gn_apply", "vq_gn_apply"),
                     ("lookup_postquant", "vq_misc")):
        if key in n:
            return cls
    return "embed_misc"


def trace_classes(fn, dev):
    """Per-kernel-class device time of one call of fn(), from CUPTI kernel records (device timestamps)."""
    try:
        import torch
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize(dev)
        out = {}
        for e in prof.events():
            if e.device_type != torch.autograd.DeviceType.CUDA:
                continue
            c = out.setdefault(kernel_class(e.name), {"total_ms": 0.0, "launches": 0})
            c["total_ms"] += (e.time_range.end - e.time_range.start) / 1000.0
            c["launches"] += 1
        return out if out else None
    except Exception as ex:      # pragma: no cover
        log(f"CUPTI trace unavailable: {ex}")
        return None


VQ_GFLOP_PER_IMAGE = {16: 252.7, 24: 570.1, 32: 1017.3}   # SURVEY §8a-7 (conv-hook count on the reference)


# ---------------------------------------------------------------------------------------------- reference arm
def run_reference(args, rank):
    """The reference's algorithm on the host cores: oracle port (the reference is Python and cannot travel to the
    GPU box), torch CPU fp32, all host threads. Each step = a BOUNDED sample of the workload: prefill + 3 decode steps
    at the full batch (the reference attends over all max_seq slots every step, so per-step cost is constant) + VQ
    decode of 1 image, extrapolated to 256 steps / `batch` images."""
    import torch
    from llamagen_b200 import GPT_models, VQ_models
    from oracle import GPTOracle, VQOracle
    if rank != 0:
        return
    cores = host_cores()
    torch.set_num_threads(cores)
    log(f"reference arm: {cores} host threads (os.cpu_count()={os.cpu_count()})")
    torch.manual_seed(args.seed)
    g = args.image_size // 16
    S = g * g
    gpt = GPT_models[args.gpt_model](block_size=S, vocab_size=16384)
    gpt.output.weight.data.normal_(std=0.02)
    c = gpt.config
    cfg = dict(n_layer=c.n_layer, n_head=c.n_head, dim=c.dim, norm_eps=c.norm_eps, rope_base=c.rope_base, num_classes=c.num_classes,
               cls_token_num=1, block_size=S, model_type="c2i")
    orc = GPTOracle(gpt.state_dict(), cfg)
    vq = VQ_models["VQ-16"](codebook_size=16384, codebook_embed_dim=8)
    vorc = VQOracle(vq.state_dict())
    B = args.batch
    n_dec = 3
    cond = torch.randint(0, 1000, (B,))

    def one_sample():
        # generate() on the oracle, truncated to 1 + n_dec tokens but with the full-length cache (max_seq = 1 + S)
        t0 = time.perf_counter()
        orc.setup(2 * B, 1 + S)
        cond_all = torch.cat([cond, torch.full_like(cond, c.num_classes)])
        orc.math_sdp = False
        logits = orc.forward(None, cond_all, torch.arange(0, 1))
        from oracle import cfg_mix_oracle, sample_oracle
        nxt = sample_oracle(cfg_mix_oracle(logits, args.cfg_scale)[:, -1], top_k=args.top_k)[0]
        t_prefill = time.perf_counter() - t0
        orc.math_sdp = True
        t1 = time.perf_counter()
        pos = torch.tensor([1], dtype=torch.int)
        for _ in range(n_dec):
            logits = orc.forward(torch.cat([nxt, nxt]).view(-1, 1), None, pos)
            nxt = sample_oracle(cfg_mix_oracle(logits, args.cfg_scale)[:, -1], top_k=args.top_k)[0]
            pos += 1
        t_dec = (time.perf_counter() - t1) / n_dec
        t2 = time.perf_counter()
        vorc.decode_code(torch.randint(0, 16384, (1, S)), [1, 8, g, g])
        t_vq = time.perf_counter() - t2
        total = t_prefill + (S - 1) * t_dec + B * t_vq
        return B / total, dict(prefill_s=t_prefill, decode_step_s=t_dec, vq_image_s=t_vq)

    with torch.no_grad():
        for _ in range(args.warmup):
            v, d = one_sample()
            log(f"reference warmup sample: {v:.4f} img/s {d}")
        vals, detail = [], None
        t0 = time.perf_counter()
        for _ in range(args.steps):
            v, detail = one_sample()
            vals.append(v)
        wall = time.perf_counter() - t0
    value = sum(vals) / len(vals)
    sample = f"prefill + {n_dec} decode steps at B={B} (R={2*B}) + VQ decode of 1 image per step, extrapolated to {S} tokens x {B} images"
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1000.0 * wall / max(1, args.steps), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            # the workload string is the one our arm prints (the driver compares the two arms' configs); what differs about this
            # arm is said in `arm`
            "config": {"workload": f"LlamaGen {args.gpt_model} c2i {args.image_size}px ({g}x{g} tokens), cfg={args.cfg_scale}, top_k={args.top_k}, "
                                   f"batch={B} per GPU (R={2 * B} rows), AR sampling + VQ-16 decode to fp32 pixels",
                       "global_batch": args.gpus * B, "arm": "oracle port of the reference on the host CPU (fp32, torch), bounded sample extrapolated to the full workload",
                       "extrapolated": True},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample, "detail": detail},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


# ---------------------------------------------------------------------------------------------- GPU reference leg
def run_gpu_reference(args):
    """The reference's own PyTorch path on THIS GPU (BASELINE.md 3.1): oracle port (bit-identical to the live reference, takes
    device tensors), bf16 GPT + fp32/TF32 VQ decode, eager and torch.compile(mode="reduce-overhead", fullgraph=True), same
    batch / cfg / top-k / tokens as our arm, CUDA-event timed. See oracle/gpu_baseline.py."""
    import torch
    from llamagen_b200 import GPT_models, VQ_models
    from oracle import gpu_baseline
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    g = args.image_size // 16
    S = g * g
    torch.manual_seed(args.seed)
    gpt = GPT_models[args.gpt_model](block_size=S, vocab_size=16384)
    gpt.output.weight.data.normal_(std=0.02)
    c = gpt.config
    cfg = dict(n_layer=c.n_layer, n_head=c.n_head, dim=c.dim, norm_eps=c.norm_eps, rope_base=c.rope_base, num_classes=c.num_classes,
               cls_token_num=1, block_size=S, model_type="c2i")
    gsd = {k: v.detach().to(device=dev, dtype=torch.bfloat16 if v.is_floating_point() else v.dtype) for k, v in gpt.state_dict().items()}
    vq = VQ_models["VQ-16"](codebook_size=16384, codebook_embed_dim=8)
    vsd = {k: v.detach().to(dev) for k, v in vq.state_dict().items()}
    out = {"kind": "oracle port of the reference (pinned bit-identical to it), torch " + torch.__version__,
           "precision": "bf16 GPT, fp32 VQ decode with TF32 allowed (sample_c2i.py:4-6,30,38)",
           "timing": "CUDA events around generate()+decode_code(), synchronised both sides", "batches": {}}
    t0 = time.time()
    for b in [int(x) for x in args.gpu_reference_batches.split(",") if x]:
        left = 780.0 - (time.time() - t0)
        if left < 60:
            out["batches"][str(b)] = {"skipped": "time budget of the leg exhausted"}
            continue
        try:
            out["batches"][str(b)] = gpu_baseline.measure(gsd, cfg, vsd, b, S, g, args.cfg_scale, args.top_k, do_compile=True, log=log,
                                                          budget_s=left - 30)
        except Exception as ex:
            out["batches"][str(b)] = {"error": f"{type(ex).__name__}: {str(ex)[-300:]}"}
        torch.cuda.empty_cache()
    emit({"impl": "gpu-reference", "gpu_reference": out})


# ---------------------------------------------------------------------------------------------- our arm
def run_ours(args):
    import ctypes
    import torch
    import torch.distributed as dist
    from llamagen_b200 import GPT_models, VQ_models, generate, _lib
    from llamagen_b200 import distributed as lgd

    rank, world, local = lgd.init_from_env()
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (there is no CPU fallback)"
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    lib = _lib.load()
    g = args.image_size // 16
    S = g * g
    B = args.batch
    R = 2 * B if args.cfg_scale > 1.0 else B

    # weights: rank 0 initialises, NCCL broadcasts once (north_star: "NCCL only for the initial weight broadcast")
    torch.manual_seed(args.seed)
    T = 120 if args.t2i else 1
    if args.t2i:
        gpt = GPT_models[args.gpt_model](block_size=S, vocab_size=16384, cls_token_num=T, model_type="t2i")
    else:
        gpt = GPT_models[args.gpt_model](block_size=S, vocab_size=16384)
    gpt.output.weight.data.normal_(std=0.02)
    gpt = gpt.to(device=dev, dtype=torch.bfloat16).eval()
    vq = VQ_models["VQ-16"](codebook_size=16384, codebook_embed_dim=8).to(dev).eval()
    bcast_bytes = lgd.broadcast_module(gpt) + lgd.broadcast_module(vq)
    torch.manual_seed(lgd.rank_seed(args.seed, rank, world))
    qz = [B, 8, g, g]
    kw = dict(cfg_scale=args.cfg_scale, cfg_interval=-1, temperature=1.0, top_k=args.top_k, top_p=1.0, sample_logits=True)

    from llamagen_b200.pipeline import SamplePipeline
    use_pipe = os.environ.get("LG_BENCH_PIPELINE", "1") != "0"
    pipe = SamplePipeline(gpt, vq, 8, **kw)

    emb_masks = None
    if args.t2i:     # SURVEY 8(d): randn(B,120,2048) x left-padded mask with valid lengths randint(8,120)
        from llamagen_b200.cond import prepare_condition, synthetic_features
        feats, fmask = synthetic_features(B, T, 2048, args.seed + 17, dev, torch.bfloat16)
        cond_t2i, emb_masks = prepare_condition(feats, fmask, left_padding=True)

    def step_resident(labels_dev):
        if use_pipe:       # VQ decode of this batch overlaps the AR sampling of the next one (decode stream)
            return pipe.submit(labels_dev, g, emb_masks=emb_masks)
        toks = generate(gpt, labels_dev, S, emb_masks=emb_masks, **kw)
        return vq.decode_code(toks, qz)

    if args.t2i:
        host_labels = cond_t2i.cpu().pin_memory()
    else:
        host_labels = torch.randint(0, 1000, (B,), dtype=torch.int64).pin_memory()
    host_pixels = torch.empty(B, args.image_size, args.image_size, 3, dtype=torch.uint8).pin_memory()

    def step_e2e():
        labels = host_labels.to(dev, non_blocking=True)                       # H2D every step
        if use_pipe:
            return pipe.submit(labels, g, to_uint8_host=host_pixels, emb_masks=emb_masks)   # decode + uint8 + D2H on the decode stream
        img = step_resident(labels)
        u8 = torch.clamp(127.5 * img + 128.0, 0, 255).permute(0, 2, 3, 1).to(torch.uint8)   # sample_c2i_ddp.py:143
        host_pixels.copy_(u8, non_blocking=True)                              # D2H every step
        return img

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        """Run fn() `steps` times between CUDA events; returns the elapsed ms and what the last call returned."""
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        ev0.record()
        for _ in range(steps):
            out = fn()
        pipe.wait()            # every decode (and D2H) submitted above is inside the timed region
        ev1.record()
        barrier()
        ms = ev0.elapsed_time(ev1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, out

    labels_dev = cond_t2i if args.t2i else torch.randint(0, 1000, (B,), device=dev)
    log(f"rank {rank}: models ready, warming up")
    for _ in range(max(args.warmup, 3)):
        t0 = time.perf_counter()
        step_resident(labels_dev)
        pipe.wait()
        torch.cuda.synchronize()
        log(f"rank {rank}: warmup step {time.perf_counter() - t0:.3f} s")
    step_e2e()
    torch.cuda.synchronize()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    lib.lg_reset_launch_count()
    ms, last_pixels = timed(lambda: step_resident(labels_dev), args.steps)
    launches = int(lib.lg_launch_count())
    ms_e2e, _ = timed(step_e2e, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    log(f"rank {rank}: timed {ms / args.steps:.1f} ms/step resident, {ms_e2e / args.steps:.1f} ms/step e2e")
    value = world * B * args.steps / (ms / 1000.0)
    e2e_value = world * B * args.steps / (ms_e2e / 1000.0)

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic",
            "config": {"workload": f"LlamaGen {args.gpt_model} {'t2i (T=120 synthetic T5 features, ragged masks)' if args.t2i else 'c2i'} {args.image_size}px ({g}x{g} tokens), cfg={args.cfg_scale}, top_k={args.top_k}, "
                                   f"batch={B} per GPU (R={R} rows), AR sampling + VQ-16 decode to fp32 pixels",
                       "kv_cache_bytes": int(4 * model_dims(args.gpt_model)[0] * R * model_dims(args.gpt_model)[2] * ((T + S + 7) // 8 * 8)),
                       "global_batch": world * B, "parallelism": f"replica-dp{world}", "weights": "random-init, output head normal(0.02)",
                       "l2": "working set per step (0.65 GB weights + KV cache up to 3.3 GB + 1 GB activations) exceeds the 126 MB L2; no flush needed",
                       "weight_broadcast_bytes": bcast_bytes,
                       "pipeline": "VQ decode of batch i on a second stream overlaps the AR sampling of batch i+1; all of it inside the timed region" if use_pipe else "sequential"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(host_labels.numel() * host_labels.element_size()),
                    "d2h_bytes_per_step": int(host_pixels.numel()), "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": launches, "clocks": clocks}

    if rank == 0:      # condition prefill alone (c2i: one position; t2i: caption MLP + 120 positions), CUDA events
        for _ in range(2):
            generate(gpt, labels_dev, 1, emb_masks=emb_masks, **kw)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        ev0.record()
        for _ in range(5):
            generate(gpt, labels_dev, 1, emb_masks=emb_masks, **kw)
        ev1.record()
        torch.cuda.synchronize()
        line["prefill_ms"] = round(ev0.elapsed_time(ev1) / 5, 3)

    # ---------------- roofline leg: device-side kernel durations (CUPTI via torch.profiler) of one extra step, rank 0
    if rank == 0 and not args.no_roofline:
        pk = peaks()
        log("roofline leg: tracing one step (CUPTI kernel timestamps)")
        # Additive, isolated kernel durations: PDL off (nothing starts early and waits on its dependency) and ONE decode chain
        # (with two chains the kernels of both run concurrently, share the SMs and summed CUPTI durations exceed wall time).
        lib.lg_set_pdl(0)
        split_env = os.environ.get("LG_SPLIT")
        os.environ["LG_SPLIT"] = "1"
        step_resident(labels_dev)
        pipe.wait()
        torch.cuda.synchronize()

        def traced():
            step_resident(labels_dev)
            pipe.wait()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        traced()
        ev1.record()
        torch.cuda.synchronize()
        traced_wall_ms = ev0.elapsed_time(ev1)
        classes = trace_classes(traced, dev)
        lib.lg_set_pdl(1 if os.environ.get("LG_PDL", "1") != "0" else 0)
        if split_env is None:
            del os.environ["LG_SPLIT"]
        else:
            os.environ["LG_SPLIT"] = split_env
        if classes is None:      # CUPTI unavailable: event-bracketed launches through the library's own profiler
            lib.lg_profile_reset()
            lib.lg_profile_enable(1)
            step_resident(labels_dev)
            torch.cuda.synchronize()
            lib.lg_profile_enable(0)
            classes, i = {}, 0
            while True:
                nm = lib.lg_profile_class_name(i)
                if nm is None:
                    break
                t, n = ctypes.c_double(), ctypes.c_uint64()
                lib.lg_profile_read(i, ctypes.byref(t), ctypes.byref(n))
                if n.value:
                    key = nm.decode()
                    key = "dense_gemm" if key.startswith("gemm_") else key
                    c = classes.setdefault(key, {"total_ms": 0.0, "launches": 0})
                    c["total_ms"] += t.value
                    c["launches"] += int(n.value)
            timing_source = "cudaEvent pairs around eager launches (includes launch latency)"
        else:
            timing_source = "CUPTI kernel timestamps inside the CUDA-graph replay (torch.profiler)"
        alg = algorithmic(args.gpt_model, R, S, T=T)
        L = model_dims(args.gpt_model)[0]
        # algorithmic work of one whole step (S tokens, B images) per kernel class
        work = {
            "attention": {"bytes": alg["per_launch"]["attention"] * L * S, "flops": alg["per_launch_flops"]["attention"] * L * S, "bound": "hbm"},
            "dense_gemm": {"bytes": sum(alg["per_launch"][k] for k in ("gemm_qkv", "gemm_wo", "gemm_w13", "gemm_w2")) * L * S + alg["per_launch"]["gemm_head"] * S,
                           "flops": sum(alg["per_launch_flops"][k] for k in ("gemm_qkv", "gemm_wo", "gemm_w13", "gemm_w2")) * L * S + alg["per_launch_flops"]["gemm_head"] * S,
                           "bound": "hbm"},
            "vq_conv_gemm": {"bytes": None, "flops": B * VQ_GFLOP_PER_IMAGE.get(g, 0.0) * 1e9, "bound": "tensor"},
        }
        total_ms = sum(v["total_ms"] for v in classes.values())
        line["kernels"] = {}
        for k, v in sorted(classes.items(), key=lambda kv: -kv[1]["total_ms"]):
            e = {"total_ms": round(v["total_ms"], 3), "launches": v["launches"], "avg_us": round(1000.0 * v["total_ms"] / v["launches"], 2),
                 "share": round(v["total_ms"] / total_ms, 4)}
            if k in work:
                if work[k]["bytes"]:
                    e["hbm_gbs"] = round(work[k]["bytes"] / (v["total_ms"] * 1e-3) / 1e9, 1)
                e["tflops"] = round(work[k]["flops"] / (v["total_ms"] * 1e-3) / 1e12, 1)
            line["kernels"][k] = e
        dom = max((k for k in classes if k in work), key=lambda k: classes[k]["total_ms"], default=None)
        traffic = None
        try:     # DRAM bytes per launch of the dominant kernel from the committed `ncu --set full` capture
            tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
            traffic = tj.get(dom, {}).get("dram_bytes_per_launch")
        except Exception:
            pass
        if dom:
            v = classes[dom]
            if work[dom]["bound"] == "hbm":
                ach = work[dom]["bytes"] / (v["total_ms"] * 1e-3) / 1e9
                line["roofline"] = {"kernel": dom, "bound": "hbm", "achieved": ach, "peak": pk["hbm_gbs"], "unit": "GB/s",
                                    "frac": ach / pk["hbm_gbs"], "traffic": traffic, "peak_source": pk["source"],
                                    "algorithmic_bytes_per_launch": work[dom]["bytes"] / v["launches"],
                                    "avg_launch_us": 1000.0 * v["total_ms"] / v["launches"],
                                    "timing": timing_source + "; traced with PDL off and a single decode chain so durations are additive and isolated",
                                    "algorithmic_bytes": "SURVEY 8(d): weight bytes of the GEMM (+ fp32 logits for the head); no activations, no split-K partials"}
            else:
                ach = work[dom]["flops"] / (v["total_ms"] * 1e-3) / 1e12
                line["roofline"] = {"kernel": dom, "bound": "tensor", "achieved": ach, "peak": pk["bf16_sustained"], "unit": "TFLOP/s",
                                    "frac": ach / pk["bf16_sustained"], "traffic": traffic, "peak_source": pk["source"],
                                    "algorithmic_flops_per_launch": work[dom]["flops"] / v["launches"],
                                    "avg_launch_us": 1000.0 * v["total_ms"] / v["launches"], "timing": timing_source + "; traced with PDL off so durations are additive"}
        step_roof_ms = 1000.0 * max(alg["step_bytes"] / (pk["hbm_gbs"] * 1e9), alg["step_flops"] / (pk["bf16_sustained"] * 1e12))
        vq_roof_ms = B * VQ_GFLOP_PER_IMAGE.get(g, 0.0) / (pk["bf16_sustained"] * 1e3) * 1e3
        total_vq = sum(v["total_ms"] for k, v in classes.items() if k.startswith("vq_"))
        line["step_roofline"] = {"decode_step_floor_us": round(step_roof_ms * 1000, 1), "ar_floor_ms": round(step_roof_ms * S, 2),
                                 "vq_floor_ms": round(vq_roof_ms, 2), "measured_ms_per_step": round(ms / args.steps, 2),
                                 "frac_of_floor": round((step_roof_ms * S + vq_roof_ms) / (ms / args.steps), 4),
                                 "traced_ar_kernel_ms": round(total_ms - total_vq, 2), "traced_vq_kernel_ms": round(total_vq, 2),
                                 "traced_step_wall_ms": round(traced_wall_ms, 2),
                                 "note": "traced_* come from the single-chain, PDL-off trace step (sum of isolated kernel durations <= its wall time); "
                                         "measured_ms_per_step is the shipped configuration"}

    # ---------------- batch-1 per-token latency (BASELINE.json metric, second half), rank 0
    if rank == 0 and not args.no_latency:
        lab1 = cond_t2i[:1].contiguous() if args.t2i else torch.randint(0, 1000, (1,), device=dev)
        em1 = emb_masks[:1].contiguous() if args.t2i else None
        for _ in range(3):
            generate(gpt, lab1, S, emb_masks=em1, **kw)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        ev0.record()
        reps = 5
        for _ in range(reps):
            generate(gpt, lab1, S, emb_masks=em1, **kw)
        ev1.record()
        torch.cuda.synchronize()
        us_tok = 1000.0 * ev0.elapsed_time(ev1) / reps / S
        alg1 = algorithmic(args.gpt_model, 2, S, T=T)
        floor_us = 1e6 * alg1["step_bytes"] / (peaks()["hbm_gbs"] * 1e9)
        line["latency_b1"] = {"us_per_token": round(us_tok, 2), "hbm_floor_us": round(floor_us, 2), "frac_of_hbm_roofline": round(floor_us / us_tok, 4),
                              "rows": 2, "note": "generate() of 1 image incl. prefill and sampling, / tokens"}

    # ---------------- north_star's per-GPU operating point (B=256 over 8 GPUs -> 32 images per GPU), our arm, rank 0
    if rank == 0 and world == 1 and not args.no_operating_points and B != 32 and not args.t2i:
        b2 = 32
        gpt._workspace, gpt._ws_shape = None, (0, 0)          # a workspace sized for R = 64 rows (the chain split keys on it)
        lab2 = torch.randint(0, 1000, (b2,), device=dev)
        for _ in range(2):
            pipe.submit(lab2, g)
        pipe.wait()
        torch.cuda.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n2 = 4
        ev0.record()
        for _ in range(n2):
            pipe.submit(lab2, g)
        pipe.wait()
        ev1.record()
        torch.cuda.synchronize()
        ms2 = ev0.elapsed_time(ev1) / n2
        line["operating_points"] = {"batch32": {"images_per_s": b2 * 1000.0 / ms2, "ms_per_step": ms2, "rows": 2 * b2,
                                                "note": "north_star headline shape: GPT-L 256-token c2i at B=256 over 8 GPUs = 32 images per GPU"}}
        gpt._workspace, gpt._ws_shape = None, (0, 0)

    # ---------------- reference PyTorch-GPU path on this same GPU (BASELINE.md 3.1; the number north_star asks us to beat), rank 0, N=1
    if rank == 0 and world == 1 and not args.no_gpu_reference and not args.t2i:
        try:
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "gpu-reference", "--gpt-model", args.gpt_model,
                                "--image-size", str(args.image_size), "--cfg-scale", str(args.cfg_scale), "--top-k", str(args.top_k),
                                "--gpu-reference-batches", ",".join([str(B)] + [b for b in args.gpu_reference_batches.split(",") if b and int(b) != B][:1])],
                               capture_output=True, text=True, timeout=900, env={**os.environ, "CUDA_VISIBLE_DEVICES": str(local)})
            ref = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
            line["gpu_reference"] = ref["gpu_reference"]
            ours = {str(B): value / world}
            if "operating_points" in line:
                ours["32"] = line["operating_points"]["batch32"]["images_per_s"]
            for b, res in line["gpu_reference"]["batches"].items():
                best = max((res.get(k, {}).get("images_per_s") or 0.0) for k in ("eager", "compiled"))
                if b in ours and best > 0:
                    res["ours_images_per_s"] = ours[b]
                    res["ours_over_best_reference"] = ours[b] / best
        except Exception as ex:   # never silently drop the leg
            tail = ""
            try:
                tail = r.stderr[-300:]
            except Exception:
                pass
            line["gpu_reference"] = {"error": f"{type(ex).__name__}: {str(ex)[-200:]} {tail}"}
        log("gpu reference leg done")

    # ---------------- CPU baseline leg (rank 0, N=1 only): bounded sample of the same workload on the host cores
    if rank == 0 and world == 1 and not args.no_cpu_baseline and not args.t2i:
        try:
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "1", "--warmup", "1",
                                "--gpt-model", args.gpt_model, "--image-size", str(args.image_size), "--batch", str(B)],
                               capture_output=True, text=True, timeout=600, env={**os.environ, "CUDA_VISIBLE_DEVICES": ""})
            ref = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
            line["cpu_baseline"] = ref["cpu_baseline"]
        except Exception as ex:   # never silently drop the leg
            line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": host_cores(), "kind": "port",
                                    "sample": f"failed: {type(ex).__name__}: {str(ex)[-300:]}"}
        log("cpu baseline leg done")
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, last_pixels)
    if rank == 0:
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


_REAL_STDOUT = None


def quiet_stdout():
    """Route everything libraries print to fd 1 (e.g. NCCL's version banner) to stderr; the single JSON line is
    written to the real stdout by emit()."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line: dict):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    args = parse()
    quiet_stdout()
    if args.impl == "gpu-reference":
        run_gpu_reference(args)
        return
    if args.impl == "reference":
        rank = int(os.environ.get("RANK", "0"))
        run_reference(args, rank)
        return
    run_ours(args)


if __name__ == "__main__":
    main()
