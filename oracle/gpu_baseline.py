"""GPU stand-in for "the reference's own PyTorch path on the same B200" (BASELINE.md §3.1) — BENCH INFRASTRUCTURE ONLY.

The reference sources are not part of this repository, so the number north_star asks us to beat (reference PyTorch-GPU
images/sec) is measured with the oracle, which is pinned bit-identically to the reference (tests/test_oracle_vs_reference.py) and
runs the same torch ops in the same order:

  * precision as the reference CLI sets it: bf16 GPT (`sample_c2i.py:38,46`), fp32 VQ with TF32 allowed
    (`sample_c2i.py:4-6,30`: `torch.backends.cuda.matmul.allow_tf32 = True`, `cudnn.allow_tf32 = True`);
  * the decode loop of `generate.py:105-123` under `sdp_kernel(math only)`, CFG mix + `sample` eager per step, `input_pos += 1`;
  * "eager": every op dispatched from Python (the reference default);
  * "compiled": `torch.compile(model, mode="reduce-overhead", fullgraph=True)` exactly as `sample_c2i.py:66-72` /
    `sample_c2i_ddp.py:169` wrap the model. The oracle keeps its weights and KV caches in plain tensors, so they are
    registered with `torch._dynamo.mark_static_address` (what nn.Module parameters/buffers get implicitly) — otherwise CUDA
    graphs would copy 0.65 GB of weights per replay or be skipped because the caches are mutated inputs. The caches are allocated
    once and zero-filled per call (the reference re-allocates them in `setup_caches` every `generate`, which would force a
    re-record per call; the stand-in gives the reference its steady-state best case).

Timed with CUDA events around whole `generate()+decode_code()` calls, synchronised on both sides (the reference's own
`time.time()` prints have no synchronisation, SURVEY §5). Only bench.py's `gpu_reference` leg imports this module.
"""
from __future__ import annotations

import time

import torch
from torch.nn.attention import SDPBackend, sdpa_kernel

from .gpt_oracle import GPTOracle
from .sampling_oracle import cfg_mix_oracle, sample_oracle
from .vq_oracle import VQOracle


class GpuReference:
    def __init__(self, gpt_state, cfg, vq_state, B, S, grid, cfg_scale=4.0, top_k=2000, temperature=1.0):
        self.orc = GPTOracle(gpt_state, cfg)
        self.vorc = VQOracle(vq_state)
        self.B, self.S, self.g = B, S, grid
        self.cfg_scale, self.top_k, self.temperature = cfg_scale, top_k, temperature
        self.dev = self.orc.device
        self.R = 2 * B if cfg_scale > 1.0 else B
        self.T = 1
        self.orc.setup(self.R, self.T + S)                   # gpt.py:316-330, once (see module docstring)
        self.orc.math_sdp = False                            # the math-only selection wraps the decode loop, generate.py:112
        self.fwd = self.orc.forward
        self.compiled = False

    def compile(self):
        import torch._dynamo as dynamo
        for t in list(self.orc.sd.values()) + self.orc.k + self.orc.v + [self.orc.mask, self.orc.freqs]:
            dynamo.mark_static_address(t)
        self.fwd = torch.compile(self.orc.forward, mode="reduce-overhead", fullgraph=True)     # sample_c2i.py:66-72
        self.compiled = True

    @torch.no_grad()
    def generate(self, cond):
        """generate.py:126-176 for c2i with CFG; returns int tokens [B, S]."""
        orc, S, B = self.orc, self.S, self.B
        for t in orc.k + orc.v:
            t.zero_()
        c = orc.cfg
        cond_all = torch.cat([cond, torch.ones_like(cond) * c.num_classes]) if self.cfg_scale > 1.0 else cond
        sk = dict(temperature=self.temperature, top_k=self.top_k, top_p=1.0, sample_logits=True)
        toks = []
        logits = self.fwd(None, cond_all, torch.arange(0, self.T, device=self.dev))                # prefill, generate.py:77-86
        mixed = cfg_mix_oracle(logits, self.cfg_scale) if self.cfg_scale > 1.0 else logits
        nxt = sample_oracle(mixed[:, -1], **sk)[0]
        toks.append(nxt)
        pos = torch.tensor([self.T], device=self.dev, dtype=torch.int)
        with sdpa_kernel(SDPBackend.MATH):                                                      # generate.py:112
            for _ in range(S - 1):
                x = torch.cat([nxt, nxt]) if self.cfg_scale > 1.0 else nxt
                logits = self.fwd(x.view(-1, 1), None, pos)
                mixed = cfg_mix_oracle(logits, self.cfg_scale) if self.cfg_scale > 1.0 else logits
                nxt = sample_oracle(mixed[:, -1], **sk)[0]
                toks.append(nxt)
                pos += 1
        return torch.cat(toks, dim=1)

    @torch.no_grad()
    def step(self, cond):
        toks = self.generate(cond)
        return self.vorc.decode_code(toks, [self.B, 8, self.g, self.g])                        # sample_c2i.py:92

    def time_steps(self, warmup, reps):
        """(ms per generate()+decode_code() of B images, ms of the AR part alone) by CUDA events."""
        cond = torch.randint(0, 1000, (self.B,), device=self.dev)
        for _ in range(warmup):
            self.step(cond)
        torch.cuda.synchronize()
        e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        tot = ar = 0.0
        for _ in range(reps):
            e[0].record()
            toks = self.generate(cond)
            e[1].record()
            self.vorc.decode_code(toks, [self.B, 8, self.g, self.g])
            e[2].record()
            torch.cuda.synchronize()
            tot += e[0].elapsed_time(e[2])
            ar += e[0].elapsed_time(e[1])
        return tot / reps, ar / reps


def measure(gpt_state, cfg, vq_state, B, S, grid, cfg_scale, top_k, do_compile=True, log=print, budget_s=400.0):
    """Returns {"eager": {...}, "compiled": {...} | {"error": ...}} for one batch size."""
    torch.backends.cuda.matmul.allow_tf32 = True            # sample_c2i.py:4-6
    torch.backends.cudnn.allow_tf32 = True
    t_start = time.time()
    out = {}
    ref = GpuReference(gpt_state, cfg, vq_state, B, S, grid, cfg_scale, top_k)
    ms, ar = ref.time_steps(1, 2)
    out["eager"] = {"images_per_s": B * 1000.0 / ms, "ms_per_step": ms, "ar_us_per_token": 1000.0 * ar / S, "vq_ms": ms - ar}
    log(f"gpu reference eager B={B}: {out['eager']}")
    if do_compile and time.time() - t_start < budget_s:
        try:
            t0 = time.time()
            ref.compile()
            ms, ar = ref.time_steps(2, 3)
            out["compiled"] = {"images_per_s": B * 1000.0 / ms, "ms_per_step": ms, "ar_us_per_token": 1000.0 * ar / S,
                               "vq_ms": ms - ar, "compile_and_warmup_s": round(time.time() - t0 - 3 * ms / 1000.0, 1),
                               "mode": "torch.compile(mode='reduce-overhead', fullgraph=True) on the model forward"}
            log(f"gpu reference compiled B={B}: {out['compiled']}")
        except Exception as ex:                              # never silently drop the leg
            out["compiled"] = {"error": f"{type(ex).__name__}: {str(ex)[-400:]}"}
            log(f"gpu reference compile failed: {out['compiled']['error']}")
    return out
