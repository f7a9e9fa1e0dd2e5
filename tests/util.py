import ctypes
import hashlib
import os
import zlib

import numpy as np
import torch

from conftest import GOLDEN


def synth_uniform(seed: int, key: str, shape):
    """Uniform values in [-1, 1) as float64, identical on every platform: splitmix64 of (seed, key, element index)
    in integer arithmetic, kept to 24-bit dyadic fractions so every value is exact in float32."""
    n = int(np.prod(shape, dtype=np.int64))
    x = np.arange(n, dtype=np.uint64) + np.uint64(((seed << 32) + zlib.crc32(key.encode())) % (1 << 64))
    x = x * np.uint64(0x9E3779B97F4A7C15)
    x = (x ^ (x >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    x = (x ^ (x >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    x = x ^ (x >> np.uint64(31))
    u = ((x >> np.uint64(40)).astype(np.int64) - (1 << 23)).astype(np.float64) / (1 << 23)
    return torch.from_numpy(u.reshape(tuple(shape)))


def synth_tensor(seed: int, key: str, shape, const: float, bound: float):
    """const + bound * U[-1, 1) in float32 (see synth_uniform)."""
    return (const + bound * synth_uniform(seed, key, shape)).float()


def synth_state_dict(spec: dict):
    """Weights of a golden case from its stored spec {"seed": s, "tensors": {name: [shape, const, bound]}}."""
    return {k: synth_tensor(spec["seed"], k, *v) for k, v in spec["tensors"].items()}


def tensor_digest(t) -> str:
    """sha256 of a tensor's bytes: equal digests <=> bit-identical tensors of the same dtype and shape."""
    t = t.detach().cpu().contiguous()
    return hashlib.sha256(str((tuple(t.shape), str(t.dtype))).encode() + t.view(torch.uint8).numpy().tobytes()).hexdigest()


def golden_inputs(name):
    """A stored golden case with its weights (and, for t2i, its caption features) regenerated from their specs. Outputs of
    the reference that are too large to store are present only as a digest and a sample ("<key>_sha256", "<key>_sample")."""
    g = torch.load(os.path.join(GOLDEN, name), map_location="cpu", weights_only=False)
    if "weights" in g:
        g["state_dict"] = synth_state_dict(g["weights"])
    if "cond_spec" in g:
        s = g["cond_spec"]
        g["cond"] = synth_tensor(s["seed"], "cond", s["shape"], 0.0, s["bound"]) * g["emb_masks"][:, :, None]
    return g


def load_golden(name):
    """golden_inputs() with the reference's per-step logits restored in full: the fp32 oracle recomputes them on the stored
    weights, and they are checked against the stored sample of the reference's logits (the CPU test
    test_oracle_golden.py pins the oracle's logits to the reference's bit for bit through the stored digests)."""
    from oracle import GPTOracle
    g = golden_inputs(name)
    for key in [k[:-len("_sample")] for k in g if k.startswith("logits_cfg") and k.endswith("_sample")]:
        cfg_scale = float(key[len("logits_cfg"):])
        _, logits = GPTOracle(g["state_dict"], g["cfg"]).generate(g["cond"], g["S"], emb_masks=g["emb_masks"], cfg_scale=cfg_scale,
                                                                  sample_logits=False)
        idx, vals = g[key + "_sample"]
        assert (logits.reshape(-1)[idx] - vals).abs().max().item() <= 1e-6, f"{name}: oracle logits drifted from the reference's"
        g[key] = logits
    return g


def build_gpt(cfg: dict, state_dict, dtype, device="cuda"):
    """Instantiate the product Transformer for an arbitrary (tiny) config and load a reference state_dict."""
    from llamagen_b200.gpt import ModelArgs, Transformer
    keys = {k: v for k, v in cfg.items() if k in ModelArgs.__dataclass_fields__}
    m = Transformer(ModelArgs(**keys))
    missing, unexpected = m.load_state_dict(state_dict, strict=False)
    assert not missing and not unexpected, (missing, unexpected)
    return m.to(device=device, dtype=dtype).eval()


def oracle_cfg(model):
    c = model.config
    return dict(n_layer=c.n_layer, n_head=c.n_head, dim=c.dim, norm_eps=c.norm_eps, rope_base=c.rope_base,
                num_classes=c.num_classes, cls_token_num=c.cls_token_num, block_size=c.block_size, model_type=c.model_type)


def cpu_state(model, dtype=None):
    return {k: (v.detach().cpu().to(dtype) if dtype is not None else v.detach().cpu()) for k, v in model.state_dict().items()}


def top2_gap(logits):
    t = torch.topk(logits, 2, dim=-1).values
    return t[..., 0] - t[..., 1]


def test_gemm(x, w):
    """y = x @ w.T through lg_test_gemm (the engine's own GEMM dispatch)."""
    from llamagen_b200 import _lib
    lib = _lib.load()
    M, K = x.shape
    N = w.shape[0]
    dt = _lib.LG_DTYPE_BF16 if x.dtype == torch.bfloat16 else _lib.LG_DTYPE_F32
    y = torch.empty(M, N, dtype=torch.float32, device=x.device)
    scratch = torch.empty(16 * M * N + 1024, dtype=torch.float32, device=x.device)
    _lib.check(lib.lg_test_gemm(_lib.ptr(x), _lib.ptr(w), M, N, K, dt, _lib.ptr(y), _lib.ptr(scratch),
                                ctypes.c_size_t(scratch.numel() * 4), _lib.current_stream(x.device)), "lg_test_gemm")
    return y


def gemm_dx(x, wa, wb=None, mode=0, normw=None, eps=1e-5, h=None):
    """The decode step's direct-epilogue GEMM (lg_test_gemm_dx): mode 0 -> y fp32, 1 -> h updated in place (returned), 2 -> ff."""
    from llamagen_b200 import _lib
    lib = _lib.load()
    M, K = x.shape
    N = wa.shape[0]
    if mode == 0:
        out = torch.empty(M, N, dtype=torch.float32, device=x.device)
    elif mode == 1:
        out = h.clone()
    else:
        out = torch.empty(M, N, dtype=torch.bfloat16, device=x.device)
    _lib.check(lib.lg_test_gemm_dx(_lib.ptr(x), _lib.ptr(wa), _lib.ptr(wb) if wb is not None else None, M, N, K, mode,
                                   _lib.ptr(normw) if normw is not None else None, ctypes.c_float(eps), _lib.ptr(out),
                                   _lib.current_stream(x.device)), "lg_test_gemm_dx")
    return out
