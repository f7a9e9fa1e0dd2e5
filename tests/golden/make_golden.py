"""Generate golden vectors by RUNNING THE REFERENCE (the original LlamaGen sources) on tiny models.

    python tests/golden/make_golden.py <path to a LlamaGen checkout>

Weights (and the t2i caption features) are not stored: every case keeps a spec from which tests/util.py regenerates them
bit for bit (synth_state_dict), and the reference runs on exactly those tensors. Outputs (committed, small):
  tests/golden/gpt_c2i.pt  gpt_t2i.pt   : weight spec + inputs + reference generate() greedy tokens; the per-step logits as a
                                          sha256 digest plus a fixed sample
  tests/golden/vq_tiny.pt               : weight spec + codes + reference decode_code pixels + argmin indices
  tests/golden/vq_enc_tiny.pt           : weight spec + image + reference z / quant / indices (VQModel.encode)
  tests/golden/sampling.pt              : logits + reference top_k_top_p_filtering / sample outputs
  tests/golden/reference_cases.pt       : the cases of tests/test_oracle_vs_reference.py (generate, RoPE table, VQ decode /
                                          encode, center crop)
  tests/golden/reference_surface.json   : model registries (parameter names and shapes) and sampling-script flags
Every tensor here is an output of the unmodified reference code; nothing is copied from its source.
"""
import json
import math
import os
import re
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.path.abspath(sys.argv[1]) if __name__ == "__main__" else None
sys.path.insert(0, os.path.dirname(HERE))
if REF:
    sys.path.insert(0, REF)

from util import synth_state_dict, synth_tensor, tensor_digest  # noqa: E402

if REF:
    from autoregressive.models.generate import generate, sample, top_k_top_p_filtering  # noqa: E402
    from autoregressive.models.gpt import ModelArgs, Transformer  # noqa: E402

LOGIT_SAMPLE = 512


def gpt_spec(model, seed):
    """Linear / embedding weights U(+-0.02 sqrt 3) (std 0.02, the reference's init), RMSNorm weights 1."""
    tensors = {}
    for k, v in model.state_dict().items():
        assert v.dim() >= 2 or "norm" in k, k
        tensors[k] = [list(v.shape), 1.0, 0.0] if v.dim() == 1 else [list(v.shape), 0.0, 0.02 * math.sqrt(3)]
    return {"seed": seed, "tensors": tensors}


def vq_spec(sd, seed):
    """PyTorch's default conv init bounds (1/sqrt(fan_in)) for weights and biases, GroupNorm 1 / 0, codebook U(+-1/n_e)."""
    tensors = {}
    for k, v in sd.items():
        if v.dim() == 1 and "norm" in k:
            tensors[k] = [list(v.shape), 1.0 if k.endswith("weight") else 0.0, 0.0]
        elif k == "quantize.embedding.weight":
            tensors[k] = [list(v.shape), 0.0, 1.0 / v.shape[0]]
        else:
            w = sd[k[:-len("bias")] + "weight"] if v.dim() == 1 else v
            tensors[k] = [list(v.shape), 0.0, 1.0 / math.sqrt(w[0].numel())]
    return {"seed": seed, "tensors": tensors}


def logit_record(out, key, logits):
    """Digest of the full fp32 logits and a fixed sample of LOGIT_SAMPLE values (the full tensor is ~100 KB)."""
    idx = torch.randperm(logits.numel(), generator=torch.Generator().manual_seed(0))[:LOGIT_SAMPLE].sort().values
    out[key + "_sha256"] = tensor_digest(logits)
    out[key + "_sample"] = (idx, logits.reshape(-1)[idx].clone())
    gap = torch.topk(logits, 2, dim=-1).values
    print(f"  {key}: smallest top-1/top-2 gap {(gap[..., 0] - gap[..., 1]).min().item():.2e}")


def ref_step_logits(model, cond, S, emb_masks, cfg_scale, tokens):
    """Teacher-forced per-step mixed logits from the reference model (fp32): replays generate()'s model
    calls with hooks-free plain forward calls on the same caches."""
    import autoregressive.models.generate as G
    logs = []
    orig = G.sample

    def spy(logits, **kw):
        logs.append(logits[:, -1, :].clone())
        return orig(logits, **kw)

    G.sample = spy
    try:
        out = generate(model, cond, S, emb_masks=emb_masks, cfg_scale=cfg_scale, temperature=1.0, top_k=0,
                       top_p=1.0, sample_logits=False)
    finally:
        G.sample = orig
    assert torch.equal(out, tokens)
    return torch.stack(logs)


def t2i_masks(B, cls, lens):
    em = torch.zeros(B, cls)
    for b, n in enumerate(lens):
        em[b, -n:] = 1
    return em


def gpt_case(model_type, seed):
    torch.manual_seed(seed)
    cls = 1 if model_type == "c2i" else 120
    cfg = dict(n_layer=2, n_head=2, dim=128, vocab_size=512, block_size=16, cls_token_num=cls, model_type=model_type,
               num_classes=10, caption_dim=64, norm_eps=1e-5, rope_base=10000)
    model = Transformer(ModelArgs(**cfg)).eval()
    spec = gpt_spec(model, seed)
    model.load_state_dict(synth_state_dict(spec))
    B, S = 3, 16
    case = dict(cfg=cfg, weights=spec, S=S)
    if model_type == "c2i":
        cond, em = torch.tensor([1, 5, 9]), None
        case["cond"] = cond
    else:
        em = t2i_masks(B, cls, [7, 30, 120])
        case["cond_spec"] = {"seed": seed, "shape": [B, cls, 64], "bound": math.sqrt(3)}
        cond = synth_tensor(seed, "cond", [B, cls, 64], 0.0, math.sqrt(3)) * em[:, :, None]
    case["emb_masks"] = em
    for cfg_scale in (1.0, 4.0):
        toks = generate(model, cond, S, emb_masks=em, cfg_scale=cfg_scale, temperature=1.0, top_k=0, top_p=1.0,
                        sample_logits=False)
        case[f"tokens_cfg{cfg_scale}"] = toks.clone()
        logit_record(case, f"logits_cfg{cfg_scale}", ref_step_logits(model, cond, S, em, cfg_scale, toks))
    # cfg_interval variant (generate.py:113-114)
    case["tokens_cfg4.0_int3"] = generate(model, cond, S, emb_masks=em, cfg_scale=4.0, cfg_interval=3, temperature=1.0,
                                          top_k=0, top_p=1.0, sample_logits=False).clone()
    return case


def vq_decoder(seed, ch_mult, n_e):
    """Tiny decoder (ch=32, z_channels=32) assembled from the reference's own classes exactly as VQModel.decode_code composes
    them (vq_model.py:47-55); VQModel itself hard-codes ch=128 (35 MB of weights)."""
    import torch.nn as nn
    from tokenizer.tokenizer_image.vq_model import Decoder, VectorQuantizer
    torch.manual_seed(seed)
    dec = Decoder(z_channels=32, ch=32, ch_mult=ch_mult).eval()
    quant = VectorQuantizer(n_e, 8, 0.25, 0.0, True, True).eval()
    pqc = nn.Conv2d(8, 32, 1).eval()
    sd = {"decoder." + k: v for k, v in dec.state_dict().items()}
    sd.update({"quantize.embedding.weight": quant.embedding.weight, "post_quant_conv.weight": pqc.weight,
               "post_quant_conv.bias": pqc.bias})
    spec = vq_spec(sd, seed)
    w = synth_state_dict(spec)
    dec.load_state_dict({k[len("decoder."):]: v for k, v in w.items() if k.startswith("decoder.")})
    quant.embedding.weight.data.copy_(w["quantize.embedding.weight"])
    pqc.weight.data.copy_(w["post_quant_conv.weight"])
    pqc.bias.data.copy_(w["post_quant_conv.bias"])
    return spec, dec, quant, pqc


def vq_encoder(seed, ch_mult, n_e):
    """Tiny encoder (ch=32, z_channels=32) + quant_conv + quantizer composed as VQModel.encode does (vq_model.py:41-45)."""
    import torch.nn as nn
    from tokenizer.tokenizer_image.vq_model import Encoder, VectorQuantizer
    torch.manual_seed(seed)
    enc = Encoder(ch=32, ch_mult=ch_mult, z_channels=32).eval()
    quant = VectorQuantizer(n_e, 8, 0.25, 0.0, True, True).eval()
    qc = nn.Conv2d(32, 8, 1).eval()
    sd = {"encoder." + k: v for k, v in enc.state_dict().items()}
    sd.update({"quantize.embedding.weight": quant.embedding.weight, "quant_conv.weight": qc.weight, "quant_conv.bias": qc.bias})
    spec = vq_spec(sd, seed)
    w = synth_state_dict(spec)
    enc.load_state_dict({k[len("encoder."):]: v for k, v in w.items() if k.startswith("encoder.")})
    quant.embedding.weight.data.copy_(w["quantize.embedding.weight"])
    qc.weight.data.copy_(w["quant_conv.weight"])
    qc.bias.data.copy_(w["quant_conv.bias"])
    return spec, enc, quant, qc


def vq_case(seed):
    spec, dec, quant, pqc = vq_decoder(seed, (1, 2), 64)
    codes = torch.randint(0, 64, (2, 16))
    with torch.no_grad():
        pix = dec(pqc(quant.get_codebook_entry(codes, [2, 8, 4, 4], True)))
        z = torch.randn(2, 8, 4, 4)
        idx = quant(z)[2][2]
    return dict(ch=32, z_channels=32, ch_mult=[1, 2], weights=spec, codes=codes, pixels=pix.clone(), z=z, argmin=idx.clone())


def vq_enc_case(seed):
    spec, enc, quant, qc = vq_encoder(seed, (1, 2), 64)
    x = torch.rand(2, 3, 16, 16) * 2 - 1
    with torch.no_grad():
        z = qc(enc(x))
        zq, _, info = quant(z)
    return dict(ch=32, z_channels=32, ch_mult=[1, 2], weights=spec, x=x, z=z.clone(), quant=zq.clone(), indices=info[2].clone())


def sampling_case(seed):
    torch.manual_seed(seed)
    V = 1024
    logits = torch.randn(4, V) * 2.5
    logits[1, 10] = logits[1, 20] = logits[1].topk(5).values[-1]      # tie at the k=5 boundary (SURVEY G8)
    out = dict(logits=logits)
    for k, p in ((0, 1.0), (5, 1.0), (50, 1.0), (V, 1.0), (0, 0.9), (100, 0.5), (1, 1.0)):
        out[f"filtered_k{k}_p{p}"] = top_k_top_p_filtering(logits.clone(), top_k=k, top_p=p)
        idx, probs = sample(logits[:, None, :].clone(), temperature=0.7, top_k=k, top_p=p, sample_logits=False)
        out[f"greedy_k{k}_p{p}"] = idx.clone()
        out[f"probs_k{k}_p{p}"] = probs.clone()
    return out


def reference_cases():
    """The cases tests/test_oracle_vs_reference.py checks the oracle (and the product's RoPE table / center crop) against."""
    from autoregressive.models.gpt import precompute_freqs_cis_2d
    from dataset.augmentation import center_crop_arr
    from PIL import Image
    out = {"generate": {}}
    for model_type, cls in (("c2i", 1), ("t2i", 120)):
        for dtype in (torch.float32, torch.bfloat16):
            cfg = dict(n_layer=2, n_head=2, dim=128, vocab_size=256, block_size=16, cls_token_num=cls, model_type=model_type,
                       num_classes=7, caption_dim=64, norm_eps=1e-5, rope_base=10000)
            m = Transformer(ModelArgs(**cfg)).eval()
            spec = gpt_spec(m, 11)
            m.load_state_dict(synth_state_dict(spec))
            m = m.to(dtype)
            case = dict(cfg=cfg, weights=spec, cfg_scale=3.0, S=16)
            if model_type == "c2i":
                cond, em = torch.tensor([3, 6]), None
                case["cond"] = cond
            else:
                em = t2i_masks(2, cls, [5, 77])
                case["cond_spec"] = {"seed": 11, "shape": [2, cls, 64], "bound": math.sqrt(3)}
                cond = (synth_tensor(11, "cond", [2, cls, 64], 0.0, math.sqrt(3)) * em[:, :, None]).to(dtype)
            case["emb_masks"] = em
            case["tokens"] = generate(m, cond, 16, emb_masks=em, cfg_scale=3.0, temperature=1.0, top_k=0, top_p=1.0,
                                      sample_logits=False).clone()
            out["generate"][f"{model_type}_{str(dtype).split('.')[-1]}"] = case
    out["rope"] = [(grid, hd, cls, tensor_digest(precompute_freqs_cis_2d(grid, hd, 10000, cls)))
                   for grid, hd, cls in ((16, 64, 1), (24, 100, 1), (32, 64, 120))]
    spec, dec, quant, pqc = vq_decoder(5, (1, 2, 2), 128)
    codes = torch.randint(0, 128, (1, 9))
    with torch.no_grad():
        pix = dec(pqc(quant.get_codebook_entry(codes, [1, 8, 3, 3], True)))
    out["vq_decode"] = dict(ch_mult=[1, 2, 2], weights=spec, codes=codes, shape=[1, 8, 3, 3], pixels=pix.clone())
    spec, enc, quant, qc = vq_encoder(6, (1, 2, 2), 128)
    x = torch.rand(1, 3, 24, 16) * 2 - 1
    with torch.no_grad():
        zq, _, info = quant(qc(enc(x)))
    out["vq_encode"] = dict(ch_mult=[1, 2, 2], weights=spec, x=x, quant=zq.clone(), indices=info[2].clone())
    rng = np.random.default_rng(1)
    out["center_crop"] = []
    for shape in [(300, 420), (1100, 900), (256, 256), (513, 2000)]:
        im = Image.fromarray(rng.integers(0, 255, (*shape, 3), dtype=np.uint8))
        for s in (256, 384):
            out["center_crop"].append((shape, s, tensor_digest(torch.from_numpy(np.array(center_crop_arr(im, s))))))
    return out


def reference_surface():
    """Registry keys with every model's parameter names and shapes, and the flags of the sampling scripts."""
    from autoregressive.models.gpt import GPT_models
    from tokenizer.tokenizer_image.vq_model import VQ_models

    def shapes(sd):
        return {k: list(v.shape) for k, v in sd.items()}
    out = {"gpt_models": sorted(GPT_models), "vq_models": sorted(VQ_models), "gpt_b": {}, "vq": {}, "cli_flags": {}}
    for kw in (dict(model_type="c2i", cls_token_num=1, block_size=256), dict(model_type="t2i", cls_token_num=120, block_size=256)):
        out["gpt_b"][kw["model_type"]] = shapes(GPT_models["GPT-B"](**kw).state_dict())
    for name in VQ_models:
        out["vq"][name] = shapes(VQ_models[name](codebook_size=16384, codebook_embed_dim=8).state_dict())
    for script in ("sample_c2i", "sample_t2i", "sample_c2i_ddp"):
        src = open(os.path.join(REF, "autoregressive", "sample", f"{script}.py")).read()
        out["cli_flags"][script] = sorted(set(re.findall(r'add_argument\(\s*"(--[a-z0-9\-]+)"', src)))
    return out


if __name__ == "__main__":
    torch.save(gpt_case("c2i", 0), os.path.join(HERE, "gpt_c2i.pt"))
    torch.save(gpt_case("t2i", 1), os.path.join(HERE, "gpt_t2i.pt"))
    torch.save(vq_case(2), os.path.join(HERE, "vq_tiny.pt"))
    torch.save(sampling_case(3), os.path.join(HERE, "sampling.pt"))
    torch.save(vq_enc_case(4), os.path.join(HERE, "vq_enc_tiny.pt"))
    torch.save(reference_cases(), os.path.join(HERE, "reference_cases.pt"))
    with open(os.path.join(HERE, "reference_surface.json"), "w") as f:
        json.dump(reference_surface(), f, sort_keys=True)
        f.write("\n")
    for f in sorted(os.listdir(HERE)):
        if f.endswith((".pt", ".json")):
            print(f, os.path.getsize(os.path.join(HERE, f)) // 1024, "KiB")
