"""CPU: the oracle restatement must reproduce the golden vectors the REFERENCE produced
(tests/golden/make_golden.py). This is what pins the oracle without the reference sources."""
import pytest
import torch

from oracle import GPTOracle, VQOracle, sample_oracle, top_k_top_p_oracle
from util import golden_inputs as _load, tensor_digest


@pytest.mark.parametrize("name", ["gpt_c2i.pt", "gpt_t2i.pt"])
@pytest.mark.parametrize("cfg_scale", [1.0, 4.0])
def test_gpt_oracle_matches_reference_golden(name, cfg_scale):
    g = _load(name)
    orc = GPTOracle(g["state_dict"], g["cfg"])
    toks, logits = orc.generate(g["cond"], g["S"], emb_masks=g["emb_masks"], cfg_scale=cfg_scale, sample_logits=False)
    assert torch.equal(toks, g[f"tokens_cfg{cfg_scale}"])          # greedy ids bit-exact
    idx, vals = g[f"logits_cfg{cfg_scale}_sample"]
    assert torch.equal(logits.reshape(-1)[idx], vals)
    assert tensor_digest(logits) == g[f"logits_cfg{cfg_scale}_sha256"]   # same ops, same order -> identical fp32


@pytest.mark.parametrize("name", ["gpt_c2i.pt", "gpt_t2i.pt"])
def test_gpt_oracle_cfg_interval(name):
    g = _load(name)
    orc = GPTOracle(g["state_dict"], g["cfg"])
    toks, _ = orc.generate(g["cond"], g["S"], emb_masks=g["emb_masks"], cfg_scale=4.0, cfg_interval=3, sample_logits=False)
    assert torch.equal(toks, g["tokens_cfg4.0_int3"])


def test_vq_oracle_matches_reference_golden():
    g = _load("vq_tiny.pt")
    orc = VQOracle(g["state_dict"], ch_mult=g["ch_mult"])
    pix = orc.decode_code(g["codes"], [2, 8, 4, 4])
    assert torch.equal(pix, g["pixels"])
    assert torch.equal(orc.argmin_indices(g["z"]), g["argmin"])


def test_vq_encode_oracle_matches_reference_golden():
    g = _load("vq_enc_tiny.pt")
    orc = VQOracle(g["state_dict"], ch_mult=g["ch_mult"])
    assert torch.equal(orc.encode_z(g["x"]), g["z"])
    quant, idx = orc.encode(g["x"])
    assert torch.equal(idx, g["indices"])
    assert torch.equal(quant, g["quant"])


@pytest.mark.parametrize("k,p", [(0, 1.0), (5, 1.0), (50, 1.0), (1024, 1.0), (0, 0.9), (100, 0.5), (1, 1.0)])
def test_sampling_oracle_matches_reference_golden(k, p):
    g = _load("sampling.pt")
    f = top_k_top_p_oracle(g["logits"], top_k=k, top_p=p)
    assert torch.equal(f, g[f"filtered_k{k}_p{p}"])
    idx, probs = sample_oracle(g["logits"], temperature=0.7, top_k=k, top_p=p, sample_logits=False)
    assert torch.equal(idx, g[f"greedy_k{k}_p{p}"])
    assert torch.equal(probs, g[f"probs_k{k}_p{p}"])


def test_topk_ties_are_kept():
    # SURVEY G8: [1,3,3,2,0], k=2 keeps both 3s; top-p keeps the first token crossing the threshold
    x = torch.tensor([[1.0, 3.0, 3.0, 2.0, 0.0]])
    f = top_k_top_p_oracle(x, top_k=2)
    assert torch.isinf(f[0, [0, 3, 4]]).all() and (f[0, [1, 2]] == 3).all()
    y = torch.tensor([[2.0, 1.0, 0.0, -1.0]])
    f = top_k_top_p_oracle(y, top_p=0.5)
    assert f[0, 0] == 2 and torch.isinf(f[0, 1:]).all()
