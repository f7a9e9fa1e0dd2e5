"""CPU: the oracle (and the product's RoPE table, registries and center crop) against outputs of the reference
itself, recorded by tests/golden/make_golden.py from the original LlamaGen sources into tests/golden/reference_cases.pt
and tests/golden/reference_surface.json."""
import json
import os

import pytest
import torch

from conftest import GOLDEN
from oracle import GPTOracle, VQOracle, rope_table_2d_oracle
from util import synth_state_dict, synth_tensor, tensor_digest

CASES = torch.load(os.path.join(GOLDEN, "reference_cases.pt"), map_location="cpu", weights_only=False)
SURFACE = json.load(open(os.path.join(GOLDEN, "reference_surface.json")))


def _shapes(sd):
    return {k: list(v.shape) for k, v in sd.items()}


@pytest.mark.parametrize("model_type,cls", [("c2i", 1), ("t2i", 120)])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_generate_matches_live_reference(model_type, cls, dtype):
    c = CASES["generate"][f"{model_type}_{str(dtype).split('.')[-1]}"]
    assert c["cfg"]["cls_token_num"] == cls
    sd = {k: v.to(dtype) for k, v in synth_state_dict(c["weights"]).items()}
    if model_type == "c2i":
        cond = c["cond"]
    else:
        s = c["cond_spec"]
        cond = (synth_tensor(s["seed"], "cond", s["shape"], 0.0, s["bound"]) * c["emb_masks"][:, :, None]).to(dtype)
    toks, _ = GPTOracle(sd, c["cfg"]).generate(cond, c["S"], emb_masks=c["emb_masks"], cfg_scale=c["cfg_scale"],
                                              sample_logits=False)
    assert torch.equal(c["tokens"], toks)


def test_rope_table_matches_live_reference():
    from llamagen_b200.gpt import rope_table_2d
    for grid, hd, cls, digest in CASES["rope"]:
        assert tensor_digest(rope_table_2d_oracle(grid, hd, 10000, cls)) == digest
        assert tensor_digest(rope_table_2d(grid, hd, 10000, cls)) == digest


def test_registry_matches_live_reference():
    """Same keys, same parameter names and shapes as the reference registries (drop-in boundary §8b)."""
    from llamagen_b200 import GPT_models
    assert SURFACE["gpt_models"] == sorted(GPT_models)
    for kw in (dict(model_type="c2i", cls_token_num=1, block_size=256), dict(model_type="t2i", cls_token_num=120, block_size=256)):
        assert _shapes(GPT_models["GPT-B"](**kw).state_dict()) == SURFACE["gpt_b"][kw["model_type"]]


def test_vq_registry_matches_live_reference():
    from llamagen_b200 import VQ_models
    assert SURFACE["vq_models"] == sorted(VQ_models)
    for name in SURFACE["vq_models"]:
        assert _shapes(VQ_models[name](codebook_size=16384, codebook_embed_dim=8).state_dict()) == SURFACE["vq"][name]


def test_vq_decode_matches_live_reference():
    c = CASES["vq_decode"]
    pix = VQOracle(synth_state_dict(c["weights"]), ch_mult=tuple(c["ch_mult"])).decode_code(c["codes"], c["shape"])
    assert torch.equal(c["pixels"], pix)


def test_vq_encode_matches_live_reference():
    c = CASES["vq_encode"]
    q, idx = VQOracle(synth_state_dict(c["weights"]), ch_mult=tuple(c["ch_mult"])).encode(c["x"])
    assert torch.equal(idx, c["indices"]) and torch.equal(q, c["quant"])


def test_center_crop_matches_live_reference():
    import numpy as np
    from PIL import Image
    from llamagen_b200.sample.vq_demo import center_crop
    rng = np.random.default_rng(1)
    cases = iter(CASES["center_crop"])
    for shape in [(300, 420), (1100, 900), (256, 256), (513, 2000)]:
        im = Image.fromarray(rng.integers(0, 255, (*shape, 3), dtype=np.uint8))
        for s in (256, 384):
            ref_shape, ref_s, digest = next(cases)
            assert (tuple(ref_shape), ref_s) == (shape, s)
            assert tensor_digest(torch.from_numpy(np.array(center_crop(im, s)))) == digest
