"""CPU oracle for the llamagen_b200 hot path — TEST INFRASTRUCTURE ONLY.

A functional PyTorch (fp32/bf16, CPU by default) restatement of the reference algorithm for the path
named in BASELINE.json:north_star:
    generate()            autoregressive/models/generate.py:16-176
    Transformer.forward   autoregressive/models/gpt.py:137-257,332-382,404-430
    VQModel.decode_code   tokenizer/tokenizer_image/vq_model.py:47-55,128-194,261-378
    VectorQuantizer.forward (index path) tokenizer/tokenizer_image/vq_model.py:215-233
    VQModel.encode        tokenizer/tokenizer_image/vq_model.py:41-45,64-124,215-255,389-397   (SURVEY §8 f-2)
Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import this
package, and only as the checker (or the timed CPU baseline) — never as a product path.

Pinning: the oracle is pinned against outputs the reference itself produced on stored cases (tests/golden/*.pt and
reference_surface.json, generator tests/golden/make_golden.py; checked by tests/test_oracle_vs_reference.py and
tests/test_oracle_golden.py).
"""
from .gpt_oracle import GPTOracle, rope_table_2d_oracle   # noqa: F401
from .sampling_oracle import sample_oracle, top_k_top_p_oracle, cfg_mix_oracle   # noqa: F401
from .vq_oracle import VQOracle   # noqa: F401
