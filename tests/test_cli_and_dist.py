"""CPU: CLI flag parity with the reference scripts, and the N>1 host logic (weight broadcast, sharding, seeds)
over gloo with world_size 2."""
import os
import socket
import sys

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from conftest import GOLDEN, ROOT


@pytest.mark.parametrize("script", ["sample_c2i", "sample_t2i", "sample_c2i_ddp"])
def test_cli_accepts_every_reference_flag(script):
    """Every flag the reference's sampling script defines (tests/golden/reference_surface.json, make_golden.py)."""
    import importlib
    import json
    mod = importlib.import_module(f"llamagen_b200.sample.{script}")
    ours = {a for act in mod.build_parser()._actions for a in act.option_strings}
    ref = set(json.load(open(os.path.join(GOLDEN, "reference_surface.json")))["cli_flags"][script])
    assert ref
    assert ref <= ours, f"missing flags: {sorted(ref - ours)}"


def test_cli_defaults_match_reference_text():
    from llamagen_b200.sample import sample_c2i, sample_t2i
    a = sample_c2i.build_parser().parse_args([])
    assert (a.gpt_model, a.image_size, a.cfg_scale, a.top_k, a.precision, a.cls_token_num) == ("GPT-B", 384, 4.0, 2000, "bf16", 1)
    b = sample_t2i.build_parser().parse_args([])
    assert (b.gpt_model, b.image_size, b.cfg_scale, b.top_k, b.cls_token_num, b.t5_feature_max_len) == ("GPT-XL", 512, 7.5, 1000, 120, 120)


def test_checkpoint_key_dispatch():
    from llamagen_b200.sample.common import pick_model_weight
    sd = {"w": 1}
    assert pick_model_weight(sd, True) is sd
    for k in ("model", "module", "state_dict"):
        assert pick_model_weight({k: sd}, False) is sd
    with pytest.raises(Exception, match="please check model weight"):
        pick_model_weight({"other": sd}, False)


def test_shard_and_index_helpers():
    from llamagen_b200 import distributed as lgd
    for total, world in ((256, 8), (10, 4), (3, 8)):
        covered = []
        for r in range(world):
            lo, hi = lgd.shard_range(total, r, world)
            covered += list(range(lo, hi))
        assert covered == list(range(total))
    assert lgd.rank_seed(3, 5, 8) == 29
    idx = sorted(lgd.image_index(i, r, 4, 8) for r in range(4) for i in range(2))
    assert idx == list(range(8, 16))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, q):
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    sys.path.insert(0, ROOT)
    from llamagen_b200 import distributed as lgd
    from llamagen_b200.gpt import ModelArgs, Transformer
    r, w, _ = lgd.init_from_env("gloo")
    torch.manual_seed(100 + rank)                       # ranks start with DIFFERENT weights
    m = Transformer(ModelArgs(n_layer=1, n_head=1, dim=64, vocab_size=32, block_size=4, num_classes=3))
    n = lgd.broadcast_module(m, src=0)
    digest = torch.cat([p.reshape(-1) for p in m.state_dict().values()]).double().sum().item()
    q.put((r, w, n, digest, lgd.rank_seed(0, r, w)))
    dist.barrier()
    dist.destroy_process_group()


def test_weight_broadcast_world2_gloo():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=120) for _ in range(2))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    (r0, w0, n0, d0, s0), (r1, w1, n1, d1, s1) = res
    assert (r0, r1, w0, w1) == (0, 1, 2, 2)
    assert n0 == n1 and n0 > 0
    assert d0 == d1, "weights differ after the broadcast"
    assert (s0, s1) == (0, 1)


def test_left_pad_features_matches_reference_loop():
    """cond.left_pad_features == the per-prompt loop of sample_t2i.py:92-103 (restated here), incl. empty and full rows."""
    import torch
    from llamagen_b200.cond import left_pad_features, load_t5_feature_files, pack_t5_features, prepare_condition
    torch.manual_seed(0)
    B, T, C = 6, 12, 5
    lens = torch.tensor([0, 1, 5, 11, 12, 7])
    masks = (torch.arange(T)[None, :] < lens[:, None]).float()
    embs = torch.randn(B, T, C)
    ref_masks = torch.flip(masks, dims=[-1])
    ref = torch.stack([torch.cat([e[int(m.sum().item()):], e[:int(m.sum().item())]]) for e, m in zip(embs, masks)])
    out, out_masks = left_pad_features(embs, masks)
    assert torch.equal(out, ref) and torch.equal(out_masks, ref_masks)
    c, m = prepare_condition(embs, masks)
    assert torch.equal(c, ref * ref_masks[:, :, None]) and torch.equal(m, ref_masks)
    c2, m2 = prepare_condition(embs, masks, left_padding=False)
    assert torch.equal(c2, embs * masks[:, :, None]) and torch.equal(m2, masks)
    # extract_t5_feature.py file layout: fp32 [1, valid_len, C]; truncated at max_len
    e, mk = pack_t5_features([torch.randn(1, 3, C).numpy(), torch.randn(1, 20, C).numpy()], max_len=T, dim=C)
    assert e.shape == (2, T, C) and mk.sum(1).tolist() == [3.0, 12.0] and (e[0, 3:] == 0).all()


def test_t2i_ddp_prompt_sharding(tmp_path):
    """prompt index map of sample_t2i_ddp.py:134-138: i*world + rank + total covers every row exactly once."""
    from llamagen_b200.sample.sample_t2i_ddp import prompt_indices, read_prompts
    tsv = tmp_path / "p.tsv"
    tsv.write_text("Prompt\tCategory\n" + "".join(f"prompt {i}\tc\n" for i in range(10)))
    assert read_prompts(str(tsv)) == [f"prompt {i}" for i in range(10)]
    world, n, seen = 2, 3, []
    for total in (0, 6):
        for rank in range(world):
            seen += prompt_indices(n, rank, world, total)
    assert sorted(seen) == list(range(12))


def test_serve_continuous_batching_host_logic():
    """Host logic of serve.LLM with the device step stubbed (next token = input + 1): requests JOIN MID-SEQUENCE of the running ones
    (iteration-level scheduling, llm_engine.py:511), a change of sampling parameters waits for the running set to drain, null-class
    twins mirror their conditional request, outputs come back sorted by request id."""
    import types
    import torch
    from llamagen_b200 import serve
    model = types.SimpleNamespace(model_type="c2i", tok_embeddings=types.SimpleNamespace(weight=torch.zeros(1)), vocab_size=64,
                                  cls_token_num=1, setup_caches=lambda **kw: None)

    def fake_device_step(self, st, params):
        B = self.max_num_seqs
        nxt = st["tok"] + 1
        for b in range(B):
            st["out"][b, int(st["pos"][b])] = nxt[b]
        st["tok"].copy_(nxt)

    serve.LLM._device_step, saved = fake_device_step, serve.LLM._device_step
    try:
        a, b = serve.SamplingParams(top_k=10, max_tokens=3), serve.SamplingParams(top_k=20, max_tokens=3)
        # --- mid-sequence join: r2 arrives after the first step and starts while r0, r1 are at depth 1
        llm = serve.LLM(model, cfg_scale=1.0, num_classes=1000, max_num_seqs=3, seed=0)
        llm.add_request([5], a)
        llm.add_request([6], a)
        outs = llm.step()
        assert outs == [] and llm._depth[:2] == [1, 1]
        llm.add_request([40], a)
        while llm.has_unfinished_requests():
            outs += llm.step()
        assert llm.steps_run == 4                             # static batching would need 3 + 3 steps
        got = {o.request_id: o.outputs[0].token_ids for o in outs}
        assert got == {"0": [6, 7, 8], "1": [7, 8, 9], "2": [41, 42, 43]}
        # --- LLM.generate surface: CFG twins, parameter change, more requests than slots
        llm = serve.LLM(model, cfg_scale=4.0, num_classes=1000, max_num_seqs=2, seed=0)
        labels = [5, 6, 7, 8]
        outs = llm.generate(prompt_token_ids=[[c] for c in labels] + [[1000]] * 4, sampling_params=[a, a, a, b] * 2)
        assert [o.request_id for o in outs] == [str(i) for i in range(8)]
        assert [o.outputs[0].token_ids for o in outs[:4]] == [[c + 1, c + 2, c + 3] for c in labels]
        assert [o.outputs[0].token_ids for o in outs[4:]] == [o.outputs[0].token_ids for o in outs[:4]]
        assert [o.prompt_token_ids for o in outs[4:]] == [[1000]] * 4
        # r0, r1 run together (3 steps); r2 joins a fresh set (3 steps); r3 has other sampling parameters: it waits for the drain (3 steps)
        assert llm.steps_run == 9
        assert not llm.has_unfinished_requests() and llm.get_num_unfinished_requests() == 0
        import pytest
        with pytest.raises(ValueError):
            llm.generate(prompt_token_ids=[[1], [2]])
        with pytest.raises(ValueError):
            llm.generate(prompts=["a"], prompt_token_ids=[[1]])
    finally:
        serve.LLM._device_step = saved


def test_serve_free_slots_carry_valid_class_ids():
    """Regression (round 2): a slot whose request finished sits at position 0, i.e. on the CLASS branch of the embedding lookup
    (launch_embed_rows). Its input must be a valid class id — the last sampled token (0..16383) left there indexed far past the
    1001-row class table on the device. The stub device step samples large token ids and checks every row it is given."""
    import types
    import torch
    from llamagen_b200 import serve
    model = types.SimpleNamespace(model_type="c2i", tok_embeddings=types.SimpleNamespace(weight=torch.zeros(1)), vocab_size=16384,
                                  cls_token_num=1, setup_caches=lambda **kw: None)
    seen = {"steps": 0}

    def fake_device_step(self, st, params):
        B = self.max_num_seqs
        pos, tok = st["pos"][:B], st["tok"]
        at_zero = pos == 0
        assert bool(((tok[at_zero] >= 0) & (tok[at_zero] <= self.num_classes)).all()), (tok.tolist(), pos.tolist())
        assert bool(((tok >= 0) & (tok < 16384)).all())
        nxt = torch.full_like(tok, 16000) + torch.arange(B, dtype=tok.dtype)          # "sampled" tokens far above num_classes
        for b in range(B):
            st["out"][b, int(st["pos"][b])] = nxt[b]
        st["tok"].copy_(nxt)
        seen["steps"] += 1

    serve.LLM._device_step, saved = fake_device_step, serve.LLM._device_step
    try:
        sp = serve.SamplingParams(top_k=10, max_tokens=4)
        llm = serve.LLM(model, cfg_scale=4.0, num_classes=1000, max_num_seqs=3, seed=0)
        llm.add_request([7], sp)
        llm.add_request([8], sp)
        for _ in range(2):
            llm.step()
        llm.add_request([9], sp)                       # joins mid-sequence; slots 0, 1 finish two steps before it does
        outs = []
        while llm.has_unfinished_requests():
            outs += llm.step()
        assert seen["steps"] == 6 and len(outs) == 3
    finally:
        serve.LLM._device_step = saved


def test_left_pad_and_index_map_properties():
    """Property checks (hypothesis): left_pad_features == per-row rotate for arbitrary ragged lengths; the DDP index map
    i*world + rank + total (sample_c2i_ddp.py:147) is a bijection onto range(total_samples) for any world / batch."""
    import torch
    from hypothesis import given, settings, strategies as st
    from llamagen_b200.cond import left_pad_features
    from llamagen_b200.distributed import image_index

    @settings(max_examples=40, deadline=None)
    @given(st.lists(st.integers(0, 9), min_size=1, max_size=5), st.integers(0, 2 ** 31 - 1))
    def rotate(lens, seed):
        T, C = 9, 3
        g = torch.Generator().manual_seed(seed)
        embs = torch.randn(len(lens), T, C, generator=g)
        masks = (torch.arange(T)[None, :] < torch.tensor(lens)[:, None]).float()
        out, om = left_pad_features(embs, masks)
        for i, n in enumerate(lens):
            assert torch.equal(out[i], torch.roll(embs[i], shifts=-n, dims=0))
            assert om[i].tolist() == [0.0] * (T - n) + [1.0] * n

    @settings(max_examples=40, deadline=None)
    @given(st.integers(1, 8), st.integers(1, 6), st.integers(1, 4))
    def bijection(world, n, iters):
        seen = []
        for it in range(iters):
            for rank in range(world):
                seen += [image_index(i, rank, world, it * n * world) for i in range(n)]
        assert sorted(seen) == list(range(world * n * iters))

    rotate()
    bijection()


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` (the arm the driver runs beside ours): one JSON line with the contract's keys, the same metric / unit /
    workload string as our arm, `impl`, a `cpu_baseline` describing the run and an `e2e` that repeats the value with zero copies."""
    import json
    import subprocess
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"].startswith("images/sec") and line["unit"] == "images/s"
    assert line["higher_is_better"] is True and line["steps"] == 1 and line["n_gpus"] == 1
    assert line["value"] > 0 and abs(line["e2e"]["value"] - line["value"]) < 1e-9
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and "decode steps" in cb["sample"]
    assert line["config"]["workload"] == ("LlamaGen GPT-L c2i 256px (16x16 tokens), cfg=4.0, top_k=2000, batch=64 per GPU (R=128 rows), "
                                          "AR sampling + VQ-16 decode to fp32 pixels")
