"""Functional oracle of the LlamaGen AR transformer + generate() loop (TEST INFRASTRUCTURE ONLY).

Restates, op for op and in the model dtype, the inference branches of
  autoregressive/models/gpt.py      RMSNorm :137-148, FeedForward :166-167, KVCache.update :177-185,
                                    Attention.forward :207-241, TransformerBlock.forward :253-257,
                                    Transformer.setup_caches :316-330, Transformer.forward :341-368,
                                    precompute_freqs_cis_2d :404-417, apply_rotary_emb :420-430,
                                    LabelEmbedder :78-83, CaptionEmbedder/MLP :110-131
  autoregressive/models/generate.py prefill :77-86, decode_one_token :89-102, decode_n_tokens :105-123,
                                    generate :126-176
over a plain state_dict (reference tensor names).  Pinned against reference outputs by
tests/test_oracle_vs_reference.py and against tests/golden/gpt_*.pt.
"""
from __future__ import annotations

from types import SimpleNamespace

import torch
import torch.nn.functional as F
from torch.nn.attention import SDPBackend, sdpa_kernel

from .sampling_oracle import cfg_mix_oracle, sample_oracle


def _round_up(n, k):
    return n if n % k == 0 else n + k - n % k


def rope_table_2d_oracle(grid: int, head_dim: int, base: float, n_cond: int) -> torch.Tensor:
    """gpt.py:404-417. [n_cond + grid^2, head_dim/2, 2]; condition rows are all-zero (cos AND sin)."""
    half = head_dim // 2
    freqs = 1.0 / (base ** (torch.arange(0, half, 2)[: half // 2].float() / half))
    ang = torch.outer(torch.arange(grid), freqs)
    grid_ang = torch.concat([ang[:, None, :].expand(-1, grid, -1), ang[None, :, :].expand(grid, -1, -1)], dim=-1)
    tab = torch.stack([torch.cos(grid_ang), torch.sin(grid_ang)], dim=-1).flatten(0, 1)
    return torch.cat([torch.zeros(n_cond, head_dim // 2, 2), tab])


def _rope(x: torch.Tensor, fr: torch.Tensor) -> torch.Tensor:
    """gpt.py:420-430: adjacent pairs (2j, 2j+1), fp32 math, cast back. x [R, T, H, hd], fr [T, hd/2, 2]."""
    xs = x.float().reshape(*x.shape[:-1], -1, 2)
    f = fr.view(1, xs.size(1), 1, xs.size(3), 2)
    out = torch.stack([xs[..., 0] * f[..., 0] - xs[..., 1] * f[..., 1],
                       xs[..., 1] * f[..., 0] + xs[..., 0] * f[..., 1]], dim=-1)
    return out.flatten(3).type_as(x)


class GPTOracle:
    def __init__(self, state_dict, cfg):
        """cfg needs: n_layer n_head dim norm_eps rope_base num_classes cls_token_num block_size model_type."""
        self.sd = state_dict
        self.cfg = cfg if not isinstance(cfg, dict) else SimpleNamespace(**cfg)
        c = self.cfg
        self.hd = c.dim // c.n_head
        self.dtype = state_dict["tok_embeddings.weight"].dtype
        self.device = state_dict["tok_embeddings.weight"].device
        self.grid = int(c.block_size ** 0.5)
        self.k = self.v = None
        self.math_sdp = False

    # ---------------------------------------------------------------- building blocks
    def _rms(self, x, w):                                   # gpt.py:143-148
        xf = x.float()
        normed = xf * torch.rsqrt(torch.mean(xf * xf, dim=-1, keepdim=True) + self.cfg.norm_eps)
        return normed.type_as(x) * w

    def setup(self, rows: int, max_seq: int):               # gpt.py:316-330
        c = self.cfg
        self.max_seq = _round_up(max_seq, 8)
        shape = (rows, c.n_head, self.max_seq, self.hd)
        self.k = [torch.zeros(shape, dtype=self.dtype, device=self.device) for _ in range(c.n_layer)]
        self.v = [torch.zeros(shape, dtype=self.dtype, device=self.device) for _ in range(c.n_layer)]
        self.mask = torch.tril(torch.ones(self.max_seq, self.max_seq, dtype=torch.bool, device=self.device)) \
            .unsqueeze(0).repeat(rows, 1, 1)
        self.freqs = rope_table_2d_oracle(self.grid, self.hd, c.rope_base, c.cls_token_num).to(self.device)

    def apply_emb_masks(self, emb_masks_rows: torch.Tensor, T: int):   # generate.py:154-163
        self.mask[:, :, :T] = self.mask[:, :, :T] * emb_masks_rows.unsqueeze(1).to(self.mask.dtype)
        eye = torch.eye(self.mask.size(1), self.mask.size(2), device=self.device)
        self.mask[:] = (self.mask * (1 - eye) + eye).to(self.mask.dtype)

    def _layer(self, l, x, fr, pos, mask):
        c, sd, p = self.cfg, self.sd, f"layers.{l}."
        R, T, D = x.shape
        H, hd = c.n_head, self.hd
        xn = self._rms(x, sd[p + "attention_norm.weight"])
        q, k, v = F.linear(xn, sd[p + "attention.wqkv.weight"]).split([D, D, D], dim=-1)     # gpt.py:214
        q = _rope(q.view(R, T, H, hd), fr).transpose(1, 2)
        k = _rope(k.view(R, T, H, hd), fr).transpose(1, 2)
        v = v.view(R, T, H, hd).transpose(1, 2)
        self.k[l][:, :, pos] = k                                                               # gpt.py:183-184
        self.v[l][:, :, pos] = v
        # gpt.py:232-236. The reference runs decode steps under sdp_kernel(math only) (generate.py:112) and the
        # prefill under the default backend selection; mirrored so the oracle is bit-identical on CPU.
        if self.math_sdp:
            with sdpa_kernel(SDPBackend.MATH):
                o = F.scaled_dot_product_attention(q, self.k[l][:R], self.v[l][:R], attn_mask=mask, dropout_p=0.0)
        else:
            o = F.scaled_dot_product_attention(q, self.k[l][:R], self.v[l][:R], attn_mask=mask, dropout_p=0.0)
        o = o.transpose(1, 2).contiguous().view(R, T, D)
        h = x + F.linear(o, sd[p + "attention.wo.weight"])                                     # gpt.py:255
        hn = self._rms(h, sd[p + "ffn_norm.weight"])
        ff = F.linear(F.silu(F.linear(hn, sd[p + "feed_forward.w1.weight"])) *
                      F.linear(hn, sd[p + "feed_forward.w3.weight"]), sd[p + "feed_forward.w2.weight"])
        return h + ff                                                                          # gpt.py:256

    def embed_cond(self, cond):
        sd = self.sd
        if self.cfg.model_type == "c2i":                    # LabelEmbedder, gpt.py:82
            return F.embedding(cond, sd["cls_embedding.embedding_table.weight"]).unsqueeze(1)
        h = F.linear(cond, sd["cls_embedding.cap_proj.fc1.weight"])     # MLP, gpt.py:127-131
        h = F.gelu(h, approximate="tanh")
        return F.linear(h, sd["cls_embedding.cap_proj.fc2.weight"])

    def forward(self, idx, cond, input_pos):
        """Inference branches of Transformer.forward (gpt.py:348-368); returns fp32 logits [R, T, V]."""
        c, sd = self.cfg, self.sd
        if cond is not None:
            x = self.embed_cond(cond)[:, : c.cls_token_num]
        else:
            x = F.embedding(idx, sd["tok_embeddings.weight"])
        R = x.shape[0]
        mask = self.mask[:R, None, input_pos]
        fr = self.freqs[input_pos]
        for l in range(c.n_layer):
            x = self._layer(l, x, fr, input_pos, mask)
        x = self._rms(x, sd["norm.weight"])
        return F.linear(x, sd["output.weight"]).float()

    # ---------------------------------------------------------------- generate.py:126-176
    @torch.no_grad()
    def generate(self, cond, max_new_tokens, emb_masks=None, cfg_scale=1.0, cfg_interval=-1, temperature=1.0,
                 top_k=0, top_p=1.0, sample_logits=True, teacher=None, generator=None):
        """Returns (tokens int32 [B,S], mixed_logits fp32 [S,B,V]).  teacher [B,S]: feed these tokens
        instead of the sampled ones (per-step teacher-forced comparison, SURVEY §8c)."""
        c = self.cfg
        B = cond.shape[0]
        use_cfg = cfg_scale > 1.0
        if c.model_type == "c2i":
            T = 1
            cond_all = torch.cat([cond, torch.ones_like(cond) * c.num_classes]) if use_cfg else cond
        else:
            T = cond.shape[1]
            null = torch.zeros_like(cond) + self.sd["cls_embedding.uncond_embedding"]
            cond_all = torch.cat([cond, null]) if use_cfg else cond
        rows = 2 * B if use_cfg else B
        self.setup(rows, T + max_new_tokens)
        if emb_masks is not None:
            self.apply_emb_masks(torch.cat([emb_masks, emb_masks]) if use_cfg else emb_masks, T)

        sk = dict(temperature=temperature, top_k=top_k, top_p=top_p, sample_logits=sample_logits, generator=generator)
        toks, mixed_all = [], []

        self.math_sdp = False
        logits = self.forward(None, cond_all, torch.arange(0, T, device=self.device))
        self.math_sdp = True
        mixed = cfg_mix_oracle(logits, cfg_scale) if use_cfg else logits                        # generate.py:79-82
        mixed_all.append(mixed[:, -1].clone())
        nxt = sample_oracle(mixed[:, -1], **sk)[0]
        toks.append(nxt)
        pos = torch.tensor([T], device=self.device, dtype=torch.int)
        cfg_flag = True
        for i in range(max_new_tokens - 1):
            if cfg_interval > -1 and i > cfg_interval:                                          # generate.py:113-114
                cfg_flag = False
            cur = nxt if teacher is None else teacher[:, i:i + 1].to(nxt.dtype)
            x = torch.cat([cur, cur]) if use_cfg else cur
            logits = self.forward(x.view(-1, 1), None, pos)
            if use_cfg:
                mixed = cfg_mix_oracle(logits, cfg_scale) if cfg_flag else logits[: logits.shape[0] // 2]
            else:
                mixed = logits
            mixed_all.append(mixed[:, -1].clone())
            nxt = sample_oracle(mixed[:, -1], **sk)[0]
            toks.append(nxt)
            pos += 1
        return torch.cat(toks, dim=1).to(torch.int32), torch.stack(mixed_all)
