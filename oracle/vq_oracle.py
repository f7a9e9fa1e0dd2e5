"""Functional oracle of the LlamaGen VQ tokenizer decode path + codebook argmin (TEST INFRASTRUCTURE ONLY).

Restates tokenizer/tokenizer_image/vq_model.py over a plain state_dict:
  VQModel.decode_code :52-55 -> get_codebook_entry :261-276 -> post_quant_conv :48 -> Decoder.forward :173-194
  ResnetBlock.forward :298-314, AttnBlock.forward :327-351, Upsample.forward :374-378,
  Normalize = GroupNorm(32, C, eps=1e-6) :359-362, nonlinearity (swish) :354-356,
  VectorQuantizer.forward index path :215-233,
  VQModel.encode :41-45 -> Encoder.forward :100-124 (Downsample :389-397) -> quant_conv -> VectorQuantizer.forward.
Pinned against reference outputs (tests/test_oracle_vs_reference.py) and tests/golden/vq_*.pt.
"""
from __future__ import annotations

import torch
import torch.nn.functional as F


def _swish(x):
    return x * torch.sigmoid(x)


class VQOracle:
    def __init__(self, state_dict, ch_mult=(1, 1, 2, 2, 4), num_res_blocks=2, l2_norm=True):
        self.sd = state_dict
        self.ch_mult = tuple(ch_mult)
        self.num_res_blocks = num_res_blocks
        self.l2_norm = l2_norm

    # ------------------------------------------------------------------ pieces
    def _conv(self, x, name, padding):
        return F.conv2d(x, self.sd[name + ".weight"], self.sd[name + ".bias"], stride=1, padding=padding)

    def _gn(self, x, name):
        return F.group_norm(x, 32, self.sd[name + ".weight"], self.sd[name + ".bias"], eps=1e-6)

    def _res(self, x, p):                                   # vq_model.py:298-314
        h = self._conv(_swish(self._gn(x, p + ".norm1")), p + ".conv1", 1)
        h = self._conv(_swish(self._gn(h, p + ".norm2")), p + ".conv2", 1)
        if (p + ".nin_shortcut.weight") in self.sd:
            x = self._conv(x, p + ".nin_shortcut", 0)
        return x + h

    def _attn(self, x, p):                                  # vq_model.py:327-351
        hn = self._gn(x, p + ".norm")
        q, k, v = (self._conv(hn, p + "." + n, 0) for n in ("q", "k", "v"))
        b, c, hh, ww = q.shape
        q = q.reshape(b, c, hh * ww).permute(0, 2, 1)
        k = k.reshape(b, c, hh * ww)
        w = torch.softmax(torch.bmm(q, k) * (int(c) ** (-0.5)), dim=2)
        v = v.reshape(b, c, hh * ww)
        o = torch.bmm(v, w.permute(0, 2, 1)).reshape(b, c, hh, ww)
        return x + self._conv(o, p + ".proj_out", 0)

    # ------------------------------------------------------------------ decode
    def codebook(self):
        e = self.sd["quantize.embedding.weight"]
        return F.normalize(e, p=2, dim=-1) if self.l2_norm else e      # vq_model.py:263-266

    def lookup(self, codes, shape):                          # vq_model.py:261-276 (channel_first=True)
        zq = self.codebook()[codes.reshape(-1).long()]
        zq = zq.reshape(shape[0], shape[2], shape[3], shape[1])
        return zq.permute(0, 3, 1, 2).contiguous()

    @torch.no_grad()
    def decode(self, z):                                     # vq_model.py:47-50,173-194
        h = self._conv(z, "post_quant_conv", 0)
        h = self._conv(h, "decoder.conv_in", 1)
        h = self._res(h, "decoder.mid.0")
        h = self._attn(h, "decoder.mid.1")
        h = self._res(h, "decoder.mid.2")
        n = len(self.ch_mult)
        for i in range(n):                                   # conv_blocks[0] is the deepest level
            for j in range(self.num_res_blocks + 1):
                h = self._res(h, f"decoder.conv_blocks.{i}.res.{j}")
                if i == 0:                                   # attention only at the deepest level (:152-153)
                    h = self._attn(h, f"decoder.conv_blocks.{i}.attn.{j}")
            if i != n - 1:
                h = F.interpolate(h, scale_factor=2.0, mode="nearest")
                h = self._conv(h, f"decoder.conv_blocks.{i}.upsample.conv", 1)
        h = _swish(self._gn(h, "decoder.norm_out"))
        return self._conv(h, "decoder.conv_out", 1)

    @torch.no_grad()
    def decode_code(self, codes, shape):
        return self.decode(self.lookup(codes, shape))

    # ------------------------------------------------------------------ encode-side index path
    @torch.no_grad()
    def argmin_indices(self, z):                             # vq_model.py:215-233
        zf = z.permute(0, 2, 3, 1).contiguous().view(-1, z.shape[1])
        e = self.sd["quantize.embedding.weight"]
        if self.l2_norm:
            zf = F.normalize(zf, p=2, dim=-1)
            e = F.normalize(e, p=2, dim=-1)
        d = torch.sum(zf ** 2, dim=1, keepdim=True) + torch.sum(e ** 2, dim=1) - 2 * (zf @ e.t())
        return torch.argmin(d, dim=1)

    # ------------------------------------------------------------------ encode (SURVEY §8 f-2)
    @torch.no_grad()
    def encode_z(self, x, ch_mult=None):                     # Encoder.forward vq_model.py:100-124 + quant_conv :42
        ch_mult = tuple(ch_mult) if ch_mult is not None else self.ch_mult
        h = self._conv(x, "encoder.conv_in", 1)
        n = len(ch_mult)
        for i in range(n):
            for j in range(self.num_res_blocks):
                h = self._res(h, f"encoder.conv_blocks.{i}.res.{j}")
                if i == n - 1:                               # attention only at the coarsest level (:84-85)
                    h = self._attn(h, f"encoder.conv_blocks.{i}.attn.{j}")
            if i != n - 1:                                   # Downsample :389-397: pad right/bottom by one, 3x3 stride 2
                p = f"encoder.conv_blocks.{i}.downsample.conv"
                h = F.conv2d(F.pad(h, (0, 1, 0, 1)), self.sd[p + ".weight"], self.sd[p + ".bias"], stride=2, padding=0)
        h = self._res(h, "encoder.mid.0")
        h = self._attn(h, "encoder.mid.1")
        h = self._res(h, "encoder.mid.2")
        h = _swish(self._gn(h, "encoder.norm_out"))
        h = self._conv(h, "encoder.conv_out", 1)
        return self._conv(h, "quant_conv", 0)

    @torch.no_grad()
    def quantize(self, z):                                   # VectorQuantizer.forward :215-255 in eval mode
        idx = self.argmin_indices(z)
        zl = z.permute(0, 2, 3, 1).contiguous()
        if self.l2_norm:
            zl = F.normalize(zl, p=2, dim=-1)
        zq = self.codebook()[idx].view(zl.shape)
        zq = zl + (zq - zl)                                  # straight-through expression, kept for its fp32 rounding (:252)
        return zq.permute(0, 3, 1, 2), idx

    @torch.no_grad()
    def encode(self, x, ch_mult=None):                       # VQModel.encode :41-45 -> (quant, indices)
        return self.quantize(self.encode_z(x, ch_mult))
