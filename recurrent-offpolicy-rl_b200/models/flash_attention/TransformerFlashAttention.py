"""`cgpt_*` encoder: pre-norm causal transformer with ALiBi attention over the trajectories packed in each row.

API- and state_dict-compatible with the reference's TransformerDecoder / DecoderLayer / PositionWiseFeedForward /
RMSNorm (ref: offpolicy_rnn/models/flash_attention/TransformerFlashAttention.py:29-121) and with the parameter
names of flash_attn's MHA it embeds (`mha.Wqkv.{weight,bias}`, `mha.out_proj.{weight,bias}`).

What runs where:
  * attention: csrc/attn.cu (tcgen05, bf16 operands, fp32 accumulation) -- the reference runs flash-attn 2 in bf16
    autocast (ref :80-82);
  * Wqkv / out_proj: tcgen05 GEMM, one bf16 MMA per product (passes = 4): bf16 operands, fp32 accumulation, as the
    reference computes them under the same autocast;
  * FFN (fc1 -> GELU -> fc2), norms, output_fc: fp32 as in the reference (two-term bf16 split GEMM, fused add+norm
    kernels).
Differences, deliberate: tokens are NOT unpadded / re-padded (ref :104-121): every per-token operation runs on the
padded [B*L] token axis, the attention kernel walks the sequences through a (start, length) work list, and the
padding tokens are zeroed once at the end, which is what pad_input produces.  Attention-probability dropout
(flash-attn's `dropout_p`, training mode) runs inside the attention kernels with a counter-hash keep mask: the
distribution is flash-attn's (Bernoulli(1 - p) per probability, survivors scaled by 1 / (1 - p)), the random stream
is not (flash-attn's Philox stream is not reproducible outside its kernels; parity fixtures use p0.0).
"""
from __future__ import annotations

import math

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

from ... import kernels as K
from ..linear import Linear
from ..RNNHidden import InferenceParams  # noqa: F401  (re-exported under the reference's name)

# The reference runs the MHA (Wqkv, attention, out_proj) under torch.cuda.amp.autocast(bfloat16) (ref :80-81): its linears
# are single bf16 GEMMs.  4 = one bf16 MMA per k-step on the tcgen05 kernel.
BF16_AUTOCAST_PASSES = 4


def get_alibi_slopes(nheads: int):
    """Same schedule as flash_attn.modules.mha.get_alibi_slopes (geometric in 2^(-8/n))."""
    def pow2(n):
        start = 2 ** (-(2 ** -(math.log2(n) - 3)))
        return [start * start ** i for i in range(n)]
    if math.log2(nheads).is_integer():
        return pow2(nheads)
    closest = 2 ** math.floor(math.log2(nheads))
    return pow2(closest) + get_alibi_slopes(2 * closest)[0::2][:nheads - closest]


class RMSNorm(nn.Module):
    def __init__(self, d_model: int, eps: float = 1e-5):
        super().__init__()
        self.eps = eps
        self.weight = nn.Parameter(torch.ones(d_model))

    def forward(self, x):
        return K.rms_norm_fn(x, self.weight, None, eps=self.eps)


class LayerNorm(nn.LayerNorm):
    def forward(self, x):
        return K.layer_norm_fn(x, self.weight, self.bias, eps=self.eps)


class MHA(nn.Module):
    """Self-attention block with flash_attn.modules.mha.MHA's parameter names (fused Wqkv, out_proj)."""
    _instances = 0

    def __init__(self, embed_dim: int, num_heads: int, dropout: float = 0.0, layer_idx=None):
        super().__init__()
        self.layer_idx = layer_idx
        assert embed_dim % num_heads == 0
        self.embed_dim, self.num_heads, self.head_dim = embed_dim, num_heads, embed_dim // num_heads
        if self.head_dim not in K.ATTN_HEAD_DIMS:
            raise NotImplementedError(f'the tcgen05 attention kernels take head dimensions 8, 16, ..., 128 (multiples of 8); '
                                      f'got {self.head_dim} (width {embed_dim} / {num_heads} heads)')
        self.attn_dropout = dropout
        self.Wqkv = Linear(embed_dim, 3 * embed_dim)
        self.out_proj = Linear(embed_dim, embed_dim)
        self.register_buffer('alibi_slopes', torch.tensor(get_alibi_slopes(num_heads), dtype=torch.float32), persistent=False)
        # attention-dropout call counter (device scalar: every call, also one replayed from a CUDA graph, draws a fresh mask)
        self.register_buffer('_drop_calls', torch.zeros(1, dtype=torch.int64), persistent=False)
        MHA._instances += 1
        self._salt = (0x51ED270B * ((layer_idx or 0) + 1) + 0x9E3779B1 * MHA._instances) & 0x7FFFFFFF   # stable across runs

    def forward(self, x, tiles):
        """x: [T, C] tokens; tiles: device (work list, gather map) of the sequences (kernels.attention_tiles).
        In training mode with dropout > 0 the attention probabilities are dropped inside the kernel, as flash-attn does
        for `MHA(dropout=p)` (ref: TransformerFlashAttention.py:65-70)."""
        T = x.shape[0]
        qkv = K.linear(x, self.Wqkv.weight, self.Wqkv.bias, passes=BF16_AUTOCAST_PASSES)
        p_drop = self.attn_dropout if self.training else 0.0
        seed = None
        if p_drop > 0.0:
            self._drop_calls += 1
            seed = self._drop_calls.clone()                  # the backward needs THIS call's value
        o = K.attn_varlen_alibi(qkv.view(T, 3, self.num_heads, self.head_dim), tiles[0], tiles[1], self.alibi_slopes,
                                1.0 / math.sqrt(self.head_dim), p_drop, seed, self._salt)
        return K.linear(o, self.out_proj.weight, self.out_proj.bias, passes=BF16_AUTOCAST_PASSES)

    def decode_step(self, x, cache):
        """One rollout step with the kv-cache: x [B, 1, C]; `cache` is the layer stack's InferenceParams
        (`key_value_memory_dict[layer_idx]` = [max_batch, max_seqlen, 2, H, hd] bf16, `seqlen_offset` = tokens already
        cached).  Same arithmetic as the training kernel on one query row: bf16 q / k / v, fp32 scores with the ALiBi
        bias -slope * (offset - j), fp32 softmax, bf16 probabilities.  (ref: flash_attn MHA with inference_params as
        called from TransformerFlashAttention.py:76-83 and rnn_base.py:437-452.)  Tiny tensors: plain CUDA ops, the same
        for every head dimension hd."""
        B = x.shape[0]
        H, hd = self.num_heads, self.head_dim
        qkv = K.linear(x, self.Wqkv.weight, self.Wqkv.bias, passes=BF16_AUTOCAST_PASSES).view(B, 3, H, hd)
        kv = cache.key_value_memory_dict.get(self.layer_idx)
        if kv is None:
            kv = torch.zeros((cache.max_batch_size, cache.max_seqlen, 2, H, hd), device=x.device, dtype=torch.bfloat16)
            cache.key_value_memory_dict[self.layer_idx] = kv
        off = int(cache.seqlen_offset)
        if off >= kv.shape[1]:
            raise RuntimeError(f'kv-cache of {kv.shape[1]} positions is full')
        kv[:B, off] = qkv[:, 1:].to(torch.bfloat16)
        q = qkv[:, 0].to(torch.bfloat16).float()                                   # [B, H, hd]
        keys, vals = kv[:B, :off + 1, 0].float(), kv[:B, :off + 1, 1].float()      # [B, T, H, hd]
        scores = torch.einsum('bhd,bthd->bht', q, keys) / math.sqrt(hd)
        dist = (off - torch.arange(off + 1, device=x.device, dtype=torch.float32))
        scores = scores - self.alibi_slopes.view(1, H, 1) * dist.view(1, 1, -1)
        p = torch.softmax(scores, dim=-1).to(torch.bfloat16).float()
        o = torch.einsum('bht,bthd->bhd', p, vals).reshape(B, 1, H * hd)
        return K.linear(o, self.out_proj.weight, self.out_proj.bias, passes=BF16_AUTOCAST_PASSES)


class PositionWiseFeedForward(nn.Module):
    def __init__(self, d_model, d_ff, dropout=0.1):
        super().__init__()
        self.fc1 = Linear(d_model, d_ff)
        self.fc2 = Linear(d_ff, d_model)
        self.act = nn.GELU()
        self.dropout = nn.Dropout(dropout)

    def forward(self, x):
        if K.linear_gelu_ok(x, self.fc1.weight):            # bias + exact GELU in fc1's GEMM epilogue; its backward fused with db
            h = K.linear_gelu(x, self.fc1.weight, self.fc1.bias)
        else:
            h = self.act(self.fc1(x))
        return self.fc2(self.dropout(h))


class DecoderLayer(nn.Module):
    def __init__(self, d_model, nhead, d_ff, dropout=0.1, layer_idx=None, ln=True):
        super().__init__()
        self.mha = MHA(d_model, nhead, dropout, layer_idx=layer_idx)
        self.ffn = PositionWiseFeedForward(d_model, d_ff, dropout)
        self.dropout = nn.Dropout(dropout)
        self.mha_norm = LayerNorm(d_model) if ln else RMSNorm(d_model)
        self.ffn_norm = LayerNorm(d_model) if ln else RMSNorm(d_model)

    def forward(self, x, tiles):
        x = self.dropout(self.mha(self.mha_norm(x), tiles)) + x                  # ref :76-83
        return self.dropout(self.ffn(self.ffn_norm(x))) + x                      # ref :84 (pre_norm)

    def forward_stream(self, branch, residual, tiles):
        """The same layer on a (branch, residual stream) pair: every `branch + x` of the reference (ref :76-84) is the
        residual add of the NEXT norm's fused add + norm kernel, so no separate add launches -- and, in the backward, no
        gradient accumulation launches on the stream -- exist.  Returns (this layer's FFN branch, the stream before it is
        added); the caller adds it in the following norm."""
        h, residual = _norm_stream(self.mha_norm, branch, residual)            # residual = x_in
        a = self.dropout(self.mha(h, tiles))
        h, residual = _norm_stream(self.ffn_norm, a, residual)                 # residual = x_in + dropout(mha)
        return self.dropout(self.ffn(h)), residual

    def decode_step(self, x, cache):
        x = self.dropout(self.mha.decode_step(self.mha_norm(x), cache)) + x
        return self.dropout(self.ffn(self.ffn_norm(x))) + x


def _norm_stream(norm, branch, residual, prenorm=True):
    """norm(branch + residual) on the fused add + norm kernel; with prenorm also the fp32 sum (the new residual stream)."""
    return K.layer_norm_fn(branch, norm.weight, getattr(norm, 'bias', None), residual=residual, eps=norm.eps, prenorm=prenorm,
                           is_rms_norm=isinstance(norm, RMSNorm))


def sequences_of(seqlens_host: np.ndarray, L: int):
    """Row-packed sequence lengths [B, <=L] -> (starts, lengths) on the padded token axis b * L + position, plus the
    number of real tokens per row.  Mirrors how unpad_input_for_concatenated_sequences reads the same array."""
    starts, lens, row_tokens = [], [], []
    for b in range(seqlens_host.shape[0]):
        pos = 0
        for n in seqlens_host[b]:
            n = int(n)
            if n > 0:
                starts.append(b * L + pos)
                lens.append(n)
                pos += n
        assert pos <= L, 'sequence lengths exceed the padded row length'
        row_tokens.append(pos)
    return starts, lens, row_tokens


class TransformerDecoder(nn.Module):
    def __init__(self, d_model, n_head, d_ff, n_layer, dropout=0.1, ln=True):
        super().__init__()
        self.d_model, self.n_head, self.d_ff, self.n_layer = d_model, n_head, d_ff, n_layer
        self.decoder_layers = nn.ModuleList([DecoderLayer(d_model, n_head, d_ff, dropout=dropout, layer_idx=i, ln=ln)
                                             for i in range(n_layer)])
        self.output_ln = LayerNorm(d_model) if ln else RMSNorm(d_model)
        self.output_fc = Linear(d_model, d_model)
        self._tiles_cache = {}

    def forward(self, x, inference_params=None, seqlens=None):
        """x: [B, L, C].  seqlens: [B, L] lengths of the sequences packed in each row (zeros padded), as the update
        path passes them (ref :104-112); None = every row is one full-length sequence.  A host copy attached as
        `seqlens._host` (numpy) avoids a device->host sync."""
        if not x.is_cuda:
            raise RuntimeError('the cgpt encoder runs on sm_100a kernels only; there is no CPU path')
        if inference_params is not None and seqlens is None and x.shape[-2] == 1:
            # rollout: one token per row against the kv-cache; the caller (RNNBase.meta_forward, ref rnn_base.py:437-452)
            # advances `seqlen_offset` after the whole stack has run
            h = x
            for layer in self.decoder_layers:
                h = layer.decode_step(h, inference_params)
            return self.output_fc(self.output_ln(h))
        B, L, C = x.shape
        if seqlens is None:
            host = np.zeros((B, 1), dtype=np.int64)
            host[:, 0] = L
        else:
            host = getattr(seqlens, '_host', None)
            if host is None:
                host = seqlens.detach().cpu().numpy()
        # the attention work list and the padding mask depend only on the length table: built once per table on the host,
        # kept on the device (a captured CUDA graph must not contain the pageable host-to-device copies that build them)
        host = np.ascontiguousarray(np.asarray(host))
        key = (host.tobytes(), host.shape, L, str(x.device))
        cached = self._tiles_cache.get(key)
        if cached is None:
            starts, lens, row_tokens = sequences_of(host, L)
            tiles = tuple(t.to(x.device) for t in K.attention_tiles(starts, lens))
            keep = None
            if any(n < L for n in row_tokens):                                   # pad_input: padding tokens -> 0
                keep = torch.zeros((B, L, 1), dtype=torch.float32)
                for b, n in enumerate(row_tokens):
                    keep[b, :n] = 1
                keep = keep.to(x.device)
            if len(self._tiles_cache) >= 16:
                self._tiles_cache.pop(next(iter(self._tiles_cache)))
            cached = self._tiles_cache[key] = (tiles, keep)
        tiles, keep = cached
        branch, residual = x.reshape(B * L, C), None
        for layer in self.decoder_layers:
            branch, residual = layer.forward_stream(branch, residual, tiles)
        h = self.output_fc(_norm_stream(self.output_ln, branch, residual, prenorm=False)).view(B, L, C)
        if keep is not None:
            h = h * keep
        return h
