"""smamba encoder: a stack of pre-norm Mamba blocks on the B200 kernels.

    residual add + LayerNorm/RMSNorm   -> kernels.layer_norm_fn       (rorl_addnorm_*)
    in_proj (two halves), x_proj, out_proj -> tcgen05 bf16x3 GEMM, token-major [B*L, .] (rorl_gemm_tn / _nt; no transposes)
    mask * x -> causal depthwise conv -> SiLU -> kernels.causal_conv1d_silu (rorl_conv1d_silu_*)
    dt_proj (K = dt_rank <= 16)        -> narrow-input kernels (rorl_skinny_linear / rorl_skinny_wgrad);
                                          B_t / C_t are read in place from x_dbl
    selective scan with reset + D skip + SiLU(z) gate -> kernels.selective_scan_tm (rorl_selscan_*)
    L == 1 (rollout)                   -> Mamba.step semantics: rolled conv window + one scan step with the carried state

Parameter names/shapes/initialisation and the forward contract (x [B, L, C], flat hidden
[1, B, (d_conv + d_state) * d_inner * blocks] returned unchanged, `rnn_start` resets only the SSM
state, `mask` zeroes the conv input) follow the reference
(ref: offpolicy_rnn/models/smamba/mamba.py:37-131 Mamba.__init__, :166-255 forward_sequential,
:355-412 Block, :415-526 BlockList, :528-539 PositionWiseFeedForward).  Everything stays token-major:
the reference's [B, D, L] transposes (:175-183, :251) do not exist here.
"""
import math
from functools import partial

import torch
import torch.nn as nn
import torch.nn.functional as F

from ... import kernels as K
from ..linear import Linear


class RMSNorm(nn.Module):
    def __init__(self, hidden_size, eps=1e-5):
        super().__init__()
        self.eps = eps
        self.weight = nn.Parameter(torch.ones(hidden_size))
        self.register_parameter("bias", None)

    def forward(self, x, residual=None, prenorm=False, residual_in_fp32=False):
        return K.rms_norm_fn(x, self.weight, None, residual=residual, eps=self.eps, prenorm=prenorm)


class Mamba(nn.Module):
    def __init__(self, d_model, d_state=16, d_conv=4, expand=2, dt_rank="auto", dt_min=0.001, dt_max=0.1,
                 dt_init="random", dt_scale=1.0, dt_init_floor=1e-4, conv_bias=True, bias=False, layer_idx=None):
        super().__init__()
        self.d_model, self.d_state, self.d_conv, self.expand = d_model, d_state, d_conv, expand
        self.d_inner = int(expand * d_model)
        self.dt_rank = math.ceil(d_model / 16) if dt_rank == "auto" else dt_rank
        self.layer_idx = layer_idx
        self.in_proj = Linear(d_model, self.d_inner * 2, bias=bias)
        self.conv_hidden_dim = d_model * expand * d_conv
        self.ssm_hidden_dim = d_model * expand * d_state
        self.desired_hidden_dim = self.conv_hidden_dim + self.ssm_hidden_dim
        self.use_conv = d_conv > 0
        if self.use_conv:
            self.conv1d = nn.Conv1d(self.d_inner, self.d_inner, bias=conv_bias, kernel_size=d_conv,
                                    groups=self.d_inner, padding=d_conv - 1)
        self.x_proj = Linear(self.d_inner, self.dt_rank + d_state * 2, bias=False)
        self.dt_proj = nn.Linear(self.dt_rank, self.d_inner, bias=True)
        std = self.dt_rank ** -0.5 * dt_scale
        if dt_init == "constant":
            nn.init.constant_(self.dt_proj.weight, std)
        elif dt_init == "random":
            nn.init.uniform_(self.dt_proj.weight, -std, std)
        else:
            raise NotImplementedError
        # softplus(dt_bias) log-uniform in [dt_min, dt_max]
        dt = torch.exp(torch.rand(self.d_inner) * (math.log(dt_max) - math.log(dt_min)) + math.log(dt_min)).clamp(min=dt_init_floor)
        with torch.no_grad():
            self.dt_proj.bias.copy_(dt + torch.log(-torch.expm1(-dt)))
        self.dt_proj.bias._no_reinit = True
        self.A_log = nn.Parameter(torch.log(torch.arange(1, d_state + 1, dtype=torch.float32).repeat(self.d_inner, 1)))
        self.A_log._no_weight_decay = True
        self.D = nn.Parameter(torch.ones(self.d_inner))
        self.D._no_weight_decay = True
        self.out_proj = Linear(self.d_inner, d_model, bias=bias)

    def forward(self, x, hidden=None, rnn_start=None, mask=None):
        """x: [B, L, d_model] -> [B, L, d_model]; the flat hidden is passed through untouched, as on the
        reference's GPU path (ref: mamba.py:160-164)."""
        Bsz, L, _ = x.shape
        Dn, N, R = self.d_inner, self.d_state, self.dt_rank
        if L == 1:
            return self.step(x, hidden)
        # the two halves of in_proj as two GEMMs on row slices of the weight: xs and z come out as separate
        # contiguous tensors, so no column-slice gradients ([B, L, 2D] zero-fill + copy + add) exist in the backward
        Wi, bi = self.in_proj.weight, self.in_proj.bias
        xs = K.linear(x, Wi[:Dn], None if bi is None else bi[:Dn])     # [B, L, D]
        z = K.linear(x, Wi[Dn:], None if bi is None else bi[Dn:])
        if self.use_conv:
            xs = K.causal_conv1d_silu(xs, self.conv1d.weight, self.conv1d.bias, mask)
        elif mask is not None:
            xs = xs * mask
        if K.ssm_core_ok(xs, z, self.x_proj.weight, self.dt_proj.weight, self.A_log):
            # x_proj + dt_proj + A = -exp(A_log) + scan as one autograd node (no slice / add / exp launches around the scan)
            y = K.ssm_core(xs, self.x_proj.weight, self.dt_proj.weight, self.A_log, self.D, z, self.dt_proj.bias, rnn_start)
        else:
            x_dbl = self.x_proj(xs)                                    # [B, L, R + 2N]
            delta = K.linear(x_dbl[..., :R], self.dt_proj.weight)      # bias + softplus happen in the scan
            y = K.selective_scan_tm(xs, delta, self.A_log.float(), x_dbl[..., R:R + N], x_dbl[..., R + N:], self.D.float(), z,
                                    self.dt_proj.bias.float(), rnn_start, True, a_log=True)
        out = self.out_proj(y)
        if hidden is None:
            hidden = torch.zeros((1, Bsz, self.desired_hidden_dim), device=x.device)
        return out, hidden


    def step(self, x, hidden=None):
        """Single-step (rollout / decoding) path, taken for L == 1 as in the reference (ref: mamba.py:133-159
        dispatch, :257-305 step).  hidden [1, B, D*d_conv + D*d_state] = [conv window | SSM state], conv FIRST;
        the window is rolled and the new input appended, the SSM state advances by one step of the same scan
        kernel (carried state in, final state out).  As in the reference, `rnn_start` and `mask` are NOT looked
        at on this path (SURVEY.md App. G)."""
        Bsz = x.shape[0]
        Dn, N, R, Kc = self.d_inner, self.d_state, self.dt_rank, self.d_conv
        if hidden is None:
            conv_state = x.new_zeros((Bsz, Dn, Kc)) if self.use_conv else None
            ssm_state = x.new_zeros((Bsz, Dn, N))
        else:
            conv_state = hidden[0, :, :self.conv_hidden_dim].reshape(Bsz, Dn, Kc) if self.use_conv else None
            ssm_state = hidden[0, :, self.conv_hidden_dim:].reshape(Bsz, Dn, N)
        xz = self.in_proj(x)                                           # [B, 1, 2D]
        xs, z = xz[..., :Dn], xz[..., Dn:]
        if self.use_conv:
            conv_state = torch.cat((conv_state[:, :, 1:], xs.transpose(1, 2)), dim=-1)      # roll left, append
            xs = torch.sum(conv_state * self.conv1d.weight[:, 0, :], dim=-1)
            if self.conv1d.bias is not None:
                xs = xs + self.conv1d.bias
            xs = F.silu(xs).unsqueeze(1)                               # [B, 1, D]
        x_dbl = self.x_proj(xs)
        delta = K.linear(x_dbl[..., :R], self.dt_proj.weight)
        y, last = K.selective_scan_tm(xs.contiguous(), delta, self.A_log.float(), x_dbl[..., R:R + N], x_dbl[..., R + N:], self.D.float(),
                                      z, self.dt_proj.bias.float(), None, True, True, ssm_state, a_log=True)
        out = self.out_proj(y)
        parts = ([conv_state.reshape(1, Bsz, -1)] if self.use_conv else []) + [last.reshape(1, Bsz, -1)]
        return out, torch.cat(parts, dim=-1)


def _init_weights(module, n_layer, rescale_prenorm_residual=True, n_residuals_per_layer=1):
    """GPT-2 style residual-branch rescale (ref: mamba.py:323-352)."""
    if isinstance(module, nn.Linear) and module.bias is not None and not getattr(module.bias, "_no_reinit", False):
        nn.init.zeros_(module.bias)
    if rescale_prenorm_residual:
        for name, p in module.named_parameters():
            if name in ("out_proj.weight", "fc2.weight"):
                nn.init.kaiming_uniform_(p, a=math.sqrt(5))
                with torch.no_grad():
                    p /= math.sqrt(n_residuals_per_layer * n_layer)


class Block(nn.Module):
    """Add -> Norm -> Mixer, returning (mixer output, residual stream) (ref: mamba.py:355-412)."""

    def __init__(self, dim, mixer_cls, norm_cls=nn.LayerNorm, fused_add_norm=True, residual_in_fp32=True):
        super().__init__()
        self.residual_in_fp32 = residual_in_fp32
        self.fused_add_norm = fused_add_norm
        self.mixer = mixer_cls(dim)
        self.norm = norm_cls(dim)

    def forward(self, hidden_states, residual=None, hidden=None, rnn_start=None, mask=None):
        hidden_states, residual = K.layer_norm_fn(
            hidden_states, self.norm.weight, self.norm.bias, residual=residual, eps=self.norm.eps, prenorm=True,
            residual_in_fp32=self.residual_in_fp32, is_rms_norm=isinstance(self.norm, RMSNorm))
        out, hidden = self.mixer(hidden_states, hidden, rnn_start, mask)
        return out, hidden, residual


class PositionWiseFeedForward(nn.Module):
    def __init__(self, d_model, dropout=0.0, eps=1e-5):
        super().__init__()
        self.w_1 = Linear(d_model, d_model)
        self.w_2 = Linear(d_model, d_model)
        self.activation = nn.GELU()
        self.dropout = nn.Dropout(dropout)
        self.layer_norm = nn.LayerNorm(d_model, eps=eps)

    def forward(self, x):
        y = self.dropout(self.w_2(self.dropout(self.activation(self.w_1(x)))))
        if not x.is_cuda:
            return self.layer_norm(y + x)
        # residual add + LayerNorm in one kernel (ATen's LayerNorm backward ran at 240 us per call on [32, 1002, 256])
        return K.layer_norm_fn(y, self.layer_norm.weight, self.layer_norm.bias, residual=x, eps=self.layer_norm.eps, prenorm=False)


class BlockList(nn.Module):
    def __init__(self, block_num, dim, d_conv=4, d_state=16, fused_add_norm=True, rms_norm=True,
                 residual_in_fp32=True, use_ff=False):
        super().__init__()
        self.block_num, self.fused_add_norm, self.rms_norm = block_num, fused_add_norm, rms_norm
        self.norm_epsilon = 1e-8
        self.d_conv = d_conv
        self.residual_in_fp32 = residual_in_fp32
        norm_cls = partial(RMSNorm if rms_norm else nn.LayerNorm, eps=self.norm_epsilon)
        self.layers = nn.ModuleList([
            Block(dim, partial(Mamba, layer_idx=i, d_conv=d_conv, d_state=d_state), norm_cls=norm_cls,
                  fused_add_norm=fused_add_norm, residual_in_fp32=residual_in_fp32) for i in range(block_num)])
        for i, blk in enumerate(self.layers):
            blk.layer_idx = i
        self.desired_hidden_dim = self.layers[0].mixer.desired_hidden_dim * block_num
        self.use_ff = use_ff
        if use_ff:
            self.head = PositionWiseFeedForward(d_model=dim, dropout=0.0, eps=self.norm_epsilon)
        else:
            self.head = Linear(dim, dim, bias=False)
            self.norm_f = norm_cls(dim)
        self.apply(partial(_init_weights, n_layer=block_num))

    def forward(self, x, hidden=None, rnn_start=None, mask=None, fuse_elu: bool = False):
        """fuse_elu: the caller's ELU after this layer (ref: rnn_base.py activation list) runs in the epilogue of the
        head projection's GEMM; honoured when the head is the plain Linear (not the position-wise FFN)."""
        if hidden is None:
            hidden = torch.zeros((x.shape[0], 1, self.desired_hidden_dim), device=x.device)
        hiddens = torch.chunk(hidden, self.block_num, dim=-1)
        residual, outs = None, []
        for i, blk in enumerate(self.layers):
            x, h, residual = blk(x, residual, hiddens[i], rnn_start, mask)
            outs.append(h)
        if not self.use_ff:
            x = K.layer_norm_fn(x, self.norm_f.weight, self.norm_f.bias, residual=residual, eps=self.norm_f.eps,
                                prenorm=False, residual_in_fp32=self.residual_in_fp32,
                                is_rms_norm=isinstance(self.norm_f, RMSNorm))
        else:
            x = (x + residual) if residual is not None else x
        if self.use_ff:
            y = self.head(x)
            return (F.elu(y) if fuse_elu else y), torch.cat(outs, dim=-1)
        return self.head(x, fuse_elu=fuse_elu), torch.cat(outs, dim=-1)
