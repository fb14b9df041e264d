"""s6 `mamba_*` encoder layer (the reference's secondary Mamba implementation) on the B200 kernels.

    RMSNorm (eps 1e-5)                      -> kernels.rms_norm_fn              (rorl_addnorm_*)
    in_proj / x_proj / out_proj             -> tcgen05 bf16x3 GEMM              (rorl_gemm_*)
    mask * x -> causal depthwise conv -> SiLU -> kernels.causal_conv1d_silu     (rorl_conv1d_silu_*)
    selective scan with reset, carried state h0, D skip and SiLU(res) gate, final state
                                             -> kernels.selective_scan_tm       (rorl_selscan_*)

Same recurrence as the smamba layer; what differs, and is kept (ref: offpolicy_rnn/models/s6/mamba.py):
  * Norm -> mixer -> plain residual add -> feed-forward tail (:41-67), not the smamba add+norm chain;
  * the conv takes an explicit left state of d_conv - 1 masked inputs and padding 0 (:133-144); the layer's
    hidden is `cat(ssm state [D*N], conv window [(K-1)*D])`, SSM first, taken in as [1, B, .] and returned
    batch-first as [B, 1, .] (:160-172,187-190); the REAL final state is returned (the smamba GPU path
    hands its hidden back unchanged);
  * `delta = softplus(dt_proj(.))` with the bias inside the Linear (:231): bias + softplus run inside the scan
    kernel here, which is the same arithmetic;
  * the reference's device path is a Triton sequential scan that writes the [B, L, D, N] state history
    (triton_scan.py:19-72, 2.1 GB per call at the bench shape); this path never materialises it.
`grad_detach` is None on the update path; a non-None flag is rejected rather than ignored.
Parameter names / shapes / initialisation follow the reference so state_dicts are interchangeable.
"""
import math

import torch
import torch.nn as nn
import torch.nn.functional as F

from ... import kernels as K
from ..linear import Linear


class RMSNorm(nn.Module):
    """ref: s6/mamba.py:240-251"""

    def __init__(self, d_model: int, eps: float = 1e-5):
        super().__init__()
        self.eps = eps
        self.weight = nn.Parameter(torch.ones(d_model))

    def forward(self, x):
        return K.rms_norm_fn(x, self.weight, None, residual=None, eps=self.eps, prenorm=False)


class PositionWiseFeedForward(nn.Module):
    """ref: s6/mamba.py:256-267 (LayerNorm at torch's default eps)"""

    def __init__(self, d_model, dropout=0.0):
        super().__init__()
        self.w_1 = Linear(d_model, d_model)
        self.w_2 = Linear(d_model, d_model)
        self.activation = nn.GELU()
        self.dropout = nn.Dropout(dropout)
        self.layer_norm = nn.LayerNorm(d_model)

    def forward(self, x):
        x_ = self.dropout(self.activation(self.w_1(x)))
        y = self.dropout(self.w_2(x_))
        if not x.is_cuda:
            return self.layer_norm(y + x)
        return K.layer_norm_fn(y, self.layer_norm.weight, self.layer_norm.bias, residual=x, eps=self.layer_norm.eps, prenorm=False)


class MambaBlock(nn.Module):
    def __init__(self, d_model, bias=False, dt_rank='auto', expand=2, d_state=16, d_conv=4):
        super().__init__()
        d_inner = int(expand * d_model)
        if dt_rank == 'auto':
            dt_rank = int(math.ceil(d_model / 16))
        self.d_inner, self.dt_rank, self.d_conv, self.d_state = d_inner, dt_rank, d_conv, d_state
        self.in_proj = Linear(d_model, d_inner * 2, bias=bias)
        self.use_conv1d = d_conv >= 1
        self.conv1d = nn.Conv1d(d_inner, d_inner, bias=True, kernel_size=d_conv, groups=d_inner, padding=0) \
            if self.use_conv1d else nn.Identity()
        self.x_proj = Linear(d_inner, dt_rank + d_state * 2, bias=False)
        self.dt_proj = nn.Linear(dt_rank, d_inner, bias=True)
        self._init_dt_proj_weight()
        self.ssm_hidden_dim = d_inner * d_state
        self.conv_hidden_dim = d_inner * max(d_conv - 1, 0)
        self.desired_hidden_dim = self.ssm_hidden_dim + self.conv_hidden_dim
        self.A_log = nn.Parameter(torch.log(torch.arange(1, d_state + 1, dtype=torch.float32).repeat(d_inner, 1)))
        self.A_log._no_weight_decay = True
        self.D = nn.Parameter(torch.ones(d_inner))
        self.D._no_weight_decay = True
        self.out_proj = Linear(d_inner, d_model, bias=bias)

    def _init_dt_proj_weight(self, dt_scale=1.0, dt_max=0.1, dt_min=0.001, dt_init_floor=1e-4):
        """ref: s6/mamba.py:111-131"""
        std = self.dt_rank ** -0.5 * dt_scale
        with torch.no_grad():
            nn.init.uniform_(self.dt_proj.weight, -std, std)
            dt = torch.exp(torch.rand(self.d_inner) * (math.log(dt_max) - math.log(dt_min)) + math.log(dt_min)).clamp(min=dt_init_floor)
            self.dt_proj.bias.copy_(dt + torch.log(-torch.expm1(-dt)))
        self.dt_proj.bias._no_reinit = True

    def forward(self, x, hidden=None, rnn_start=None, mask=None, grad_detach=None):
        if grad_detach is not None:
            raise NotImplementedError('grad_detach is not part of the update path (it is None there)')
        Bsz, L, _ = x.shape
        Dn, Ns, R, Kc = self.d_inner, self.d_state, self.dt_rank, self.d_conv
        Wi, bi = self.in_proj.weight, self.in_proj.bias                 # two GEMMs: see smamba/mamba.py
        xs = K.linear(x, Wi[:Dn], None if bi is None else bi[:Dn])
        res = K.linear(x, Wi[Dn:], None if bi is None else bi[Dn:])
        carried = hidden is not None and not getattr(hidden, '_rorl_zero', False)
        h_ssm = h_conv = None
        if carried:
            if self.use_conv1d:
                h_ssm, h_conv = torch.split(hidden, [self.ssm_hidden_dim, self.conv_hidden_dim], dim=-1)
                h_conv = h_conv.reshape(Bsz, Kc - 1, Dn)
            else:
                h_ssm = hidden
            h_ssm = h_ssm.reshape(Bsz, Dn, Ns)
        if self.use_conv1d:
            w = self.conv1d.weight
            if h_conv is None:
                # zero left state == the kernel's zero padding; keep the masked inputs' tail for the new hidden
                conv_in_tail = (xs if mask is None else xs * mask)[:, -(Kc - 1):, :] if Kc > 1 else xs[:, :0]
                if L < Kc - 1:
                    conv_in_tail = F.pad(conv_in_tail, (0, 0, Kc - 1 - L, 0))
                xs = K.causal_conv1d_silu(xs, w, self.conv1d.bias, mask)
            else:
                # carried conv window: run the same kernel over [window | masked x] and drop the window's rows
                xm = xs if mask is None else xs * mask
                x_in = torch.cat((h_conv, xm), dim=1)
                conv_in_tail = x_in[:, -(Kc - 1):, :] if Kc > 1 else x_in[:, :0]
                xs = K.causal_conv1d_silu(x_in, w, self.conv1d.bias, None)[:, Kc - 1:, :]
        else:
            xs = F.silu(xs if mask is None else xs * mask)
            conv_in_tail = None
        x_dbl = self.x_proj(xs)                                         # [B, L, R + 2N]
        delta = K.linear(x_dbl[..., :R], self.dt_proj.weight)           # bias + softplus happen in the scan
        A = -torch.exp(self.A_log.float())
        y, last = K.selective_scan_tm(xs, delta, A, x_dbl[..., R:R + Ns], x_dbl[..., R + Ns:], self.D.float(), res,
                                      self.dt_proj.bias.float(), rnn_start, True, True, h_ssm)
        out = self.out_proj(y)
        parts = [last.reshape(Bsz, 1, -1)]
        if self.use_conv1d:
            parts.append(conv_in_tail.detach().reshape(Bsz, 1, -1))
        return out, torch.cat(parts, dim=-1)


class MambaResidualBlock(nn.Module):
    def __init__(self, input_dim, output_dim, bias=False, dt_rank='auto', expand=2, d_state=16, d_conv=4,
                 use_ff=True, norm_type='rms'):
        super().__init__()
        assert input_dim == output_dim
        d_model = output_dim
        self.mixer = MambaBlock(input_dim, bias, dt_rank, expand, d_state, d_conv)

        def get_norm(kind):
            if kind == 'ln':
                return nn.LayerNorm(d_model)
            if kind == 'rms':
                return RMSNorm(d_model)
            if kind == 'none':
                return nn.Identity()
            raise NotImplementedError(f'{kind} has not been implemented!!')
        self.norm = get_norm(norm_type)
        self.use_ff = use_ff
        if use_ff:
            self.ff = PositionWiseFeedForward(d_model, 0.0)
        else:
            self.ff = Linear(d_model, d_model, bias=False)
            self.norm_f = get_norm(norm_type)
        self.d_conv = d_conv

    def forward(self, x, hidden=None, rnn_start=None, mask=None, grad_detach=None):
        output, hidden = self.mixer(self.norm(x), hidden, rnn_start, mask, grad_detach)
        output = output + x
        if self.use_ff:
            output = self.ff(output)
        else:
            output = self.ff(self.norm_f(output))
        return output, hidden
