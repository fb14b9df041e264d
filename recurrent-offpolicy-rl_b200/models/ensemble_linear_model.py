"""Ensemble of E independent linear maps (the `efc-E` layer and the 2/3-way input projections of
GILR / LRU).  Same parameters (`weight [E, in, out]`, `bias [E, 1, out]`), same rank dispatch and
`desire_ndim` switch as the reference (ref: offpolicy_rnn/models/ensemble_linear_model.py:8-60); the
contraction itself is a batched GEMM (torch.matmul -> cuBLAS) instead of einsum.
"""
import torch
import torch.nn as nn
import torch.nn.functional as F

from .. import kernels as K


class EnsembleLinear(nn.Module):
    def __init__(self, input_dim: int, output_dim: int, num_ensemble: int, bias: bool = True, desire_ndim: int = None):
        super().__init__()
        self.use_bias = bias
        self.desire_ndim = desire_ndim
        self.num_ensemble = num_ensemble
        self.weight = nn.Parameter(torch.zeros(num_ensemble, input_dim, output_dim))
        if bias:
            self.bias = nn.Parameter(torch.zeros(num_ensemble, 1, output_dim))
        nn.init.trunc_normal_(self.weight, std=1 / (2 * input_dim ** 0.5))

    def forward(self, x: torch.Tensor, fuse_elu: bool = False) -> torch.Tensor:
        W, E = self.weight, self.num_ensemble
        nd = x.dim()
        # tensor-core path (tcgen05 bf16x3 GEMM, bias + ELU fused) for the two shapes the update uses:
        # a shared [.., in] input fanned out to E members, and a per-member [E, .., in] input
        if x.is_cuda and nd in (3, 4):
            per_member = x.shape[0] == E and (self.desire_ndim is None or self.desire_ndim == nd)
            if nd == 3 or per_member:
                y = K.ensemble_linear(x, W, self.bias if self.use_bias else None, fuse_elu, shared=not per_member)
                if y is not None:
                    return y
        if nd == 2:                                   # [i, j] -> [E, i, k]
            y = torch.matmul(x.unsqueeze(0), W)
        elif nd == 3:
            if (self.desire_ndim is None or self.desire_ndim == 3) and x.shape[0] == E:
                y = torch.bmm(x, W)                   # per-member input [E, i, j]
            else:                                     # shared input [c, i, j] -> [E, c, i, k]
                y = torch.matmul(x.unsqueeze(0), W.unsqueeze(1))
        elif nd == 4:
            if (self.desire_ndim is None or self.desire_ndim == 4) and x.shape[0] == E:
                y = torch.matmul(x, W.unsqueeze(1))   # [E, b, i, j] @ [E, 1, j, k]
            else:                                     # [c, d, i, j] -> [E, c, d, i, k]
                y = torch.matmul(x.unsqueeze(0), W[:, None, None])
        elif nd == 5:
            y = torch.matmul(x, W[:, None, None])
        else:
            raise ValueError(f'EnsembleLinear: unsupported input rank {nd}')
        if self.use_bias:
            b = self.bias
            assert y.shape[0] == b.shape[0] and y.shape[-1] == b.shape[-1]
            y = y + b.reshape((E,) + (1,) * (y.dim() - 2) + (b.shape[-1],))
        return F.elu(y) if fuse_elu else y
