"""nn.Linear whose forward runs on the tcgen05 bf16x3 GEMM (kernels.linear) with an optional fused ELU
epilogue.  Same parameters / state_dict keys as torch.nn.Linear, so it is a drop-in for every `fc` layer and
projection of the reference (ref: offpolicy_rnn/models/rnn_base.py:57,102-103)."""
import torch.nn as nn

from .. import kernels as K


class Linear(nn.Linear):
    def forward(self, x, fuse_elu: bool = False):
        return K.linear(x, self.weight, self.bias, elu=fuse_elu)
