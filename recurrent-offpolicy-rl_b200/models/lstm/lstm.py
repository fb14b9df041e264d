"""`lstm` encoder layer: torch.nn.LSTM(batch_first=True) parameters and call contract (ref: offpolicy_rnn/models/
rnn_base.py, layer table entry 'lstm').  Subclassing nn.LSTM keeps the reference's state_dict keys (weight_ih_l0,
weight_hh_l0, bias_ih_l0, bias_hh_l0) so checkpoints interchange; the arithmetic does not go through cuDNN: the input
projection is one tensor-core GEMM over all steps and the L dependent steps run in the persistent cluster kernel of
csrc/lstm.cu.
"""
import torch.nn as nn

from ... import kernels as K


class LSTMLayer(nn.LSTM):
    def __init__(self, input_size, hidden_size, batch_first=True):
        assert batch_first, "the encoder stack is batch-first"
        super().__init__(input_size, hidden_size, batch_first=batch_first)

    def forward(self, x, hx=None):
        """x [B, L, I]; hx = (h0, c0), each [1, B, H] -> (out [B, L, H], (h_n, c_n) each [1, B, H]), as torch.nn.LSTM
        returns them."""
        if not x.is_cuda:
            raise RuntimeError("rorl_b200 LSTM runs on the sm_100a persistent kernel only; there is no CPU path")
        h0, c0 = (None, None) if hx is None else (hx[0][0], hx[1][0])
        gi = K.linear(x, self.weight_ih_l0, self.bias_ih_l0)
        out, h_last, c_last = K.lstm_scan(gi, self.weight_hh_l0, self.bias_hh_l0, h0, c0)
        return out, (h_last.unsqueeze(0), c_last.unsqueeze(0))
