"""CPU oracle of the `lstm` encoder layer for the parity tests: torch.nn.LSTM's own arithmetic (torch._VF.lstm, the
reference's `nn.LSTM` on CPU) on the layer's flat weights, and `rnn_base`, oracle.model.rnn_base with the `lstm` layer
type added.  Tests install it with `monkeypatch.setattr(oracle.model, "rnn_base", lstm_oracle.rnn_base)`, so that
oracle.model's policy / value forwards and oracle.update's complete update run an `lstm` encoder too."""
from typing import Dict, List

import torch
import torch.nn.functional as F

from oracle import model as OM

_BASE_RNN_BASE = OM.rnn_base


def lstm_layer(p: Dict[str, torch.Tensor], pre: str, x: torch.Tensor, hidden=None):
    """torch.nn.LSTM(batch_first=True), gate order i, f, g, o; the initial (h, c) is zero unless a tuple of two [1, B, H]
    is carried in.  Returns (out [B, L, H], (h_n, c_n)).  ref: rnn_base.py layer table 'lstm' -> nn.LSTM"""
    width = p[pre + 'weight_hh_l0'].shape[1]
    if hidden is None:
        z = torch.zeros((1, x.shape[0], width), dtype=x.dtype)
        hidden = (z, z)
    flat = [p[pre + 'weight_ih_l0'], p[pre + 'weight_hh_l0'], p[pre + 'bias_ih_l0'], p[pre + 'bias_hh_l0']]
    out, h_n, c_n = torch._VF.lstm(x, tuple(hidden), flat, True, 1, 0.0, False, False, True)
    return out, (h_n, c_n)


def rnn_base(p: Dict[str, torch.Tensor], layer_types: List[str], acts: List[str], x, side=None, desire_ndim=None):
    """oracle.model.rnn_base, plus `lstm` layers (carried state from side.h0[i], final (h, c) left in side.h_out).
    Every other layer runs through oracle.model.rnn_base itself, one layer at a time."""
    if 'lstm' not in layer_types:
        return _BASE_RNN_BASE(p, layer_types, acts, x, side, desire_ndim)
    side = side or OM.Side()
    for i, (lt, act) in enumerate(zip(layer_types, acts)):
        pre, apre = f'layer_list.{i}.', f'activation_list.{i}.'
        if lt == 'lstm':
            x, side.h_out = lstm_layer(p, pre, x, side.h0.get(i))
            if '+' in act:
                x = F.layer_norm(x, x.shape[-1:], p[apre + '0.weight'], p[apre + '0.bias'])
                act = act.split('+')[1]
            x = OM.ACT[act](x)
            continue
        sub = {}
        for k, v in p.items():
            if k.startswith(pre):
                sub['layer_list.0.' + k[len(pre):]] = v
            elif k.startswith(apre):
                sub['activation_list.0.' + k[len(apre):]] = v
        h0 = side.h0
        side.h0 = {0: h0[i]} if i in h0 else {}
        try:
            x = _BASE_RNN_BASE(sub, [lt], [act], x, side, desire_ndim)
        finally:
            side.h0 = h0
    return x
