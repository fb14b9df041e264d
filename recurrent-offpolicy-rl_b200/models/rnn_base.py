"""Layer registry: a list of layer-ID strings + activation strings -> a stack of modules, with the
recurrent-state side-band threaded through every encoder call.

API-compatible with the reference's RNNBase (ref: offpolicy_rnn/models/rnn_base.py): same
constructor, same layer-ID grammar (SURVEY.md App. C; ref :100-249), same attribute names
(`layer_list`, `activation_list`, `layer_type`, `activation_type`, `rnn_num`, `rnn_layer_type`,
`rnn_hidden_state_input_size`), same per-type call signatures (ref :424-454), same state_dict keys,
same Xavier re-initialisation (ref :265-354), soft-update and l2 helpers (ref :475-532).
"""
from __future__ import annotations

import copy
import os
from typing import Dict, List, Optional, Tuple, Union

import torch
import torch.nn as nn

from .. import kernels as K
from .RNNHidden import RNNHidden
from .ensemble_linear_model import EnsembleLinear
from .linear import Linear
from .gilr.gilr import GILRLayer
from .gilr.egilr import EnsembleGILRLayer
from .lru.lru import LRULayer
from .lru.elru import EnsembleLRULayer
from .conv1d.econv1d import EConv1d
from .smamba.mamba import BlockList as MambaBlockList
from .s6.mamba import MambaResidualBlock
from .conv1d.conv1d import Conv1d
from .gilr_lstm.gilr_lstm import GILRLSTMLayer
from .gru.gru import GRULayer
from .lstm.lstm import LSTMLayer

try:
    from .flash_attention.TransformerFlashAttention import TransformerDecoder
except Exception:  # pragma: no cover - optional encoder
    TransformerDecoder = None

ACTIVATIONS = {'tanh': nn.Tanh, 'relu': nn.ReLU, 'sigmoid': nn.Sigmoid, 'leaky_relu': nn.LeakyReLU,
               'linear': nn.Identity, 'elu': nn.ELU, 'gelu': nn.GELU}
_RNN_NAMES = {'lstm', 'gru', 'cgru', 'lru', 'gilr', 'mamba', 'gilr_lstm', 'smamba', 'transformer', 'gpt', 'cgpt'}
_RNN_PREFIXES = ('conv1d', 'econv1d', 'mamba', 'smamba', 'transformer', 'gpt', 'cgpt')


def check_is_rnn(layer_id: str) -> bool:
    """ref: rnn_base.py:73-76"""
    return (layer_id in _RNN_NAMES or (layer_id.startswith('e') and layer_id[1:].split('-')[0] in _RNN_NAMES)
            or layer_id.startswith(_RNN_PREFIXES))


def parse_layer_id(layer_id: str) -> Tuple[str, Dict]:
    """Split a layer-ID string into (family, options).  Grammar: SURVEY.md App. C.2."""
    if layer_id == 'fc':
        return 'fc', {}
    if layer_id.startswith('efc'):
        return 'efc', {'ensemble': int(layer_id.split('-')[-1])}
    toks = layer_id.split('_')[1:]
    if layer_id.startswith('smamba'):
        cfg = dict(d_state=16, d_conv=4, block_num=2, rms_norm=True, use_ff=False)
        for t in toks:
            if t.startswith('s'):
                cfg['d_state'] = int(t[1:])
            elif t.startswith('c'):
                cfg['d_conv'] = int(t[1:])
            elif t.startswith('b'):
                cfg['block_num'] = int(t[1:])
            elif t.startswith('n'):
                cfg['rms_norm'] = t[1:] != 'ln'
            elif t.startswith('f'):
                cfg['use_ff'] = cfg['use_ff'] or t[1:] == 'f'
            else:
                raise ValueError(f'Pattern {t} has not been implemented!')
        return 'smamba', cfg
    if layer_id.startswith('mamba'):                           # s6 layer, ref: rnn_base.py:118-136
        cfg = dict(d_state=16, d_conv=4, use_ff=True)
        for t in toks:
            if t.startswith('s'):
                cfg['d_state'] = int(t[1:])
            elif t.startswith('c'):
                cfg['d_conv'] = int(t[1:])
            elif t.startswith('no'):
                if t[2:] == 'ff':
                    cfg['use_ff'] = False
            else:
                raise ValueError(f'Pattern {t} has not been implemented!')
        return 'mamba', cfg
    if layer_id.startswith('cgpt'):
        cfg = dict(nhead=8, nlayer=4, pdrop=0.1, maxlength=1024, ln=True)
        for t in toks:
            if t.startswith('h'):
                cfg['nhead'] = int(t[1:])
            elif t.startswith('l'):
                cfg['nlayer'] = int(t[1:])
            elif t.startswith('p'):
                cfg['pdrop'] = float(t[1:])
            elif t.startswith('ml'):
                cfg['maxlength'] = int(t[2:])
            elif t.startswith('rms'):
                cfg['ln'] = False
            else:
                raise ValueError(f'Pattern {t} has not been implemented!')
        return 'cgpt', cfg
    if layer_id in ('gru', 'lstm', 'lru', 'gilr', 'gilr_lstm'):
        return layer_id, {}
    if layer_id.startswith('conv1d'):                          # ref: rnn_base.py:227-234
        return 'conv1d', {'d_conv': int(layer_id.split('_')[-1]) if '_' in layer_id else 4}
    # ensemble encoders: one independent encoder per ensemble member, output [E, B, L, C]  (ref: rnn_base.py:110-117,235-244)
    if layer_id.startswith('e') and layer_id[1:].split('-')[0] in ('lru', 'gilr_lstm'):
        return 'elru', {'ensemble': int(layer_id.split('-')[-1])}      # `egilr_lstm-E` builds EnsembleLRULayer too (ref :110-113)
    if layer_id.startswith('egilr'):
        return 'egilr', {'ensemble': int(layer_id.split('-')[-1])}
    if layer_id.startswith('econv1d'):
        name, ens = layer_id.split('-')
        return 'econv1d', {'ensemble': int(ens), 'd_conv': int(name.split('_')[-1]) if '_' in name else 4}
    if layer_id == 'cgru':
        raise NotImplementedError("'cgru' is listed among the reference's recurrent type names (ref: rnn_base.py:70) but has no "
                                  "constructor there (its layer_dict has no such key, ref :55-69): it cannot be built in the reference either")
    raise NotImplementedError(
        f'layer type {layer_id!r} is outside the update hot path this package covers '
        f'(fc, efc-E, gru, lstm, lru, gilr, gilr_lstm, conv1d_*, smamba_*, mamba_*, cgpt_*, elru-E, egilr-E, egilr_lstm-E, econv1d_*-E)')


class RNNBase(nn.Module):
    def __init__(self, input_size: int, output_size: int, hidden_size_list: List[int], activation: List[str],
                 layer_type: List[str]):
        super().__init__()
        assert len(activation) - 1 == len(hidden_size_list), \
            "number of activation should be larger by 1 than size of hidden layers."
        assert len(activation) == len(layer_type), "number of layer type should equal to the activate"
        self.activation_dict = ACTIVATIONS
        self.check_is_rnn = check_is_rnn
        self.layer_type = copy.deepcopy(layer_type)
        self.activation_type = copy.deepcopy(activation)
        self.layer_list = nn.ModuleList()
        self.activation_list = nn.ModuleList()
        self.rnn_hidden_state_input_size: List[int] = []
        self.rnn_layer_type: List[str] = []
        self.rnn_num = 0
        width_in = input_size
        for ind, width in enumerate(hidden_size_list + [output_size]):
            lid = self.layer_type[ind]
            kind, cfg = parse_layer_id(lid)
            if kind == 'fc':
                self.layer_list.append(Linear(width_in, width))
            elif kind == 'efc':
                self.layer_list.append(EnsembleLinear(width_in, width, cfg['ensemble']))
            else:
                self.rnn_num += 1
                self.rnn_layer_type.append(lid)
                if kind == 'lru':
                    self.layer_list.append(LRULayer(width_in, width, batch_first=True))
                    self.rnn_hidden_state_input_size.append(width * 2)
                elif kind == 'gilr':
                    self.layer_list.append(GILRLayer(width_in, width, batch_first=True))
                    self.rnn_hidden_state_input_size.append(width)
                elif kind == 'gru':
                    self.layer_list.append(GRULayer(width_in, width, batch_first=True))
                    self.rnn_hidden_state_input_size.append(width)
                elif kind == 'lstm':
                    self.layer_list.append(LSTMLayer(width_in, width, batch_first=True))
                    self.rnn_hidden_state_input_size.append(width)
                elif kind == 'gilr_lstm':
                    self.layer_list.append(GILRLSTMLayer(width_in, width, batch_first=True))
                    self.rnn_hidden_state_input_size.append(width * 2)
                elif kind == 'conv1d':
                    blk = Conv1d(width_in, width, d_conv=cfg['d_conv'])
                    self.layer_list.append(blk)
                    self.rnn_hidden_state_input_size.append(blk.desired_hidden_dim)
                elif kind == 'elru':
                    self.layer_list.append(EnsembleLRULayer(width_in, width, cfg['ensemble'], batch_first=True))
                    self.rnn_hidden_state_input_size.append(width * 2 * cfg['ensemble'])
                elif kind == 'egilr':
                    self.layer_list.append(EnsembleGILRLayer(width_in, width, cfg['ensemble'], batch_first=True))
                    self.rnn_hidden_state_input_size.append(width * cfg['ensemble'])
                elif kind == 'econv1d':
                    blk = EConv1d(width_in, width, num_ensemble=cfg['ensemble'], d_conv=cfg['d_conv'])
                    self.layer_list.append(blk)
                    self.rnn_hidden_state_input_size.append(blk.desired_hidden_dim)
                elif kind == 'smamba':
                    assert width_in == width, f'mamba_simple require input_dim == output_dim, while got {width_in} and {width}'
                    blk = MambaBlockList(cfg['block_num'], width_in, d_conv=cfg['d_conv'], d_state=cfg['d_state'],
                                         rms_norm=cfg['rms_norm'], use_ff=cfg['use_ff'])
                    self.layer_list.append(blk)
                    self.rnn_hidden_state_input_size.append(blk.desired_hidden_dim)
                elif kind == 'mamba':
                    blk = MambaResidualBlock(width_in, width, d_conv=cfg['d_conv'], d_state=cfg['d_state'], use_ff=cfg['use_ff'])
                    self.layer_list.append(blk)
                    self.rnn_hidden_state_input_size.append(blk.mixer.desired_hidden_dim)
                elif kind == 'cgpt':
                    if TransformerDecoder is None:
                        raise RuntimeError('cgpt encoder unavailable in this build')
                    self.layer_list.append(TransformerDecoder(width_in, cfg['nhead'], 4 * width_in, cfg['nlayer'],
                                                              cfg['pdrop'], cfg['ln']))
                    self.rnn_hidden_state_input_size.append(cfg['maxlength'])
            act = activation[ind]
            if '+' in act:
                norm, act_name = act.split('+')
                if norm.startswith('eln'):
                    self.activation_list.append(nn.ModuleList([nn.LayerNorm([int(norm.split('-')[-1]), width]), ACTIVATIONS[act_name]()]))
                else:
                    self.activation_list.append(nn.ModuleList([nn.LayerNorm(width), ACTIVATIONS[act_name]()]))
            else:
                self.activation_list.append(ACTIVATIONS[act]())
            width_in = width
        self.input_size = input_size
        self.xavier_initialize_weights()

    # ---- initialisation (ref: rnn_base.py:265-354) -----------------------------------------------------
    @staticmethod
    def _xavier_efc(efc: EnsembleLinear):
        for i in range(efc.weight.shape[0]):
            nn.init.xavier_uniform_(efc.weight[i].transpose(0, 1))
        if getattr(efc, 'bias', None) is not None:
            nn.init.constant_(efc.bias, 0)

    @staticmethod
    def _xavier_multi(mefc):
        for i in range(mefc.weight.shape[0]):
            for j in range(mefc.weight.shape[1]):
                nn.init.xavier_uniform_(mefc.weight[i, j].transpose(0, 1))
        if getattr(mefc, 'bias', None) is not None:
            nn.init.constant_(mefc.bias, 0)

    def xavier_initialize_weights(self):
        for m in self.layer_list:
            if isinstance(m, nn.Linear):
                nn.init.xavier_uniform_(m.weight)
                if m.bias is not None:
                    nn.init.constant_(m.bias, 0)
            elif isinstance(m, EnsembleLinear):
                self._xavier_efc(m)
            elif isinstance(m, LRULayer):
                self._xavier_efc(m.in_proj)
                self._xavier_efc(m.middle_proj)
            elif isinstance(m, GILRLayer):
                nn.init.xavier_uniform_(m.out_proj.weight)
                nn.init.constant_(m.out_proj.bias, 0)
                self._xavier_efc(m.in_proj)
            elif isinstance(m, GILRLSTMLayer):
                nn.init.xavier_uniform_(m.out_proj.weight)
                nn.init.constant_(m.out_proj.bias, 0)
                self._xavier_efc(m.in_proj)
                self._xavier_efc(m.middle_proj)
            elif isinstance(m, EnsembleLRULayer):
                self._xavier_multi(m.in_proj)
                self._xavier_multi(m.middle_proj)
            elif isinstance(m, EnsembleGILRLayer):
                self._xavier_efc(m.out_proj)
                self._xavier_multi(m.in_proj)
            elif isinstance(m, (MambaBlockList, MambaResidualBlock, Conv1d, EConv1d)) or (TransformerDecoder is not None and isinstance(m, TransformerDecoder)):
                pass
            else:   # GRU, LSTM and anything else with plain weight/bias tensors
                for name, param in m.named_parameters():
                    if 'weight' in name:
                        nn.init.xavier_uniform_(param.data)
                    elif 'bias' in name:
                        nn.init.constant_(param.data, 0)

    def rnn_parameters(self, recursive=True):
        params = []
        for lid, layer in zip(self.layer_type, self.layer_list):
            if check_is_rnn(lid):
                params += list(layer.rnn_parameters()) if hasattr(layer, 'rnn_parameters') else list(layer.parameters(recursive))
        return params

    # ---- state -------------------------------------------------------------------------------------------
    def make_init_state(self, batch_size: int, device=torch.device("cpu")) -> RNNHidden:
        st = RNNHidden(self.rnn_num, self.rnn_layer_type, device)
        for size, lid in zip(self.rnn_hidden_state_input_size, self.rnn_layer_type):
            st.append(st.init_hidden_by_type(lid, batch_size, size, device))
        return st

    def make_rnd_init_state(self, batch_size: int, device=torch.device("cpu")) -> RNNHidden:
        st = RNNHidden(self.rnn_num, self.rnn_layer_type, device)
        for size, lid in zip(self.rnn_hidden_state_input_size, self.rnn_layer_type):
            st.append(st.init_random_hidden_by_type(lid, batch_size, size, device))
        return st

    # ---- forward (ref: rnn_base.py:397-472) ----------------------------------------------------------------
    def meta_forward(self, x: torch.Tensor, hidden_state: Optional[RNNHidden] = None, require_full_hidden: bool = False):
        assert x.shape[-1] == self.input_size, f"inputting size does not match!!!! input is {x.shape[-1]}, expected: {self.input_size}"
        if hidden_state is None:
            hidden_state = self.make_init_state(x.shape[0], x.device)
        assert len(hidden_state) == self.rnn_num, f"rnn num does not match, input is {len(hidden_state)}, expected: {self.rnn_num}"
        x_dim = x.dim()
        assert x_dim >= 2, f"dim of input is {x_dim}, which < 1"
        if x_dim == 2 and self.rnn_num > 0:
            x = x.unsqueeze(0)
        out_state = RNNHidden(self.rnn_num, self.rnn_layer_type, device=x.device, batch_first=False)
        full = RNNHidden(self.rnn_num, self.rnn_layer_type, device=x.device, batch_first=True) if require_full_hidden else None
        k = 0
        fused_tail = self._fused_tail(x)
        for ind, layer in enumerate(self.layer_list):
            lid = self.layer_type[ind]
            if check_is_rnn(lid):
                h_in = hidden_state[k]
                if 'gilr' in lid:
                    x, h = layer(x, h_in, hidden_state.rnn_start)
                elif 'lru' in lid:
                    x, h = layer(x, h_in, hidden_state.rnn_start, hidden_state.grad_detach)
                elif lid.startswith('smamba'):
                    # the full-hidden record takes the layer output BEFORE the activation, so no fusion when it is asked for
                    fuse = isinstance(self.activation_list[ind], nn.ELU) and x.is_cuda and not require_full_hidden
                    x, h = layer(x, h_in, hidden_state.rnn_start, hidden_state.mask, fuse_elu=fuse)
                    if fuse:                               # the ELU ran in the layer's last GEMM
                        k += 1
                        out_state.append(h)
                        continue
                elif lid.startswith('mamba'):
                    x, h = layer(x, h_in, hidden_state.rnn_start, hidden_state.mask, hidden_state.grad_detach)
                elif 'conv1d' in lid:
                    x, h = layer(x, h_in, hidden_state.mask)
                elif lid.startswith('cgpt'):
                    if x.dim() == 3 and x.shape[-2] > 1:
                        cache, seqlens = None, hidden_state.attention_concat_mask
                    else:
                        cache, seqlens = h_in, None
                    x = layer(x, inference_params=cache, seqlens=seqlens)
                    h = h_in
                    if cache is not None:
                        cache.seqlen_offset += x.shape[-2]
                else:
                    x, h = layer(x, h_in)
                k += 1
                out_state.append(h)
                if require_full_hidden:
                    full.append(x)
            else:
                if ind == fused_tail and K.ensemble_hidden_to_scalar_ok(x, layer.weight, self.layer_list[ind + 1].weight):
                    # efc-E (ELU) -> efc-E (out_dim 1): the ensemble-Q head's last two layers as one fused node
                    nxt = self.layer_list[ind + 1]
                    x = K.EnsembleHiddenToScalar.apply(x, layer.weight, layer.bias if layer.use_bias else None,
                                                       nxt.weight, nxt.bias if nxt.use_bias else None)
                    break
                if isinstance(self.activation_list[ind], nn.ELU):
                    x = layer(x, fuse_elu=True)          # bias + ELU in the GEMM epilogue
                    continue
                x = layer(x)
            act = self.activation_list[ind]
            if isinstance(act, nn.ModuleList):
                if self.activation_type[ind].startswith('eln'):
                    x = act[0](x.transpose(-2, 0)).transpose(-2, 0)
                else:
                    x = act[0](x)
                x = act[1](x)
            else:
                x = act(x)
        if x_dim == 2 and self.rnn_num > 0:
            x = x.squeeze(0)
        return x, out_state, full

    def _fused_tail(self, x) -> int:
        """Index of the layer at which the fused `efc (ELU) -> efc (out 1, linear)` tail starts, or -1.  The tail needs
        a per-member [E, ..., C] input (what an earlier efc layer leaves), so a network whose FIRST layer would be the
        tail's hidden layer is not fused."""
        n = len(self.layer_list)
        if n < 3 or not x.is_cuda:
            return -1
        a, b = self.layer_list[n - 2], self.layer_list[n - 1]
        if not (isinstance(a, EnsembleLinear) and isinstance(b, EnsembleLinear) and isinstance(self.activation_list[n - 2], nn.ELU)
                and isinstance(self.activation_list[n - 1], nn.Identity) and isinstance(self.layer_list[n - 3], EnsembleLinear)):
            return -1
        if a.desire_ndim not in (None, x.dim() + 1) or b.weight.shape[-1] != 1 or a.weight.shape[-1] not in (128, 256, 384, 512):
            return -1
        return n - 2

    # ---- soft update / persistence (ref: rnn_base.py:475-532) -------------------------------------------------
    @staticmethod
    def _copy_weight_from(dst_net: nn.Module, src_net: nn.Module, tau: float):
        with torch.no_grad():
            if tau == 0.0:
                dst_net.load_state_dict(src_net.state_dict())
                return
            if tau == 1.0:
                return
            src, dst = list(src_net.parameters(True)), list(dst_net.parameters(True))
            assert len(src) == len(dst), "parameter number show be equal!"
            for p, t in zip(src, dst):
                t.data.copy_(t.data * tau + (1 - tau) * p.data)

    def copy_weight_from(self, src_net: "RNNBase", tau: float):
        RNNBase._copy_weight_from(self, src_net, tau)

    def save(self, path):
        os.makedirs(os.path.dirname(path), exist_ok=True)
        torch.save(self.state_dict(), path)

    def load(self, path, **kwargs):
        self.load_state_dict(torch.load(path, map_location=kwargs.get('map_location')))

    def l2_norm_square(self) -> torch.Tensor:
        return sum(torch.sum(p ** 2) for p in self.parameters(True))
