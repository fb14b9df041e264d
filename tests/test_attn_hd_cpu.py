"""Host-side checks of the cgpt encoder at head dimensions other than 64 that need no GPU: the C ABI's `_hd` entry points
(declared, exported, and their argument checks, which return before any CUDA call), and model construction with the
reference's state_dict layout at the widths and head counts users configure."""
import ctypes

import pytest
import torch

HD_FNS = ("rorl_attn_prep_hd", "rorl_attn_fwd_hd", "rorl_attn_bwd_hd")
DUMMY = 4096                                  # never dereferenced: every call below fails its checks first


def _calls(L):
    prep = lambda hd, src=DUMMY, ld=96: L.rorl_attn_prep_hd(src, ld, 3, 2, 100, 128, None, DUMMY, DUMMY, None, 0, None, hd, None)
    fwd = lambda hd, q=DUMMY, ld=32: L.rorl_attn_fwd_hd(q, DUMMY, DUMMY, DUMMY, 1, DUMMY, 0.25, DUMMY, ld, None, 2, 100, 128, 0.0,
                                                        None, 0, hd, None)
    bwd = lambda hd, q=DUMMY, ld=96: L.rorl_attn_bwd_hd(q, *([DUMMY] * 9), 1, DUMMY, 0.25, DUMMY, DUMMY, DUMMY, ld, 2, 100, 128, 0.0,
                                                        None, 0, hd, None)
    return prep, fwd, bwd


def test_attn_hd_abi_exports_and_version():
    import rorl_b200._native as N
    lib = ctypes.CDLL(N.LIB_PATH)
    protos = N.declared_prototypes()
    for name in HD_FNS:
        assert hasattr(lib, name) and name in protos
        assert protos[name][1][-2] is ctypes.c_int64            # head_dim, just before the stream
        assert len(protos[name][1]) == len(protos[name[:-3]][1]) + 1
    assert N.lib().rorl_abi_version() == 6


@pytest.mark.parametrize("hd", [0, 4, 12, 136, 256])
def test_attn_hd_rejects_unsupported_head_dim(hd):
    import rorl_b200._native as N
    for fn in _calls(N.lib()):
        assert fn(hd) == -1


def test_attn_hd_null_and_misaligned_arguments():
    """The `_hd` calls check null pointers and strides as the head-dim-64 calls do."""
    import rorl_b200._native as N
    L = N.lib()
    prep, fwd, bwd = _calls(L)
    for hd in (8, 32, 128):
        assert prep(hd, src=None) == -3 and fwd(hd, q=None) == -3 and bwd(hd, q=None) == -3
        assert prep(hd, ld=98) == -2
        assert fwd(hd, ld=30) == -1 and bwd(hd, ld=94) == -1
    assert L.rorl_attn_prep(None, 96, 3, 2, 100, 128, None, DUMMY, DUMMY, None, 0, None, None) == -3
    assert L.rorl_attn_prep(DUMMY, 98, 3, 2, 100, 128, None, DUMMY, DUMMY, None, 0, None, None) == -2


def _cgpt_layout(C, nl):
    keys = []
    for i in range(nl):
        pre = f'layer_list.1.decoder_layers.{i}.'
        keys += [(pre + 'mha.Wqkv.weight', (3 * C, C)), (pre + 'mha.Wqkv.bias', (3 * C,)),
                 (pre + 'mha.out_proj.weight', (C, C)), (pre + 'mha.out_proj.bias', (C,)),
                 (pre + 'ffn.fc1.weight', (4 * C, C)), (pre + 'ffn.fc1.bias', (4 * C,)),
                 (pre + 'ffn.fc2.weight', (C, 4 * C)), (pre + 'ffn.fc2.bias', (C,)),
                 (pre + 'mha_norm.weight', (C,)), (pre + 'mha_norm.bias', (C,)),
                 (pre + 'ffn_norm.weight', (C,)), (pre + 'ffn_norm.bias', (C,))]
    return keys + [('layer_list.1.output_ln.weight', (C,)), ('layer_list.1.output_ln.bias', (C,)),
                   ('layer_list.1.output_fc.weight', (C, C)), ('layer_list.1.output_fc.bias', (C,))]


@pytest.mark.parametrize("C,lid,heads", [(256, 'cgpt', 8), (512, 'cgpt_h4', 4), (128, 'cgpt_h8_l2', 8), (64, 'cgpt_h8_l1', 8)])
def test_rnnbase_builds_cgpt_at_other_head_dims(C, lid, heads):
    """The default `cgpt` at width 256 (head dim 32), `cgpt_h4` at 512 (128) and 8 heads at widths 128 and 64 (16, 8),
    with the state_dict keys and shapes of the reference's TransformerDecoder over flash_attn's MHA."""
    from rorl_b200.models.rnn_base import RNNBase
    from rorl_b200.models.flash_attention.TransformerFlashAttention import MHA
    net = RNNBase(10, 6, [C, C], ['elu', 'elu', 'linear'], ['fc', lid, 'fc'])
    nl = net.layer_list[1].n_layer
    got = [(k, tuple(v.shape)) for k, v in net.state_dict().items() if k.startswith('layer_list.1.')]
    assert got == _cgpt_layout(C, nl)
    mha = [m for m in net.modules() if isinstance(m, MHA)]
    assert len(mha) == nl and all(m.num_heads == heads and m.head_dim == C // heads for m in mha)


@pytest.mark.parametrize("C,heads", [(96, 8), (512, 2), (24, 2), (100, 1)])
def test_cgpt_rejects_unsupported_head_dim(C, heads):
    """Head dims 12, 256, 12 and 100: not a multiple of 8 from 8 to 128."""
    from rorl_b200.models.flash_attention.TransformerFlashAttention import MHA
    with pytest.raises(NotImplementedError, match='multiples of 8'):
        MHA(C, heads)


def test_attn_varlen_rejects_unsupported_head_dim():
    import rorl_b200.kernels as K
    assert K.ATTN_HEAD_DIMS == tuple(range(8, 129, 8))
    with pytest.raises(NotImplementedError, match='multiple of 8'):
        K.AttnVarlen.forward(None, torch.zeros(4, 3, 2, 12), None, torch.zeros(8, dtype=torch.int32), None, 0.25)
