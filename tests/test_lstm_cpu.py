"""Host-side checks of the `lstm` encoder that need no GPU: layer-ID grammar, parameters and state_dict keys of
torch.nn.LSTM, the (h, c) recurrent state, model construction with the RESeL split, nest-stacking, and the C ABI's
argument checks (they return before any CUDA call), and the CPU oracle the GPU parity tests compare against."""
import ctypes
from types import SimpleNamespace

import pytest
import torch

KW = dict(state_dim=3, action_dim=2, embedding_size=8, embedding_hidden=[16, 16], embedding_activations=['elu', 'elu', 'linear'],
          embedding_layer_type=['fc', 'lstm', 'fc'], uni_model_hidden=[16, 16], uni_model_activations=['elu', 'elu', 'linear'],
          fix_rnn_length=0, uni_model_input_mapping_dim=8, reward_input=False, last_action_input=True, last_state_input=True,
          separate_encoder=True)


def test_lstm_layer_id():
    from rorl_b200.models.rnn_base import check_is_rnn, parse_layer_id
    assert parse_layer_id('lstm') == ('lstm', {})
    assert check_is_rnn('lstm')
    with pytest.raises(NotImplementedError, match='lstm'):       # not in the reference's grammar; the message lists lstm
        parse_layer_id('elstm-3')


def test_rnnbase_lstm_matches_torch_lstm_layout():
    from rorl_b200.models.rnn_base import RNNBase
    net = RNNBase(12, 8, [16, 16], ['elu', 'elu', 'linear'], ['fc', 'lstm', 'fc'])
    ref = torch.nn.LSTM(16, 16, batch_first=True)
    sd = {k[len('layer_list.1.'):]: v for k, v in net.state_dict().items() if k.startswith('layer_list.1.')}
    assert list(sd) == list(ref.state_dict())
    for k, v in ref.state_dict().items():
        assert sd[k].shape == v.shape, k
    assert net.rnn_hidden_state_input_size == [16] and net.rnn_layer_type == ['lstm'] and net.rnn_num == 1
    # Xavier weights and zero biases, as for every plain-parameter layer
    assert float(sd['bias_ih_l0'].abs().max()) == 0.0 and float(sd['bias_hh_l0'].abs().max()) == 0.0
    bound = (6.0 / (16 + 64)) ** 0.5
    assert float(sd['weight_hh_l0'].abs().max()) <= bound
    for st in (net.make_init_state(5), net.make_rnd_init_state(5)):
        h = st[0]
        assert isinstance(h, tuple) and len(h) == 2
        assert all(t.shape == (1, 5, 16) for t in h)
    assert float(net.make_init_state(5)[0][1].abs().max()) == 0.0


def test_lstm_random_hidden_draws_h_then_c():
    from rorl_b200.models.rnn_base import RNNBase
    net = RNNBase(12, 8, [16, 16], ['elu', 'elu', 'linear'], ['fc', 'lstm', 'fc'])
    torch.manual_seed(11)
    h, c = net.make_rnd_init_state(4)[0]
    torch.manual_seed(11)
    first, second = torch.rand((1, 4, 16)) * 2 - 1, torch.rand((1, 4, 16)) * 2 - 1
    assert torch.equal(h, first) and torch.equal(c, second)


def test_lstm_layer_has_no_cpu_path():
    from rorl_b200.models.lstm.lstm import LSTMLayer
    with pytest.raises(RuntimeError, match='no CPU path'):
        LSTMLayer(4, 16)(torch.zeros(2, 3, 4))


@pytest.mark.parametrize("algo", ["sac", "td3"])
def test_models_with_lstm_encoder_and_resel_split(algo):
    from rorl_b200.algorithm.full_length_update import FullLengthRNNUpdate, prepare_param_list
    from rorl_b200.policy_value_models.make_models import make_policy_model, make_value_model
    pol = make_policy_model(dict(KW, uni_model_layer_type=['fc'] * 3), algo, False)
    val = make_value_model(dict(KW, uni_model_layer_type=['efc-8'] * 3), algo, False)
    for model in (pol, val):
        assert isinstance(model.embedding_network.layer_list[1], torch.nn.LSTM)
        groups = prepare_param_list(model, 1e-5, 0.0)
        slow = {id(p) for gr in groups if gr.get("lr") == 1e-5 for p in gr["params"]}
        assert slow == {id(p) for p in model.embedding_network.parameters()}
        lstm_params = {id(p) for p in model.embedding_network.layer_list[1].parameters()}
        assert len(lstm_params) == 4 and lstm_params <= slow
        h = model.make_init_state(3, torch.device('cpu'))
        assert len(h) == 1 and isinstance(h[0], tuple) and h[0][0].shape == (1, 3, 16)
    # several trajectories share a batch row with an LSTM encoder, as in the reference (only gru / transformer stop it)
    assert FullLengthRNNUpdate.allow_nest_stack_trajs(SimpleNamespace(values=[val], policy=pol))


def test_lstm_abi_exports_and_argument_checks():
    import rorl_b200._native as N
    lib = ctypes.CDLL(N.LIB_PATH)
    for name in ("rorl_lstm_fwd", "rorl_lstm_bwd", "rorl_lstm_save_floats_per_step"):
        assert hasattr(lib, name) and name in N.declared_prototypes()
    L = N.lib()
    assert L.rorl_lstm_save_floats_per_step(256) == 5 * 256
    assert L.rorl_abi_version() == 6
    dummy = 4096                                  # never dereferenced: every call below fails its checks first
    fwd = lambda gi, w, out, B, Ln, H: L.rorl_lstm_fwd(gi, w, None, None, None, out, None, None, None, B, Ln, H, None)
    bwd = lambda dout, w, save, dg, B, Ln, H: L.rorl_lstm_bwd(dout, None, None, w, save, None, dg, None, None, B, Ln, H, None)
    for H in (8, 24, 48, 96, 512):
        assert fwd(dummy, dummy, dummy, 2, 3, H) == -1
        assert bwd(dummy, dummy, dummy, dummy, 2, 3, H) == -1
    assert fwd(dummy, dummy, dummy, 0, 3, 64) == -1 and fwd(dummy, dummy, dummy, 2, 0, 64) == -1
    assert bwd(dummy, dummy, dummy, dummy, 0, 3, 64) == -1
    assert fwd(None, dummy, dummy, 2, 3, 64) == -3
    assert fwd(dummy, None, dummy, 2, 3, 64) == -3
    assert fwd(dummy, dummy, None, 2, 3, 64) == -3
    for i in range(4):
        args = [dummy] * 4
        args[i] = None
        assert bwd(*args, 2, 3, 64) == -3
    assert fwd(dummy, dummy + 4, dummy, 2, 3, 64) == -2      # W_hh must be 16-byte aligned (float4 loads)


def test_lstm_oracle_matches_torch_lstm():
    """The parity tests' CPU oracle (tests/lstm_oracle.py) is torch.nn.LSTM's arithmetic, with a carried (h, c), and its
    rnn_base leaves every other layer type to oracle.model.rnn_base."""
    import torch.nn.functional as F
    import lstm_oracle as LO
    from oracle import model as OM
    torch.manual_seed(0)
    lstm, fc0, fc2 = torch.nn.LSTM(16, 16, batch_first=True), torch.nn.Linear(12, 16), torch.nn.Linear(16, 8)
    p = {**{f'layer_list.0.{k}': v for k, v in fc0.state_dict().items()},
         **{f'layer_list.1.{k}': v for k, v in lstm.state_dict().items()},
         **{f'layer_list.2.{k}': v for k, v in fc2.state_dict().items()}}
    x = torch.randn(3, 9, 12)
    hc = (torch.randn(1, 3, 16), torch.randn(1, 3, 16))
    side = OM.Side(h0={1: hc})
    with torch.no_grad():
        got = LO.rnn_base(p, ['fc', 'lstm', 'fc'], ['elu', 'elu', 'linear'], x, side)
        y, (h_n, c_n) = lstm(F.elu(fc0(x)), hc)
        assert torch.allclose(got, fc2(F.elu(y)), atol=1e-6)
        assert torch.allclose(side.h_out[0], h_n, atol=1e-6) and torch.allclose(side.h_out[1], c_n, atol=1e-6)
        y0, _ = LO.lstm_layer(p, 'layer_list.1.', F.elu(fc0(x)))
        assert torch.allclose(y0, lstm(F.elu(fc0(x)))[0], atol=1e-6)
        plain = ['fc', 'fc']
        q = {k: v for k, v in p.items() if k.startswith('layer_list.0.')}
        q.update({k.replace('layer_list.2.', 'layer_list.1.'): v for k, v in p.items() if k.startswith('layer_list.2.')})
        xx = torch.randn(3, 9, 12)
        assert torch.equal(LO.rnn_base(q, plain, ['elu', 'linear'], xx), OM.rnn_base(q, plain, ['elu', 'linear'], xx))
