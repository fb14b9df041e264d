"""Host-side checks of the discrete-action SAC kernels that need no GPU: the categorical-head and discrete-loss entry
points are exported and declared, the ABI version is unchanged, their argument checks return before any CUDA call, and
the policy's one-hot of the action index equals F.one_hot bit for bit."""
import ctypes

import pytest
import torch
import torch.nn.functional as F

NEW = ("rorl_categorical_fwd", "rorl_categorical_bwd", "rorl_discrete_target_expect", "rorl_discrete_actor_loss_fwd_bwd")
KW = dict(state_dim=3, action_dim=5, embedding_size=8, embedding_hidden=[16, 16], embedding_activations=['elu', 'elu', 'linear'],
          embedding_layer_type=['fc', 'gilr', 'fc'], uni_model_hidden=[16, 16], uni_model_activations=['elu', 'elu', 'linear'],
          uni_model_layer_type=['fc'] * 3, fix_rnn_length=0, uni_model_input_mapping_dim=8, reward_input=False,
          last_action_input=True, last_state_input=True, separate_encoder=True)


def test_discrete_abi_exports_and_version():
    import rorl_b200._native as N
    lib = ctypes.CDLL(N.LIB_PATH)
    for name in NEW:
        assert hasattr(lib, name) and name in N.declared_prototypes(), name
    assert N.lib().rorl_abi_version() == 6


def test_categorical_argument_checks():
    import rorl_b200._native as N
    L = N.lib()
    d = 4096                                      # never dereferenced: every call below fails its checks first
    fwd = lambda z, ld, u, p, lp, mo, sa, M, A: L.rorl_categorical_fwd(z, ld, u, p, lp, mo, sa, M, A, None)
    bwd = lambda z, ld, g, dz, M, A: L.rorl_categorical_bwd(z, ld, g, dz, M, A, None)
    for A in (0, 257, -1):
        assert fwd(d, 300, d, d, d, d, d, 4, A) == -1
        assert bwd(d, 300, d, d, 4, A) == -1
    assert fwd(d, 4, d, d, d, d, d, -1, 4) == -1 and bwd(d, 4, d, d, -1, 4) == -1
    assert fwd(d, 3, d, d, d, d, d, 4, 4) == -1 and bwd(d, 3, d, d, 4, 4) == -1        # row stride below A
    for i in range(4):                                                                   # logits, probs, logp, mode
        args = [d] * 4
        args[i] = None
        assert fwd(args[0], 4, None, args[1], args[2], args[3], None, 4, 4) == -3
    assert fwd(d, 4, d, d, d, d, None, 4, 4) == -3                                       # u given, no sample buffer
    for i in range(3):
        args = [d] * 3
        args[i] = None
        assert bwd(args[0], 4, args[1], args[2], 4, 4) == -3
    assert fwd(d, 4, None, d, d, d, None, 0, 4) == 0 and bwd(d, 4, d, d, 0, 4) == 0     # no rows: nothing to launch


def test_discrete_loss_argument_checks():
    import rorl_b200._native as N
    L = N.lib()
    d = 4096
    tgt = lambda q, sel, nsel, E, M, A, lp, la, m, g, w: L.rorl_discrete_target_expect(q, sel, nsel, E, M, A, lp, la, m, g, w, None)
    act = lambda q, lp, mk, nv, la, mode, out, dl, w, E, M, A: L.rorl_discrete_actor_loss_fwd_bwd(q, lp, mk, nv, la, mode, out, dl,
                                                                                                 w, E, M, A, None)
    for A in (0, 257):
        assert tgt(d, d, 2, 4, 10, A, d, d, d, d, d) == -1
        assert act(d, d, d, d, d, 0, d, d, d, 4, 10, A) == -1
    assert tgt(d, d, 2, 4, -1, 4, d, d, d, d, d) == -1 and act(d, d, d, d, d, 0, d, d, d, 4, -1, 4) == -1
    assert tgt(d, d, 5, 4, 10, 4, d, d, d, d, d) == -1 and tgt(d, d, 0, 4, 10, 4, d, d, d, d, d) == -1
    assert act(d, d, d, d, d, 2, d, d, d, 4, 10, 4) == -1 and act(d, d, d, d, d, 0, d, d, d, 0, 10, 4) == -1
    for i in range(7):
        args = [d] * 7
        args[i] = None
        q, sel, lp, la, m, g, w = args
        assert tgt(q, sel, 2, 4, 10, 4, lp, la, m, g, w) == -3
    for i in range(8):
        args = [d] * 8
        args[i] = None
        q, lp, mk, nv, la, out, dl, w = args
        assert act(q, lp, mk, nv, la, 1, out, dl, w, 4, 10, 4) == -3


@pytest.mark.parametrize("shape", [(7, 11, 1), (3, 1), (1, 1), (5,), (2, 3, 4, 1)])
def test_action2onehot_matches_f_one_hot(shape):
    from rorl_b200.policy_value_models.contextual_sac_discrete_policy import ContextualSACDiscretePolicy
    pol = ContextualSACDiscretePolicy(**KW)
    g = torch.Generator().manual_seed(1)
    action = torch.randint(0, KW['action_dim'], shape, generator=g).float()
    got = pol.action2onehot(action)
    ref = F.one_hot(action.squeeze(-1).long(), num_classes=KW['action_dim']).float()
    assert got.dtype == ref.dtype and got.shape == ref.shape and torch.equal(got, ref)


def test_discrete_value_embed_then_forward_matches_forward():
    """The discrete value's context encoder can run ahead of the forward (the update runs it on the side stream)."""
    from rorl_b200.policy_value_models.contextual_sac_discrete_value import ContextualSACDiscreteValue
    kw = dict(KW, embedding_layer_type=['fc', 'fc', 'fc'], uni_model_layer_type=['fc'] * 3)
    val = ContextualSACDiscreteValue(**kw)
    torch.manual_seed(0)
    B, T, S, A = 2, 6, kw['state_dim'], kw['action_dim']
    s, ls, la, r = torch.randn(B, T, S), torch.randn(B, T, S), torch.randn(B, T, A), torch.randn(B, T, 1)
    with torch.no_grad():
        ref = val.forward(s, ls, la, None, val.make_init_state(B, torch.device('cpu')), r)[0]
        h = val.make_init_state(B, torch.device('cpu'))
        got = val.forward(s, ls, la, None, h, r, embedded=val.embed(s, ls, la, h, r))[0]
    assert torch.equal(got, ref)
