"""Host-side checks of the decode-step kernels and the rollout actor that need no GPU: the new entry points are exported
and declared, the ABI version is unchanged, their argument checks return before any CUDA call, and `make_actor` refuses
the cgpt encoder and a CPU policy."""
import ctypes
from types import SimpleNamespace

import pytest
import torch

NEW = ("rorl_small_linear", "rorl_mamba_step_conv", "rorl_mamba_step_ssm")


def _kw(enc):
    return dict(state_dim=3, action_dim=2, embedding_size=8, embedding_hidden=[16, 16],
                embedding_activations=['elu', 'elu', 'linear'], embedding_layer_type=['fc', enc, 'fc'], uni_model_hidden=[16, 16],
                uni_model_activations=['elu', 'elu', 'linear'], uni_model_layer_type=['fc'] * 3, fix_rnn_length=0,
                uni_model_input_mapping_dim=8, reward_input=False, last_action_input=True, last_state_input=True,
                separate_encoder=True)


def test_step_abi_exports_and_version():
    import rorl_b200._native as N
    lib = ctypes.CDLL(N.LIB_PATH)
    for name in NEW:
        assert hasattr(lib, name) and name in N.declared_prototypes(), name
    assert N.lib().rorl_abi_version() == 6


def test_small_linear_argument_checks():
    import rorl_b200._native as N
    L = N.lib()
    d = 4096                                      # never dereferenced: every call below fails its checks first
    f = lambda x, ldx, xg, W, b, y, ldy, M, Nn, K, G, layout, elu=0: L.rorl_small_linear(x, ldx, xg, W, b, y, ldy, M, Nn, K, G,
                                                                                          layout, elu, None)
    assert f(d, 8, 0, d, None, d, 8, 65, 8, 8, 1, 0) == -1                  # more than 64 rows
    assert f(d, 8, 0, d, None, d, 8, 0, 8, 8, 1, 0) == -1
    assert f(d, 8, 0, d, None, d, 8, 4, 0, 8, 1, 0) == -1                   # N < 1
    assert f(d, 8, 0, d, None, d, 8, 4, 8, 0, 1, 0) == -1                   # K < 1
    assert f(d, 7, 0, d, None, d, 8, 4, 8, 8, 1, 0) == -1                   # ldx < K
    assert f(d, 8, 0, d, None, d, 7, 4, 8, 8, 1, 0) == -1                   # ldy < N
    assert f(d, 8, 0, d, None, d, 8, 4, 8, 8, 0, 1) == -1                   # G < 1
    for i in (0, 1, 2):                                                      # x, W, y
        a = [d, d, d]
        a[i] = None
        assert f(a[0], 8, 0, a[1], None, a[2], 8, 4, 8, 8, 1, 0) == -3
    assert f(d, 8, 0, d, None, d, 8, 4, 8, 8, 1, 2) == -3                   # unknown layout
    assert f(d, 8, 0, d, None, d, 8, 4, 8, 8, 2, 0) == -3                   # [N, K] weights have no member axis
    assert f(d, 8, 64, d, None, d, 8, 4, 8, 8, 1, 0) == -3                  # ... and no per-member input


def test_mamba_step_argument_checks():
    import rorl_b200._native as N
    L = N.lib()
    d = 4096
    conv = lambda xz, w, wi, wo, u, B=2, D=8, Kc=4, ldxz=16, ldi=32, ldo=32: L.rorl_mamba_step_conv(
        xz, ldxz, w, None, wi, ldi, wo, ldo, u, B, D, Kc, None)
    for i in range(5):
        a = [d] * 5
        a[i] = None
        assert conv(*a) == -3
    assert conv(d, d, d, d, d, B=0) == -1 and conv(d, d, d, d, d, Kc=0) == -1
    assert conv(d, d, d, d, d, ldxz=7) == -1 and conv(d, d, d, d, d, ldi=31) == -1 and conv(d, d, d, d, d, ldo=31) == -1
    ssm = lambda ptrs, B=2, D=8, R=1, Ns=16, ldx=33, ldz=8, ldi=128, ldo=128: L.rorl_mamba_step_ssm(
        ptrs[0], ptrs[1], ldx, ptrs[2], ldz, ptrs[3], ptrs[4], ptrs[5], None, ptrs[6], ldi, ptrs[7], ldo, ptrs[8], B, D, R, Ns, None)
    for i in range(9):                                                       # u, x_dbl, z, dt_w, dt_b, A_log, h_in, h_out, y
        a = [d] * 9
        a[i] = None
        assert ssm(a) == -3
    a = [d] * 9
    assert ssm(a, B=0) == -1 and ssm(a, Ns=0) == -1 and ssm(a, R=0) == -1
    assert ssm(a, ldx=32) == -1 and ssm(a, ldz=7) == -1 and ssm(a, ldi=127) == -1 and ssm(a, ldo=127) == -1


def test_decode_step_selection_without_gpu():
    """CPU tensors never take the decode kernels, whatever their shape."""
    import rorl_b200.kernels as K
    x = torch.zeros(4, 1, 8)
    assert not K.decode_step_ok(x, 4)


@pytest.mark.parametrize("enc", ["cgpt_h2_l1", "gilr"])
def test_make_actor_refusals(enc):
    from rorl_b200.algorithm.full_length_update import FullLengthRNNUpdate
    from rorl_b200.policy_value_models.make_models import make_policy_model
    policy = make_policy_model(_kw(enc), 'sac', False)                       # stays on the CPU
    fake = SimpleNamespace(policy=policy, use_cuda_graph=True, model_generation=0)
    if enc.startswith('cgpt'):
        with pytest.raises(NotImplementedError, match="seqlen_offset"):
            FullLengthRNNUpdate.make_actor(fake, 4)
    else:
        with pytest.raises(RuntimeError, match="no CPU path"):
            FullLengthRNNUpdate.make_actor(fake, 4)
