"""The decode-step kernels and the rollout actor on the GPU: `rorl_small_linear` against float64, the fused Mamba step
against the torch chain it replaces, and `PolicyActor` (one graph replay per environment step) against the eager L = 1
loop, through weight updates, `load_models()` and `load_state_dict()`."""
import numpy as np
import pytest
import torch

from helpers import rel_err
from test_resume_gpu import _engine

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")


# ---- rorl_small_linear ----------------------------------------------------------------------------------------------------
def _ref_linear(x, W, b, elu, layout, G):
    x64, W64 = x.double(), W.double()
    if layout == 0:
        y = x64 @ W64.t() + (0 if b is None else b.double())
    else:
        y = torch.einsum('mk,gkn->gmn', x64, W64) + (0 if b is None else b.double().view(G, 1, -1))
    return torch.nn.functional.elu(y) if elu else y


@pytest.mark.parametrize("K", [1, 6, 16, 256, 1024])
@pytest.mark.parametrize("layout,G", [(0, 1), (1, 1), (1, 2), (1, 3), (1, 8)])
def test_small_linear_matches_float64(K, layout, G):
    import rorl_b200.kernels as Kn
    torch.manual_seed(K * 10 + G)
    Nn = 40 if layout == 0 else 36
    for M in (1, 7, 64):
        for bias in (False, True):
            for elu in (False, True):
                x = torch.randn(M, K, device=DEV)
                W = torch.randn((Nn, K) if layout == 0 else (G, K, Nn), device=DEV) / K ** 0.5
                b = torch.randn((Nn,) if layout == 0 else (G, Nn), device=DEV) if bias else None
                y = Kn.small_linear(x, W, b, elu, layout=layout)
                e = rel_err(y, _ref_linear(x, W, b, elu, layout, G))
                assert e < 2e-6, (M, bias, elu, e)


def test_small_linear_strided_and_per_member_inputs():
    import rorl_b200.kernels as Kn
    torch.manual_seed(1)
    wide = torch.randn(13, 300, device=DEV)
    x = wide[:, 17:17 + 256]                                                 # row stride 300, unaligned base
    W = torch.randn(96, 256, device=DEV) / 16
    assert rel_err(Kn.small_linear(x, W, None), _ref_linear(x, W, None, False, 0, 1)) < 2e-6
    out = torch.zeros(13, 200, device=DEV)
    Kn.small_linear(x, W, None, out=out[:, 50:146])                          # into a column block
    assert rel_err(out[:, 50:146], _ref_linear(x, W, None, False, 0, 1)) < 2e-6 and out[:, :50].abs().max() == 0
    Wg = torch.randn(4, 64, 40, device=DEV) / 8
    bg = torch.randn(4, 1, 40, device=DEV)
    xg = torch.randn(4, 9, 64, device=DEV)                                   # one input per member
    y = Kn.small_linear(xg, Wg, bg, True, layout=1, shared=False)
    ref = torch.nn.functional.elu(torch.bmm(xg.double(), Wg.double()) + bg.double())
    assert rel_err(y, ref) < 2e-6


def test_small_linear_run_to_run_bit_identical():
    import rorl_b200.kernels as Kn
    torch.manual_seed(2)
    x = torch.randn(64, 1024, device=DEV)
    W = torch.randn(1024, 1024, device=DEV)
    Wg = torch.randn(3, 1024, 256, device=DEV)
    a, b = Kn.small_linear(x, W, None), Kn.small_linear(x, W, None)
    c, d = Kn.small_linear(x, Wg, None, layout=1), Kn.small_linear(x, Wg, None, layout=1)
    assert torch.equal(a, b) and torch.equal(c, d)


def test_decode_step_selection(monkeypatch):
    """Only [.., 1, K] inputs with at most 64 rows, passes 2 and no autograd recording take the decode kernel."""
    import rorl_b200.kernels as Kn
    calls = []
    real = Kn.small_linear
    monkeypatch.setattr(Kn, "small_linear", lambda *a, **k: calls.append(1) or real(*a, **k))
    W = torch.randn(32, 48, device=DEV, requires_grad=True)
    We = torch.randn(2, 48, 32, device=DEV, requires_grad=True)

    def taken(fn):
        calls.clear()
        fn()
        return len(calls) > 0
    x1 = torch.randn(5, 1, 48, device=DEV)
    assert not taken(lambda: Kn.linear(x1, W))                                # autograd records the call
    with torch.no_grad():
        assert taken(lambda: Kn.linear(x1, W))
        assert taken(lambda: Kn.ensemble_linear(x1, We, None, False, True))
        assert not taken(lambda: Kn.linear(x1, W, passes=4))
        assert not taken(lambda: Kn.linear(torch.randn(5, 2, 48, device=DEV), W))
        assert not taken(lambda: Kn.linear(torch.randn(65, 1, 48, device=DEV), W))
        assert not taken(lambda: Kn.linear(torch.randn(5, 48, device=DEV), W))
        y_fast = Kn.linear(x1, W)
        Kn.DECODE_STEP_KERNELS = False
        try:
            y_tc = Kn.linear(x1, W)
        finally:
            Kn.DECODE_STEP_KERNELS = True
    assert tuple(y_fast.shape) == (5, 1, 32) and rel_err(y_fast, y_tc) < 1e-5


# ---- fused Mamba step -------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("d_state", [16, 32, 64])
@pytest.mark.parametrize("d_conv", [2, 4, 8, 16])
def test_fused_mamba_step_matches_torch_chain(d_state, d_conv):
    import rorl_b200.kernels as Kn
    from rorl_b200.models.smamba.mamba import Mamba
    torch.manual_seed(d_state + d_conv)
    m = Mamba(64, d_state=d_state, d_conv=d_conv).to(DEV)
    B = 11
    h = torch.randn(1, B, m.desired_hidden_dim, device=DEV) * 0.5
    h_keep = h.clone()
    with torch.no_grad():
        for _ in range(3):                                                    # carried over three steps
            x = torch.randn(B, 1, 64, device=DEV)
            y_new, h_new = m.step(x, h)
            Kn.DECODE_STEP_KERNELS = False
            try:
                y_old, h_old = m.step(x, h)
            finally:
                Kn.DECODE_STEP_KERNELS = True
            assert torch.equal(h, h_keep)                                     # the carried hidden is only read
            # the torch chain's projections run on the two-term bf16 GEMM (about 2^-17 relative)
            assert rel_err(y_new, y_old) < 5e-5 and rel_err(h_new, h_old) < 5e-5
            h, h_keep = h_old, h_old.clone()


# ---- the actor --------------------------------------------------------------------------------------------------------------
S, A = 5, 3


def _policy(enc, algo, discrete, width=32):
    from rorl_b200.policy_value_models.make_models import make_policy_model
    kw = dict(state_dim=S, action_dim=A, embedding_size=16, embedding_hidden=[width, width],
              embedding_activations=['elu', 'elu', 'linear'], embedding_layer_type=['fc', enc, 'fc'], uni_model_hidden=[width, width],
              uni_model_activations=['elu', 'elu', 'linear'], uni_model_layer_type=['fc'] * 3, fix_rnn_length=0,
              uni_model_input_mapping_dim=16, reward_input=True, last_action_input=True, last_state_input=True, separate_encoder=True)
    if algo == 'td3':
        kw['sample_std'] = 0.1
    p = make_policy_model(kw, algo, discrete)
    p.to(DEV)
    p.need_full_hidden = False
    return p


class _Draws:
    """Graph-safe injected randomness: the policy reads a static device buffer the test refills before every step."""

    def __init__(self, n, discrete):
        self.buf = torch.zeros(n, 1, 1 if discrete else A, device=DEV)
        self.discrete = discrete

    def refill(self, gen):
        v = torch.from_numpy(gen.random(self.buf.shape) if self.discrete else gen.standard_normal(self.buf.shape)).float()
        self.buf.copy_(v)

    def install(self, policy):
        if self.discrete:
            buf = self.buf

            def sample_fn(probs):
                return (probs.cumsum(-1) < buf).sum(-1, keepdim=True).clamp(max=probs.shape[-1] - 1)
            sample_fn.graph_safe = True
            policy.sample_fn = sample_fn
        else:
            buf = self.buf

            def noise_fn(t):                                                  # an update's own draws stay random
                return buf.view(t.shape) if t.numel() == buf.numel() else torch.randn_like(t)
            noise_fn.graph_safe = True
            policy.noise_fn = noise_fn


def _flat_hidden(h):
    out = []
    for s in h._data:
        out += [t.reshape(-1) for t in (s if isinstance(s, tuple) else (s,))]
    return torch.cat(out)


def _eager_step(policy, hidden, inputs, start, n):
    """The eager L = 1 loop: environments beginning an episode continue from fresh init-state rows."""
    st, ls, la, r = (torch.from_numpy(v).float().to(DEV).view(n, 1, -1) for v in inputs)
    if hidden is None:
        hidden = policy.make_init_state(n, DEV)
    else:
        fresh = policy.make_init_state(n, DEV)
        mask = torch.from_numpy(start > 0.5).to(DEV).view(1, n, 1)
        for i, s in enumerate(hidden._data):
            if isinstance(s, tuple):
                hidden._data[i] = tuple(torch.where(mask, f, t.reshape(f.shape)) for f, t in zip(fresh._data[i], s))
            else:
                hidden._data[i] = torch.where(mask, fresh._data[i], s.reshape(fresh._data[i].shape))
    with torch.no_grad():
        out = policy.forward(st, ls, la, hidden, reward=r)
    return out, out[4]


ENCODERS = ["smamba_s16_c4_b2", "mamba_s16_c4", "gilr", "lru", "gru", "lstm", "gilr_lstm", "conv1d_4"]


@pytest.mark.parametrize("enc", ENCODERS)
@pytest.mark.parametrize("algo,discrete", [("sac", False), ("td3", False), ("sac", True)])
def test_actor_matches_eager_loop(enc, algo, discrete):
    from rorl_b200.algorithm.actor import PolicyActor
    n, steps = 6, 300
    torch.manual_seed(0)
    policy = _policy(enc, algo, discrete)
    draws = _Draws(n, discrete)
    draws.install(policy)
    graph_actor = PolicyActor(policy, n)
    plain_actor = PolicyActor(policy, n, use_cuda_graph=False)
    gen = np.random.default_rng(7)
    hidden = None
    got, ref = [], []
    for t in range(steps):
        start = (gen.random(n) < 0.03).astype(np.float32) if t else np.ones(n, np.float32)
        state, last_state, reward = gen.standard_normal((n, S)), gen.standard_normal((n, S)), gen.standard_normal((n, 1))
        last_action = (np.eye(A)[gen.integers(0, A, n)] if discrete else np.tanh(gen.standard_normal((n, A))))
        draws.refill(gen)
        a = graph_actor.step(state, last_state, last_action, reward, start)
        b = plain_actor.step(state, last_state, last_action, reward, start)
        for u, v in zip(a, b):                                                # replay == the actor's eager body, bit for bit
            assert np.array_equal(u, v), t
        assert torch.equal(_flat_hidden(graph_actor.hidden), _flat_hidden(plain_actor.hidden)), t
        out, hidden = _eager_step(policy, hidden, (state, last_state, last_action, reward), start, n)
        ref_t = [out[0], out[2], out[3]]
        got.append(a)
        ref.append([r.reshape(n, -1).cpu().numpy() for r in ref_t])
        e = rel_err(_flat_hidden(graph_actor.hidden), _flat_hidden(hidden))
        assert e < 1e-4, (t, e)
    assert graph_actor.captured and not plain_actor.captured
    for i in range(3):
        g = np.stack([x[i] for x in got]).astype(np.float64)
        r = np.stack([x[i] for x in ref]).astype(np.float64)
        if discrete and i < 2:                                                # action indices: ties / boundary draws only
            assert (g != r).mean() < 2e-3, i
        else:
            assert rel_err(torch.from_numpy(g), torch.from_numpy(r)) < 1e-4, i


def test_actor_beyond_64_envs_and_reset():
    from rorl_b200.algorithm.actor import PolicyActor
    torch.manual_seed(1)
    policy = _policy("gilr", "sac", False)
    draws = _Draws(70, False)
    draws.install(policy)
    actor = PolicyActor(policy, 70)
    gen = np.random.default_rng(3)
    hidden = None
    for t in range(5):
        start = np.ones(70, np.float32) if t == 0 else np.zeros(70, np.float32)
        inputs = (gen.standard_normal((70, S)), gen.standard_normal((70, S)), np.tanh(gen.standard_normal((70, A))),
                  gen.standard_normal((70, 1)))
        draws.refill(gen)
        a = actor.step(*inputs, start)
        out, hidden = _eager_step(policy, hidden, inputs, start, 70)
        assert rel_err(torch.from_numpy(a[1]), out[2].reshape(70, -1).cpu()) < 1e-4
    assert actor.captured
    actor.reset()
    assert float(_flat_hidden(actor.hidden).abs().max()) == 0.0


def _act_once(alg, actor, draws, gen, n):
    """One actor step against the eager policy with the engine's current weights, both from zero hidden state."""
    inputs = (gen.standard_normal((n, S)), gen.standard_normal((n, S)), np.tanh(gen.standard_normal((n, 3))),
              gen.standard_normal((n, 1)))
    start = np.ones(n, np.float32)
    draws.refill(gen)
    a = actor.step(*inputs, start)
    out, _ = _eager_step(alg.policy, None, inputs, start, n)
    assert rel_err(torch.from_numpy(a[0]), out[0].reshape(n, -1).cpu()) < 1e-4
    assert rel_err(torch.from_numpy(a[1]), out[2].reshape(n, -1).cpu()) < 1e-4


def test_actor_follows_training_and_reloads():
    """The graph reads the engine's parameters in place: after train_one_batch() and load_state_dict() the next step
    uses the new weights without recapture; after load_models() (new arenas) it recaptures."""
    alg = _engine("sac_redq_sep_smamba", True, 0)
    n = 4
    draws = _Draws(n, False)
    draws.install(alg.policy)
    actor = alg.make_actor(n)
    gen = np.random.default_rng(11)
    for _ in range(3):
        _act_once(alg, actor, draws, gen, n)
    graph0 = actor._graph
    assert graph0 is not None
    sd = alg.state_dict()
    alg.train_one_batch()
    _act_once(alg, actor, draws, gen, n)
    assert actor._graph is graph0
    alg.train_one_batch()
    alg.load_state_dict(sd)                                                   # back to the saved weights, in place
    _act_once(alg, actor, draws, gen, n)
    assert actor._graph is graph0
    w = {k: {n_: t.clone() * 0.9 for n_, t in v.items()} for k, v in alg.policy.state_dict().items()}
    alg.load_models(policy_sd=w)
    _act_once(alg, actor, draws, gen, n)                                             # eager again (warm-up) ...
    _act_once(alg, actor, draws, gen, n)                                             # ... then a fresh capture
    assert actor._graph is not None and actor._graph is not graph0
    _act_once(alg, actor, draws, gen, n)
