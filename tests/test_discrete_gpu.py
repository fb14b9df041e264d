"""The discrete-action SAC update on sm_100a: the categorical head (csrc/categorical.cu) against the torch formula and
autograd, its inverse-CDF draw, the discrete target / actor reductions (csrc/losses.cu) against their torch
expressions, whole updates against the oracle's CPU update, and CUDA-graph replay and the side stream against eager,
single-stream launches."""
import numpy as np
import pytest
import torch

from helpers import assert_close

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")


def torch_head(z):
    """ContextualSACDiscretePolicy.process_model_out's torch formula (ref: contextual_sac_discrete_policy.py:106-111)."""
    p = (z - z.max(dim=-1, keepdim=True).values).exp()
    p = p / p.sum(dim=-1, keepdim=True)
    p = p + 0.01
    p = p / p.sum(dim=-1, keepdim=True)
    return p, torch.log(p)


def logits_cases(A, g):
    rows = [torch.randn(300, A, generator=g) * 3, torch.randn(40, A, generator=g) * 1e4,        # large: softmax one-hot
            torch.randn(40, A, generator=g) * 1e-6 - 50.0, torch.full((3, A), -1e30),           # tiny spread, huge negative
            torch.zeros(4, A)]                                                                  # all tied
    t = torch.randint(-2, 2, (60, A), generator=g).float()                                      # many ties
    rows.append(t)
    return torch.cat(rows)


@pytest.mark.parametrize("A", [1, 2, 3, 4, 7, 18, 33, 256])
def test_categorical_head_forward_matches_torch(A):
    import rorl_b200.kernels as K
    g = torch.Generator().manual_seed(A)
    z = logits_cases(A, g)
    wide = torch.randn(z.shape[0], A + 5, generator=g)
    wide[:, 2:2 + A] = z
    for logits in (z.to(DEV), wide.to(DEV)[:, 2:2 + A]):           # contiguous and row-strided (read in place)
        mode, sample, logp, probs = K.categorical_head(logits)
        assert sample is None and mode.shape == (z.shape[0], 1) and mode.dtype == torch.float32
        p_ref, lp_ref = torch_head(logits)
        assert float((probs - p_ref).abs().max()) <= 2e-6 * float(p_ref.abs().max())
        assert float((logp - lp_ref).abs().max()) <= 4e-6 * max(1.0, float(lp_ref.abs().max()))
        ref_mode = p_ref.argmax(dim=-1)
        top2 = p_ref.topk(min(2, A), dim=-1).values
        clear = (top2[:, 0] - top2[:, -1]) > 1e-6 * top2[:, 0] if A > 1 else torch.ones_like(top2[:, 0], dtype=torch.bool)
        got = mode[:, 0].long()
        assert torch.equal(got[clear], ref_mode[clear])
        # near-ties: the kernel's mode is the first index of its own maximum, and a maximum of the torch probabilities
        assert torch.equal(got, probs.argmax(dim=-1))
        assert bool((p_ref.gather(-1, got[:, None])[:, 0] >= top2[:, 0] * (1 - 2e-6)).all())
    # exact ties go to the first index, as torch.argmax
    zt = torch.zeros(2, A, device=DEV)
    if A >= 3:
        zt[0, 1] = zt[0, A - 1] = 5.0
        zt[1, A - 2:] = 2.0
        assert K.categorical_head(zt)[0][:, 0].tolist() == [1.0, float(A - 2)]
    assert K.categorical_head(torch.zeros(2, A, device=DEV))[0][:, 0].tolist() == [0.0, 0.0]


@pytest.mark.parametrize("A", [1, 3, 7, 33, 256])
def test_categorical_sample_is_inverse_cdf(A):
    import rorl_b200.kernels as K
    g = torch.Generator().manual_seed(10 + A)
    z = (torch.randn(5000, A, generator=g) * 2).to(DEV)
    u = torch.rand(5000, generator=g).to(DEV)
    u[:3] = torch.tensor([0.0, 1.0 - 2 ** -24, 0.5])
    _, sample, _, probs = K.categorical_head(z, u)
    p = probs.double().cpu()
    cum = p.cumsum(-1)
    thr = u.double().cpu()[:, None] * cum[:, -1:]
    ref = (cum > thr).double().argmax(-1)
    ref = torch.where((cum > thr).any(-1), ref, torch.full_like(ref, A - 1))
    got = sample[:, 0].long().cpu()
    bad = (got != ref).nonzero()[:, 0]
    # only a draw within fp32 rounding of a CDF step may land on its neighbour
    for i in bad.tolist():
        assert abs(int(got[i]) - int(ref[i])) == 1
        edge = cum[i, min(int(got[i]), int(ref[i]))]
        assert abs(float(edge - thr[i, 0])) < 1e-5, (i, float(edge), float(thr[i, 0]))
    assert bad.numel() <= 5


def test_categorical_sample_chi_square():
    import rorl_b200.kernels as K
    from scipy.stats import chisquare
    g = torch.Generator().manual_seed(3)
    A, n = 7, 1_000_000
    z = (torch.randn(1, A, generator=g) * 1.5).repeat(n, 1).to(DEV)
    u = torch.rand(n, generator=g).to(DEV)
    _, sample, _, probs = K.categorical_head(z, u)
    counts = torch.bincount(sample[:, 0].long(), minlength=A).cpu().double().numpy()
    expected = probs[0].double().cpu().numpy() * n
    stat, pval = chisquare(counts, expected * counts.sum() / expected.sum())
    assert pval > 1e-3, (stat, pval, counts, expected)


@pytest.mark.parametrize("A", [1, 2, 4, 7, 18, 33, 256])
def test_categorical_head_backward_matches_autograd(A):
    import rorl_b200.kernels as K
    g = torch.Generator().manual_seed(100 + A)
    z = torch.cat([torch.randn(200, A, generator=g) * 2, torch.randn(20, A, generator=g) * 30])
    wide = torch.randn(z.shape[0], A + 3, generator=g)
    wide[:, 1:1 + A] = z
    d_logp = torch.randn(z.shape[0], A, generator=g)
    d_probs = torch.randn(z.shape[0], A, generator=g)
    z64 = z.double().requires_grad_()
    p64, lp64 = torch_head(z64)
    ref = torch.autograd.grad(lp64, z64, d_logp.double(), retain_graph=True)[0]
    ref_both = torch.autograd.grad((lp64 * d_logp.double()).sum() + (p64 * d_probs.double()).sum(), z64)[0]
    zc = wide.to(DEV)[:, 1:1 + A].requires_grad_()
    _, _, logp, probs = K.categorical_head(zc)
    got = torch.autograd.grad(logp, zc, d_logp.to(DEV), retain_graph=True)[0]
    assert_close(got.cpu().double(), ref, 1e-5, "d logits")
    got_both = torch.autograd.grad((logp * d_logp.to(DEV)).sum() + (probs * d_probs.to(DEV)).sum(), zc)[0]
    assert_close(got_both.cpu().double(), ref_both, 1e-5, "d logits through logp and probs")


def _loss_inputs(E, A, B, L, g):
    q = torch.randn(E, B, L, A, generator=g) * 3
    z = torch.randn(B, L, A, generator=g) * 2
    _, logp = torch_head(z)
    mask = torch.ones(B, L, 1)
    for b in range(B):
        mask[b, int(torch.randint(1, L + 1, (1,), generator=g)):] = 0       # ragged
    mask[B - 1] = 0                                                           # one all-masked row
    return q, logp, mask


@pytest.mark.parametrize("A,sel", [(4, [3, 5]), (18, [6]), (33, list(range(8))), (256, [0, 7, 2])])
def test_discrete_target_expect_matches_torch(A, sel):
    import rorl_b200._native as N
    import rorl_b200.kernels as K
    g = torch.Generator().manual_seed(A)
    E, B, L = 8, 6, 37
    q, logp, _ = _loss_inputs(E, A, B, L, g)
    log_alpha = torch.tensor([-1.2])
    ref = ((q[sel].double().min(dim=0).values - log_alpha.double().exp() * logp.double()) * logp.double().exp()).sum(-1)
    guard = torch.tensor([1e6, -1e6, 0.0, 1.0], dtype=torch.float64, device=DEV)
    work = torch.zeros(int(N.lib().rorl_loss_work_floats(0)), device=DEV)
    sel_d = torch.tensor(sel, dtype=torch.int32, device=DEV)
    m = K.discrete_target_expect(q.to(DEV), sel_d, logp.to(DEV), log_alpha.to(DEV), guard, work)
    assert_close(m.cpu().double().view(B, L), ref, 1e-5, "m")
    assert guard[2].item() == 1.0
    assert guard[0].item() == float(m.min()) and guard[1].item() == float(m.max())
    m2 = K.discrete_target_expect(q.to(DEV), sel_d, logp.to(DEV), log_alpha.to(DEV), guard, work)
    assert torch.equal(m, m2) and guard[0].item() == float(m.min())      # initialised once; deterministic


@pytest.mark.parametrize("A", [4, 18, 33, 256])
@pytest.mark.parametrize("mode", [0, 1])
def test_discrete_actor_loss_matches_torch(A, mode):
    import rorl_b200._native as N
    import rorl_b200.kernels as K
    g = torch.Generator().manual_seed(7 * A + mode)
    E, B, L = 8, 5, 41
    q, logp, mask = _loss_inputs(E, A, B, L, g)
    log_alpha = torch.tensor([-0.7])
    lp = logp.double().requires_grad_()
    agg = q.double().mean(0) if mode == 1 else q.double().min(0).values
    alpha = log_alpha.double().exp()
    n_valid = mask.sum()
    loss = (((alpha * lp - agg) * lp.exp()).sum(-1, keepdim=True) * mask.double()).sum() / n_valid.double()
    ent = (((lp * lp.exp()).sum(-1, keepdim=True)) * mask.double()).sum() / n_valid.double()
    dref = torch.autograd.grad(loss, lp)[0]
    out = torch.zeros(2, device=DEV)
    work = torch.zeros(int(N.lib().rorl_loss_work_floats(0)), device=DEV)
    dlogp = K.discrete_actor_loss(q.to(DEV), logp.to(DEV), mask.to(DEV), n_valid.reshape(1).to(DEV), log_alpha.to(DEV), mode,
                                  out, work)
    assert abs(float(out[0]) - float(loss)) <= 1e-5 * max(1.0, abs(float(loss)))
    assert abs(float(out[1]) - float(ent)) <= 1e-5 * max(1.0, abs(float(ent)))
    assert_close(dlogp.cpu().double(), dref, 1e-5, "dlogp")
    assert float(dlogp[B - 1].abs().max()) == 0.0                               # the all-masked row gets no gradient
    out2 = torch.zeros(2, device=DEV)
    dlogp2 = K.discrete_actor_loss(q.to(DEV), logp.to(DEV), mask.to(DEV), n_valid.reshape(1).to(DEV), log_alpha.to(DEV), mode,
                                   out2, work)
    assert torch.equal(out, out2) and torch.equal(dlogp, dlogp2)


# ------------------------------------------------------------------------------------------------------------------
# whole updates
# ------------------------------------------------------------------------------------------------------------------
CLASSES = {"redq": "sac_rnn_full_horizon_redQ_sep_optim", "ensembleq": "sac_rnn_full_horizon_ensemble_q_sep_optim"}


def _kw(enc, S, A, H, value, emb=32, last_action=True):
    return dict(state_dim=S, action_dim=A, embedding_size=emb, embedding_hidden=[H, H], embedding_activations=['elu', 'elu', 'linear'],
                embedding_layer_type=['fc', enc, 'fc'], uni_model_hidden=[H, H], uni_model_activations=['elu', 'elu', 'linear'],
                uni_model_layer_type=(['efc-8'] * 3 if value else ['fc'] * 3), fix_rnn_length=0, uni_model_input_mapping_dim=emb,
                reward_input=False, last_action_input=last_action, last_state_input=True, separate_encoder=True)


def _hp(lens, **kw):
    return dict(dict(gamma=0.99, sac_tau=0.995, policy_update_per=1, redq_m=2, policy_lr=3e-4, value_lr=1e-3, rnn_policy_lr=1e-5,
                     rnn_value_lr=1e-5, alpha_lr=1e-4, target_entropy_ratio=1.0, sac_batch_size=sum(lens) - 1, sac_alpha=0.2,
                     max_buffer_transition_num=max(1000, sum(lens) + 8), policy_l2_norm=0.0, value_l2_norm=0.0), **kw)


def _build(kind, enc, S, A, H, lens, emb=32, **hp):
    from rorl_b200.utility.alg_init import alg_class
    from rorl_b200.buffers.transition_buffer.replay_memory import Transition
    from test_update_gpu import fill_buffer_discrete
    cls = alg_class(CLASSES[kind])
    # the ensembleQ classes hand the target policy the raw action index as its last action (ref :141): no last-action input
    last_action = kind == "redq"
    alg = cls(_hp(lens, **hp), _kw(enc, S, A, H, False, emb, last_action), _kw(enc, S, A, H, True, emb, last_action), max(lens),
              device=DEV, discrete_env=True)
    fill_buffer_discrete(alg.replay_buffer, Transition, np.random.RandomState(4), lens, S, A)
    return alg, last_action


@pytest.mark.parametrize("enc,kind,A,H,lens", [
    ("gilr", "redq", 4, 64, [40, 13, 25, 37, 9, 30]),
    ("gilr", "ensembleq", 18, 64, [40, 13, 25, 37, 9, 30]),
    ("smamba_s16_c4_b1", "redq", 18, 64, [40, 13, 25, 37, 9, 30]),
    ("smamba_s16_c4_b1", "ensembleq", 4, 64, [33, 40, 11, 26, 19]),
    ("gilr", "redq", 18, 256, [1000] * 32),
])
def test_discrete_update_vs_oracle(enc, kind, A, H, lens):
    """Whole discrete SAC updates (nest-stacked rows) against the oracle's CPU update on the same weights, replay and
    numpy RNG stream: losses and gradients to 1e-3, updated parameters to 1e-3 with AdamW's eps-regime allowance."""
    from oracle import model as OM, sampler as OS, update as OU
    from test_update_gpu import fill_buffer_discrete
    S = 5
    torch.manual_seed(3)
    emb = 128 if H == 256 else 32
    alg, last_action = _build(kind, enc, S, A, H, lens, emb)
    with torch.no_grad():
        for m in (alg.policy, alg.values[0]):
            for p in m.parameters():
                if p.dim() == 1:
                    p.add_(0.05 * torch.randn_like(p))
    alg._finalize_models()
    cpu_sd = lambda model: {k: {n: t.detach().cpu().clone() for n, t in sd.items()} for k, sd in model.state_dict().items()}
    obuf = OS.RefNestedReplay(max(1000, sum(lens) + 8), max(lens), additional_history_len=alg._get_skip_len())
    fill_buffer_discrete(obuf, OS.Transition, np.random.RandomState(4), lens, S, A)
    hp = _hp(lens)
    upd = OU.RefUpdate(cpu_sd(alg.policy), cpu_sd(alg.values[0]), OM.ModelSpec(**_kw(enc, S, A, H, False, emb, last_action)),
                       OM.ModelSpec(**_kw(enc, S, A, H, True, emb, last_action)), hp, obuf, None, algo="sac",
                       redq=kind == "redq", allow_nest_stack=alg.allow_nest_stack, discrete=True)
    eps_zone = {}
    for call in range(2):
        np.random.seed(100 + call)
        ref = upd.train_one_batch()
        np.random.seed(100 + call)
        log = alg.train_one_batch()
        for k in ("critic_loss", "actor_loss", "log_prob", "target_q_max", "clip_min", "clip_max", "log_alpha"):
            if k in ref:
                assert abs(log[k] - ref[k]) <= 1e-3 * max(1.0, abs(ref[k])), (k, log[k], ref[k])
        for grads, model in ((upd.value_grads, alg.values[0]), (upd.policy_grads, alg.policy)):
            for mod, mm in model.contextual_modules.items():
                for n, p_ in mm.named_parameters():
                    if grads[mod][n] is not None and p_.grad is not None:
                        assert_close(p_.grad, grads[mod][n], 1e-3, f"grad/{mod}/{n}")
        for which, model, osd, ograds in (("policy", alg.policy, upd.policy, upd.policy_grads),
                                          ("value", alg.values[0], upd.value, upd.value_grads),
                                          ("target", alg.target_values[0], upd.target, upd.value_grads)):
            for mod, params in model.state_dict().items():
                for n, t in params.items():
                    r = osd[mod][n].detach()
                    diff = (t.cpu() - r).abs()
                    scale = float(r.abs().max()) + 1e-30
                    gref = ograds.get(mod, {}).get(n)
                    small = eps_zone.get((which, mod, n), torch.zeros_like(r, dtype=torch.bool))
                    if gref is not None:
                        small = small | (gref.detach().abs() < 1e-6)
                    eps_zone[(which, mod, n)] = small
                    if (~small).any():
                        bound = 1e-3 * scale + 0.01 * hp["value_lr"] * (call + 1)
                        assert float(diff[~small].max()) <= bound, f"{which}/{mod}/{n}: {float(diff[~small].max()):.3e} > {bound:.3e}"
                    if small.any():
                        assert float(diff[small].max()) <= 2.2 * hp["value_lr"] * (call + 1), f"{which}/{mod}/{n} (eps regime)"


def _snapshot(alg, logs):
    sd = {f"{w}/{m}/{n}": t.detach().clone() for w, model in (("p", alg.policy), ("v", alg.values[0]), ("t", alg.target_values[0]))
          for m, params in model.state_dict().items() for n, t in params.items()}
    keys = ("critic_loss", "actor_loss", "log_prob", "target_q_max", "clip_min", "clip_max")
    return [tuple(l[k] for k in keys) for l in logs], sd, alg.Q_guard.state.clone()


def _assert_bit_identical(a, b):
    (la, sa, ga), (lb, sb, gb) = a, b
    assert la == lb
    assert torch.equal(ga, gb)
    for k in sa:
        assert torch.equal(sa[k], sb[k]), k


@pytest.mark.parametrize("enc,kind,A", [("gilr", "redq", 4), ("smamba_s16_c4_b1", "ensembleq", 18)])
def test_discrete_graph_replay_matches_eager(enc, kind, A):
    """From the third update on the discrete update is replayed from captured CUDA graphs (nothing in it reads back to the
    host, or capture would fail); five replayed updates leave exactly what five eager updates leave."""
    lens = [40, 40, 40, 40]
    runs = []
    for graph in (False, True):
        torch.manual_seed(3)
        alg, _ = _build(kind, enc, 5, A, 64, lens, use_cuda_graph=graph)
        np.random.seed(50)
        logs = []
        for i in range(5):
            logs.append(alg.train_one_batch())
            if graph and i == 2:
                assert any(isinstance(v, dict) for v in alg._graphs.values()), "no graph was captured"
        if not graph:
            assert not alg._graphs
        runs.append(_snapshot(alg, logs))
    _assert_bit_identical(*runs)


def test_discrete_graph_refused_for_unsafe_sample_fn():
    alg, _ = _build("redq", "gilr", 5, 4, 64, [40, 40])
    assert alg._graph_allowed()
    alg.policy.sample_fn = lambda probs: probs.argmax(-1, keepdim=True)
    assert not alg._graph_allowed()
    alg.policy.sample_fn.graph_safe = True
    assert alg._graph_allowed()


@pytest.mark.parametrize("enc,kind", [("gilr", "ensembleq"), ("smamba_s16_c4_b1", "redq")])
def test_discrete_side_stream_bit_identical(enc, kind, monkeypatch):
    lens = [40, 33, 25, 37]
    runs = []
    for side in ("1", "0"):
        monkeypatch.setenv("RORL_SIDE_STREAM", side)
        torch.manual_seed(3)
        alg, _ = _build(kind, enc, 5, 18, 64, lens)
        assert (alg._side_stream is not None) == (side == "1")
        np.random.seed(60)
        runs.append(_snapshot(alg, [alg.train_one_batch() for _ in range(4)]))
    _assert_bit_identical(*runs)
