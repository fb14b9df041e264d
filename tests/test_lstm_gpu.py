"""GPU parity of the `lstm` encoder (csrc/lstm.cu + kernels.LSTMScan + models/lstm) against torch.nn.LSTM on CPU:
the layer with all gradients, the rollout path with a carried (h, c), the complete update against the oracle's CPU
update (SAC and TD3, nest-stacked rows), graph replay against eager launches, and one update at the benchmark's size.
Tolerance: <= 1e-3 relative (fp32), as for every fp32 path."""
import numpy as np
import pytest
import torch

import lstm_oracle as LO
from helpers import assert_close
from test_update_gpu import fill_buffer

pytestmark = pytest.mark.gpu
TOL = 1e-3


def _layer_vs_torch(B, L, I, H, with_h0, seed=0):
    from rorl_b200.models.lstm.lstm import LSTMLayer
    gen = torch.Generator().manual_seed(seed)
    ref = torch.nn.LSTM(I, H, batch_first=True)
    with torch.no_grad():
        for p in ref.parameters():                      # non-zero biases, so that b_ih and b_hh are both exercised
            p.copy_((torch.rand(p.shape, generator=gen) * 2 - 1) / H ** 0.5)
    mine = LSTMLayer(I, H).cuda()
    mine.load_state_dict(ref.state_dict())
    x = torch.randn(B, L, I, generator=gen)
    gout, gh, gc = torch.randn(B, L, H, generator=gen), torch.randn(1, B, H, generator=gen), torch.randn(1, B, H, generator=gen)
    hx = (0.5 * torch.randn(1, B, H, generator=gen), 0.5 * torch.randn(1, B, H, generator=gen)) if with_h0 else None

    def run(layer, dev):
        xx = x.to(dev).requires_grad_()
        h = None if hx is None else tuple(t.to(dev).requires_grad_() for t in hx)
        out, (hn, cn) = layer(xx, h)
        loss = (out * gout.to(dev)).sum() + (hn * gh.to(dev)).sum() + (cn * gc.to(dev)).sum()
        params = list(layer.parameters())
        grads = torch.autograd.grad(loss, [xx] + params + ([] if h is None else list(h)))
        return (out, hn, cn), grads

    (o_r, h_r, c_r), g_r = run(ref, "cpu")
    (o_m, h_m, c_m), g_m = run(mine, "cuda")
    assert_close(o_m, o_r, TOL, "out")
    assert_close(h_m, h_r, TOL, "h_n")
    assert_close(c_m, c_r, TOL, "c_n")
    names = ["dx"] + [n for n, _ in ref.named_parameters()] + (["dh0", "dc0"] if with_h0 else [])
    for n, a, b in zip(names, g_m, g_r):
        assert_close(a, b, TOL, n)


@pytest.mark.parametrize("H", [16, 32, 64, 128, 256])
@pytest.mark.parametrize("with_h0", [False, True])
def test_lstm_layer_vs_torch_cpu(H, with_h0):
    _layer_vs_torch(5, 37, 12, H, with_h0, seed=H)


def test_lstm_layer_more_rows_than_clusters():
    """150 rows: more batch groups than co-resident clusters, so every cluster walks several groups."""
    _layer_vs_torch(150, 20, 24, 64, True, seed=1)
    _layer_vs_torch(150, 9, 16, 256, True, seed=2)


def test_lstm_layer_benchmark_shape():
    _layer_vs_torch(32, 1002, 256, 256, False, seed=3)


def test_lstm_scan_graph_replay_bit_identical():
    """Forward + backward of the recurrence captured in a CUDA graph leave exactly what the eager launches leave."""
    import rorl_b200.kernels as K
    B, L, H = 32, 200, 256
    gen = torch.Generator().manual_seed(5)
    base = [torch.randn(B, L, 4 * H, generator=gen), 0.06 * torch.randn(4 * H, H, generator=gen), torch.randn(4 * H, generator=gen),
            torch.randn(B, H, generator=gen), torch.randn(B, H, generator=gen)]
    base = [t.cuda() for t in base]
    dout = torch.randn(B, L, H, generator=gen).cuda()

    def step():              # fresh leaves per call: no autograd node outlives the stream it was created on
        ins = [t.detach().requires_grad_() for t in base]
        out, hl, cl = K.lstm_scan(*ins)
        return (out, hl, cl) + torch.autograd.grad((out * dout).sum() + hl.sum() + cl.sum(), ins)

    eager = [t.clone() for t in step()]
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        step()                                           # warm-up on the capture stream
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        static = step()
    g.replay()
    torch.cuda.synchronize()
    for a, r in zip(static, eager):
        assert torch.equal(a, r)


def _net(H=64):
    from rorl_b200.models.rnn_base import RNNBase
    torch.manual_seed(7)
    net = RNNBase(12, 8, [H, H], ['elu', 'elu', 'linear'], ['fc', 'lstm', 'fc'])
    with torch.no_grad():
        for p in net.parameters():
            if p.dim() == 1:
                p.add_(0.1 * torch.randn_like(p))
    return net.cuda()


def test_lstm_rollout_carry_matches_full_pass_and_oracle():
    """L = 1 calls through RNNBase.meta_forward with (h, c) carried equal one full pass and the oracle's CPU layer;
    two pieces with the state handed over equal the single pass."""
    from oracle import model as OM
    net = _net()
    B, L = 6, 23
    x = torch.randn(B, L, 12).cuda()
    torch.manual_seed(9)
    st0 = net.make_rnd_init_state(B, torch.device("cuda"))
    h0, c0 = st0[0]
    with torch.no_grad():
        full, st_full, _ = net.meta_forward(x, st0)
        st, outs = st0, []
        for t in range(L):
            y, st, _ = net.meta_forward(x[:, t:t + 1], st)
            outs.append(y)
        steps = torch.cat(outs, dim=1)
        a, st_a, _ = net.meta_forward(x[:, :10], st0)
        b, st_b, _ = net.meta_forward(x[:, 10:], st_a)
    sd = {k: v.detach().cpu() for k, v in net.state_dict().items()}
    side = OM.Side(h0={1: (h0.cpu(), c0.cpu())})
    ref = LO.rnn_base(sd, ['fc', 'lstm', 'fc'], ['elu', 'elu', 'linear'], x.cpu(), side)
    h_ref, c_ref = side.h_out
    assert_close(full, ref, TOL, "full pass vs oracle")
    assert_close(steps, ref, TOL, "L = 1 steps vs oracle")
    assert_close(torch.cat((a, b), dim=1), ref, TOL, "two pieces vs oracle")
    for got in (st_full[0], st[0], st_b[0]):
        assert_close(got[0], h_ref, TOL, "h_n")
        assert_close(got[1], c_ref, TOL, "c_n")


def _kw(S, A, H, value, emb=32):
    return dict(state_dim=S, action_dim=A, embedding_size=emb, embedding_hidden=[H, H], embedding_activations=['elu', 'elu', 'linear'],
                embedding_layer_type=['fc', 'lstm', 'fc'], uni_model_hidden=[H, H], uni_model_activations=['elu', 'elu', 'linear'],
                uni_model_layer_type=(['efc-8'] * 3 if value else ['fc'] * 3), fix_rnn_length=0, uni_model_input_mapping_dim=emb,
                reward_input=False, last_action_input=True, last_state_input=True, separate_encoder=True)


def _update_vs_oracle(monkeypatch, algo, S, A, H, lens, calls, randomize_first_hidden=False, check_params=True, emb=32,
                      nested=True):
    from oracle import model as OM, sampler as OS, update as OU
    monkeypatch.setattr(OM, "rnn_base", LO.rnn_base)            # the oracle's model stack with the lstm layer
    from rorl_b200.algorithm.sac_full_length_rnn_redq_sep_optim import SACFullLengthRNNREDQ_SEP_OPTIM
    from rorl_b200.algorithm.td3_full_length_rnn_redq_sep_optim import TD3FullLengthRNNREDQ_SEP_OPTIM
    from rorl_b200.buffers.transition_buffer.replay_memory import Transition
    from rorl_b200.models import RNNHidden as RH
    hp = dict(gamma=0.99, sac_tau=0.995, policy_update_per=1, redq_m=2, policy_lr=3e-4, value_lr=1e-3, rnn_policy_lr=1e-5,
              rnn_value_lr=1e-5, alpha_lr=1e-4, target_entropy_ratio=1.0, sac_batch_size=sum(lens) - 1,
              max_buffer_transition_num=sum(lens) + 1000, sample_std=0.1, target_action_noise_std=0.04,
              target_action_noise_clip=0.12, policy_l2_norm=0.0, value_l2_norm=0.0,
              randomize_first_hidden=randomize_first_hidden)
    torch.manual_seed(3)
    cls = SACFullLengthRNNREDQ_SEP_OPTIM if algo == "sac" else TD3FullLengthRNNREDQ_SEP_OPTIM
    alg = cls(dict(hp), _kw(S, A, H, False, emb), _kw(S, A, H, True, emb), max(lens), device=torch.device("cuda:0"))
    assert alg.allow_nest_stack
    with torch.no_grad():
        for m in (alg.policy, alg.values[0]):
            for p in m.parameters():
                if p.dim() == 1:
                    p.add_(0.05 * torch.randn_like(p))
    alg._finalize_models()
    cpu_sd = lambda model: {k: {n: t.detach().cpu().clone() for n, t in sd.items()} for k, sd in model.state_dict().items()}
    pol_sd, val_sd = cpu_sd(alg.policy), cpu_sd(alg.values[0])
    fill_buffer(alg.replay_buffer, Transition, np.random.RandomState(4), lens, S, A)
    obuf = OS.RefNestedReplay(sum(lens) + 1000, max(lens), additional_history_len=alg._get_skip_len())
    fill_buffer(obuf, OS.Transition, np.random.RandomState(4), lens, S, A)
    gen = torch.Generator().manual_seed(8)
    drawn, hdraws = [], []

    def o_noise(shape):
        n = torch.randn(tuple(shape), generator=gen)
        drawn.append(n)
        return n

    def hidden_fn(spec, batch):          # (h, c) of the embedding network's LSTM (layer 1), h drawn first (RNNHidden order)
        h, c = (torch.rand((1, batch, H), generator=gen) for _ in range(2))
        hdraws.extend([h, c])                # the raw uniform draws: RNNHidden maps them to [-1, 1) itself
        return {1: (h * 2 - 1, c * 2 - 1)}

    upd = OU.RefUpdate(pol_sd, val_sd, OM.ModelSpec(**_kw(S, A, H, False, emb)), OM.ModelSpec(**_kw(S, A, H, True, emb)), hp, obuf,
                       o_noise, algo=algo, redq=True, allow_nest_stack=alg.allow_nest_stack, hidden_fn=hidden_fn)
    try:
        for call in range(calls):
            np.random.seed(100 + call)
            plan = alg.replay_buffer.plan_trajs(hp["sac_batch_size"], None, nest_stack_trajs=alg.allow_nest_stack)
            if nested:           # the (h, c) state runs on from one trajectory into the next in the same row (no reset)
                assert int((plan.lens[:, 1:] > 0).sum(1).max()) >= 2, "no batch row holds two trajectories"
            drawn.clear(), hdraws.clear()
            np.random.seed(100 + call)
            ref = upd.train_one_batch()
            it = iter([d.cuda() for d in drawn])
            alg.policy.noise_fn = alg.target_policy.noise_fn = lambda like: next(it)
            if randomize_first_hidden:
                from test_update_gpu import _TorchWithRand
                RH.torch = _TorchWithRand(iter([d.cuda() for d in hdraws]))
            np.random.seed(100 + call)
            log = alg.train_one_batch()
            RH.torch = torch
            for k in ("critic_loss", "actor_loss", "alpha_loss", "log_prob", "target_q_max"):
                if k in ref and k in log:
                    assert abs(log[k] - ref[k]) <= TOL * max(1.0, abs(ref[k])), (k, log[k], ref[k])
            for grads, model in ((upd.value_grads, alg.values[0]), (upd.policy_grads, alg.policy)):
                for mod, m in model.contextual_modules.items():
                    for n, p_ in m.named_parameters():
                        if grads[mod][n] is not None and p_.grad is not None:
                            if check_params:
                                assert_close(p_.grad, grads[mod][n], TOL, f"grad/{mod}/{n}")
                            else:                 # one gradient norm per parameter
                                gn, rn = float(p_.grad.norm()), float(grads[mod][n].norm())
                                assert abs(gn - rn) <= TOL * max(rn, 1e-12), (f"|grad|/{mod}/{n}", gn, rn)
            if not check_params:
                continue
            for which, model, osd, ograds in (("policy", alg.policy, upd.policy, upd.policy_grads),
                                              ("value", alg.values[0], upd.value, upd.value_grads)):
                for mod, params in model.state_dict().items():
                    for n, t in params.items():
                        r = osd[mod][n].detach()
                        diff = (t.cpu() - r).abs()
                        g = ograds.get(mod, {}).get(n)
                        small = torch.zeros_like(r, dtype=torch.bool) if g is None else g.detach().abs() < 1e-6
                        # as in test_update_vs_oracle_wide: AdamW steps of entries inside the eps regime may flip
                        bound = TOL * (float(r.abs().max()) + 1e-30) + 0.01 * hp["value_lr"] * (call + 1)
                        if (~small).any():
                            assert float(diff[~small].max()) <= bound, f"{which}/{mod}/{n}"
                        if small.any():
                            assert float(diff[small].max()) <= 2.2 * hp["value_lr"] * (call + 1), f"{which}/{mod}/{n} (eps regime)"
    finally:
        RH.torch = torch


@pytest.mark.parametrize("algo", ["sac", "td3"])
def test_lstm_update_vs_oracle_wide(algo, monkeypatch):
    _update_vs_oracle(monkeypatch, algo, 5, 3, 64, [40, 12, 25, 15, 9, 37], calls=2)


def test_lstm_update_vs_oracle_random_first_hidden(monkeypatch):
    _update_vs_oracle(monkeypatch, "sac", 5, 3, 64, [40, 12, 25, 15, 9, 37], calls=2, randomize_first_hidden=True)


def test_lstm_update_benchmark_size_vs_oracle(monkeypatch):
    """One SAC update at the benchmark's size (32 rows x 1000 steps, width 256) against the oracle's CPU update:
    logged scalars and one gradient norm per parameter (obs 9, act 6, embedding 128, as in bench.py)."""
    _update_vs_oracle(monkeypatch, "sac", 9, 6, 256, [1000] * 32, calls=1, check_params=False, emb=128, nested=False)


def test_lstm_cuda_graph_replay_matches_eager():
    """Modelled on test_update_gpu.test_cuda_graph_replay_matches_eager: the update replayed from a captured graph
    leaves what the eager launches leave.  The LSTM kernels are deterministic; the K < 32 input projections run through
    cuBLAS, which may pick another algorithm under capture, so rounding-level differences are allowed there."""
    from rorl_b200.algorithm.sac_full_length_rnn_redq_sep_optim import SACFullLengthRNNREDQ_SEP_OPTIM
    from rorl_b200.buffers.transition_buffer.replay_memory import Transition
    S, A, H = 5, 3, 64
    lens = [40, 40, 40, 40]
    hp = dict(gamma=0.99, sac_tau=0.995, policy_update_per=1, redq_m=2, policy_lr=3e-4, value_lr=1e-3, rnn_policy_lr=1e-5,
              rnn_value_lr=1e-5, alpha_lr=1e-4, target_entropy_ratio=1.0, sac_batch_size=sum(lens) - 1,
              max_buffer_transition_num=1000)

    def noise(like):
        n = like.numel()
        return torch.sin(torch.arange(n, device=like.device, dtype=torch.float32) * 12.9898).reshape(like.shape)
    noise.graph_safe = True
    results = []
    for graph in (False, True):
        torch.manual_seed(3)
        alg = SACFullLengthRNNREDQ_SEP_OPTIM(dict(hp, use_cuda_graph=graph), _kw(S, A, H, False), _kw(S, A, H, True), max(lens),
                                             device=torch.device("cuda:0"))
        alg.policy.noise_fn = alg.target_policy.noise_fn = noise
        fill_buffer(alg.replay_buffer, Transition, np.random.RandomState(4), lens, S, A)
        np.random.seed(50)
        logs = [alg.train_one_batch() for _ in range(5)]
        if graph:
            assert any(isinstance(v, dict) for v in alg._graphs.values()), "no graph was captured"
        sd = {f"{w}/{m}/{n}": t.detach().clone() for w, model in (("p", alg.policy), ("v", alg.values[0]), ("t", alg.target_values[0]))
              for m, params in model.state_dict().items() for n, t in params.items()}
        results.append((logs, sd))
    (le, se), (lg, sg) = results
    for a, b in zip(le, lg):
        for k in ("critic_loss", "actor_loss", "target_q_max", "log_alpha"):
            if k in a:
                assert abs(a[k] - b[k]) <= 1e-5 * max(1.0, abs(a[k])), (k, a[k], b[k])
    exact = True
    for k in se:
        exact = exact and torch.equal(se[k], sg[k])
        assert_close(sg[k], se[k], 2e-4, k)
    print(f"lstm graph vs eager after 5 updates: bit-identical={exact}")
