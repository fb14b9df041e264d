"""GPU parity of the tcgen05 attention kernels and the cgpt encoder at head dimensions other than 64 (every multiple of 8
from 8 to 128; the operands are padded to 64 or 128 along d): the kernels against the fp32 oracle and against
flash-attn 2's recorded results, the decoder stack and the kv-cache rollout, full SAC / TD3 updates against the oracle's
CPU update, and graph replay.  Tolerance 1e-2 relative (max-norm), as for head dimension 64 (bf16 operands)."""
import math

import numpy as np
import pytest
import torch

from helpers import assert_close
from test_attn_gpu import _seqs
from test_update_gpu import fill_buffer

pytestmark = pytest.mark.gpu
TOL = 1e-2

LAYOUTS = {"ragged": ([1, 130, 1, 300, 64, 128, 129], [0, 0, 3, 0, 1, 0, 5]), "long": ([1001, 1, 1001], [0, 0, 0]),
           "one": ([17], [2]), "tiles": ([256, 512], [0, 0])}


def _slopes(H):
    from oracle import attention as OA
    return OA.alibi_slopes(H)


@pytest.mark.parametrize("layout", list(LAYOUTS))
@pytest.mark.parametrize("hd", [8, 16, 32, 48, 96, 128])
def test_attention_hd_vs_oracle(hd, layout):
    """Output and qkv gradients against the fp32 oracle on ragged sequences with gaps, 1-token and 1001-token sequences
    and 128-row tile boundaries; rows outside every sequence stay exactly zero."""
    import rorl_b200.kernels as K
    from oracle import attention as OA
    lens, gaps = LAYOUTS[layout]
    H = 8 if hd <= 64 else 4
    starts, used = _seqs(lens, gaps)
    T = used + 7
    gen = torch.Generator().manual_seed(T + hd)
    qkv = torch.randn(T, 3, H, hd, generator=gen)
    dout = torch.randn(T, H * hd, generator=gen)
    scale = 1.0 / math.sqrt(hd)
    ref_in = qkv.clone().requires_grad_()
    ref = OA.attention_varlen(ref_in, starts, lens, _slopes(H), scale)
    inside = torch.zeros(T, 1)
    for s, n in zip(starts, lens):
        inside[s:s + n] = 1
    (ref * dout * inside).sum().backward()
    x = qkv.cuda().requires_grad_()
    tiles, gmap = (t.cuda() for t in K.attention_tiles(starts, lens))
    out = K.attn_varlen_alibi(x, tiles, gmap, torch.tensor(_slopes(H), dtype=torch.float32, device="cuda"), scale)
    (out * (dout * inside).cuda()).sum().backward()
    assert out.shape == (T, H * hd)
    assert_close(out, ref, TOL, "out")
    outside = inside[:, 0] == 0
    if outside.any():
        assert float(out.detach().cpu()[outside].abs().max()) == 0.0
        assert float(x.grad.cpu()[outside].abs().max()) == 0.0
    for i, name in enumerate("qkv"):
        assert_close(x.grad[:, i], ref_in.grad[:, i], TOL, f"d{name}")


@pytest.mark.parametrize("hd", [32, 128])
def test_attention_hd_dropout_explicit_mask(hd):
    """The kernels' keep mask (kernels.attention_dropout_mask) applied in an fp32 torch attention reproduces the kernel's
    output and gradients at head dimensions 32 and 128."""
    import rorl_b200.kernels as K
    H, p_drop = 4, 0.25
    lens, gaps = [100, 37, 130], [0, 0, 3]
    starts, used = _seqs(lens, gaps)
    T = used + 5
    gen = torch.Generator().manual_seed(11 + hd)
    qkv = torch.randn(T, 3, H, hd, generator=gen)
    dout = torch.randn(T, H * hd, generator=gen)
    slopes = _slopes(H)
    scale = 1.0 / math.sqrt(hd)
    tiles, gmap = K.attention_tiles(starts, lens)
    Ta = gmap.shape[0]
    Tp = (Ta + 63) // 64 * 64
    seed_val, salt = 2024 + hd, 99
    mask = K.attention_dropout_mask(seed_val, salt, H, Ta, Tp, p_drop)
    pos = {row[3]: row[0] for row in tiles.tolist()}            # attention-space start of each sequence
    ref_in = qkv.clone().requires_grad_()
    ref = torch.zeros(T, H * hd)
    sl = torch.tensor(slopes).view(H, 1, 1)
    for s0, n in zip(starts, lens):
        q, k, v = (ref_in[s0:s0 + n, i].transpose(0, 1) for i in range(3))
        idx = torch.arange(n)
        rel = (idx.view(n, 1) - idx.view(1, n)).float()
        sc = (scale * q @ k.transpose(1, 2) - sl * rel).masked_fill(rel.unsqueeze(0) < 0, float("-inf"))
        a0 = pos[s0]
        pd = torch.softmax(sc, dim=-1) * mask[:, a0:a0 + n, a0:a0 + n]
        ref = ref.index_add(0, torch.arange(s0, s0 + n), (pd @ v).transpose(0, 1).reshape(n, H * hd))
    inside = torch.zeros(T, 1)
    for s0, n in zip(starts, lens):
        inside[s0:s0 + n] = 1
    (ref * dout * inside).sum().backward()
    x = qkv.cuda().requires_grad_()
    seed = torch.tensor([seed_val], dtype=torch.int64, device="cuda")
    out = K.attn_varlen_alibi(x, tiles.cuda(), gmap.cuda(), torch.tensor(slopes, dtype=torch.float32, device="cuda"), scale, p_drop,
                              seed, salt)
    (out * (dout * inside).cuda()).sum().backward()
    assert_close(out, ref, 2e-2, "out with dropout")
    for i, name in enumerate("qkv"):
        assert_close(x.grad[:, i], ref_in.grad[:, i], 2e-2, f"d{name} with dropout")


# flash-attn comparison cases: head dimension -> heads.  Inputs and sampled rows as for the head-dim-64 fixture.
FLASH_HD_CASES = {32: 8, 128: 4}
FLASH_HD_LENS = [1, 1001, 1, 700, 301]
FLASH_HD_PROBE = 4099


def flash_attn_hd_case(hd):
    """Inputs of the flash-attn comparison at head dimension hd (CPU): sequence starts, lengths, heads, packed qkv
    [T, 3, H, hd], output gradient [T, H * hd]."""
    H = FLASH_HD_CASES[hd]
    starts, T = _seqs(FLASH_HD_LENS, [0] * len(FLASH_HD_LENS))
    gen = torch.Generator().manual_seed(3 + hd)
    qkv = torch.randn(T, 3, H, hd, generator=gen)
    dout = torch.randn(T, H * hd, generator=gen)
    return starts, FLASH_HD_LENS, H, qkv, dout


@pytest.mark.parametrize("hd", list(FLASH_HD_CASES))
def test_attention_hd_vs_flash_attn(hd):
    """flash-attn 2.8.3's varlen kernel (bf16, ALiBi, causal) on the same inputs, as recorded on a B200 by
    tests/golden/make_golden_flash_attn_hd.py (attn_flash_varlen_hd{32,128}.npz)."""
    import rorl_b200.kernels as K
    from helpers import load_npz
    g = load_npz(f"attn_flash_varlen_hd{hd}.npz")
    starts, lens, H, qkv, dout = flash_attn_hd_case(hd)
    assert np.array_equal(qkv.reshape(-1)[::FLASH_HD_PROBE].numpy(), g["qkv_probe"])
    assert np.array_equal(dout.reshape(-1)[::FLASH_HD_PROBE].numpy(), g["dout_probe"])
    x = qkv.cuda().requires_grad_()
    tiles, gmap = (t.cuda() for t in K.attention_tiles(starts, lens))
    out = K.attn_varlen_alibi(x, tiles, gmap, torch.tensor(_slopes(H), dtype=torch.float32, device="cuda"), 1.0 / math.sqrt(hd))
    out.backward(dout.cuda())
    rows = torch.from_numpy(g["rows"])
    bf16 = lambda bits: torch.from_numpy(bits.view(np.int16)).view(torch.bfloat16).float()
    assert_close(out.detach().cpu()[rows], bf16(g["out_bf16"]), 2e-2, "out vs flash-attn (both bf16)")
    assert_close(x.grad.cpu()[rows], bf16(g["dqkv_bf16"]), 3e-2, "dqkv vs flash-attn (both bf16)")


@pytest.mark.parametrize("case", ["c256_h8_ln_stacked", "c512_h4_rms_rows"])
def test_cgpt_encoder_hd_vs_oracle(case):
    """TransformerDecoder at head dims 32 and 128 against oracle.attention.decoder_forward: forward, dx and every
    parameter gradient."""
    from oracle import attention as OA
    from rorl_b200.models.flash_attention.TransformerFlashAttention import TransformerDecoder
    torch.manual_seed(0)
    if case == "c256_h8_ln_stacked":
        C, Hh, B, L, ln = 256, 8, 3, 300, True
        seq = np.zeros((B, L), dtype=np.int64)
        seq[0, :2] = (200, 100); seq[1, :3] = (1, 150, 99); seq[2, :1] = (212,)
    else:
        C, Hh, B, L, ln = 512, 4, 2, 1002, False
        seq = np.zeros((B, L), dtype=np.int64)
        seq[:, 0] = 1; seq[:, 1] = 1001
    net = TransformerDecoder(C, Hh, 4 * C, 2, dropout=0.0, ln=ln)
    with torch.no_grad():
        for p in net.parameters():
            if p.dim() == 1:
                p.add_(0.1 * torch.randn_like(p))
    sd = {k: v.detach().clone().requires_grad_() for k, v in net.state_dict().items()}
    x = torch.randn(B, L, C)
    dy = torch.randn(B, L, C)
    xr = x.clone().requires_grad_()
    ref = OA.decoder_forward(sd, xr, seq, Hh, ln)
    (ref * dy).sum().backward()
    net.cuda().train()
    xg = x.cuda().requires_grad_()
    s_dev = torch.from_numpy(seq).to(torch.int32).cuda()
    s_dev._host = seq
    out = net(xg, None, s_dev)
    (out * dy.cuda()).sum().backward()
    assert_close(out, ref, TOL, "y")
    assert_close(xg.grad, xr.grad, TOL, "dx")
    for n, p in net.named_parameters():
        assert_close(p.grad, sd[n].grad, 2e-2, n)


@pytest.mark.parametrize("lid", ["cgpt_h8_l2_p0.0_ml64", "cgpt_h2_l2_p0.0_ml64"])
def test_cgpt_hd_kv_cache_decode_matches_full_forward(lid):
    """Rollout at width 256 with head dims 32 and 128: decoding one token at a time against the kv-cache reproduces the
    causal full-sequence forward at every position."""
    from rorl_b200.models.rnn_base import RNNBase
    torch.manual_seed(2)
    net = RNNBase(10, 6, [256, 256], ['elu', 'elu', 'linear'], ['fc', lid, 'fc']).cuda().eval()
    B, T = 3, 37
    x = torch.randn(B, T, 10, device="cuda")
    with torch.no_grad():
        y_full, _, _ = net.meta_forward(x, net.make_init_state(B, x.device))
        hid = net.make_init_state(B, x.device)
        ys = []
        for t in range(T):
            y, hid, _ = net.meta_forward(x[:, t:t + 1], hid)
            ys.append(y)
    assert hid[0].seqlen_offset == T
    assert_close(torch.cat(ys, dim=1), y_full, TOL, "decoded steps vs full forward")


def _kw(S, A, H, enc, value, emb=32):
    return dict(state_dim=S, action_dim=A, embedding_size=emb, embedding_hidden=[H, H], embedding_activations=['elu', 'elu', 'linear'],
                embedding_layer_type=['fc', enc, 'fc'], uni_model_hidden=[H, H], uni_model_activations=['elu', 'elu', 'linear'],
                uni_model_layer_type=(['efc-8'] * 3 if value else ['fc'] * 3), fix_rnn_length=0, uni_model_input_mapping_dim=emb,
                reward_input=False, last_action_input=True, last_state_input=True, separate_encoder=True)


def _update_vs_oracle(algo, enc, S, A, H, lens, calls, check_params=True, emb=32):
    """Modelled on test_update_gpu.test_update_vs_oracle_wide (cgpt branch): logged scalars, gradients and (with
    check_params) updated parameters against the oracle's CPU update; without it one gradient norm per parameter."""
    from oracle import model as OM, sampler as OS, update as OU
    from rorl_b200.algorithm.sac_full_length_rnn_redq_sep_optim import SACFullLengthRNNREDQ_SEP_OPTIM
    from rorl_b200.algorithm.td3_full_length_rnn_redq_sep_optim import TD3FullLengthRNNREDQ_SEP_OPTIM
    from rorl_b200.buffers.transition_buffer.replay_memory import Transition
    hp = dict(gamma=0.99, sac_tau=0.995, policy_update_per=1, redq_m=2, policy_lr=3e-4, value_lr=1e-3, rnn_policy_lr=1e-5,
              rnn_value_lr=1e-5, alpha_lr=1e-4, target_entropy_ratio=1.0, sac_batch_size=sum(lens) - 1,
              max_buffer_transition_num=sum(lens) + 1000, sample_std=0.1, target_action_noise_std=0.04,
              target_action_noise_clip=0.12, policy_l2_norm=0.0, value_l2_norm=0.0)
    torch.manual_seed(3)
    cls = SACFullLengthRNNREDQ_SEP_OPTIM if algo == "sac" else TD3FullLengthRNNREDQ_SEP_OPTIM
    alg = cls(dict(hp), _kw(S, A, H, enc, False, emb), _kw(S, A, H, enc, True, emb), max(lens), device=torch.device("cuda:0"))
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
    drawn = []

    def o_noise(shape):
        n = torch.randn(tuple(shape), generator=gen)
        drawn.append(n)
        return n

    upd = OU.RefUpdate(pol_sd, val_sd, OM.ModelSpec(**_kw(S, A, H, enc, False, emb)), OM.ModelSpec(**_kw(S, A, H, enc, True, emb)), hp,
                       obuf, o_noise, algo=algo, redq=True, allow_nest_stack=alg.allow_nest_stack)
    for call in range(calls):
        drawn.clear()
        np.random.seed(100 + call)
        ref = upd.train_one_batch()
        it = iter([d.cuda() for d in drawn])
        alg.policy.noise_fn = alg.target_policy.noise_fn = lambda like: next(it)
        np.random.seed(100 + call)
        log = alg.train_one_batch()
        for k in ("critic_loss", "actor_loss", "alpha_loss", "log_prob", "target_q_max"):
            if k in ref and k in log:
                assert abs(log[k] - ref[k]) <= TOL * max(1.0, abs(ref[k])), (k, log[k], ref[k])
        for grads, model in ((upd.value_grads, alg.values[0]), (upd.policy_grads, alg.policy)):
            for mod, m in model.contextual_modules.items():
                for n, p_ in m.named_parameters():
                    if grads[mod][n] is not None and p_.grad is not None:
                        if check_params:
                            assert_close(p_.grad, grads[mod][n], TOL, f"grad/{mod}/{n}")
                        else:
                            gn, rn = float(p_.grad.norm()), float(grads[mod][n].norm())
                            assert abs(gn - rn) <= TOL * max(rn, 1e-12), (f"|grad|/{mod}/{n}", gn, rn)
        if not check_params:
            continue
        # as in test_update_vs_oracle_wide for cgpt: 1e-2 of max|theta| plus one flipped AdamW step per update taken
        for which, model, osd in (("policy", alg.policy, upd.policy), ("value", alg.values[0], upd.value),
                                  ("target", alg.target_values[0], upd.target)):
            for mod, params in model.state_dict().items():
                for n, t in params.items():
                    r = osd[mod][n].detach()
                    bound = TOL * (float(r.abs().max()) + 1e-30) + 2.2 * hp["value_lr"] * (call + 1)
                    assert float((t.cpu() - r).abs().max()) <= bound, f"{which}/{mod}/{n}"


@pytest.mark.parametrize("algo,enc,H", [("sac", "cgpt_h2_l2_p0.0_rms", 64), ("sac", "cgpt_h8_l1_p0.0", 64),
                                        ("td3", "cgpt_h1_l1_p0.0", 128)])
def test_cgpt_hd_update_vs_oracle(algo, enc, H):
    """Head dims 32, 8 and 128 through the whole update."""
    _update_vs_oracle(algo, enc, 5, 3, H, [40, 33, 25, 37], calls=2)


def test_cgpt_hd32_update_benchmark_size_vs_oracle():
    """One SAC update at the benchmark's size (32 rows x 1000 steps, width 256, 6 layers of 8 heads: head dim 32) against
    the oracle's CPU update: logged scalars and one gradient norm per parameter (obs 9, act 6, embedding 128)."""
    _update_vs_oracle("sac", "cgpt_h8_l6_p0.0_ml1024_rms", 9, 6, 256, [1000] * 32, calls=1, check_params=False, emb=128)


def test_cgpt_hd32_cuda_graph_replay_bit_identical(monkeypatch):
    """SAC with `cgpt_h8_l2_p0.1` at width 256 (head dim 32, dropout on): the update replayed from a captured graph leaves
    bit for bit what the eager launches leave, so the device-side dropout counter draws the same masks on replay."""
    from rorl_b200.algorithm.sac_full_length_rnn_redq_sep_optim import SACFullLengthRNNREDQ_SEP_OPTIM
    from rorl_b200.buffers.transition_buffer.replay_memory import Transition
    from rorl_b200.models.flash_attention.TransformerFlashAttention import MHA
    S, A, H = 16, 4, 256                     # input width 16 + 4 + 16 >= 32: every projection runs on the project's GEMM
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
        monkeypatch.setattr(MHA, "_instances", 0)            # the same per-layer dropout salts in both runs
        enc = "cgpt_h8_l2_p0.1"
        alg = SACFullLengthRNNREDQ_SEP_OPTIM(dict(hp, use_cuda_graph=graph), _kw(S, A, H, enc, False), _kw(S, A, H, enc, True),
                                             max(lens), device=torch.device("cuda:0"))
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
                assert a[k] == b[k], (k, a[k], b[k])
    for k in se:
        assert torch.equal(se[k], sg[k]), k
