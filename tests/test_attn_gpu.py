"""GPU parity of the tcgen05 attention kernels and of the cgpt encoder built on them.  Tolerance 1e-2 relative
(max-norm): the path computes with bf16 operands like the reference's flash-attn autocast region (BASELINE.json)."""
import math

import numpy as np
import pytest
import torch

from helpers import assert_close

pytestmark = pytest.mark.gpu
TOL = 1e-2


def _seqs(lens, gaps):
    starts, pos = [], 0
    for n, g in zip(lens, gaps):
        pos += g
        starts.append(pos)
        pos += n
    return starts, pos


@pytest.mark.parametrize("lens,gaps", [([1, 130, 1, 300, 64, 128, 129], [0, 0, 3, 0, 1, 0, 5]), ([1001, 1, 1001], [0, 0, 0]),
                                       ([17], [2]), ([256, 512], [0, 0])])
def test_attention_vs_oracle(lens, gaps):
    import rorl_b200.kernels as K
    from oracle import attention as OA
    H, hd = 8, 64
    starts, used = _seqs(lens, gaps)
    T = used + 7
    gen = torch.Generator().manual_seed(T)
    qkv = torch.randn(T, 3, H, hd, generator=gen)
    dout = torch.randn(T, H * hd, generator=gen)
    slopes = OA.alibi_slopes(H)
    scale = 1.0 / math.sqrt(hd)
    ref_in = qkv.clone().requires_grad_()
    ref = OA.attention_varlen(ref_in, starts, lens, slopes, scale)
    inside = torch.zeros(T, 1)
    for s, n in zip(starts, lens):
        inside[s:s + n] = 1
    (ref * dout * inside).sum().backward()
    x = qkv.cuda().requires_grad_()
    tiles, gmap = (t.cuda() for t in K.attention_tiles(starts, lens))
    out = K.attn_varlen_alibi(x, tiles, gmap, torch.tensor(slopes, dtype=torch.float32, device="cuda"), scale)
    (out * (dout * inside).cuda()).sum().backward()
    assert_close(out, ref, TOL, "out")
    assert float(out.cpu()[inside[:, 0] == 0].abs().max() if (inside == 0).any() else 0.0) == 0.0
    for i, name in enumerate("qkv"):
        assert_close(x.grad[:, i], ref_in.grad[:, i], TOL, f"d{name}")


FLASH_LENS, FLASH_H, FLASH_HD = [1, 1001, 1, 700, 301], 8, 64
FLASH_PROBE = 4099          # stride of the input entries the fixture records, to confirm the inputs are regenerated exactly


def flash_attn_case():
    """Inputs of the flash-attn comparison (CPU): sequence starts, packed qkv [T, 3, H, hd], output gradient [T, H * hd]."""
    starts, T = _seqs(FLASH_LENS, [0] * len(FLASH_LENS))
    gen = torch.Generator().manual_seed(3)
    qkv = torch.randn(T, 3, FLASH_H, FLASH_HD, generator=gen)
    dout = torch.randn(T, FLASH_H * FLASH_HD, generator=gen)
    return starts, qkv, dout


def test_attention_vs_flash_attn():
    """Pins the third-party arithmetic: flash-attn 2's own varlen kernel (bf16, ALiBi, causal) on the same inputs, as
    recorded on a B200 by tests/golden/make_golden_flash_attn.py (attn_flash_varlen.npz: its output and qkv gradient
    on a fixed, seeded sample of token rows that includes the first and last row of every sequence)."""
    import rorl_b200.kernels as K
    from helpers import load_npz
    from oracle import attention as OA
    g = load_npz("attn_flash_varlen.npz")
    starts, qkv, dout = flash_attn_case()
    assert np.array_equal(qkv.reshape(-1)[::FLASH_PROBE].numpy(), g["qkv_probe"])
    assert np.array_equal(dout.reshape(-1)[::FLASH_PROBE].numpy(), g["dout_probe"])
    slopes = torch.tensor(OA.alibi_slopes(FLASH_H), dtype=torch.float32, device="cuda")
    x = qkv.cuda().requires_grad_()
    tiles, gmap = (t.cuda() for t in K.attention_tiles(starts, FLASH_LENS))
    out = K.attn_varlen_alibi(x, tiles, gmap, slopes, 1.0 / math.sqrt(FLASH_HD))
    out.backward(dout.cuda())
    rows = torch.from_numpy(g["rows"])
    bf16 = lambda bits: torch.from_numpy(bits.view(np.int16)).view(torch.bfloat16).float()    # stored as raw bf16 bits
    assert_close(out.detach().cpu()[rows], bf16(g["out_bf16"]), 2e-2, "out vs flash-attn (both bf16)")
    assert_close(x.grad.cpu()[rows], bf16(g["dqkv_bf16"]), 3e-2, "dqkv vs flash-attn (both bf16)")


@pytest.mark.parametrize("case", ["stacked_ln", "rows_rms"])
def test_cgpt_encoder_vs_oracle(case):
    from oracle import attention as OA
    from rorl_b200.models.flash_attention.TransformerFlashAttention import TransformerDecoder
    torch.manual_seed(0)
    C, Hh = 512, 8
    if case == "stacked_ln":
        B, L, ln, nl = 3, 300, True, 2
        seq = np.zeros((B, L), dtype=np.int64)
        seq[0, :2] = (200, 100); seq[1, :3] = (1, 150, 99); seq[2, :1] = (212,)
    else:
        B, L, ln, nl = 2, 1002, False, 2
        seq = np.zeros((B, L), dtype=np.int64)
        seq[:, 0] = 1; seq[:, 1] = 1001
    net = TransformerDecoder(C, Hh, 4 * C, nl, dropout=0.0, ln=ln)
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
    worst = 0.0
    for n, p in net.named_parameters():
        worst = max(worst, assert_close(p.grad, sd[n].grad, 2e-2, n))


def test_cgpt_kv_cache_decode_matches_full_forward():
    """Rollout path: decoding one token at a time against the kv-cache reproduces the causal full-sequence forward
    (same weights, eval mode) at every position -- the property flash-attn's own kv-cache path has; bf16 tolerance."""
    from rorl_b200.models.rnn_base import RNNBase
    torch.manual_seed(2)
    net = RNNBase(10, 6, [128, 128], ['elu', 'elu', 'linear'], ['fc', 'cgpt_h2_l2_p0.0_ml64', 'fc']).cuda().eval()
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
    y_dec = torch.cat(ys, dim=1)
    err = float((y_dec - y_full).abs().max() / y_full.abs().max())
    print(f"kv-cache decode vs full forward: max-norm relative error {err:.2e}")
    assert err < 1e-2


def _fixture(name):
    import os
    from helpers import GOLDEN, load_npz
    if not os.path.exists(os.path.join(GOLDEN, name)):
        pytest.skip(f"{name}: generated on the GPU box by tests/golden/make_golden_gpu.py (needs flash-attn), not present")
    return load_npz(name)


@pytest.mark.parametrize("tag", ["cgpt_ln", "cgpt_rms"])
def test_cgpt_layer_matches_reference(tag):
    """The cgpt encoder against the UNMODIFIED reference's TransformerDecoder run with flash-attn on a B200
    (tests/golden/layer_cgpt_*.npz, tests/golden/make_golden_gpu.py): forward, input gradient, every parameter gradient.
    Tolerance 1e-2 (bf16 attention region, BASELINE.json)."""
    from helpers import T
    from rorl_b200.models.rnn_base import RNNBase
    g = _fixture(f"layer_{tag}.npz")
    lid = str(g["layer_id"])
    net = RNNBase(12, 8, [128, 128], ['elu', 'elu', 'linear'], ['fc', lid, 'fc'])
    net.load_state_dict({k[2:]: T(v) for k, v in g.items() if k.startswith("p/")})
    net.cuda().train()
    x = T(g["x"], "cuda", grad=True)
    seq = g["seqlens"]
    s_dev = torch.from_numpy(seq).to(torch.int32).cuda()
    s_dev._host = seq
    hid = net.make_init_state(x.shape[0], x.device)
    hid.set_attention_concat_mask(s_dev)
    y, _, _ = net.meta_forward(x, hid)
    assert_close(y, g["y"], TOL, "y")
    params = dict(net.named_parameters())
    names = [k[2:] for k in g if k.startswith("g/")]
    gs = torch.autograd.grad(y, [x] + [params[n] for n in names], T(g["dy"], "cuda"))
    assert_close(gs[0], g["dx"], TOL, "dx")
    worst = 0.0
    for n, got in zip(names, gs[1:]):
        worst = max(worst, assert_close(got, g["g/" + n], 2e-2, n))
    print(f"{tag}: worst parameter-gradient error vs the reference on flash-attn {worst:.2e}")


def test_cgpt_kv_cache_matches_reference():
    """Rollout path against the reference decoding one token at a time with flash-attn's kv-cache (step_cgpt.npz)."""
    from helpers import T
    from rorl_b200.models.rnn_base import RNNBase
    g = _fixture("step_cgpt.npz")
    net = RNNBase(10, 6, [128, 128], ['elu', 'elu', 'linear'], ['fc', str(g["layer_id"]), 'fc'])
    net.load_state_dict({k[2:]: T(v) for k, v in g.items() if k.startswith("p/")})
    net.cuda().eval()
    x = T(g["x"], "cuda")
    with torch.no_grad():
        hid = net.make_init_state(x.shape[0], x.device)
        ys = []
        for t in range(x.shape[1]):
            y, hid, _ = net.meta_forward(x[:, t:t + 1], hid)
            ys.append(y)
        y_full, _, _ = net.meta_forward(x, net.make_init_state(x.shape[0], x.device))
    assert_close(torch.cat(ys, dim=1), g["y_steps"], TOL, "decoded steps")
    assert_close(y_full, g["y_full"], TOL, "full forward")


def test_attention_dropout_explicit_mask():
    """Attention-probability dropout: the kernels' keep mask (a counter hash, restated in kernels.attention_dropout_mask)
    applied in an fp32 torch attention must reproduce the kernel's output and gradients -- forward and both backward
    kernels regenerate the same mask.  Also: the keep rate is 1 - p."""
    import rorl_b200.kernels as K
    from oracle import attention as OA
    H, hd, p_drop = 4, 64, 0.25
    lens, gaps = [100, 37, 130], [0, 0, 3]
    starts, used = _seqs(lens, gaps)
    T = used + 5
    gen = torch.Generator().manual_seed(11)
    qkv = torch.randn(T, 3, H, hd, generator=gen)
    dout = torch.randn(T, H * hd, generator=gen)
    slopes = OA.alibi_slopes(H)
    scale = 1.0 / math.sqrt(hd)
    tiles, gmap = K.attention_tiles(starts, lens)
    Ta = gmap.shape[0]
    Tp = (Ta + 63) // 64 * 64
    seed_val, salt = 12345, 777
    mask = K.attention_dropout_mask(seed_val, salt, H, Ta, Tp, p_drop)           # [H, Ta, Ta]
    keep_rate = float((mask > 0).float().mean())
    assert abs(keep_rate - (1 - p_drop)) < 5e-3, keep_rate
    pos = {}                                                                       # attention-space start of each sequence
    for row in tiles.tolist():
        pos[row[3]] = row[0]
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
    out = K.attn_varlen_alibi(x, tiles.cuda(), gmap.cuda(), torch.tensor(slopes, dtype=torch.float32, device="cuda"), scale, p_drop, seed, salt)
    (out * (dout * inside).cuda()).sum().backward()
    assert_close(out, ref, 2e-2, "out with dropout")
    for i, name in enumerate("qkv"):
        assert_close(x.grad[:, i], ref_in.grad[:, i], 2e-2, f"d{name} with dropout")
    # a different seed value gives a different mask; p = 0 ignores the seed
    out2 = K.attn_varlen_alibi(qkv.cuda(), tiles.cuda(), gmap.cuda(), torch.tensor(slopes, dtype=torch.float32, device="cuda"), scale,
                               p_drop, seed + 1, salt)
    assert float((out2 - out).abs().max()) > 1e-3


def test_cgpt_dropout_active_only_in_training():
    """cgpt_*_p0.1: train() draws a fresh attention / residual dropout mask per call, eval() is deterministic and equals
    the p0.0 network (ref: TransformerFlashAttention.py:57,65-70,83-84)."""
    from rorl_b200.models.rnn_base import RNNBase
    torch.manual_seed(4)
    net = RNNBase(10, 6, [128, 128], ['elu', 'elu', 'linear'], ['fc', 'cgpt_h2_l2_p0.1_ml512', 'fc']).cuda()
    ref = RNNBase(10, 6, [128, 128], ['elu', 'elu', 'linear'], ['fc', 'cgpt_h2_l2_p0.0_ml512', 'fc']).cuda()
    ref.load_state_dict(net.state_dict())
    x = torch.randn(2, 200, 10, device="cuda")
    net.eval(); ref.eval()
    with torch.no_grad():
        a, _, _ = net.meta_forward(x, net.make_init_state(2, x.device))
        b, _, _ = ref.meta_forward(x, ref.make_init_state(2, x.device))
        assert torch.equal(a, b)
        net.train()
        c, _, _ = net.meta_forward(x, net.make_init_state(2, x.device))
        d, _, _ = net.meta_forward(x, net.make_init_state(2, x.device))
    assert float((c - a).abs().max()) > 1e-4 and float((c - d).abs().max()) > 1e-4
    assert float((c - a).abs().mean() / a.abs().mean()) < 0.5          # a perturbation, not garbage
