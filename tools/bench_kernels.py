#!/usr/bin/env python
"""Per-kernel micro-benchmark at the workload shapes (SURVEY.md 8d): CUDA-event time per launch, algorithmic
bytes / FLOPs, fraction of the measured peak.  Inputs are larger than L2 or rotated so launches do not hit in cache.

    python tools/bench_kernels.py [--only gilr,lru,selscan,conv,addnorm,gru,lstm,gemm,attn,attn_hd] [--out kernels.json]
"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import rorl_b200.kernels as K  # noqa: E402
import rorl_b200._native as N  # noqa: E402

dev = torch.device("cuda:0")
try:
    PEAKS = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
except Exception:
    PEAKS = {}
HBM = float(PEAKS.get("hbm_gbs", 6650.0))
TF = float(PEAKS.get("bf16_tflops", 1590.0))


def timeit(fn, n=20, warm=3):
    """CUDA-event time per call.  The n calls are captured into one CUDA graph and replayed, so that what is
    measured is device time, not the Python / ctypes launch path (tens of microseconds per call, which hides
    kernels shorter than that); falls back to eager launches if the callable cannot be captured."""
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    graph = None
    if not os.environ.get("RORL_BENCH_EAGER"):
        try:
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph, capture_error_mode="thread_local"):
                for _ in range(n):
                    fn()
            graph.replay()
            torch.cuda.synchronize()
        except Exception:
            graph = None
            torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    if graph is not None:
        graph.replay()
    else:
        for _ in range(n):
            fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n * 1e-3


def rn(*s):
    return torch.randn(*s, device=dev)


RES = {}


def rec(name, t, nbytes=None, flops=None, note=""):
    r = {"us": t * 1e6}
    if nbytes:
        r.update(GBps=nbytes / t / 1e9, hbm_frac=nbytes / t / 1e9 / HBM, bytes=nbytes)
    if flops:
        r.update(TFLOPs=flops / t / 1e12, bf16_peak_frac=flops / t / 1e12 / TF, flops=flops)
    if note:
        r["note"] = note
    RES[name] = r
    print(name, json.dumps(r), flush=True)


def bench_gilr():
    B, L, C = 32, 1003, 256
    uv, uf, dh = rn(B, L, C), rn(B, L, C), rn(B, L, C)
    start = torch.zeros(B, L, device=dev); start[:, 0] = 1
    h = torch.empty_like(uv)
    du, df = torch.empty_like(uv), torch.empty_like(uv)
    rec("gilr_fused_fwd", timeit(lambda: N.call("rorl_gilr_fused_fwd", N.ptr(uv), N.ptr(uf), N.ptr(start), N.ptr(h), B, L, C, N.stream())),
        12 * B * L * C)
    rec("gilr_fused_bwd", timeit(lambda: N.call("rorl_gilr_fused_bwd", N.ptr(dh), N.ptr(uv), N.ptr(uf), N.ptr(h), N.ptr(start),
                                                N.ptr(du), N.ptr(df), B, L, C, N.stream())), 24 * B * L * C)
    # L2-cold variant: 8 rotating operand sets (8 x 98 MB > 126 MB L2)
    sets = [(rn(B, L, C), rn(B, L, C), torch.empty(B, L, C, device=dev)) for _ in range(8)]
    it = [0]

    def cold():
        a, b, c = sets[it[0] % 8]
        it[0] += 1
        N.call("rorl_gilr_fused_fwd", N.ptr(a), N.ptr(b), N.ptr(start), N.ptr(c), B, L, C, N.stream())
    rec("gilr_fused_fwd_L2cold", timeit(cold, n=24), 12 * B * L * C)


def bench_lru():
    B, L, C = 32, 1003, 256
    vr, vi, fr, fi = rn(B, L, C), rn(B, L, C), 0.9 * torch.rand(B, L, C, device=dev), 0.1 * rn(B, L, C)
    hr, hi = torch.empty_like(vr), torch.empty_like(vr)
    rec("lru_scan_fwd", timeit(lambda: N.call("rorl_lru_scan_fwd", N.ptr(vr), N.ptr(vi), N.ptr(fr), N.ptr(fi), None, None,
                                              N.ptr(hr), N.ptr(hi), B, L, C, N.stream())), 24 * B * L * C,
        note="per-step decay tensors as the reference materialises them: 6 x [B,L,C] floats")
    g1, g2 = rn(B, L, C), rn(B, L, C)
    o = [torch.empty_like(vr) for _ in range(4)]
    rec("lru_scan_bwd", timeit(lambda: N.call("rorl_lru_scan_bwd", N.ptr(g1), N.ptr(g2), N.ptr(fr), N.ptr(fi), N.ptr(hr), N.ptr(hi),
                                              None, None, None, N.ptr(o[0]), N.ptr(o[1]), N.ptr(o[2]), N.ptr(o[3]), B, L, C, N.stream())),
        40 * B * L * C)


def bench_lru_fused():
    B, L, C = 32, 1003, 256
    u_re, u_im = rn(B, L, C).requires_grad_(), rn(B, L, C).requires_grad_()
    lam_re, lam_im, gamma = (0.6 * torch.rand(C, device=dev)).requires_grad_(), (0.6 * torch.rand(C, device=dev)).requires_grad_(), (0.5 + torch.rand(C, device=dev)).requires_grad_()
    start = torch.zeros(B, L, device=dev); start[:, 0] = 1
    g1, g2 = rn(B, L, C), rn(B, L, C)
    with torch.no_grad():
        t_f = timeit(lambda: K.lru_fused_scan(u_re, u_im, lam_re, lam_im, gamma, start))
    t_fb = timeit(lambda: torch.autograd.grad(K.lru_fused_scan(u_re, u_im, lam_re, lam_im, gamma, start), (u_re, u_im, lam_re, lam_im, gamma), (g1, g2)), n=10)
    rec("lru_fused_fwd", t_f, 16 * B * L * C, note="lambda / gamma as [C] vectors, reset flags [B, L] (SURVEY.md 8d formula)")
    rec("lru_fused_bwd(+partial sums)", t_fb - t_f, 24 * B * L * C)


def bench_selscan():
    B, L, D, Ns = 32, 1019, 512, 32
    u, delta, z = rn(B, L, D).requires_grad_(), (0.5 * rn(B, L, D) - 1).requires_grad_(), rn(B, L, D).requires_grad_()
    Bm, Cm = rn(B, L, Ns).requires_grad_(), rn(B, L, Ns).requires_grad_()
    A = (-torch.exp(0.3 * rn(D, Ns))).requires_grad_()
    Dk, bias = rn(D).requires_grad_(), rn(D).requires_grad_()
    start = torch.zeros(B, L, device=dev); start[:, :19] = 1
    dy = rn(B, L, D)
    with torch.no_grad():
        t_fwd = timeit(lambda: K.selective_scan_tm(u, delta, A, Bm, Cm, Dk, z, bias, start, True))
    t_fwd_ck = timeit(lambda: K.selective_scan_tm(u, delta, A, Bm, Cm, Dk, z, bias, start, True), n=10)
    t_both = timeit(lambda: torch.autograd.grad(K.selective_scan_tm(u, delta, A, Bm, Cm, Dk, z, bias, start, True),
                                                (u, delta, A, Bm, Cm, Dk, z, bias), dy), n=10)
    bf = 4 * (4 * B * D * L + 2 * B * Ns * L + B * L)
    bb = 4 * (7 * B * D * L + 4 * B * Ns * L)
    rec("selscan_fwd", t_fwd, bf, note="MUFU floor ~115 us (App. F)")
    rec("selscan_fwd_ckpt", t_fwd_ck, bf)
    rec("selscan_bwd(+partial sums)", t_both - t_fwd_ck, bb)


def bench_conv():
    B, L, D, Kc = 32, 1019, 512, 16
    x, w, b = rn(B, L, D).requires_grad_(), rn(D, 1, Kc).requires_grad_(), rn(D).requires_grad_()
    mask = torch.ones(B, L, device=dev)
    dy = rn(B, L, D)
    with torch.no_grad():
        t_f = timeit(lambda: K.causal_conv1d_silu(x, w, b, mask))
    t_fb = timeit(lambda: torch.autograd.grad(K.causal_conv1d_silu(x, w, b, mask), (x, w, b), dy), n=10)
    rec("conv1d_silu_fwd", t_f, 8 * B * L * D)
    rec("conv1d_silu_bwd(+partials)", t_fb - t_f, 12 * B * L * D)


def bench_addnorm():
    rows, C = 32 * 1019, 256
    x, r, w, b = rn(rows, C).requires_grad_(), rn(rows, C).requires_grad_(), rn(C).requires_grad_(), rn(C).requires_grad_()
    dy = rn(rows, C)
    with torch.no_grad():
        t_f = timeit(lambda: K.layer_norm_fn(x, w, b, r, 1e-5, True))
    rec("addnorm_fwd", t_f, 16 * rows * C)
    t_fb = timeit(lambda: torch.autograd.grad(K.layer_norm_fn(x, w, b, r, 1e-5, True), (x, r, w, b), (dy, dy)), n=10)
    rec("addnorm_bwd", t_fb - t_f, 16 * rows * C)


def bench_gru():
    from rorl_b200.models.gru.gru import GRULayer
    B, L, H = 32, 1003, 256
    gi, w, bh = rn(B, L, 3 * H), 0.06 * rn(3 * H, H), rn(3 * H)
    out, hl, save = torch.empty(B, L, H, device=dev), torch.empty(B, H, device=dev), torch.empty(B, L, 4 * H, device=dev)
    t = timeit(lambda: N.call("rorl_gru_fwd", N.ptr(gi), N.ptr(w), N.ptr(bh), None, N.ptr(out), N.ptr(save), N.ptr(hl), B, L, H, N.stream()), n=10)
    rec("gru_fwd_persistent", t, note=f"{t / L * 1e6:.3f} us/step, {B} rows, H={H}")
    dout = rn(B, L, H)
    dgi, dghn, dh0 = torch.empty(B, L, 3 * H, device=dev), torch.empty(B, L, H, device=dev), torch.empty(B, H, device=dev)
    t = timeit(lambda: N.call("rorl_gru_bwd", N.ptr(dout), None, N.ptr(w), N.ptr(save), N.ptr(out), None, N.ptr(dgi), N.ptr(dghn),
                              N.ptr(dh0), B, L, H, N.stream()), n=10)
    rec("gru_bwd_persistent", t, note=f"{t / L * 1e6:.3f} us/step")
    ref = torch.nn.GRU(H, H, batch_first=True).to(dev)
    x = rn(B, L, H)
    with torch.no_grad():
        t = timeit(lambda: ref(x), n=10)
    rec("cudnn_gru_fwd(library, for scale)", t, note=f"{t / L * 1e6:.3f} us/step")
    mine = GRULayer(H, H).to(dev)
    xg = x.clone().requires_grad_()
    t = timeit(lambda: torch.autograd.grad(mine(xg)[0], [xg] + list(mine.parameters()), dout), n=10)
    rec("gru_layer_fwd+bwd(ours, incl. GEMMs)", t)
    xr = x.clone().requires_grad_()
    t = timeit(lambda: torch.autograd.grad(ref(xr)[0], [xr] + list(ref.parameters()), dout), n=10)
    rec("cudnn_gru_fwd+bwd(library, for scale)", t)


def bench_lstm():
    from rorl_b200.models.lstm.lstm import LSTMLayer
    B, L, H = 32, 1002, 256
    gi, w, bh = rn(B, L, 4 * H), 0.06 * rn(4 * H, H), rn(4 * H)
    out, hl, cl = torch.empty(B, L, H, device=dev), torch.empty(B, H, device=dev), torch.empty(B, H, device=dev)
    save = torch.empty(B, L, int(N.lib().rorl_lstm_save_floats_per_step(H)), device=dev)
    t = timeit(lambda: N.call("rorl_lstm_fwd", N.ptr(gi), N.ptr(w), N.ptr(bh), None, None, N.ptr(out), N.ptr(save), N.ptr(hl),
                              N.ptr(cl), B, L, H, N.stream()), n=10)
    rec("lstm_fwd_persistent", t, note=f"{t / L * 1e6:.3f} us/step, {B} rows, H={H}")
    dout = rn(B, L, H)
    dg, dh0, dc0 = torch.empty(B, L, 4 * H, device=dev), torch.empty(B, H, device=dev), torch.empty(B, H, device=dev)
    t = timeit(lambda: N.call("rorl_lstm_bwd", N.ptr(dout), None, None, N.ptr(w), N.ptr(save), None, N.ptr(dg), N.ptr(dh0),
                              N.ptr(dc0), B, L, H, N.stream()), n=10)
    rec("lstm_bwd_persistent", t, note=f"{t / L * 1e6:.3f} us/step")
    ref = torch.nn.LSTM(H, H, batch_first=True).to(dev)
    x = rn(B, L, H)
    with torch.no_grad():
        t = timeit(lambda: ref(x), n=10)
    rec("cudnn_lstm_fwd(library, for scale)", t, note=f"{t / L * 1e6:.3f} us/step")
    mine = LSTMLayer(H, H).to(dev)
    xg = x.clone().requires_grad_()
    t = timeit(lambda: torch.autograd.grad(mine(xg)[0], [xg] + list(mine.parameters()), dout), n=10)
    rec("lstm_layer_fwd+bwd(ours, incl. GEMMs)", t)
    xr = x.clone().requires_grad_()
    t = timeit(lambda: torch.autograd.grad(ref(xr)[0], [xr] + list(ref.parameters()), dout), n=10)
    rec("cudnn_lstm_fwd+bwd(library, for scale)", t)


def bench_gemm():
    M = 32 * 1019
    for (n, k, g, tag) in [(256, 256, 1, "fc 256x256"), (1024, 256, 1, "in_proj"), (256, 512, 1, "out_proj"), (256, 384, 8, "efc-8 L1 (shared x)"),
                           (256, 256, 8, "efc-8 L2")]:
        a = rn(M, k) if (g == 1 or k == 384) else rn(g, M, k)
        b = rn(n, k) if g == 1 else rn(g, n, k)
        bias = rn(n) if g == 1 else rn(g, n)
        for passes in (2, 4):
            t = timeit(lambda: K.gemm_tn(a, b, bias, 1, passes=passes))
            fl = 2.0 * M * n * k * g
            rec(f"gemm_tn {tag} passes={passes}", t, flops=fl * (3 if passes == 2 else 1), nbytes=4 * (a.numel() + b.numel() + M * n * g),
                note=f"useful fp32 TFLOP/s {fl / t / 1e12:.1f}")
    # weight gradient
    gq, xq = rn(M, 256), rn(M, 256)
    for passes in (2, 4):
        t = timeit(lambda: K.gemm_nt(gq, xq, passes=passes))
        rec(f"gemm_nt 256x256 R=32608 passes={passes}", t, flops=(3 if passes == 2 else 1) * 2.0 * M * 256 * 256, nbytes=4 * (gq.numel() + xq.numel()))
    g8, x8 = rn(8, M, 256), rn(8, M, 256)
    for passes in (2, 4):
        t = timeit(lambda: K.gemm_nt(x8, g8, passes=passes))
        rec(f"gemm_nt efc-8 L2 dW 8x[256x256] R=32608 passes={passes}", t, flops=(3 if passes == 2 else 1) * 2.0 * M * 256 * 256 * 8, nbytes=4 * (g8.numel() + x8.numel()))
    c = torch.empty(M, 256, device=dev)
    a2, w2 = rn(M, 256), rn(256, 256)
    t = timeit(lambda: torch.mm(a2, w2, out=c))
    rec("cublas sgemm 32608x256x256 (library, for scale)", t, flops=2.0 * M * 256 * 256)


def bench_reduce():
    M = 32 * 1019
    for shape in ((16, 32 * 1019 * 64), (4, 512 * 256), (32, 512 * 32)):
        x = rn(*shape)
        t = timeit(lambda: K.sum_leading(x))
        rec(f"sum_leading {list(shape)}", t, 4 * x.numel())
    for n, k in ((128, 9), (128, 6), (512, 16)):
        x, W, b = rn(M, k), rn(n, k), rn(n)
        out = torch.empty(M, n, device=dev)
        t = timeit(lambda: K.skinny_encoders([x], [W], [b]))
        rec(f"skinny_linear N={n} K={k}", t, 4 * M * (n + k))
    g6, W6 = rn(M, 128), rn(128, 6)
    t = timeit(lambda: K.skinny_dgrad(g6, W6))
    rec("skinny_dgrad N=128 K=6", t, 4 * M * (128 + 6))
    for n in (128, 256, 512, 1024):
        x = rn(M, n)
        t = timeit(lambda: K.colsum(x))
        rec(f"colsum [{M},{n}]", t, 4 * M * n)
        t = timeit(lambda: x.sum(0))
        rec(f"aten sum(0) [{M},{n}] (library, for scale)", t, 4 * M * n)
    dy, y = rn(8, M, 256), rn(8, M, 256)
    t = timeit(lambda: K.elu_bwd_colsum(dy, y))
    rec("elu_bwd_colsum [8,32608,256]", t, 12 * dy.numel())
    t = timeit(lambda: torch.ops.aten.elu_backward(dy, 1.0, 1.0, 1.0, True, y).sum(1))
    rec("aten elu_backward + sum (library, for scale)", t, 12 * dy.numel())
    for n, k in ((128, 9), (512, 16)):
        g, x = rn(M, n), rn(M, k)
        t = timeit(lambda: K.skinny_wgrad(g, x))
        rec(f"skinny_wgrad N={n} K={k}", t, 4 * M * (n + k))
        t = timeit(lambda: g.t() @ x)
        rec(f"cublas wgrad N={n} K={k} (library, for scale)", t, 4 * M * (n + k))


def bench_attn():
    """cgpt attention at the config-4 shape (32 rows, each a 1-token + a 1002-token sequence, 8 heads x 64) next to the
    kernel the reference calls on the same box: flash-attn 2's varlen kernel (FA2 `mma.sync` build for sm_100)."""
    import math
    import numpy as np
    H, hd, B = 8, 64, 32
    lens, starts, pos = [], [], 0
    for _ in range(B):
        for n in (1, 1002):
            starts.append(pos); lens.append(n); pos += n
    T = pos
    qkv = rn(T, 3, H, hd).requires_grad_()
    dout = rn(T, H * hd)
    slopes = torch.tensor([2 ** (-(i + 1)) for i in range(H)], dtype=torch.float32, device=dev)
    scale = 1.0 / math.sqrt(hd)
    tiles, gmap = (t.to(dev) for t in K.attention_tiles(starts, lens))
    fl_f = sum(4.0 * n * (n + 1) / 2 * hd for n in lens) * H          # causal QK^T + PV
    with torch.no_grad():
        t_f = timeit(lambda: K.attn_varlen_alibi(qkv, tiles, gmap, slopes, scale))
    t_fb = timeit(lambda: torch.autograd.grad(K.attn_varlen_alibi(qkv, tiles, gmap, slopes, scale), qkv, dout), n=10)
    rec("attn_fwd (ours: prep + tcgen05 kernel, fp32 in/out)", t_f, flops=fl_f)
    rec("attn_fwd+bwd (ours)", t_fb, flops=3.5 * fl_f)
    try:
        import flash_attn as fa
        cu = torch.tensor(np.concatenate(([0], np.cumsum(lens))), dtype=torch.int32, device=dev)
        a = qkv.detach().to(torch.bfloat16).requires_grad_()
        do16 = dout.view(T, H, hd).to(torch.bfloat16)
        with torch.no_grad():
            t_f = timeit(lambda: fa.flash_attn_varlen_qkvpacked_func(a, cu, max(lens), 0.0, softmax_scale=scale, causal=True, alibi_slopes=slopes))
        t_fb = timeit(lambda: torch.autograd.grad(fa.flash_attn_varlen_qkvpacked_func(a, cu, max(lens), 0.0, softmax_scale=scale, causal=True,
                                                                                      alibi_slopes=slopes), a, do16), n=10)
        rec("flash-attn 2 varlen fwd (library, same box, bf16 in/out)", t_f, flops=fl_f, note=f"flash_attn {fa.__version__}")
        rec("flash-attn 2 varlen fwd+bwd (library, same box)", t_fb, flops=3.5 * fl_f)
        # like for like with the reference's call site: the fp32 -> bf16 casts autocast inserts around the kernel
        q32 = qkv.detach().clone().requires_grad_()
        t_fb = timeit(lambda: torch.autograd.grad(fa.flash_attn_varlen_qkvpacked_func(q32.to(torch.bfloat16), cu, max(lens), 0.0, softmax_scale=scale,
                                                  causal=True, alibi_slopes=slopes).float(), q32, dout.view(T, H, hd)), n=10)
        rec("flash-attn 2 varlen fwd+bwd incl. fp32<->bf16 casts (library, same box)", t_fb, flops=3.5 * fl_f)
    except Exception as e:  # pragma: no cover
        print("flash-attn unavailable:", e)


def attn_flops(lens, H, hd):
    """Algorithmic FLOPs of causal attention over sequences `lens`: Q K^T and P V, 2 * hd each per (query, key <= query)
    pair.  The backward's five products are counted as 2.5 forwards (forward + backward = 3.5x)."""
    return sum(4.0 * n * (n + 1) / 2 * hd for n in lens) * H


def bench_attn_hd():
    """cgpt attention at other head dimensions (32 sequences x 1001 tokens; width / heads = hd), next to flash-attn 2's
    varlen kernel on the same inputs when it imports.  hd <= 64 runs on operands padded to 64, hd > 64 on 128; the
    FLOP/s below count the real hd only."""
    import math
    import numpy as np
    lens = [1001] * 32
    starts = [1001 * i for i in range(32)]
    T = sum(lens)
    tiles, gmap = (t.to(dev) for t in K.attention_tiles(starts, lens))
    try:
        import flash_attn as fa
    except Exception as e:  # pragma: no cover
        fa = None
        print("flash-attn unavailable:", e)
    cu = torch.tensor(np.concatenate(([0], np.cumsum(lens))), dtype=torch.int32, device=dev)
    for width, H in ((256, 8), (512, 8), (512, 4), (1024, 8)):
        hd = width // H
        qkv = rn(T, 3, H, hd).requires_grad_()
        dout = rn(T, H * hd)
        slopes = torch.tensor([2 ** (-(i + 1)) for i in range(H)], dtype=torch.float32, device=dev)
        scale = 1.0 / math.sqrt(hd)
        fl_f = attn_flops(lens, H, hd)
        tag = f"C={width} H={H} hd={hd}"
        with torch.no_grad():
            t_f = timeit(lambda: K.attn_varlen_alibi(qkv, tiles, gmap, slopes, scale))
        t_fb = timeit(lambda: torch.autograd.grad(K.attn_varlen_alibi(qkv, tiles, gmap, slopes, scale), qkv, dout), n=10)
        rec(f"attn_fwd {tag} (ours: prep + tcgen05 kernel, fp32 in/out)", t_f, flops=fl_f)
        rec(f"attn_fwd+bwd {tag} (ours)", t_fb, flops=3.5 * fl_f)
        if fa is not None:
            a = qkv.detach().to(torch.bfloat16).requires_grad_()
            do16 = dout.view(T, H, hd).to(torch.bfloat16)
            call = lambda: fa.flash_attn_varlen_qkvpacked_func(a, cu, max(lens), 0.0, softmax_scale=scale, causal=True, alibi_slopes=slopes)
            with torch.no_grad():
                t_f = timeit(call)
            t_fb = timeit(lambda: torch.autograd.grad(call(), a, do16), n=10)
            rec(f"flash-attn 2 varlen fwd {tag} (library, same box, bf16 in/out)", t_f, flops=fl_f, note=f"flash_attn {fa.__version__}")
            rec(f"flash-attn 2 varlen fwd+bwd {tag} (library, same box)", t_fb, flops=3.5 * fl_f)
        del qkv, dout


def bench_refs():
    """The reference's own in-tree Triton scans (K6 / K7) on the same box, imported UNMODIFIED from oracle/_ref
    (ref: gilr/scan_triton/real_rnn_tie_input_gate.py:170-264, lru/scan_triton/complex_rnn.py:174-244)."""
    sys.path.insert(0, ROOT)
    from oracle import refload
    if not refload.available():
        print("reference not staged (oracle/make_ref.py)")
        return
    refload.load_reference()
    B, L, C = 32, 1003, 256
    try:
        from offpolicy_rnn.models.gilr.scan_triton.real_rnn_tie_input_gate import real_scan_tie_input_gate
        v, f = rn(B, L, C).requires_grad_(), torch.sigmoid(rn(B, L, C)).requires_grad_()
        dh = rn(B, L, C)
        with torch.no_grad():
            t_f = timeit(lambda: real_scan_tie_input_gate(v, f), n=10)
        rec("reference Triton gilr scan fwd (K6, same box)", t_f, 12 * B * L * C)
        # the reference's backward overwrites its saved tensors in place, so time forward + backward together
        t_fb = timeit(lambda: torch.autograd.grad(real_scan_tie_input_gate(v.clone(), f.clone()), (v, f), dh, allow_unused=True), n=10)
        rec("reference Triton gilr scan fwd+bwd incl. 2 clones (K6, same box)", t_fb, 36 * B * L * C + 16 * B * L * C)
    except Exception as e:
        print("reference gilr Triton scan failed:", repr(e))
    try:
        from offpolicy_rnn.models.lru.scan_triton.complex_rnn import complex_scan
        vr, vi = rn(B, L, C).requires_grad_(), rn(B, L, C).requires_grad_()
        fr, fi = (0.9 * torch.rand(B, L, C, device=dev)).requires_grad_(), (0.1 * rn(B, L, C)).requires_grad_()
        h0r, h0i = torch.zeros(B, 1, C, device=dev), torch.zeros(B, 1, C, device=dev)
        gd = torch.zeros(B, L, 1, device=dev)
        g1, g2 = rn(B, L, C), rn(B, L, C)
        with torch.no_grad():
            t_f = timeit(lambda: complex_scan(vr, vi, fr, fi, h0r, h0i, gd), n=10)
        rec("reference Triton lru scan fwd (K7, same box)", t_f, 24 * B * L * C)
        t_fb = timeit(lambda: torch.autograd.grad(complex_scan(vr.clone(), vi.clone(), fr.clone(), fi.clone(), h0r, h0i, gd), (vr, vi, fr, fi), (g1, g2),
                                                  allow_unused=True), n=10)
        rec("reference Triton lru scan fwd+bwd incl. 4 clones (K7, same box)", t_fb, (24 + 40 + 32) * B * L * C)
    except Exception as e:
        print("reference lru Triton scan failed:", repr(e))


ALL = {"attn": bench_attn, "attn_hd": bench_attn_hd, "refs": bench_refs, "reduce": bench_reduce, "gilr": bench_gilr, "lru": bench_lru, "lru_fused": bench_lru_fused, "selscan": bench_selscan, "conv": bench_conv, "addnorm": bench_addnorm,
       "gru": bench_gru, "lstm": bench_lstm, "gemm": bench_gemm}

if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--only", default="")
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    names = [n for n in a.only.split(",") if n] or list(ALL)
    for n in names:
        ALL[n]()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        json.dump({"peaks": {"hbm_gbs": HBM, "bf16_tflops": TF}, "kernels": RES}, open(a.out, "w"), indent=1)
