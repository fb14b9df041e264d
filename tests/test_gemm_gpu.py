"""tcgen05 GEMM (two-term bf16 split, passes = 2; its hi * hi term alone, passes = 4) vs float64 matmul.  The split keeps
16 mantissa bits per operand: ~2^-17 relative per product, 30x inside the 1e-3 parity budget.  K only has to be a
multiple of 4: shapes with K % 8 == 4 exercise the padded rows of B's split copy."""
import pytest
import torch

from helpers import rel_err

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def K():
    import rorl_b200.kernels as K
    return K


def test_linear_and_ensemble_autograd(K):
    g = torch.Generator(device="cuda").manual_seed(9)
    B_, L, Kin, Nout, E = 4, 300, 384, 256, 8
    x = torch.randn(B_, L, Kin, device="cuda", generator=g, requires_grad=True)
    W = (0.1 * torch.randn(Nout, Kin, device="cuda", generator=g)).requires_grad_()
    b = torch.randn(Nout, device="cuda", generator=g).requires_grad_()
    dy = torch.randn(B_, L, Nout, device="cuda", generator=g)
    y = K.linear(x, W, b, elu=True)
    got = torch.autograd.grad(y, (x, W, b), dy)
    xd, Wd, bd = (t.detach().double().requires_grad_() for t in (x, W, b))
    yr = torch.nn.functional.elu(torch.nn.functional.linear(xd, Wd, bd))
    ref = torch.autograd.grad(yr, (xd, Wd, bd), dy.double())
    assert rel_err(y, yr) < 3e-5
    for a, r, n in zip(got, ref, "x W b".split()):
        assert rel_err(a, r) < 1e-4, n
    # ensemble, shared input then per-member input
    We = (0.1 * torch.randn(E, Kin, Nout, device="cuda", generator=g)).requires_grad_()
    be = torch.randn(E, 1, Nout, device="cuda", generator=g).requires_grad_()
    y1 = K.ensemble_linear(x, We, be, True, True)
    dy1 = torch.randn_like(y1)
    got = torch.autograd.grad(y1, (x, We, be), dy1)
    xd, Wd, bd = (t.detach().double().requires_grad_() for t in (x, We, be))
    yr = torch.nn.functional.elu(torch.einsum('cij,bjk->bcik', xd, Wd) + bd.unsqueeze(1))
    ref = torch.autograd.grad(yr, (xd, Wd, bd), dy1.double())
    assert rel_err(y1, yr) < 3e-5
    for a, r, n in zip(got, ref, "x W b".split()):
        assert rel_err(a, r) < 1e-4, n
    h = torch.randn(E, B_, L, Kin, device="cuda", generator=g, requires_grad=True)
    y2 = K.ensemble_linear(h, We, be, False, False)
    dy2 = torch.randn_like(y2)
    got = torch.autograd.grad(y2, (h, We, be), dy2)
    hd = h.detach().double().requires_grad_()
    yr = torch.einsum('cbij,cjk->cbik', hd, Wd) + bd.unsqueeze(1)
    ref = torch.autograd.grad(yr, (hd, Wd, bd), dy2.double())
    assert rel_err(y2, yr) < 3e-5
    for a, r, n in zip(got, ref, "h W b".split()):
        assert rel_err(a, r) < 1e-4, n


@pytest.mark.parametrize("R,M,N,G", [(128, 128, 128, 1), (1000, 80, 512, 1), (32576, 256, 384, 1), (5000, 384, 256, 8), (333, 12, 260, 2)])
@pytest.mark.parametrize("passes", [2, 4])
def test_gemm_nt_weight_gradient_form(K, R, M, N, G, passes):
    """passes = 4 is checked against the product of the bf16-rounded operands (what its single MMA computes)."""
    g = torch.Generator(device="cuda").manual_seed(R + M)
    A = torch.randn((G, R, M) if G > 1 else (R, M), device="cuda", generator=g)
    B = torch.randn((G, R, N) if G > 1 else (R, N), device="cuda", generator=g)
    r = (lambda t: t.double()) if passes == 2 else (lambda t: t.to(torch.bfloat16).double())
    D = K.gemm_nt(A, B, passes=passes)
    ref = r(A).transpose(-1, -2) @ r(B)
    e = rel_err(D, ref)
    print(f"NT R={R} M={M} N={N} G={G}: passes={passes} err {e:.2e}")
    assert e < 5e-5
    if G > 1:       # shared A (first efc layer: one input, E output gradients)
        D2 = K.gemm_nt(A[0], B, passes=passes)
        assert rel_err(D2, r(A[0]).t() @ r(B)) < 5e-5


@pytest.mark.parametrize("M,N,K_", [(128, 128, 32), (300, 12, 256), (1000, 80, 512), (32608, 256, 384), (4097, 1024, 256),
                                     (77, 132, 36), (513, 260, 64), (2000, 200, 96), (129, 2048, 384), (255, 256, 40),
                                     (32576, 256, 384), (32608, 256, 36), (1000, 80, 36), (300, 260, 44), (4097, 1024, 100),
                                     (129, 2048, 36), (513, 132, 12), (2000, 12, 68), (64, 4, 20)])
def test_gemm_tn_bf16_split(K, M, N, K_):
    """passes = 2: two-term bf16 split (hi*hi + hi*lo + lo*hi on kind::f16).  Error ~2^-17 relative per product,
    measured against float64; tolerance 3e-5 of max|D| (30x inside the 1e-3 parity budget)."""
    g = torch.Generator(device="cuda").manual_seed(M + N + 7)
    A = torch.randn(M, K_, device="cuda", generator=g)
    B = torch.randn(N, K_, device="cuda", generator=g)
    bias = torch.randn(N, device="cuda", generator=g)
    ref = A.double() @ B.double().t() + bias.double()
    D = K.gemm_tn(A, B, bias, passes=2)
    e = rel_err(D, ref)
    print(f"M={M} N={N} K={K_}: bf16x3 err {e:.2e}")
    assert e < 3e-5
    Delu = K.gemm_tn(A, B, bias, act=1, passes=2)
    assert rel_err(Delu, torch.nn.functional.elu(ref)) < 3e-5


def test_gemm_tn_bf16_split_batched(K):
    g = torch.Generator(device="cuda").manual_seed(6)
    E, M, N, K_ = 8, 1500, 256, 384
    big = torch.randn(M, 2 * K_, device="cuda", generator=g)
    A = big[:, K_:]
    W = torch.randn(E, N, K_, device="cuda", generator=g)
    b = torch.randn(E, N, device="cuda", generator=g)
    D = K.gemm_tn(A, W, b, passes=2)                  # shared, row-strided A; batched B
    ref = torch.einsum('mk,enk->emn', A.double(), W.double()) + b.double()[:, None]
    assert rel_err(D, ref) < 3e-5
    Ab = torch.randn(E, M, K_, device="cuda", generator=g)
    D2 = K.gemm_tn(Ab, W, b, act=1, passes=2)         # per-member A, ELU
    ref2 = torch.nn.functional.elu(torch.einsum('emk,enk->emn', Ab.double(), W.double()) + b.double()[:, None])
    assert rel_err(D2, ref2) < 3e-5
    D3 = K.gemm_tn(Ab, W, reduce_g=True, passes=2)    # sum over members: one K = 8 * 384 reduction
    ref3 = torch.einsum('emk,enk->mn', Ab.double(), W.double())
    assert rel_err(D3, ref3) < 1e-4
    A4, W4 = Ab[:3, :, :36].contiguous(), W[:3, :, :36].contiguous()      # K % 8 == 4: padded split-copy rows per member
    D4 = K.gemm_tn(A4, W4, reduce_g=True, passes=2)
    assert rel_err(D4, torch.einsum('emk,enk->mn', A4.double(), W4.double())) < 1e-4


@pytest.mark.parametrize("M,N,K_,G", [(1000, 512, 256, 1), (700, 16, 512, 1), (300, 80, 512, 1), (1500, 256, 384, 8), (129, 36, 40, 3),
                                     (129, 36, 44, 3), (700, 132, 36, 1)])
def test_gemm_tn_transposed_weights(K, M, N, K_, G):
    """transb: B handed over as [K, N] (nn.Linear's weight for its input-gradient GEMM, EnsembleLinear's [E, in, out]
    weight for its forward); the kernel's pre-split pass transposes it -- no transposed copy is made by the caller."""
    g = torch.Generator(device="cuda").manual_seed(M + N)
    A = torch.randn(M, K_, device="cuda", generator=g)
    if G == 1:
        Bt = torch.randn(K_, N, device="cuda", generator=g)
        ref = A.double() @ Bt.double()
    else:
        Bt = torch.randn(G, K_, N, device="cuda", generator=g)
        ref = torch.einsum('mk,gkn->gmn', A.double(), Bt.double())
    D = K.gemm_tn(A, Bt, passes=2, transb=True)
    assert D.shape == ref.shape
    assert rel_err(D, ref) < 3e-5


@pytest.mark.parametrize("M,N,K_", [(1000, 512, 256), (32608, 1536, 512), (300, 80, 64), (1000, 520, 36)])
def test_gemm_bf16_single_pass(K, M, N, K_):
    """passes = 4: the hi * hi term alone (one bf16 MMA per k-step), for the layers the reference runs under bf16 autocast.
    Checked against the product of the bf16-ROUNDED operands in float64 (exact up to fp32 accumulation), forward, the
    transposed-weight form and the weight-gradient form."""
    g = torch.Generator(device="cuda").manual_seed(M + K_)
    A = torch.randn(M, K_, device="cuda", generator=g)
    B = torch.randn(N, K_, device="cuda", generator=g)
    bias = torch.randn(N, device="cuda", generator=g)
    r = lambda t: t.to(torch.bfloat16).double()
    ref = r(A) @ r(B).t() + bias.double()
    assert rel_err(K.gemm_tn(A, B, bias, passes=4), ref) < 2e-5
    assert rel_err(K.gemm_tn(A, B.t().contiguous(), bias, passes=4, transb=True), ref) < 2e-5
    G_ = torch.randn(M, N, device="cuda", generator=g)
    assert rel_err(K.gemm_nt(G_, A, passes=4), r(G_).t() @ r(A)) < 2e-5


@pytest.mark.parametrize("Kh,M", [(256, 1000), (128, 37), (384, 513), (512, 130)])
def test_ensemble_hidden_to_scalar(K, Kh, M):
    """Fused `efc (ELU) -> efc (out 1)` tail of the ensemble-Q head vs the same two layers in float64."""
    g = torch.Generator(device="cuda").manual_seed(Kh + M)
    E, Kin = 8, 96
    x = torch.randn(E, 3, M, Kin, device="cuda", generator=g, requires_grad=True)
    W2 = (0.2 * torch.randn(E, Kin, Kh, device="cuda", generator=g)).requires_grad_()
    b2 = torch.randn(E, 1, Kh, device="cuda", generator=g).requires_grad_()
    W3 = (0.2 * torch.randn(E, Kh, 1, device="cuda", generator=g)).requires_grad_()
    b3 = torch.randn(E, 1, 1, device="cuda", generator=g).requires_grad_()
    assert K.ensemble_hidden_to_scalar_ok(x, W2, W3)
    q = K.EnsembleHiddenToScalar.apply(x, W2, b2, W3, b3)
    dq = torch.randn_like(q)
    got = torch.autograd.grad(q, (x, W2, b2, W3, b3), dq)
    xd, W2d, b2d, W3d, b3d = (t.detach().double().requires_grad_() for t in (x, W2, b2, W3, b3))
    y = torch.nn.functional.elu(torch.einsum('ebmi,eik->ebmk', xd, W2d) + b2d.unsqueeze(1))
    qr = torch.einsum('ebmk,eko->ebmo', y, W3d) + b3d.unsqueeze(1)
    ref = torch.autograd.grad(qr, (xd, W2d, b2d, W3d, b3d), dq.double())
    assert q.shape == qr.shape
    assert rel_err(q, qr) < 3e-5
    for a, r, n in zip(got, ref, "x W2 b2 W3 b3".split()):
        assert a.shape == r.shape, n
        assert rel_err(a, r) < 1e-4, n


@pytest.mark.parametrize("M,N,K_", [(1000, 2048, 512), (32608, 2048, 512), (77, 132, 40), (300, 260, 36)])
def test_linear_gelu_fused(K, M, N, K_):
    """gelu(x W^T + b) with the exact (erf) GELU in the GEMM epilogue and its backward fused with the bias gradient
    (rorl_gelu_bwd_colsum), against torch in float64: output, dx, dW, db."""
    g = torch.Generator(device="cuda").manual_seed(M + N)
    x = torch.randn(M, K_, device="cuda", generator=g, requires_grad=True)
    W = (torch.randn(N, K_, device="cuda", generator=g) / K_ ** 0.5).requires_grad_()
    b = torch.randn(N, device="cuda", generator=g, requires_grad=True)
    assert K.linear_gelu_ok(x, W)
    y = K.linear_gelu(x, W, b)
    dy = torch.randn(M, N, device="cuda", generator=g)
    got = torch.autograd.grad(y, (x, W, b), dy)
    xd, Wd, bd = (t.detach().double().requires_grad_() for t in (x, W, b))
    yr = torch.nn.functional.gelu(torch.nn.functional.linear(xd, Wd, bd))
    ref = torch.autograd.grad(yr, (xd, Wd, bd), dy.double())
    assert rel_err(y, yr) < 3e-5
    for a, r, n in zip(got, ref, ("dx", "dW", "db")):
        assert rel_err(a, r) < 1e-4, (n, rel_err(a, r))
    with torch.no_grad():
        assert rel_err(K.linear_gelu(x, W, b), yr) < 3e-5


@pytest.mark.parametrize("K_", [36, 64])
def test_gemm_tn_accumulate(K, K_):
    """accumulate=True: out += A B^T in the GEMM epilogue, into a column block of a wider buffer (as SSMCore's backward adds
    x_proj's input gradient onto the scan's du), at 128- and 256-column tiles, plain and with transposed weights; the
    columns outside the block stay untouched."""
    g = torch.Generator(device="cuda").manual_seed(K_)
    M = 1000
    for N, transb in ((260, False), (100, True)):
        A = torch.randn(M, K_, device="cuda", generator=g)
        B = torch.randn((K_, N) if transb else (N, K_), device="cuda", generator=g)
        buf = torch.randn(M, N + 8, device="cuda", generator=g)
        base = buf.clone()
        K.gemm_tn(A, B, transb=transb, out=buf[:, 4:N + 4], accumulate=True)
        prod = A.double() @ (B.double() if transb else B.double().t())
        assert rel_err(buf[:, 4:N + 4], base[:, 4:N + 4].double() + prod) < 3e-5
        assert torch.equal(buf[:, :4], base[:, :4]) and torch.equal(buf[:, N + 4:], base[:, N + 4:])


def test_weight_split_cache_contract(K):
    """kernels.WeightSplitCache: B operands that are views into a registered arena get a persistent bf16 hi | lo copy,
    rebuilt by refresh() (one launch for the whole arena); GEMMs between two refreshes read that copy -- so a weight change
    becomes visible at the next refresh, which is why the update engine refreshes after every optimizer step -- and
    operands outside the arena are never cached."""
    g = torch.Generator(device="cuda").manual_seed(11)
    n0, n1 = 512 * 256, 512 * 256 + 8 * 256 * 384
    arena = torch.randn(n1 + 260 * 36, device="cuda", generator=g)
    W = arena[:n0].view(512, 256)                              # nn.Linear layout [N, K]
    We = arena[n0:n1].view(8, 256, 384)                        # EnsembleLinear layout [E, in, out] -> transb
    Wk = arena[n1:].view(260, 36)                              # K % 8 == 4: the kept copy has padded rows
    A = torch.randn(1000, 256, device="cuda", generator=g)
    cache = K.WeightSplitCache(torch.device("cuda", 0))
    owner = cache.add_owner(arena)
    ref = lambda: (A.double() @ W.double().t(), torch.einsum('mk,ekn->emn', A.double(), We.double()),
                   A[:, :36].double() @ Wk.double().t())
    with cache.active():
        y0, e0, k0 = K.gemm_tn(A, W[:256]), K.gemm_tn(A, We, transb=True), K.gemm_tn(A[:, :36], Wk)   # first sighting:
        assert len(cache.entries) == 3                                          # own pre-split, entries recorded
        cache.refresh(owner)
        y1, e1, k1 = K.gemm_tn(A, W[:256]), K.gemm_tn(A, We, transb=True), K.gemm_tn(A[:, :36], Wk)   # from the cache
        assert torch.equal(y0, y1) and torch.equal(e0, e1) and torch.equal(k0, k1)
        r = ref()
        assert rel_err(y1, r[0][:, :256]) < 3e-5 and rel_err(e1, r[1]) < 3e-5 and rel_err(k1, r[2]) < 3e-5
        old = ref()
        arena.mul_(-0.5)                                                        # the weights change ...
        y2 = K.gemm_tn(A, W[:256])
        assert rel_err(y2, old[0][:, :256]) < 3e-5                               # ... the kept copy does not, until
        cache.refresh(owner)                                                    # the owner says so
        r = ref()
        assert rel_err(K.gemm_tn(A, W[:256]), r[0][:, :256]) < 3e-5
        assert rel_err(K.gemm_tn(A, We, transb=True), r[1]) < 3e-5
        assert rel_err(K.gemm_tn(A[:, :36], Wk), r[2]) < 3e-5
        cache.invalidate(owner)
        arena.mul_(2.0)
        assert rel_err(K.gemm_tn(A, W[:256]), ref()[0][:, :256]) < 3e-5         # invalidated: per-call pre-split again
        other = torch.randn(128, 256, device="cuda", generator=g)
        K.gemm_tn(A, other)
        assert len(cache.entries) == 3                                          # not in a registered arena: never cached
    assert K._ACTIVE_SPLIT_CACHE is None
