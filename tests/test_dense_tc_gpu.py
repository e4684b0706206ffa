"""K8 on tcgen05 (csrc/dense_tc.cuh): bns_dense_tn_3xtf32 / bns_dense_nt_3xtf32 against an f64 torch reference.

Tolerance: 2e-5 of max|C| (cuBLAS fp32 itself sits at ~2e-6 on these shapes; one TF32 pass would be ~5e-4)."""
import pytest
import torch

pytestmark = pytest.mark.gpu

TOL = 2e-5


def _rel(got, ref):
    return ((got.double() - ref).abs().max() / ref.abs().max().clamp_min(1e-30)).item()


@pytest.fixture(scope="module")
def dense(built):
    from bns_gcn_b200.module import dense as d
    return d


@pytest.mark.parametrize("M,N,K,bias", [(128, 128, 32, False), (1, 4, 4, True), (300, 136, 100, True), (1000, 256, 1204, True),
                                        (4099, 44, 256, False), (20000, 256, 512, True)])
def test_tn_matches_f64(dense, M, N, K, bias):
    g = torch.Generator().manual_seed(M + N + K)
    a, b = torch.randn(M, K, generator=g).cuda(), torch.randn(N, K, generator=g).cuda()
    bi = torch.randn(N, generator=g).cuda() if bias else None
    got = dense.tc_mm_tn(a, b, bi)
    ref = a.double() @ b.double().t() + (bi.double() if bias else 0)
    assert _rel(got, ref) < TOL


@pytest.mark.parametrize("R,N1,N2", [(32, 128, 128), (7, 4, 8), (1000, 136, 100), (5000, 256, 1204), (150000, 256, 256)])
def test_nt_matches_f64_and_is_deterministic(dense, R, N1, N2):
    g = torch.Generator().manual_seed(R + N1 + N2)
    a, b = torch.randn(R, N1, generator=g).cuda(), torch.randn(R, N2, generator=g).cuda()
    got = dense.tc_mm_nt(a, b)
    ref = a.double().t() @ b.double()
    assert _rel(got, ref) < TOL
    assert torch.equal(got, dense.tc_mm_nt(a, b)), "split-K combine must be deterministic"


def test_strided_rows_and_onehot_are_exact(dense):
    """Leading dimensions larger than the row (views into wider buffers) and an exactness check: one-hot A picks
    integer-coded B entries, any layout / descriptor slip shows up as a wrong integer."""
    buf = torch.zeros(256, 96, device="cuda")
    a = buf[:, 8:72]                                              # [256, 64], ld 96, 32-byte offset
    a[torch.arange(256), torch.arange(256) % 64] = 1.0
    b = (torch.arange(200, device="cuda", dtype=torch.float32)[:, None] * 1000 + torch.arange(64, device="cuda")[None, :])
    got = dense.tc_mm_tn(a, b)
    assert torch.equal(got, (a.double() @ b.double().t()).float())
    at = torch.zeros(96, 136, device="cuda")
    at[torch.arange(136) % 96, torch.arange(136)] = 1.0
    bt = (torch.arange(96, device="cuda", dtype=torch.float32)[:, None] * 1000 + torch.arange(60, device="cuda")[None, :])
    assert torch.equal(dense.tc_mm_nt(at, bt), (at.double().t() @ bt.double()).float())


def test_linear_autograd_matches_f64_and_pads_odd_widths(dense):
    """`linear()` runs on the tcgen05 kernels (not the cuBLAS fallback): forward, dX, dW, db against f64 -- including
    41 output columns (padded to 44)."""
    from bns_gcn_b200._lib import lib
    for n_out in (64, 41):
        g = torch.Generator().manual_seed(n_out)
        x = torch.randn(3000, 256, generator=g).cuda().requires_grad_()
        w = (torch.randn(n_out, 256, generator=g) / 16).cuda().requires_grad_()
        b = torch.randn(n_out, generator=g).cuda().requires_grad_()
        dy = torch.randn(3000, n_out, generator=g).cuda()
        launches = lib.bns_launch_count()
        y = dense.linear(x, w, b)
        assert lib.bns_launch_count() > launches, "linear() did not reach the tcgen05 kernels"
        assert y.shape == (3000, n_out)
        y.backward(dy)
        xd, wd, bd, dyd = x.detach().double(), w.detach().double(), b.detach().double(), dy.double()
        assert _rel(y.detach(), xd @ wd.t() + bd) < TOL
        assert _rel(x.grad, dyd @ wd) < TOL
        assert _rel(w.grad, dyd.t() @ xd) < TOL
        assert _rel(b.grad, dyd.sum(0)) < 1e-5


def test_rejects_unaligned_operands(dense):
    from bns_gcn_b200._lib import BnsError
    a = torch.randn(64, 30, device="cuda")          # 120-byte rows: TMA cannot address them
    b = torch.randn(16, 30, device="cuda")
    with pytest.raises(BnsError):
        dense.tc_mm_tn(a, b)
    y = dense.linear(a, b)                          # linear() falls back to the library GEMM instead
    assert _rel(y, a.double() @ b.double().t()) < 1e-5


def test_fused_addend_and_colsum(dense):
    g = torch.Generator().manual_seed(7)
    x = torch.randn(2500, 128, generator=g).cuda().requires_grad_()
    w = (torch.randn(41, 128, generator=g) / 11).cuda().requires_grad_()
    b = torch.randn(41, generator=g).cuda().requires_grad_()
    add = torch.randn(2500, 44, generator=g).cuda().requires_grad_()      # padded width: fused into the epilogue
    dy = torch.randn(2500, 41, generator=g).cuda()
    y = dense.linear(x, w, b, addend=add)
    y.backward(dy)
    ref = x.detach().double() @ w.detach().double().t() + b.detach().double() + add.detach().double()[:, :41]
    assert _rel(y.detach(), ref) < TOL
    assert torch.equal(add.grad[:, :41], dy) and float(add.grad[:, 41:].abs().max()) == 0.0
    assert _rel(b.grad, dy.double().sum(0)) < 1e-5
    # unfusable width (40 columns for 41 outputs): same result through the plain add
    add2 = torch.randn(2500, 41, generator=g).cuda()
    y2 = dense.linear(x.detach(), w.detach(), b.detach(), addend=add2)
    assert _rel(y2, x.detach().double() @ w.detach().double().t() + b.detach().double() + add2.double()) < TOL
    big = torch.randn(100000, 256, generator=g).cuda()
    s1, s2 = dense.colsum(big), dense.colsum(big)
    assert torch.equal(s1, s2)
    assert _rel(s1, big.double().sum(0)) < 1e-5
