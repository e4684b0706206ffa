"""GPU parity of every C-ABI compute entry point against the oracle (oracle/spmm_ref.c, oracle/philox.py,
torch CPU fp32), on seeded inputs the oracle finishes in seconds.  Tolerances: index / integer work is
bit-exact; f32 sums 1e-5 relative (north_star allows 1e-4 on layer outputs)."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

RTOL = 1e-5


def _rand_csr(n_rows, n_cols, avg_deg, seed, heavy=0, empty_frac=0.1):
    g = torch.Generator().manual_seed(seed)
    deg = torch.poisson(torch.full((n_rows,), float(avg_deg)), generator=g).long()
    deg[torch.rand(n_rows, generator=g) < empty_frac] = 0
    for i in range(heavy):                       # rows far longer than one chunk
        deg[(i * 7919) % n_rows] = 3000 + 1700 * i
    deg.clamp_(max=n_cols * 4)
    indptr = torch.zeros(n_rows + 1, dtype=torch.int64)
    indptr[1:] = deg.cumsum(0)
    nnz = int(indptr[-1])
    idx = torch.randint(0, n_cols, (nnz,), generator=g, dtype=torch.int64)
    return indptr, idx


def _ref_spmm(indptr, idx, x, row_scale=None, col_scale=None, col_map=None, n_direct=None, row_map=None,
              n_out=None, y0=None):
    """Oracle: C SpMM on the (mapped, filtered) edge list, scalings applied the way the reference does."""
    from oracle import bns_oracle as O
    n_rows = indptr.numel() - 1
    rows = torch.repeat_interleave(torch.arange(n_rows), indptr[1:] - indptr[:-1])
    cols = idx.clone()
    xrow = cols.clone()
    if col_map is not None:
        m = cols >= n_direct
        xrow[m] = col_map[cols[m] - n_direct].long()
    keep = xrow >= 0
    orow = rows.clone()
    if row_map is not None:
        orow = row_map[rows].long()
        keep &= orow >= 0
    n_out = n_out if n_out is not None else n_rows
    # scale sources per EDGE (col_scale is indexed by the original column id)
    if col_scale is not None:
        contrib = x[xrow[keep]] * col_scale[cols[keep]].unsqueeze(1)
        out = torch.zeros(n_out, x.shape[1]).index_add_(0, orow[keep], contrib)
    else:
        g = O.EdgeList(xrow[keep], orow[keep], x.shape[0], n_out)
        out = O.CopyUSum.apply(g, x)
    if row_scale is not None:
        rs = torch.zeros(n_out)
        if row_map is None:
            rs = row_scale
        else:
            ok = row_map >= 0
            rs[row_map[ok].long()] = row_scale[ok]
        out = out * rs.unsqueeze(1)
    if y0 is not None:
        out = out + y0
    return out


def _relerr(a, b):
    return ((a - b).norm() / b.norm().clamp(min=1e-30)).item()


@pytest.mark.parametrize("F", [256, 128, 64, 4, 100, 602, 41, 1, 300, 44, 48, 40])
def test_spmm_plain(built, F):
    from bns_gcn_b200 import ops
    dev = torch.device("cuda:0")
    indptr, idx = _rand_csr(700, 900, 12, seed=F, heavy=2)
    x = torch.randn(900, F, generator=torch.Generator().manual_seed(F + 1))
    g = ops.DeviceGraph.from_csr(indptr.to(dev), idx.int().to(dev), 900)
    assert g.n_split_rows >= 2
    y = ops.spmm(g, x.to(dev)).cpu()
    ref = _ref_spmm(indptr, idx, x)
    assert _relerr(y, ref) < RTOL
    # rows without entries must be written as zeros
    empty = (indptr[1:] - indptr[:-1]) == 0
    assert empty.any() and torch.all(y[empty] == 0)


@pytest.mark.parametrize("F", [256, 604, 128, 44])
@pytest.mark.parametrize("slab", [0, 256, 128, 64, 32])
def test_spmm_every_slab_variant(built, F, slab):
    """Every column-slab instantiation of spmm_kernel against oracle/spmm_ref.c -- including the ones the default
    heuristic only picks on graphs too large for a unit test: <4,32,1> with n_tiles > 1 (F = 256 as two 128-float slabs,
    the instantiation behind the headline bench number), <4,16,1> and <4,8,1> multi-tile (sub-warp row groups), with the
    GUARD path where the slab does not divide F (604, 44).  Rows longer than one chunk exercise the partial sums."""
    from bns_gcn_b200 import ops
    dev = torch.device("cuda:0")
    indptr, idx = _rand_csr(900, 1100, 14, seed=F + slab, heavy=3)
    x = torch.randn(1100, F, generator=torch.Generator().manual_seed(F + slab + 1))
    g = ops.DeviceGraph.from_csr(indptr.to(dev), idx.int().to(dev), 1100)
    assert g.n_split_rows >= 3
    y = ops.spmm(g, x.to(dev), slab=slab).cpu()
    ref = _ref_spmm(indptr, idx, x)
    assert _relerr(y, ref) < RTOL
    # full-warp slabs (256 / 128) keep the per-row summation order of the unblocked kernel: bit-identical; sub-warp
    # row groups (64 / 32) sum the entries of a chunk in a different order: equal to rounding
    y_full = ops.spmm(g, x.to(dev), slab=256).cpu()
    if slab in (128, 256):
        assert torch.equal(y, y_full)
    else:
        assert _relerr(y, y_full) < 1e-6


@pytest.mark.parametrize("slab", [256, 128, 64])
@pytest.mark.parametrize("F", [256, 604, 128])
def test_spmm_slab_variants_with_maps_scales_accumulate(built, F, slab):
    """The per-epoch forms (slot-mapped halo columns + col/row scales + accumulate; row-mapped backward) under a forced
    slab: the MAP / CSCALE instantiations of the blocked kernels."""
    from bns_gcn_b200 import ops
    dev = torch.device("cuda:0")
    gen = torch.Generator().manual_seed(31 + F + slab)
    n_rows, n_direct, n_halo, n_slab = 500, 500, 420, 150
    indptr, idx = _rand_csr(n_rows, n_direct + n_halo, 18, seed=F + slab, heavy=2)
    slot = torch.full((n_halo,), -1, dtype=torch.int32)
    chosen = torch.randperm(n_halo, generator=gen)[:n_slab]
    slot[chosen] = torch.randperm(n_slab, generator=gen).int()
    x = torch.randn(n_direct + n_slab, F, generator=gen)
    cs = torch.rand(n_direct + n_halo, generator=gen) + 0.5
    rs = torch.rand(n_rows, generator=gen) + 0.5
    col_map = torch.where(slot >= 0, slot + n_direct, slot)
    g = ops.DeviceGraph.from_csr(indptr.to(dev), idx.int().to(dev), n_direct + n_halo)
    y0 = torch.randn(n_rows, F, generator=gen)
    y = y0.clone().to(dev)
    ops.spmm(g, x.to(dev), y, row_scale=rs.to(dev), col_scale=cs.to(dev), col_map=col_map.to(dev),
             n_direct=n_direct, accumulate=True, slab=slab)
    ref = _ref_spmm(indptr, idx, x, row_scale=rs, col_scale=cs, col_map=col_map, n_direct=n_direct) + y0
    assert _relerr(y.cpu(), ref) < RTOL
    ind2, idx2 = _rand_csr(n_halo, n_rows, 20, seed=F + slab + 100, heavy=1, empty_frac=0.0)
    dy = torch.randn(n_rows, F, generator=gen)
    g2 = ops.DeviceGraph.from_csr(ind2.to(dev), idx2.int().to(dev), n_rows)
    out = torch.full((n_slab, F), 7.0, device=dev)
    ops.spmm(g2, dy.to(dev), out, row_map=slot.to(dev), row_scale=cs[n_direct:].to(dev), slab=slab)
    ref2 = _ref_spmm(ind2, idx2, dy, row_scale=cs[n_direct:], row_map=slot, n_out=n_slab)
    assert _relerr(out.cpu(), ref2) < RTOL


def test_spmm_roundtrip_csr_and_transpose(built):
    from bns_gcn_b200 import ops
    dev = torch.device("cuda:0")
    indptr, idx = _rand_csr(500, 300, 9, seed=3, heavy=1)
    g = ops.DeviceGraph.from_csr(indptr.to(dev), idx.int().to(dev), 300)
    ip, ix = g.csr()
    assert torch.equal(ip.cpu(), indptr) and torch.equal(ix.cpu().long(), idx)        # bit-exact copy
    gt = g.transpose()
    assert (gt.n_rows, gt.n_cols, gt.nnz) == (300, 500, g.nnz)
    tp, tx = (t.cpu() for t in gt.csr())
    rows = torch.repeat_interleave(torch.arange(500), indptr[1:] - indptr[:-1])
    order = torch.argsort(idx * 500 + rows, stable=True)                                # by column, rows ascending
    assert torch.equal(tx.long(), rows[order])
    cnt = torch.bincount(idx, minlength=300)
    assert torch.equal(tp[1:] - tp[:-1], cnt)
    # backward of the aggregation == SpMM on the transpose == oracle's reversed-graph SpMM
    dy = torch.randn(500, 64, generator=torch.Generator().manual_seed(5))
    dx = ops.spmm(gt, dy.to(dev)).cpu()
    from oracle import bns_oracle as O
    e = O.EdgeList(idx, rows, 300, 500)
    tip, tcols = e.csr_t()
    ref = O._spmm(tip, tcols, dy, 300)
    assert _relerr(dx, ref) < RTOL


@pytest.mark.parametrize("F", [256, 128, 36, 7, 44])
def test_spmm_scales_maps_accumulate(built, F):
    """The per-epoch form: halo columns resolved through a slot map (-1 = unsampled), GCN-style col / row
    scales, accumulation on top of the inner-edge pass, and the row-mapped backward."""
    from bns_gcn_b200 import ops
    dev = torch.device("cuda:0")
    gen = torch.Generator().manual_seed(11 + F)
    n_rows, n_direct, n_halo, n_slab = 400, 400, 350, 120
    indptr, idx = _rand_csr(n_rows, n_direct + n_halo, 15, seed=F, heavy=1)
    slot = torch.full((n_halo,), -1, dtype=torch.int32)
    chosen = torch.randperm(n_halo, generator=gen)[:n_slab]
    slot[chosen] = torch.randperm(n_slab, generator=gen).int()
    x = torch.randn(n_direct + n_slab, F, generator=gen)
    cs = torch.rand(n_direct + n_halo, generator=gen) + 0.5
    rs = torch.rand(n_rows, generator=gen) + 0.5
    col_map = torch.where(slot >= 0, slot + n_direct, slot)        # absolute row of x
    g = ops.DeviceGraph.from_csr(indptr.to(dev), idx.int().to(dev), n_direct + n_halo)
    y0 = torch.randn(n_rows, F, generator=gen)
    y = y0.clone().to(dev)
    ops.spmm(g, x.to(dev), y, row_scale=rs.to(dev), col_scale=cs.to(dev), col_map=col_map.to(dev),
             n_direct=n_direct, accumulate=True)
    ref = _ref_spmm(indptr, idx, x, row_scale=rs, col_scale=cs, col_map=col_map, n_direct=n_direct) + y0
    assert _relerr(y.cpu(), ref) < RTOL
    # row-mapped (backward over sampled halo rows): rows = halo nodes, output row = slab slot
    ind2, idx2 = _rand_csr(n_halo, n_rows, 20, seed=F + 100, heavy=1, empty_frac=0.0)
    dy = torch.randn(n_rows, F, generator=gen)
    g2 = ops.DeviceGraph.from_csr(ind2.to(dev), idx2.int().to(dev), n_rows)
    out = torch.full((n_slab, F), 7.0, device=dev)
    ops.spmm(g2, dy.to(dev), out, row_map=slot.to(dev), row_scale=cs[n_direct:].to(dev), col_scale=rs.to(dev))
    ref2 = _ref_spmm(ind2, idx2, dy, row_scale=cs[n_direct:], col_scale=rs, row_map=slot, n_out=n_slab)
    assert _relerr(out.cpu(), ref2) < RTOL


def test_spmm_edge_cases(built):
    from bns_gcn_b200 import ops, _lib
    dev = torch.device("cuda:0")
    # empty graph (no rows), graph with rows but no entries
    g0 = ops.DeviceGraph.from_csr(torch.zeros(1, dtype=torch.int64, device=dev), torch.empty(0, dtype=torch.int32, device=dev), 5)
    assert ops.spmm(g0, torch.randn(5, 8, device=dev)).shape == (0, 8)
    g1 = ops.DeviceGraph.from_csr(torch.zeros(4, dtype=torch.int64, device=dev), torch.empty(0, dtype=torch.int32, device=dev), 5)
    assert torch.all(ops.spmm(g1, torch.randn(5, 8, device=dev)) == 0)
    # non-contiguous leading dimension (a column slice) takes the scalar / strided path
    indptr, idx = _rand_csr(64, 64, 5, seed=1)
    g = ops.DeviceGraph.from_csr(indptr.to(dev), idx.int().to(dev), 64)
    big = torch.randn(64, 40)
    y = ops.spmm(g, big.to(dev)[:, 3:35]).cpu()
    assert _relerr(y, _ref_spmm(indptr, idx, big[:, 3:35].contiguous())) < RTOL
    # out-of-range column index is rejected at creation, with a message
    bad = idx.clone()
    bad[0] = 64
    with pytest.raises(_lib.BnsError, match="outside"):
        ops.DeviceGraph.from_csr(indptr.to(dev), bad.int().to(dev), 64)
    with pytest.raises(_lib.BnsError):
        ops.spmm(g, torch.randn(64, 8))          # CPU tensor: no CPU path


def test_aggregate_autograd_matches_oracle(built):
    from bns_gcn_b200 import ops
    from oracle import bns_oracle as O
    dev = torch.device("cuda:0")
    indptr, idx = _rand_csr(300, 300, 10, seed=9, heavy=1, empty_frac=0.0)
    rows = torch.repeat_interleave(torch.arange(300), indptr[1:] - indptr[:-1])
    deg = (indptr[1:] - indptr[:-1]).clamp(min=1).float()
    x = torch.randn(300, 128, generator=torch.Generator().manual_seed(2), requires_grad=True)
    w = torch.randn(300, 128, generator=torch.Generator().manual_seed(3))
    ref = O.CopyUSum.apply(O.EdgeList(idx, rows, 300, 300), x) / deg.unsqueeze(1)
    (ref * w).sum().backward()
    xg = x.detach().to(dev).requires_grad_(True)
    g = ops.DeviceGraph.from_csr(indptr.to(dev), idx.int().to(dev), 300)
    y = ops.AggregateSum.apply(xg, g, (1.0 / deg).to(dev), None)
    (y * w.to(dev)).sum().backward()
    assert _relerr(y.detach().cpu(), ref.detach()) < RTOL
    assert _relerr(xg.grad.cpu(), x.grad) < RTOL


@pytest.mark.parametrize("F", [256, 41, 602])
def test_gather_scatter(built, F):
    from bns_gcn_b200 import ops
    dev = torch.device("cuda:0")
    gen = torch.Generator().manual_seed(F)
    h = torch.randn(500, F, generator=gen)
    idx = torch.randperm(500, generator=gen)[:123]
    ratio = 123 / 500
    out = ops.gather_div(h.to(dev), idx.to(dev), ratio).cpu()
    assert torch.equal(out, h[idx] / ratio)                       # true division: bit-exact vs torch CPU
    grad = torch.randn(500, F, generator=gen)
    src = torch.randn(123, F, generator=gen)
    ref = grad.clone()
    ref[idx] += src / ratio
    got = ops.scatter_add_div(grad.clone().to(dev), idx.to(dev), src.to(dev), ratio).cpu()
    assert torch.equal(got, ref)
    # empty selection is a no-op
    e = torch.empty(0, dtype=torch.int64, device=dev)
    assert ops.gather_div(h.to(dev), e, 1.0).shape == (0, F)


def test_sampler_exact_vs_philox_replay(built):
    from bns_gcn_b200 import ops
    from oracle import philox
    dev = torch.device("cuda:0")
    gen = torch.Generator().manual_seed(0)
    boundary = [None, torch.sort(torch.randperm(5000, generator=gen)[:1733])[0], torch.empty(0, dtype=torch.int64),
                torch.sort(torch.randperm(9000, generator=gen)[:4000])[0]]
    send = [0, int(0.1 * 1733), 0, int(0.37 * 4000)]
    s = ops.BoundarySampler(boundary, send, dev)
    for seed, off in [(0, 0), (12345, 7), (2**40 + 3, 2**33 + 1)]:
        _, views = s.sample(seed, off)
        ref = philox.sample_boundary([b.numpy() for b in boundary if b is not None], [send[j] for j in s.peers], seed, off)
        for i, j in enumerate(s.peers):
            assert torch.equal(views[j].cpu(), torch.from_numpy(ref[i])), (seed, off, j)      # exact, ordered
            v = views[j].cpu()
            assert v.numel() == send[j] and v.unique().numel() == v.numel()                    # no duplicates
            assert torch.isin(v, boundary[j]).all()                                            # subset
    # different epochs give different samples; same (seed, offset) is reproducible
    a = s.sample(1, 5)[0].clone()
    assert torch.equal(a, s.sample(1, 5)[0]) and not torch.equal(a, s.sample(1, 6)[0])


def test_sampler_uniform_inclusion(built):
    """chi-square on inclusion counts: every boundary node is sampled with probability k/b."""
    from bns_gcn_b200 import ops
    dev = torch.device("cuda:0")
    b, k, trials = 200, 50, 2000
    s = ops.BoundarySampler([None, torch.arange(b)], [0, k], dev)
    cnt = torch.zeros(b)
    for t in range(trials):
        cnt += torch.bincount(s.sample(99, t)[0].cpu(), minlength=b)
    exp = trials * k / b
    chi2 = (((cnt - exp) ** 2) / (exp * (1 - k / b))).sum().item()      # ~ chi2(b-1): mean 199, sd ~20
    assert 120 < chi2 < 290, chi2


def test_halo_slot_update(built):
    from bns_gcn_b200 import ops
    dev = torch.device("cuda:0")
    n_in, n_halo, part = 100, 60, 80
    gen = torch.Generator().manual_seed(4)
    pos = torch.full((part,), -1, dtype=torch.int64)
    owned = torch.randperm(part, generator=gen)[:n_halo]
    pos[owned] = n_in + torch.arange(n_halo)
    one_hops = owned[torch.randperm(n_halo, generator=gen)[:25]]
    slot = torch.empty(n_halo, dtype=torch.int32, device=dev)
    ops.fill_i32(slot, -1)
    ops.halo_slot_update(pos.to(dev), one_hops.to(dev), n_in, 1000, slot)
    ref = torch.full((n_halo,), -1, dtype=torch.int32)
    ref[pos[one_hops] - n_in] = 1000 + torch.arange(25, dtype=torch.int32)
    assert torch.equal(slot.cpu(), ref)


@pytest.mark.parametrize("F,p", [(256, 0.0), (256, 0.5), (64, 0.3), (600, 0.5), (16, 0.0)])
def test_fused_layernorm_relu_dropout(built, F, p):
    """ops.LnReluDropout == dropout(relu(layer_norm(x))) forward and backward (mask recovered from the output),
    mask keep-rate ~ 1-p, masks differ across offsets and repeat for the same (seed, offset)."""
    import torch.nn.functional as Fn
    from bns_gcn_b200 import ops
    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(F)
    n = 3000
    x = (torch.randn(n, F, generator=g) * 2 + 0.3).to(dev).requires_grad_(True)
    gamma = (torch.rand(F, generator=g) + 0.5).to(dev).requires_grad_(True)
    beta = (torch.randn(F, generator=g) * 0.2).to(dev).requires_grad_(True)
    dy = torch.randn(n, F, generator=g).to(dev)
    ops.RNG.update(seed=123, offset=5, offset_dev=None)
    y = ops.LnReluDropout.apply(x, gamma, beta, 1e-5, p, 77)
    y.backward(dy)
    got = (y.detach().clone(), x.grad.clone(), gamma.grad.clone(), beta.grad.clone())
    # reference with the same mask
    xr, gr, br = (t.detach().clone().requires_grad_(True) for t in (x, gamma, beta))
    z = Fn.relu(Fn.layer_norm(xr, (F,), gr, br, 1e-5))
    if p > 0:
        mask = ((y.detach() != 0) | (z.detach() <= 0)).float()
        keep = mask[z.detach() > 0].mean().item()
        assert abs(keep - (1 - p)) < 0.01, keep
        ref = z * mask / (1 - p)
    else:
        ref = z
    ref.backward(dy)
    for a, b in zip(got, (ref.detach(), xr.grad, gr.grad, br.grad)):
        assert _relerr(a.cpu(), b.cpu()) < 2e-5
    if p > 0:
        y2 = ops.LnReluDropout.apply(x.detach(), gamma.detach(), beta.detach(), 1e-5, p, 77)
        assert torch.equal(y2, y.detach())                            # same (seed, offset) -> same mask
        off_dev = torch.tensor([1], dtype=torch.int64, device=dev)    # 5 + 1: offset read from the device
        ops.RNG.update(offset=5, offset_dev=off_dev)
        y3 = ops.LnReluDropout.apply(x.detach(), gamma.detach(), beta.detach(), 1e-5, p, 77)
        ops.RNG.update(offset=6, offset_dev=None)
        y4 = ops.LnReluDropout.apply(x.detach(), gamma.detach(), beta.detach(), 1e-5, p, 77)
        assert torch.equal(y3, y4) and not torch.equal(y3, y.detach())
    ops.RNG.update(seed=0, offset=0, offset_dev=None)


@pytest.mark.parametrize("F", [64, 256, 44])
def test_weighted_spmm_perm_and_sddmm(built, F):
    """GAT primitives: per-entry weights in the SpMM, the transpose's entry permutation, and the SDDMM dot."""
    from bns_gcn_b200 import ops
    dev = torch.device("cuda:0")
    gen = torch.Generator().manual_seed(F)
    n_rows, n_direct, n_halo, n_slab = 300, 300, 200, 70
    indptr, idx = _rand_csr(n_rows, n_direct + n_halo, 14, seed=F + 3, heavy=1)
    nnz = idx.numel()
    rows = torch.repeat_interleave(torch.arange(n_rows), indptr[1:] - indptr[:-1])
    w = torch.rand(nnz, generator=gen)
    slot = torch.full((n_halo,), -1, dtype=torch.int32)
    chosen = torch.randperm(n_halo, generator=gen)[:n_slab]
    slot[chosen] = torch.randperm(n_slab, generator=gen).int()
    col_map = torch.where(slot >= 0, slot + n_direct, slot)
    x = torch.randn(n_direct + n_slab, F, generator=gen)
    g = ops.DeviceGraph.from_csr(indptr.to(dev), idx.int().to(dev), n_direct + n_halo, 64)
    y = ops.spmm(g, x.to(dev), edge_weight=w.to(dev), col_map=col_map.to(dev), n_direct=n_direct).cpu()
    xrow = idx.clone()
    m = idx >= n_direct
    xrow[m] = col_map[idx[m] - n_direct].long()
    keep = xrow >= 0
    ref = torch.zeros(n_rows, F).index_add_(0, rows[keep], x[xrow[keep]] * w[keep].unsqueeze(1))
    assert _relerr(y, ref) < RTOL
    # transpose permutation: entry k of g^T is entry perm[k] of g
    gt = g.transpose()
    perm = gt.perm().cpu().long()
    tp, tx = (t.cpu() for t in gt.csr())
    assert torch.equal(tx.long(), rows[perm])
    tcols = torch.repeat_interleave(torch.arange(gt.n_rows), tp[1:] - tp[:-1])
    assert torch.equal(tcols, idx[perm])
    # weighted transpose SpMM == autograd of the forward
    dy = torch.randn(n_rows, F, generator=gen)
    dx = ops.spmm(gt, dy.to(dev), edge_weight=w[perm].to(dev)).cpu()
    ref_dx = torch.zeros(n_direct + n_halo, F).index_add_(0, idx, dy[rows] * w.unsqueeze(1))
    assert _relerr(dx, ref_dx) < RTOL
    # SDDMM dot with the column map: d w_k = <dy[row_k], x[xrow_k]>, 0 for skipped entries
    if F % 4 == 0:
        dw = ops.sddmm_dot(g, dy.to(dev), x.to(dev), col_map=col_map.to(dev), n_direct=n_direct).cpu()
        ref_dw = torch.zeros(nnz)
        ref_dw[keep] = (dy[rows[keep]] * x[xrow[keep]]).sum(1)
        assert _relerr(dw, ref_dw) < RTOL
        assert torch.all(dw[~keep] == 0)


# =====================================================================================================================
# ABI 2: the one-launch-per-step kernels of csrc/fused.cuh
# =====================================================================================================================
@pytest.mark.parametrize("n,C,Cp", [(3000, 41, 44), (500, 5, 8), (1000, 100, 100)])
def test_fused_cross_entropy_loss_and_gradient(built, n, C, Cp):
    """bns_xent_f32 == CrossEntropyLoss(reduction='sum') over the masked rows, forward and d(logits) (train.py:358-361,
    406-408); pad columns and unmasked rows get exact zeros; the loss is bit-reproducible."""
    from bns_gcn_b200 import fused
    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(n + C)
    logits = (torch.randn(n, Cp, generator=g) * 3).to(dev)
    labels = torch.randint(0, C, (n,), generator=g).to(dev)
    mask = (torch.rand(n, generator=g) < 0.6).to(dev)
    scale = 1.0 / 777.0
    loss, dl = fused.softmax_xent(logits, C, labels, mask, scale)
    x = logits[:, :C].detach().clone().requires_grad_(True)
    ref = torch.nn.functional.cross_entropy(x[mask], labels[mask], reduction="sum")
    ref.backward()
    assert abs(loss.item() - ref.item()) <= 2e-6 * abs(ref.item())
    assert _relerr(dl[:, :C].cpu(), (x.grad * scale).cpu()) < 2e-6
    assert torch.all(dl[:, C:] == 0) and torch.all(dl[~mask] == 0)
    loss2, dl2 = fused.softmax_xent(logits, C, labels, mask, scale)
    assert loss2.item() == loss.item() and torch.equal(dl, dl2)


def test_fused_bce_with_logits_loss_and_gradient(built):
    from bns_gcn_b200 import fused
    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(5)
    n, C, Cp = 2000, 6, 8
    logits = (torch.randn(n, Cp, generator=g) * 4).to(dev)
    y = (torch.rand(n, C, generator=g) < 0.2).float().to(dev)
    mask = (torch.rand(n, generator=g) < 0.7).to(dev)
    loss, dl = fused.softmax_xent(logits, C, y, mask, 0.5)
    x = logits[:, :C].detach().clone().requires_grad_(True)
    ref = torch.nn.functional.binary_cross_entropy_with_logits(x[mask], y[mask], reduction="sum")
    ref.backward()
    assert abs(loss.item() - ref.item()) <= 2e-6 * abs(ref.item())
    assert _relerr(dl[:, :C].cpu(), (x.grad * 0.5).cpu()) < 2e-6
    assert torch.all(dl[:, C:] == 0) and torch.all(dl[~mask] == 0)


@pytest.mark.parametrize("wd", [0.0, 5e-4])
def test_fused_adam_matches_torch_adam(built, wd):
    """bns_adam_step_f32 over the flat arena + bns_derive_refresh == torch.optim.Adam on the same parameters, several
    steps; padded slots stay zero; cached transposes and bias sums follow the parameters."""
    from bns_gcn_b200 import fused
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    net = torch.nn.Sequential(torch.nn.Linear(30, 41), torch.nn.LayerNorm(41), torch.nn.Linear(41, 7)).to(dev)
    ref = [p.detach().clone().requires_grad_(True) for p in net.parameters()]
    arena = fused.ParamArena(net)
    opt = fused.FusedAdam(arena, lr=1e-2, weight_decay=wd)
    ropt = torch.optim.Adam(ref, lr=1e-2, weight_decay=wd)
    w0 = net[0].weight
    wt = arena.transposed(w0)                   # [30, 44] cache of the padded weight
    bsum = arena.bias_sum(net[0].bias, net[1].bias)
    assert arena.padded(w0).shape == (44, 30) and torch.all(arena.padded(w0)[41:] == 0)
    g = torch.Generator().manual_seed(1)
    for step in range(5):
        for p, r in zip(net.parameters(), ref):
            gr = torch.randn(p.shape, generator=g).to(dev)
            p.grad.copy_(gr)                    # the arena's gradient views
            r.grad = gr.clone()
        opt.step()
        ropt.step()
        for p, r in zip(net.parameters(), ref):
            assert _relerr(p.detach().cpu(), r.detach().cpu()) < 2e-6, step
        assert torch.all(arena.padded(w0)[41:] == 0)
        assert torch.equal(wt[:, :41], w0.detach().t()) and torch.all(wt[:, 41:] == 0)
        assert torch.equal(bsum[:41], net[0].bias.detach() + net[1].bias.detach())
    assert int(opt.step_dev.item()) == 5


def test_scatter_rows_all_equals_successive_scatter_adds(built):
    """bns_scatter_rows_all_f32 over the inverse maps of bns_epoch_maps_update == the P-1 successive
    bns_scatter_add_div_f32 calls of the reference's order (helper/feature_buffer.py:111-129), bit for bit; the slot
    map part of the same kernel == fill + per-peer bns_halo_slot_update."""
    import ctypes
    from bns_gcn_b200 import ops
    from bns_gcn_b200._lib import EpochMaps, check, lib
    dev = torch.device("cuda:0")
    gen = torch.Generator().manual_seed(3)
    n_in, n_halo, F, peers = 700, 500, 256, 3
    sel = [torch.randperm(n_in, generator=gen)[:k] for k in (150, 0, 260)]
    ratios = [0.3, 0.0, 0.26]
    part_sizes = [400, 300, 500]
    pos, hops, halo_next = [], [], n_in
    for s_, ps in enumerate(part_sizes):
        p_ = torch.full((ps,), -1, dtype=torch.int64)
        cnt = [120, 200, 180][s_]
        owned = torch.randperm(ps, generator=gen)[:cnt]
        p_[owned] = halo_next + torch.arange(cnt)
        halo_next += cnt
        pos.append(p_)
        hops.append(owned[torch.randperm(cnt, generator=gen)[:[40, 0, 77][s_]]])
    sel_cat, hops_cat = torch.cat(sel).to(dev), torch.cat(hops).to(dev)
    maps = torch.full((n_halo + peers * n_in,), 5, dtype=torch.int32, device=dev)
    pos_d = [p_.to(dev) for p_ in pos]
    m = EpochMaps()
    m.n_seg = peers
    a = b = 0
    for s_ in range(peers):
        m.sel_begin[s_], m.hop_begin[s_] = a, b
        a += sel[s_].numel()
        b += hops[s_].numel()
        m.pos[s_] = pos_d[s_].data_ptr()
        m.inv[s_] = maps[n_halo + s_ * n_in:].data_ptr()
    m.sel_begin[peers], m.hop_begin[peers] = a, b
    m.selected_cat, m.one_hops_cat, m.slot, m.n_in = sel_cat.data_ptr(), hops_cat.data_ptr(), maps.data_ptr(), n_in
    check(lib.bns_epoch_maps_update(ctypes.byref(m), maps.data_ptr(), maps.numel() * 4,
                                    torch.cuda.current_stream().cuda_stream))
    slot_ref = torch.empty(n_halo, dtype=torch.int32, device=dev)
    ops.fill_i32(slot_ref, -1)
    off = 0
    for s_ in range(peers):
        if hops[s_].numel():
            ops.halo_slot_update(pos_d[s_], hops[s_].to(dev), n_in, off, slot_ref)
        off += hops[s_].numel()
    assert torch.equal(maps[:n_halo], slot_ref)
    for s_ in range(peers):
        inv = maps[n_halo + s_ * n_in:n_halo + (s_ + 1) * n_in].cpu()
        want = torch.full((n_in,), -1, dtype=torch.int32)
        want[sel[s_]] = torch.arange(sel[s_].numel(), dtype=torch.int32)
        assert torch.equal(inv, want)
    G0 = torch.randn(n_in, F, generator=gen).to(dev)
    recv = [torch.randn(max(sel[s_].numel(), 1), F, generator=gen).to(dev) for s_ in range(peers)]
    order = [2, 0]                                   # the reference's ring order, peers with an empty sample skipped
    ref = G0.clone()
    for s_ in order:
        ops.scatter_add_div(ref, sel[s_].to(dev), recv[s_][:sel[s_].numel()], ratios[s_])
    got = G0.clone()
    inv_p = (ctypes.c_void_p * 2)(*[maps[n_halo + s_ * n_in:].data_ptr() for s_ in order])
    rcv_p = (ctypes.c_void_p * 2)(*[recv[s_].data_ptr() for s_ in order])
    div = (ctypes.c_float * 2)(*[ratios[s_] for s_ in order])
    check(lib.bns_scatter_rows_all_f32(got.data_ptr(), got.stride(0), n_in, F, 2, inv_p, rcv_p, F, div,
                                       torch.cuda.current_stream().cuda_stream))
    assert torch.equal(got, ref)


@pytest.mark.parametrize("F", [256, 44, 604])
def test_compacted_halo_spmm_is_bit_identical_to_the_column_mapped_one(built, F):
    """bns_graph_compact_cols + bns_spmm_compact_f32 == bns_spmm_sum_f32(col_map): same entries, same order."""
    from bns_gcn_b200 import ops
    dev = torch.device("cuda:0")
    gen = torch.Generator().manual_seed(17 + F)
    n_rows, n_halo, n_slab = 600, 900, 90                        # ~10 % of the halo columns sampled
    indptr, idx = _rand_csr(n_rows, n_halo, 40, seed=F, heavy=2)
    slot = torch.full((n_halo,), -1, dtype=torch.int32)
    chosen = torch.randperm(n_halo, generator=gen)[:n_slab]
    slot[chosen] = torch.randperm(n_slab, generator=gen).int()
    x = torch.randn(n_slab, F, generator=gen).to(dev)
    rs = (torch.rand(n_rows, generator=gen) + 0.5).to(dev)
    cs = (torch.rand(n_halo, generator=gen) + 0.5).to(dev)
    g = ops.DeviceGraph.from_csr(indptr.to(dev), idx.int().to(dev), n_halo, 64)
    y0 = torch.randn(n_rows, F, generator=gen).to(dev)
    for weights in (False, True):
        ref = y0.clone()
        ops.spmm(g, x, ref, row_scale=rs, col_scale=cs if weights else None, col_map=slot.to(dev), n_direct=0,
                 accumulate=True)
        c = ops.CompactedCols(g, with_weights=weights)
        c.refresh(slot.to(dev), 0, cs if weights else None)
        got = y0.clone()
        ops.spmm_compact(c, x, got, row_scale=rs, accumulate=True)
        if F >= 128:      # full-warp slabs: the same entries added in the same order
            assert torch.equal(got, ref), weights
        else:             # sub-warp row groups split a chunk's entries between them by position: equal to rounding
            assert _relerr(got.cpu(), ref.cpu()) < 1e-6, weights
        live = int((slot[idx] >= 0).sum())
        assert int(c.chunk_cnt.sum()) == live
    # a second epoch with another sample reuses the buffers
    slot2 = torch.full((n_halo,), -1, dtype=torch.int32)
    slot2[torch.randperm(n_halo, generator=gen)[:n_slab]] = torch.randperm(n_slab, generator=gen).int()
    c.refresh(slot2.to(dev), 0, cs)
    ref = torch.zeros(n_rows, F, device=dev)
    ops.spmm(g, x, ref, col_scale=cs, col_map=slot2.to(dev), n_direct=0)
    got = torch.zeros(n_rows, F, device=dev)
    ops.spmm_compact(c, x, got)
    assert torch.equal(got, ref) if F >= 128 else _relerr(got.cpu(), ref.cpu()) < 1e-6


def test_dropout_and_scale_rows_kernels(built):
    from bns_gcn_b200 import fused, ops
    dev = torch.device("cuda:0")
    x = torch.randn(4000, 1204, generator=torch.Generator().manual_seed(0)).to(dev)
    ops.RNG.update(seed=9, offset=3, offset_dev=None)
    y = fused.dropout(x, 0.5, 1234)
    keep = (y != 0)
    assert abs(keep.float().mean().item() - 0.5) < 0.005
    assert torch.equal(y[keep], (x * 2.0)[keep])
    assert torch.equal(y, fused.dropout(x, 0.5, 1234))
    ops.RNG.update(offset=4)
    assert not torch.equal(y, fused.dropout(x, 0.5, 1234))
    ops.RNG.update(seed=0, offset=0, offset_dev=None)
    assert fused.dropout(x, 0.0, 1) is x
    rs = torch.rand(4000, device=dev)
    assert torch.equal(fused.scale_rows(x, rs), x * rs.unsqueeze(1))


def test_dense_epilogue_row_scale_and_in_place_addend(built):
    from bns_gcn_b200.module import dense
    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(2)
    a = torch.randn(5000, 256, generator=g).to(dev)
    w = (torch.rand(256, 256, generator=g) - 0.5).to(dev)
    rs = (torch.rand(5000, generator=g) + 0.5).to(dev)
    ref = (a.double() @ w.double().t()) * rs.double().unsqueeze(1)
    got = dense.tc_mm_tn(a, w, row_scale=rs)
    assert _relerr(got.double().cpu(), ref.cpu()) < 1e-5
    acc = torch.randn(6000, 256, generator=g).to(dev)
    want = acc.clone()
    want[:5000] += (a.double() @ w.double().t()).float()
    dense.tc_mm_tn(a, w, addend=acc[:5000], out=acc[:5000])          # C aliases the addend: accumulate in place
    assert _relerr(acc.cpu(), want.cpu()) < 1e-5
    o1, o2 = torch.empty(256, device=dev), torch.empty(256, device=dev)
    dense.colsum(a, out=o1, out2=o2)
    assert torch.equal(o1, o2) and _relerr(o1.cpu(), a.double().sum(0).float().cpu()) < 1e-5


def _gat_case(H, Fo, seed, with_halo=True):
    """A partition-like graph on the device + the per-entry lists a torch reference needs."""
    from bns_gcn_b200 import ops
    from bns_gcn_b200.graph import PartitionGraph
    dev = torch.device("cuda:0")
    gen = torch.Generator().manual_seed(seed)
    n_in, n_halo, n_slab = 300, 260, 70
    ip_in, ix_in = _rand_csr(n_in, n_in, 9, seed=seed, heavy=1, empty_frac=0.05)
    a_in = ops.DeviceGraph.from_csr(ip_in.to(dev), ix_in.int().to(dev), n_in, 64)
    a_out = None
    ip_out = ix_out = None
    if with_halo:
        ip_out, ix_out = _rand_csr(n_in, n_halo, 12, seed=seed + 1, heavy=1, empty_frac=0.2)
        a_out = ops.DeviceGraph.from_csr(ip_out.to(dev), ix_out.int().to(dev), n_halo, 64)
    g = PartitionGraph(n_in, n_halo if with_halo else 0, a_in, a_out, dev)
    g.want_positions = True
    n_u = n_in
    slot = None
    if with_halo:
        slot = torch.full((n_halo,), -1, dtype=torch.int32)
        chosen = torch.randperm(n_halo, generator=gen)[:n_slab]
        slot[chosen] = torch.randperm(n_slab, generator=gen).int()
        g.slot.copy_(slot.to(dev))
        g.refresh_compaction()
        n_u = n_in + n_slab
    rows_in = torch.repeat_interleave(torch.arange(n_in), ip_in[1:] - ip_in[:-1])
    u = [ix_in]
    v = [rows_in]
    if with_halo:
        rows_out = torch.repeat_interleave(torch.arange(n_in), ip_out[1:] - ip_out[:-1])
        x = slot[ix_out].long()
        keep = x >= 0
        u.append(n_in + x[keep])
        v.append(rows_out[keep])
    return g, n_in, n_u, torch.cat(u), torch.cat(v), gen


@pytest.mark.parametrize("H,Fo,with_halo", [(1, 64, True), (2, 8, True), (4, 16, False), (1, 256, True), (1, 100, True)])
def test_fused_gat_attention_matches_the_per_entry_reference(built, H, Fo, with_halo):
    """graph.GatAttention == the u_add_v / leaky_relu / edge_softmax / u_mul_e+sum algebra of dgl.nn.GATConv written with
    torch ops on explicit entry lists (what module/gat.py's op-by-op path and oracle.GATConvRef do), forward and the
    gradients with respect to ft, el and er; attention dropout off."""
    from bns_gcn_b200.graph import GatAttention
    dev = torch.device("cuda:0")
    g, n_in, n_u, u, v, gen = _gat_case(H, Fo, 100 + H + Fo, with_halo)
    ft = torch.randn(n_u, H * Fo, generator=gen)
    el = torch.randn(n_u, H, generator=gen)
    er = torch.randn(n_in, H, generator=gen)
    d = torch.randn(n_in, H * Fo, generator=gen)
    # reference (f64 on the CPU)
    ftr, elr, err = (t.double().clone().requires_grad_(True) for t in (ft, el, er))
    e = torch.nn.functional.leaky_relu(elr[u] + err[v], 0.2)
    m = torch.full((n_in, H), float("-inf"), dtype=torch.float64).scatter_reduce(0, v.unsqueeze(1).expand(-1, H), e.detach(), "amax")
    ex = torch.exp(e - m[v])
    den = torch.zeros(n_in, H, dtype=torch.float64).index_add(0, v, ex)
    a = ex / den[v]
    ref = torch.zeros(n_in, H, Fo, dtype=torch.float64).index_add(0, v, a.unsqueeze(-1) * ftr.view(-1, H, Fo)[u]).reshape(n_in, H * Fo)
    (ref * d.double()).sum().backward()
    ftg, elg, erg = (t.to(dev).requires_grad_(True) for t in (ft, el, er))
    out = GatAttention.apply(ftg, elg, erg, g, H, Fo, 0.2, 0.0, 1)
    (out * d.to(dev)).sum().backward()
    assert _relerr(out.detach().cpu(), ref.detach().float()) < 2e-5
    assert _relerr(ftg.grad.cpu(), ftr.grad.float()) < 2e-5
    assert _relerr(elg.grad.cpu(), elr.grad.float()) < 5e-5
    assert _relerr(erg.grad.cpu(), err.grad.float()) < 5e-5
    # rows without any entry produce zeros
    deg = torch.bincount(v, minlength=n_in)
    assert torch.all(out.detach().cpu()[deg == 0] == 0)


def test_fused_gat_attention_dropout_is_consistent_between_forward_and_backward(built):
    """With attention dropout the layer is still linear in ft for fixed scores: <rst(ft), d> == <ft, d_ft(d)> holds only
    if the backward regenerates exactly the forward's Philox mask; the keep rate is 1 - p; a new offset gives a new mask."""
    from bns_gcn_b200 import ops
    from bns_gcn_b200.graph import GatAttention
    dev = torch.device("cuda:0")
    H, Fo, p = 2, 32, 0.4
    g, n_in, n_u, u, v, gen = _gat_case(H, Fo, 7, True)
    ft = torch.randn(n_u, H * Fo, generator=gen).to(dev).requires_grad_(True)
    el = torch.randn(n_u, H, generator=gen).to(dev)
    er = torch.randn(n_in, H, generator=gen).to(dev)
    d = torch.randn(n_in, H * Fo, generator=gen).to(dev)
    ops.RNG.update(seed=5, offset=11, offset_dev=None)
    out = GatAttention.apply(ft, el, er, g, H, Fo, 0.2, p, 3)
    out.backward(d)
    lhs, rhs = (out.detach() * d).sum().item(), (ft.detach() * ft.grad).sum().item()
    assert abs(lhs - rhs) <= 1e-4 * max(abs(lhs), 1.0), (lhs, rhs)
    out2 = GatAttention.apply(ft.detach(), el, er, g, H, Fo, 0.2, p, 3)
    assert torch.equal(out2, out.detach())
    ops.RNG.update(offset=12)
    assert not torch.equal(GatAttention.apply(ft.detach(), el, er, g, H, Fo, 0.2, p, 3), out.detach())
    # keep rate: compare the total attention mass of every row (sum of a' over its entries ~ 1) via ft = ones
    ones = torch.ones(n_u, H * Fo, device=dev)
    mass = GatAttention.apply(ones, el, er, g, H, Fo, 0.2, p, 3)[:, ::Fo]           # [n_in, H]: sum of a'_uv per head
    deg = torch.bincount(v, minlength=n_in).to(dev)
    big = deg >= 8
    assert abs(mass[big].mean().item() - 1.0) < 0.1
    ops.RNG.update(seed=0, offset=0, offset_dev=None)


@pytest.mark.parametrize("H,Fo,n_src,n_dst", [(1, 256, 3001, 2000), (2, 8, 777, 700), (8, 128, 300, 300), (1, 100, 513, 1), (3, 4, 50, 0)])
def test_gat_projection_matches_torch(built, H, Fo, n_src, n_dst):
    """graph.GatProjection (el / er of GATConv and their backward) == (ft.view(n, H, Fo) * attn).sum(-1) under autograd."""
    from bns_gcn_b200.graph import GatProjection
    dev = torch.device("cuda:0")
    gen = torch.Generator().manual_seed(H * 1000 + Fo)
    fs, fd = torch.randn(n_src, H * Fo, generator=gen), torch.randn(n_dst, H * Fo, generator=gen)
    al, ar = torch.randn(1, H, Fo, generator=gen), torch.randn(1, H, Fo, generator=gen)
    g1, g2 = torch.randn(n_src, H, generator=gen), torch.randn(n_dst, H, generator=gen)
    ref_in = [t.double().clone().requires_grad_(True) for t in (fs, fd, al, ar)]
    rel = (ref_in[0].view(-1, H, Fo) * ref_in[2]).sum(-1)
    rer = (ref_in[1].view(-1, H, Fo) * ref_in[3]).sum(-1)
    ((rel * g1.double()).sum() + (rer * g2.double()).sum()).backward()
    got_in = [t.to(dev).requires_grad_(True) for t in (fs, fd, al, ar)]
    el, er = GatProjection.apply(*got_in, H, Fo)
    ((el * g1.to(dev)).sum() + (er * g2.to(dev)).sum()).backward()
    assert _relerr(el.detach().cpu(), rel.detach().float()) < 1e-5
    if n_dst:
        assert _relerr(er.detach().cpu(), rer.detach().float()) < 1e-5
    for got, ref in zip(got_in, ref_in):
        assert got.grad.shape == ref.grad.shape
        if ref.grad.numel():
            assert _relerr(got.grad.cpu(), ref.grad.float()) < 2e-5
    # deterministic
    got2 = [t.to(dev).requires_grad_(True) for t in (fs, fd, al, ar)]
    e2, r2 = GatProjection.apply(*got2, H, Fo)
    ((e2 * g1.to(dev)).sum() + (r2 * g2.to(dev)).sum()).backward()
    assert torch.equal(got2[2].grad, got_in[2].grad) and torch.equal(got2[0].grad, got_in[0].grad)
