"""Graph handles passed to the layers in place of DGL graphs.

``PartitionGraph`` is what ``train.construct_graph`` returns: the reference rebuilds a bipartite ``_U -> _V``
``dgl.heterograph`` every epoch (train.py:256-281); here the structure is static -- ``a_in`` (inner -> inner) and
``a_out`` (halo -> inner), each with its transpose, all built once -- and an epoch only rewrites ``slot``:
``slot[h]`` = row of halo node ``h`` in this epoch's receive slab (U-numbering minus ``n_in``), or -1 when the
owner did not sample it.  Callers see the same surface the layers use: ``num_nodes('_V')``.

``FullGraphHandle`` is the homogeneous graph of the evaluation branch (module/layer.py:39-45, 93-102).
"""
from __future__ import annotations

from typing import Dict, Optional

import torch

from . import ops


class PartitionGraph:
    def __init__(self, n_in: int, n_halo: int, a_in: ops.DeviceGraph, a_out: Optional[ops.DeviceGraph], device):
        self.n_in, self.n_halo = n_in, n_halo
        self.a_in, self.a_out = a_in, a_out
        self.a_in_t = a_in.transpose()
        self.a_out_t = a_out.transpose() if a_out is not None else None
        self.device = device
        self.slot = torch.full((max(n_halo, 1),), -1, dtype=torch.int32, device=device)
        self.n_u = n_in
        self._recip: Dict[int, torch.Tensor] = {}
        # per-epoch compaction of a_out to the sampled halo columns (ops.CompactedCols), refreshed by construct_graph
        self.compact: Optional[ops.CompactedCols] = None
        self.halo_col_scale: Optional[torch.Tensor] = None      # GCN: 1/sqrt(out_deg) of the halo nodes (static)
        self.want_positions = False                             # GAT: the compaction also records CSR positions

    def refresh_compaction(self) -> None:
        """Call after every change of ``slot`` (train.construct_graph does)."""
        if self.a_out is None or self.a_out.nnz == 0:
            return
        if self.compact is None:
            self.compact = ops.CompactedCols(self.a_out, with_weights=self.halo_col_scale is not None,
                                             with_positions=self.want_positions)
        self.compact.refresh(self.slot, 0, self.halo_col_scale)

    def num_nodes(self, ntype: str = '_V') -> int:
        return self.n_in if ntype == '_V' else self.n_u

    def num_edges(self) -> int:
        return self.a_in.nnz + (self.a_out.nnz if self.a_out is not None else 0)

    def recip(self, t: torch.Tensor) -> torch.Tensor:
        """``1 / t`` as f32, cached per source tensor (degree / norm vectors are static)."""
        # keyed on the tensor OBJECT (kept alive here, so its id cannot be recycled) and its in-place version counter:
        # a freed-and-reallocated buffer at the same address, or a norm updated in place, never returns a stale value
        key = id(t)
        hit = self._recip.get(key)
        if hit is None or hit[0] is not t or hit[1] != t._version:
            hit = (t, t._version, (1.0 / t.to(torch.float32)).contiguous())
            self._recip[key] = hit
        return hit[2]


class FullGraphHandle:
    def __init__(self, a: ops.DeviceGraph, in_deg: torch.Tensor, out_deg: torch.Tensor):
        self.a = a
        self._in, self._out = in_deg, out_deg

    def num_nodes(self, ntype: str = '_V') -> int:
        return self.a.n_rows

    def in_degrees(self):
        return self._in

    def out_degrees(self):
        return self._out


def halo_aggregate(g: PartitionGraph, x_halo: torch.Tensor, y: torch.Tensor, rs, cs_halo) -> None:
    """``y += rs * A_out[:, sampled] (cs_halo * x_halo)``.  With the epoch's compaction (the default) the kernel walks
    the sampled entries only; without it (a graph whose slot map was set by hand) every halo entry is looked up."""
    c = g.compact
    if c is not None and (c.cw is not None) == (cs_halo is not None):
        ops.spmm_compact(c, x_halo, y, row_scale=rs, accumulate=True)
    else:
        ops.spmm(g.a_out, x_halo, y, row_scale=rs, col_scale=cs_halo, col_map=g.slot, n_direct=0, accumulate=True)


class PartitionAggregate(torch.autograd.Function):
    """K1 + K2 (+ K1b in backward) on a ``PartitionGraph``:

        Y = rs * ( A_in (cs_in * H_U[:n_in])  +  A_out[:, sampled] (cs_halo * H_U[n_in:]) )

    The inner-edge pass only needs the local rows, so it is issued first; the halo pass waits for the exchange
    (``ready`` event recorded by ``Buffer.update(..., overlap=True)``) -- that is the comm/compute overlap.
    """

    @staticmethod
    def forward(ctx, h_u, g: PartitionGraph, rs, cs_in, cs_halo, ready):
        ctx.g, ctx.rs, ctx.cs_in, ctx.cs_halo = g, rs, cs_in, cs_halo
        ctx.n_u = h_u.shape[0]
        h_u = h_u.contiguous()
        # a per-source scale is applied ONCE per row here, not once per edge inside the gather (each source row is
        # gathered ~degree times; the fused col_scale path costs an extra scalar gather per edge)
        x_in = h_u[:g.n_in] if cs_in is None else h_u[:g.n_in] * cs_in.unsqueeze(1)
        y = ops.spmm_auto(g.a_in, x_in, row_scale=rs)
        if ready is not None:
            torch.cuda.current_stream(h_u.device).wait_event(ready)
        if g.a_out is not None and ctx.n_u > g.n_in:
            halo_aggregate(g, h_u[g.n_in:], y, rs, cs_halo)
        return y

    @staticmethod
    def backward(ctx, dy):
        g = ctx.g
        dy = dy.contiguous() if ctx.rs is None else dy * ctx.rs.unsqueeze(1)      # pre-scale once (see forward)
        du = torch.empty(ctx.n_u, dy.shape[1], dtype=torch.float32, device=dy.device)
        if ctx.n_u > g.n_in:
            tail = du[g.n_in:]
            tail.zero_()
            if g.a_out_t is not None:
                ops.spmm(g.a_out_t, dy, tail, row_scale=ctx.cs_halo, row_map=g.slot)
        ops.spmm_auto(g.a_in_t, dy, du[:g.n_in], row_scale=ctx.cs_in)
        return du, None, None, None, None, None


def _entry_rows(a: ops.DeviceGraph):
    """(row id, column id) of every CSR entry of ``a`` as int64 vectors (static, built once)."""
    indptr, indices = a.csr()
    rows = torch.repeat_interleave(torch.arange(a.n_rows, device=indptr.device), indptr[1:] - indptr[:-1])
    return rows, indices.long()


def gat_entries(g: PartitionGraph):
    """Static per-entry index vectors the attention scores are computed on (rows / cols of a_in and a_out)."""
    if getattr(g, "_gat_entries", None) is None:
        rin, cin = _entry_rows(g.a_in)
        if g.a_out is not None:
            rout, cout = _entry_rows(g.a_out)
        else:
            rout = cout = torch.empty(0, dtype=torch.int64, device=g.device)
        g._gat_entries = (rin, cin, rout, cout)
    return g._gat_entries


class WeightedAggregate(torch.autograd.Function):
    """``rst[v] = sum_k w_k * ft_u[xrow(c_k)]`` over the inner entries (weights ``w_in``) and the sampled halo entries
    (``w_out``; unsampled entries are skipped through the slot map) -- DGL's ``update_all(u_mul_e, sum)`` of GATConv.
    Backward: ``d ft = A_w^T d rst`` (weights carried to the transposes by their entry permutation) and
    ``d w_k = <d rst[v], ft_u[xrow(c_k)]>`` (``bns_sddmm_dot_f32``)."""

    @staticmethod
    def forward(ctx, ft_u, w_in, w_out, g: PartitionGraph):
        ft_u, w_in, w_out = ft_u.contiguous(), w_in.contiguous(), w_out.contiguous()
        ctx.g = g
        ctx.save_for_backward(ft_u, w_in, w_out)
        y = ops.spmm(g.a_in, ft_u, edge_weight=w_in)
        if g.a_out is not None and ft_u.shape[0] > g.n_in:
            ops.spmm(g.a_out, ft_u[g.n_in:], y, edge_weight=w_out, col_map=g.slot, n_direct=0, accumulate=True)
        return y

    @staticmethod
    def backward(ctx, dy):
        g = ctx.g
        ft_u, w_in, w_out = ctx.saved_tensors
        dy = dy.contiguous()
        n_u, n_in = ft_u.shape[0], g.n_in
        d_ft = torch.empty_like(ft_u)
        ops.spmm(g.a_in_t, dy, d_ft[:n_in], edge_weight=w_in[g.a_in_t.perm().long()])
        d_w_in = ops.sddmm_dot(g.a_in, dy, ft_u)
        d_w_out = torch.zeros_like(w_out)
        if n_u > n_in:
            tail = d_ft[n_in:]
            tail.zero_()
            if g.a_out_t is not None:
                ops.spmm(g.a_out_t, dy, tail, edge_weight=w_out[g.a_out_t.perm().long()], row_map=g.slot)
                ops.sddmm_dot(g.a_out, dy, ft_u[n_in:], col_map=g.slot, n_direct=0, out=d_w_out)
        return d_ft, d_w_in, d_w_out, None


_PROJ_WS = {}


class GatProjection(torch.autograd.Function):
    """``el = <ft_src, attn_l>``, ``er = <ft_dst, attn_r>`` per head (the two ``(feat * attn).sum(-1)`` of
    ``dgl.nn.GATConv``) on ``bns_gat_proj_f32``; the backward (``bns_gat_proj_bwd_f32``) makes ``d ft = s (x) attn`` and
    the deterministic ``d attn = sum_r s_r ft_r`` in one pass over ``ft`` each."""

    @staticmethod
    def forward(ctx, ft_src, ft_dst, attn_l, attn_r, H: int, Fo: int):
        from ._lib import check, lib
        ft_src, ft_dst = ft_src.contiguous(), ft_dst.contiguous()
        al, ar = attn_l.reshape(-1).contiguous(), attn_r.reshape(-1).contiguous()
        dev = ft_src.device
        el = torch.empty(ft_src.shape[0], H, dtype=torch.float32, device=dev)
        er = torch.empty(ft_dst.shape[0], H, dtype=torch.float32, device=dev)
        st = torch.cuda.current_stream(dev).cuda_stream
        with torch.cuda.device(dev):
            check(lib.bns_gat_proj_f32(ft_src.data_ptr(), ft_src.stride(0), ft_src.shape[0], H, Fo, al.data_ptr(), el.data_ptr(),
                                       st), "bns_gat_proj_f32")
            check(lib.bns_gat_proj_f32(ft_dst.data_ptr(), ft_dst.stride(0), ft_dst.shape[0], H, Fo, ar.data_ptr(), er.data_ptr(),
                                       st), "bns_gat_proj_f32")
        ctx.save_for_backward(ft_src, ft_dst, al, ar)
        ctx.cfg = (H, Fo, attn_l.shape)
        return el, er

    @staticmethod
    def backward(ctx, d_el, d_er):
        from ._lib import check, lib
        ft_src, ft_dst, al, ar = ctx.saved_tensors
        H, Fo, shape = ctx.cfg
        dev = ft_src.device
        st = torch.cuda.current_stream(dev).cuda_stream
        key = (dev, H * Fo, st)
        ws = _PROJ_WS.get(key)
        if ws is None:
            ws = _PROJ_WS[key] = torch.empty(lib.bns_colsum_workspace_bytes(H * Fo), dtype=torch.uint8, device=dev)
        outs = []
        with torch.cuda.device(dev):
            for ft, a, s in ((ft_src, al, d_el), (ft_dst, ar, d_er)):
                s = s.contiguous()
                d_ft = torch.empty_like(ft)
                d_a = torch.empty_like(a)
                check(lib.bns_gat_proj_bwd_f32(ft.data_ptr(), ft.stride(0), ft.shape[0], H, Fo, a.data_ptr(), s.data_ptr(),
                                               d_ft.data_ptr(), d_ft.stride(0), 0, d_a.data_ptr(), ws.data_ptr(), ws.numel(),
                                               st), "bns_gat_proj_bwd_f32")
                outs.append((d_ft, d_a.view(shape)))
        return outs[0][0], outs[1][0], outs[0][1], outs[1][1], None, None


class GatAttention(torch.autograd.Function):
    """The attention of ``dgl.nn.GATConv`` for all heads:

        rst_v = sum_u attn_drop(edge_softmax(leaky_relu(el_u + er_v)))_uv * ft_u

    over the inner entries and this epoch's sampled halo entries (the partition graph's compaction with positions).
    ``ft [n_u, H * Fo]``, ``el [n_u, H]``, ``er [n_in, H]`` -> ``[n_in, H * Fo]``; gradients for all three.

    Stages (include/bnsgcn.h): ``bns_gat_scores_f32`` (scalars: probabilities + dropped attention per entry) ->
    ``bns_spmm_weighted_f32`` / ``bns_spmm_compact_f32`` per head; backward ``bns_sddmm_dot_f32`` ->
    ``bns_gat_softmax_bwd_f32`` -> ``bns_gat_colsum_f32`` -> ``bns_spmm_weighted_f32`` on the transposes."""

    @staticmethod
    def forward(ctx, ft, el, er, g: PartitionGraph, H: int, Fo: int, slope: float, p: float, seed: int):
        from ._lib import check, lib
        ft, el, er = ft.contiguous(), el.contiguous(), er.contiguous()
        n_in, dev = g.n_in, ft.device
        c = g.compact if (g.a_out is not None and ft.shape[0] > n_in) else None
        if c is not None and c.cpos is None:
            raise RuntimeError("GatAttention: the partition graph was compacted without positions (want_positions)")
        rst = torch.empty(n_in, H * Fo, dtype=torch.float32, device=dev)
        p_in = torch.empty(max(g.a_in.nnz, 1), H, dtype=torch.float32, device=dev)
        p_out = torch.empty(max(g.a_out.nnz, 1), H, dtype=torch.float32, device=dev) if c is not None else None
        off, off_dev = ops.RNG["offset"], ops.RNG["offset_dev"]
        head = (g.a_in._h, None if c is None else g.a_out._h, None if c is None else c.cidx.data_ptr(),
                None if c is None else c.chunk_cnt.data_ptr(), None if c is None else c.cpos.data_ptr(), n_in)
        tail = (H, el.data_ptr(), er.data_ptr(), float(slope), float(p), seed & (2 ** 64 - 1), off & (2 ** 64 - 1),
                ops._ptr(off_dev))
        st = torch.cuda.current_stream(dev).cuda_stream
        w_in = w_out = None
        if p > 0:
            w_in = torch.empty_like(p_in)
            w_out = torch.empty_like(p_out) if p_out is not None else None
        wc = torch.empty_like(p_out) if p_out is not None else None          # halo attention, compacted positions
        with torch.cuda.device(dev):
            check(lib.bns_gat_scores_f32(*head, *tail, p_in.data_ptr(), ops._ptr(p_out), ops._ptr(w_in), ops._ptr(w_out),
                                         ops._ptr(wc), st), "bns_gat_scores_f32")
        for h in range(H):
            cols = slice(h * Fo, (h + 1) * Fo)
            ops.spmm_weighted(g.a_in, ft[:n_in, cols], rst[:, cols], p_in if w_in is None else w_in, h)
            if c is not None:
                ops.spmm_compact(c, ft[n_in:, cols], rst[:, cols], accumulate=True, weights=wc, head=h)
        ctx.g, ctx.c, ctx.head, ctx.tail, ctx.cfg = g, c, head, tail, (H, Fo, float(p))
        saved = [ft, el, er, p_in] + ([p_out] if p_out is not None else [])
        if w_in is not None:
            saved += [w_in] + ([w_out] if w_out is not None else [])
        ctx.n_w = 0 if w_in is None else (2 if w_out is not None else 1)
        ctx.save_for_backward(*saved)
        return rst

    @staticmethod
    def backward(ctx, d_rst):
        from ._lib import check, lib
        g, c = ctx.g, ctx.c
        H, Fo, p = ctx.cfg
        ft, el, er, p_in, *rest = ctx.saved_tensors
        p_out = rest.pop(0) if c is not None else None
        d_rst = d_rst.contiguous()
        dev, n_in, n_u = ft.device, g.n_in, ft.shape[0]
        de_in = torch.empty_like(p_in)
        de_out = torch.empty_like(p_out) if p_out is not None else None
        d_er = torch.empty(n_in, H, dtype=torch.float32, device=dev)
        st = torch.cuda.current_stream(dev).cuda_stream
        w_in, w_out = p_in, p_out
        if ctx.n_w:
            w_in = rest.pop(0)
            w_out = rest.pop(0) if ctx.n_w == 2 else None
        for h in range(H):                                 # d a'_uv = <d rst_v, ft_u> (0 for an unsampled halo node)
            cols = slice(h * Fo, (h + 1) * Fo)
            ops.sddmm_dot(g.a_in, d_rst[:, cols], ft[:n_in, cols], out=de_in[:, h])
            if c is not None:
                ops.sddmm_dot(g.a_out, d_rst[:, cols], ft[n_in:, cols], col_map=g.slot, n_direct=0, out=de_out[:, h])
        with torch.cuda.device(dev):
            check(lib.bns_gat_softmax_bwd_f32(*ctx.head, *ctx.tail, p_in.data_ptr(), ops._ptr(p_out), de_in.data_ptr(),
                                              ops._ptr(de_out), d_er.data_ptr(), st), "bns_gat_softmax_bwd_f32")
        with torch.cuda.device(dev):
            d_el = torch.empty(n_u, H, dtype=torch.float32, device=dev)
            check(lib.bns_gat_colsum_f32(g.a_in_t._h, de_in.data_ptr(), H, None, 0, d_el.data_ptr(), st),
                  "bns_gat_colsum_f32")
            if c is not None:
                check(lib.bns_gat_colsum_f32(g.a_out_t._h, de_out.data_ptr(), H, g.slot.data_ptr(), n_in, d_el.data_ptr(),
                                             st), "bns_gat_colsum_f32")
        d_ft = torch.empty(n_u, H * Fo, dtype=torch.float32, device=dev)
        for h in range(H):
            cols = slice(h * Fo, (h + 1) * Fo)
            ops.spmm_weighted(g.a_in_t, d_rst[:, cols], d_ft[:n_in, cols], w_in, h, through_perm=True)
            if c is not None:
                ops.spmm_weighted(g.a_out_t, d_rst[:, cols], d_ft[n_in:, cols], w_out, h, through_perm=True,
                                  row_map=g.slot)
        return d_ft, d_el, d_er, None, None, None, None, None, None
