"""``GATConv``: the layer ``module/model.py:102`` takes from ``dgl.nn.GATConv`` (DGL 0.9, README.md:41; not
vendored with the reference).  Same constructor arguments, parameter names (``fc.weight``, ``attn_l``, ``attn_r``,
``bias``), initialisation (xavier-normal with the ReLU gain, zero bias) and forward contract as DGL's layer for the
call the reference makes -- ``layer(g, (h_src, h_dst))`` on the bipartite ``_U -> _V`` graph in training:

    ft = fc(feat_drop(h))            el = <ft_src, attn_l>      er = <ft_dst, attn_r>
    e_uv = leaky_relu(el_u + er_v)   a = attn_drop(edge_softmax(e))     rst_v = sum_u a_uv ft_u + bias

Everything after ``fc`` runs as kernels of libbnsgcn.so (``graph.GatProjection``, ``graph.GatAttention``; feature
dropout on the Philox kernel).  The op-by-op fallback (a per-head width that is not a multiple of 4) writes the
per-entry score / softmax algebra as torch ops on ``[nnz, heads]`` vectors over the STATIC entry lists of the
partition graph (an unsampled halo entry gets e = -inf, i.e. weight 0) around the weighted SpMM, its transpose and the
SDDMM-dot of the attention gradient (``graph.WeightedAggregate``)."""
import torch
import torch.nn.functional as F
from torch import nn

from .. import fused, ops
from ..graph import GatAttention, GatProjection, PartitionGraph, WeightedAggregate, gat_entries
from . import dense


class GATConv(nn.Module):

    def __init__(self, in_feats, out_feats, num_heads, feat_drop=0., attn_drop=0., negative_slope=0.2,
                 residual=False, activation=None, allow_zero_in_degree=False, bias=True):
        super(GATConv, self).__init__()
        if residual or activation is not None:
            raise NotImplementedError("the reference constructs GATConv(in, out, heads, dropout, dropout) only")
        self._num_heads, self._in_feats, self._out_feats = num_heads, in_feats, out_feats
        self.fc = nn.Linear(in_feats, out_feats * num_heads, bias=False)
        self.attn_l = nn.Parameter(torch.empty(1, num_heads, out_feats))
        self.attn_r = nn.Parameter(torch.empty(1, num_heads, out_feats))
        self.feat_drop = nn.Dropout(feat_drop)
        self.attn_drop = nn.Dropout(attn_drop)
        self.negative_slope = negative_slope
        self.bias = nn.Parameter(torch.empty(num_heads * out_feats)) if bias else None
        self.reset_parameters()

    def reset_parameters(self):
        gain = nn.init.calculate_gain('relu')
        nn.init.xavier_normal_(self.fc.weight, gain=gain)
        nn.init.xavier_normal_(self.attn_l, gain=gain)
        nn.init.xavier_normal_(self.attn_r, gain=gain)
        if self.bias is not None:
            nn.init.constant_(self.bias, 0)

    def forward(self, graph, feat):
        if not isinstance(graph, PartitionGraph) or not isinstance(feat, tuple):
            raise NotImplementedError("GATConv: only the training call layer(g, (h_src, h_dst)) of the reference")
        H, Fo = self._num_heads, self._out_feats
        n_in = graph.n_in
        ready = getattr(feat[0], '_bns_ready', None)
        if ready is not None:          # every row of h_src is read below: wait for the overlapped exchange
            torch.cuda.current_stream(feat[0].device).wait_event(ready)
        # the attention (u_add_v, leaky_relu, edge_softmax, attn_drop, u_mul_e + sum of DGL's GATConv) as kernels
        # (graph.GatAttention); per-head widths that are not multiples of 4: the op-by-op torch path below
        kernels = Fo % 4 == 0 and H <= 8 and H * Fo <= 1024 and \
            (graph.a_out is None or (graph.compact is not None and graph.compact.cpos is not None))
        salt = ops.RNG["seed"] + 15485863 * (1 + getattr(self, "_layer_index", 0))
        pf = self.feat_drop.p if self.training else 0.0
        if kernels and pf > 0 and fused.dropout_supported(feat[0]) and fused.dropout_supported(feat[1]):
            # two independent masks, as DGL draws them (feat_drop is applied to the source and the destination rows)
            h_src, h_dst = fused.DropoutFn.apply(feat[0], pf, salt + 1), fused.DropoutFn.apply(feat[1], pf, salt + 2)
        else:
            h_src, h_dst = self.feat_drop(feat[0]), self.feat_drop(feat[1])
        ft_src = dense.linear(h_src, self.fc.weight).view(-1, H, Fo)
        ft_dst = dense.linear(h_dst, self.fc.weight).view(-1, H, Fo)
        if kernels:
            # el / er, score -> edge softmax -> dropout -> weighted aggregation (and their backward) as kernels
            ft2 = ft_src.reshape(-1, H * Fo)
            el, er = GatProjection.apply(ft2, ft_dst.reshape(-1, H * Fo), self.attn_l, self.attn_r, H, Fo)
            p = self.attn_drop.p if self.training else 0.0
            rst = GatAttention.apply(ft2, el, er, graph, H, Fo, self.negative_slope, p, salt)
            if self.bias is not None:
                rst += self.bias                                    # in place: the attention saved nothing of it
            return rst.view(-1, H, Fo)
        el = (ft_src * self.attn_l).sum(dim=-1)                     # [n_U, H]
        er = (ft_dst * self.attn_r).sum(dim=-1)                     # [n_in, H]
        rin, cin, rout, cout = gat_entries(graph)
        e_in = F.leaky_relu(el[cin] + er[rin], self.negative_slope)                                  # [nnz_in, H]
        n_u = ft_src.shape[0]
        if rout.numel() and n_u > n_in:
            xrow = graph.slot.long()[cout]                                                           # -1 = unsampled
            valid = (xrow >= 0).unsqueeze(1)
            e_out = F.leaky_relu(el[n_in + xrow.clamp(min=0)] + er[rout], self.negative_slope)
            e_out = torch.where(valid, e_out, torch.full_like(e_out, float('-inf')))
        else:
            rout = cout = rout[:0]
            e_out = e_in.new_empty(0, H)
        # edge softmax over each destination's in-entries (inner + sampled halo)
        m = torch.full((n_in, H), float('-inf'), device=e_in.device)
        m = m.scatter_reduce(0, rin.unsqueeze(1).expand(-1, H), e_in.detach(), 'amax')
        if e_out.numel():
            m = m.scatter_reduce(0, rout.unsqueeze(1).expand(-1, H), e_out.detach(), 'amax')
        ex_in = torch.exp(e_in - m[rin])
        ex_out = torch.exp(e_out - m[rout]) if e_out.numel() else e_out
        den = torch.zeros(n_in, H, device=e_in.device).index_add(0, rin, ex_in)
        if e_out.numel():
            den = den.index_add(0, rout, ex_out)
        a_in = self.attn_drop(ex_in / den[rin])
        a_out = self.attn_drop(ex_out / den[rout]) if e_out.numel() else ex_out
        # weighted aggregation, one head at a time (16-byte lanes need the per-head width padded to 4)
        pad = (-Fo) % 4
        outs = []
        for h in range(H):
            ft_h = ft_src[:, h, :]
            if pad:
                ft_h = F.pad(ft_h, (0, pad))
            w_out_h = a_out[:, h] if a_out.numel() else a_in.new_empty(graph.a_out.nnz if graph.a_out is not None else 0)
            if a_out.numel() == 0 and graph.a_out is not None:
                w_out_h = a_in.new_zeros(graph.a_out.nnz)
            r = WeightedAggregate.apply(ft_h.contiguous(), a_in[:, h], w_out_h, graph)
            outs.append(r[:, :Fo])
        rst = torch.stack(outs, dim=1)                              # [n_in, H, Fo]
        if self.bias is not None:
            rst = rst + self.bias.view(1, H, Fo)
        return rst
