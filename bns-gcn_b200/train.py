"""The training driver: same function names and call order as the reference's train.py, on the DGL-free
partition contract and the CUDA path.

``run(graph, node_dict, gpb, args)`` is the reference entry point (train.py:300-456).  It is split into
``setup(...) -> TrainState`` and ``train_epoch(state, epoch)`` so that bench.py / tests can time or inspect single
epochs; ``run`` is the loop around them with the reference's log line.
"""
from __future__ import annotations

import dataclasses
import time
from typing import List, Optional

import numpy as np
import torch
import torch.nn.functional as F

from . import ops
from .data.partition import NID, LocalGraph
from .graph import FullGraphHandle, PartitionGraph
from .helper import context as ctx
from .helper.timer.timer import comm_timer
from .helper.utils import (TransferTag, data_transfer, get_boundary, get_layer_size, merge_feature, minus_one_tensor,
                           nonzero_idx, print_memory)
from .module.model import GAT, GCN, GraphSAGE


def _rank_size():
    c = ctx.comm()
    return c.rank, c.size


def calc_acc(logits, labels):
    """train.py:13-19 (micro-F1 for multi-label without sklearn's host round trip)."""
    if labels.dim() == 1:
        return (logits.argmax(dim=1) == labels).sum().item() / labels.shape[0]
    pred = logits > 0
    tp = (pred & (labels > 0)).sum().item()
    fp = (pred & ~(labels > 0)).sum().item()
    fn = (~pred & (labels > 0)).sum().item()
    return 2 * tp / max(2 * tp + fp + fn, 1)


def move_to_cuda(graph, in_graph, out_graph, node_dict, boundary, device=None):
    """train.py:64-74.  ``in_graph`` / ``out_graph`` are already device-resident ``DeviceGraph`` s."""
    rank, size = _rank_size()
    dev = torch.device(device if device is not None else torch.cuda.current_device())
    for i in range(size):
        if i != rank:
            boundary[i] = boundary[i].to(dev)
    for key in node_dict.keys():
        node_dict[key] = node_dict[key].to(dev)
    return graph, in_graph, out_graph, node_dict, boundary


def get_in_out_graph(graph: LocalGraph, node_dict, device=None, chunk_nnz: int = 0):
    """train.py:77-87.  ``in_graph``: edges between inner nodes; ``out_graph``: edges halo -> inner (stored with
    halo-local column ids ``src - n_in``).  Both become static CSR matrices in HBM, int32 ids (train.py:71-73)."""
    dev = torch.device(device if device is not None else torch.cuda.current_device())
    n_in = graph.n_in
    indptr, idx = graph.indptr.to(dev), graph.indices.to(dev)
    inner = idx < n_in
    rows = torch.repeat_interleave(torch.arange(n_in, device=dev), indptr[1:] - indptr[:-1])

    def csr_of(mask, shift):
        cnt = torch.bincount(rows[mask], minlength=n_in)
        ip = torch.zeros(n_in + 1, dtype=torch.int64, device=dev)
        ip[1:] = torch.cumsum(cnt, 0)
        return ip, (idx[mask] - shift).to(torch.int32)

    ip_in, ix_in = csr_of(inner, 0)
    in_graph = ops.DeviceGraph.from_csr(ip_in, ix_in, n_in, chunk_nnz)
    out_graph = None
    if graph.n_halo > 0:
        ip_out, ix_out = csr_of(~inner, n_in)
        out_graph = ops.DeviceGraph.from_csr(ip_out, ix_out, graph.n_halo, chunk_nnz)
    return in_graph, out_graph


def get_pos(node_dict, gpb):
    """train.py:90-104: ``pos[i][owner-local id] = my local id`` of that node, -1 if it is not one of my halo nodes."""
    rank, size = _rank_size()
    dev = node_dict['part_id'].device
    pos = []
    for i in range(size):
        if i == rank:
            pos.append(None)
            continue
        start, end = int(gpb.ranges[i]), int(gpb.ranges[i + 1])
        p = minus_one_tensor(end - start, dev)
        in_idx = nonzero_idx(node_dict['part_id'] == i)
        p[node_dict[NID][in_idx] - start] = in_idx
        pos.append(p)
    return pos


def get_send_size(boundary, prob):
    """train.py:107-119.  An empty boundary makes the reference divide by zero; here it sends nothing at ratio 1."""
    rank, size = _rank_size()
    res, ratio = [], []
    for i, b in enumerate(boundary):
        if i == rank:
            res.append(0)
            ratio.append(0)
            continue
        s = int(prob * b.shape[0])
        res.append(s)
        ratio.append(s / b.shape[0] if b.shape[0] else 1.0)
    return res, ratio


def get_recv_size(node_dict, prob):
    """train.py:122-131."""
    rank, size = _rank_size()
    counts = torch.bincount(node_dict['part_id'], minlength=size).tolist()
    return [0 if i == rank else int(prob * counts[i]) for i in range(size)]


def _halo_counts(node_dict):
    rank, size = _rank_size()
    counts = torch.bincount(node_dict['part_id'], minlength=size).tolist()
    return [None if i == rank else counts[i] for i in range(size)]


def collect_out_degree(node_dict, boundary):
    """train.py:148-167: out-degrees of my halo nodes, fetched from their owners -> ``[inner | halo]`` vector."""
    rank, size = _rank_size()
    out_deg = node_dict['out_deg']
    if size == 1:
        return out_deg
    send_info = [None if i == rank else out_deg[b] for i, b in enumerate(boundary)]
    recv_shape = [None if c is None else torch.Size([c]) for c in _halo_counts(node_dict)]
    recv_out_deg = data_transfer(send_info, recv_shape, tag=TransferTag.DEG, dtype=torch.long)
    return merge_feature(out_deg, recv_out_deg)


def select_node(boundary, send_size, sampler: Optional[ops.BoundarySampler] = None, seed: int = 0, epoch: int = 0):
    """train.py:225-236 (K6).  The reference draws ``np.random.choice(b, k, replace=False)`` per peer on the host
    and copies the ids to the GPU; here one Philox kernel draws all peers' samples on the device."""
    if sampler is None:
        dev = next(b for b in boundary if b is not None).device
        sampler = ops.BoundarySampler(boundary, send_size, dev)
    return sampler.sample(seed, epoch)[1]


def construct_graph(part: PartitionGraph, graph, pos, one_hops, hops_cat=None):
    """train.py:256-281 (K7).  Instead of a new heterograph: refresh the slot map of the static graph.
    U-numbering = ``[inner | sampled halo of peer 0 | peer 1 ...]`` in the order of the received ``one_hops``.
    ``hops_cat`` (the received lists as ONE tensor, from ``Buffer.exchange_ids``): all peers in one launch, together
    with the inverse maps of the gradient scatter (``Buffer.update_maps``); otherwise one small launch per peer.
    Either way the halo matrix is then compacted to this epoch's sampled columns."""
    rank, size = _rank_size()
    tot = part.n_in
    if hops_cat is not None:
        buf = ctx.buffer._get()
        buf.update_maps(buf._selected_cat, hops_cat, part.slot)
        tot += int(hops_cat.shape[0])
    else:
        if part.n_halo:
            ops.fill_i32(part.slot, -1)
        for i in range(size):
            if i == rank:
                continue
            u = one_hops[i]
            if u is None or u.shape[0] == 0:
                continue
            ops.halo_slot_update(pos[i], u, part.n_in, tot - part.n_in, part.slot)
            tot += u.shape[0]
    part.n_u = tot
    if size > 1:
        part.refresh_compaction()
    return part


def order_graph(part, graph, gpb, node_dict, pos):
    """train.py:134-145: the full-halo graph (every halo node present, sorted by owner-local id)."""
    rank, size = _rank_size()
    one_hops = []
    for i in range(size):
        if i == rank:
            one_hops.append(None)
            continue
        nodes = node_dict[NID][node_dict['part_id'] == i] - int(gpb.ranges[i])
        one_hops.append(torch.sort(nodes)[0])
    return construct_graph(part, graph, pos, one_hops)


def construct_out_norm(num, norm, pos, one_hops):
    """train.py:245-253 rebuilds a U-ordered ``out_norm`` per epoch; the slot map makes that unnecessary --
    ``GCNLayer`` takes the static ``[inner | halo]`` vector, so this returns it unchanged."""
    return norm


def construct_feat(num, feat, pos, one_hops):
    """train.py:284-297 (GAT layer 0): ``[inner features | stored features of this epoch's sampled halo nodes]``."""
    rank, size = _rank_size()
    res = [feat[0:num]]
    for i in range(size):
        if i == rank:
            continue
        u = one_hops[i]
        if u is None or u.shape[0] == 0:
            continue
        res.append(feat[pos[i][u]])
    return torch.cat(res)


def precompute(part: PartitionGraph, graph, node_dict, boundary, model, gpb, pos, out_deg_all=None):
    """train.py:170-211: the one-time layer-0 aggregation over ALL boundary nodes (sampling rate 1)."""
    rank, size = _rank_size()
    g = order_graph(part, graph, gpb, node_dict, pos)
    feat = node_dict['feat']
    if size > 1:
        send_info = [None if i == rank else feat[b] for i, b in enumerate(boundary)]
        recv_shape = [None if c is None else torch.Size([c, feat.shape[1]]) for c in _halo_counts(node_dict)]
        recv_feat = data_transfer(send_info, recv_shape, tag=TransferTag.FEAT, dtype=torch.float)
    else:
        recv_feat = [None]
    h_u = merge_feature(feat, recv_feat)
    n_feat = feat.shape[1]
    pad = (-n_feat) % 4                       # 16-byte vector path of the SpMM (602 -> 604 columns)
    if pad:
        h_u = F.pad(h_u, (0, pad))
    from .graph import PartitionAggregate
    with torch.no_grad():
        if model == 'gcn':
            in_norm = torch.sqrt(node_dict['in_deg'].float())
            out_norm = torch.sqrt(out_deg_all.float())
            cs = 1.0 / out_norm
            h = PartitionAggregate.apply(h_u, g, 1.0 / in_norm, cs[:g.n_in].contiguous(), cs[g.n_in:].contiguous(), None)
            return h[:, :n_feat].contiguous()
        elif model == 'graphsage':
            # fn.mean divides by the number of messages = the full in-degree (every in-edge is present here)
            mean = PartitionAggregate.apply(h_u, g, 1.0 / node_dict['in_deg'].float(), None, None, None)
            return torch.cat([feat, mean[:, :n_feat]], dim=1)
        elif model == 'gat':
            return h_u[:, :n_feat]
        raise Exception


def precompute_streaming(part: PartitionGraph, node_dict, boundary, model):
    """``precompute`` for GraphSAGE without ever materialising the full halo feature matrix (train.py:189, :202 fetch the
    features of ALL boundary nodes at once: ~42 GB per rank on the papers100M shape under a random partition).  The halo
    columns of ``a_out`` are grouped by owner, so the aggregation is a sum over peers: step i of the reference's ring
    (helper/utils.py:204-206) receives the rows of ONE peer, multiplies them with that peer's column block of ``a_out``
    (accumulating), and frees both.  Peak extra memory: one peer's rows + one column block."""
    rank, size = _rank_size()
    if model != 'graphsage':
        raise NotImplementedError("precompute_streaming: GraphSAGE only (GCN needs the out-degrees too, GAT keeps the rows)")
    feat = node_dict['feat']
    n_in, n_feat = feat.shape
    pad = (-n_feat) % 4
    x_in = F.pad(feat, (0, pad)) if pad else feat
    c = ctx.comm()
    with torch.no_grad():
        acc = ops.spmm_auto(part.a_in, x_in)                                     # raw sums over the inner edges
        if size > 1 and part.a_out is not None and part.a_out.nnz:
            counts = _halo_counts(node_dict)
            first = [0] * size                                                   # first halo column of each owner
            tot = 0
            for j in range(size):
                first[j] = tot
                tot += 0 if j == rank else counts[j]
            ip, ix = part.a_out.csr()
            rows = torch.repeat_interleave(torch.arange(n_in, device=feat.device), ip[1:] - ip[:-1])
            for i in range(1, size):
                right, left = (rank + i) % size, (rank - i + size) % size
                send = [None] * size
                recv = [None] * size
                send[right] = x_in[boundary[right]]
                recv[left] = torch.empty(counts[left], x_in.shape[1], dtype=torch.float32, device=feat.device)
                c.alltoall(send, recv, tag=TransferTag.FEAT * 1000 + i)
                m = (ix >= first[left]) & (ix < first[left] + counts[left])
                ipb = torch.zeros(n_in + 1, dtype=torch.int64, device=feat.device)
                ipb[1:] = torch.cumsum(torch.bincount(rows[m], minlength=n_in), 0)
                blk = ops.DeviceGraph.from_csr(ipb, (ix[m] - first[left]).to(torch.int32), counts[left])
                ops.spmm(blk, recv[left], acc, accumulate=True)
                torch.cuda.current_stream(feat.device).synchronize()             # the block and the rows die here
                del blk, recv, send, m, ipb
        from . import fused
        mean = fused.scale_rows(acc, 1.0 / node_dict['in_deg'].float())
    return torch.cat([feat, mean[:, :n_feat]], dim=1)


def create_model(layer_size, args):
    """train.py:214-222."""
    if args.model == 'gcn':
        return GCN(layer_size, F.relu, norm=args.norm, use_pp=args.use_pp, dropout=args.dropout,
                   train_size=args.n_train, n_linear=args.n_linear)
    elif args.model == 'graphsage':
        return GraphSAGE(layer_size, F.relu, norm=args.norm, use_pp=args.use_pp, dropout=args.dropout,
                         train_size=args.n_train, n_linear=args.n_linear)
    elif args.model == 'gat':
        return GAT(layer_size, F.relu, use_pp=True, heads=args.heads, norm=args.norm, dropout=args.dropout)
    raise NotImplementedError(args.model)


def reduce_hook(param, name, n_train):
    """train.py:239-242.  The rank's reducer is bound here: the hook fires on autograd's device thread."""
    red = ctx.reducer._get()

    def fn(grad):
        red.reduce(param, name, grad, n_train)
    return fn


@dataclasses.dataclass
class TrainState:
    args: object
    part: PartitionGraph
    model: torch.nn.Module
    optimizer: torch.optim.Optimizer
    loss_fcn: torch.nn.Module
    feat: torch.Tensor
    labels: torch.Tensor
    train_mask: torch.Tensor
    in_norm: torch.Tensor
    out_norm: Optional[torch.Tensor]
    boundary: list
    pos: list
    send_size: list
    recv_size: list
    ratio: list
    sampler: Optional[ops.BoundarySampler]
    part_train: int
    selected: Optional[list] = None
    one_hops: Optional[list] = None
    last_logits: Optional[torch.Tensor] = None
    epoch_dev: Optional[torch.Tensor] = None     # int64 [1] on the device: epochs started so far
    graph_mode: bool = False
    train_idx: Optional[torch.Tensor] = None     # nonzero(train_mask), computed once (mask indexing would sync)
    arena: Optional[object] = None               # fused.ParamArena when the fused training step is on


def _fused_eligible(args, layer_size, dev) -> bool:
    """The fused training step (fused.py) covers the BASELINE configuration families: GraphSAGE / GCN, --use-pp, LayerNorm +
    ReLU between the layers, no trailing linear layers, widths the 16-byte vector / TMA paths take.  Every other
    configuration runs the op-by-op autograd path."""
    if dev.type != "cuda":
        return False
    if args.model not in ('graphsage', 'gcn') or not args.use_pp or args.n_linear != 0 or args.norm != 'layer':
        return False
    k0 = 2 * layer_size[0] if args.model == 'graphsage' else layer_size[0]       # width of the precomputed layer-0 input
    widths_ok = k0 % 4 == 0 and all(w % 4 == 0 and w <= 1024 for w in layer_size[1:-1])
    return widths_ok and len(layer_size) >= 3


def setup(graph: LocalGraph, node_dict, gpb, args, device=None) -> TrainState:
    """Everything ``run`` does before its epoch loop (train.py:300-383)."""
    rank, size = _rank_size()
    dev = torch.device(device if device is not None else torch.cuda.current_device())
    node_dict = dict(node_dict)
    in_graph, out_graph = get_in_out_graph(graph, node_dict, dev, getattr(args, 'chunk_nnz', 0))
    part = PartitionGraph(graph.n_in, graph.n_halo, in_graph, out_graph, dev)
    part.want_positions = args.model == 'gat'          # the fused attention keeps per-entry values at CSR positions
    boundary = get_boundary({k: v.to(dev) for k, v in node_dict.items() if k in ('part_id', NID)}, gpb)
    layer_size = get_layer_size(args.n_feat, args.n_hidden, args.n_class, args.n_layers)
    _, _, _, node_dict, boundary = move_to_cuda(graph, in_graph, out_graph, node_dict, boundary, dev)
    print(f'Process {rank} has {graph.num_nodes()} nodes, {graph.num_edges()} edges '
          f'{in_graph.n_rows} inner nodes, and {in_graph.nnz} inner edges.')
    seed_lock = getattr(ctx.comm(), 'fabric', None)
    lock = seed_lock._lock if seed_lock is not None else None
    if lock is not None:
        lock.acquire()
    try:
        torch.manual_seed(args.seed)                                        # train.py:331-333
        model = create_model(layer_size, args)
    finally:
        if lock is not None:
            lock.release()
    model.to(dev)
    arena = None
    if _fused_eligible(args, layer_size, dev):
        from . import fused
        arena = fused.ParamArena(model)
        model._arena = arena
        ctx.reducer.init_arena(arena)
    else:
        ctx.reducer.init(model)
        for name, param in model.named_parameters():
            param.register_hook(reduce_hook(param, name, args.n_train))     # train.py:337-338
    labels = node_dict['label']
    part_train = int(node_dict['train_mask'].int().sum().item())
    pos = get_pos(node_dict, gpb)
    send_size, ratio = get_send_size(boundary, args.sampling_rate)
    recv_size = get_recv_size(node_dict, args.sampling_rate)
    ctx.buffer.init_buffer(in_graph.n_rows, ratio, send_size, recv_size,
                           layer_size[:args.n_layers - args.n_linear], use_pp=args.use_pp, backend=args.backend,
                           device=dev)
    if size > 1 and ctx.buffer._get()._p2p is not None:
        # slot map + the inverse maps of the gradient scatter in ONE allocation (one memset + one kernel per epoch)
        n_slot = max(graph.n_halo, 1)
        maps = torch.full((n_slot + (size - 1) * graph.n_in,), -1, dtype=torch.int32, device=dev)
        part.slot = maps[:n_slot]
        ctx.buffer._get().set_maps(maps, n_slot, pos)
    out_deg_all = collect_out_degree(node_dict, boundary)                   # train.py:350
    if args.use_pp:
        halo_bytes = graph.n_halo * node_dict['feat'].shape[1] * 4
        stream = getattr(args, 'streaming_precompute', None)
        if stream is None:                  # automatic: when all the halo rows together would not fit comfortably
            stream = args.model == 'graphsage' and halo_bytes > (16 << 30)
        if stream and args.model == 'graphsage':
            node_dict['feat'] = precompute_streaming(part, node_dict, boundary, args.model)
        else:
            node_dict['feat'] = precompute(part, graph, node_dict, boundary, args.model, gpb, pos, out_deg_all)
    if getattr(args, 'multilabel', False) or args.dataset == 'yelp':
        loss_fcn = torch.nn.BCEWithLogitsLoss(reduction='sum')              # train.py:358-361
    else:
        loss_fcn = torch.nn.CrossEntropyLoss(reduction='sum')
    if arena is not None:
        from . import fused
        optimizer = fused.FusedAdam(arena, lr=args.lr, weight_decay=args.weight_decay)
    else:
        # capturable: the step counter lives on the device, so the optimizer step can sit inside a CUDA graph
        optimizer = torch.optim.Adam(model.parameters(), lr=args.lr, weight_decay=args.weight_decay, capturable=True)
    out_norm = None
    if args.model == 'gcn':
        in_norm = torch.sqrt(node_dict['in_deg'].float())                   # train.py:377-378
        out_norm = torch.sqrt(out_deg_all.float())
        if graph.n_halo:
            part.halo_col_scale = part.recip(out_norm)[graph.n_in:].contiguous()
            part.compact = None
    else:
        in_norm = node_dict['in_deg']                                       # train.py:380 (unused by GAT)
    sampler = ops.BoundarySampler(boundary, send_size, dev) if size > 1 else None
    return TrainState(args, part, model, optimizer, loss_fcn, node_dict['feat'], labels, node_dict['train_mask'],
                      in_norm, out_norm, boundary, pos, send_size, recv_size, ratio, sampler, part_train,
                      epoch_dev=torch.zeros(1, dtype=torch.int64, device=dev),
                      train_idx=torch.nonzero(node_dict['train_mask'], as_tuple=True)[0], arena=arena)


def _forward_logits(st: TrainState, epoch: int, selected: Optional[list] = None) -> torch.Tensor:
    """train.py:388-402: sample the boundary, exchange the ids, refresh the graph, run the model (training mode)."""
    rank, size = _rank_size()
    args = st.args
    st.epoch_dev.add_(1)
    # Philox stream of this epoch's dropout masks (ops.LnReluDropout): (model seed, epoch index)
    ops.RNG["seed"] = int(getattr(args, 'seed', 0)) * 1000003 + rank
    if st.graph_mode:
        ops.RNG["offset"], ops.RNG["offset_dev"] = 2 ** 64 - 1, st.epoch_dev
    else:
        ops.RNG["offset"], ops.RNG["offset_dev"] = int(epoch), None
        comm_timer.clear()                  # train.py:425 (interval names are per epoch)
    hops_cat = None
    if size > 1:
        sel_cat = None
        if selected is None and st.graph_mode:
            # replayed from a CUDA graph: the Philox offset is (device epoch counter - 1), i.e. the same epoch
            # index an eager run passes as an immediate
            sel_cat, selected = st.sampler.sample(getattr(args, 'sampler_seed', 0), 2 ** 64 - 1, st.epoch_dev)
        elif selected is None:
            sel_cat, selected = st.sampler.sample(getattr(args, 'sampler_seed', 0), epoch)      # K6
        buf = ctx.buffer._get()
        buf.set_selected(selected, sel_cat)
        if buf.uses_p2p_ids():
            hops_cat, one_hops = buf.exchange_ids(buf._selected_cat)                            # C3 over peer memory
        else:
            recv_shape = [torch.Size([s]) for s in st.recv_size]
            one_hops = data_transfer(selected, recv_shape, tag=TransferTag.NODE, dtype=torch.long)  # C3
    else:
        selected, one_hops = [None], [None]
    st.selected, st.one_hops = selected, one_hops
    g = construct_graph(st.part, None, st.pos, one_hops, hops_cat)                              # K7
    st.model.train()
    if args.model == 'gcn':
        return st.model(g, st.feat, st.in_norm, st.out_norm)
    elif args.model == 'graphsage':
        return st.model(g, st.feat, st.in_norm)
    elif args.model == 'gat':
        return st.model(g, construct_feat(g.num_nodes('_V'), st.feat, st.pos, one_hops))        # train.py:401-402
    raise NotImplementedError


def train_epoch(st: TrainState, epoch: int, selected: Optional[list] = None) -> torch.Tensor:
    """One pass of the epoch body (train.py:388-413).  Returns the local sum-reduced loss (device scalar).
    ``selected`` injects the sampled sets (parity runs); by default they come from the Philox sampler."""
    logits = _forward_logits(st, epoch, selected)
    if st.arena is not None:
        # fused step: loss + d(logits) in one kernel (the 1/n_train of helper/reducer.py:34 rides on d(logits)), backward
        # through the layer functions (gradients land in the arena = the all-reduce bucket), one all-reduce, one Adam
        from . import fused
        pad = st.model._scratch.value
        loss, dl = fused.softmax_xent(pad.detach(), st.args.n_class, st.labels, st.train_mask, 1.0 / st.args.n_train)
        pad.backward(dl)
        ctx.reducer.synchronize()
        st.optimizer.step()
        st.last_logits = logits
        return loss
    # train.py:406 indexes with the boolean mask; the equivalent index list avoids a host sync per epoch
    loss = st.loss_fcn(logits[st.train_idx], st.labels[st.train_idx])
    st.optimizer.zero_grad(set_to_none=True)
    loss.backward()
    ctx.reducer.synchronize()
    st.optimizer.step()
    st.last_logits = logits
    return loss.detach()


def probe_loss(st: TrainState, epoch: int = 0, selected: Optional[list] = None) -> torch.Tensor:
    """The training-mode forward of ``epoch`` with every dropout switched off: no backward, no update, the epoch
    counter restored.  A loss that the CPU oracle (``OracleRank.epoch(forward_only=True)``) and any other arrangement
    of the same ranks (threads of one process / one process per GPU) must reproduce whatever the dropout rate of the
    run is -- bench.py prints it as ``parity_probe``."""
    drops = [(m, m.p) for m in st.model.modules() if isinstance(m, torch.nn.Dropout)]
    for m, _ in drops:
        m.p = 0.0
    try:
        with torch.no_grad():
            logits = _forward_logits(st, epoch, selected)
            loss = st.loss_fcn(logits[st.train_idx], st.labels[st.train_idx]).double().reshape(1)
    finally:
        for m, p_ in drops:
            m.p = p_
        st.epoch_dev.sub_(1)
    # the sum over ranks -- and the rendezvous that keeps a fast rank's NEXT exchange out of the slabs a slow rank is
    # still reading (a training epoch ends with the gradient all-reduce; a forward-only pass must bring its own)
    ctx.comm().all_reduce_sum(loss)
    return loss.detach()


class GraphedEpoch:
    """One whole training epoch -- boundary sampling, id exchange, slot-map refresh, forward (feature exchange on
    the comm stream + SpMM + dense), loss, backward (SpMM^T + gradient exchange), weight-gradient all-reduce, Adam --
    captured ONCE into a CUDA graph and replayed.  At 4-8 partitions of the Reddit-shape graph the eager epoch is
    bound by the ~10 ms the host needs to enqueue ~300 launches (profiles/kineto_n4_r01.txt); a replay costs one.

    What changes between replays is read from device memory, not baked into kernel arguments: the Philox offset of
    the sampler and the flag sequence number of the p2p exchange both come from ``st.epoch_dev``; dropout uses
    torch's graph-safe Philox state.  Sizes (sample counts, slab rows) are fixed for the run (train.py:344-345).
    """

    def __init__(self, st: TrainState, warmup: int = 3):
        self.st = st
        dev = st.feat.device
        cur = torch.cuda.current_stream(dev)
        if cur == torch.cuda.default_stream(dev):
            raise RuntimeError(
                "GraphedEpoch must be built -- and train.setup() must have run -- under `with torch.cuda.stream(s)` "
                "for one non-default stream s: autograd ties each parameter's gradient accumulator to the stream "
                "that was current when its hook was registered, and a capturing stream may not synchronise with the "
                "legacy default stream")
        # eager warm-up on the capture stream (allocator, cuBLAS workspaces, lazy kernel loads)
        for _ in range(warmup):
            train_epoch(st, int(st.epoch_dev.item()))
        torch.cuda.synchronize(dev)
        buf, red = ctx.buffer._get(), ctx.reducer._get()
        if _rank_size()[1] > 2 and getattr(buf, "_backend", None) == 'nccl':
            # Measured (tools/dist_check.py --graph, 4 x B200): the staged transport replayed from a graph is correct at
            # 2 ranks and WRONG at 4 (its NCCL send/recv batches sit on three streams of the captured graph); the
            # peer-mapped transport -- the default, flags in peer memory -- is bit-identical to the eager run at 2/4/8.
            raise NotImplementedError("GraphedEpoch with more than 2 partitions needs --backend p2p (the staged NCCL "
                                      "transport is only replay-safe at 2 ranks)")
        st.graph_mode = buf.graph_mode = red.graph_mode = True
        buf.seq_dev = st.epoch_dev
        # flag values of the replays: seq_base + epoch counter, strictly above every value the eager epochs (and any
        # forward-only probe) have already published
        # (the staged transport publishes no flags: its dict of sequence numbers is empty)
        buf.seq_base = max(max(buf._seq.values(), default=0) - int(st.epoch_dev.item()), 0)
        self.graph = torch.cuda.CUDAGraph()
        try:
            # thread_local: other threads of the process (NCCL watchdog, copy threads) may keep calling CUDA meanwhile
            with torch.cuda.graph(self.graph, stream=cur, capture_error_mode="thread_local"):
                self.loss = train_epoch(st, -1)
        except BaseException:
            st.graph_mode = buf.graph_mode = red.graph_mode = False      # stay usable in eager mode
            raise
        torch.cuda.synchronize(dev)

    def __call__(self) -> torch.Tensor:
        self.graph.replay()
        return self.loss


def run(graph, node_dict, gpb, args, device=None, full_graph=None):
    """train.py:300-456.  With ``args.eval`` rank 0 also runs the evaluation / checkpoint branch (:308-321, 427-456)
    through ``evaluate.Evaluator`` -- on the GPU with the same kernels, synchronously, instead of a CPU thread pool;
    ``full_graph``: the un-partitioned ``FullGraph`` to evaluate on (default: regenerated from ``args.dataset``)."""
    rank, size = _rank_size()
    st = setup(graph, node_dict, gpb, args, device)
    dev = st.feat.device
    evaluator = None
    if getattr(args, 'eval', False) and rank == 0:
        if args.model == 'gat':
            import warnings
            warnings.warn('--eval: the full-graph GAT forward (dgl.nn.GATConv on a homogeneous graph) is not rebuilt; '
                          'training runs without the evaluation branch')
        else:
            from .data import make_graph
            from .evaluate import Evaluator
            fg = full_graph if full_graph is not None else make_graph(args.dataset, seed=getattr(args, 'graph_seed', 0),
                                                                      device=dev)
            evaluator = Evaluator(args, fg, dev)
    train_dur, comm_dur, reduce_dur = [], [], []
    torch.cuda.reset_peak_memory_stats(dev)
    print(f'Process {rank} start training')
    loss = None
    for epoch in range(args.n_epochs):
        torch.cuda.synchronize(dev)
        t0 = time.time()
        loss = train_epoch(st, epoch)
        torch.cuda.synchronize(dev)
        if epoch >= 5:                                                      # train.py:415-418
            train_dur.append(time.time() - t0)
            comm_dur.append(comm_timer.tot_time())
            reduce_dur.append(ctx.reducer.last_reduce_seconds())
        if (epoch + 1) % args.log_every == 0:
            print("Process {:03d} | Epoch {:05d} | Time(s) {:.4f} | Comm(s) {:.4f} | Reduce(s) {:.4f} | Loss {:.4f}".format(
                rank, epoch, np.mean(train_dur) if train_dur else float('nan'),
                np.mean(comm_dur) if comm_dur else float('nan'),
                np.mean(reduce_dur) if reduce_dur else float('nan'), loss.item() / max(st.part_train, 1)))
            if evaluator is not None:                                       # train.py:427-442
                evaluator.after_epoch(st.model, epoch)
    print_memory("memory stats")
    if evaluator is not None:                                               # train.py:446-456
        evaluator.finish(st.model)
    return st, {"time": train_dur, "comm": comm_dur, "reduce": reduce_dur,
                "loss": None if loss is None else loss.item()}
