"""oracle/bns_oracle.py -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

CPU (torch fp32 + the C SpMM of ``spmm_ref.c``) restatement of the BNS-GCN hot path, written to
check the CUDA path of ``bns-gcn_b200`` and to serve as the CPU baseline of ``bench.py``.  Only
``tests/``, ``__graft_entry__.smoke()`` and ``bench.py`` (``cpu_baseline`` / ``--impl reference``)
may import this module.

PARITY PINNING.  The reference (/root/reference, 100 % Python) ships no tests, fixtures or golden
vectors, and cannot be imported as is: it needs ``dgl``/``ogb`` (absent, un-vendored third-party
wheels: ``dgl-cu113`` README.md:41 says 0.9.1, ``torch==1.12.0+cu113`` requirements.txt:3-5) and a
CUDA device.  The restatement below is therefore pinned two ways: (1) ``tests/golden/`` holds vectors
produced by running the reference's own ``module/``, ``helper/`` and ``train.py`` functions on CPU
under a small DGL shim (``tests/golden/make_golden.py``), which this oracle must reproduce; (2) the
known-answer properties of SURVEY.md §4 (P-invariance at sampling rate 1, exchange exactness).

Every function cites the reference lines it follows.  Graph ids here are int64 CPU tensors.
"""
from __future__ import annotations

import ctypes
import math
import os
import queue
import subprocess
import threading
from typing import Dict, List, Optional, Sequence

import numpy as np
import torch
import torch.nn.functional as F
from torch import nn

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None
_SEED_LOCK = threading.Lock()


def _lib():
    """Load (building on first use) the C restatement of the DGL SpMM."""
    global _LIB
    if _LIB is None:
        so = os.path.join(_HERE, "_build", "libspmm_ref.so")
        if not os.path.exists(so):
            subprocess.check_call(["make", "-s", "-C", _HERE])
        lib = ctypes.CDLL(so)
        i64, p = ctypes.c_int64, ctypes.c_void_p
        lib.bns_ref_coo_to_csr.argtypes = [i64, i64, p, p, p, p]
        lib.bns_ref_coo_to_csr.restype = ctypes.c_int
        lib.bns_ref_spmm_sum_f32.argtypes = [i64, p, p, p, i64, i64, p, i64]
        lib.bns_ref_spmm_sum_f32.restype = ctypes.c_int
        lib.bns_ref_set_threads.argtypes = [ctypes.c_int]
        lib.bns_ref_set_threads.restype = None
        _LIB = lib
    return _LIB


def set_threads(n: int) -> None:
    """OpenMP threads per SpMM / COO->CSR call (0 = OpenMP default).  bench.py sets it explicitly because torchrun
    exports OMP_NUM_THREADS=1."""
    _lib().bns_ref_set_threads(int(n))


# --------------------------------------------------------------------------------------------
# communication shim: the reference talks to ``torch.distributed`` (gloo) directly; the oracle
# goes through this tiny interface so that the same rank code runs under real gloo processes
# (``GlooComm``) or as P threads of one process (``ThreadComm``), which is what most tests use.
# --------------------------------------------------------------------------------------------
class _Done:
    def wait(self):
        return None


class ThreadFabric:
    """Mailboxes shared by the P ``ThreadComm`` endpoints of one in-process group."""

    def __init__(self, size: int):
        self.size = size
        self._box: Dict[tuple, "queue.Queue"] = {}
        self._lock = threading.Lock()
        self._bar = threading.Barrier(size)
        self._red: List[Optional[torch.Tensor]] = [None] * size

    def box(self, src: int, dst: int, tag: int) -> "queue.Queue":
        with self._lock:
            return self._box.setdefault((src, dst, tag), queue.Queue())

    def comm(self, rank: int) -> "ThreadComm":
        return ThreadComm(self, rank)


class ThreadComm:
    def __init__(self, fabric: ThreadFabric, rank: int):
        self.fabric, self.rank, self.size = fabric, rank, fabric.size

    def isend(self, t: torch.Tensor, dst: int, tag: int = 0):
        self.fabric.box(self.rank, dst, tag).put(t.detach().clone())
        return _Done()

    def recv(self, t: torch.Tensor, src: int, tag: int = 0):
        t.copy_(self.fabric.box(src, self.rank, tag).get(timeout=300))

    def irecv(self, t: torch.Tensor, src: int, tag: int = 0):
        comm = self

        class _R:
            def wait(self_inner):
                comm.recv(t, src, tag)
        return _R()

    def all_reduce_sum(self, t: torch.Tensor):
        f = self.fabric
        f._red[self.rank] = t.detach().clone()
        f._bar.wait()
        tot = f._red[0].clone()
        for r in range(1, self.size):     # fixed rank order => every endpoint gets the same bits
            tot += f._red[r]
        f._bar.wait()
        t.copy_(tot)

    def barrier(self):
        self.fabric._bar.wait()


class GlooComm:
    """Same interface over ``torch.distributed`` (gloo), i.e. the reference's default backend
    (``helper/parser.py:48``)."""

    def __init__(self):
        import torch.distributed as dist
        self._d = dist
        self.rank, self.size = dist.get_rank(), dist.get_world_size()

    def isend(self, t, dst, tag=0):
        return self._d.isend(t.contiguous(), dst=dst, tag=tag)

    def recv(self, t, src, tag=0):
        self._d.recv(t, src=src, tag=tag)

    def irecv(self, t, src, tag=0):
        return self._d.irecv(t, src=src, tag=tag)

    def all_reduce_sum(self, t):
        self._d.all_reduce(t, op=self._d.ReduceOp.SUM)

    def barrier(self):
        self._d.barrier()


class SoloComm:
    """World of one rank (P=1: plain full-graph training, the known-answer reference of SURVEY §4)."""
    rank, size = 0, 1

    def all_reduce_sum(self, t):
        return None

    def barrier(self):
        return None


TAG_NODE, TAG_FEAT, TAG_DEG = 0, 1, 2          # helper/utils.py:15-18
TAG_FWD, TAG_BWD, TAG_BND = 16, 64, 128        # per-layer feature / gradient messages, boundary setup


# --------------------------------------------------------------------------------------------
# the DGL pieces the path relies on, restated over COO edge lists
# --------------------------------------------------------------------------------------------
class EdgeList:
    """A bipartite ``_U -> _V`` graph held as COO, as ``dgl.heterograph`` receives it (train.py:276)."""

    def __init__(self, u: torch.Tensor, v: torch.Tensor, n_u: int, n_v: int):
        self.u, self.v, self.n_u, self.n_v = u.contiguous(), v.contiguous(), int(n_u), int(n_v)
        self._csr = None      # by destination (forward)
        self._csr_t = None    # by source (backward), built lazily like DGL does

    def num_nodes(self, ntype: str = "_V") -> int:
        return self.n_v if ntype == "_V" else self.n_u

    def num_edges(self) -> int:
        return int(self.u.numel())

    @staticmethod
    def _build(n_rows: int, rows: torch.Tensor, cols: torch.Tensor):
        indptr = torch.empty(n_rows + 1, dtype=torch.int64)
        out = torch.empty_like(cols)
        rc = _lib().bns_ref_coo_to_csr(n_rows, rows.numel(), rows.data_ptr(), cols.data_ptr(),
                                       indptr.data_ptr(), out.data_ptr())
        if rc != 0:
            raise RuntimeError(f"bns_ref_coo_to_csr failed ({rc})")
        return indptr, out

    def csr(self):
        if self._csr is None:
            self._csr = self._build(self.n_v, self.v, self.u)
        return self._csr

    def csr_t(self):
        if self._csr_t is None:
            self._csr_t = self._build(self.n_u, self.u, self.v)
        return self._csr_t


def _spmm(indptr: torch.Tensor, cols: torch.Tensor, x: torch.Tensor, n_rows: int) -> torch.Tensor:
    x = x.contiguous()
    y = torch.empty(n_rows, x.shape[1], dtype=torch.float32)
    _lib().bns_ref_spmm_sum_f32(n_rows, indptr.data_ptr(), cols.data_ptr(), x.data_ptr(), x.stride(0),
                                x.shape[1], y.data_ptr(), y.stride(0))
    return y


class CopyUSum(torch.autograd.Function):
    """``graph['_E'].update_all(fn.copy_u('h','m'), fn.sum('m','h'))`` (module/layer.py:35-37, 88-90)."""

    @staticmethod
    def forward(ctx, g: EdgeList, h_u: torch.Tensor):
        assert h_u.shape[0] == g.n_u, (h_u.shape, g.n_u)
        ctx.g = g
        indptr, cols = g.csr()
        return _spmm(indptr, cols, h_u, g.n_v)

    @staticmethod
    def backward(ctx, dy):
        g = ctx.g
        indptr, cols = g.csr_t()
        return None, _spmm(indptr, cols, dy, g.n_u)


def copy_u_sum_indexadd(g: EdgeList, h_u: torch.Tensor) -> torch.Tensor:
    """Second, independent statement of the same sum (``index_add_``); cross-checks the C kernel."""
    out = torch.zeros(g.n_v, h_u.shape[1], dtype=h_u.dtype)
    return out.index_add_(0, g.v, h_u[g.u])


# --------------------------------------------------------------------------------------------
# per-rank setup: train.py:77-131, helper/utils.py:150-223
# --------------------------------------------------------------------------------------------
class RankInput:
    """What ``load_partition`` hands to ``run`` (helper/utils.py:101-140), as plain tensors."""

    def __init__(self, n_in, n_halo, indptr, indices, nid, part_id, feat, label, in_deg, out_deg, train_mask,
                 ranges, n_train, n_class):
        self.n_in, self.n_halo = int(n_in), int(n_halo)
        self.indptr, self.indices = indptr, indices
        self.nid, self.part_id = nid, part_id
        self.feat, self.label = feat, label
        self.in_deg, self.out_deg, self.train_mask = in_deg, out_deg, train_mask
        self.ranges, self.n_train, self.n_class = ranges, int(n_train), int(n_class)

    @classmethod
    def from_partition(cls, p) -> "RankInput":
        nd = p.node_dict
        return cls(p.graph.n_in, p.graph.n_halo, p.graph.indptr, p.graph.indices, nd["_ID"], nd["part_id"],
                   nd["feat"], nd["label"], nd["in_deg"], nd["out_deg"], nd["train_mask"], p.gpb.ranges,
                   p.meta["n_train"], p.meta["n_class"])


def ring_exchange(comm, send: Sequence[Optional[torch.Tensor]], recv_shape, tag: int, dtype) -> list:
    """``data_transfer`` (helper/utils.py:190-213): tagged ring isend / recv, ``right=(rank+i)%P``."""
    rank, size = comm.rank, comm.size
    res: List[Optional[torch.Tensor]] = [None] * size
    for i in range(1, size):
        left, right = (rank - i + size) % size, (rank + i) % size
        req = comm.isend(send[right].to(dtype), right, tag)
        buf = torch.zeros(recv_shape[left], dtype=dtype)
        comm.recv(buf, left, tag)
        res[left] = buf
        req.wait()
    return res


def merge_feature(own: torch.Tensor, recv: list) -> torch.Tensor:
    """``merge_feature`` (helper/utils.py:216-223): ``[own | recv_0 | recv_1 ...]`` in rank order, self skipped."""
    return torch.cat([own] + [r for r in recv if r is not None])


class OracleRank:
    """One partition's state: everything ``train.run`` builds before the epoch loop (train.py:300-383)."""

    def __init__(self, inp: RankInput, comm, model: str = "graphsage", n_layers: int = 3, n_hidden: int = 16,
                 sampling_rate: float = 1.0, use_pp: bool = True, dropout: float = 0.0, norm: Optional[str] = "layer",
                 lr: float = 1e-2, weight_decay: float = 0.0, seed: int = 0, n_linear: int = 0,
                 multilabel: bool = False, heads: int = 1):
        self.inp, self.comm = inp, comm
        self.rank, self.size = comm.rank, comm.size
        self.model_name, self.rate = model, sampling_rate
        n_in = inp.n_in
        self.n_in = n_in
        # get_in_out_graph (train.py:77-87): inner->inner edges / halo->inner edges
        dst = torch.repeat_interleave(torch.arange(n_in, dtype=torch.int64), inp.indptr[1:] - inp.indptr[:-1])
        src = inp.indices
        inner = src < n_in
        self.in_u, self.in_v = src[inner], dst[inner]
        self.out_u, self.out_v = src[~inner], dst[~inner]
        # out_graph.out_degrees / out_edges need halo rows: CSR of the halo->inner edges by halo source
        n_loc = n_in + inp.n_halo
        self.out_indptr, self.out_cols = EdgeList._build(n_loc, self.out_u, self.out_v)
        self.boundary = self._get_boundary()
        self.pos = self._get_pos()
        self.send_size, self.ratio = self._get_send_size()
        self.recv_size = self._get_recv_size()
        self.layer_size = [inp.feat.shape[1]] + [n_hidden] * (n_layers - 1) + [inp.n_class]   # utils.py:143-147
        # Buffer.__init_pl_pr (helper/feature_buffer.py:23-33)
        self.pl, self.pr, tot = [None] * self.size, [None] * self.size, n_in
        for j in range(self.size):
            if j != self.rank:
                self.pl[j], tot = tot, tot + self.recv_size[j]
                self.pr[j] = tot
        if not use_pp:
            raise NotImplementedError("init_buffer raises unless use_pp (helper/feature_buffer.py:36-37)")
        self.out_deg_all = self._collect_out_degree()                                        # train.py:350
        self.feat = self._precompute()                                                       # train.py:351-352
        with _SEED_LOCK:          # ranks may be threads of one process: the global RNG is shared
            torch.manual_seed(seed)                                                          # train.py:331
            self.net = build_model(model, self.layer_size, use_pp, dropout, norm, inp.n_train, n_linear, heads)
        self.net.oracle = self
        for m in self.net.modules():
            if isinstance(m, SyncBNRef):
                m.comm = comm
        self.loss_fn = (nn.BCEWithLogitsLoss(reduction="sum") if multilabel
                        else nn.CrossEntropyLoss(reduction="sum"))                            # train.py:358-361
        self.opt = torch.optim.Adam(self.net.parameters(), lr=lr, weight_decay=weight_decay)
        if model == "gcn":
            self.in_norm = torch.sqrt(inp.in_deg.float())                                    # train.py:377-378
            self.out_norm = torch.sqrt(self.out_deg_all.float())
        else:
            self.in_norm = inp.in_deg                                                        # train.py:380
        self.selected: List[Optional[torch.Tensor]] = [None] * self.size
        self.trace: Dict[str, torch.Tensor] = {}
        self.relu_masks: Optional[Dict[int, torch.Tensor]] = None
        self.kink = {"flips": 0, "max_abs_z": 0.0}
        self.comm_bytes = 0

    # ---- helper/utils.py:150-184 ---------------------------------------------------------
    def _get_boundary(self):
        inp, comm, rank, size = self.inp, self.comm, self.rank, self.size
        boundary: List[Optional[torch.Tensor]] = [None] * size
        for i in range(1, size):
            left, right = (rank - i + size) % size, (rank + i) % size
            belong_right = inp.part_id == right
            v = inp.nid[belong_right] - int(inp.ranges[right])
            num_right = torch.tensor([v.numel()], dtype=torch.int64)
            num_left = torch.zeros(1, dtype=torch.int64)
            req = comm.isend(num_right, right, TAG_BND)
            comm.recv(num_left, left, TAG_BND)
            req.wait()
            req = comm.isend(v, right, TAG_BND + 1)
            u = torch.zeros(int(num_left), dtype=torch.int64)
            comm.recv(u, left, TAG_BND + 1)
            boundary[left] = torch.sort(u)[0]
            req.wait()
        return boundary

    # ---- train.py:90-104 -------------------------------------------------------------------
    def _get_pos(self):
        inp = self.inp
        pos: List[Optional[torch.Tensor]] = []
        for i in range(self.size):
            if i == self.rank:
                pos.append(None)
                continue
            start, end = int(inp.ranges[i]), int(inp.ranges[i + 1])
            p = torch.full((end - start,), -1, dtype=torch.int64)
            in_idx = torch.nonzero(inp.part_id == i, as_tuple=True)[0]
            p[inp.nid[in_idx] - start] = in_idx
            pos.append(p)
        return pos

    # ---- train.py:107-131 ------------------------------------------------------------------
    def _get_send_size(self):
        res, ratio = [], []
        for i, b in enumerate(self.boundary):
            if i == self.rank:
                res.append(0)
                ratio.append(0)
                continue
            s = int(self.rate * b.shape[0])
            res.append(s)
            # the reference divides by b.shape[0] unguarded (ZeroDivisionError on an empty boundary)
            ratio.append(s / b.shape[0] if b.shape[0] else 1.0)
        return res, ratio

    def _get_recv_size(self):
        return [0 if i == self.rank else int(self.rate * int((self.inp.part_id == i).sum()))
                for i in range(self.size)]

    # ---- train.py:148-167 ------------------------------------------------------------------
    def _halo_shapes(self, width=None):
        out = []
        for i in range(self.size):
            if i == self.rank:
                out.append(None)
            else:
                s = int((self.inp.part_id == i).sum())
                out.append((s,) if width is None else (s, width))
        return out

    def _collect_out_degree(self):
        if self.size == 1:
            return self.inp.out_deg
        send = [None if i == self.rank else self.inp.out_deg[b] for i, b in enumerate(self.boundary)]
        recv = ring_exchange(self.comm, send, self._halo_shapes(), TAG_DEG, torch.int64)
        return merge_feature(self.inp.out_deg, recv)

    # ---- train.py:134-145, 256-281 -----------------------------------------------------------
    def construct_graph(self, one_hops) -> EdgeList:
        tot = self.n_in
        u_list, v_list = [self.in_u], [self.in_v]
        for i in range(self.size):
            if i == self.rank:
                continue
            u = one_hops[i]
            if u.shape[0] == 0:
                continue
            u = self.pos[i][u]                                    # my local halo ids, sender's order
            deg = self.out_indptr[u + 1] - self.out_indptr[u]      # graph.out_degrees(u)
            u_list.append(torch.repeat_interleave(torch.arange(u.shape[0], dtype=torch.int64), deg) + tot)
            tot += u.shape[0]
            # graph.out_edges(u): edges grouped in the order of u
            seg = torch.repeat_interleave(self.out_indptr[u] - torch.cumsum(deg, 0) + deg, deg)
            v_list.append(self.out_cols[seg + torch.arange(int(deg.sum()), dtype=torch.int64)])
        u, v = torch.cat(u_list), torch.cat(v_list)
        # dgl.heterograph infers n_V = max(v)+1 (== n_in thanks to the self loops); _U is padded to tot
        return EdgeList(u, v, tot, self.n_in)

    def order_graph(self) -> EdgeList:
        one_hops = [None if i == self.rank else
                    torch.sort(self.inp.nid[self.inp.part_id == i] - int(self.inp.ranges[i]))[0]
                    for i in range(self.size)]
        return self.construct_graph(one_hops)

    # ---- train.py:170-211 --------------------------------------------------------------------
    def _precompute(self):
        inp, feat = self.inp, self.inp.feat
        g = self.order_graph()
        if self.size > 1:
            send = [None if i == self.rank else feat[b] for i, b in enumerate(self.boundary)]
            recv = ring_exchange(self.comm, send, self._halo_shapes(feat.shape[1]), TAG_FEAT, torch.float32)
        else:
            recv = [None]
        h_u = merge_feature(feat, recv)
        if self.model_name == "gcn":
            in_norm = torch.sqrt(inp.in_deg.float())
            out_norm = torch.sqrt(self.out_deg_all.float())
            h = CopyUSum.apply(g, h_u / out_norm.unsqueeze(-1))
            return h / in_norm.unsqueeze(-1)
        if self.model_name == "graphsage":
            s = CopyUSum.apply(g, h_u)
            cnt = (g.csr()[0][1:] - g.csr()[0][:-1]).clamp(min=1).unsqueeze(-1)     # fn.mean: / #messages
            return torch.cat([feat, s / cnt], dim=1)
        if self.model_name == "gat":
            return h_u                                                                       # train.py:208-209
        raise NotImplementedError(self.model_name)

    # ---- train.py:225-236 --------------------------------------------------------------------
    def select_node(self, rng: np.random.RandomState):
        sel: List[Optional[torch.Tensor]] = []
        for i in range(self.size):
            if i == self.rank:
                sel.append(None)
                continue
            b = self.boundary[i]
            idx = torch.as_tensor(rng.choice(b.shape[0], self.send_size[i], replace=False), dtype=torch.int64)
            sel.append(b[idx])
        return sel

    # ---- helper/feature_buffer.py:93-129 (gloo variant) ---------------------------------------
    def exchange_forward(self, layer: int, h: torch.Tensor) -> torch.Tensor:
        rank, size, comm = self.rank, self.size, self.comm
        recv: List[Optional[torch.Tensor]] = [None] * size
        reqs = []
        for i in range(1, size):
            left, right = (rank - i + size) % size, (rank + i) % size
            msg = h[self.selected[right]] / self.ratio[right]                     # :117
            reqs.append(comm.isend(msg, right, TAG_FWD + layer))
            self.comm_bytes += msg.numel() * 4
            recv[left] = torch.zeros(self.recv_size[left], h.shape[1])
        for i in range(1, size):
            left = (rank - i + size) % size
            comm.recv(recv[left], left, TAG_FWD + layer)
        for r in reqs:
            r.wait()
        return torch.cat([h] + [recv[j] for j in range(size) if j != rank])       # __feat_concat :85-91

    def exchange_backward(self, layer: int, grad: torch.Tensor) -> torch.Tensor:
        rank, size, comm = self.rank, self.size, self.comm
        grad = grad.clone()
        reqs = []
        for i in range(1, size):
            right = (rank + i) % size
            msg = grad[self.pl[right]:self.pr[right]]                             # :119
            reqs.append(comm.isend(msg, right, TAG_BWD + layer))
            self.comm_bytes += msg.numel() * 4
        for i in range(1, size):
            left = (rank - i + size) % size
            buf = torch.zeros(self.send_size[left], grad.shape[1])
            comm.recv(buf, left, TAG_BWD + layer)
            grad[self.selected[left]] += buf / self.ratio[left]                   # :129
        for r in reqs:
            r.wait()
        return grad

    # ---- train.py:385-425 ---------------------------------------------------------------------
    def epoch(self, selected: Optional[list] = None, rng: Optional[np.random.RandomState] = None,
              step: bool = True, trace: bool = False, relu_masks: Optional[Dict[int, torch.Tensor]] = None,
              forward_only: bool = False) -> float:
        """One training epoch; returns the local (sum-reduced) loss.  ``selected`` injects the sampled sets.
        ``forward_only``: the training-mode forward with every dropout switched off, no backward, no update (bench.py's
        ``parity_probe``: a loss both sides can compute at the initial weights whatever the dropout rate is).

        ``relu_masks`` ({norm index i: bool [n_in, F]}): the active set another implementation of the SAME forward took
        at the ReLU after norm i.  Gradient parity is only defined on a common active set: where a pre-activation sits
        within f32 rounding of zero the two forwards may land on different sides of the kink (tests/harness.py).  The
        given mask then replaces ``z > 0``; ``self.kink`` counts the entries where it differed and how far from zero
        the furthest of them was (a large distance means a real forward disagreement, not a kink)."""
        self.trace = {} if trace else None
        self.relu_masks = relu_masks
        if selected is None:
            selected = self.select_node(rng if rng is not None else np.random)
        self.selected = selected
        if self.size > 1:
            one_hops = ring_exchange(self.comm, selected, [None if s is None else (r,) for s, r in
                                                           zip(selected, self.recv_size)], TAG_NODE, torch.int64)
        else:
            one_hops = [None]
        self.one_hops = one_hops
        g = self.construct_graph(one_hops)
        self.graph = g
        self.net.train()
        if forward_only:
            drops = [(m, m.p) for m in self.net.modules() if isinstance(m, nn.Dropout)]
            for m, _ in drops:
                m.p = 0.0
            try:
                with torch.no_grad():
                    logits = self._forward_logits(g, one_hops)
            finally:
                for m, p_ in drops:
                    m.p = p_
            mask = self.inp.train_mask
            return float(self.loss_fn(logits[mask], self.inp.label[mask]).item())
        logits = self._forward_logits(g, one_hops)
        mask = self.inp.train_mask
        loss = self.loss_fn(logits[mask], self.inp.label[mask])
        self.opt.zero_grad(set_to_none=True)
        loss.backward()
        # Reducer.reduce / synchronize (helper/reducer.py:28-38): grad /= n_train, SUM all-reduce per parameter
        for prm in self.net.parameters():
            if prm.grad is None:
                continue
            prm.grad.div_(self.inp.n_train)
            self.comm.all_reduce_sum(prm.grad)
        if step:
            self.opt.step()
        if trace:
            self.trace["logits"] = logits.detach().clone()
        return float(loss.item())

    def _forward_logits(self, g, one_hops):
        if self.model_name == "gcn":
            parts = [self.out_norm[:self.n_in]] + [self.out_norm[self.pos[i][one_hops[i]]]
                                                   for i in range(self.size) if i != self.rank]   # train.py:245-253
            logits = self.net(g, self.feat, self.in_norm, torch.cat(parts))
        elif self.model_name == "gat":
            res = [self.feat[0:self.n_in]]                                                   # construct_feat, train.py:284-297
            for i in range(self.size):
                if i != self.rank and one_hops[i].shape[0] > 0:
                    res.append(self.feat[self.pos[i][one_hops[i]]])
            logits = self.net(g, torch.cat(res))
        else:
            logits = self.net(g, self.feat, self.in_norm)
        return logits


class _Exchange(torch.autograd.Function):
    """``Buffer.update`` + its grad hook (helper/feature_buffer.py:93-99, 169-174)."""

    @staticmethod
    def forward(ctx, h, rk: OracleRank, layer: int):
        ctx.rk, ctx.layer, ctx.n_in = rk, layer, h.shape[0]
        return rk.exchange_forward(layer, h)

    @staticmethod
    def backward(ctx, grad):
        if ctx.rk.trace is not None:
            ctx.rk.trace[f"grad_u{ctx.layer}"] = grad.detach().clone()          # before the gradient exchange
        g = ctx.rk.exchange_backward(ctx.layer, grad)
        if ctx.rk.trace is not None:
            ctx.rk.trace[f"grad_h{ctx.layer}"] = g[:ctx.n_in].detach().clone()
        return g[:ctx.n_in], None, None


# --------------------------------------------------------------------------------------------
# module/layer.py and module/model.py
# --------------------------------------------------------------------------------------------
def _uniform_reset(*linears):
    """``reset_parameters`` (module/layer.py:20-24, 65-77): U(-1/sqrt(in), 1/sqrt(in)), weights first."""
    stdv = 1.0 / math.sqrt(linears[0].weight.size(1))
    for lin in linears:
        lin.weight.data.uniform_(-stdv, stdv)
    for lin in linears:
        if lin.bias is not None:
            lin.bias.data.uniform_(-stdv, stdv)


class SAGELayerRef(nn.Module):
    """``GraphSAGELayer`` (module/layer.py:49-103)."""

    def __init__(self, in_feats, out_feats, use_pp=False):
        super().__init__()
        self.use_pp = use_pp
        if use_pp:
            self.linear = nn.Linear(2 * in_feats, out_feats)
            _uniform_reset(self.linear)
        else:
            self.linear1 = nn.Linear(in_feats, out_feats)
            self.linear2 = nn.Linear(in_feats, out_feats)
            _uniform_reset(self.linear1, self.linear2)

    def forward(self, g, feat, in_norm):
        if self.training:
            if self.use_pp:
                return self.linear(feat)                                         # :82-83
            degs = in_norm.unsqueeze(1)
            ah = CopyUSum.apply(g, feat) / degs                                  # :88-91
            return self.linear1(feat[0:g.num_nodes("_V")]) + self.linear2(ah)    # :92
        degs = (g.csr()[0][1:] - g.csr()[0][:-1]).unsqueeze(1)                   # :94
        ah = CopyUSum.apply(g, feat) / degs
        if self.use_pp:
            return self.linear(torch.cat((feat, ah), dim=1))                     # :99-100
        return self.linear1(feat) + self.linear2(ah)


class GCNLayerRef(nn.Module):
    """``GCNLayer`` (module/layer.py:8-46)."""

    def __init__(self, in_feats, out_feats, use_pp=False):
        super().__init__()
        self.use_pp = use_pp
        self.linear = nn.Linear(in_feats, out_feats)
        _uniform_reset(self.linear)

    def forward(self, g, feat, in_norm, out_norm):
        if self.training:
            if self.use_pp:
                return self.linear(feat)                                         # :29-30
            h = CopyUSum.apply(g, feat / out_norm.unsqueeze(1))                  # :34-37
            return self.linear(h / in_norm.unsqueeze(1))                         # :38
        indptr_t = g.csr_t()[0]
        in_n = torch.sqrt((g.csr()[0][1:] - g.csr()[0][:-1]).float()).unsqueeze(1)
        out_n = torch.sqrt((indptr_t[1:] - indptr_t[:-1]).float()).unsqueeze(1)
        return self.linear(CopyUSum.apply(g, feat / out_n) / in_n)               # :40-45


class _SyncBNFunc(torch.autograd.Function):
    """``SyncBatchNormFunc`` (module/sync_bn.py:7-39), four all-reduces as in the reference."""

    @staticmethod
    def forward(ctx, x, weight, bias, whole_size, running_mean, running_var, training, momentum, eps, comm):
        if not training:
            mean, var = running_mean, running_var
        else:
            sum_x, sum_x2 = x.sum(axis=0), (x ** 2).sum(axis=0)
            comm.all_reduce_sum(sum_x)
            comm.all_reduce_sum(sum_x2)
            mean = sum_x / whole_size
            var = (sum_x2 - mean * sum_x) / whole_size
            running_mean.mul_(1 - momentum).add_(mean * momentum)
            running_var.mul_(1 - momentum).add_(var * momentum)
        std = torch.sqrt(var + eps)
        x_hat = (x - mean) / std
        if training:
            ctx.save_for_backward(x_hat, weight, std)
            ctx.whole_size, ctx.comm = whole_size, comm
        return x_hat * weight + bias

    @staticmethod
    def backward(ctx, grad):
        x_hat, weight, std = ctx.saved_tensors
        dbias, dweight = grad.sum(axis=0), (grad * x_hat).sum(axis=0)
        ctx.comm.all_reduce_sum(dbias)
        ctx.comm.all_reduce_sum(dweight)
        n = ctx.whole_size
        dx = (weight / n) / std * (n * grad - dbias - x_hat * dweight)
        return dx, dweight, dbias, None, None, None, None, None, None, None


class SyncBNRef(nn.Module):
    """``SyncBatchNorm`` (module/sync_bn.py:42-56)."""

    def __init__(self, num_features, whole_size, eps=1e-5, momentum=0.1):
        super().__init__()
        self.register_buffer("running_mean", torch.zeros(num_features))
        self.register_buffer("running_var", torch.ones(num_features))
        self.whole_size, self.eps, self.momentum = whole_size, eps, momentum
        self.weight = nn.Parameter(torch.ones(num_features))
        self.bias = nn.Parameter(torch.zeros(num_features))
        self.comm = None

    def forward(self, x):
        return _SyncBNFunc.apply(x, self.weight, self.bias, self.whole_size, self.running_mean, self.running_var,
                                 self.training, self.momentum, self.eps, self.comm)


class GNNRef(nn.Module):
    """``GCN`` / ``GraphSAGE`` (module/model.py:26-93)."""

    def __init__(self, kind, layer_size, use_pp, dropout, norm, train_size, n_linear):
        super().__init__()
        self.kind = kind
        self.n_layers = len(layer_size) - 1
        self.n_linear = n_linear
        self.use_pp = use_pp
        self.layers = nn.ModuleList()
        self.use_norm = norm is not None
        if self.use_norm:
            self.norm = nn.ModuleList()
        self.dropout = nn.Dropout(p=dropout)
        layer_cls = SAGELayerRef if kind == "graphsage" else GCNLayerRef
        pp = use_pp
        for i in range(self.n_layers):
            if i < self.n_layers - n_linear:
                self.layers.append(layer_cls(layer_size[i], layer_size[i + 1], use_pp=pp))
            else:
                self.layers.append(nn.Linear(layer_size[i], layer_size[i + 1]))
            if i < self.n_layers - 1 and self.use_norm:
                if norm == "layer":
                    self.norm.append(nn.LayerNorm(layer_size[i + 1], elementwise_affine=True))
                else:
                    self.norm.append(SyncBNRef(layer_size[i + 1], train_size))            # model.py:37-39
            pp = False                                                           # model.py:40,75
        self.oracle: Optional[OracleRank] = None

    def forward(self, g, feat, in_norm=None, out_norm=None):
        h = feat
        rk = self.oracle
        for i in range(self.n_layers):
            h = self.dropout(h)
            if i < self.n_layers - self.n_linear:
                if self.training and (i > 0 or not self.use_pp):
                    h = _Exchange.apply(h, rk, i) if rk.size > 1 else h           # ctx.buffer.update(i, h)
                    if rk.trace is not None:
                        rk.trace[f"h_u{i}"] = h.detach().clone()
                h = self.layers[i](g, h, in_norm) if self.kind == "graphsage" else \
                    self.layers[i](g, h, in_norm, out_norm)
            else:
                h = self.layers[i](h)
            if rk is not None and rk.trace is not None:
                rk.trace[f"layer{i}"] = h.detach().clone()
            if i < self.n_layers - 1:
                if self.use_norm:
                    h = self.norm[i](h)
                h = _relu_on_active_set(h, rk, i)
        return h


def _relu_on_active_set(z, rk, i):
    """``F.relu(z)``, or ``z * mask`` when the caller prescribed the active set (``OracleRank.epoch(relu_masks=...)``)."""
    if rk is not None and rk.trace is not None:
        rk.trace[f"z{i}"] = z.detach().clone()
    m = rk.relu_masks.get(i) if (rk is not None and rk.relu_masks) else None
    if m is None:
        return F.relu(z)
    d = (z.detach() > 0) != m
    if bool(d.any()):
        rk.kink["flips"] += int(d.sum())
        rk.kink["max_abs_z"] = max(rk.kink["max_abs_z"], float(z.detach()[d].abs().max()))
    return z * m.to(z.dtype)


class GATConvRef(nn.Module):
    """``dgl.nn.GATConv(in, out, heads, feat_drop, attn_drop)`` as module/model.py:102 constructs it.  DGL 0.9 is not
    vendored with the reference, so this restates its published layer (Velickovic et al. 2018 as implemented in
    python/dgl/nn/pytorch/conv/gatconv.py): shared ``fc`` for source and destination, ``attn_l`` / ``attn_r``,
    LeakyReLU(0.2), softmax over each destination's in-edges, dropout on features and on attention, bias, no residual
    or activation; xavier-normal init with the ReLU gain, zero bias.  Pinned by hand-computed outputs derived from the
    layer's published definition (tests/test_gat_pin_cpu.py: uniform attention, both LeakyReLU branches, two heads with a
    non-trivial fc and destination scores); DGL's own kernels cannot be run here."""

    def __init__(self, in_feats, out_feats, num_heads, feat_drop=0.0, attn_drop=0.0, negative_slope=0.2):
        super().__init__()
        self.H, self.Fo = num_heads, out_feats
        self.fc = nn.Linear(in_feats, out_feats * num_heads, bias=False)
        self.attn_l = nn.Parameter(torch.empty(1, num_heads, out_feats))
        self.attn_r = nn.Parameter(torch.empty(1, num_heads, out_feats))
        self.feat_drop, self.attn_drop = nn.Dropout(feat_drop), nn.Dropout(attn_drop)
        self.negative_slope = negative_slope
        self.bias = nn.Parameter(torch.empty(num_heads * out_feats))
        gain = nn.init.calculate_gain("relu")
        nn.init.xavier_normal_(self.fc.weight, gain=gain)
        nn.init.xavier_normal_(self.attn_l, gain=gain)
        nn.init.xavier_normal_(self.attn_r, gain=gain)
        nn.init.constant_(self.bias, 0)

    def forward(self, g: EdgeList, feat):
        H, Fo = self.H, self.Fo
        h_src, h_dst = (self.feat_drop(feat[0]), self.feat_drop(feat[1])) if isinstance(feat, tuple) \
            else (self.feat_drop(feat),) * 2
        ft_src = self.fc(h_src).view(-1, H, Fo)
        ft_dst = self.fc(h_dst).view(-1, H, Fo)
        el = (ft_src * self.attn_l).sum(-1)
        er = (ft_dst * self.attn_r).sum(-1)
        e = F.leaky_relu(el[g.u] + er[g.v], self.negative_slope)                        # u_add_v, leaky_relu
        idx = g.v.unsqueeze(1).expand(-1, H)
        m = torch.full((g.n_v, H), float("-inf")).scatter_reduce(0, idx, e.detach(), "amax")
        ex = torch.exp(e - m[g.v])
        den = torch.zeros(g.n_v, H).index_add(0, g.v, ex)
        a = self.attn_drop(ex / den[g.v])                                               # edge_softmax
        rst = torch.zeros(g.n_v, H, Fo).index_add(0, g.v, a.unsqueeze(-1) * ft_src[g.u])   # u_mul_e, sum
        return rst + self.bias.view(1, H, Fo)


class GATRef(nn.Module):
    """``GAT`` (module/model.py:96-132)."""

    def __init__(self, layer_size, use_pp, heads, dropout, norm, train_size, n_linear):
        super().__init__()
        self.n_layers, self.n_linear, self.use_pp = len(layer_size) - 1, n_linear, use_pp
        self.layers = nn.ModuleList()
        self.use_norm = norm is not None
        if self.use_norm:
            self.norm = nn.ModuleList()
        self.dropout = nn.Dropout(p=dropout)
        for i in range(self.n_layers):
            if i < self.n_layers - n_linear:
                self.layers.append(GATConvRef(layer_size[i], layer_size[i + 1], heads, dropout, dropout))
            else:
                self.layers.append(nn.Linear(layer_size[i], layer_size[i + 1]))
            if i < self.n_layers - 1 and self.use_norm:
                self.norm.append(nn.LayerNorm(layer_size[i + 1], elementwise_affine=True) if norm == "layer"
                                 else SyncBNRef(layer_size[i + 1], train_size))
        self.oracle: Optional[OracleRank] = None

    def forward(self, g, feat):
        h, rk = feat, self.oracle
        for i in range(self.n_layers):
            if i < self.n_layers - self.n_linear:
                if self.training:
                    if i > 0 or not self.use_pp:
                        h1 = _Exchange.apply(h, rk, i) if rk.size > 1 else h          # model.py:117-118
                    else:
                        h1, h = h, h[0:g.num_nodes("_V")]                              # :120-121
                    h = self.layers[i](g, (h1, h))
                else:
                    h = self.layers[i](g, h)
                h = h.mean(1)
            else:
                h = self.layers[i](self.dropout(h))
            if rk is not None and rk.trace is not None:
                rk.trace[f"layer{i}"] = h.detach().clone()
            if i < self.n_layers - 1:
                if self.use_norm:
                    h = self.norm[i](h)
                h = _relu_on_active_set(h, rk, i)
        return h


def build_model(kind, layer_size, use_pp, dropout, norm, train_size, n_linear, heads=1):
    if kind == "gat":
        return GATRef(layer_size, True, heads, dropout, norm, train_size, n_linear)     # train.py:222: use_pp=True
    if kind not in ("graphsage", "gcn"):
        raise NotImplementedError(kind)
    return GNNRef(kind, layer_size, use_pp, dropout, norm, train_size, n_linear)


# --------------------------------------------------------------------------------------------
# running P ranks inside one process
# --------------------------------------------------------------------------------------------
def run_threads(n_ranks: int, fn, *args):
    """Run ``fn(comm, rank, *args)`` on ``n_ranks`` threads sharing a ``ThreadFabric``; returns the results."""
    if n_ranks == 1:
        return [fn(SoloComm(), 0, *args)]
    fabric = ThreadFabric(n_ranks)
    out: List = [None] * n_ranks
    err: List = [None] * n_ranks

    def work(r):
        try:
            out[r] = fn(fabric.comm(r), r, *args)
        except BaseException as e:          # noqa: BLE001 - surfaced below
            err[r] = e
            fabric._bar.abort()

    ts = [threading.Thread(target=work, args=(r,), daemon=True) for r in range(n_ranks)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    for e in err:
        if e is not None and not isinstance(e, threading.BrokenBarrierError):
            raise e
    for e in err:
        if e is not None:
            raise e
    return out
