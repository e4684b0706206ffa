"""bench.py -- the driver's measurement contract.

  python bench.py [--gpus N] [--steps K] [--warmup W]                (N>1: launched under torchrun, one rank per GPU)
  python bench.py --impl reference [--gpus N] [--steps K] [--warmup W]
  python bench.py [...] --dump-outputs DIR    (also writes the last timed step's outputs, see dump_outputs)

Workload (BASELINE.json metric, configs[1]): 3-layer GraphSAGE (hidden 256, --use-pp, LayerNorm, dropout 0.5,
lr 0.01, sampling rate 0.1) on the Reddit-shape synthetic power-law graph (232,965 nodes, ~114.6M edges, 602
features, 41 classes), vertex-partitioned over the N GPUs (random partition).  A "step" is one training epoch:
boundary sampling -> id exchange -> forward (feature exchange + SpMM + dense) -> loss -> backward (SpMM^T +
gradient exchange) -> weight-gradient all-reduce -> Adam.  The graph is fixed, so more GPUs = less work per GPU
("scaling": "strong").  value = epochs/sec of the whole job (max over ranks of the device-timed region).
Besides the contract keys the line carries `roofline` (the SpMM, the dominant kernel: algorithmic bytes / CUDA-event
time per launch, measured in an eager pass of the same step), `dense_roofline` (the tcgen05 GEMM family), `e2e`
(inputs copied from pinned host memory every epoch, loss read back), `cpu_baseline` (N=1), `exchange`, `clocks`.

`--impl reference` times the CPU restatement of the reference (oracle/: torch CPU fp32 + C/OpenMP SpMM, P in-process
ranks for N>1) on the host cores with the same config; the real reference cannot run here (needs DGL + CUDA 11.3
wheels, see DESIGN.md).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

WORKLOAD = dict(shape="reddit", model="graphsage", n_layers=3, n_hidden=256, sampling_rate=0.1, dropout=0.5,
                lr=0.01, norm="layer", partition="random")


def METRIC():
    if (WORKLOAD["shape"], WORKLOAD["model"], WORKLOAD["n_layers"]) == ("reddit", "graphsage", 3):
        return "epochs/sec (3-layer GraphSAGE, Reddit-shape graph)"
    return f"epochs/sec ({WORKLOAD['n_layers']}-layer {WORKLOAD['model']}, {WORKLOAD['shape']}-shape graph)"


def workload_string(gstats: dict, world: int) -> str:
    """`config.workload`, identical in both arms (our CUDA path and `--impl reference`)."""
    head = "BASELINE configs[1]: " if (WORKLOAD["shape"], WORKLOAD["model"]) == ("reddit", "graphsage") else ""
    return (f"{head}{WORKLOAD['shape']}-shape synthetic power-law graph, {gstats['n_nodes']} nodes, {gstats['n_edges']} edges, "
            f"{gstats['n_feat']} feat; {WORKLOAD['model']} {WORKLOAD['n_layers']}-layer hidden {WORKLOAD['n_hidden']} --use-pp, "
            f"sampling-rate {WORKLOAD['sampling_rate']}, dropout {WORKLOAD['dropout']}, {world} random partition(s)")


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.idx)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def make_args(n_parts: int, backend: str, extra: dict):
    ns = argparse.Namespace(dataset=WORKLOAD["shape"], model=WORKLOAD["model"], n_layers=WORKLOAD["n_layers"],
                            n_hidden=WORKLOAD["n_hidden"], sampling_rate=WORKLOAD["sampling_rate"], use_pp=True,
                            dropout=WORKLOAD["dropout"], norm=WORKLOAD["norm"], lr=WORKLOAD["lr"], weight_decay=0.0,
                            seed=0, n_linear=0, backend=backend, sampler_seed=0, n_epochs=0, log_every=10 ** 9,
                            heads=1, n_partitions=n_parts, inductive=False, partition_method=WORKLOAD["partition"],
                            eval=False, chunk_nnz=0, multilabel=(WORKLOAD["shape"] == "yelp"))
    for k, v in extra.items():
        setattr(ns, k, v)
    return ns


SCALE = 1.0          # --scale: shrinks the per-rank generated shapes (papers100m) in nodes and edges alike


def build_partition(shape: str, n_parts: int, rank: int, device):
    from bns_gcn_b200.data import SHAPES, make_graph, make_local_partition, partition_graph
    if shape == "papers100m":
        # never built as one graph: every rank generates its own piece on its GPU (data.make_local_partition)
        part = make_local_partition(shape, rank, n_parts, seed=0, device=device, scale=SCALE)
        stats = {"n_nodes": int(part.gpb.ranges[-1]), "n_edges": part.graph.num_edges() * n_parts,
                 "n_feat": SHAPES[shape]["n_feat"]}
        return part, stats
    fg = make_graph(shape, seed=0, device=device)
    stats = {"n_nodes": fg.n_nodes, "n_edges": fg.n_edges, "n_feat": fg.n_feat}
    part = partition_graph(fg, n_parts, WORKLOAD["partition"], seed=0, ranks=[rank], device=device)[0]
    del fg
    return part, stats


DUMP_BYTES = 64 << 20            # --dump-outputs writes at most this much, all ranks together


def dump_outputs(d: str, st, loss, rank: int, world: int) -> None:
    """`--dump-outputs DIR`: what the last timed step computed, one `.npy` file per array, so that two builds run with
    the same arguments can be compared output for output.  `loss` is the step's summed training loss on this rank,
    `logits` this rank's inner nodes x classes, `param.<name>` the weights after the step's Adam update (identical on
    every rank, so rank 0 writes them).  Logits larger than the budget are a fixed seeded sample of rows whose indices
    go to `logits_rows`.  With several ranks, loss and logits carry a `.rank<r>` suffix."""
    import numpy as np
    os.makedirs(d, exist_ok=True)
    sfx = f".rank{rank}" if world > 1 else ""
    params = {f"param.{n}": p.detach().float() for n, p in st.model.named_parameters()}
    out = {f"loss{sfx}": loss.detach().float().reshape(1)}
    if rank == 0:
        out.update(params)
    logits = st.last_logits.detach().float()
    n, c = logits.shape
    budget = (DUMP_BYTES - sum(4 * p.numel() for p in params.values())) // world - 4
    if 4 * n * c > budget:
        keep = max(budget // (4 * c + 8), 0)
        rows = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:keep].sort().values
        out[f"logits_rows{sfx}"] = rows.double()
        logits = logits[rows.to(logits.device)]
    out[f"logits{sfx}"] = logits
    for name, t in out.items():
        np.save(os.path.join(d, name + ".npy"), t.cpu().numpy())


# =====================================================================================================
# our arm
# =====================================================================================================
def run_ours(a):
    import torch.distributed as dist
    from bns_gcn_b200 import ops, train
    from bns_gcn_b200._lib import lib
    from bns_gcn_b200.helper import context as ctx
    from bns_gcn_b200.helper.timer.timer import comm_timer

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != a.gpus:
        if world == 1 and a.gpus > 1:
            raise SystemExit(f"--gpus {a.gpus} needs torchrun (one rank per GPU); WORLD_SIZE is 1")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    K, W = a.steps, max(a.warmup, 3)
    # everything runs on ONE non-default stream: the epoch is later captured on it (see train.GraphedEpoch)
    main_stream = torch.cuda.Stream(dev)
    torch.cuda.set_stream(main_stream)
    part, gstats = build_partition(a.shape, world, rank, dev)
    args = make_args(world, a.backend, {"n_feat": part.meta["n_feat"], "n_class": part.meta["n_class"],
                                        "n_train": part.meta["n_train"], "dataset": a.shape})
    import contextlib
    with contextlib.redirect_stdout(sys.stderr):          # stdout carries exactly one JSON line
        st = train.setup(part.graph, part.node_dict, part.gpb, args, dev)
    torch.cuda.synchronize(dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # one device per process: run backward on this thread (no hand-off to autograd's device thread; it also keeps
    # the NVTX range below around the backward kernels for the ncu launch list)
    torch.autograd.set_multithreading_enabled(False)
    # ---------------- parity probe (correctness carried by every bench line, N = 8 included) ------------------
    # The forward loss of epoch 0 at the initial weights with dropout off, summed over ranks, against (N = 1) the CPU
    # oracle's value and (N > 1) the same ranks run as threads of one process on rank 0's GPU -- the arrangement
    # tests/ pins to the oracle, bench shape included (tests/test_bench_shape_gpu.py).
    probe = None
    # the probe's reference side rebuilds every partition in one process (N > 1) or runs the CPU oracle (N = 1): bounded
    # to graphs of at most 20 M nodes (the papers100M shape above --scale 0.18 skips it; use --scale 0.05 to probe it)
    too_big = gstats["n_nodes"] > 20_000_000
    if too_big and not a.no_probe and rank == 0:
        print(f"[bench] parity probe skipped: {gstats['n_nodes']} nodes", file=sys.stderr)
    if not a.no_probe and not too_big:
        probe = {"loss_epoch0_dropout_off": float(train.probe_loss(st, 0).item())}     # summed over ranks inside
    epoch = 0
    for _ in range(W):                                   # untimed warm-up
        train.train_epoch(st, epoch)
        epoch += 1

    from bns_gcn_b200.module import dense as dense_mod
    dense_prof = []
    last_loss = [None]                                   # what the most recent timed step returned

    def timed(step_fn, n_steps, profile_spmm):
        """n_steps of step_fn between barriers; device time by CUDA events, max over ranks."""
        barrier()
        if profile_spmm:
            ops.PROFILE = []
            dense_mod.PROFILE = []
        c0 = lib.bns_launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record(torch.cuda.current_stream(dev))
        torch.cuda.nvtx.range_push("bns_timed")          # ncu --nvtx --nvtx-include "bns_timed/" lists the steps
        for _ in range(n_steps):
            last_loss[0] = step_fn()
        torch.cuda.nvtx.range_pop()
        e1.record(torch.cuda.current_stream(dev))
        barrier()
        pr, ops.PROFILE = ops.PROFILE, None
        if profile_spmm:
            dense_prof[:] = dense_mod.PROFILE or []
        dense_mod.PROFILE = None
        return max_over_ranks(e0.elapsed_time(e1)), lib.bns_launch_count() - c0, pr

    comm_log, reduce_log = [], []

    def eager_step():
        nonlocal epoch
        loss = train.train_epoch(st, epoch)
        epoch += 1
        if world > 1:                                    # Comm(s) / Reduce(s) of EVERY eager epoch (train.py:415-418)
            comm_log.append(comm_timer.tot_time())
            reduce_log.append(ctx.reducer.last_reduce_seconds())
        return loss

    # ---------------- eager pass: per-kernel CUDA events (roofline), Comm(s)/Reduce(s) -----------------------
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    K_eager = K if a.mode == "eager" else min(K, 5)
    eager_ms, eager_launches, prof = timed(eager_step, K_eager, True)
    # Comm(s) / Reduce(s) per epoch: mean over the eager epochs of this rank, then the max over ranks
    comm_last = max_over_ranks(sum(comm_log) / len(comm_log)) if world > 1 and comm_log else 0.0
    reduce_last = max_over_ranks(sum(reduce_log) / len(reduce_log)) if world > 1 and reduce_log else 0.0
    launches_per_step = eager_launches / K_eager
    mode = "eager"
    dev_ms, n_launch = eager_ms * K / K_eager, eager_launches * K // K_eager
    step_fn = eager_step
    # ---------------- timed region proper: the epoch replayed from one CUDA graph ----------------------------
    if a.mode == "graph":
        try:
            ge = train.GraphedEpoch(st, warmup=1)
            epoch += 1
            for _ in range(2):
                ge()
            step_fn, mode = ge, "cuda-graph"
            dev_ms, _, _ = timed(step_fn, K, False)
            n_launch = int(launches_per_step * K)        # the same kernels, launched by the graph
        except Exception as e:                           # noqa: BLE001
            import traceback
            traceback.print_exc(file=sys.stderr)
            print(f"[bench] CUDA-graph capture failed, staying eager: {type(e).__name__}: {e}", file=sys.stderr)
            if a.strict:
                raise
            dev_ms, n_launch, _ = timed(eager_step, K, False)
    n0, n1 = 0, n_launch
    clk = clocks.stop() if rank == 0 else None
    if a.dump_outputs:                                   # before the e2e pass below trains the model further
        dump_outputs(a.dump_outputs, st, last_loss[0], rank, world)
    spmm_ms = sum(s.elapsed_time(e) for s, e, *_ in prof)
    spmm_alg = sum(p[2] for p in prof)
    spmm_gather = sum(4 * p[3] + 4 * p[4] * p[5] for p in prof)        # p[5]: entries actually gathered (estimate)
    gemm_ms = sum(s.elapsed_time(e) for s, e, *_ in dense_prof)
    gemm_flops = sum(p[2] for p in dense_prof)
    gemm_bytes = sum(p[3] for p in dense_prof)
    # ---------------- e2e: host-resident inputs, H2D + D2H inside the timed region -------------------
    feat_dev, lab_dev, mask_dev = st.feat, st.labels, st.train_mask
    feat_pin = feat_dev.cpu().pin_memory()
    lab_pin, mask_pin = lab_dev.cpu().pin_memory(), mask_dev.cpu().pin_memory()
    bufs = [(torch.empty_like(feat_dev), torch.empty_like(lab_dev), torch.empty_like(mask_dev)) for _ in range(2)]
    copy_stream = torch.cuda.Stream(dev)
    ready = [torch.cuda.Event(), torch.cuda.Event()]
    consumed = [torch.cuda.Event(), torch.cuda.Event()]
    h2d = feat_pin.numel() * 4 + lab_pin.numel() * lab_pin.element_size() + mask_pin.numel()

    def prefetch(i):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[i % 2])
            f, l, m = bufs[i % 2]
            f.copy_(feat_pin, non_blocking=True)
            l.copy_(lab_pin, non_blocking=True)
            m.copy_(mask_pin, non_blocking=True)
            ready[i % 2].record(copy_stream)

    for i in range(2):
        consumed[i].record(torch.cuda.current_stream(dev))
    # the step's result (the loss) goes to pinned host memory with an async copy and is READ one step late: the host
    # never stalls the queue, every loss is still read inside the timed region (the last one before the clock stops)
    loss_pin = [torch.zeros(1, dtype=torch.float32).pin_memory() for _ in range(2)]
    loss_ev = [torch.cuda.Event(), torch.cuda.Event()]
    losses_read = []
    barrier()
    t0 = time.perf_counter()
    prefetch(0)
    for i in range(K):
        if i + 1 < K:
            prefetch(i + 1)                              # next step's inputs stream in behind this step's compute
        cur = torch.cuda.current_stream(dev)
        cur.wait_event(ready[i % 2])
        if mode == "cuda-graph":                         # the graph reads fixed addresses: stage -> device copy
            feat_dev.copy_(bufs[i % 2][0]); lab_dev.copy_(bufs[i % 2][1]); mask_dev.copy_(bufs[i % 2][2])
            consumed[i % 2].record(cur)
            loss = step_fn()
        else:
            st.feat, st.labels, st.train_mask = bufs[i % 2]
            loss = train.train_epoch(st, epoch)
            consumed[i % 2].record(cur)
            epoch += 1
        loss_pin[i % 2].copy_(loss.reshape(1), non_blocking=True)      # D2H of the step's result
        loss_ev[i % 2].record(cur)
        if i > 0:
            loss_ev[(i - 1) % 2].synchronize()
            losses_read.append(float(loss_pin[(i - 1) % 2][0]))
    loss_ev[(K - 1) % 2].synchronize()
    losses_read.append(float(loss_pin[(K - 1) % 2][0]))
    barrier()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    assert len(losses_read) == K
    st.feat, st.labels, st.train_mask = feat_dev, lab_dev, mask_dev

    if a.profile and rank == 0:                            # diagnosis only (kineto); never a reported number
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof_:
            for _ in range(3):
                step_fn()
            torch.cuda.synchronize(dev)
        with open(a.profile, "w") as f:
            f.write(prof_.key_averages().table(sort_by="cuda_time_total", row_limit=45, max_name_column_width=70))
    elif a.profile:
        for _ in range(3):
            step_fn()
    # host-side enqueue time of one epoch (no sync inside): if it is close to ms_per_step the step is CPU-bound
    barrier()
    th = time.perf_counter()
    for _ in range(5):
        step_fn()
    host_ms = (time.perf_counter() - th) / 5 * 1e3
    barrier()

    # ---------------- parity probe, reference side (N > 1): the same ranks as threads of ONE process ------------
    if probe is not None and world > 1:
        if rank == 0:
            try:
                ref = inprocess_probe_loss(a.shape, world, dev)
                probe.update({"reference": "same ranks as threads of one process on rank 0's GPU (staged transport), "
                                           "the arrangement tests/ pins to the CPU oracle",
                              "loss_reference": ref,
                              "rel_err": abs(probe["loss_epoch0_dropout_off"] - ref) / max(abs(ref), 1e-30)})
                probe["ok"] = bool(probe["rel_err"] < 1e-5)
            except Exception as e:                       # noqa: BLE001
                probe.update({"reference": f"in-process run failed: {type(e).__name__}: {e}", "ok": None})
        barrier()
    if rank != 0:
        _leave(world)
        return
    peak, peak_src = load_peaks()
    n_spmm = max(len(prof), 1)
    feat_mb = st.feat.numel() * 4 / 2 ** 20
    csr_mb = part.graph.num_edges() * 4 * 2 / 2 ** 20
    ws_mb = feat_mb + csr_mb + 8 * part.graph.n_in * WORKLOAD["n_hidden"] * 4 / 2 ** 20
    # boundary exchange (per rank, per epoch): rows sent forward + gradient rows returned, on every communicating layer
    n_comm_layers = max(WORKLOAD["n_layers"] - 1, 0)
    ex_bytes = 4 * WORKLOAD["n_hidden"] * (sum(st.send_size) + sum(st.recv_size)) * n_comm_layers if world > 1 else 0
    traffic, traffic_src = None, None
    tp = os.path.join(ROOT, "profiles", "spmm_traffic.json")
    if os.path.exists(tp) and WORKLOAD["shape"] == "reddit":
        # not measurable inside this run (ncu replays kernels): the per-launch DRAM bytes of the F = 256 inner SpMM from
        # the committed capture of the same kernel on the same shape (tools/ncu_spmm_traffic.sh; world 1 and 4)
        with open(tp) as f:
            tj = json.load(f)
        ent = tj.get(str(world)) or (tj if world == 1 else {})
        traffic, traffic_src = ent.get("dram_bytes_per_launch"), ent.get("source")
    ach = spmm_alg / (spmm_ms * 1e-3) / 1e9 if spmm_ms > 0 else 0.0
    out = {
        "metric": METRIC(), "value": K / (dev_ms * 1e-3),
        "unit": "epochs/s", "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": dev_ms / K,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_string(gstats, world),
                   "l2": f"no flush between timed epochs: one epoch of rank 0 streams {ws_mb:.0f} MB (features "
                         f"{feat_mb:.0f} MB + CSR and transposes {csr_mb:.0f} MB + activations), L2 is 126 MB",
                   "parallelism": f"partition-parallel x{world}", "exchange": a.backend, "execution": mode,
                   "n_in_rank0": part.graph.n_in, "n_halo_rank0": part.graph.n_halo,
                   "local_edges_rank0": part.graph.num_edges()},
        "comm_s_per_epoch": comm_last, "reduce_s_per_epoch": reduce_last,
        "comm_note": f"mean over the {K_eager} eager epochs of this run (CUDA events on the comm / reduce streams), max over "
                     "ranks; the replayed graph runs the same kernels but cannot be timed from inside",
        "host_enqueue_ms_per_step": host_ms,
        "eager_ms_per_step": eager_ms / K_eager,
        "e2e": {"value": K / e2e_s, "unit": "epochs/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": 4,
                "note": "features+labels+mask copied from pinned host memory every epoch (prefetched one step ahead on "
                        "a copy stream), loss read back every epoch"},
        "exchange": {"bytes_per_epoch_per_rank": int(ex_bytes), "comm_s_per_epoch": comm_last,
                     "GBs_over_comm_time": (ex_bytes / comm_last / 1e9) if comm_last > 0 else None,
                     "note": "comm_s = CUDA-event time of the exchanges on the comm stream (pack + NVLink transfer + "
                             "waiting for the peers' data), measured in the eager pass; it overlaps the inner-edge SpMM"},
        "gpu_launches": int(n1 - n0),
        "clocks": clk,
        "roofline": {"bound": "hbm", "kernel": "spmm_kernel (bns_spmm_sum_f32)", "achieved": ach, "peak": peak,
                     "unit": "GB/s", "frac": ach / peak, "traffic": traffic, "traffic_source": traffic_src,
                     "peak_source": peak_src,
                     "launches_timed": len(prof), "avg_launch_ms": spmm_ms / n_spmm,
                     "share_of_step": spmm_ms / eager_ms if eager_ms else None,
                     "gather_GBs": spmm_gather / (spmm_ms * 1e-3) / 1e9 if spmm_ms > 0 else 0.0,
                     "note": "per-launch CUDA events from the eager pass of the same step inside this run (events cannot sit between nodes of the captured graph); achieved = algorithmic bytes (each distinct operand byte once, SURVEY 8d) / CUDA-event time; "
                             "gather_GBs counts one 4F-byte row read per edge (what actually crosses L2->SM): that is the "
                             "binding resource on this degree-492 graph, see DESIGN.md"},
    }
    if dense_prof and gemm_ms > 0:
        # second kernel family of the step: the dense layers on tcgen05 (csrc/dense_tc.cuh).  3xTF32 issues three
        # tensor-core products per useful f32 one; TF32 dense peak is taken as half the measured bf16 cuBLAS rate
        # (MEASURED_PEAKS.json holds no TF32 figure; sustained, because the kernel runs inside a long step)
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
                pk = json.load(f)
            tf32_peak, tf32_src = 0.5 * float(pk.get("bf16_tflops_sustained") or pk["bf16_tflops"]), "0.5 x measured sustained bf16 (MEASURED_PEAKS.json)"
        except Exception:   # noqa: BLE001
            tf32_peak, tf32_src = 0.5 * 1400.0, "0.5 x fallback sustained bf16 (B200_PROFILING.md)"
        useful = gemm_flops / (gemm_ms * 1e-3) / 1e12
        out["dense_roofline"] = {"bound": "tensor", "kernel": "gemm3x_kernel (bns_dense_tn_3xtf32 / bns_dense_nt_3xtf32)",
                                 "achieved": 3.0 * useful, "peak": tf32_peak, "unit": "TFLOP/s", "frac": 3.0 * useful / tf32_peak,
                                 "f32_equivalent_TFLOPs": useful, "peak_source": tf32_src, "launches_timed": len(dense_prof),
                                 "share_of_step": gemm_ms / eager_ms if eager_ms else None,
                                 "algorithmic_GBs": gemm_bytes / (gemm_ms * 1e-3) / 1e9,
                                 "note": "achieved = 3 x useful f32 FLOPs (hi*hi + hi*lo + lo*hi) / CUDA-event time of the "
                                         "launches in the eager pass; the kernel is shared-memory-bandwidth bound (ncu: tensor "
                                         "pipe 46 %, LSU + tensor-core shared-memory wavefronts 53 % + 51 %), see "
                                         "profiles/ncu_gemm3x_r01.md"}
    if world == 1 and not a.no_cpu_baseline:
        out["cpu_baseline"] = cpu_epochs_per_sec(a.shape, 1, steps=1, warmup=1, probe=probe is not None)
        out["cpu_baseline"].pop("gstats", None)
        if probe is not None and "probe_loss" in out["cpu_baseline"]:
            ref = out["cpu_baseline"].pop("probe_loss")
            probe.update({"reference": "CPU oracle (oracle/bns_oracle.py), forward at the initial weights, dropout off",
                          "loss_reference": ref,
                          "rel_err": abs(probe["loss_epoch0_dropout_off"] - ref) / max(abs(ref), 1e-30)})
            probe["ok"] = bool(probe["rel_err"] < 1e-4)
    if probe is not None:
        out["parity_probe"] = probe
    emit(out)
    _leave(world)


def _leave(world: int) -> None:
    """Multi-rank runs end here, right after the last barrier / the JSON line: flush and leave without tearing down
    NCCL, the captured graphs and the peer-mapped slabs.  (Round 1: an N=2 run printed its line and then sat in
    interpreter teardown until the box's time limit; nothing after this point is measured or needed.)"""
    if world > 1:
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


def inprocess_probe_loss(shape: str, world: int, dev) -> float:
    """`train.probe_loss` of epoch 0 with the `world` ranks as threads of this process on `dev` (ThreadComm, staged
    transport), summed over ranks."""
    import contextlib
    from bns_gcn_b200 import train
    from bns_gcn_b200.data import make_graph, partition_graph
    from bns_gcn_b200.helper.comm import run_threads
    if shape == "papers100m":
        parts = [build_partition(shape, world, r, dev)[0] for r in range(world)]     # per-rank generator (never one graph)
    else:
        fg = make_graph(shape, seed=0, device=dev)
        parts = partition_graph(fg, world, WORKLOAD["partition"], seed=0, device=dev)
        del fg

    def fn(comm, r):
        p = parts[r]
        args = make_args(world, "nccl", {"n_feat": p.meta["n_feat"], "n_class": p.meta["n_class"],
                                         "n_train": p.meta["n_train"], "dataset": shape})
        st = train.setup(p.graph, p.node_dict, p.gpb, args, dev)
        return float(train.probe_loss(st, 0).item())          # already the sum over the ranks

    # redirect ONCE, around the threads: contextlib.redirect_stdout swaps the process-wide sys.stdout, so entering /
    # leaving it from several threads can leave stdout pointing at stderr for good (and the JSON line with it)
    with contextlib.redirect_stdout(sys.stderr):
        out = run_threads(world, fn, device=str(dev))
    return float(out[0])


# =====================================================================================================
# CPU arm (the oracle as the reference's stand-in)
# =====================================================================================================
def _oracle_rank(part, comm):
    from oracle import bns_oracle as O
    return O.OracleRank(O.RankInput.from_partition(part), comm, model=WORKLOAD["model"], n_layers=WORKLOAD["n_layers"],
                        n_hidden=WORKLOAD["n_hidden"], sampling_rate=WORKLOAD["sampling_rate"], use_pp=True,
                        dropout=WORKLOAD["dropout"], norm=WORKLOAD["norm"], lr=WORKLOAD["lr"], seed=0,
                        multilabel=(WORKLOAD["shape"] == "yelp"))


def _cpu_rank_loop(rk, comm, r, per_rank, steps, warmup, budget_s, probe):
    """The timed loop of one CPU rank: `warmup` + up to `steps` full epochs between barriers, stopped early (after at
    least one timed epoch) once `budget_s` is spent.  Returns (per-epoch seconds, probe loss or None)."""
    import numpy as np
    torch.set_num_threads(per_rank)          # OpenMP's thread count is per calling thread
    probe_loss = None
    if probe:                                # forward at the initial weights, dropout off, the epoch-0 Philox sets
        sel = None
        if comm.size > 1:
            from oracle import philox
            peers = [j for j in range(comm.size) if j != r]
            ref = philox.sample_boundary([rk.boundary[j].numpy() for j in peers], [rk.send_size[j] for j in peers], 0, 0)
            sel = [None] * comm.size
            for i, j in enumerate(peers):
                sel[j] = torch.from_numpy(ref[i])
        probe_loss = rk.epoch(selected=sel, forward_only=True)
    rng = np.random.RandomState(1234 + r)
    times = []
    t_begin = time.perf_counter()
    for e in range(warmup + steps):
        comm.barrier()
        t0 = time.perf_counter()
        rk.epoch(rng=rng)
        comm.barrier()
        dt = time.perf_counter() - t0
        if e >= warmup:
            times.append(dt)
        stop = torch.tensor([1.0 if (time.perf_counter() - t_begin > budget_s and e >= warmup) else 0.0])
        comm.all_reduce_sum(stop)
        if float(stop) > 0:
            break
    return times, probe_loss


def cpu_worker(a):
    """One gloo process of the CPU arm (spawned by cpu_epochs_per_sec for P > 1): loads its partition from the
    hand-over directory, joins the gloo group on 127.0.0.1 and runs the timed loop."""
    import torch.distributed as dist
    from oracle import bns_oracle as O
    d = a.cpu_worker
    with open(os.path.join(d, "job.json")) as f:
        job = json.load(f)
    WORKLOAD.update(job["workload"])
    r, P = a.cpu_rank, job["world"]
    torch.set_num_threads(job["per_rank"])
    O.set_threads(job["per_rank"])
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{job['port']}", rank=r, world_size=P)
    part = torch.load(os.path.join(d, f"part{r}.pt"), weights_only=False)
    comm = O.GlooComm()
    rk = _oracle_rank(part, comm)
    times, pl = _cpu_rank_loop(rk, comm, r, job["per_rank"], job["steps"], job["warmup"], job["budget_s"], job["probe"])
    with open(os.path.join(d, f"out{r}.json"), "w") as f:
        json.dump({"times": times, "probe_loss": pl}, f)
    dist.barrier()
    dist.destroy_process_group()


def cpu_epochs_per_sec(shape: str, n_parts: int, steps: int, warmup: int, budget_s: float = 150.0,
                       probe: bool = False) -> dict:
    """The CPU restatement of the reference (oracle/) on the host cores: P = 1 in this process, P > 1 as P gloo
    processes on 127.0.0.1 with floor(cores / P) threads each (BASELINE.md section 3), full epochs of the same workload."""
    import shutil
    import tempfile
    from bns_gcn_b200.data import make_graph, partition_graph
    from oracle import bns_oracle as O
    cores = os.cpu_count() or 1
    per_rank = max(1, cores // n_parts)
    torch.set_num_threads(per_rank)          # torchrun exports OMP_NUM_THREADS=1: set both pools explicitly
    O.set_threads(per_rank)
    fg = make_graph(shape, seed=0, device=torch.device("cuda") if torch.cuda.is_available() else None)
    gstats = {"n_nodes": fg.n_nodes, "n_edges": fg.n_edges, "n_feat": fg.n_feat}
    parts = partition_graph(fg, n_parts, WORKLOAD["partition"], seed=0)
    del fg
    if n_parts == 1:
        comm = O.SoloComm()
        per_rank_times, pl = _cpu_rank_loop(_oracle_rank(parts[0], comm), comm, 0, per_rank, steps, warmup, budget_s, probe)
        all_times, probe_loss, how = [per_rank_times], pl, "this process"
    else:
        d = tempfile.mkdtemp(prefix="bns_cpu_arm_")
        try:
            for r, p_ in enumerate(parts):
                torch.save(p_, os.path.join(d, f"part{r}.pt"))
            del parts
            import socket
            with socket.socket() as sk:
                sk.bind(("127.0.0.1", 0))
                port = sk.getsockname()[1]
            with open(os.path.join(d, "job.json"), "w") as f:
                json.dump({"world": n_parts, "per_rank": per_rank, "steps": steps, "warmup": warmup, "budget_s": budget_s,
                           "probe": probe, "port": port, "workload": WORKLOAD}, f)
            # the workers form their OWN gloo group: nothing of the launcher's rendezvous may leak into them (with
            # TORCHELASTIC_USE_AGENT_STORE set, a tcp:// init makes every rank a store CLIENT and nobody serves)
            env = {k: v for k, v in os.environ.items()
                   if k not in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT", "OMP_NUM_THREADS",
                                "GROUP_RANK", "ROLE_RANK", "LOCAL_WORLD_SIZE", "GROUP_WORLD_SIZE", "ROLE_WORLD_SIZE",
                                "ROLE_NAME") and not k.startswith(("TORCHELASTIC_", "TORCH_NCCL_"))}
            env["OMP_NUM_THREADS"] = str(per_rank)
            env["CUDA_VISIBLE_DEVICES"] = ""             # the CPU arm never touches a GPU
            procs = [subprocess.Popen([sys.executable, os.path.abspath(__file__), "--cpu-worker", d, "--cpu-rank", str(r)],
                                      env=env, stdout=sys.stderr, stderr=sys.stderr) for r in range(n_parts)]
            rcs = [p_.wait() for p_ in procs]
            if any(rcs):
                raise RuntimeError(f"CPU arm: worker exit codes {rcs}")
            outs = []
            for r in range(n_parts):
                with open(os.path.join(d, f"out{r}.json")) as f:
                    outs.append(json.load(f))
            all_times = [o["times"] for o in outs]
            probe_loss = sum(o["probe_loss"] for o in outs) if probe else None
            how = f"{n_parts} gloo processes on 127.0.0.1"
        finally:
            shutil.rmtree(d, ignore_errors=True)
    done = min(len(t) for t in all_times)
    per_epoch = [max(t[i] for t in all_times) for i in range(done)]
    mean = sum(per_epoch) / len(per_epoch)
    res = {"value": 1.0 / mean, "unit": "epochs/s", "cores": cores, "kind": "port",
           "sample": f"{done} full epoch(s) of the same workload ({how}) after {warmup} warm-up, oracle/bns_oracle.py + "
                     f"oracle/spmm_ref.c (OpenMP), {cores} host threads ({per_rank} per rank)",
           "seconds_per_epoch": mean, "epochs_timed": done, "seconds_per_epoch_min": min(per_epoch),
           "seconds_per_epoch_median": statistics.median(per_epoch), "gstats": gstats}
    if probe_loss is not None:
        res["probe_loss"] = probe_loss
    return res


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    K, W = a.steps, a.warmup
    res = cpu_epochs_per_sec(a.shape, a.gpus, steps=K, warmup=min(W, 1))
    gstats = res.pop("gstats")
    done = res["epochs_timed"]
    out = {"impl": "reference", "metric": METRIC(), "value": res["value"],
           "unit": "epochs/s", "n_gpus": a.gpus, "steps": done, "steps_requested": K, "warmup": min(W, 1),
           "ms_per_step": 1e3 * res["seconds_per_epoch"],
           "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": workload_string(gstats, a.gpus),
                      "parallelism": f"host cores: {a.gpus} rank(s), OpenMP SpMM + torch CPU f32",
                      "note": "steps = epochs actually timed inside the 150 s budget (each epoch is a full pass of the "
                              "same workload); steps_requested = --steps"},
           "cpu_baseline": res,
           "e2e": {"value": res["value"], "unit": "epochs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(out)


_JSON_FD = None


def protect_stdout() -> None:
    """The contract is ONE JSON line on stdout.  C libraries write to file descriptor 1 behind Python's back (NCCL prints
    its version banner there at NCCL_DEBUG=VERSION / WARN), so keep a private duplicate of the real stdout for `emit`
    and point descriptor 1 at stderr for everything else -- in this process and every child it starts."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def emit(out: dict) -> None:
    data = (json.dumps(out) + "\n").encode()
    fd = 1 if _JSON_FD is None else _JSON_FD
    while data:
        data = data[os.write(fd, data):]


def main():
    global WORKLOAD
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--shape", default=WORKLOAD["shape"])
    ap.add_argument("--backend", default="p2p", choices=["nccl", "p2p"])
    ap.add_argument("--mode", default="graph", choices=["graph", "eager"],
                    help="graph: the epoch is captured once into a CUDA graph and replayed (default); eager: launched op by op")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--watchdog", type=int, default=int(os.environ.get("BNS_BENCH_WATCHDOG", "0")),
                    help="seconds after which every rank dumps the Python stacks of all its threads to stderr and exits "
                         "(post-mortem of a hang on a box nobody can attach to); 0 = off")
    ap.add_argument("--strict", action="store_true", help="fail instead of falling back to eager when capture fails")
    ap.add_argument("--profile", default="", help="write a torch.profiler kernel table of 3 epochs (rank 0) to this file")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write the loss, logits and weights of the last timed step to DIR/<name>.npy")
    # non-default workloads (the other BASELINE.json configs); the driver's contract run uses the defaults above
    ap.add_argument("--model", default=None, choices=["graphsage", "gcn", "gat"])
    ap.add_argument("--n-layers", type=int, default=None)
    ap.add_argument("--n-hidden", type=int, default=None)
    ap.add_argument("--rate", type=float, default=None)
    ap.add_argument("--dropout", type=float, default=None)
    ap.add_argument("--no-probe", action="store_true", help="skip the parity probe")
    ap.add_argument("--scale", type=float, default=1.0, help="papers100m only: fraction of the 111 M nodes / 1.6 B edges")
    ap.add_argument("--cpu-worker", default="", help=argparse.SUPPRESS)      # internal: one gloo process of the CPU arm
    ap.add_argument("--cpu-rank", type=int, default=0, help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.watchdog > 0:
        import faulthandler
        faulthandler.dump_traceback_later(a.watchdog, exit=True)
    if a.cpu_worker:
        cpu_worker(a)
        return
    protect_stdout()
    global SCALE
    SCALE = a.scale
    for k, v in (("model", a.model), ("n_layers", a.n_layers), ("n_hidden", a.n_hidden), ("sampling_rate", a.rate),
                 ("dropout", a.dropout), ("shape", a.shape)):
        if v is not None:
            WORKLOAD[k] = v
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)


if __name__ == "__main__":
    main()
