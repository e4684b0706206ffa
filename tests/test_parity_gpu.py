"""End-to-end parity of the CUDA path against the CPU oracle: per-layer outputs, logits, all-reduced weight
gradients and the weights after the optimizer steps, within 1e-4 relative (BASELINE.json north_star); sampled
index sets, boundary sets and exchanged id lists bit-exact.  P ranks run as threads on one GPU."""
import pytest
import torch

pytestmark = pytest.mark.gpu

TOL = 1e-4   # north_star: "within 1e-4 relative on layer outputs"


def _run(**kw):
    from tests.harness import run_parity_case
    res = run_parity_case(device="cuda:0", **kw)
    bad = {k: v for k, v in res["detail"].items() if v >= TOL}
    assert not bad, bad
    assert res["index_sets_equal"]
    for a, b in zip(res["loss"], res["loss_oracle"]):
        assert abs(a - b) <= 1e-4 * abs(b)
    return res


@pytest.mark.parametrize("model", ["graphsage", "gcn"])
@pytest.mark.parametrize("n_parts,rate", [(1, 1.0), (2, 1.0), (3, 0.5), (4, 0.1)])
def test_training_parity_tiny(built, model, n_parts, rate):
    _run(shape="tiny", n_parts=n_parts, model=model, sampling_rate=rate, n_epochs=3)


@pytest.mark.parametrize("backend", ["nccl", "p2p"])
def test_training_parity_small_both_transports(built, backend):
    """BASELINE configs[0]-like plumbing case at a size the oracle finishes in seconds; hidden 64 takes the
    16-byte vector path, rows longer than a chunk exist (chunk_nnz=64)."""
    _run(shape="small", n_parts=4, model="graphsage", sampling_rate=0.3, n_epochs=2, backend=backend, n_hidden=64,
         chunk_nnz=64)


@pytest.mark.parametrize("backend", ["nccl", "p2p"])
def test_training_parity_eight_partitions(built, backend):
    """8 partitions (the largest BASELINE rank count) as 8 in-process ranks: 7 peers per rank on both transports.

    graph_seed=3 on purpose.  With graph_seed=0 this configuration has, in epoch 2, one LayerNorm output at -2.8e-6
    (rank 0, row 64, feature 17): the f32 forward of the CUDA path lands on the other side of the ReLU kink, the
    mask of that single entry flips and the gradients upstream differ by 1e-3 -- from the oracle AND from the
    reference itself, which the oracle matches to 1e-7 there (tests/localize_gradient_mismatch.py localises it; the same inputs with
    the sets the reference drew have no such entry and agree to 2e-5, see the golden test below)."""
    _run(shape="small", n_parts=8, model="graphsage", sampling_rate=0.5, n_epochs=2, backend=backend, n_hidden=32,
         graph_seed=3)


def test_config0_two_partitions_rate1(built):
    """BASELINE.json configs[0]: 10K-node / 100K-edge random graph, 2 partitions, GraphSAGE, sampling rate 1.0."""
    _run(shape="synthetic-10k", n_parts=2, model="graphsage", sampling_rate=1.0, n_epochs=2, n_hidden=64)


def test_p_invariance_on_gpu(built):
    """At sampling rate 1 the P-partition run equals the single-partition run (SURVEY §4 pin 1): summed loss and
    all-reduced gradients agree."""
    from tests.harness import make_args, run_product
    from bns_gcn_b200.data import make_graph, partition_graph
    fg = make_graph("tiny")
    ref = None
    for P in (1, 3):
        parts = partition_graph(fg, P, "random")
        args = make_args(model="graphsage", sampling_rate=1.0, n_hidden=16, n_partitions=P)
        out = run_product(parts, args, "cuda:0", 2, capture=False)
        loss = [sum(o["loss"][e] for o in out) for e in range(2)]
        if ref is None:
            ref = (loss, out[0]["grads"])
        else:
            for a, b in zip(loss, ref[0]):
                assert abs(a - b) <= 1e-4 * abs(b)
            for a, b in zip(out[0]["grads"], ref[1]):
                assert ((a - b).norm() / b.norm()).item() < TOL


def test_metis_standin_partition_parity(built):
    _run(shape="tiny", n_parts=3, model="graphsage", sampling_rate=0.5, n_epochs=2, partition_method="metis")


@pytest.mark.parametrize("name", ["graphsage", "gcn", "graphsage_bn"])
def test_cuda_path_reproduces_reference_golden(built, name):
    """The CUDA path, fed the index sets the REFERENCE drew (tests/golden/make_golden.py ran the reference's own
    train.run), reproduces the reference's precomputed features, layer outputs, logits, reduced gradients and
    updated weights within 1e-4, and its boundary sets exactly."""
    import os
    from tests.harness import make_args, run_product, _relerr
    from bns_gcn_b200.data import make_graph, partition_graph
    gold = torch.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", f"ref_{name}_p2.pt"))
    cfg, ranks = gold["config"], gold["ranks"]
    fg = make_graph(cfg["shape"], seed=0, **cfg.get("graph_override", {}))
    parts = partition_graph(fg, cfg["n_parts"], "random", seed=0)
    args = make_args(dataset=cfg["shape"], model=cfg["model"], sampling_rate=cfg["rate"], n_layers=cfg["n_layers"],
                     n_hidden=cfg["n_hidden"], n_partitions=cfg["n_parts"], norm=cfg.get("norm", "layer"))
    sel = [[ranks[r]["selected"][e] for r in range(cfg["n_parts"])] for e in range(cfg["epochs"])]
    out = run_product(parts, args, "cuda:0", cfg["epochs"], selected_per_epoch=sel)
    bn, last = cfg.get("norm") == "batch", cfg["n_layers"] - 1      # see tests/test_oracle_cpu.py on the BN case
    for r, o in enumerate(out):
        g = ranks[r]
        for j, b in enumerate(g["boundary"]):
            if b is not None:
                assert torch.equal(o["boundary"][j], b)
        assert _relerr(o["feat0"], g["feat0"]) < TOL
        for i, lo in enumerate(g["layer_out"][-1]):
            if bn and i < last:
                continue
            assert _relerr(o["layers"][f"layer{i}"], lo) < TOL, (r, i)
        assert _relerr(o["logits"], g["logits"][-1]) < TOL
        for k, (p, gp, gg) in enumerate(zip(o["params"], g["params"], g["grads"])):
            nm = g["param_names"][k]
            if bn and nm.endswith("bias") and nm.startswith("layers.") and int(nm.split(".")[1]) < last:
                continue
            assert _relerr(p, gp) < TOL, (r, nm)
            assert _relerr(o["grads"][k], gg) < TOL, (r, nm)


def test_training_parity_through_a_relu_kink(built):
    """The graph_seed=0 twin of the test above: epoch 2 has one LayerNorm output at -2.8e-6 on rank 0 and the CUDA
    forward takes the other side of the ReLU kink.  run_parity_case must notice the mismatch, re-run both sides on the
    CUDA path's active sets, find exactly that kind of entry (|z| < 1e-4) and then agree within the bar."""
    from tests.harness import run_parity_case
    res = run_parity_case(shape="small", n_parts=8, model="graphsage", sampling_rate=0.5, n_epochs=2, n_hidden=32,
                          graph_seed=0)
    # Which side of the kink the CUDA forward lands on depends on its rounding (the op-by-op path of round 1 took the
    # other side; the fused layer functions happen to agree with the CPU): either no retry was needed, or the retry found
    # exactly that kind of entry.  Both ways the comparison must end inside the bar.
    if res["kink"] is not None:
        assert res["kink"]["flips"] >= 1 and res["kink"]["max_abs_z"] < 1e-4, res["kink"]
    assert res["max_rel_err"] < TOL, {k: v for k, v in res["detail"].items() if v >= TOL}
    assert res["index_sets_equal"]


def test_cuda_path_reproduces_reference_golden_eight_partitions(built):
    """The reference's own train.run on 8 gloo processes (tests/golden/make_golden.py, config graphsage_small):
    6000-node graph, 7 peers per rank, sampling rate 0.5, two epochs.  Rank 0's layer outputs / logits and the
    all-reduced gradients and updated weights (identical on every rank) are stored."""
    import os
    from tests.harness import make_args, run_product, _relerr
    from bns_gcn_b200.data import make_graph, partition_graph
    gold = torch.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_graphsage_small_p8.pt"))
    cfg, ranks = gold["config"], gold["ranks"]
    fg = make_graph(cfg["shape"], seed=0)
    parts = partition_graph(fg, cfg["n_parts"], "random", seed=0)
    args = make_args(dataset=cfg["shape"], model=cfg["model"], sampling_rate=cfg["rate"], n_layers=cfg["n_layers"],
                     n_hidden=cfg["n_hidden"], n_partitions=cfg["n_parts"])
    sel = [[ranks[r]["selected"][e] for r in range(cfg["n_parts"])] for e in range(cfg["epochs"])]
    out = run_product(parts, args, "cuda:0", cfg["epochs"], selected_per_epoch=sel)
    for r, o in enumerate(out):
        for j, b in enumerate(ranks[r]["boundary"]):
            if b is not None:
                assert torch.equal(o["boundary"][j], b)
    g0, o = ranks[0], out[0]
    errs = {f"layer{i}": _relerr(o["layers"][f"layer{i}"], lo) for i, lo in enumerate(g0["layer_out"][-1])}
    errs["logits"] = _relerr(o["logits"], g0["logits"][-1])
    for r, o in enumerate(out):
        for k, (gp, gg) in enumerate(zip(g0["params"], g0["grads"])):
            errs[f"r{r}/param/{g0['param_names'][k]}"] = _relerr(o["params"][k], gp)
            errs[f"r{r}/grad/{g0['param_names'][k]}"] = _relerr(o["grads"][k], gg)
    bad = {k: v for k, v in errs.items() if v >= TOL}
    if bad:
        # A ReLU kink (see test_training_parity_through_a_relu_kink): compare instead with the oracle -- which
        # tests/test_oracle_cpu.py pins to this very golden at 1e-7 -- on the active sets the CUDA forward took; the
        # harness accepts that only if every switched entry sat within 1e-4 of zero in the oracle's own forward.
        from tests.harness import run_parity_case
        res = run_parity_case(shape=cfg["shape"], n_parts=cfg["n_parts"], model=cfg["model"], sampling_rate=cfg["rate"],
                              n_epochs=cfg["epochs"], n_layers=cfg["n_layers"], n_hidden=cfg["n_hidden"], device="cuda:0",
                              selected_per_epoch=sel)
        assert res["kink"] is not None and res["kink"]["flips"] >= 1 and res["kink"]["max_abs_z"] < 1e-4, (bad, res["kink"])
        assert res["max_rel_err"] < TOL, ({k: v for k, v in res["detail"].items() if v >= TOL}, bad)


@pytest.mark.parametrize("model", ["graphsage", "gcn"])
def test_eval_branch_full_graph(built, model):
    """module/layer.py:39-45, 93-102: evaluation on the full homogeneous graph (degrees from the graph itself)."""
    from bns_gcn_b200 import ops
    from bns_gcn_b200.data import make_graph
    from bns_gcn_b200.graph import FullGraphHandle
    from bns_gcn_b200.module.model import GCN, GraphSAGE
    from oracle import bns_oracle as O
    import torch.nn.functional as F
    dev = torch.device("cuda:0")
    fg = make_graph("tiny", seed=3)
    layer_size = [fg.n_feat, 16, 16, fg.n_class]
    torch.manual_seed(0)
    net = (GraphSAGE if model == "graphsage" else GCN)(layer_size, F.relu, use_pp=False, dropout=0.5, norm="layer")
    torch.manual_seed(0)
    ref = O.build_model(model, layer_size, False, 0.5, "layer", None, 0)
    for a, b in zip(net.parameters(), ref.parameters()):
        assert torch.equal(a, b)                                   # same init order as the reference
    net.to(dev).eval()
    ref.eval()
    a = ops.DeviceGraph.from_csr(fg.indptr.to(dev), fg.src.int().to(dev), fg.n_nodes)
    g = FullGraphHandle(a, fg.in_degrees().to(dev), fg.out_degrees().to(dev))
    with torch.no_grad():
        out = net(g, fg.feat.to(dev)).cpu()
        e = O.EdgeList(fg.src, fg.dst(), fg.n_nodes, fg.n_nodes)
        want = ref(e, fg.feat)
    assert ((out - want).norm() / want.norm()).item() < TOL


@pytest.mark.parametrize("model", ["graphsage", "gcn"])
def test_cuda_graph_epoch_equals_eager(built, model):
    """train.GraphedEpoch: replaying the captured epoch gives the losses and weights of the eager loop."""
    import argparse
    from tests.harness import make_args
    from bns_gcn_b200 import train
    from bns_gcn_b200.data import make_graph, partition_graph
    from bns_gcn_b200.helper import context as ctx
    dev = torch.device("cuda:0")
    fg = make_graph("tiny", seed=0)
    part = partition_graph(fg, 1, "random", seed=0)[0]

    def fresh():
        ctx.reset()
        a = make_args(model=model, n_hidden=16)
        a.n_feat, a.n_class, a.n_train = part.meta["n_feat"], part.meta["n_class"], part.meta["n_train"]
        return train.setup(part.graph, part.node_dict, part.gpb, a, dev)
    prev = torch.autograd.is_multithreading_enabled()
    torch.autograd.set_multithreading_enabled(False)
    prev_stream = torch.cuda.current_stream(dev)
    torch.cuda.set_stream(torch.cuda.Stream(dev))       # setup + eager + capture on one non-default stream
    try:
        st = fresh()
        eager = [train.train_epoch(st, e).item() for e in range(5)]
        w_eager = [p.detach().clone() for p in st.model.parameters()]
        st = fresh()
        ge = train.GraphedEpoch(st, warmup=2)               # epochs 0, 1 eager
        replay = [ge().item() for _ in range(3)]            # epochs 2, 3, 4 from the graph
        w_graph = [p.detach().clone() for p in st.model.parameters()]
    finally:
        torch.cuda.synchronize(dev)
        torch.cuda.set_stream(prev_stream)
        torch.autograd.set_multithreading_enabled(prev)
        ctx.reset()
    for a_, b_ in zip(replay, eager[2:]):
        assert abs(a_ - b_) <= 1e-5 * abs(b_), (replay, eager)
    for a_, b_ in zip(w_graph, w_eager):
        assert ((a_ - b_).norm() / b_.norm()).item() < 1e-5


@pytest.mark.parametrize("kw", [
    dict(n_parts=3, sampling_rate=0.004),                 # int(p * b) == 0 for every peer: nothing is exchanged
    dict(n_parts=3, sampling_rate=0.004, backend="p2p"),  # ... over peer memory: zero-row puts still publish their flags
    dict(n_parts=2, sampling_rate=0.5, n_linear=1),       # --n-linear: the last layer is a plain nn.Linear
    dict(n_parts=2, sampling_rate=0.5, inductive=True),   # --inductive: partition the train-node subgraph
    dict(n_parts=2, sampling_rate=0.5, shape="tiny-ml", multilabel=True),          # BCE-with-logits (yelp-style)
    dict(n_parts=2, sampling_rate=0.5, model="gcn", n_layers=4, backend="p2p"),    # deeper GCN over the p2p transport
    dict(n_parts=3, sampling_rate=0.5, norm="batch", graph_override={"train": 1.0}),   # --norm batch (SyncBatchNorm)
], ids=["zero-sample", "zero-sample-p2p", "n-linear", "inductive", "multilabel", "gcn4-p2p", "sync-bn"])
def test_training_parity_variants(built, kw):
    kw = dict(kw)
    kw.setdefault("shape", "tiny")
    if kw.get("norm") == "batch":
        # Three epochs, everything compared -- layer outputs, logits, gradients, weights -- except the gradients and
        # values of the biases that sit directly in front of a batch norm (parameters 1, 3, 5: layers.0.linear.bias,
        # layers.1.linear1.bias, layers.1.linear2.bias) -- logits, every other gradient and weight included.  Their true gradient is exactly zero (the mean subtraction
        # removes any constant shift), what is computed is rounding noise, Adam turns noise into +-lr steps, and the
        # next normalisation removes the shift again: they differ between any two implementations and influence nothing.
        from tests.harness import run_parity_case
        res = run_parity_case(device="cuda:0", n_epochs=3, **kw)
        # ... except through what is recorded BEFORE the normalisation: the raw outputs of layers 0 and 1 carry the bias.
        skip = tuple(f"/{k}{i}" for k in ("grad", "param") for i in (1, 3, 5)) + ("/layer0", "/layer1")
        bad = {k: v for k, v in res["detail"].items() if v >= TOL and not k.endswith(skip)}
        assert not bad, sorted(bad.items())
        assert res["index_sets_equal"]
        for a, b in zip(res["loss"], res["loss_oracle"]):
            assert abs(a - b) <= 1e-4 * abs(b)
        return
    _run(n_epochs=2, **kw)


@pytest.mark.parametrize("kw", [
    dict(n_parts=1, sampling_rate=1.0),
    dict(n_parts=2, sampling_rate=1.0, heads=2),
    dict(n_parts=3, sampling_rate=0.5),
    dict(n_parts=3, sampling_rate=0.3, heads=2, backend="p2p", n_layers=3),
    dict(n_parts=2, sampling_rate=0.5, shape="tiny"),            # single-label CE, 5 classes (per-head width padded to 8)
], ids=["p1", "p2-heads2", "p3", "p3-heads2-p2p", "tiny-ce"])
def test_gat_training_parity(built, kw):
    """GAT (module/model.py:96-132 + dgl.nn.GATConv) against the oracle's explicit-edge-list restatement:
    BASELINE configs[3]-style multi-label BCE by default."""
    kw = dict(kw)
    shape = kw.pop("shape", "tiny-ml")
    kw.setdefault("n_layers", 2)
    _run(shape=shape, model="gat", n_epochs=2, multilabel=(shape == "tiny-ml"), **kw)


def test_run_with_eval_writes_checkpoints_and_results(built, tmp_path, monkeypatch):
    """train.run with --eval (train.py:427-456): every log_every epochs rank 0 saves a checkpoint, evaluates on the full
    graph with the same kernels and appends the result line; at the end the best model is saved and tested."""
    import argparse
    import os
    from tests.harness import make_args
    from bns_gcn_b200 import train
    from bns_gcn_b200.data import make_graph, partition_graph
    from bns_gcn_b200.evaluate import checkpoint_path, load_checkpoint, result_file_name
    from bns_gcn_b200.helper.comm import run_threads
    monkeypatch.chdir(tmp_path)
    fg = make_graph("tiny", seed=0)
    parts = partition_graph(fg, 2, "random", seed=0)
    args = make_args(dataset="tiny", model="graphsage", sampling_rate=0.5, n_hidden=16, n_partitions=2, n_epochs=4,
                     log_every=2, eval=True, graph_name="tiny-2-random-vol-trans")

    def fn(comm, r):
        a = argparse.Namespace(**vars(args))
        p = parts[r]
        a.n_feat, a.n_class, a.n_train = p.meta["n_feat"], p.meta["n_class"], p.meta["n_train"]
        st, stats = train.run(p.graph, p.node_dict, p.gpb, a, "cuda:0", full_graph=fg)
        return st.model if r == 0 else None

    model = run_threads(2, fn, device="cuda:0")[0]
    with open(result_file_name(args)) as f:
        lines = f.read().strip().splitlines()
    assert len(lines) == 2 and all("Validation Accuracy" in ln and "Test Accuracy" in ln for ln in lines)
    for e in (1, 3):
        assert os.path.exists(checkpoint_path(args, e))
    assert os.path.exists(checkpoint_path(args))
    load_checkpoint(model, checkpoint_path(args, 3))          # the last periodic checkpoint is the final weights
    sd = torch.load(checkpoint_path(args, 3))
    assert list(sd.keys()) == [k for k, _ in model.named_parameters()]


def test_streaming_precompute_equals_the_materialised_one(built):
    """train.precompute_streaming (one peer's halo rows at a time) == train.precompute (all halo rows at once,
    train.py:170-211), 3 ranks, and the locally generated partitions of data.make_local_partition train to parity with
    the oracle like the ones cut from a full graph."""
    import argparse
    from tests.harness import make_args, run_oracle, run_product, _compare
    from bns_gcn_b200.data import make_local_partition
    P = 3
    parts = [make_local_partition("papers100m", r, P, seed=1, device=torch.device("cpu"), scale=3e-5) for r in range(P)]
    for p in parts:                               # a small feature width keeps the oracle quick
        p.node_dict["feat"] = p.node_dict["feat"][:, :24].contiguous()
        p.meta["n_feat"] = 24
    outs = {}
    for stream in (False, True):
        args = make_args(dataset="papers100m", model="graphsage", sampling_rate=0.5, n_hidden=16, n_partitions=P,
                         streaming_precompute=stream)
        outs[stream] = run_product(parts, args, "cuda:0", 2)
    for r in range(P):
        a, b = outs[True][r]["feat0"], outs[False][r]["feat0"]
        assert ((a - b).norm() / b.norm()).item() < 1e-6
    sel = [[outs[True][r]["selected"][e] for r in range(P)] for e in range(2)]
    args = make_args(dataset="papers100m", model="graphsage", sampling_rate=0.5, n_hidden=16, n_partitions=P)
    orc = run_oracle(parts, args, 2, sel)
    worst, detail = _compare(outs[True], orc, P)
    assert worst < TOL, {k: v for k, v in detail.items() if v >= TOL}


def test_cuda_gat_reproduces_the_reference_golden(built):
    """tests/golden/ref_gat_p2.pt: the reference's OWN GAT model, precompute, construct_feat and epoch loop
    (module/model.py:96-132, train.py:208-209, :284-297, :401-402) run by tests/golden/make_golden.py on 2 gloo
    processes, 2 heads, with dgl.nn.GATConv supplied as a DENSE masked-softmax restatement of DGL 0.9's layer.  The
    CUDA path (entry-list kernels; the 5-class output layer takes the op-by-op path), fed the index sets the reference
    drew, reproduces its stored halo features, head-averaged layer outputs, logits, reduced gradients and updated
    weights within 1e-4 and its boundary sets exactly.

    Epoch 3 of this run has one LayerNorm output about 1e-7 from zero (found by the oracle, which reproduces the golden to
    1e-5), so the f32 forward on the GPU may take the other side of that ReLU kink; the fallback below is the one of the
    eight-partition golden test."""
    import os
    from tests.harness import make_args, run_product, _relerr
    from bns_gcn_b200.data import make_graph, partition_graph
    gold = torch.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_gat_p2.pt"))
    cfg, ranks = gold["config"], gold["ranks"]
    fg = make_graph(cfg["shape"], seed=0)
    parts = partition_graph(fg, cfg["n_parts"], "random", seed=0)
    args = make_args(dataset=cfg["shape"], model=cfg["model"], sampling_rate=cfg["rate"], n_layers=cfg["n_layers"],
                     n_hidden=cfg["n_hidden"], n_partitions=cfg["n_parts"], heads=cfg["heads"])
    sel = [[ranks[r]["selected"][e] for r in range(cfg["n_parts"])] for e in range(cfg["epochs"])]
    out = run_product(parts, args, "cuda:0", cfg["epochs"], selected_per_epoch=sel)
    errs = {}
    for r, o in enumerate(out):
        g = ranks[r]
        for j, b in enumerate(g["boundary"]):
            if b is not None:
                assert torch.equal(o["boundary"][j], b)
        errs[f"r{r}/feat0"] = _relerr(o["feat0"], g["feat0"])
        for i, lo in enumerate(g["layer_out"][-1]):
            errs[f"r{r}/layer{i}"] = _relerr(o["layers"][f"layer{i}"], lo.mean(1))       # the model averages the heads
        errs[f"r{r}/logits"] = _relerr(o["logits"], g["logits"][-1])
        for k, (p, gp, gg) in enumerate(zip(o["params"], g["params"], g["grads"])):
            errs[f"r{r}/param/{g['param_names'][k]}"] = _relerr(p, gp)
            errs[f"r{r}/grad/{g['param_names'][k]}"] = _relerr(o["grads"][k], gg)
    bad = {k: v for k, v in errs.items() if v >= TOL}
    if bad:
        # the oracle (tests/test_oracle_cpu.py pins it to this golden) on the active sets the CUDA forward took; accepted
        # only if every switched entry sat within 1e-4 of zero in the oracle's own forward
        from tests.harness import run_parity_case
        res = run_parity_case(shape=cfg["shape"], n_parts=cfg["n_parts"], model=cfg["model"], sampling_rate=cfg["rate"],
                              n_epochs=cfg["epochs"], n_layers=cfg["n_layers"], n_hidden=cfg["n_hidden"],
                              heads=cfg["heads"], device="cuda:0", selected_per_epoch=sel)
        assert res["kink"] is not None and res["kink"]["flips"] >= 1 and res["kink"]["max_abs_z"] < 1e-4, \
            (sorted(bad.items()), res["kink"])
        assert res["max_rel_err"] < TOL, ({k: v for k, v in res["detail"].items() if v >= TOL}, sorted(bad.items()))
