"""GPU: evaluation over a held-out split.  The record and reduction kernels per element against the float64 references
of test_eval.py (records bit for bit where the definition is exact, the reduction bit for bit against the emulation
of its fixed order); ``evaluate`` on both pipelines against the hand-written loop a user would otherwise write; no
interference with CUDA-graph-replayed training; one device->host read; errors; two ranks over NCCL."""
import math
import os
import socket
import tempfile
from argparse import Namespace

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from dummynode4graphlearning_b200 import ops, synth
from dummynode4graphlearning_b200._lib import lib
from dummynode4graphlearning_b200.datasets import ResidentCountingDataset, ResidentTUDataset
from dummynode4graphlearning_b200.graph import _stream, check_errors
from dummynode4graphlearning_b200.subgraph_isomorphism.losses import eval_criterion
from test_eval import reduce_bound, ref_class_rows, ref_count_rows, ref_reduce

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
GUARD = 67          # rows of guard band after the outputs (and pos0 rows before the batch) that must stay untouched


def _bits_equal_f32(a, b):
    """bitwise equality of float32 arrays, any NaN equal to any NaN."""
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    nan = np.isnan(a)
    return np.array_equal(nan, np.isnan(b)) and np.array_equal(a[~nan].view(np.int32), b[~nan].view(np.int32))


# ---- kernels ---------------------------------------------------------------------------------------------------------
def _class_case(B, C, seed):
    g = torch.Generator().manual_seed(seed)
    logp = torch.log_softmax(torch.randn(B, C, generator=g) * 3, 1)
    logp[::4] = logp[::4].round(decimals=0)                 # exact ties inside rows
    if B > 3:
        logp[1] = -0.5                                      # a whole row tied
        logp[2, C // 2] = float("nan")                      # a NaN row
    y = torch.randint(0, C, (B,), generator=g)
    if B > 5:
        y[4], y[5] = -1, C                                  # targets outside [0, C)
    return logp, y


@pytest.mark.parametrize("C", [1, 2, 3, 32])
@pytest.mark.parametrize("B", [1, 31, 32, 33, 20000])
def test_class_rows_kernel(B, C):
    logp, y = _class_case(B, C, 17 * B + C)
    pos0 = 5
    n = pos0 + B + GUARD
    d_logp, d_y = logp.to(DEV), y.to(DEV)
    runs = []
    for _ in range(2):
        pred = torch.full((n,), -777, dtype=torch.int32, device=DEV)
        nll = torch.full((n,), float("nan"), device=DEV)
        correct = torch.full((n,), float("nan"), device=DEV)
        ops.eval_class_rows(d_logp, d_y, pos0, pred, nll, correct)
        runs.append((pred.cpu(), nll.cpu(), correct.cpu()))
    (p0, l0, c0), (p1, l1, c1) = runs
    assert torch.equal(p0, p1) and _bits_equal_f32(l0, l1) and _bits_equal_f32(c0, c1)
    rp, rl, rc = ref_class_rows(logp, y)
    sl = slice(pos0, pos0 + B)
    assert torch.equal(p0[sl].long(), rp)
    assert _bits_equal_f32(l0[sl], rl.float()), "nll is a negation: bit for bit"
    assert torch.equal(c0[sl].double(), rc)
    for band in (slice(0, pos0), slice(pos0 + B, n)):      # nothing written outside the batch's rows
        assert (p0[band] == -777).all() and torch.isnan(l0[band]).all() and torch.isnan(c0[band]).all()


@pytest.mark.parametrize("B", [1, 31, 32, 33, 20000])
def test_count_rows_kernel(B):
    g = torch.Generator().manual_seed(B)
    pred_c = (torch.randn(B, 1, generator=g) * 8).float()          # about half negative: the relu matters
    pred_c[::3] = pred_c[::3].round()                              # exact hits and |d| < 1 terms
    counts = torch.randint(0, 12, (B,), generator=g)
    if B > 2:
        counts[1] = 3 ** 30                                        # not exactly representable in float32
    pos0 = 9
    n = pos0 + B + GUARD
    runs = []
    for _ in range(2):
        pred = torch.full((n,), float("nan"), device=DEV)
        err = torch.full((n, 3), float("nan"), device=DEV)
        ops.eval_count_rows(pred_c.to(DEV), counts.to(DEV), pos0, pred, err)
        runs.append((pred.cpu(), err.cpu()))
    (q0, e0), (q1, e1) = runs
    assert _bits_equal_f32(q0, q1) and _bits_equal_f32(e0, e1)
    sl = slice(pos0, pos0 + B)
    assert _bits_equal_f32(q0[sl], pred_c.view(-1))
    ref = ref_count_rows(pred_c, counts.float())                   # t = float(count), as loss_fn converts it
    got = e0[sl].double()
    assert ((got - ref).abs() <= 4 * 2.0 ** -24 * ref.abs()).all(), float(((got - ref).abs() / ref.abs().clamp_min(1e-30)).max())
    for band in (slice(0, pos0), slice(pos0 + B, n)):
        assert torch.isnan(q0[band]).all() and torch.isnan(e0[band]).all()


@pytest.mark.parametrize("k", [1, 3])
@pytest.mark.parametrize("n", [0, 1, 1000, 4 * 148 * 1024 * 2 + 12345])
def test_reduce_kernel_fixed_order(n, k):
    """bit for bit the emulated fixed order (so: independent of the grid, which the wrapper sizes from the SM count and n
    -- at the largest n the grid is smaller than the tile count, each CTA takes several tiles), within n 2^-53 sum|v| of
    the exact sum, twice the same bits, the ticket counter left at zero."""
    rng = np.random.default_rng(n + k)
    v = (rng.normal(size=(n, k)) * np.exp(rng.uniform(-30, 30, (n, k)))).astype(np.float32)   # order-sensitive sums
    dv = torch.from_numpy(v).to(DEV)
    outs = []
    for _ in range(2):
        out = torch.full((k + 2,), float("nan"), dtype=torch.float64, device=DEV)
        ops.eval_reduce(dv if k > 1 else dv.view(-1), out[:k])
        outs.append(out.cpu().numpy())
    assert np.array_equal(outs[0].view(np.int64), outs[1].view(np.int64))
    assert np.isnan(outs[0][k:]).all()
    got = outs[0][:k]
    assert np.array_equal(got.view(np.int64), ref_reduce(v).view(np.int64)), (got, ref_reduce(v))
    exact = np.array([math.fsum(v[:, c].astype(np.float64)) for c in range(k)])
    assert (np.abs(got - exact) <= reduce_bound(v)).all()
    cnt = ops._tc_scratch[(DEV.index, _stream())][1]
    assert int(cnt.abs().sum()) == 0
    if n == 0:
        assert got.tolist() == [0.0] * k


def test_reduce_counts_correct_rows_exactly():
    n = 3 * 1024 * 1024 + 7
    v = torch.zeros(n, device=DEV)
    v[::3] = 1.0
    out = ops.eval_reduce(v)
    assert float(out[0]) == float((n + 2) // 3)


# ---- pipelines ---------------------------------------------------------------------------------------------------------
def _tu_raw(kind, n, seed):
    if kind == "mutag":
        return synth.tu_batch("mutag", n, seed=seed)
    raw = synth.tu_batch("proteins", n, seed=seed)
    return raw if kind == "proteins_attr" else {k: v for k, v in raw.items() if k != "vattr"}


CLASS_CASES = {
    # name: (data, model, pipeline keywords, num_features)
    "gin_conj_closed_form": ("proteins", "GIN", dict(mode="conj", num_node_labels=2, node_label_min=0), 2),
    "gin_conj_general": ("proteins", "GIN", dict(mode="conj", num_node_labels=2), 2),
    "gin_dummy": ("proteins_attr", "GIN", dict(mode="dummy", num_node_labels=4, node_label_min=0), 5),
    "rgin_edge_attr": ("mutag", "RGIN", dict(mode="dummy", num_node_labels=8, node_label_min=0, num_edge_labels=5,
                                             with_edge_attr=True), 8),
}


def _classifier(name, nf, dropout=0.0, seed=0, device=DEV):
    from dummynode4graphlearning_b200.graph_classification.models import GIN, RGIN
    torch.manual_seed(seed)
    args = Namespace(num_features=nf, hidden_dim=32, num_classes=2, dropout_ratio=dropout, num_relations=5,
                     additional={"train_eps": True, "num_layers": 4, "aggregation": "sum"}, epochs=1, device=str(device))
    return (GIN if name == "GIN" else RGIN)(args).to(device)


def _class_pipe(case, cuda_graphs=True, overlap=None, seed=0, device=DEV):
    from dummynode4graphlearning_b200.optim import FlatAdam
    from dummynode4graphlearning_b200.pipelines import ClassificationPipeline
    data, name, kw, nf = CLASS_CASES[case]
    model = _classifier(name, nf, seed=seed, device=device)
    return ClassificationPipeline(model, FlatAdam(model.parameters(), lr=0.01), cuda_graphs=cuda_graphs, overlap=overlap,
                                  **kw), data


def _batches(idx, bs):
    return [idx[s:s + bs] for s in range(0, len(idx), bs)]


def _hand_loop_class(pipe, ds, idx, bs):
    """what a user writes without evaluate: eval mode, transform, forward, one host read per batch, train mode."""
    pipe.model.eval()
    outs, ys, correct, loss = [], [], 0.0, 0.0
    with torch.no_grad():
        for sel in _batches(idx, bs):
            b = ds.batch(sel)
            if pipe.mode != "conj":
                b.pop("conj_sizes")
            data = pipe.transform(b)
            out = pipe.model(data)
            correct += out.max(1)[1].eq(data.y).sum().item()                 # main.py eval_test
            loss += F.nll_loss(out, data.y, reduction="sum").item()
            outs.append(out.clone())
            ys.append(data.y.clone())
    pipe.model.train()
    return torch.cat(outs), torch.cat(ys), correct / len(idx), loss / len(idx)


@pytest.mark.parametrize("case", sorted(CLASS_CASES))
def test_classification_evaluate_equals_the_hand_written_loop(case):
    pipe, data = _class_pipe(case)
    raw = _tu_raw(data, 300, 21)
    ds = ResidentTUDataset(raw, DEV)
    idx = np.random.default_rng(3).permutation(300)[:251]
    bs = 64
    res = pipe.evaluate(ds, idx, batch_size=bs, log_probs=True)
    m = res.metrics()
    assert pipe.model.training
    out, y, acc_ref, loss_ref = _hand_loop_class(pipe, ds, idx, bs)
    p = res.predictions
    assert torch.equal(p["log_probs"], out)
    assert torch.equal(p["pred"].long(), out.max(1)[1])
    assert torch.equal(p["nll"], -out.gather(1, y.view(-1, 1)).view(-1))
    rp, rl, rc = ref_class_rows(out.cpu(), y.cpu())
    # the metrics are the fixed-order float64 sums of exactly these per-graph values
    assert m["accuracy"] == ref_reduce(rc.float().numpy())[0] / len(idx) == float(rc.sum()) / len(idx)
    assert m["loss"] == ref_reduce(rl.float().numpy())[0] / len(idx)
    assert abs(m["loss"] - math.fsum(rl.tolist()) / len(idx)) <= reduce_bound(rl.float().numpy())[0] / len(idx)
    # ... and agree with the reference's eval_test arithmetic on the same outputs
    assert m["accuracy"] == acc_ref
    assert math.isclose(m["loss"], loss_ref, rel_tol=1e-6)
    # the default split is every graph in order
    full = pipe.evaluate(ds, batch_size=128)
    assert full.predictions["pred"].numel() == 300 and "log_probs" not in full.predictions
    full.metrics()


def _counter(name, device=DEV):
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    from bench_counting import build
    over = dict(rep_rgin_regularizer="bdd", rep_rgin_num_bases=4) if name == "RGIN" else {}
    return build(name, "small", over, device)


@pytest.mark.parametrize("name", ["RGIN", "DMPNN"])
def test_counting_evaluate_equals_the_hand_written_loop(name):
    from dummynode4graphlearning_b200.optim import FlatAdam
    from dummynode4graphlearning_b200.pipelines import CountingPipeline
    model, cfg, kw = _counter(name)
    assert kw["pred_net"] == "SumPredictNet"
    pipe = CountingPipeline(model, FlatAdam(model.parameters(), lr=1e-3), cfg, add_dummy=True)
    samples = synth.counting_samples("small", 120, seed=23)
    ds = ResidentCountingDataset(samples, DEV)
    idx = np.random.default_rng(4).permutation(120)[:101]
    bs = 24
    res = pipe.evaluate(ds, idx, batch_size=bs)
    m = res.metrics()
    assert pipe.model.training
    model.eval()
    preds, cnts = [], []
    with torch.no_grad():
        for sel in _batches(idx, bs):
            p, g, c = ds.batch(sel)
            preds.append(model(*pipe.transform(p, g))["pred_c"].view(-1).clone())
            cnts.append(c.clone())
    model.train()
    pred, counts = torch.cat(preds), torch.cat(cnts)
    assert torch.equal(res.predictions["pred_c"], pred)
    err = ref_count_rows(pred.cpu(), counts.cpu().float())
    n = len(idx)
    for key, col in (("MAE", 0), ("MSE", 1), ("SMSE", 2)):
        assert math.isclose(m[key], float(err[:, col].sum()) / n, rel_tol=1e-6), key
        assert math.isclose(m[key], float(eval_criterion(key)(pred.double().cpu().view(-1, 1), counts.double().cpu().view(-1, 1))),
                            rel_tol=1e-6), key
    assert m["RMSE"] == math.sqrt(m["MSE"])


def _bn_buffers(model):
    return {k: v.detach().clone() for k, v in model.named_buffers()}


def _tensors(obj):
    """every tensor inside a (nested) optimizer state dict, cloned, in a fixed order."""
    if isinstance(obj, torch.Tensor):
        return [obj.detach().clone()]
    if isinstance(obj, dict):
        return [t for k in sorted(obj, key=str) for t in _tensors(obj[k])]
    if isinstance(obj, (list, tuple)):
        return [t for x in obj for t in _tensors(x)]
    return []


def test_evaluate_does_not_disturb_replayed_training():
    """train steps replayed from CUDA graphs with captured transforms on the second stream, interleaved with evaluations:
    every loss and every final parameter equals the same training without evaluations, bit for bit."""
    raw = _tu_raw("proteins", 400, 31)
    ds = ResidentTUDataset(raw, DEV)
    train = [np.arange(s, s + 80) for s in (0, 80, 160)]
    valid = np.arange(240, 400)
    runs = []
    for with_eval in (True, False):
        pipe, _ = _class_pipe("gin_conj_closed_form", cuda_graphs=True, overlap=True, seed=1)
        assert pipe.overlap and pipe.cuda_graphs
        losses = []
        for epoch in range(4):
            for sel in train:
                losses.append(pipe.step_indices(ds, sel))
            if with_eval:
                torch.cuda.synchronize()
                before, caches = _bn_buffers(pipe.model), (dict(pipe._graphs), dict(pipe._tgraphs))
                opt_state = _tensors(pipe.opt.state_dict())
                res = pipe.evaluate(ds, valid, batch_size=48)
                res.metrics()
                torch.cuda.synchronize()
                assert pipe.model.training and all(m.training for m in pipe.model.modules())
                after = _bn_buffers(pipe.model)
                assert all(torch.equal(before[k], after[k]) for k in before), "evaluate changed a BatchNorm buffer"
                assert (dict(pipe._graphs), dict(pipe._tgraphs)) == caches, "evaluate touched the capture caches"
                now = _tensors(pipe.opt.state_dict())
                assert len(now) == len(opt_state) and all(torch.equal(a, b) for a, b in zip(now, opt_state))
        losses = [p.result() for p in losses]
        assert pipe.replayed_library_kernels() > 0 and any(not isinstance(e, str) for e in pipe._tgraphs.values())
        runs.append((losses, {k: v.detach().clone() for k, v in pipe.model.state_dict().items()}))
    (l0, s0), (l1, s1) = runs
    assert l0 == l1
    for k in s0:
        assert torch.equal(s0[k], s1[k]), k


def test_metrics_is_the_only_host_read():
    from torch.profiler import ProfilerActivity, profile
    pipe, data = _class_pipe("gin_conj_closed_form")
    ds = ResidentTUDataset(_tu_raw(data, 600, 41), DEV)
    pipe.evaluate(ds, batch_size=100).metrics()                 # warm-up
    torch.cuda.synchronize()
    reads = lambda prof: [e.name for e in prof.events()                                  # noqa: E731
                          if "DtoH" in e.name or e.name in ("aten::item", "aten::_local_scalar_dense")]
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        res = pipe.evaluate(ds, batch_size=100)
    assert not reads(prof), reads(prof)                         # evaluate itself reads nothing back
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        k0 = lib().kernel_launches()
        m = res.metrics()
        assert lib().kernel_launches() == k0                    # metrics() launches nothing
    d2h = [e.name for e in prof.events() if "DtoH" in e.name]
    assert len(d2h) == 1, d2h
    assert 0.0 <= m["accuracy"] <= 1.0 and m["loss"] > 0


def test_malformed_batch_raises_in_metrics():
    """a graph whose node has more in-edges than DN4GL_MAX_ROW_DEGREE: the CSR build flags it, metrics() raises."""
    hub = 30000
    raw = _tu_raw("proteins_attr", 20, 51)
    n0 = int(raw["node_ptr"][-1])
    src = np.concatenate([raw["src"], n0 + np.arange(1, hub + 1)]).astype(raw["src"].dtype)
    dst = np.concatenate([raw["dst"], np.full(hub, n0)]).astype(raw["dst"].dtype)
    bad = dict(raw, num_graphs=21, src=src, dst=dst, y=np.concatenate([raw["y"], [0]]).astype(raw["y"].dtype),
               node_ptr=np.concatenate([raw["node_ptr"], [n0 + hub + 1]]).astype(raw["node_ptr"].dtype),
               edge_ptr=np.concatenate([raw["edge_ptr"], [raw["edge_ptr"][-1] + hub]]).astype(raw["edge_ptr"].dtype),
               vlabel=np.concatenate([raw["vlabel"], np.ones(hub + 1, raw["vlabel"].dtype)]),
               elabel=np.concatenate([raw["elabel"], np.ones(hub, raw["elabel"].dtype)]),
               vattr=np.concatenate([raw["vattr"], np.zeros((hub + 1,) + raw["vattr"].shape[1:], raw["vattr"].dtype)]))
    pipe, _ = _class_pipe("gin_dummy", cuda_graphs=False)
    ds = ResidentTUDataset(bad, DEV)
    res = pipe.evaluate(ds, batch_size=32)
    with pytest.raises(RuntimeError, match="builder kernel"):
        res.metrics()
    check_errors()                                              # the flag was read and cleared


def test_empty_or_invalid_index_lists_raise_before_device_work():
    pipe, data = _class_pipe("gin_conj_closed_form")
    ds = ResidentTUDataset(_tu_raw(data, 50, 61), DEV)
    torch.cuda.synchronize()
    for bad in ([], np.zeros(0, np.int64), [50], [[1, 2]]):
        k0, m0 = lib().kernel_launches(), torch.cuda.memory_stats(DEV).get("allocation.all.allocated", 0)
        with pytest.raises(ValueError):
            pipe.evaluate(ds, bad)
        assert lib().kernel_launches() == k0
        assert torch.cuda.memory_stats(DEV).get("allocation.all.allocated", 0) == m0


# ---- two ranks over NCCL -----------------------------------------------------------------------------------------------
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


N_DIST, BS_DIST = 203, 64          # the last batch holds 11 graphs: 5 on rank 0, 6 on rank 1


def _dist_eval(dev):
    pipe, data = _class_pipe("gin_conj_closed_form", seed=7, device=dev)
    ds = ResidentTUDataset(_tu_raw(data, N_DIST, 71), dev)
    res = pipe.evaluate(ds, batch_size=BS_DIST)
    return res.metrics(), {k: v.cpu() for k, v in res.predictions.items()}


def _dist_worker(rank, world, port, out_dir):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        m, p = _dist_eval(dev)
        torch.save(dict(metrics=m, predictions=p), os.path.join(out_dir, "rank%d.pt" % rank))
        dist.barrier()
    finally:
        dist.destroy_process_group()


def test_two_rank_nccl_evaluate_equals_single_process():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import torch.multiprocessing as mp
    with tempfile.TemporaryDirectory() as d:
        mp.spawn(_dist_worker, args=(2, _free_port(), d), nprocs=2, join=True)
        r0, r1 = torch.load(os.path.join(d, "rank0.pt")), torch.load(os.path.join(d, "rank1.pt"))
    m1, p1 = _dist_eval(DEV)
    for r in (r0, r1):
        for k in p1:
            assert torch.equal(r["predictions"][k].view(torch.int32), p1[k].view(torch.int32)), k
    bits = lambda m: {k: np.float64(v).view(np.int64) for k, v in m.items()}      # noqa: E731
    assert bits(r0["metrics"]) == bits(r1["metrics"]) == bits(m1)
