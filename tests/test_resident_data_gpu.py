"""Resident data sets on the GPU: batches assembled by the segmented gather are bitwise the uploaded host collations, the
gather kernel writes every output item deterministically in one launch per level, and step_indices trains exactly as
step does on the host-collated batch."""
from argparse import Namespace

import numpy as np
import pytest
import torch

from dummynode4graphlearning_b200 import ops, synth, transforms as T
from dummynode4graphlearning_b200._lib import lib
from dummynode4graphlearning_b200.datasets import ResidentCountingDataset, ResidentTUDataset
from dummynode4graphlearning_b200.pipelines import pin_batch
from dummynode4graphlearning_b200.subgraph_isomorphism import io as sio
from dummynode4graphlearning_b200.subgraph_isomorphism.matching import pack_subisomorphisms
from helpers import nasty_tu_batch
from test_resident_data import collate_tu

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")


def _assert_same(a, b, what):
    assert set(a) == set(b), (what, sorted(a), sorted(b))
    for k in a:
        x, y = a[k], b[k]
        if isinstance(y, torch.Tensor):
            assert x.dtype == y.dtype and x.shape == y.shape and x.device == y.device, (what, k, x.dtype, y.dtype, x.shape, y.shape)
            assert torch.equal(x.view(torch.int32) if x.is_floating_point() else x,
                               y.view(torch.int32) if y.is_floating_point() else y), (what, k)
        else:
            assert x == y and type(x) is type(y), (what, k, x, y)


def _tu_sets():
    mutag = synth.tu_batch("mutag", 60, seed=4)
    proteins = synth.tu_batch("proteins", 80, seed=5)
    wide = dict(proteins, vattr=np.random.default_rng(0).normal(size=(int(proteins["node_ptr"][-1]), 2)).astype(np.float32),
                eattr=np.random.default_rng(1).normal(size=int(proteins["edge_ptr"][-1])))
    nasty = nasty_tu_batch(np.random.default_rng(2), 40)        # self loops, single-node and edgeless graphs
    return dict(mutag=mutag, proteins=proteins, wide=wide, nasty=nasty)


@pytest.mark.parametrize("name", ["mutag", "proteins", "wide", "nasty"])
def test_tu_batch_is_the_uploaded_host_collation(name):
    raw = _tu_sets()[name]
    ds = ResidentTUDataset(raw, DEV)
    rng = np.random.default_rng(7)
    B = len(ds)
    for i in range(6):
        idx = rng.permutation(B)[:int(rng.integers(1, B))] if i % 2 else rng.integers(0, B, int(rng.integers(1, 2 * B)))
        host = collate_tu(raw, idx)
        host["conj_sizes"] = T.tu_conjugate_sizes_ex(host, with_dummy=True)
        _assert_same(ds.batch(idx), T.to_device(host, DEV), (name, i))


def _counting_sets():
    shared = synth.counting_samples("small", 48, seed=3, num_patterns=4)
    own = synth.counting_samples("small", 48, seed=4)
    return dict(shared=shared, own=own)


@pytest.mark.parametrize("name", ["shared", "own"])
def test_counting_batch_is_the_uploaded_collation(name):
    samples = _counting_sets()[name]
    ds = ResidentCountingDataset(samples, DEV)
    if name == "shared":
        assert ds.graphs.num_nodes.size == 12 and ds.patterns.num_nodes.size == 4      # each graph stored once
    rng = np.random.default_rng(8)
    for i in range(5):
        idx = rng.integers(0, len(samples), int(rng.integers(1, 64))) if i % 2 else rng.permutation(len(samples))[:20]
        p, g, counts, mats = sio.collate([samples[j] for j in idx])
        pd_, gd_, cd_, sub = ds.batch(idx, subisomorphisms=True)
        _assert_same(pd_, T.to_device(p, DEV), (name, "pattern"))
        _assert_same(gd_, T.to_device(g, DEV), (name, "graph"))
        _assert_same(dict(c=cd_), dict(c=torch.from_numpy(counts).to(DEV)), (name, "counts"))
        _assert_same(sub, pack_subisomorphisms(mats, DEV), (name, "subisomorphisms"))
        three = ds.batch(idx)
        assert len(three) == 3 and torch.equal(three[2], cd_)


def test_gather_kernel_writes_every_item_deterministically():
    """one level with an int32 rebased column, a 3-wide float column and an int64 column, segments of length 0..9 taken
    in any order with repeats: outputs pre-filled with a sentinel come back equal to the numpy gather, twice."""
    rng = np.random.default_rng(11)
    n_seg = 500
    lens = rng.integers(0, 10, n_seg)
    lens[::7] = 0
    ptr_in = np.concatenate([[0], np.cumsum(lens)])
    rebase_in = np.concatenate([[0], np.cumsum(rng.integers(0, 5, n_seg))])
    M = int(ptr_in[-1])
    a = rng.integers(-1000, 1000, M).astype(np.int32)
    f = rng.normal(size=(M, 3)).astype(np.float32)
    y = rng.integers(-2 ** 40, 2 ** 40, M)
    idx = rng.integers(0, n_seg, 3000)
    ptr_out = np.concatenate([[0], np.cumsum(lens[idx])])
    rebase_out = np.concatenate([[0], np.cumsum(rng.integers(0, 5, len(idx)))])
    sel = np.concatenate([np.arange(ptr_in[g], ptr_in[g + 1]) for g in idx])
    shift = np.repeat(rebase_out[:-1] - rebase_in[idx], lens[idx])
    want = [a[sel] + shift, f[sel], y[sel]]
    d = lambda x: torch.from_numpy(np.ascontiguousarray(x)).to(DEV)     # noqa: E731
    i32 = lambda x: d(np.asarray(x, np.int32))                           # noqa: E731
    cols = [d(a), d(f), d(y)]
    outs = []
    for run in range(2):
        out = [torch.full((int(ptr_out[-1]),) + tuple(c.shape[1:]), -7, dtype=c.dtype, device=DEV) for c in cols]
        k0 = lib().kernel_launches()
        ops.gather_segments(i32(idx), i32(ptr_in), i32(ptr_out), cols, out, [True, False, False], i32(rebase_in),
                            i32(rebase_out))
        assert lib().kernel_launches() - k0 == 1
        torch.cuda.synchronize()
        for o, w in zip(out, want):
            assert np.array_equal(o.cpu().numpy(), w.astype(o.cpu().numpy().dtype))
        outs.append(out)
    for x, z in zip(*outs):
        assert torch.equal(x, z)


def test_launches_per_batch_and_validation_before_device_work():
    raw = _tu_sets()["wide"]                    # vattr (2 wide) and eattr share their level's launch
    ds = ResidentTUDataset(raw, DEV)
    L = lib()
    k0 = L.kernel_launches()
    ds.batch(np.arange(0, 80, 3))
    assert L.kernel_launches() - k0 == 3        # nodes, edges, graphs
    cs = ResidentCountingDataset(_counting_sets()["shared"], DEV)
    k0 = L.kernel_launches()
    cs.batch(np.arange(10))
    assert L.kernel_launches() - k0 == 5        # pattern nodes, pattern edges, graph nodes, graph edges, samples
    k0 = L.kernel_launches()
    cs.batch(np.arange(10), subisomorphisms=True)
    assert L.kernel_launches() - k0 == 6        # ... and the subisomorphism values
    torch.cuda.synchronize()
    for bad_tu, bad_cs in (([80], [48]), ([-1], [-1]), (np.array([0, 1.0]), np.array([0, 1.0])), ([[1]], [[1]])):
        k0, m0 = L.kernel_launches(), torch.cuda.memory_stats(DEV).get("allocation.all.allocated", 0)
        with pytest.raises(ValueError):
            ds.batch(bad_tu)
        with pytest.raises(ValueError):
            cs.batch(bad_cs)
        assert L.kernel_launches() == k0
        assert torch.cuda.memory_stats(DEV).get("allocation.all.allocated", 0) == m0


# ---- pipelines ---------------------------------------------------------------------------------------------------------
def _gin(num_features):
    from dummynode4graphlearning_b200.graph_classification.models import GIN
    torch.manual_seed(0)
    args = Namespace(num_features=num_features, hidden_dim=32, num_classes=2, dropout_ratio=0.0,
                     additional={"train_eps": True, "num_layers": 4, "aggregation": "sum"}, epochs=1, device="cuda:0")
    return GIN(args).to(DEV)


def _params(model):
    return {k: v.detach().clone() for k, v in model.state_dict().items()}


@pytest.mark.parametrize("mode", ["conj", "dummy"])
def test_classification_step_indices_equals_step_on_host_collation(mode):
    from dummynode4graphlearning_b200.optim import FlatAdam
    from dummynode4graphlearning_b200.pipelines import ClassificationPipeline
    raw = synth.tu_batch("proteins", 300, seed=9)
    if mode == "conj":          # the closed-form CONJ_ builder: labels only, size hint attached
        raw = {k: v for k, v in raw.items() if k != "vattr"}
        nf, kw = 2, dict(num_node_labels=2, node_label_min=0)
    else:                       # DUMMY_ graphs with the node attribute: x = [vattr, one-hot(label 0..3)]
        nf, kw = 5, dict(num_node_labels=4, node_label_min=0)
    ds = ResidentTUDataset(raw, DEV)
    rng = np.random.default_rng(12)
    sets = [rng.permutation(300)[:n] for n in (111, 97, 120)]
    runs = []
    for resident in (True, False):
        model = _gin(nf)
        pipe = ClassificationPipeline(model, FlatAdam(model.parameters(), lr=0.01), mode=mode, **kw)
        losses = []
        for idx in sets:
            if resident:
                losses.append(pipe.step_indices(ds, idx).result())
            else:
                host = collate_tu(raw, idx)
                if mode == "conj":
                    host["conj_sizes"] = T.tu_conjugate_sizes_ex(host, with_dummy=True)
                losses.append(pipe.step(pin_batch(host)))
        runs.append((losses, _params(model)))
    (l0, s0), (l1, s1) = runs
    assert l0 == l1, (l0, l1)
    for k in s0:
        assert torch.equal(s0[k], s1[k]), k


def test_classification_step_indices_reads_nothing_back_in_conj_mode():
    """with the hint and the label range, the transform is the closed-form builder: no device->host copy in the step."""
    from dummynode4graphlearning_b200.optim import FlatAdam
    from dummynode4graphlearning_b200.pipelines import ClassificationPipeline
    raw = {k: v for k, v in synth.tu_batch("proteins", 200, seed=10).items() if k != "vattr"}
    ds = ResidentTUDataset(raw, DEV)
    model = _gin(2)
    pipe = ClassificationPipeline(model, FlatAdam(model.parameters(), lr=0.01), mode="conj", num_node_labels=2,
                                  node_label_min=0)
    pipe.step_indices(ds, np.arange(0, 100)).result()
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        pending = pipe.step_indices(ds, np.arange(100, 200))
        torch.cuda.synchronize()
    pending.result()
    d2h = [e.name for e in prof.events() if "DtoH" in e.name]
    assert len(d2h) <= 2, d2h       # the loss and the error flag PendingLoss queues behind the step; nothing else
    assert not [e for e in prof.events() if e.name in ("aten::item", "aten::_local_scalar_dense")]


def test_counting_step_indices_equals_step_on_host_collation():
    import os
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    from bench_counting import build
    from dummynode4graphlearning_b200.optim import FlatAdam
    from dummynode4graphlearning_b200.pipelines import CountingPipeline
    samples = synth.counting_samples("small", 96, seed=13)
    ds = ResidentCountingDataset(samples, DEV)
    rng = np.random.default_rng(14)
    sets = [rng.permutation(96)[:n] for n in (32, 29, 35)]
    runs = []
    for resident in (True, False):
        model, cfg, _ = build("RGIN", "small", dict(rep_rgin_regularizer="bdd", rep_rgin_num_bases=4), DEV)
        opt = FlatAdam(model.parameters(), lr=1e-3, weight_decay=1e-2, amsgrad=True, decoupled_weight_decay=True)
        pipe = CountingPipeline(model, opt, cfg, add_dummy=True, rep_reg_w=1e-3)
        losses = []
        for idx in sets:
            if resident:
                losses.append(pipe.step_indices(ds, idx).result())
            else:
                p, g, counts, _ = sio.collate([samples[j] for j in idx])
                losses.append(pipe.step(pin_batch(p), pin_batch(g), torch.from_numpy(counts)))
        runs.append((losses, _params(model)))
    (l0, s0), (l1, s1) = runs
    assert l0 == l1, (l0, l1)
    for k in s0:
        assert torch.equal(s0[k], s1[k]), k
