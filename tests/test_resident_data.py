"""Host side of the resident data sets (no GPU): the epoch sampler and the per-graph tables the batch offsets and the
conj_sizes hint come from."""
import os

import numpy as np
import pytest

from dummynode4graphlearning_b200 import synth, transforms as T
from dummynode4graphlearning_b200.datasets import EpochSampler, TUGraphTables
from dummynode4graphlearning_b200.graph_classification.io import load_tu_dir
from helpers import nasty_tu_batch


def collate_tu(raw, idx):
    """plain per-graph loop: the raw TU-shaped host batch of graphs idx, in the layout of synth.tu_batch."""
    node_ptr, edge_ptr = [0], [0]
    parts = {k: [] for k in ("src", "dst", "vlabel", "elabel", "vattr", "eattr", "y") if k in raw}
    for g in idx:
        n0, n1 = int(raw["node_ptr"][g]), int(raw["node_ptr"][g + 1])
        e0, e1 = int(raw["edge_ptr"][g]), int(raw["edge_ptr"][g + 1])
        for k in parts:
            if k in ("src", "dst"):
                parts[k].append(np.asarray(raw[k][e0:e1], np.int64) - n0 + node_ptr[-1])
            elif k in ("vlabel", "vattr"):
                parts[k].append(np.asarray(raw[k][n0:n1]))
            elif k in ("elabel", "eattr"):
                parts[k].append(np.asarray(raw[k][e0:e1]))
            else:
                parts[k].append(np.asarray(raw[k][g:g + 1]))
        node_ptr.append(node_ptr[-1] + n1 - n0)
        edge_ptr.append(edge_ptr[-1] + e1 - e0)
    out = {k: np.concatenate(v) if v else np.zeros((0,) + np.shape(raw[k])[1:], np.asarray(raw[k]).dtype)
           for k, v in parts.items()}
    out.update(num_graphs=len(idx), node_ptr=np.asarray(node_ptr, np.int32), edge_ptr=np.asarray(edge_ptr, np.int32))
    if "has_edge_labels" in raw:
        out["has_edge_labels"] = raw["has_edge_labels"]
    return out


# ---- sampler ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,bs,shuffle", [(103, 10, True), (100, 10, True), (7, 10, True), (50, 8, False)])
def test_sampler_covers_every_index_once_per_epoch(n, bs, shuffle):
    s = EpochSampler(n, bs, shuffle=shuffle, seed=3)
    for epoch in range(3):
        s.set_epoch(epoch)
        steps = list(s)
        assert len(steps) == len(s) == -(-n // bs)
        seen = np.concatenate([idx for idx, _ in steps])
        assert seen.dtype == np.int64
        assert np.array_equal(np.sort(seen), np.arange(n))
        assert all(len(idx) == gb for idx, gb in steps)
        assert all(len(idx) == bs for idx, _ in steps[:-1])
    if not shuffle:
        assert np.array_equal(np.concatenate([i for i, _ in s]), np.arange(n))


def test_sampler_is_a_function_of_seed_and_epoch():
    a = [EpochSampler(1000, 64, seed=5, rank=r, world_size=2) for r in range(2)]
    assert np.array_equal(a[0].permutation(2), a[1].permutation(2))
    assert np.array_equal(a[0].permutation(2), EpochSampler(1000, 64, seed=5).permutation(2))
    assert not np.array_equal(a[0].permutation(0), a[0].permutation(1))
    assert not np.array_equal(a[0].permutation(0), EpochSampler(1000, 64, seed=6).permutation(0))
    s = EpochSampler(1000, 64, seed=5)
    s.set_epoch(4)
    assert np.array_equal(np.concatenate([i for i, _ in s]), s.permutation(4))
    assert np.array_equal(np.concatenate([i for i, _ in s.batches(1)]), s.permutation(1))


@pytest.mark.parametrize("drop_last", [False, True])
@pytest.mark.parametrize("n,bs,world", [(1000, 64, 4), (1003, 100, 3), (257, 16, 8), (64, 64, 1)])
def test_rank_slices_partition_every_global_batch(n, bs, world, drop_last):
    ranks = [list(EpochSampler(n, bs, seed=1, drop_last=drop_last, rank=r, world_size=world).batches(2))
             for r in range(world)]
    whole = list(EpochSampler(n, bs, seed=1, drop_last=drop_last).batches(2))
    assert all(len(r) == len(whole) for r in ranks)
    total = 0
    for step, (g, gb) in enumerate(whole):
        parts = [ranks[r][step][0] for r in range(world)]
        assert all(ranks[r][step][1] == gb == len(g) for r in range(world))
        assert np.array_equal(np.concatenate(parts), g)          # contiguous slices in rank order, disjoint
        assert max(len(p) for p in parts) - min(len(p) for p in parts) <= 1
        total += gb
    assert total == (n // bs * bs if drop_last else n)


def test_sampler_rejects_bad_arguments():
    for kw in (dict(num_items=-1, batch_size=4), dict(num_items=10, batch_size=0), dict(num_items=10, batch_size=4, rank=2,
               world_size=2), dict(num_items=10, batch_size=2, world_size=4), dict(num_items=10, batch_size=4, seed=-1)):
        with pytest.raises(ValueError):
            EpochSampler(**kw)


# ---- per-graph tables ------------------------------------------------------------------------------------------------
def _write_tu_dir(d, b, trailing_edgeless):
    """TU text files of batch b followed by `trailing_edgeless` graphs without edges (1-based global node ids)."""
    B, N = int(b["num_graphs"]), int(b["node_ptr"][-1])
    gi = np.repeat(np.arange(1, B + 1), np.diff(b["node_ptr"]))
    extra = np.repeat(np.arange(B + 1, B + 1 + len(trailing_edgeless)), trailing_edgeless)
    os.makedirs(d)
    with open(os.path.join(d, "X_A.txt"), "w") as f:
        f.writelines("%d, %d\n" % (s + 1, t + 1) for s, t in zip(b["src"], b["dst"]))
    with open(os.path.join(d, "X_graph_indicator.txt"), "w") as f:
        f.writelines("%d\n" % g for g in np.concatenate([gi, extra]))
    with open(os.path.join(d, "X_node_labels.txt"), "w") as f:
        f.writelines("%d\n" % v for v in np.concatenate([b["vlabel"], np.ones(len(extra), np.int64)]))
    with open(os.path.join(d, "X_graph_labels.txt"), "w") as f:
        f.writelines("%d\n" % v for v in np.concatenate([b["y"], np.zeros(len(trailing_edgeless), np.int64)]))
    return N


def _check_hint(raw, rng, sets=20):
    t = TUGraphTables(raw)
    B = int(raw["num_graphs"])
    for i in range(sets):
        K = int(rng.integers(1, 2 * B + 1))
        idx = rng.integers(0, B, K) if i % 2 else rng.permutation(B)[:min(K, B)]     # with / without repeats
        host = collate_tu(raw, idx)
        assert t.conj_sizes(idx) == T.tu_conjugate_sizes_ex(host, with_dummy=True), idx
        node_ptr, edge_ptr = t.offsets(idx)
        assert np.array_equal(node_ptr, host["node_ptr"]) and np.array_equal(edge_ptr, host["edge_ptr"])
    assert t.conj_sizes([]) == T.tu_conjugate_sizes_ex(collate_tu(raw, []), with_dummy=True)


def test_hint_from_tables_equals_host_hint_synthetic():
    rng = np.random.default_rng(0)
    _check_hint(synth.tu_batch("proteins", 60, seed=2), rng)
    _check_hint(synth.tu_batch("mutag", 40, seed=3), rng)


def test_hint_from_tables_equals_host_hint_nasty(tmp_path):
    """self loops, duplicate and unsorted edges, single-node graphs, graphs without edges -- also trailing ones, which
    load_tu_dir keeps only with keep_trailing_edgeless=True (such graphs have a node but no edge)."""
    rng = np.random.default_rng(1)
    for trial in range(4):
        b = nasty_tu_batch(rng, 30)
        _check_hint(b, rng)
        d = str(tmp_path / ("t%d" % trial))
        _write_tu_dir(d, b, trailing_edgeless=[1, 3, 1])
        raw = load_tu_dir(d, keep_trailing_edgeless=True)
        assert raw["num_graphs"] == 33 and np.diff(raw["edge_ptr"])[-3:].tolist() == [0, 0, 0]
        _check_hint(raw, rng)
        t = TUGraphTables(raw)
        assert t.conj_sizes([32, 30])[3] and t.conj_sizes([31])[:3] == (1, 0, 1)   # single-node graph: just its dummy
    sorted_only = synth.tu_batch("mutag", 5, seed=1)
    assert TUGraphTables(sorted_only).conj_sizes(np.arange(5))[4]


def test_tables_validate_indices_and_data_set():
    raw = synth.tu_batch("mutag", 6, seed=1)
    t = TUGraphTables(raw)
    for bad in ([6], [-1], [[0, 1]], np.array([0.5]), np.array([True])):
        with pytest.raises(ValueError):
            t.conj_sizes(bad)
    broken = dict(raw, dst=raw["dst"].copy())
    broken["dst"][0] = int(raw["node_ptr"][-1]) - 1        # an edge of graph 0 pointing into the last graph
    with pytest.raises(ValueError, match="leaves its graph"):
        TUGraphTables(broken)
