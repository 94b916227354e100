"""Training data sets that stay resident in HBM, and shuffled mini-batches assembled from them on the device.

Replaces the host-side batching of the reference: PyG ``DataLoader(shuffle=True)`` on the classification side and
``GraphAdjDataset.batchify`` (subgraph_isomorphism/dataset.py:1604-1636) on the counting side.  A data set's columns are
uploaded once.  A mini-batch is an array of graph (sample) indices; for it the host only computes the batch's offsets
from per-graph size tables (a few cumulative sums over the batch), stages ``[indices | offsets]`` in one pinned buffer
and uploads it with one asynchronous copy, and one segmented-gather launch per level (``ops.gather_segments``:
nodes, edges, graphs / samples) writes the batch in the layout the pipelines take.  Nothing is read back from the device.

``EpochSampler`` yields the index arrays of an epoch (shuffled, sharded over data-parallel ranks);
``ClassificationPipeline.step_indices`` / ``CountingPipeline.step_indices`` train on them.
"""
import numpy as np
import torch

from . import ops
from . import transforms as T
from .subgraph_isomorphism.io import _pack

_I32_MAX = 2 ** 31 - 1


class EpochSampler:
    """Mini-batches of indices into a data set of ``num_items`` items, epoch by epoch.

    The order of an epoch is a function of ``(seed, epoch)`` only (numpy's default generator seeded with both), so every
    rank computes the same permutation without communicating; it does not reproduce the order of torch's
    ``RandomSampler``.  Global batch ``s`` of an epoch is ``perm[s * batch_size : (s + 1) * batch_size]``, the last one
    short unless ``drop_last``.  Under ``world_size > 1`` rank ``r`` takes the contiguous slice
    ``[r * n // world_size, (r + 1) * n // world_size)`` of a global batch of ``n`` items (a short last batch with fewer
    items than ranks leaves some ranks an empty slice: pass ``drop_last=True`` then).

    Iterating yields ``(idx, global_batch)``: this rank's host int64 indices and the item count of the whole global
    batch, which ``step_indices(..., global_batch=...)`` uses to weight this rank's gradient by ``len(idx) / global_batch``.
    ``set_epoch(e)`` selects the epoch the next iteration walks (as with torch's ``DistributedSampler``)."""

    def __init__(self, num_items, batch_size, shuffle=True, seed=0, drop_last=False, rank=0, world_size=1):
        num_items, batch_size, world_size, rank = int(num_items), int(batch_size), int(world_size), int(rank)
        if num_items < 0 or batch_size < 1 or world_size < 1 or not 0 <= rank < world_size or int(seed) < 0:
            raise ValueError("EpochSampler: needs num_items >= 0, batch_size >= 1, seed >= 0 and 0 <= rank < world_size")
        if batch_size < world_size:
            raise ValueError("EpochSampler: batch_size %d gives some of the %d ranks no item" % (batch_size, world_size))
        self.num_items, self.batch_size, self.shuffle, self.seed = num_items, batch_size, bool(shuffle), int(seed)
        self.drop_last, self.rank, self.world_size = bool(drop_last), rank, world_size
        self.epoch = 0

    def set_epoch(self, epoch):
        self.epoch = int(epoch)

    def permutation(self, epoch=None):
        """the global order of the items in `epoch` (default: the current one), int64."""
        if not self.shuffle:
            return np.arange(self.num_items, dtype=np.int64)
        e = self.epoch if epoch is None else int(epoch)
        return np.random.default_rng([self.seed, e]).permutation(self.num_items).astype(np.int64)

    def __len__(self):
        full, rest = divmod(self.num_items, self.batch_size)
        return full + (1 if rest and not self.drop_last else 0)

    def batches(self, epoch=None):
        """yields ``(idx, global_batch)`` for every step of `epoch` (default: the current one)."""
        perm = self.permutation(epoch)
        for s in range(len(self)):
            g = perm[s * self.batch_size:(s + 1) * self.batch_size]
            n = len(g)
            yield g[self.rank * n // self.world_size:(self.rank + 1) * n // self.world_size], n

    def __iter__(self):
        return self.batches()


def _offsets(sizes):
    out = np.zeros(len(sizes) + 1, dtype=np.int64)
    np.cumsum(sizes, out=out[1:])
    return out


def _check_indices(idx, n, what):
    """host validation of a batch's index array -> int64 numpy (ValueError before any device work)."""
    if isinstance(idx, torch.Tensor):
        if idx.device.type != "cpu":
            raise ValueError("%s: the indices must be a host array" % what)
        idx = idx.numpy()
    idx = np.asarray(idx)
    if idx.ndim != 1 or not (np.issubdtype(idx.dtype, np.integer) or idx.size == 0):
        raise ValueError("%s: the indices must be a 1-D integer array" % what)
    idx = idx.astype(np.int64, copy=False)
    if idx.size > _I32_MAX:
        raise ValueError("%s: more than 2^31 - 1 indices" % what)
    if idx.size and (int(idx.min()) < 0 or int(idx.max()) >= n):
        raise ValueError("%s: index outside [0, %d)" % (what, n))
    return idx


class _Staging:
    """pinned int32 host buffers for the per-batch index / offset upload.  A buffer is handed out again only after the
    event recorded behind its copy has completed (the copy reads it asynchronously), as PendingLoss does with its pairs."""

    def __init__(self):
        self._bufs = []         # [pinned tensor, event of its latest copy or None]

    def upload(self, parts, device):
        """concatenation of the int64 numpy arrays `parts` as one int32 device tensor (one asynchronous copy on the
        current stream) -> the device views of the parts."""
        n = sum(len(p) for p in parts)
        ent = next((e for e in self._bufs if e[0].numel() >= n and (e[1] is None or e[1].query())), None)
        if ent is None:
            cap = 1 << max(10, (n - 1).bit_length())
            ent = [torch.empty(cap, dtype=torch.int32).pin_memory(), None]
            self._bufs.append(ent)
        host = ent[0].numpy()
        o = 0
        for p in parts:
            host[o:o + len(p)] = p
            o += len(p)
        dev = torch.empty(n, dtype=torch.int32, device=device)
        dev.copy_(ent[0][:n], non_blocking=True)
        ent[1] = torch.cuda.Event()
        ent[1].record()
        views, o = [], 0
        for p in parts:
            views.append(dev[o:o + len(p)])
            o += len(p)
        return views


def _empty_like_rows(col, rows):
    return torch.empty((int(rows),) + tuple(col.shape[1:]), dtype=col.dtype, device=col.device)


def _gather_level(idx_d, ptr_in, ptr_out, cols, rows, rebase=None, rebase_in=None, rebase_out=None):
    """{name: resident column} -> {name: batch column of `rows` items} (one launch for all of them)."""
    names = list(cols)
    out = {k: _empty_like_rows(cols[k], rows) for k in names}
    if names:
        ops.gather_segments(idx_d, ptr_in, ptr_out, [cols[k] for k in names], [out[k] for k in names],
                            [k in (rebase or ()) for k in names], rebase_in, rebase_out)
    return out


# the per-graph columns of a raw TU-shaped data set (graph_classification.io.load_tu_dir / synth.tu_batch) by level
_TU_NODE, _TU_EDGE, _TU_GRAPH = ("vlabel", "vattr"), ("src", "dst", "elabel", "eattr"), ("y",)


class TUGraphTables:
    """Host tables of a raw TU-shaped data set, one entry per graph: node and edge counts and the inputs of
    ``transforms.tu_conjugate_sizes_ex`` (edges, sum over nodes of in-degree * out-degree, has a node, edges sorted by
    source).  A batch's offsets and its size hint are sums and maxima over the selected graphs' entries."""

    def __init__(self, raw):
        node_ptr, edge_ptr = np.asarray(raw["node_ptr"], np.int64), np.asarray(raw["edge_ptr"], np.int64)
        B = len(node_ptr) - 1
        src, dst = np.asarray(raw["src"], np.int64), np.asarray(raw["dst"], np.int64)
        N, E = int(node_ptr[-1]), int(edge_ptr[-1])
        if (B != int(raw["num_graphs"]) or len(edge_ptr) != B + 1 or node_ptr[0] != 0 or edge_ptr[0] != 0
                or (np.diff(node_ptr) < 0).any() or (np.diff(edge_ptr) < 0).any() or len(src) != E or len(dst) != E
                or len(raw["vlabel"]) != N):
            raise ValueError("TU data set: inconsistent node_ptr / edge_ptr / column lengths")
        if N > _I32_MAX or E > _I32_MAX:
            raise ValueError("TU data set: more than 2^31 - 1 nodes or edges")
        e2g = np.repeat(np.arange(B), np.diff(edge_ptr))
        lo, hi = node_ptr[e2g], node_ptr[e2g + 1]
        if ((src < lo) | (src >= hi) | (dst < lo) | (dst >= hi)).any():
            raise ValueError("TU data set: an edge leaves its graph")
        self.num_graphs = B
        self.num_nodes, self.num_edges = np.diff(node_ptr), np.diff(edge_ptr)
        deg = np.bincount(dst, minlength=N) * np.bincount(src, minlength=N)
        self.pairs = np.diff(np.concatenate([[0], np.cumsum(deg)])[node_ptr])
        self.has_node = self.num_nodes > 0
        # edges stay inside their graph and graphs follow each other, so a batch's src is sorted exactly when every
        # selected graph's is
        self.unsorted = np.zeros(B, dtype=bool)
        down = np.flatnonzero(np.diff(src) < 0)
        self.unsorted[e2g[down]] = True

    def check(self, idx):
        return _check_indices(idx, self.num_graphs, "TU data set")

    def offsets(self, idx):
        """(node_ptr, edge_ptr) of the batch of graphs idx (int64)."""
        node_ptr, edge_ptr = _offsets(self.num_nodes[idx]), _offsets(self.num_edges[idx])
        if node_ptr[-1] > _I32_MAX or edge_ptr[-1] > _I32_MAX:
            raise ValueError("TU data set: the batch exceeds 2^31 - 1 nodes or edges")
        return node_ptr, edge_ptr

    def conj_sizes(self, idx):
        """``transforms.tu_conjugate_sizes_ex(<host collation of graphs idx>, with_dummy=True)``."""
        idx = self.check(idx)
        m, has = self.num_edges[idx], self.has_node[idx]
        return (int(m.sum() + has.sum()), int(self.pairs[idx].sum() + 2 * m.sum()), int((m + has).max()) if len(idx) else 0,
                bool(has.all()), not bool(self.unsorted[idx].any()))


class ResidentTUDataset:
    """A raw TU-shaped data set (what ``graph_classification.io.load_tu_dir`` or ``synth.tu_batch`` returns) resident on
    `device`.  ``batch(idx)`` is the raw device batch of graphs ``idx`` (any order, repeats allowed) in exactly the layout
    and dtypes of ``transforms.to_device`` applied to the host collation of those graphs: ``num_graphs``,
    ``has_edge_labels`` (when the data set has it), ``node_ptr``, ``edge_ptr``, ``src`` / ``dst`` (batch-global node
    ids), ``vlabel``, ``elabel`` and, when the data set has them, ``vattr``, ``eattr``, ``y``; plus ``conj_sizes``, the hint
    ``transforms.tu_conjugate_sizes_ex(<that collation>, with_dummy=True)`` computed from the per-graph ``tables``."""

    def __init__(self, raw, device):
        self.device = torch.device(device)
        self.tables = TUGraphTables(raw)
        self._scalars = {k: raw[k] for k in ("has_edge_labels",) if k in raw}
        cols = T.to_device({k: raw[k] for k in _TU_NODE + _TU_EDGE + _TU_GRAPH if k in raw}, self.device)
        self._node = {k: cols[k] for k in _TU_NODE if k in cols}
        self._edge = {k: cols[k] for k in _TU_EDGE if k in cols}
        self._graph = {k: cols[k] for k in _TU_GRAPH if k in cols}
        ptrs = T.to_device(dict(node_ptr=raw["node_ptr"], edge_ptr=raw["edge_ptr"], graph_ptr=np.arange(len(self) + 1)),
                           self.device)
        self._node_ptr, self._edge_ptr, self._graph_ptr = ptrs["node_ptr"], ptrs["edge_ptr"], ptrs["graph_ptr"]
        self._staging = _Staging()
        torch.cuda.synchronize(self.device)

    def __len__(self):
        return self.tables.num_graphs

    def batch(self, idx):
        """raw device batch of graphs `idx` (host integer array, validated here: ValueError before any device work).
        Queued on the current stream: one host->device copy and one gather launch per level with columns."""
        idx = self.tables.check(idx)
        K = len(idx)
        node_ptr, edge_ptr = self.tables.offsets(idx)
        hint = self.tables.conj_sizes(idx)
        idx_d, np_d, ep_d, gp_d = self._staging.upload([idx, node_ptr, edge_ptr, np.arange(K + 1)], self.device)
        out = dict(self._scalars, num_graphs=K, node_ptr=np_d, edge_ptr=ep_d, conj_sizes=hint)
        out.update(_gather_level(idx_d, self._node_ptr, np_d, self._node, node_ptr[-1]))
        out.update(_gather_level(idx_d, self._edge_ptr, ep_d, self._edge, edge_ptr[-1], ("src", "dst"), self._node_ptr, np_d))
        out.update(_gather_level(idx_d, self._graph_ptr, gp_d, self._graph, K))
        return out


_SUB_NODE, _SUB_EDGE = ("vid", "vlabel"), ("src", "dst", "eid", "elabel")


class _ResidentGraphs:
    """distinct pattern or data graphs of a counting data set, packed as ``io._pack`` packs a batch, on the device."""

    def __init__(self, graphs, device):
        b = _pack(graphs)           # ValueError beyond the int32 range
        cols = T.to_device(b, device)
        self.num_nodes, self.num_edges = np.diff(b["node_ptr"].astype(np.int64)), np.diff(b["edge_ptr"].astype(np.int64))
        self.node_ptr, self.edge_ptr = cols["node_ptr"], cols["edge_ptr"]
        self.node = {k: cols[k] for k in _SUB_NODE}
        self.edge = {k: cols[k] for k in _SUB_EDGE}

    def ptrs(self, sel):
        node_ptr, edge_ptr = _offsets(self.num_nodes[sel]), _offsets(self.num_edges[sel])
        if node_ptr[-1] > _I32_MAX or edge_ptr[-1] > _I32_MAX:
            raise ValueError("ResidentCountingDataset: the batch exceeds 2^31 - 1 nodes or edges")
        return node_ptr, edge_ptr

    def gather(self, sel_d, np_d, ep_d, n_nodes, n_edges):
        """the ``io._pack`` batch of the graphs selected by device indices `sel_d` (two launches)."""
        out = dict(num_graphs=int(sel_d.numel()), node_ptr=np_d, edge_ptr=ep_d)
        out.update(_gather_level(sel_d, self.node_ptr, np_d, self.node, n_nodes))
        out.update(_gather_level(sel_d, self.edge_ptr, ep_d, self.edge, n_edges, ("src", "dst"), self.node_ptr, np_d))
        return out


class ResidentCountingDataset:
    """One split of a counting data set (the sample list ``subgraph_isomorphism.io.load_data`` returns per split:
    ``{pattern, graph, subisomorphisms, counts}`` dicts) resident on `device`.  Every distinct pattern and every distinct
    graph (by object identity: the graphs of a shared-graph data set are stored once) is uploaded once; a sample is
    (pattern id, graph id, count, subisomorphism block).

    ``batch(idx)`` -> ``(p_dev, g_dev, counts_dev)``: the device tensors of ``io.collate`` of the samples `idx` (the
    ``io._pack`` layout with int32 indices, ``eid`` = position in the graph; counts int64).  With
    ``subisomorphisms=True`` a fourth item is the ``matching.pack_subisomorphisms`` dict of the same samples on the
    device, for the match-weight targets."""

    def __init__(self, samples, device):
        self.device = torch.device(device)
        pats, gras, pid, gid, where = [], [], [], [], {}
        for x in samples:
            for obj, table, ids, kind in ((x["pattern"], pats, pid, "p"), (x["graph"], gras, gid, "g")):
                key = (kind, id(obj))
                if key not in where:
                    where[key] = len(table)
                    table.append(obj)
                ids.append(where[key])
        self.num_samples = len(pid)
        self._pid, self._gid = np.asarray(pid, np.int64), np.asarray(gid, np.int64)
        self.patterns, self.graphs = _ResidentGraphs(pats, self.device), _ResidentGraphs(gras, self.device)
        mats = []
        for x in samples:           # io.collate's view of the ground truth
            m = np.asarray(x["subisomorphisms"], dtype=np.int64)
            mats.append(m.reshape(-1, x["pattern"]["num_nodes"]) if m.ndim != 2 else m)
        self._val_sizes = np.asarray([m.size for m in mats], np.int64)
        self._rows = np.asarray([m.shape[0] for m in mats], np.int64)    # host copy: the dummy column's offsets
        val_ptr = _offsets(self._val_sizes)
        if val_ptr[-1] > _I32_MAX:
            raise ValueError("ResidentCountingDataset: more than 2^31 - 1 subisomorphism entries")
        values = np.concatenate([m.reshape(-1) for m in mats]) if mats else np.zeros(0, np.int64)
        cols = T.to_device(dict(val_ptr=val_ptr, values=values, rows=self._rows,
                                sample_ptr=np.arange(self.num_samples + 1)), self.device)
        self._val_ptr, self._sample_ptr, self._values, self._rows_d = (cols[k] for k in ("val_ptr", "sample_ptr", "values", "rows"))
        self._counts = torch.as_tensor(np.asarray([int(x["counts"]) for x in samples], np.int64)).to(self.device)
        self._staging = _Staging()
        torch.cuda.synchronize(self.device)

    def __len__(self):
        return self.num_samples

    def batch(self, idx, subisomorphisms=False, dummy_column=False):
        """device batch of samples `idx` (host integer array, validated here: ValueError before any device work); queued
        on the current stream: one host->device copy and 5 gather launches (6 with subisomorphisms).  dummy_column (with
        subisomorphisms): the subisomorphisms come with the dummy column ``add_dummy_nodes_edges`` appends
        (``matching.append_dummy_column``, one more launch; its offsets are computed here on the host)."""
        idx = _check_indices(idx, self.num_samples, "ResidentCountingDataset")
        K = len(idx)
        P, G = self._pid[idx], self._gid[idx]
        pn, pe = self.patterns.ptrs(P)
        gn, ge = self.graphs.ptrs(G)
        parts = [idx, P, G, pn, pe, gn, ge, np.arange(K + 1)]
        if subisomorphisms:
            val_ptr = _offsets(self._val_sizes[idx])
            parts.append(val_ptr)
            if dummy_column:
                from .subgraph_isomorphism.matching import dummy_column_offsets
                parts.append(dummy_column_offsets(self._val_sizes[idx], self._rows[idx]))
            if parts[-1][-1] > _I32_MAX:
                raise ValueError("ResidentCountingDataset: the batch exceeds 2^31 - 1 subisomorphism entries")
        views = self._staging.upload(parts, self.device)
        idx_d, P_d, G_d, pn_d, pe_d, gn_d, ge_d, sp_d = views[:8]
        p_dev = self.patterns.gather(P_d, pn_d, pe_d, pn[-1], pe[-1])
        g_dev = self.graphs.gather(G_d, gn_d, ge_d, gn[-1], ge[-1])
        per_sample = dict(counts=self._counts, rows=self._rows_d) if subisomorphisms else dict(counts=self._counts)
        s = _gather_level(idx_d, self._sample_ptr, sp_d, per_sample, K)
        if not subisomorphisms:
            return p_dev, g_dev, s["counts"]
        vp_d = views[8]
        v = _gather_level(idx_d, self._val_ptr, vp_d, dict(values=self._values), val_ptr[-1])
        sub = dict(val_ptr=vp_d, values=v["values"], rows=s["rows"])
        if dummy_column:
            from .subgraph_isomorphism.matching import append_dummy_column
            sub = append_dummy_column(sub, g_dev, views[9], int(parts[-1][-1]))
        return p_dev, g_dev, s["counts"], sub
