"""End-to-end public API: host graph batches in, loss out.

``ClassificationPipeline.step(host_batch)`` is the call a user of the classification side makes per
mini-batch: pinned host arrays of RAW TU-shaped graphs -> H2D -> dummy augmentation -> edge-to-vertex
transform -> PyG canonicalisation -> CSR build -> GIN forward + nll_loss + backward -> (gradient all-reduce)
-> Adam step -> loss read back.  Everything between the two copies runs on the GPU; it replaces the
reference's offline ``tu_data_processing.py`` + ``PYGDataset`` + ``main.py:train`` loop body
(tu_data_processing.py:417-455, graph_neural_networks/dataset.py:141-168, main.py:37-43).

``CountingPipeline.step(pattern, graph, counts)`` does the same for the subgraph-counting side
(train.py:1322-1334 augmentation + train_epoch body :753-838).
"""
import contextlib

import numpy as np
import torch
import torch.nn.functional as F

from . import ops
from . import transforms as T
from .graph import BatchedGraph
from .graph_classification.data import Batch
from .parallel import GradientBucket, is_distributed, sync_padded_lengths

_HOST_KEYS = ("node_ptr", "edge_ptr", "src", "dst", "vlabel", "elabel", "vid", "eid", "y", "vattr", "e_is_reversed")


def pin_batch(b):
    """numpy batch dict -> pinned host tensors (int32 / float32 / int64 for y)."""
    out = {}
    for k, v in b.items():
        if k in _HOST_KEYS:
            t = torch.as_tensor(np.ascontiguousarray(v))
            out[k] = t.pin_memory() if torch.cuda.is_available() else t
        else:
            out[k] = v
    return out


def host_bytes(b):
    return int(sum(v.numel() * v.element_size() for v in b.values() if isinstance(v, torch.Tensor)))


def upload(b, device):
    out = {}
    for k, v in b.items():
        out[k] = v.to(device, non_blocking=True) if isinstance(v, torch.Tensor) else v
    return out


def _structure_tensors(data):
    """every device tensor the GIN / RGIN train step reads from a compiled Batch, in a fixed order, plus the host
    scalars that are baked into kernel arguments (the CUDA-graph signature)."""
    s = data.structure
    tensors = [data.x, data.y, s.node_ptr, s.row2seg]
    scalars = [s.num_nodes]
    for csr in (s.csr_in, s.csr_out):
        tensors += [csr.row_ptr, csr.col, csr.heavy_rows, csr.heavy_count]
        scalars += [csr.n_rows, csr.nnz, csr.heavy_thr, csr.max_seg]
        for key in sorted(csr._tiles):
            t = csr._tiles[key]
            tensors += [t["desc"], t["heavy_list"], t["heavy_count"]]
            scalars += [key] + [t[k] for k in ("T", "heavy_cap", "smem", "stages", "npr", "window", "cap_rows", "warps")]
    return tensors, scalars


def _signature(tensors, scalars):
    """CUDA-graph signature of a train step from the tensors it reads and the host scalars baked into its launches."""
    return (tuple(None if t is None else (tuple(t.shape), t.dtype) for t in tensors), tuple(scalars))


def _static_clone(data):
    """a Batch with the same compiled structure whose tensors are private copies (the buffers a captured CUDA graph
    reads).  The tilings are copied: the captured forward reads them as they are (_structure_tensors lists them)."""
    import copy
    s0 = data.structure
    d = Batch(data.x.clone(), None, None, y=data.y.clone())
    s = copy.copy(s0)
    s.node_ptr = s0.node_ptr.clone()
    s._row2seg = None if s0.row2seg is None else s0.row2seg.clone()
    s._rel = {}
    for name in ("csr_in", "csr_out"):
        setattr(s, name, getattr(s0, name).clone(s.node_ptr, eid=False, tiles=True))
    d._structure = s
    return d


class PendingLoss:
    """loss of a step that is still in flight: the device->host copy has been queued behind the step on its stream;
    ``result()`` waits for that copy only (not for later work) and returns the python float."""

    _free = {}      # device index -> pinned (loss, error code) buffers that no unresolved PendingLoss owns

    def __init__(self, loss):
        from .graph import error_flag
        self.dev = loss.device.index
        pool = PendingLoss._free.setdefault(self.dev, [])
        # one private pinned pair per unresolved result (handed back by result()): any number of steps may be in flight
        self.buf, self.err = pool.pop() if pool else (torch.empty(1, dtype=torch.float32).pin_memory(),
                                                     torch.empty(1, dtype=torch.int32).pin_memory())
        self.buf.copy_(loss.detach().reshape(1), non_blocking=True)
        # the builder kernels' sticky asynchronous error flag travels with the loss: result() raises instead of returning
        # a number computed from a malformed CSR (row above DN4GL_MAX_ROW_DEGREE, unsorted keys, wrong size hint)
        self.flag = error_flag(loss.device)
        self.err.copy_(self.flag, non_blocking=True)
        self.event = torch.cuda.Event()
        self.event.record()
        self.value = None

    def result(self):
        if self.value is None:
            self.event.synchronize()
            self.value, code = float(self.buf[0]), int(self.err[0])
            PendingLoss._free[self.dev].append((self.buf, self.err))
            self.buf = self.err = None
            if code != 0:
                from .graph import check_errors
                check_errors()          # reads, clears and raises with the code table
        return self.value


class EvalResult:
    """what ``evaluate`` returns before the device has finished: ``predictions`` (device tensors in the order of the
    evaluated indices) and the queued float64 sums behind ``metrics()``."""

    def __init__(self, sums, n, finish, predictions):
        self._sums, self.n, self._finish, self.predictions = sums, n, finish, predictions
        self._metrics = None

    def metrics(self):
        """host dict of the split's metrics.  The one device->host read of the evaluation: the column sums together with
        the builder kernels' sticky error flag, which raises here (as in ``PendingLoss.result()``) instead of returning
        numbers computed from a malformed batch structure."""
        if self._metrics is None:
            host = self._sums.cpu().tolist()
            if host[-1] != 0:
                from .graph import check_errors
                check_errors()          # reads, clears and raises with the code table
            self._metrics = self._finish(host[:-1], self.n)
        return dict(self._metrics)


class _CapturedGraph:
    """one CUDA graph of ``fn()``, captured on `stream` (default: torch's own capture stream).  ``replay()`` does the
    captured work again and returns what ``fn()`` returned during the capture (static tensors)."""

    def __init__(self, fn, stream=None):
        from ._lib import lib
        self.graph, self.replays = torch.cuda.CUDAGraph(), 0
        k0 = lib().kernel_launches()
        with torch.cuda.graph(self.graph, stream=stream):
            self.out = fn()
        self.library_kernels = lib().kernel_launches() - k0   # libdn4gl kernels inside the graph (launched per replay)

    def replay(self):
        self.graph.replay()
        self.replays += 1
        return self.out


class _CapturedStep(_CapturedGraph):
    """one train step (forward, loss, backward, gradient all-reduce, optimizer step) for ONE batch signature, captured as
    ``body(*batch)`` on `batch`, a private copy of a batch whose tensors ``describe(*batch)`` lists.  ``load()`` of
    another batch of the signature followed by ``replay()`` does all of that work again on that batch's data."""

    def __init__(self, body, batch, describe):
        self.batch, self.static = batch, describe(*batch)[0]
        torch.cuda.synchronize()
        # the AccumulateGrad nodes were created by the eager steps on the default stream; capture runs them on the
        # capture stream, which is intended here
        torch.autograd.graph.set_warn_on_accumulate_grad_stream_mismatch(False)
        super().__init__(lambda: body(*batch))

    def load(self, tensors):
        """copies a batch's tensors (in ``describe`` order) into the buffers the graph reads."""
        pairs = [(d, s) for d, s in zip(self.static, tensors) if d is not None]
        torch._foreach_copy_([d for d, _ in pairs], [s for _, s in pairs])


class _CapturedTransform(_CapturedGraph):
    """CUDA graph of the whole transform (dummy augmentation, edge-to-vertex transform, canonicalisation, both CSR builds,
    tilings) for ONE raw-batch signature.  Only possible when the transform has no device->host read, i.e. when the
    loader attached ``conj_sizes`` (transforms.tu_conjugate_sizes).  The ~60 small launches that the eager transform paces
    from the host (0.6 ms of host time per C2 batch) become one graph launch; the outputs are static tensors, so a replay
    must not start before the train step that consumes the previous outputs has copied them (``wait`` event)."""

    def __init__(self, pipe, dev_batch):
        cur = torch.cuda.current_stream()
        cur.synchronize()
        self.static_in = {k: (v.clone() if isinstance(v, torch.Tensor) else v) for k, v in dev_batch.items()}
        on_side = cur != torch.cuda.default_stream(cur.device)      # capture must not run on the legacy default stream
        super().__init__(lambda: pipe._transform_eager(self.static_in), stream=cur if on_side else None)

    def run(self, batch, wait=None):
        """batch: device OR pinned-host tensors of the captured signature (copied into the graph's input buffers)."""
        if wait is not None:
            torch.cuda.current_stream().wait_event(wait)
        for k, v in batch.items():
            if isinstance(v, torch.Tensor):
                d = self.static_in[k]
                d.copy_(v if v.dtype == d.dtype else v.to(d.dtype), non_blocking=True)
        return self.replay()


def _raw_signature(b):
    return tuple(sorted((k, (tuple(v.shape), str(v.dtype)) if isinstance(v, torch.Tensor) else
                         (tuple(v) if isinstance(v, (tuple, list)) else v)) for k, v in b.items()))


class _Pipeline:
    """what both pipelines share: the CUDA-graph cache of the train step and the overlapped step, whose transform runs on
    a second stream while the previous train step still runs on the current one."""

    _caches = ("_graphs",)      # attributes that hold captured graphs by signature

    def __init__(self, model, optimizer, cuda_graphs, max_graphs, overlap):
        self.model, self.opt = model, optimizer
        self.bucket = getattr(optimizer, "bucket", None) or GradientBucket(model.parameters())
        self.device = next(model.parameters()).device
        self.global_batch = None
        capturable = all(g.get("capturable", False) for g in optimizer.param_groups)
        self.cuda_graphs = capturable if cuda_graphs is None else bool(cuda_graphs)
        if self.cuda_graphs and not capturable:
            raise ValueError("cuda_graphs=True needs an optimizer built with capturable=True")
        self._graphs, self._max_graphs = {}, max_graphs     # captured train steps by batch signature
        self.overlap = bool(self.cuda_graphs if overlap is None else overlap) and self.device.type == "cuda"
        self._tstream = None
        self._inflight = []      # completion events of the train steps queued so far (bounded lead, see _throttle)

    def _captured(self, cache, sig, capture):
        """the CUDA graph to replay for a batch of signature `sig`, or None when the batch runs eagerly.  The first
        occurrence of a signature runs eagerly and is remembered as "seen" (while `cache` holds fewer than max_graphs
        signatures), the second is captured by ``capture()``, later ones replay that graph."""
        ent = cache.get(sig)
        if ent is None:
            if len(cache) < self._max_graphs:
                cache[sig] = "seen"
        elif isinstance(ent, str):
            ent = cache[sig] = capture()
        return ent

    def replayed_library_kernels(self):
        """libdn4gl kernels launched through CUDA-graph replays so far (they bypass the library's launch counter)."""
        return sum(e.replays * e.library_kernels for name in self._caches for e in getattr(self, name).values()
                   if isinstance(e, _CapturedGraph))

    def _transform_stream(self):
        if self._tstream is None:
            # high priority: the host blocks on the transform's two size read-backs, so its small kernels should be
            # scheduled ahead of the queued CTAs of the train step that runs concurrently on the main stream
            self._tstream = torch.cuda.Stream(self.device, priority=-1)
        return self._tstream

    def _throttle(self):
        """bounds the host's lead over the train stream to ONE step: before the transform of step k+1 starts, the train
        step k-1 must have finished (step k may still be running -- that is the overlap).  Without the bound the host
        (whose transform only synchronises with its own stream) runs several steps ahead whenever the train stream is
        the slower side; every step in flight pins a full set of transform outputs, the caching allocator answers with
        cudaMalloc, and single steps stall for 5-50 ms (profiles/r1f)."""
        while len(self._inflight) >= 2:
            self._inflight.pop(0).synchronize()

    def _mark_step(self):
        ev = torch.cuda.Event()
        ev.record()
        self._inflight.append(ev)

    def _hand_over(self, tensors, tstream):
        """transform outputs (`tensors`, allocated and produced on `tstream`) -> consumable on the current (train) stream."""
        main = torch.cuda.current_stream()
        done = torch.cuda.Event()
        done.record(tstream)
        main.wait_event(done)
        for t in tensors:       # the caching allocator must not recycle them before the train stream is done
            t.record_stream(main)

    @contextlib.contextmanager
    def _global_batch(self, n):
        """``global_batch`` = n (when given) for the steps queued inside the block."""
        prev = self.global_batch
        if n is not None:
            self.global_batch = int(n)
        try:
            yield
        finally:
            self.global_batch = prev

    def _step_overlapped(self, transform, train, assume_ready):
        """``train(transform())`` with the transform on the second stream (see ClassificationPipeline.step_resident);
        ``_transform_outputs`` names the tensors of its result that the train stream takes over."""
        ts = self._transform_stream()
        self._throttle()
        if not assume_ready:
            ts.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(ts):
            out = transform()
            tensors = self._transform_outputs(out)
        self._hand_over(tensors, ts)
        loss = train(out)
        self._mark_step()
        return loss

    def _evaluate(self, ds, idx, batch_size, words, assemble, score, columns, finish):
        """the shared body of ``evaluate``: validates, then for each batch of the fixed order ``score(assemble(sel),
        pos0)`` with the model in eval mode under no_grad (assembly on the second stream with ``overlap``).  ``words``:
        int32 words of the zero-filled record buffer that ``columns(buf)`` cuts into (float32 sum columns, predictions);
        -> EvalResult."""
        import torch.distributed as dist

        from .datasets import EpochSampler, _check_indices
        from .graph import error_flag
        idx = np.arange(len(ds), dtype=np.int64) if idx is None else _check_indices(idx, len(ds), "evaluate")
        if idx.size == 0:
            raise ValueError("evaluate: no samples to evaluate")
        world, rank = (dist.get_world_size(), dist.get_rank()) if is_distributed() else (1, 0)
        # the evaluation order is idx itself; each rank takes its contiguous slice of every batch, as in training
        order = EpochSampler(idx.size, batch_size, shuffle=False, rank=rank, world_size=world)
        n = int(idx.size)
        buf = torch.zeros(words(n), dtype=torch.int32, device=self.device)
        sum_cols, predictions = columns(buf, n)
        modes = [(m, m.training) for m in self.model.modules()]
        self.model.eval()
        try:
            with torch.no_grad():
                for pos, _ in order.batches():
                    if len(pos) == 0:           # a short last batch leaves this rank nothing
                        self._eval_skip()
                        continue
                    sel, pos0 = idx[pos], int(pos[0])
                    if not self.overlap:
                        score(assemble(sel), pos0)
                    else:
                        self._step_overlapped(lambda: assemble(sel), lambda out: score(out, pos0), assume_ready=True)
        finally:
            for m, training in modes:
                m.training = training
        if world > 1:
            # every rank wrote its own positions only; as int32 words the sum adds exact zeros to every bit pattern
            # (NaN included), so all ranks hold the same records, bit for bit
            dist.all_reduce(buf)
        k = [1 if c.dim() == 1 else c.size(1) for c in sum_cols]
        sums = torch.empty(sum(k) + 1, dtype=torch.float64, device=self.device)
        for col, o in zip(sum_cols, np.cumsum([0] + k[:-1])):
            ops.eval_reduce(col, sums[int(o):int(o) + col.numel() // n])
        sums[-1:].copy_(error_flag(self.device))
        return EvalResult(sums, n, finish, predictions)

    def _eval_skip(self):
        """a batch of the evaluation order that holds nothing for this rank (collectives the others issue go here)."""


class ClassificationPipeline(_Pipeline):
    _caches = ("_graphs", "_tgraphs")

    def __init__(self, model, optimizer, mode="conj", num_node_labels=None, num_edge_labels=None,
                 node_label_min=None, with_edge_attr=False, cuda_graphs=None, max_graphs=8, overlap=None):
        """mode: 'dummy' (DUMMY_ graphs), 'conj' (CONJ_: dummy + edge-to-vertex), 'line' (LINE_), 'raw'.

        overlap: run the graph transforms on a second CUDA stream so that the transform of mini-batch k+1 (host-bound:
        ~60 small launches and two size read-backs) overlaps the train step of mini-batch k on the main stream -- the
        data-loader prefetch of the reference's DataLoader workers, done on the device.  Default: on when the train
        step is replayed as a CUDA graph (the host is free as soon as the replay is queued).

        cuda_graphs: replay the train step (forward + loss + backward + all-reduce + optimizer) as a CUDA graph when a
        batch has the same signature (tensor shapes + tiling scalars) as an earlier one: the first occurrence of a
        signature runs eagerly, the second is captured, later ones are replayed (a ~300-launch step is host-bound
        otherwise, profiles/).  Needs an optimizer whose step is capturable (``torch.optim.Adam(capturable=True)``);
        default: on exactly when the optimizer is."""
        super().__init__(model, optimizer, cuda_graphs, max_graphs, overlap)
        self.mode = mode
        self.nvl, self.nel = num_node_labels, num_edge_labels
        self.node_label_min, self.with_edge_attr = node_label_min, with_edge_attr
        self._tgraphs = {}       # captured transforms by raw-batch signature
        self._consumed = None    # event: the latest train step no longer reads its batch's own tensors

    def transform(self, batch):
        """raw TU-shaped batch (device tensors, or pinned host tensors of an int32 / float32 / int64-y batch) -> PyG-style
        Batch with compiled structure.  A batch that carries the loader's ``conj_sizes`` hint and whose signature has been
        seen before is transformed by replaying a captured CUDA graph (see _CapturedTransform); everything else runs the
        kernels eagerly."""
        on_host = any(isinstance(v, torch.Tensor) and not v.is_cuda for v in batch.values())
        capturable = (self.cuda_graphs and self.mode == "conj" and batch.get("conj_sizes") is not None and
                      not self.with_edge_attr and not torch.cuda.is_current_stream_capturing())
        if capturable:
            norm = {k: (v.to(torch.int32) if isinstance(v, torch.Tensor) and v.dtype == torch.int64 and k != "y" else v)
                    for k, v in batch.items()} if on_host else batch
            ent = self._captured(self._tgraphs, _raw_signature(norm),
                                 lambda: _CapturedTransform(self, self._upload(batch) if on_host else batch))
            if ent is not None:
                # the outputs are static tensors: the consumer of the previous replay must be done with them -- a replayed
                # train step right after its copy into its own buffers, an eager one at its end (train_on sets the event)
                return ent.run(norm, wait=self._consumed)
        return self._transform_eager(self._upload(batch) if on_host else batch)

    def _transform_eager(self, dev_batch):
        b = dev_batch
        hint = b.get("conj_sizes")
        if (self.mode == "conj" and not self.with_edge_attr and hint is not None and len(hint) >= 5 and hint[3]
                and self.nvl is not None and self.node_label_min is not None and "vattr" not in b):
            # CONJ_ structure in closed form from the raw graphs' CSRs (transforms.tu_conj_structure): the loader's extended
            # hint (tu_conjugate_sizes_ex) says every graph has a node, and the model reads x, y and the structure only
            data = T.tu_conj_structure(b, self.nvl, self.node_label_min)
            s = data.structure
            hid = getattr(self.model, "hidden_dim", None)
            if hid in ops._TILED_D:
                s.csr_in.tiles(hid)
                s.csr_out.tiles(hid)
            s.row2seg
            return data
        if self.mode in ("dummy", "conj"):
            b = T.tu_add_dummy(b)
        if self.mode in ("conj", "line"):
            b = T.tu_conjugate(b)
            b.pop("eattr", None)
        b["has_edge_labels"] = True
        # GIN never reads edge_attr (gconv.py:204); RGIN does (rgconv.py:109-111)
        can = T.pyg_canonicalize(b, self.nvl, self.nel, node_label_min=self.node_label_min,
                                 with_edge_attr=self.with_edge_attr, defer_count=not self.with_edge_attr)
        data = Batch.from_canonical(can)
        s = data.structure  # compile the CSR pair now (part of the transform cost)
        hid = getattr(self.model, "hidden_dim", None)
        if hid in ops._TILED_D and s.node_ptr is not None:   # ... and the aggregation tiling for the model's width
            s.csr_in.tiles(hid)
            s.csr_out.tiles(hid)
        s.row2seg
        return data

    def _train_body(self, data):
        self.bucket.zero()
        out = self.model(data)
        loss = ops.nll_loss(out, data.y) if out.is_cuda else F.nll_loss(out, data.y)    # main.py:41
        loss.backward()
        self.bucket.gather()                                # gradients live in one flat buffer (one multi-tensor copy)
        if is_distributed():
            gb = self.global_batch or data.num_graphs * torch.distributed.get_world_size()
            self.bucket.all_reduce(data.num_graphs / gb)
        self.opt.step()                                     # main.py:43
        # detached: a caller holding the loss must not keep this step's autograd graph (and its AccumulateGrad nodes,
        # bound to the stream they were created on) alive into the next step / a CUDA-graph capture
        return loss.detach()

    def train_on(self, data):
        if not self.model.training:      # Module.train() walks every submodule (~0.2 ms of host time per step)
            self.model.train()
        if not self.cuda_graphs:
            return self._train_body(data)
        tensors, scalars = _structure_tensors(data)
        ent = self._captured(self._graphs, _signature(tensors, scalars),
                             lambda: _CapturedStep(self._train_body, (_static_clone(data),), _structure_tensors))
        if ent is None:
            loss = self._train_body(data)
        else:
            ent.load(tensors)
        # from here on the batch's own tensors may be overwritten (captured transform): after an eager step's end, right
        # after a replay's copy into the graph's buffers
        self._consumed = torch.cuda.Event()
        self._consumed.record()
        return loss if ent is None else ent.replay()

    def _transform_outputs(self, data):
        """every device tensor a compiled Batch holds (what the train step may read from it)."""
        s = data.structure
        out = [t for t in _structure_tensors(data)[0] if t is not None]
        out += [t for t in (s.src, s.dst, s.csr_in.eid, s.csr_out.eid) if t is not None]
        return out

    def step_resident(self, dev_batch, assume_ready=False):
        """inputs already in HBM: transform + train step; returns the loss tensor (no host sync).

        With ``overlap`` the transform runs on the pipeline's second stream.  ``assume_ready=True``: the caller
        guarantees that ``dev_batch`` is complete (written before any still-running work was queued), so the transform
        does not wait for the train stream and overlaps the previous step; otherwise it is ordered behind everything
        queued on the current stream so far (always safe, no GPU-side overlap)."""
        if not self.overlap:
            return self.train_on(self.transform(dev_batch))
        return self._step_overlapped(lambda: self.transform(dev_batch), self.train_on, assume_ready)

    def _upload(self, host_batch):
        dev = upload(host_batch, self.device)
        return {k: (v.to(torch.int32) if isinstance(v, torch.Tensor) and v.dtype == torch.int64 and k != "y" else v)
                for k, v in dev.items()}

    def step_async(self, host_batch):
        """host buffers in, ``PendingLoss`` out: H2D + transform (second stream when ``overlap``) + train step + queued D2H
        of the loss.  The host returns as soon as everything is queued; ``PendingLoss.result()`` yields the float.  A
        loop that reads the previous step's result after submitting the next one keeps both streams busy."""
        if not self.overlap:
            return PendingLoss(self.step_resident(self._upload(host_batch)))
        # the upload is ordered on the transform stream: no wait on the train stream
        return PendingLoss(self._step_overlapped(lambda: self.transform(host_batch), self.train_on, assume_ready=True))

    def step(self, host_batch):
        """host buffers in, python float out: H2D + transform + train step + D2H of the loss (blocking)."""
        return self.step_async(host_batch).result()

    def step_indices(self, ds, idx, global_batch=None):
        """one train step on graphs `idx` (host integer array) of a ``datasets.ResidentTUDataset``, assembled on the device
        by ``ds.batch(idx)``; returns a ``PendingLoss`` as ``step_async`` does.  With ``overlap`` the staging copy and the
        gathers run inside the transform on the second stream, next to the previous train step (the resident columns
        never change, so nothing waits for the train stream).  In 'conj' mode the batch carries its size hint: with
        ``num_node_labels`` and ``node_label_min`` given and every graph holding a node, the closed-form CONJ_ builder runs
        and the step reads nothing back from the device.  global_batch: graphs of the whole data-parallel step (as
        ``EpochSampler`` yields it); default: this batch times the world size."""
        def assemble():
            b = ds.batch(idx)
            if self.mode != "conj":
                b.pop("conj_sizes")     # the hint describes the dummy-augmented edge-to-vertex transform only
            return self.transform(b)

        with self._global_batch(global_batch):
            if not self.overlap:
                return PendingLoss(self.train_on(assemble()))
            return PendingLoss(self._step_overlapped(assemble, self.train_on, assume_ready=True))

    def evaluate(self, ds, idx=None, batch_size=512, log_probs=False):
        """accuracy and mean NLL of the model over graphs `idx` (host integer array; default: every graph, in order) of a
        ``datasets.ResidentTUDataset`` -- the reference's ``eval_test`` (main.py:54, 90-104), whose numbers drive early
        stopping and the choice of ``best.pt``.  Returns an ``EvalResult`` as soon as the work is queued:
        ``metrics()`` -> ``{"accuracy", "loss"}`` (correct / n and the summed ``F.nll_loss`` / n); ``predictions`` ->
        ``pred`` (int32 arg-max, ``out.max(1)[1]``), ``nll`` (per graph) and, with ``log_probs``, the (n, C)
        log-probabilities, all in the order of `idx`.

        Batches of ``batch_size`` graphs in the order of `idx` are assembled by ``ds.batch``, transformed, and scored by
        the model's own eval-mode forward under ``torch.no_grad()``; one kernel writes each batch's records at its offset
        and one fixed-order reduction per column gives the sums, so the metrics do not depend on the batching.  The
        model's train / eval modes are restored afterwards; no parameter, BatchNorm buffer or optimizer state changes.
        Under torch.distributed each rank scores its contiguous slice of every batch and the records are all-reduced:
        every rank returns the same bits.  Kept from the reference: GIN's layer-0 dropout is applied without
        ``training=`` (gconv.py:210), so with ``dropout_ratio > 0`` the scores are random, as there."""
        C = getattr(self.model, "num_classes", None)
        if log_probs and not C:
            raise ValueError("evaluate(log_probs=True) needs a model with num_classes")
        rec = {}

        def columns(buf, n):
            rec["pred"] = buf[:n]
            rec["nll"], rec["correct"] = buf[n:2 * n].view(torch.float32), buf[2 * n:3 * n].view(torch.float32)
            preds = dict(pred=rec["pred"], nll=rec["nll"])
            if log_probs:
                preds["log_probs"] = rec["log_probs"] = buf[3 * n:].view(torch.float32).view(n, C)
            return [rec["correct"], rec["nll"]], preds

        def assemble(sel):
            b = ds.batch(sel)
            if self.mode != "conj":
                b.pop("conj_sizes")
            # the eager transform, also where train steps replay a captured one: a captured transform writes static
            # buffers that the next train step reads (the _consumed protocol), and evaluation batches would take
            # signatures in the train-time cache; the eager transform shares nothing with training
            return self._transform_eager(b)

        def score(data, pos0):
            out = self.model(data)
            ops.eval_class_rows(out, data.y.long(), pos0, rec["pred"], rec["nll"], rec["correct"])
            if log_probs:
                rec["log_probs"][pos0:pos0 + out.size(0)].copy_(out)

        def finish(s, n):
            return {"accuracy": s[0] / n, "loss": s[1] / n}

        return self._evaluate(ds, idx, batch_size, lambda n: (3 + (C if log_probs else 0)) * n, assemble, score,
                              columns, finish)


def _graph_tensors(g):
    """device tensors a counting-model step reads from a BatchedGraph (fixed order) + the host scalars baked into kernel
    arguments and tensor shapes (padded lengths come from the per-graph maxima)."""
    tensors = [g.src, g.dst, g.node_ptr, g.edge_ptr]
    scalars = [g.batch_size, g.number_of_nodes(), g.number_of_edges(), g.max_num_nodes(), g.max_num_edges(),
               g.padded_num_nodes(), g.padded_num_edges()]
    for frame in (g.ndata, g.edata):
        for k in sorted(frame):
            tensors.append(frame[k])
            scalars.append(k)
    for csr in (g._csr_in, g._csr_out):
        if csr is None:
            tensors += [None] * 5
            scalars.append(None)
        else:
            tensors += [csr.row_ptr, csr.col, csr.eid, csr.heavy_rows, csr.heavy_count]
            scalars += [csr.n_rows, csr.nnz, csr.heavy_thr, csr.max_seg]
    return tensors, scalars


def _counting_tensors(pattern, graph, counts, node_weights=None, edge_weights=None):
    """every device tensor a counting train step reads (fixed order) + the host scalars of its CUDA-graph signature.  The
    match weights are among the tensors (None when absent), so a matched step has a signature of its own."""
    tp, sp = _graph_tensors(pattern)
    tg, sg = _graph_tensors(graph)
    return tp + tg + [counts, node_weights, edge_weights], [tuple(sp), tuple(sg)]


def _static_graph(g):
    """private copy of a BatchedGraph (the buffers a captured CUDA graph reads); caches that the model fills during its
    forward (relation CSRs, int32 views, tilings) start empty so that the captured forward recomputes them.  Tilings
    copied from this batch would not be among the tensors a replay copies in (_graph_tensors), so later replays would
    run on this batch's tiles."""
    c = BatchedGraph(g.src.clone(), g.dst.clone(), g.node_ptr.clone(), g.edge_ptr.clone(),
                     {k: v.clone() for k, v in g.ndata.items()}, {k: v.clone() for k, v in g.edata.items()})
    c._n, c._host_sizes, c._pad_lengths = g._n, g._host_sizes, g._pad_lengths
    for name in ("_csr_in", "_csr_out"):
        c0 = getattr(g, name)
        if c0 is not None:
            setattr(c, name, c0.clone(c.node_ptr, eid=True, tiles=False))
    return c


def _match_kinds(match_weights):
    """the reference's --match_weights flag (None, "node", "edge", "node,edge") -> (node, edge) booleans."""
    if match_weights is None:
        return None
    kinds = [k.strip() for k in str(match_weights).split(",")]
    if not kinds or any(k not in ("node", "edge") for k in kinds) or len(set(kinds)) != len(kinds):
        raise ValueError("match_weights: None, 'node', 'edge' or 'node,edge', got %r" % (match_weights,))
    return "node" in kinds, "edge" in kinds


def _check_identity_refine(model):
    """the fused match loss reads the weights as they are: refuse a model that refines them."""
    from .subgraph_isomorphism.models.basemodel import _CountingBase
    for name in ("refine_node_weights", "refine_edge_weights"):
        if getattr(type(model), name, None) is not getattr(_CountingBase, name):
            raise ValueError("match weights: %s overrides %s; the fused match loss reads the weights unrefined"
                             % (type(model).__name__, name))


class CountingPipeline(_Pipeline):
    def __init__(self, model, optimizer, config, add_dummy=True, rep_reg_w=0.0, neg_slp=0.01, max_grad_norm=8.0,
                 cuda_graphs=None, max_graphs=8, overlap=None, exact_sharding=False, bp_loss="MSE", match_loss_w=0.0,
                 match_reg_w=0.0, remove_loops=False, add_rev=False, convert_conj=False, share_emb_net=True,
                 match_weights=None):
        """config: the dataset maxima BEFORE augmentation (max_npv ... max_ngel).  cuda_graphs / overlap: as in
        ClassificationPipeline (defaults: graphs on exactly when the optimizer was built with capturable=True, the
        augmentation + CSR builds on a second stream exactly when graphs are on).  exact_sharding: under
        torch.distributed, all-reduce(max) the four padded lengths of every mini-batch (one 4-int collective and one
        host read per step) so that a sharded batch gives exactly the single-process head / filter numbers
        (SURVEY.md 8(e) i, v); off by default -- each rank then pads to its own shard's maxima.  bp_loss / match_loss_w /
        match_reg_w: criterion and weights of the match terms (train.py:620-627, 776-813); they only enter steps that
        are given per-node / per-edge match weights (``train_on(..., node_weights=, edge_weights=)``, or ``step_indices``
        with ``match_weights``).  Such steps compute the match terms with one kernel each way (``ops.match_loss``) and
        are captured and replayed like the others: the weights are among the tensors a replay copies in, and
        match_loss_w / match_reg_w live in device scalars like neg_slp.  match_weights: the reference's --match_weights
        (None, "node", "edge", "node,edge"): ``step_indices`` then also gathers the samples' subisomorphisms, appends the
        dummy column (with add_dummy) and trains on the match-weight targets of the augmented batch
        (``matching.node_weights`` / ``edge_weights``).  Refused with convert_conj, and for a model that overrides
        ``refine_node_weights`` / ``refine_edge_weights``.  remove_loops / add_rev / convert_conj: the reference's other
        data-set level preprocessing switches, applied per mini-batch on the GPU in the reference's order
        (train.py:1271-1340: loops, reversed edges, dummy, edge-to-vertex), each with the maxima the previous steps
        leave behind; build the model with ``transforms.process_model_config`` of the same switches."""
        self.match_weights = _match_kinds(match_weights)
        if self.match_weights is not None:
            if convert_conj:
                raise ValueError("match_weights with convert_conj: the conjugate graph's node-weight numbering is not "
                                 "pinned against the reference")
            _check_identity_refine(model)
        super().__init__(model, optimizer, cuda_graphs, max_graphs, overlap)
        self.cfg, self.add_dummy = config, add_dummy
        # neg_slp and rep_reg_w change every step in the reference (train.py:648-740 recomputes them from their
        # schedules): they live in device scalars that the (possibly captured) train step READS, so an update through the
        # properties below is seen by the next step / CUDA-graph replay
        # (match_reg_w too: anneal_cosine$0.01$0.0 by default, losses.py:30)
        self._neg_slp_t = torch.zeros((), dtype=torch.float32, device=self.device)
        self._rep_reg_w_t = torch.zeros((), dtype=torch.float32, device=self.device)
        self._match_loss_w_t = torch.zeros((), dtype=torch.float32, device=self.device)
        self._match_reg_w_t = torch.zeros((), dtype=torch.float32, device=self.device)
        self._neg_slp = self._rep_reg_w = self._match_loss_w = self._match_reg_w = None
        self.neg_slp, self.rep_reg_w, self.max_grad_norm = neg_slp, rep_reg_w, max_grad_norm
        self.share_emb_net = bool(share_emb_net)
        self.exact_sharding = bool(exact_sharding)
        self.bp_loss, self.match_loss_w, self.match_reg_w = bp_loss, match_loss_w, match_reg_w
        self.remove_loops, self.add_rev, self.convert_conj = bool(remove_loops), bool(add_rev), bool(convert_conj)

    @property
    def neg_slp(self):
        return self._neg_slp

    @neg_slp.setter
    def neg_slp(self, v):
        if v != self._neg_slp:
            self._neg_slp = float(v)
            self._neg_slp_t.fill_(self._neg_slp)

    @property
    def rep_reg_w(self):
        return self._rep_reg_w

    @rep_reg_w.setter
    def rep_reg_w(self, v):
        if v != self._rep_reg_w:
            self._rep_reg_w = float(v)
            self._rep_reg_w_t.fill_(self._rep_reg_w)

    @property
    def match_loss_w(self):
        return self._match_loss_w

    @match_loss_w.setter
    def match_loss_w(self, v):
        if v != self._match_loss_w:
            self._match_loss_w = float(v)
            self._match_loss_w_t.fill_(self._match_loss_w)

    @property
    def match_reg_w(self):
        return self._match_reg_w

    @match_reg_w.setter
    def match_reg_w(self, v):
        if v != self._match_reg_w:
            self._match_reg_w = float(v)
            self._match_reg_w_t.fill_(self._match_reg_w)

    def augment(self, p_dev, g_dev):
        """flat device batches -> flat device batches after the configured preprocessing switches (no CSR yet)."""
        c = self.cfg
        npv, npvl, npe, npel = c["max_npv"], c["max_npvl"], c["max_npe"], c["max_npel"]
        ngv, ngvl, nge, ngel = c["max_ngv"], c["max_ngvl"], c["max_nge"], c["max_ngel"]
        if self.share_emb_net:      # train.py:1276-1289: pattern and graph share the embedding tables, so the pattern side is
            npv, npvl, npe, npel = ngv, ngvl, nge, ngel      # augmented with the GRAPH maxima (same dummy / reversed ids and labels)
        if self.remove_loops:                                   # train.py:1271-1274
            p_dev, g_dev = T.sub_remove_loops(p_dev), T.sub_remove_loops(g_dev)
        if self.add_rev:                                        # train.py:1310-1319: maxima double afterwards
            p_dev, g_dev = T.sub_add_reversed(p_dev, npe, npel), T.sub_add_reversed(g_dev, nge, ngel)
            npe, npel, nge, ngel = 2 * npe, 2 * npel, 2 * nge, 2 * ngel
        if self.add_dummy:                                      # train.py:1322-1334
            p_dev = T.sub_add_dummy(p_dev, npv, npvl, npe, npel)
            g_dev = T.sub_add_dummy(g_dev, ngv, ngvl, nge, ngel)
        if self.convert_conj:                                   # train.py:1337-1340 -> convert_to_conjugate :564-593
            p_dev, g_dev = T.sub_conjugate(p_dev), T.sub_conjugate(g_dev)
        return p_dev, g_dev

    def transform(self, p_dev, g_dev):
        return self._compile(*self.augment(p_dev, g_dev))

    def _compile(self, p_dev, g_dev):
        """augmented flat batches -> BatchedGraph pair with both CSRs (and the shared padded lengths)."""
        pattern, graph = BatchedGraph.from_batch(p_dev, self.device), BatchedGraph.from_batch(g_dev, self.device)
        for g in (pattern, graph):   # compile both CSRs + degrees now (calculate_degrees, train.py:1355-1356)
            g.in_degrees()
            g.out_degrees()
        if self.exact_sharding and is_distributed():
            gv, ge, pv, pe = sync_padded_lengths(graph.max_num_nodes(), graph.max_num_edges(),
                                                 pattern.max_num_nodes(), pattern.max_num_edges())
            graph.set_padded_lengths(gv, ge)
            pattern.set_padded_lengths(pv, pe)
        return pattern, graph

    def loss_fn(self, out, counts):
        """train.py:620-627 + :801-811 with the configured criterion; the negative slope and the regulariser weight are
        read from device scalars (leaky_relu(x, s) = where(x > 0, x, x * s): same values as F.leaky_relu)."""
        from .subgraph_isomorphism.losses import _CRITERIA
        if self.bp_loss not in _CRITERIA:
            raise NotImplementedError(self.bp_loss)
        fn = _CRITERIA[self.bp_loss]
        pred = out["pred_c"]
        loss = fn(torch.where(pred > 0, pred, pred * self._neg_slp_t), counts.float().view(-1, 1))
        if self._rep_reg_w != 0.0 or self.cuda_graphs:      # a captured step keeps the term: the weight may change later
            for k in ("p_v_rep", "p_e_rep", "g_v_rep", "g_e_rep"):                      # train.py:801-811 (slope 1: identity)
                if out[k] is not None:
                    loss = loss + self._rep_reg_w_t * fn(out[k], torch.zeros_like(out[k])) * out[k].size(1)
        return loss

    def match_loss_fn(self, out, counts, graph, node_weights, edge_weights):
        """the reference's full bp_loss (losses.counting_bp_loss) with flat per-node / per-edge match weights of the
        augmented graph batch (matching.node_weights / edge_weights), left-padded here like the model's outputs.  The
        tensor restatement of what a matched train step computes with ``fused_loss_fn``; it zeroes out["pred_v"] /
        out["pred_e"] on masked positions in place, as the reference does."""
        from .subgraph_isomorphism.losses import counting_bp_loss, pad_match_weights
        nw = None if node_weights is None else pad_match_weights(node_weights, graph.node_ptr, graph.padded_num_nodes())
        ew = None if edge_weights is None else pad_match_weights(edge_weights, graph.edge_ptr, graph.padded_num_edges())
        return counting_bp_loss(out, counts, nw, ew, model=self.model, bp_loss=self.bp_loss, neg_slp=self.neg_slp,
                                rep_reg_w=self.rep_reg_w, match_loss_w=self.match_loss_w, match_reg_w=self.match_reg_w)[0]

    def fused_loss_fn(self, out, counts, graph, node_weights, edge_weights):
        """``match_loss_fn``'s value with the match terms from ``ops.match_loss`` (one kernel each way, flat weights read
        in place, every weight and the slope from device scalars); the model's outputs are left unchanged.  A kind
        whose weights or prediction is None contributes nothing (losses.py:95-96)."""
        loss = self.loss_fn(out, counts)
        pv = out.get("pred_v") if node_weights is not None else None
        pe = out.get("pred_e") if edge_weights is not None else None
        if pv is None and pe is None:
            return loss
        return loss + ops.match_loss(out["pred_c"], pv, out.get("g_v_mask"), node_weights, graph.node_ptr, pe,
                                     out.get("g_e_mask"), edge_weights, graph.edge_ptr, self.bp_loss, self._neg_slp_t,
                                     self._match_loss_w_t, self._match_reg_w_t)

    def _train_body(self, pattern, graph, counts, node_weights=None, edge_weights=None):
        self.bucket.zero()
        out = self.model(pattern, graph)
        if node_weights is None and edge_weights is None:
            loss = self.loss_fn(out, counts)
        else:
            loss = self.fused_loss_fn(out, counts, graph, node_weights, edge_weights)
        loss.backward()
        self.bucket.gather()
        if is_distributed():
            gb = self.global_batch or pattern.batch_size * torch.distributed.get_world_size()
            self.bucket.all_reduce(pattern.batch_size / gb)
        if self.max_grad_norm and self.max_grad_norm > 0:   # clip AFTER the reduction (train.py:833-834)
            flat = self.bucket.flat      # clip_grad_norm_ on the flat buffer: norm, coefficient, scale = 4 launches
            coef = (self.max_grad_norm / (torch.linalg.vector_norm(flat) + 1e-6)).clamp(max=1.0)
            flat.mul_(coef)
        self.opt.step()
        return loss.detach()   # see ClassificationPipeline._train_body

    def train_on(self, pattern, graph, counts, node_weights=None, edge_weights=None):
        if not self.model.training:      # Module.train() walks every submodule (~0.2 ms of host time per step)
            self.model.train()
        if node_weights is not None or edge_weights is not None:
            _check_identity_refine(self.model)
        if not self.cuda_graphs:
            return self._train_body(pattern, graph, counts, node_weights, edge_weights)
        tensors, scalars = _counting_tensors(pattern, graph, counts, node_weights, edge_weights)
        ent = self._captured(self._graphs, _signature(tensors, scalars), lambda: _CapturedStep(
            self._train_body, (_static_graph(pattern), _static_graph(graph), counts.clone(),
                               *(None if w is None else w.clone() for w in (node_weights, edge_weights))),
            _counting_tensors))
        if ent is None:
            return self._train_body(pattern, graph, counts, node_weights, edge_weights)
        ent.load(tensors)
        return ent.replay()

    def _transform_outputs(self, out):
        """every device tensor of both graphs (out[:2]) and the match weights that may follow them; everything the
        captured step copies out of the batch exists before the hand-over (the CSRs are built here, on the transform's
        stream, if the transform left one out)."""
        graphs = out[:2]
        for g in graphs:
            g.csr_in, g.csr_out
        return [t for g in graphs for t in _graph_tensors(g)[0] if t is not None] + [t for t in out[2:] if t is not None]

    def step_resident(self, p_dev, g_dev, counts_dev, assume_ready=False):
        """see ClassificationPipeline.step_resident: with ``overlap`` the augmentation + CSR builds of this mini-batch run
        on the second stream while the previous train step is still executing."""
        if not self.overlap:
            return self.train_on(*self.transform(p_dev, g_dev), counts_dev)
        return self._step_overlapped(lambda: self.transform(p_dev, g_dev),
                                     lambda graphs: self.train_on(*graphs, counts_dev), assume_ready)

    def step(self, p_host, g_host, counts_host):
        p_dev, g_dev = upload(p_host, self.device), upload(g_host, self.device)
        counts = counts_host.to(self.device, non_blocking=True)
        return PendingLoss(self.step_resident(p_dev, g_dev, counts)).result()    # also raises on a builder-kernel error

    def step_indices(self, ds, idx, global_batch=None):
        """one train step on samples `idx` (host integer array) of a ``datasets.ResidentCountingDataset``, assembled on the
        device by ``ds.batch(idx)``; returns a ``PendingLoss``.  With ``overlap`` the staging copy and the gathers run with
        the augmentation on the second stream, next to the previous train step.  The augmentation's own device->host
        reads (``BatchedGraph.from_batch``) stay.  global_batch: as in ClassificationPipeline.step_indices.

        With ``match_weights`` the batch also carries its samples' subisomorphisms (with the dummy column when
        ``add_dummy``), and the match-weight targets are computed on the augmented batch in the same place: node weights
        add no device->host read, edge weights the one of ``matching.edge_weights``."""
        counts = []

        def assemble():
            if self.match_weights is None:
                p_dev, g_dev, c = ds.batch(idx)
                counts.append(c)
                return self.transform(p_dev, g_dev)
            from .subgraph_isomorphism import matching as M
            p_dev, g_dev, c, sub = ds.batch(idx, subisomorphisms=True, dummy_column=self.add_dummy)
            counts.append(c)
            p_aug, g_aug = self.augment(p_dev, g_dev)
            node, edge = self.match_weights
            nw = M.node_weights_i32(sub, g_aug) if node else None
            ew = M.edge_weights_i32(sub, p_aug, g_aug) if edge else None
            return self._compile(p_aug, g_aug) + (nw, ew)

        def train(out):
            if self.overlap:        # allocated on the transform stream, read by the train stream
                counts[0].record_stream(torch.cuda.current_stream())
            return self.train_on(out[0], out[1], counts[0], *out[2:])

        with self._global_batch(global_batch):
            if not self.overlap:
                return PendingLoss(train(assemble()))
            return PendingLoss(self._step_overlapped(assemble, train, assume_ready=True))

    def evaluate(self, ds, idx=None, batch_size=512):
        """the reference's ``evaluate`` (train.py:609-618 criteria) over samples `idx` (host integer array; default: every
        sample, in order) of a ``datasets.ResidentCountingDataset``; returns an ``EvalResult`` as soon as the work is
        queued: ``metrics()`` -> ``{"MAE", "MSE", "SMSE", "RMSE"}`` (``losses.eval_criterion`` over the whole split:
        relu(pred_c) against the counts; RMSE = sqrt(MSE)); ``predictions`` -> ``pred_c`` in the order of `idx`.

        Batching, records, reduction, modes and distributed behaviour as in ``ClassificationPipeline.evaluate``; the
        augmentation's own device->host reads (``BatchedGraph.from_batch``) stay.  Kept from the reference: the
        prediction head's L * bias term depends on the batch's padded length (SURVEY.md App. A-7), so a sample's
        prediction depends on which samples share its batch; under torch.distributed ``exact_sharding`` pads every
        rank's slice to the whole batch's lengths, as in training."""
        rec, counts = {}, []

        def columns(buf, n):
            rec["pred"] = buf[:n].view(torch.float32)
            rec["err"] = buf[n:].view(torch.float32).view(n, 3)
            return [rec["err"]], dict(pred_c=rec["pred"])

        def assemble(sel):
            p_dev, g_dev, c = ds.batch(sel)
            counts.append(c)
            return self.transform(p_dev, g_dev)

        def score(graphs, pos0):
            c = counts.pop()
            if self.overlap:        # allocated on the transform stream, read here
                c.record_stream(torch.cuda.current_stream())
            out = self.model(*graphs)
            ops.eval_count_rows(out["pred_c"], c, pos0, rec["pred"], rec["err"])

        def finish(s, n):
            return {"MAE": s[0] / n, "MSE": s[1] / n, "SMSE": s[2] / n, "RMSE": float(np.sqrt(s[1] / n))}

        return self._evaluate(ds, idx, batch_size, lambda n: 4 * n, assemble, score, columns, finish)

    def _eval_skip(self):
        if self.exact_sharding and is_distributed():    # the other ranks agree on this batch's padded lengths
            sync_padded_lengths(0, 0, 0, 0)
