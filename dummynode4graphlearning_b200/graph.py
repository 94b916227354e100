"""Batched (block-diagonal) graph container living in HBM.

Replaces, for the hot path, what the reference gets from ``dgl.batch`` /
``Graph(dgl.DGLGraph)`` (subgraph_isomorphism/dataset.py:1053-1373, 1604-1636) and from PyG's
``Batch`` (graph_classification/graph_neural_networks/main.py:245): frames are dicts of
tensors keyed by the reference's constants (``"id"``, ``"label"``, ``"is_dummy"``,
``"is_reversed"``, ``"in_deg"``, ``"out_deg"`` -- subgraph_isomorphism/constants.py:12-35), and
the structure is an immutable pair of int32 CSRs (by destination for the forward gather, by
source for the backward) built ONCE per mini-batch by the CUDA builder kernels.

Layout in HBM (DESIGN.md section 3): ``src``/``dst`` int32[E] in edge-id order, ``node_ptr``/
``edge_ptr`` int32[B+1], CSR ``row_ptr`` int32[N+1], ``col`` int32[E], ``eid`` int32[E]; features
fp32 row-major.
"""
import os

import torch

from ._lib import lib, ptr

HEAVY_THRESHOLD = 64  # rows with more in-edges than this are reduced by a whole CTA (dummy nodes)
TILE_SMEM = int(os.environ.get("DN4GL_TILE_SMEM", str(200 * 1024)))   # shared-memory ring of the pipelined aggregation kernel
TILE_WARPS = int(os.environ.get("DN4GL_TILE_WARPS", "32"))             # warps per CTA for D <= 128 (16 | 32)

_dev_bound = {}


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def _stream():
    """cudaStream_t of torch's current stream on the current device (raw handle: torch.cuda.current_stream() builds a
    Python Stream object per call, ~15 us -- a fifth of the transform's host time in profiles/r1e)."""
    if _raw_stream is not None:
        return _raw_stream(torch.cuda.current_device())
    return torch.cuda.current_stream().cuda_stream


def bind_device(device):
    """cudaSetDevice for the library's (statically linked) runtime on this host thread."""
    idx = device.index if device.index is not None else torch.cuda.current_device()
    if _dev_bound.get("idx") != idx:
        lib().call("dn4gl_set_device", idx)
        _dev_bound["idx"] = idx


def require_cuda(t, what="tensor"):
    if not t.is_cuda:
        raise RuntimeError("dummynode4graphlearning_b200: %s must live on a CUDA device -- the hot path has no "
                           "CPU fallback" % what)
    bind_device(t.device)


class CSR:
    """row_ptr[n_rows+1], col[nnz], eid[nnz] (all int32, device) + the heavy-row list."""

    __slots__ = ("row_ptr", "col", "eid", "n_rows", "nnz", "heavy_rows", "heavy_count", "heavy_thr", "seg_ptr",
                 "max_seg", "_tiles", "block_diagonal")

    def __init__(self, row_ptr, col, eid, n_rows, nnz):
        self.row_ptr, self.col, self.eid, self.n_rows, self.nnz = row_ptr, col, eid, n_rows, nnz
        self.heavy_rows = self.heavy_count = None
        self.heavy_thr = 0
        self.seg_ptr = None   # per-graph row offsets when rows AND columns are block-diagonal over the same graphs
        self.max_seg = None   # rows of the largest graph if the host knows it (lets every tile be graph-aligned)
        self.block_diagonal = False   # True: built graph by graph over seg_ptr (the tiling skips its column verification)
        self._tiles = {}

    def clone(self, seg_ptr, *, eid, tiles):
        """private copy of the device arrays over the row offsets `seg_ptr` (the buffers a captured CUDA graph reads);
        the edge ids and the cached tilings are copied only when asked for (else None / empty)."""
        c = CSR(self.row_ptr.clone(), self.col.clone(), self.eid.clone() if eid else None, self.n_rows, self.nnz)
        c.heavy_rows = None if self.heavy_rows is None else self.heavy_rows.clone()
        c.heavy_count = None if self.heavy_count is None else self.heavy_count.clone()
        c.heavy_thr, c.seg_ptr, c.max_seg, c.block_diagonal = self.heavy_thr, seg_ptr, self.max_seg, self.block_diagonal
        if tiles:
            c._tiles = {key: {k: (v.clone() if isinstance(v, torch.Tensor) else v) for k, v in t.items()}
                        for key, t in self._tiles.items()}
        return c

    def tiles(self, D, smem_bytes=None):
        """tiling + launch configuration of the pipelined aggregation kernel for feature width D (cached).

        One persistent CTA per SM owns `smem_bytes` of shared memory as a ring of `stages` buffers.  The window is
        chosen so that a tile (window + the graph straddling its end) always fits one stage: cap - max_seg when the
        host knows the largest graph, else cap / 2.  Graphs longer than the window are cut; rows with more than 64
        neighbours inside cut tiles go on the heavy list (reduced CTA-wide inside the same launch)."""
        smem_bytes = TILE_SMEM if smem_bytes is None else int(smem_bytes)
        key = (D, smem_bytes)
        if key in self._tiles:
            return self._tiles[key]
        L = lib()
        npr = min(max(-(-self.nnz // max(self.n_rows, 1)) + 1, 2), 32)
        stages = cap = None
        for s in (4, 3, 2):
            c = L.size("dn4gl_spmm_tiled_cap_rows", D, smem_bytes, s, npr)
            if self.max_seg is None:
                if s == 3:
                    stages, cap = s, c
                    break
            elif 2 * self.max_seg <= c:
                stages, cap = s, c
                break
        if stages is None:
            stages = 2
            cap = L.size("dn4gl_spmm_tiled_cap_rows", D, smem_bytes, stages, npr)
        aligned = self.max_seg is not None and 2 * self.max_seg <= cap
        window = max(cap - self.max_seg if aligned else cap // 2, 1)
        T = (self.n_rows + window - 1) // window
        dev = self.row_ptr.device
        desc = torch.empty(4 * max(T, 1), dtype=torch.int32, device=dev)
        heavy_list = heavy_count = None
        heavy_cap = 0
        warps = TILE_WARPS if D <= 128 else 16
        scratch = (warps - 1) * (32 // min(D // 4, 32)) * D * 4   # CTA-wide reduction scratch must fit one stage
        if not aligned and scratch <= ((smem_bytes // stages) & ~127):
            heavy_cap = self.nnz // 64 + 1
            heavy_list = torch.empty(heavy_cap, dtype=torch.int32, device=dev)
            heavy_count = torch.empty(1, dtype=torch.int32, device=dev)   # zeroed by dn4gl_make_row_tiles
        L.call("dn4gl_make_row_tiles", ptr(self.seg_ptr), int(self.seg_ptr.numel()) - 1, window, ptr(self.row_ptr),
               None if self.block_diagonal else ptr(self.col), self.n_rows, ptr(desc), T, ptr(heavy_list), heavy_cap, ptr(heavy_count), _stream())
        cfg = dict(desc=desc, T=T, heavy_list=heavy_list, heavy_count=heavy_count, heavy_cap=heavy_cap,
                   smem=smem_bytes, stages=stages, npr=npr, window=window, cap_rows=cap, warps=warps)
        self._tiles[key] = cfg
        return cfg


def build_csr(key, val, n_rows, heavy_threshold=HEAVY_THRESHOLD, sorted_keys=False, trash_row=False):
    """Stable CSR of the items 0..E-1 grouped by key (see dn4gl_build_csr).  sorted_keys: the caller guarantees
    non-decreasing keys (a coalesced edge list keyed by its row): one boundary-marking pass (dn4gl_build_csr_sorted);
    a violation is reported through check_errors().  trash_row: keys / values may also be n_rows (padding of a list
    whose true length only the device knows, transforms.pyg_canonicalize): the CSR is built over n_rows + 1 rows and handed
    out with n_rows logical rows -- kernels never visit the last row, `nnz` is the capacity."""
    require_cuda(key, "CSR key")
    L = lib()
    E = int(key.numel())
    dev = key.device
    logical_rows = n_rows
    if trash_row:
        n_rows = n_rows + 1
    row_ptr = torch.empty(n_rows + 1, dtype=torch.int32, device=dev)
    col = torch.empty(E, dtype=torch.int32, device=dev)
    eid = torch.empty(E, dtype=torch.int32, device=dev)
    if sorted_keys:
        L.call("dn4gl_build_csr_sorted", ptr(key), ptr(val), n_rows, E, ptr(row_ptr), ptr(col), ptr(eid),
               ptr(error_flag(dev)), _stream())
    else:
        ws_bytes = L.size("dn4gl_csr_workspace_bytes", n_rows, E)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        L.call("dn4gl_build_csr", ptr(key), ptr(val), n_rows, E, ptr(row_ptr), ptr(col), ptr(eid),
               ptr(ws), ws_bytes, ptr(error_flag(dev)), _stream())   # flag checked lazily by check_errors()
    csr = CSR(row_ptr, col, eid, logical_rows, E)
    if heavy_threshold and heavy_threshold > 0 and E > 0:
        cap = E // heavy_threshold + 1
        csr.heavy_rows = torch.empty(cap, dtype=torch.int32, device=dev)
        csr.heavy_count = torch.empty(1, dtype=torch.int32, device=dev)   # zeroed by dn4gl_collect_heavy_rows
        csr.heavy_thr = heavy_threshold
        L.call("dn4gl_collect_heavy_rows", ptr(row_ptr), logical_rows, heavy_threshold, ptr(csr.heavy_rows), cap,
               ptr(csr.heavy_count), _stream())
    return csr


_err_flags = {}   # device index -> persistent int32[1]; builder kernels only ever write a non-zero error code into it


def error_flag(device):
    """The device's sticky asynchronous error flag (one allocation per device instead of a zero-fill launch per
    builder call; kernels raise it with atomicExch, check_errors() reads and clears it)."""
    idx = device.index if device.index is not None else torch.cuda.current_device()
    f = _err_flags.get(idx)
    if f is None:
        f = _err_flags[idx] = torch.zeros(1, dtype=torch.int32, device=torch.device("cuda", idx))
    return f


def check_errors():
    """Synchronising check of the asynchronous capacity flags raised by builder kernels since the last check."""
    for idx, f in list(_err_flags.items()):
        code = int(f.item())
        if code != 0:
            f.zero_()
            raise RuntimeError("dn4gl builder kernel reported error %d on cuda:%d (-3: row degree above "
                               "DN4GL_MAX_ROW_DEGREE; -1: keys passed as sorted were not; -5: a conj_sizes hint did not match "
                               "the sizes the device counted)" % (code, idx))


def cached_for_tensor(cache, name, tensor, extra, make):
    """value derived from `tensor` (e.g. a CSR compiled from an edge list), cached in the dict `cache` under `name`.
    The entry is valid only for the SAME tensor object at the SAME version with the same `extra`; it holds a reference
    to the tensor, so neither its id nor its storage address can be handed to another batch while the entry lives
    (a key built from data_ptr() silently matched a later batch that the caching allocator placed at the same address)."""
    ent = cache.get(name)
    if ent is not None and ent[0] is tensor and ent[1] == tensor._version and ent[2] == extra:
        return ent[3]
    value = make()
    cache[name] = (tensor, tensor._version, extra, value)
    return value


def _i32(t, device):
    return torch.as_tensor(t).to(device=device, dtype=torch.int32).contiguous()


class BatchedGraph:
    """DGL-flavoured view of a batch: ``ndata`` / ``edata`` frames + cached CSRs.

    The message-passing layers accept this object wherever the reference passes a batched
    ``dgl.DGLGraph`` (rgin.py:156, dmpnn.py:158)."""

    def __init__(self, src, dst, node_ptr, edge_ptr, ndata=None, edata=None):
        require_cuda(src, "graph structure")
        self.src, self.dst = src.to(torch.int32).contiguous(), dst.to(torch.int32).contiguous()
        self.node_ptr, self.edge_ptr = node_ptr.to(torch.int32).contiguous(), edge_ptr.to(torch.int32).contiguous()
        self.ndata = dict(ndata or {})
        self.edata = dict(edata or {})
        self._n = None
        self._csr_in = self._csr_out = None
        self._cache = {}
        self._host_sizes = None
        self._pad_lengths = (None, None)   # (nodes, edges) overrides of the padded lengths, see set_padded_lengths

    # ---- construction -----------------------------------------------------------------------
    @staticmethod
    def from_batch(b, device, flavour="subgraph"):
        """from a flat batch dict (synth.py / transforms.py layout, numpy or tensors)."""
        dev = torch.device(device)
        g = BatchedGraph(_i32(b["src"], dev), _i32(b["dst"], dev), _i32(b["node_ptr"], dev), _i32(b["edge_ptr"], dev))
        names_n = {"vid": "id", "vlabel": "label", "v_is_dummy": "is_dummy", "v_is_reversed": "is_reversed"}
        names_e = {"eid": "id", "elabel": "label", "e_is_dummy": "is_dummy", "e_is_reversed": "is_reversed"}
        for k, name in names_n.items():
            if k in b:
                t = torch.as_tensor(b[k]).to(dev)
                g.ndata[name] = t.bool() if name.startswith("is_") else t.long()
        for k, name in names_e.items():
            if k in b:
                t = torch.as_tensor(b[k]).to(dev)
                g.edata[name] = t.bool() if name.startswith("is_") else t.long()
        g._n = int(b["node_ptr"][-1])
        g._host_sizes = (torch.as_tensor(b["node_ptr"]).cpu().long(), torch.as_tensor(b["edge_ptr"]).cpu().long())
        return g

    # ---- DGL-like queries -----------------------------------------------------------------------
    @property
    def device(self):
        return self.src.device

    @property
    def batch_size(self):
        return int(self.node_ptr.numel()) - 1

    def number_of_nodes(self):
        if self._n is None:
            self._n = int(self.node_ptr[-1].item())
        return self._n

    def number_of_edges(self):
        return int(self.src.numel())

    def host_ptrs(self):
        """(node_ptr, edge_ptr) as host int64 tensors (one D2H copy per batch, cached)."""
        if self._host_sizes is None:
            self._host_sizes = (self.node_ptr.cpu().long(), self.edge_ptr.cpu().long())
        return self._host_sizes

    def batch_num_nodes(self):
        p = self.node_ptr.long()
        return p[1:] - p[:-1]

    def batch_num_edges(self):
        p = self.edge_ptr.long()
        return p[1:] - p[:-1]

    def max_num_nodes(self):
        p = self.host_ptrs()[0]
        return int((p[1:] - p[:-1]).max().item()) if p.numel() > 1 else 0

    def max_num_edges(self):
        p = self.host_ptrs()[1]
        return int((p[1:] - p[:-1]).max().item()) if p.numel() > 1 else 0

    def set_padded_lengths(self, nodes=None, edges=None):
        """pad the (B, L, .) readout tensors of this batch to `nodes` / `edges` rows instead of this batch's own maxima.
        Under data-parallel sharding the counting head and the label filter depend on the padded length of the WHOLE
        mini-batch (SURVEY.md App. A-7, A-14: padded rows contribute the head's bias, pattern padding leaks label 0
        into the gate); a rank that holds a shard passes the batch-wide maxima (``parallel.sync_padded_lengths``) to
        reproduce the single-process numbers exactly.  None keeps the shard's own maximum."""
        for name, v, own in (("nodes", nodes, self.max_num_nodes()), ("edges", edges, self.max_num_edges())):
            if v is not None and int(v) < own:
                raise ValueError("padded %s length %d is smaller than this batch's longest graph (%d)" % (name, v, own))
        self._pad_lengths = (None if nodes is None else int(nodes), None if edges is None else int(edges))
        return self

    def padded_num_nodes(self):
        """L of the left-padded (B, L, .) node tensors (split_and_batchify_graph_feats, utils/dl.py:51-81)."""
        return self._pad_lengths[0] if self._pad_lengths[0] is not None else self.max_num_nodes()

    def padded_num_edges(self):
        return self._pad_lengths[1] if self._pad_lengths[1] is not None else self.max_num_edges()

    def all_edges(self, form="uv", order="eid"):
        if order != "eid":
            raise NotImplementedError("only order='eid' is provided on the hot path")
        u, v = self.src.long(), self.dst.long()
        if form == "uv":
            return u, v
        if form == "all":
            return u, v, torch.arange(u.numel(), device=u.device)
        raise ValueError(form)

    def to(self, device):
        if torch.device(device) != self.device:
            raise NotImplementedError("BatchedGraph is built directly in HBM; build it on the target device")
        return self

    # ---- structure caches ---------------------------------------------------------------------------
    @property
    def csr_in(self):
        """in-edges of every node: row v lists (src, eid) of edges with dst = v, ascending eid."""
        if self._csr_in is None:
            self._csr_in = build_csr(self.dst, self.src, self.number_of_nodes())
            self._csr_in.seg_ptr, self._csr_in.max_seg = self.node_ptr, self._max_seg()
        return self._csr_in

    @property
    def csr_out(self):
        """out-edges of every node (transpose): row u lists (dst, eid) of edges with src = u."""
        if self._csr_out is None:
            self._csr_out = build_csr(self.src, self.dst, self.number_of_nodes())
            self._csr_out.seg_ptr, self._csr_out.max_seg = self.node_ptr, self._max_seg()
        return self._csr_out

    def _max_seg(self):
        """rows of the largest graph when the host already holds the sizes (no device sync otherwise)."""
        return self.max_num_nodes() if self._host_sizes is not None else None

    def in_degrees(self):
        if "in_deg" not in self.ndata:
            rp = self.csr_in.row_ptr.long()
            self.ndata["in_deg"] = rp[1:] - rp[:-1]
        return self.ndata["in_deg"]

    def out_degrees(self):
        if "out_deg" not in self.ndata:
            rp = self.csr_out.row_ptr.long()
            self.ndata["out_deg"] = rp[1:] - rp[:-1]
        return self.ndata["out_deg"]

    def cached(self, key, builder):
        if key not in self._cache:
            self._cache[key] = builder()
        return self._cache[key]
