"""Match-weight targets from ground-truth subisomorphisms (SURVEY.md section 8(f), rank 2).

With ``--match_weights node`` / ``edge`` the reference attaches to every sample a per-graph-node (per-graph-edge) count of
how many subisomorphisms use it: ``GraphAdjDataset.calculate_node_weights`` / ``calculate_edge_weights``
(subgraph_isomorphism/dataset.py:1491-1520) around the numba loops ``compute_nodeseq_subisoweights`` /
``compute_edgeseq_subisoweights`` (:54-108).  Here the whole mini-batch is done by two kernels (csrc/subiso.cu).

A batch of subisomorphisms is ``dict(val_ptr int32[B+1], values int32[total])``: sample b owns ``S_b`` rows of
``np_b`` (= its pattern's node count) graph-local node ids, concatenated row-major; ``pack_subisomorphisms`` builds it
from the per-sample ``(S_b, np_b)`` matrices the reference stores (``x["subisomorphisms"]``).
"""
import numpy as np
import torch

from .._lib import lib, ptr
from ..graph import _stream, build_csr, error_flag, require_cuda


def pack_subisomorphisms(mats, device=None):
    """list of (S_b, np_b) integer arrays -> dict(val_ptr, values, rows) (numpy, or device tensors if device given)."""
    sizes = [int(np.asarray(m).size) for m in mats]
    val_ptr = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int32)
    values = (np.concatenate([np.asarray(m).reshape(-1) for m in mats]) if mats else np.zeros(0)).astype(np.int32)
    rows = np.array([int(np.asarray(m).shape[0]) if np.asarray(m).ndim == 2 else 0 for m in mats], dtype=np.int32)
    out = dict(val_ptr=val_ptr, values=values, rows=rows)
    if device is not None:
        out = {k: torch.from_numpy(v).to(device) for k, v in out.items()}
    return out


def add_dummy_to_subisomorphisms(mats, graph_b):
    """what ``add_dummy_nodes_edges`` does to a sample's ground truth (train.py:467-472): every subisomorphism also maps
    the pattern's dummy node to the graph's dummy node, whose graph-local id is the graph's ORIGINAL node count.
    mats: per-sample (S_b, np_b) arrays; graph_b: the batch BEFORE augmentation (host numpy)."""
    n = np.diff(np.asarray(graph_b["node_ptr"]))
    out = []
    for b, m in enumerate(mats):
        m = np.asarray(m, dtype=np.int64)
        if m.ndim != 2:
            m = m.reshape(0, 0)
        out.append(np.concatenate([m, np.full((m.shape[0], 1), int(n[b]), dtype=np.int64)], axis=1))
    return out


def dummy_column_offsets(val_sizes, rows):
    """host int64 (B + 1) offsets of a packed subisomorphism batch after ``add_dummy_to_subisomorphisms``: sample b's
    ``val_sizes[b]`` ids in ``rows[b]`` rows become ``val_sizes[b] + rows[b]`` ids."""
    sizes = np.asarray(val_sizes, np.int64) + np.asarray(rows, np.int64)
    out = np.zeros(len(sizes) + 1, dtype=np.int64)
    np.cumsum(sizes, out=out[1:])
    return out


def append_dummy_column(subiso, graph_b, out_ptr, out_total):
    """``add_dummy_to_subisomorphisms`` of a packed device batch (one launch, no device->host read): every row also maps
    the pattern's dummy node to the graph's, whose graph-local id is the graph's node count in `graph_b`, the batch
    BEFORE augmentation.  out_ptr: int32 device (B + 1) offsets of the result and out_total its last entry, both from
    ``dummy_column_offsets`` on the host.  -> dict(val_ptr=out_ptr, values, rows) in the ``pack_subisomorphisms`` layout."""
    from .. import ops
    values = ops.subiso_append_dummy(subiso["val_ptr"], subiso["values"], subiso["rows"], graph_b["node_ptr"], out_ptr,
                                     out_total)
    return dict(val_ptr=out_ptr, values=values, rows=subiso["rows"])


def node_weights(subiso, graph_b):
    """(N_g,) int64: number of subisomorphism entries that hit each graph node (zeros for samples without matches)."""
    return node_weights_i32(subiso, graph_b).long()


def node_weights_i32(subiso, graph_b):
    """``node_weights`` as the kernel writes it (int32), what the fused match loss reads."""
    require_cuda(graph_b["src"], "graph batch")
    dev = graph_b["src"].device
    B, Ng = int(graph_b["num_graphs"]), int(graph_b["vlabel"].numel())
    w = torch.empty(Ng, dtype=torch.int32, device=dev)
    lib().call("dn4gl_subiso_node_weights", B, ptr(subiso["val_ptr"]), ptr(subiso["values"]), int(subiso["values"].numel()),
               ptr(graph_b["node_ptr"]), Ng, ptr(w), _stream())
    return w


def _sorted_out_lists(graph_b):
    """CSR by source with rows sorted by (dst, edge id): all_edges(order="srcdst"), dataset.py:1508 / train.py:573."""
    L = lib()
    dev = graph_b["src"].device
    Ng = int(graph_b["vlabel"].numel())
    csr = build_csr(graph_b["src"], graph_b["dst"], Ng, heavy_threshold=0)
    wsb = L.size("dn4gl_sort_rows_workspace_bytes", Ng)
    ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
    L.call("dn4gl_sort_csr_rows", ptr(csr.row_ptr), Ng, ptr(csr.eid), ptr(graph_b["dst"]), ptr(ws), wsb, ptr(error_flag(dev)),
           _stream())
    return csr


def _work_ptr(subiso, pattern_b, dev):
    B = int(pattern_b["num_graphs"])
    m = (pattern_b["edge_ptr"][1:] - pattern_b["edge_ptr"][:-1]).long()
    work = torch.zeros(B + 1, dtype=torch.int64, device=dev)
    work[1:] = torch.cumsum(subiso["rows"].long() * m, 0)
    total = int(work[-1].item())
    if total >= 2 ** 31:
        raise ValueError("more than 2^31 (subisomorphism, pattern edge) pairs in one batch")
    return work.to(torch.int32), total


def conjugate_subisomorphisms(subiso, pattern_b, graph_b):
    """node maps -> edge maps for the conjugate (edge-to-vertex) graphs: ``get_conjugate_subisomorphisms``
    (utils/graph.py:294-330) + the ``g_eid[...]`` gather of ``convert_to_conjugate`` (train.py:577-587), batched.
    Returns (work_ptr int32[B+1], conj int64[total]): sample b's (S_b, m_b) matrix of graph-local edge ids is
    ``conj[work_ptr[b]:work_ptr[b+1]].view(S_b, m_b)``."""
    require_cuda(graph_b["src"], "graph batch")
    dev = graph_b["src"].device
    B, Ep = int(graph_b["num_graphs"]), int(pattern_b["src"].numel())
    work, total = _work_ptr(subiso, pattern_b, dev)
    conj = torch.empty(max(total, 1), dtype=torch.int32, device=dev)
    if total > 0:
        csr = _sorted_out_lists(graph_b)
        active = torch.empty(max(Ep, 1), dtype=torch.int32, device=dev)
        lib().call("dn4gl_subiso_conjugate", B, ptr(work), total, ptr(subiso["val_ptr"]), ptr(subiso["values"]),
                   ptr(pattern_b["node_ptr"]), ptr(pattern_b["edge_ptr"]), ptr(pattern_b["src"]), ptr(pattern_b["dst"]),
                   ptr(pattern_b["elabel"]), Ep, ptr(active), ptr(graph_b["node_ptr"]), ptr(graph_b["edge_ptr"]),
                   ptr(csr.row_ptr), ptr(csr.eid), ptr(graph_b["dst"]), ptr(graph_b["elabel"]), ptr(conj), _stream())
    return work, conj[:total].long()


def edge_weights(subiso, pattern_b, graph_b):
    """(E_g,) int64 in edge-id order: for every subisomorphism and pattern edge (u, v, l), +1 on every graph edge
    (map[u], map[v]) with label l -- with the reference's run/dict semantics for repeated pattern pairs."""
    return edge_weights_i32(subiso, pattern_b, graph_b).long()


def edge_weights_i32(subiso, pattern_b, graph_b):
    """``edge_weights`` as the kernel writes it (int32); one device->host read (the work total)."""
    require_cuda(graph_b["src"], "graph batch")
    L = lib()
    dev = graph_b["src"].device
    B = int(graph_b["num_graphs"])
    Ng, Eg, Ep = int(graph_b["vlabel"].numel()), int(graph_b["src"].numel()), int(pattern_b["src"].numel())
    w = torch.empty(Eg, dtype=torch.int32, device=dev)
    # out-lists sorted by (dst, edge id): all_edges(order="srcdst"), dataset.py:1508
    csr = build_csr(graph_b["src"], graph_b["dst"], Ng, heavy_threshold=0)
    wsb = L.size("dn4gl_sort_rows_workspace_bytes", Ng)
    ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
    L.call("dn4gl_sort_csr_rows", ptr(csr.row_ptr), Ng, ptr(csr.eid), ptr(graph_b["dst"]), ptr(ws), wsb, ptr(error_flag(dev)),
           _stream())
    m = (pattern_b["edge_ptr"][1:] - pattern_b["edge_ptr"][:-1]).long()
    work = torch.zeros(B + 1, dtype=torch.int64, device=dev)
    work[1:] = torch.cumsum(subiso["rows"].long() * m, 0)
    total = int(work[-1].item())
    if total >= 2 ** 31:
        raise ValueError("edge_weights: more than 2^31 (subisomorphism, pattern edge) pairs in one batch")
    active = torch.empty(max(Ep, 1), dtype=torch.int32, device=dev)
    L.call("dn4gl_subiso_edge_weights", B, ptr(work.to(torch.int32)), total, ptr(subiso["val_ptr"]), ptr(subiso["values"]),
           ptr(pattern_b["node_ptr"]), ptr(pattern_b["edge_ptr"]), ptr(pattern_b["src"]), ptr(pattern_b["dst"]),
           ptr(pattern_b["elabel"]), Ep, ptr(active), ptr(graph_b["node_ptr"]), ptr(csr.row_ptr), ptr(csr.eid),
           ptr(graph_b["dst"]), ptr(graph_b["elabel"]), Eg, ptr(w), _stream())
    return w
