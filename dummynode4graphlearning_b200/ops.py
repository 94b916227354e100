"""torch.autograd wrappers over the C-ABI kernels (forward AND hand-written backward).

PyTorch supplies device memory, streams and the autograd tape; every aggregation, readout and
per-edge op below runs in libdn4gl.so.  None of these functions has a CPU or pure-PyTorch
implementation: tensors must be CUDA fp32, otherwise an error is raised.
"""
import os

import torch

from ._lib import lib, ptr
from .graph import CSR, _stream, bind_device, require_cuda


def _f32c(t):
    if t.dtype != torch.float32:
        raise TypeError("expected float32, got %s" % t.dtype)
    return t.contiguous()


SPMM_MODE = os.environ.get("DN4GL_SPMM", "tiled")          # "tiled" (pipelined shared-memory staging) | "rows" (per-row gathers)
TILE_SMEM = None                                           # override of graph.TILE_SMEM (tests / sweeps)
_TILED_D = (16, 32, 64, 128, 256, 512)


def _spmm(csr: CSR, x, n_out, self_scale, eps_dev=None):
    """eps_dev: optional device scalar; the kernel then uses self_scale = 1 + eps_dev (no host read)."""
    require_cuda(x, "features")
    x = _f32c(x)
    D = x.size(1)
    out = torch.empty((n_out, D), dtype=torch.float32, device=x.device)
    if SPMM_MODE == "tiled" and csr.seg_ptr is not None and x.size(0) == n_out and D in _TILED_D:
        t = csr.tiles(D, TILE_SMEM)
        lib().call("dn4gl_spmm_tiled_f32", ptr(csr.row_ptr), ptr(csr.col), ptr(x), ptr(out), n_out, D,
                   float(self_scale), ptr(eps_dev), ptr(t["desc"]), t["T"], ptr(t["heavy_list"]), ptr(t["heavy_count"]),
                   t["heavy_cap"], t["smem"], t["stages"], t["npr"], t["warps"], _stream())
        return out
    lib().call("dn4gl_spmm_sum_f32", ptr(csr.row_ptr), ptr(csr.col), ptr(x), ptr(out), n_out, x.size(0), D,
               float(self_scale), ptr(eps_dev), ptr(csr.heavy_rows), ptr(csr.heavy_count), csr.heavy_thr, _stream())
    return out


class _SpmmSum(torch.autograd.Function):
    """out[v] = self_scale * x[v] + sum_{p in row v} x[col[p]]   (K1).  The adjoint is the same
    kernel on the transposed CSR, so the backward is deterministic and atomic-free."""

    @staticmethod
    def forward(ctx, x, csr_fwd, csr_bwd, self_scale):
        ctx.csr_bwd, ctx.self_scale, ctx.n_src = csr_bwd, self_scale, x.size(0)
        return _spmm(csr_fwd, x, csr_fwd.n_rows, self_scale)

    @staticmethod
    def backward(ctx, g):
        return _spmm(ctx.csr_bwd, g, ctx.n_src, ctx.self_scale), None, None, None


def spmm_sum(x, csr_fwd, csr_bwd, self_scale=0.0):
    """Sum aggregation over a CSR; ``csr_bwd`` must be the transpose of ``csr_fwd``."""
    return _SpmmSum.apply(x, csr_fwd, csr_bwd, float(self_scale))


def graph_sum_aggregate(graph, x, self_scale=0.0):
    """agg[v] = self_scale*x[v] + sum over in-edges (u -> v) of x[u]: DGL ``update_all(copy_u, fn.sum)`` /
    PyG ``propagate(aggr='add')``."""
    return spmm_sum(x, graph.csr_in, graph.csr_out, self_scale)


# ---------------------------------------------------------------------------------------------
class _SegmentSum(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, seg_ptr, mask, mode):
        require_cuda(x, "features")
        x = _f32c(x)
        B, D = seg_ptr.numel() - 1, x.size(1)
        out = torch.empty((B, D), dtype=torch.float32, device=x.device)
        lib().call("dn4gl_segment_sum_f32", ptr(seg_ptr), ptr(mask), ptr(x), ptr(out), B, D, mode, _stream())
        ctx.seg_ptr, ctx.mask, ctx.mode, ctx.n = seg_ptr, mask, mode, x.size(0)
        return out

    @staticmethod
    def backward(ctx, g):
        g = _f32c(g)
        B, D = g.shape
        gx = torch.empty((ctx.n, D), dtype=torch.float32, device=g.device)
        lib().call("dn4gl_segment_bcast_f32", ptr(ctx.seg_ptr), ptr(ctx.mask), ptr(g), ptr(gx), B, ctx.n, D,
                   ctx.mode, _stream())
        return gx, None, None, None


def segment_sum(x, seg_ptr, mask=None, mean=False):
    """per-graph readout over contiguous segments (K3); mask: uint8/bool, 1 = skip row."""
    if mask is not None:
        mask = mask.to(torch.uint8).contiguous()
    return _SegmentSum.apply(x, seg_ptr, mask, 1 if mean else 0)


class _PadSegments(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, seg_ptr, mask, Lmax):
        require_cuda(x, "features")
        x = _f32c(x)
        B, D = seg_ptr.numel() - 1, x.size(1)
        out = torch.empty((B, Lmax, D), dtype=torch.float32, device=x.device)
        lib().call("dn4gl_pad_segments_f32", ptr(seg_ptr), ptr(mask), ptr(x), ptr(out), B, Lmax, D, _stream())
        ctx.seg_ptr, ctx.mask, ctx.n = seg_ptr, mask, x.size(0)
        return out

    @staticmethod
    def backward(ctx, g):
        g = _f32c(g)
        B, Lmax, D = g.shape
        gx = torch.empty((ctx.n, D), dtype=torch.float32, device=g.device)
        lib().call("dn4gl_unpad_segments_f32", ptr(ctx.seg_ptr), ptr(ctx.mask), ptr(g), ptr(gx), B, Lmax, D, ctx.n,
                   _stream())
        return gx, None, None, None


def pad_segments(x, seg_ptr, Lmax, mask=None):
    """left-padded (B, Lmax, D) batchify of ragged rows; rows with mask=1 are zeroed
    (split_and_batchify_graph_feats(pre_pad=True) + masked_fill, utils/dl.py:51-81)."""
    if mask is not None:
        mask = mask.to(torch.uint8).contiguous()
    return _PadSegments.apply(x, seg_ptr, mask, int(Lmax))


def label_filter_gate(graph, pattern, Lp_max, kind="node"):
    """(N_g, 1) float gate of ScalarFilter (filter.py:10-16) without the (B, Lg, Lp) temporary.
    kind="node": node labels vs the pattern's node labels (basemodel.py:830-847);
    kind="edge": edge labels vs the pattern's edge labels (basemodel.py:1434-1442)."""
    if kind == "node":
        g_lab, p_lab, g_ptr, p_ptr = graph.ndata["label"], pattern.ndata["label"], graph.node_ptr, pattern.node_ptr
    else:
        g_lab, p_lab, g_ptr, p_ptr = graph.edata["label"], pattern.edata["label"], graph.edge_ptr, pattern.edge_ptr
    g_label = graph.cached("label_i32_" + kind, lambda: g_lab.to(torch.int32).contiguous())
    p_label = pattern.cached("label_i32_" + kind, lambda: p_lab.to(torch.int32).contiguous())
    require_cuda(g_label, "labels")
    Ng = g_label.numel()
    gate = torch.empty((Ng, 1), dtype=torch.float32, device=g_label.device)
    lib().call("dn4gl_label_filter_gate", ptr(g_ptr), ptr(g_label), ptr(p_ptr), ptr(p_label),
               graph.batch_size, int(Lp_max), Ng, ptr(gate), _stream())
    return gate


class _NllMean(torch.autograd.Function):
    """F.nll_loss(log_probs, y) (mean reduction, main.py:41) as one small kernel each way."""

    @staticmethod
    def forward(ctx, logp, y):
        require_cuda(logp, "log-probabilities")
        logp = _f32c(logp)
        y = y.contiguous()
        B, C = logp.shape
        loss = torch.empty((), dtype=torch.float32, device=logp.device)
        lib().call("dn4gl_nll_mean_f32", ptr(logp), ptr(y), B, C, ptr(loss), _stream())
        ctx.save_for_backward(y)
        ctx.shape = (B, C)
        return loss

    @staticmethod
    def backward(ctx, g):
        (y,) = ctx.saved_tensors
        B, C = ctx.shape
        g = _f32c(g).reshape(1)
        out = torch.empty((B, C), dtype=torch.float32, device=g.device)
        lib().call("dn4gl_nll_mean_bwd_f32", ptr(g), ptr(y), B, C, ptr(out), _stream())
        return out, None


JK_HEAD_MAX_LAYERS, JK_HEAD_MAX_CLASSES = 16, 32


def jk_head_supported(L, D, C):
    """shapes dn4gl_jk_head_{fwd,bwd}_f32 take (include/dn4gl.h)."""
    return 1 <= L <= JK_HEAD_MAX_LAYERS and 1 <= C <= JK_HEAD_MAX_CLASSES and ((C + 8) * L * D + 10 * C + 8) * 4 <= 48 * 1024


def _ptr_array(tensors):
    import ctypes
    return (ctypes.c_void_p * len(tensors))(*[t.data_ptr() for t in tensors])


class _JkHead(torch.autograd.Function):
    """log_softmax(sum_l Linear_l(pooled_l)) of the GIN classifier (gconv.py:205-214, dropout 0) as one kernel each way;
    seg_ptr: sum pooling, layer 0's bias is counted once per pooled row (gconv.py:210)."""

    @staticmethod
    def forward(ctx, seg_ptr, L, *tensors):
        pooled = [_f32c(t) for t in tensors[:L]]
        W = [_f32c(t) for t in tensors[L:2 * L]]
        bias = [_f32c(t) for t in tensors[2 * L:3 * L]]
        require_cuda(pooled[0], "pooled rows")
        B, D = pooled[0].shape
        C = W[0].size(0)
        logp = torch.empty((B, C), dtype=torch.float32, device=pooled[0].device)
        lib().call("dn4gl_jk_head_fwd_f32", _ptr_array(pooled), _ptr_array(W), _ptr_array(bias), L, B, D, C, ptr(seg_ptr),
                   ptr(logp), _stream())
        ctx.save_for_backward(logp, *pooled, *W)
        ctx.seg_ptr, ctx.dims = seg_ptr, (L, B, D, C)
        return logp

    @staticmethod
    def backward(ctx, g):
        L, B, D, C = ctx.dims
        logp, pooled, W = ctx.saved_tensors[0], ctx.saved_tensors[1:1 + L], ctx.saved_tensors[1 + L:]
        dev = logp.device
        g_pooled = torch.empty((L, B, D), dtype=torch.float32, device=dev)
        dW = torch.empty((L, C, D), dtype=torch.float32, device=dev)
        db = torch.empty((L, C), dtype=torch.float32, device=dev)
        if B == 0:
            g_pooled.zero_(), dW.zero_(), db.zero_()
        else:
            lb = lib()
            wsb = lb.size("dn4gl_jk_head_workspace_bytes", L, B, D, C)
            ws, counter = _tc_ws(dev, wsb)
            lb.call("dn4gl_jk_head_bwd_f32", ptr(_f32c(g)), ptr(logp), _ptr_array(pooled), _ptr_array(W), L, B, D, C,
                    ptr(ctx.seg_ptr), _ptr_array(list(g_pooled)), _ptr_array(list(dW)), _ptr_array(list(db)), ptr(ws), wsb,
                    ptr(counter), _stream())
        return (None, None) + tuple(g_pooled) + tuple(dW) + tuple(db)


def jk_head(pooled, weights, biases, seg_ptr=None):
    """log_softmax(sum_l pooled[l] @ weights[l].T + n_b * biases[0] + sum_{l >= 1} biases[l]); n_b = rows of graph b when
    seg_ptr is given, else 1.  jk_head_supported(L, D, C) must hold."""
    L = len(pooled)
    return _JkHead.apply(seg_ptr, L, *pooled, *weights, *biases)


def nll_loss(logp, y):
    """mean negative log-likelihood of int64 targets y under row-wise log-probabilities logp (B, C)."""
    if y.dtype != torch.int64:
        y = y.long()
    return _NllMean.apply(logp, y)


# ---------------------------------------------------------------------------------------------
def _rev_u8(graph):
    if "is_reversed" not in graph.edata:
        return None
    return graph.cached("rev_u8", lambda: graph.edata["is_reversed"].to(torch.uint8).contiguous())


class _DmpNodeAgg(torch.autograd.Function):
    """S[v] = [sum_{in(v), rev} ef | sum_{in(v), !rev} ef]   (K4)."""

    @staticmethod
    def forward(ctx, ef, graph):
        require_cuda(ef, "edge features")
        ef = _f32c(ef)
        N, D = graph.number_of_nodes(), ef.size(1)
        csr = graph.csr_in
        S = torch.empty((N, 2 * D), dtype=torch.float32, device=ef.device)
        lib().call("dn4gl_dmp_node_agg_f32", ptr(csr.row_ptr), ptr(csr.eid), ptr(_rev_u8(graph)), ptr(ef), ptr(S), N, D,
                   ptr(csr.heavy_rows), ptr(csr.heavy_count), csr.heavy_thr, _stream())
        ctx.graph = graph
        return S

    @staticmethod
    def backward(ctx, gS):
        graph = ctx.graph
        gS = _f32c(gS)
        E, D = graph.number_of_edges(), gS.size(1) // 2
        gef = torch.empty((E, D), dtype=torch.float32, device=gS.device)
        lib().call("dn4gl_dmp_node_agg_bwd_f32", ptr(graph.dst), ptr(_rev_u8(graph)), ptr(gS), ptr(gef), E, D, _stream())
        return gef, None


def dmp_node_agg(ef, graph):
    return _DmpNodeAgg.apply(ef, graph)


class _DmpEdgeUpdate(torch.autograd.Function):
    """out[e] = T[e,:D] + c_e T[e,D:] + (rev ? P[src]-Q[dst] : P[dst]-Q[src]) + bias   (K5)."""

    @staticmethod
    def forward(ctx, PQ, T, bias, graph):
        require_cuda(PQ, "node projections")
        PQ, T = _f32c(PQ), _f32c(T)
        E, D = graph.number_of_edges(), T.size(1) // 2
        out_deg = graph.cached("out_deg_i32", lambda: graph.out_degrees().to(torch.int32).contiguous())
        out = torch.empty((E, D), dtype=torch.float32, device=T.device)
        b = None if bias is None else _f32c(bias)
        lib().call("dn4gl_dmp_edge_update_f32", ptr(graph.src), ptr(graph.dst), ptr(_rev_u8(graph)), ptr(out_deg),
                   ptr(PQ), ptr(T), ptr(b), ptr(out), E, D, _stream())
        ctx.graph, ctx.has_bias, ctx.out_deg = graph, bias is not None, out_deg
        return out

    @staticmethod
    def backward(ctx, g):
        graph = ctx.graph
        g = _f32c(g)
        E, D = g.shape
        N = graph.number_of_nodes()
        gT = torch.empty((E, 2 * D), dtype=torch.float32, device=g.device)
        lib().call("dn4gl_dmp_edge_update_bwd_T_f32", ptr(graph.dst), ptr(ctx.out_deg), ptr(g), ptr(gT), E, D, _stream())
        gPQ = torch.empty((N, 2 * D), dtype=torch.float32, device=g.device)
        ci, co = graph.csr_in, graph.csr_out
        lib().call("dn4gl_dmp_edge_update_bwd_PQ_f32", ptr(ci.row_ptr), ptr(ci.eid), ptr(co.row_ptr), ptr(co.eid),
                   ptr(_rev_u8(graph)), ptr(g), ptr(gPQ), N, D, _stream())
        gb = g.sum(dim=0) if ctx.has_bias else None
        return gPQ, gT, gb, None


def dmp_edge_update(PQ, T, bias, graph):
    return _DmpEdgeUpdate.apply(PQ, T, bias, graph)


class _CompEdge(torch.autograd.Function):
    """C[e] = a[src e] * comp(h[src e], ef[e]) for comp in {sub, mult} (compgcn.py:214-240 without the weights)."""

    @staticmethod
    def forward(ctx, h, ef, graph, op, a):
        require_cuda(ef, "edge features")
        h, ef = _f32c(h), _f32c(ef)
        E, D = ef.shape
        a = None if a is None else _f32c(a).view(-1)
        C = torch.empty((E, D), dtype=torch.float32, device=ef.device)
        lib().call("dn4gl_comp_edge_f32", ptr(graph.src), ptr(a), ptr(h), ptr(ef), ptr(C), E, D, op, _stream())
        ctx.save_for_backward(h, ef, a)
        ctx.graph, ctx.op = graph, op
        return C

    @staticmethod
    def backward(ctx, gC):
        h, ef, a = ctx.saved_tensors
        graph, op = ctx.graph, ctx.op
        gC = _f32c(gC)
        E, D = gC.shape
        gh = gef = None
        if ctx.needs_input_grad[1]:
            gef = torch.empty_like(gC)
            lib().call("dn4gl_comp_edge_bwd_ef_f32", ptr(graph.src), ptr(a), ptr(h), ptr(gC), ptr(gef), E, D, op, _stream())
        if ctx.needs_input_grad[0]:
            co = graph.csr_out
            gh = torch.empty_like(h)
            lib().call("dn4gl_comp_edge_bwd_h_f32", ptr(co.row_ptr), ptr(co.eid), ptr(a), ptr(ef), ptr(gC), ptr(gh),
                       h.size(0), D, op, _stream())
        return gh, gef, None, None, None


COMP_SUB, COMP_MULT = 0, 1


def comp_edge(h, ef, graph, op, src_scale=None):
    """per-edge CompGCN composition with the source half of the edge normalisation folded in."""
    return _CompEdge.apply(h, ef, graph, int(op), src_scale)


def gather_rows(x, idx_i32):
    """out[i] = x[idx[i]] (no autograd; used for attribute plumbing of the transforms)."""
    require_cuda(x, "rows")
    x = _f32c(x)
    n, D = idx_i32.numel(), x.size(1)
    out = torch.empty((n, D), dtype=torch.float32, device=x.device)
    lib().call("dn4gl_gather_rows_f32", ptr(idx_i32), ptr(x), ptr(out), n, D, _stream())
    return out


# ---------------------------------------------------------------------------------------------
# dense helpers: forward / input-gradient GEMMs are plain library GEMMs (cuBLAS through torch); the WEIGHT gradient
# is a reduction over all N rows with a tiny output and runs in libdn4gl (dn4gl_atb_f32).
def atb_supported(ka, kb):
    return ((ka + 3) // 4) * ((kb + 3) // 4) <= 256


def atb(A, B, want_colsum=False):
    """(A^T B, colsum(A) or None) for row-major A (N, Ka), B (N, Kb)."""
    require_cuda(A, "activations")
    A, B = _f32c(A), _f32c(B)
    N, Ka = A.shape
    Kb = B.size(1)
    if not atb_supported(Ka, Kb):   # wide outputs (e.g. the (D, R*D) relation table) are regular GEMMs: library
        return A.t() @ B, (A.sum(0) if want_colsum else None)
    C = torch.empty((Ka, Kb), dtype=torch.float32, device=A.device)
    cs = torch.empty(Ka, dtype=torch.float32, device=A.device) if want_colsum else None
    L = lib()
    wsb = L.size("dn4gl_atb_workspace_bytes", N, Ka, Kb)
    ws = torch.empty(wsb, dtype=torch.uint8, device=A.device)
    L.call("dn4gl_atb_f32", ptr(A), ptr(B), ptr(C), ptr(cs), N, Ka, Kb, ptr(ws), wsb, _stream())
    return C, cs


# Forward and data-gradient products on the tensor cores (dn4gl_gemm_f32: 3xTF32 with fp32 register accumulation across
# the contraction, csrc/gemm3x.cu) instead of the library's SIMT SGEMM.  DN4GL_GEMM_TC=0 restores the library GEMMs.
GEMM_TENSOR_CORES = os.environ.get("DN4GL_GEMM_TC", "1") == "1"
B_IS_WEIGHT, B_IS_KXM = 0, 1      # b_layout of dn4gl_gemm_f32: (M x K) nn.Linear weight / (K x M) matrix

_gemm_ws = {}


def gemm(a, b, b_layout, bias=None):
    """a (N, K) @ b^T (b: (M, K), b_layout 0) or a @ b (b: (K, M), b_layout 1), + bias; fp32, no autograd."""
    require_cuda(a, "the left operand")
    a, b = _f32c(a), _f32c(b)
    N, K = a.shape
    M = b.size(0) if b_layout == B_IS_WEIGHT else b.size(1)
    assert (b.size(1) if b_layout == B_IS_WEIGHT else b.size(0)) == K, "inner dimensions differ"
    out = torch.empty((N, M), dtype=torch.float32, device=a.device)
    if N == 0 or M == 0:
        return out
    if K == 0:
        return out.zero_() if bias is None else out.copy_(bias.expand(N, M))
    L = lib()
    wsb = L.size("dn4gl_gemm_workspace_bytes", K, M)
    if torch.cuda.is_current_stream_capturing():
        ws = torch.empty(wsb, dtype=torch.uint8, device=a.device)
    else:                       # one growing workspace per (device, stream): consumed before the next launch on that stream
        key = (a.device.index, _stream())
        ws = _gemm_ws.get(key)
        if ws is None or ws.numel() < wsb:
            ws = _gemm_ws[key] = torch.empty(max(wsb, 1 << 20), dtype=torch.uint8, device=a.device)
    L.call("dn4gl_gemm_f32", ptr(a), N, K, K, ptr(b), b.size(1), int(b_layout), M, ptr(None if bias is None else _f32c(bias)),
           ptr(out), M, ptr(ws), wsb, _stream())
    return out


GEMM_MIN_MACS = float(os.environ.get("DN4GL_GEMM_MIN_MACS", "0"))      # below N * K * M: the library GEMM (measurement switch)
# Products with fewer rows than this stay on the library GEMM: they are the per-GRAPH layers of the counting head (B = 8 .. 512
# rows), not the per-node / per-edge products of the message-passing path.  Two reasons, both measured: at 512 rows the
# two-kernel tensor-core GEMM takes 8-11 us against 2-4 us (profiles/r4j_bench_gemm.txt), and the head multiplies sum-pooled
# representations of magnitude 1e3 straight into the prediction -- the tensor core's truncating accumulation, harmless
# everywhere else, moved the DMPNN 'large' loss from 3e-6 to 3.4e-5 of the oracle when pred_fc1 / pred_fc2 ran on it
# (profiles/r4l_parity_errors_head_on_tensor_cores.json).
GEMM_MIN_ROWS = int(os.environ.get("DN4GL_GEMM_MIN_ROWS", "1024"))


_gemm_scope = [None]      # innermost gemm_tensor_cores(...) override, None = the module default


class gemm_tensor_cores:
    """``with ops.gemm_tensor_cores(False): ...`` -- products issued inside use the library fp32 GEMM (True: dn4gl_gemm_f32)
    whatever the module default is; the decision taken in a forward is kept for its backward."""

    def __init__(self, flag):
        self.flag = None if flag is None else bool(flag)

    def __enter__(self):
        self.prev = _gemm_scope[0]
        if self.flag is not None:
            _gemm_scope[0] = self.flag
        return self

    def __exit__(self, *exc):
        _gemm_scope[0] = self.prev
        return False


def _use_gemm(a, b):
    on = GEMM_TENSOR_CORES if _gemm_scope[0] is None else (_gemm_scope[0] and os.environ.get("DN4GL_GEMM_TC", "1") == "1")
    if not (on and a.is_cuda and b.is_cuda and a.dtype == torch.float32 and b.dtype == torch.float32):
        return False
    if a.size(0) < GEMM_MIN_ROWS:
        return False
    return GEMM_MIN_MACS <= 0 or a.size(0) * b.numel() >= GEMM_MIN_MACS


class _Linear(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight, bias):
        ctx.save_for_backward(x, weight)
        ctx.has_bias = bias is not None
        ctx.use_gemm = _use_gemm(x, weight)
        if ctx.use_gemm:
            return gemm(x, weight, B_IS_WEIGHT, bias)
        return torch.addmm(bias, x, weight.t()) if bias is not None else x @ weight.t()

    @staticmethod
    def backward(ctx, g):
        x, weight = ctx.saved_tensors
        gx = gw = gb = None
        if ctx.needs_input_grad[0]:
            gx = gemm(g, weight, B_IS_KXM) if ctx.use_gemm else g @ weight
        if ctx.needs_input_grad[1] or (ctx.has_bias and ctx.needs_input_grad[2]):
            gw, gb = atb(g, x, want_colsum=ctx.has_bias)
        return gx, gw, gb


def linear(x, weight, bias=None):
    """F.linear with the weight/bias gradient computed by the row-reduction kernel."""
    lead = x.shape[:-1]
    y = _Linear.apply(x.reshape(-1, x.size(-1)), weight, bias)
    return y.view(lead + (weight.size(0),))


class _MatmulXW(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, w):
        ctx.save_for_backward(x, w)
        ctx.use_gemm = _use_gemm(x, w)
        return gemm(x, w, B_IS_KXM) if ctx.use_gemm else x @ w

    @staticmethod
    def backward(ctx, g):
        x, w = ctx.saved_tensors
        gx = None
        if ctx.needs_input_grad[0]:
            gx = gemm(g, w, B_IS_WEIGHT) if ctx.use_gemm else g @ w.t()
        gw = atb(x, g)[0] if ctx.needs_input_grad[1] else None
        return gx, gw


def matmul_xw(x, w):
    """x (N, K) @ w (K, M) for a parameter (or parameter expression) w; dW = x^T g by the row-reduction kernel."""
    return _MatmulXW.apply(x, w)


class Linear(torch.nn.Linear):
    """nn.Linear (same parameters / state_dict keys) whose backward uses dn4gl_atb_f32 for dW, db."""

    def forward(self, x):
        return linear(x, self.weight, self.bias)


# ---------------------------------------------------------------------------------------------
# tensor-core MLP stages (csrc/mlp_tc.cu): Linear with the neighbouring BatchNorm / activation folded in
ACT_NONE, ACT_RELU, ACT_LEAKY_RELU = 0, 1, 2
_tc_scratch = {}


def lin_supported(K, M):
    return bool(lib().raw("dn4gl_lin_supported")(int(K), int(M)))


_tc_counter = {}   # device index -> persistent zeroed int32 counter shared by every captured launch on that device


def _tc_ws(device, nbytes):
    """(workspace, zeroed int32 counter) per (device, stream): the kernels consume the workspace before the next
    launch on the same stream starts, and leave the counter at zero.

    Under CUDA-graph capture the workspace comes from the graph's pool, and the counter is ONE persistent per-device
    tensor allocated outside any capture (captured launches of a device are serialised on the replaying stream, and
    each kernel leaves the counter at zero) -- not a fresh torch.zeros per call, which put ~25 fill kernels into every
    replayed train step."""
    if torch.cuda.is_current_stream_capturing():   # a CUDA graph owns its scratch (allocated from the graph's pool)
        cnt = _tc_counter.get(device.index)
        if cnt is None:                            # no eager call came first: allocate inside the capture (one fill node)
            cnt = torch.zeros(64, dtype=torch.int32, device=device)
        return torch.empty(max(nbytes, 1 << 20), dtype=torch.uint8, device=device), cnt
    if device.index not in _tc_counter:
        _tc_counter[device.index] = torch.zeros(64, dtype=torch.int32, device=device)
    key = (device.index, _stream())
    ent = _tc_scratch.get(key)
    if ent is None or ent[0].numel() < nbytes:
        ent = (torch.empty(max(nbytes, 1 << 20), dtype=torch.uint8, device=device),
               ent[1] if ent is not None else torch.zeros(64, dtype=torch.int32, device=device))
        _tc_scratch[key] = ent
    return ent


def lin_fwd(x, weight, bias=None, in_bn=None, in_act=ACT_NONE, in_slope=0.0, bn=None):
    """Y = act(bn_in(x)) W^T + b on the tensor cores (3xTF32).  bn = None, or a dict(gamma, beta, eps, momentum,
    running_mean, running_var, num_batches_tracked) -> also returns the BatchNorm record of Y's batch statistics
    (and updates the running buffers in place).  Returns (Y, record | None)."""
    require_cuda(x, "rows")
    x = _f32c(x)
    N, K = x.shape
    M = weight.size(0)
    L = lib()
    Y = torch.empty((N, M), dtype=torch.float32, device=x.device)
    rec = None
    wsb = L.size("dn4gl_lin_workspace_bytes", N, K, M)
    ws, counters = _tc_ws(x.device, wsb)
    g = b = rm = rv = nbt = None
    eps = mom = 0.0
    if bn is not None:
        rec = torch.empty(4 * M, dtype=torch.float32, device=x.device)
        g, b, eps, mom = bn.get("gamma"), bn.get("beta"), float(bn["eps"]), float(bn.get("momentum") or 0.0)
        rm, rv, nbt = bn.get("running_mean"), bn.get("running_var"), bn.get("num_batches_tracked")
    L.call("dn4gl_lin_fwd_f32", ptr(x), N, K, ptr(in_bn), int(in_act), float(in_slope), ptr(_f32c(weight)),
           ptr(None if bias is None else _f32c(bias)), M, ptr(Y), ptr(g), ptr(b), eps, mom, ptr(rec), ptr(rm), ptr(rv),
           ptr(nbt), ptr(ws), wsb, ptr(counters), _stream())
    return Y, rec


def lin_bwd(G, weight, X, Yout=None, bn=None, sums=None, g_masked=False, in_bn=None, in_act=ACT_NONE, in_slope=0.0,
            want_gx=True, want_dw=True, want_db=True, gseg=None, row2seg=None):
    """backward of one stage (see include/dn4gl.h): -> (GX | None, sums_prev | None, dW | None, db | None).
    The upstream gradient is G (N x M, may be None) + gseg[row2seg] (per-graph readout gradient, may be None)."""
    X = _f32c(X)
    require_cuda(X, "rows")
    G = None if G is None else _f32c(G)
    N, K = X.shape
    M = weight.size(0)
    dev = X.device
    L = lib()
    GX = torch.empty((N, K), dtype=torch.float32, device=dev) if want_gx else None
    sp = torch.empty(2 * K, dtype=torch.float32, device=dev) if (want_gx and in_bn is not None) else None
    dW = torch.empty((M, K), dtype=torch.float32, device=dev) if want_dw else None
    db = torch.empty(M, dtype=torch.float32, device=dev) if want_db else None
    wsb = L.size("dn4gl_lin_workspace_bytes", N, K, M)
    ws, counters = _tc_ws(dev, wsb)
    L.call("dn4gl_lin_bwd_f32", ptr(G), ptr(None if gseg is None else _f32c(gseg)), ptr(row2seg),
           ptr(None if Yout is None else _f32c(Yout)), N, M, ptr(bn), ptr(sums),
           1 if g_masked else 0, ptr(_f32c(weight)), K, ptr(X), ptr(in_bn), int(in_act), float(in_slope), ptr(GX), ptr(sp),
           ptr(dW), ptr(db), ptr(ws), wsb, ptr(counters), _stream())
    return GX, sp, dW, db


def bn_act(Y, rec, act=ACT_RELU, slope=0.0):
    """act(bn(Y)) elementwise (rec None = identity normalisation)."""
    require_cuda(Y, "rows")
    Y = _f32c(Y)
    out = torch.empty_like(Y)
    lib().call("dn4gl_bn_act_f32", ptr(Y), Y.size(0), Y.size(1), ptr(rec), int(act), float(slope), ptr(out), _stream())
    return out


def bn_act_pool(Y, rec, seg_ptr, mean=False, act=ACT_RELU, slope=0.0):
    """(act(bn(Y)), per-graph sum / mean of it) in one pass over contiguous row segments."""
    require_cuda(Y, "rows")
    Y = _f32c(Y)
    B = seg_ptr.numel() - 1
    out = torch.empty_like(Y)
    pooled = torch.empty((B, Y.size(1)), dtype=torch.float32, device=Y.device)
    lib().call("dn4gl_bn_act_pool_f32", ptr(Y), Y.size(0), Y.size(1), ptr(rec), int(act), float(slope), ptr(out),
               ptr(seg_ptr), B, 1 if mean else 0, ptr(pooled), _stream())
    return out, pooled


def segment_ids(seg_ptr, n_rows):
    """int32 row -> segment index (PyG's ``batch`` vector) for contiguous segments."""
    require_cuda(seg_ptr, "segment offsets")
    out = torch.empty(int(n_rows), dtype=torch.int32, device=seg_ptr.device)
    lib().call("dn4gl_segment_ids_i32", ptr(seg_ptr), seg_ptr.numel() - 1, int(n_rows), ptr(out), _stream())
    return out


def bn_bwd_sums(G, Y, rec, act=ACT_RELU, slope=0.0, gseg=None, row2seg=None):
    """{sum gm, sum gm * xhat} (2*M) with gm = (G + gseg[row2seg]) * act'(bn(Y))."""
    Y = _f32c(Y)
    G = None if G is None else _f32c(G)
    N, M = Y.shape
    L = lib()
    sums = torch.empty(2 * M, dtype=torch.float32, device=Y.device)
    wsb = L.size("dn4gl_bn_bwd_sums_workspace_bytes", N, M)
    ws, counters = _tc_ws(Y.device, wsb)
    L.call("dn4gl_bn_bwd_sums_f32", ptr(G), ptr(None if gseg is None else _f32c(gseg)), ptr(row2seg), ptr(Y), N, M,
           ptr(rec), int(act), float(slope), ptr(sums), ptr(ws), wsb, ptr(counters), _stream())
    return sums


def _bn_dict(bn):
    return dict(gamma=bn.weight, beta=bn.bias, eps=bn.eps, momentum=bn.momentum, running_mean=bn.running_mean,
                running_var=bn.running_var, num_batches_tracked=bn.num_batches_tracked)


def dot(a, b, out=None, counter_slot=0):
    """sum(a * b) as a 1-element tensor, fixed-order.  counter_slot: which of the device's ticket counters the launch
    uses (a launch that may run next to the stage kernels must not share theirs)."""
    a, b = _f32c(a), _f32c(b)
    L = lib()
    if out is None:
        out = torch.empty(1, dtype=torch.float32, device=a.device)
    if a.numel() == 0:      # an empty CUDA tensor has no storage (data_ptr() == 0), and its sum is 0: nothing to launch
        return out.zero_()
    wsb = L.size("dn4gl_dot_workspace_bytes", a.numel())
    ws, counter = _tc_ws(a.device, wsb)
    L.call("dn4gl_dot_f32", ptr(a), ptr(b), a.numel(), ptr(out), ptr(ws), wsb, counter.data_ptr() + 4 * counter_slot, _stream())
    return out


_side_streams = {}
SIDE_STREAM_DOT = os.environ.get("DN4GL_SIDE_DOT", "1") == "1"


def _side_stream(device):
    s = _side_streams.get(device.index)
    if s is None:
        s = _side_streams[device.index] = torch.cuda.Stream(device=device)
    return s


def dot_beside(a, b):
    """dot(a, b) launched on a second stream, forked from and joined back into the current one by the caller:
    ``out, join = dot_beside(a, b); <launch independent work on the current stream>; join()``.  The bandwidth-bound
    reduction then runs next to a latency-bound kernel (the backward aggregation) instead of after it; inside a CUDA-graph
    capture the two become parallel branches."""
    a, b = _f32c(a), _f32c(b)
    out = torch.empty(1, dtype=torch.float32, device=a.device)     # allocated on the current stream, which consumes it
    cur, side = torch.cuda.current_stream(a.device), _side_stream(a.device)
    side.wait_stream(cur)
    with torch.cuda.stream(side):
        dot(a, b, out=out, counter_slot=32)
    return out, lambda: cur.wait_stream(side)


class _GinLayer(torch.autograd.Function):
    """one GIN layer as ONE autograd node (gconv.py:210-213 + :190-196):

        z = (1 + eps) x + sum_{j->i} x_j          (skipped when csr_in is None: layer 0 applies the MLP to x itself)
        h = ReLU(BN2(Linear2(ReLU(BN1(Linear1(z))))))      training-mode batch statistics
        pooled = global_add_pool / global_mean_pool (h)    (when seg_ptr is given)

    Forward: aggregation, two tensor-core stages (+ their statistics merges), one elementwise + readout pass.  Backward:
    the readout gradient is added row-wise inside the stage prologues (never materialised), the BatchNorm sums of the
    inner stage come out of the outer stage's epilogue; eps is read on the device, d eps = sum(g_z * x)."""

    @staticmethod
    def forward(ctx, x, eps, W1, b1, g1, be1, W2, b2, g2, be2, bn1, bn2, csr_in, csr_out, seg_ptr, row2seg, mean):
        ctx.set_materialize_grads(False)
        x = _f32c(x)
        z = _spmm(csr_in, x, csr_in.n_rows, 1.0, eps) if csr_in is not None else x
        y1, rec1 = lin_fwd(z, W1, b1, bn=bn1)
        y2, rec2 = lin_fwd(y1, W2, b2, in_bn=rec1, in_act=ACT_RELU, bn=bn2)
        if seg_ptr is not None:
            h, pooled = bn_act_pool(y2, rec2, seg_ptr, mean, ACT_RELU)
        else:
            h, pooled = bn_act(y2, rec2, ACT_RELU), None
        ctx.save_for_backward(x, eps, z, y1, y2, rec1, rec2, W1, W2)
        ctx.csr_out, ctx.seg_ptr, ctx.row2seg, ctx.mean = csr_out, seg_ptr, row2seg, mean
        return h, pooled

    @staticmethod
    def backward(ctx, gh, gpooled):
        x, eps, z, y1, y2, rec1, rec2, W1, W2 = ctx.saved_tensors
        D1, D2 = W1.size(0), W2.size(0)
        gh = None if gh is None else _f32c(gh)
        gseg = row2seg = None
        if gpooled is not None:
            gseg, row2seg = _f32c(gpooled), ctx.row2seg
            if ctx.mean:
                cnt = (ctx.seg_ptr[1:] - ctx.seg_ptr[:-1]).clamp_min(1).to(gseg.dtype).unsqueeze(1)
                gseg = gseg / cnt
        if gh is None and gseg is None:
            gh = torch.zeros_like(y2)
        sums2 = bn_bwd_sums(gh, y2, rec2, ACT_RELU, gseg=gseg, row2seg=row2seg)
        ga1, sums1, dW2, db2 = lin_bwd(gh, W2, y1, Yout=y2, bn=rec2, sums=sums2, g_masked=False, in_bn=rec1,
                                       in_act=ACT_RELU, gseg=gseg, row2seg=row2seg)
        has_agg = ctx.csr_out is not None
        need_eps = has_agg and eps is not None and ctx.needs_input_grad[1]
        need_z = ctx.needs_input_grad[0] or need_eps
        gz, _, dW1, db1 = lin_bwd(ga1, W1, z, Yout=y1, bn=rec1, sums=sums1, g_masked=True, want_gx=need_z)
        gx = geps = None
        join = None
        if need_eps and SIDE_STREAM_DOT and ctx.needs_input_grad[0]:
            geps, join = dot_beside(gz, x)          # d eps next to the backward aggregation (both only read gz)
            geps = geps.view_as(eps)
        if ctx.needs_input_grad[0]:
            gx = _spmm(ctx.csr_out, gz, x.size(0), 1.0, eps) if has_agg else gz
        if join is not None:
            join()
        elif need_eps:
            geps = dot(gz, x).view_as(eps)
        return (gx, geps, dW1, db1, sums1[D1:], sums1[:D1], dW2, db2, sums2[D2:], sums2[:D2],
                None, None, None, None, None, None, None)


class _BnActTrain(torch.autograd.Function):
    """act(BatchNorm1d(y)) in training mode for widths above the fused stages' (<= 128): batch statistics, running-statistics
    update and both backward reductions by the fixed-order kernels (dn4gl_bn_stats_f32, dn4gl_bn_bwd_sums_f32,
    dn4gl_bn_bwd_apply_f32) instead of ATen's fp32 batch-norm reductions."""

    @staticmethod
    def forward(ctx, y, gamma, beta, bn, act):
        require_cuda(y, "rows")
        y = _f32c(y)
        N, M = y.shape
        L = lib()
        rec = torch.empty(4 * M, dtype=torch.float32, device=y.device)
        wsb = L.size("dn4gl_bn_stats_workspace_bytes", N, M)
        ws, _ = _tc_ws(y.device, wsb)
        L.call("dn4gl_bn_stats_f32", ptr(y), N, M, ptr(gamma), ptr(beta), float(bn["eps"]), float(bn.get("momentum") or 0.0),
               ptr(bn.get("running_mean")), ptr(bn.get("running_var")), ptr(bn.get("num_batches_tracked")), ptr(rec), ptr(ws), wsb,
               _stream())
        out = bn_act(y, rec, act)
        ctx.save_for_backward(y, rec)
        ctx.act = act
        return out

    @staticmethod
    def backward(ctx, g):
        y, rec = ctx.saved_tensors
        g = _f32c(g)
        N, M = y.shape
        sums = bn_bwd_sums(g, y, rec, ctx.act)
        gx = torch.empty_like(y)
        lib().call("dn4gl_bn_bwd_apply_f32", ptr(g), ptr(y), N, M, ptr(rec), ptr(sums), int(ctx.act), 0.0, ptr(gx), _stream())
        return gx, sums[M:], sums[:M], None, None


def gin_mlp_wide_ok(seq):
    """True for the reference's GIN MLP (Linear, BatchNorm1d, ReLU, Linear, BatchNorm1d, ReLU) in training mode at widths the
    fused stages do not take but the stand-alone BatchNorm kernels do (<= 128 columns per BatchNorm)."""
    import torch.nn as nn
    if not (isinstance(seq, nn.Sequential) and len(seq) == 6):
        return False
    l1, n1, a1, l2, n2, a2 = seq
    if not (isinstance(l1, nn.Linear) and isinstance(l2, nn.Linear) and isinstance(n1, nn.BatchNorm1d)
            and isinstance(n2, nn.BatchNorm1d) and isinstance(a1, nn.ReLU) and isinstance(a2, nn.ReLU)):
        return False
    for n in (n1, n2):
        if not (n.training and n.affine and n.track_running_stats and n.momentum is not None and n.num_features <= 128):
            return False
    return True


def gin_mlp_wide(seq, z):
    """the GIN MLP `seq` on z (N >= 1 rows): Linear through ops.linear (tensor-core GEMM), BatchNorm + ReLU through the
    stand-alone fixed-order BatchNorm kernels; gin_mlp_wide_ok(seq) must hold."""
    l1, n1, _, l2, n2, _ = seq
    for lin, bn in ((l1, n1), (l2, n2)):
        z = linear(z, lin.weight, lin.bias)
        z = _BnActTrain.apply(z, bn.weight, bn.bias, _bn_dict(bn), ACT_RELU)
    return z


def apply_gin_mlp(seq, z):
    """the GIN MLP on CUDA rows by the best available path: fused tensor-core stages (widths <= 64), stand-alone
    BatchNorm kernels + tensor-core GEMM (<= 128), else the module as it is."""
    if z.is_cuda and z.size(0) > 0:
        if gin_mlp_fusable(seq):
            return gin_mlp(seq, z)
        if gin_mlp_wide_ok(seq):
            return gin_mlp_wide(seq, z)
    return seq(z)


def gin_layer(seq, x, eps=None, csr_in=None, csr_out=None, seg_ptr=None, row2seg=None, mean=False):
    """fused GIN layer -> (h, pooled | None); gin_mlp_fusable(seq) must hold.  csr_in None: no aggregation (layer 0)."""
    l1, n1, _, l2, n2, _ = seq
    return _GinLayer.apply(x, eps, l1.weight, l1.bias, n1.weight, n1.bias, l2.weight, l2.bias, n2.weight, n2.bias,
                           _bn_dict(n1), _bn_dict(n2), csr_in, csr_out, seg_ptr, row2seg, mean)


def gin_conv(seq, x, eps, csr_in, csr_out):
    """fused GINConv (aggregation + MLP)."""
    return gin_layer(seq, x, eps, csr_in, csr_out)[0]


def gin_mlp(seq, z):
    """the GIN MLP `seq` applied to z through the fused tensor-core stages."""
    return gin_layer(seq, z)[0]


class _Mlp2(torch.autograd.Function):
    """``Linear, act, Linear`` (rgin.py:52, dmpnn.py:47,55 with the default num_mlp_layers=2, no BatchNorm) as two
    tensor-core stages: the activation is the second stage's prologue, its derivative the backward epilogue."""

    @staticmethod
    def forward(ctx, x, W1, b1, W2, b2, act, slope):
        x = _f32c(x)
        y1, _ = lin_fwd(x, W1, b1)
        y2, _ = lin_fwd(y1, W2, b2, in_act=act, in_slope=slope)
        ctx.save_for_backward(x, y1, W1, W2)
        ctx.act, ctx.slope, ctx.has_b = act, slope, (b1 is not None, b2 is not None)
        return y2

    @staticmethod
    def backward(ctx, g):
        x, y1, W1, W2 = ctx.saved_tensors
        ga1, _, dW2, db2 = lin_bwd(_f32c(g), W2, y1, in_act=ctx.act, in_slope=ctx.slope, want_db=ctx.has_b[1])
        gx, _, dW1, db1 = lin_bwd(ga1, W1, x, want_gx=ctx.needs_input_grad[0], want_db=ctx.has_b[0])
        return gx, dW1, db1, dW2, db2, None, None


def _act_code(m):
    import torch.nn as nn
    if isinstance(m, nn.ReLU):
        return ACT_RELU, 0.0
    if isinstance(m, nn.LeakyReLU):
        return ACT_LEAKY_RELU, float(m.negative_slope)
    if type(m).__name__ == "Identity":
        return ACT_NONE, 0.0
    return None


# `Linear, act, Linear` of the counting models on the tensor cores.  Round 1 kept this opt-in: the truncating fp32
# accumulation of the tensor core is a BIASED error that the counting models (12 such GEMMs per forward, 512-node sum
# aggregations, no normalisation) add up coherently -- 2-4e-5 on the DMPNN "large" loss, above the 1e-5 bar.  Round 2's stage
# kernels issue the A_lo products first and spread the A_hi k-steps over four accumulators added in round-to-nearest
# (csrc/mlp_pipe.cu): 8.5e-6 on that loss, every other recorded quantity <= 5.4e-6 (profiles/r2n_parity_errors_mlp2tc.json),
# so the tensor-core path is the default; DN4GL_MLP2_TC=0 restores the library GEMMs.
MLP2_TENSOR_CORES = os.environ.get("DN4GL_MLP2_TC", "1") == "1"


def mlp2_fusable(seq, force=False):
    """True for ``Sequential(Linear, act, Linear)`` with act in {ReLU, LeakyReLU, Identity} and supported widths
    (and the opt-in switch above, unless force)."""
    import torch.nn as nn
    if not (MLP2_TENSOR_CORES or force):
        return False
    if not (isinstance(seq, nn.Sequential) and len(seq) == 3):
        return False
    l1, a, l2 = seq
    if not (isinstance(l1, nn.Linear) and isinstance(l2, nn.Linear) and _act_code(a) is not None):
        return False
    return lin_supported(l1.in_features, l1.out_features) and lin_supported(l2.in_features, l2.out_features)


def mlp2(seq, x):
    """apply ``Sequential(Linear, act, Linear)`` through the tensor-core stages (mlp2_fusable(seq) must hold)."""
    l1, a, l2 = seq
    act, slope = _act_code(a)
    lead = x.shape[:-1]
    y = _Mlp2.apply(x.reshape(-1, x.size(-1)), l1.weight, l1.bias, l2.weight, l2.bias, act, slope)
    return y.view(lead + (l2.out_features,))


def gin_mlp_fusable(seq):
    """True if `seq` is the reference's GIN MLP (Linear, BatchNorm1d, ReLU, Linear, BatchNorm1d, ReLU) in a state
    the fused stages reproduce: training-mode batch statistics with a fixed momentum, affine BN, supported widths."""
    import torch.nn as nn
    if not (isinstance(seq, nn.Sequential) and len(seq) == 6):
        return False
    l1, n1, a1, l2, n2, a2 = seq
    if not (isinstance(l1, nn.Linear) and isinstance(l2, nn.Linear) and isinstance(n1, nn.BatchNorm1d)
            and isinstance(n2, nn.BatchNorm1d) and isinstance(a1, nn.ReLU) and isinstance(a2, nn.ReLU)):
        return False
    for n in (n1, n2):
        if not (n.training and n.affine and n.track_running_stats and n.momentum is not None):
            return False
    if l1.bias is None or l2.bias is None:
        return False
    return lin_supported(l1.in_features, l1.out_features) and lin_supported(l2.in_features, l2.out_features)


GATHER_MAX_COLUMNS = 8


def gather_segments(idx, ptr_in, ptr_out, cols_in, cols_out, rebase=None, rebase_in=None, rebase_out=None):
    """one level of a mini-batch assembled from a resident data set (dn4gl_gather_segments, one launch): segment
    ``idx[k]`` of every column of ``cols_in`` (items ``ptr_in[idx[k]] ..``) lands at item ``ptr_out[k]`` of the matching
    column of ``cols_out``; columns flagged in ``rebase`` (int32) also get ``rebase_out[k] - rebase_in[idx[k]]`` added.
    idx / ptr_in / ptr_out / rebase_*: int32 device tensors; columns: contiguous device tensors of 4- or 8-byte items
    whose leading dimension is the item count.  The caller checks that idx lies in the data set (datasets.py does)."""
    import ctypes
    import math
    n = len(cols_in)
    if n != len(cols_out) or not 1 <= n <= GATHER_MAX_COLUMNS:
        raise ValueError("gather_segments: 1..%d input columns and as many outputs" % GATHER_MAX_COLUMNS)
    words = []
    for a, b in zip(cols_in, cols_out):
        if (not (a.is_contiguous() and b.is_contiguous()) or a.dtype != b.dtype or a.shape[1:] != b.shape[1:]
                or a.element_size() not in (4, 8)):
            raise ValueError("gather_segments: columns must be contiguous, of 4- or 8-byte items, with matching dtype "
                             "and item shape")
        words.append(math.prod(a.shape[1:]) * a.element_size() // 4)
    if cols_out[0].numel() == 0:        # the selected segments hold no items on this level
        return
    reb = [int(bool(r)) for r in (rebase or [0] * n)]
    lib().call("dn4gl_gather_segments", int(idx.numel()), ptr(idx), ptr(ptr_in), int(ptr_in.numel()) - 1, ptr(ptr_out),
               ptr(rebase_in), ptr(rebase_out), n, _ptr_array(cols_in), _ptr_array(cols_out),
               (ctypes.c_int32 * n)(*words), (ctypes.c_int32 * n)(*reb), _stream())


# ---- evaluation records and their fixed-order reduction (csrc/eval.cu) ------------------------------------------------
EVAL_REDUCE_MAX_COLUMNS = 8


def _eval_tensor(what, t, dtype, ndim, device=None):
    """host-side check of one argument of the evaluation kernels (ValueError before any launch)."""
    if not isinstance(t, torch.Tensor):
        raise ValueError("%s must be a tensor" % what)
    if t.dtype != dtype:
        raise ValueError("%s must be %s, got %s" % (what, dtype, t.dtype))
    if t.dim() != ndim or not t.is_contiguous():
        raise ValueError("%s must be a contiguous %d-D tensor, got shape %s" % (what, ndim, tuple(t.shape)))
    if not t.is_cuda:
        raise ValueError("%s must live on a CUDA device (there is no CPU path)" % what)
    if device is not None and t.device != device:
        raise ValueError("%s is on %s, expected %s" % (what, t.device, device))


def _eval_span(what, B, pos0, n):
    """-> pos0 as an int, checked: the batch's records pos0 .. pos0 + B - 1 lie inside the n-row outputs."""
    import operator
    try:
        pos0 = operator.index(pos0)
    except TypeError:
        raise ValueError("%s: pos0 must be an integer, got %r" % (what, pos0)) from None
    if not (0 <= pos0 and pos0 + B <= n):
        raise ValueError("%s: records %d .. %d do not fit the %d-row outputs" % (what, pos0, pos0 + B - 1, n))
    if B > 2 ** 31 - 1:
        raise ValueError("%s: more than 2^31 - 1 rows in one batch" % what)
    return pos0


def eval_class_rows(logp, y, pos0, pred, nll, correct):
    """per-graph records of a classification batch (dn4gl_eval_class_rows_f32, one launch): for row b of the (B, C)
    log-probabilities ``logp`` and the int64 targets ``y``, position ``pos0 + b`` of the split-sized outputs gets
    ``pred`` (int32 arg-max, lowest index on ties, as ``out.max(1)[1]``), ``nll`` (-logp[b, y[b]]) and ``correct``
    (1.0 / 0.0).  A target outside [0, C) gives nll 0 and is never correct; a row holding a NaN gives nll NaN and is
    never correct."""
    _eval_tensor("eval_class_rows: logp", logp, torch.float32, 2)
    dev = logp.device
    B, C = logp.shape
    if C < 1:
        raise ValueError("eval_class_rows: logp needs at least one class column")
    _eval_tensor("eval_class_rows: y", y, torch.int64, 1, dev)
    if y.numel() != B:
        raise ValueError("eval_class_rows: %d targets for %d rows" % (y.numel(), B))
    _eval_tensor("eval_class_rows: pred", pred, torch.int32, 1, dev)
    _eval_tensor("eval_class_rows: nll", nll, torch.float32, 1, dev)
    _eval_tensor("eval_class_rows: correct", correct, torch.float32, 1, dev)
    n = pred.numel()
    if nll.numel() != n or correct.numel() != n:
        raise ValueError("eval_class_rows: pred, nll and correct must have the same length")
    pos0 = _eval_span("eval_class_rows", B, pos0, n)
    if B == 0:
        return
    bind_device(dev)
    lib().call("dn4gl_eval_class_rows_f32", ptr(logp), ptr(y), B, C, pos0, ptr(pred), ptr(nll), ptr(correct), _stream())


def eval_count_rows(pred_c, counts, pos0, pred, err):
    """per-sample records of a counting batch (dn4gl_eval_count_rows_f32, one launch): for sample b with prediction
    ``pred_c`` (B or B x 1, float32) and int64 ``counts``, position ``pos0 + b`` of the split-sized outputs gets ``pred``
    (pred_c itself) and the row ``err`` (n x 3) = |r - t|, (r - t)^2, smooth-L1(r - t) with r = relu(pred_c),
    t = float(count): the per-element terms of the MAE, MSE and SMSE criteria (losses.eval_criterion)."""
    if isinstance(pred_c, torch.Tensor) and pred_c.dim() == 2 and pred_c.size(1) == 1:
        pred_c = pred_c.view(-1)
    _eval_tensor("eval_count_rows: pred_c", pred_c, torch.float32, 1)
    dev = pred_c.device
    B = pred_c.numel()
    _eval_tensor("eval_count_rows: counts", counts, torch.int64, 1, dev)
    if counts.numel() != B:
        raise ValueError("eval_count_rows: %d counts for %d predictions" % (counts.numel(), B))
    _eval_tensor("eval_count_rows: pred", pred, torch.float32, 1, dev)
    _eval_tensor("eval_count_rows: err", err, torch.float32, 2, dev)
    n = pred.numel()
    if tuple(err.shape) != (n, 3):
        raise ValueError("eval_count_rows: err must be (%d, 3), got %s" % (n, tuple(err.shape)))
    pos0 = _eval_span("eval_count_rows", B, pos0, n)
    if B == 0:
        return
    bind_device(dev)
    lib().call("dn4gl_eval_count_rows_f32", ptr(pred_c), ptr(counts), B, pos0, ptr(pred), ptr(err), _stream())


def eval_reduce(v, out=None):
    """float64 sums of the columns of ``v`` (n, or n x k with 1 <= k <= 8, float32) in an order fixed by n alone
    (dn4gl_eval_reduce_f32, one launch; n == 0: zeros).  out: a float64 tensor of k elements to write (default: new)."""
    if isinstance(v, torch.Tensor) and v.dim() == 1:
        v = v.view(-1, 1)
    _eval_tensor("eval_reduce: v", v, torch.float32, 2)
    dev = v.device
    n, k = v.shape
    if not 1 <= k <= EVAL_REDUCE_MAX_COLUMNS:
        raise ValueError("eval_reduce: 1..%d columns, got %d" % (EVAL_REDUCE_MAX_COLUMNS, k))
    if out is None:
        out = torch.empty(k, dtype=torch.float64, device=dev)
    _eval_tensor("eval_reduce: out", out, torch.float64, 1, dev)
    if out.numel() != k:
        raise ValueError("eval_reduce: out must hold %d values" % k)
    bind_device(dev)
    L = lib()
    wsb = L.size("dn4gl_eval_reduce_workspace_bytes", n, k)
    ws, counter = _tc_ws(dev, wsb)
    L.call("dn4gl_eval_reduce_f32", ptr(v) if n else None, n, k, ptr(out), ptr(ws), wsb, ptr(counter), _stream())
    return out


# ---- the matching objective of the counting models (csrc/match.cu) -----------------------------------------------------
MATCH_CRITERIA = {"MAE": 0, "MSE": 1, "SMSE": 2}       # losses._CRITERIA: F.l1_loss, F.mse_loss, F.smooth_l1_loss


def _i32_vector(what, t, n=None, device=None):
    _eval_tensor(what, t, torch.int32, 1, device)
    if n is not None and t.numel() != n:
        raise ValueError("%s must hold %d values, got %d" % (what, n, t.numel()))


def subiso_append_dummy(val_ptr, values, rows, g_node_ptr, out_ptr, out_total):
    """the dummy column of a packed subisomorphism batch (dn4gl_subiso_append_dummy, one launch): row s of sample b
    becomes its np_b ids followed by n_b = g_node_ptr[b + 1] - g_node_ptr[b] (the graph's node count BEFORE
    augmentation), written at ``out_ptr[b] + s * (np_b + 1)``.  All arguments int32 device tensors; out_ptr (B + 1) holds
    the output offsets ``val_ptr[b] + sum_{b' < b} rows[b']`` and out_total = out_ptr[B], both computed by the caller on
    the host (``matching.dummy_column_offsets``).  -> int32 (out_total,)."""
    _i32_vector("subiso_append_dummy: val_ptr", val_ptr)
    dev = val_ptr.device
    B = val_ptr.numel() - 1
    if B < 0:
        raise ValueError("subiso_append_dummy: val_ptr needs B + 1 >= 1 offsets")
    _i32_vector("subiso_append_dummy: values", values, None, dev)
    _i32_vector("subiso_append_dummy: rows", rows, B, dev)
    _i32_vector("subiso_append_dummy: g_node_ptr", g_node_ptr, B + 1, dev)
    _i32_vector("subiso_append_dummy: out_ptr", out_ptr, B + 1, dev)
    out_total = int(out_total)
    if not values.numel() <= out_total <= 2 ** 31 - 1:
        raise ValueError("subiso_append_dummy: out_total %d is outside [%d, 2^31 - 1]" % (out_total, values.numel()))
    out = torch.empty(out_total, dtype=torch.int32, device=dev)
    if B == 0 or out_total == 0:
        return out
    bind_device(dev)
    lib().call("dn4gl_subiso_append_dummy", B, ptr(val_ptr), ptr(values), ptr(rows), ptr(g_node_ptr), ptr(out_ptr),
               out_total, ptr(out), _stream())
    return out


def _match_kind(what, pred, mask, weights, seg_ptr, B, dev):
    """checked (pred, mask, weights, seg_ptr, L) of one kind of the match terms, or None when the kind is left out."""
    if pred is None or weights is None:
        return None
    if isinstance(pred, torch.Tensor) and isinstance(mask, torch.Tensor):
        pred, mask = pred.contiguous(), mask.contiguous()
    _eval_tensor(what + " prediction", pred, torch.float32, 2, dev)
    if pred.size(0) != B:
        raise ValueError("match_loss: %s prediction has %d rows for %d graphs" % (what, pred.size(0), B))
    L = pred.size(1)
    _eval_tensor(what + " mask", mask, torch.bool, 2, dev)
    if tuple(mask.shape) != (B, L):
        raise ValueError("match_loss: %s mask must be (%d, %d), got %s" % (what, B, L, tuple(mask.shape)))
    _i32_vector("match_loss: %s seg_ptr" % what, seg_ptr, B + 1, dev)
    if not isinstance(weights, torch.Tensor) or weights.dtype not in (torch.int32, torch.int64):
        raise ValueError("match_loss: %s weights must be an int32 or int64 tensor" % what)
    weights = weights.to(torch.int32) if weights.dtype == torch.int64 else weights
    _i32_vector("match_loss: %s weights" % what, weights, None, dev)
    return pred, mask, weights, seg_ptr, L


def _kind_args(k):
    return (None, None, None, None, 0) if k is None else (ptr(k[0]), ptr(k[1]), ptr(k[2]), ptr(k[3]), k[4])


class _MatchLoss(torch.autograd.Function):
    """match_loss_w * (loss_v + loss_e) + match_reg_w * (reg_v + reg_e) as one kernel each way (csrc/match.cu)."""

    @staticmethod
    def forward(ctx, pred_c, pred_v, pred_e, kv, ke, crit, scalars):
        dev = pred_c.device
        B = pred_c.size(0)
        L = lib()
        out = torch.empty((), dtype=torch.float32, device=dev)
        wsb = L.size("dn4gl_match_loss_workspace_bytes", B)
        ws, counter = _tc_ws(dev, wsb)
        L.call("dn4gl_match_loss_f32", B, ptr(pred_c), *_kind_args(kv), *_kind_args(ke), crit, *(ptr(s) for s in scalars),
               ptr(out), ptr(ws), wsb, ptr(counter), _stream())
        ctx.kv, ctx.ke, ctx.crit, ctx.scalars, ctx.B = kv, ke, crit, scalars, B
        ctx.shape_c = pred_c.shape
        ctx.pred_c = pred_c
        return out

    @staticmethod
    def backward(ctx, g):
        g = _f32c(g).reshape(1)
        kv, ke = ctx.kv, ctx.ke
        gc = torch.empty(ctx.shape_c, dtype=torch.float32, device=g.device)
        gv = None if kv is None else torch.empty_like(kv[0])
        ge = None if ke is None else torch.empty_like(ke[0])
        lib().call("dn4gl_match_loss_bwd_f32", ctx.B, ptr(g), ptr(ctx.pred_c), *_kind_args(kv), *_kind_args(ke), ctx.crit,
                   *(ptr(s) for s in ctx.scalars), ptr(gv), ptr(ge), ptr(gc), _stream())
        return gc, gv, ge, None, None, None, None


def match_loss(pred_c, pred_v, mask_v, node_weights, node_ptr, pred_e, mask_e, edge_weights, edge_ptr, bp_loss, neg_slp,
               match_loss_w, match_reg_w):
    """the match terms of the counting models' bp_loss (losses.counting_bp_loss with the identity refine_*_weights) as a
    0-d float32 tensor with a gradient for pred_c (B, 1), pred_v and pred_e: dn4gl_match_loss_f32 / _bwd_f32, one launch
    each way.  pred_v / pred_e: the model's left-padded (B, L) predictions with its own g_v_mask / g_e_mask; node_weights /
    edge_weights: the FLAT int32 (or int64) weights of the augmented graph batch with their row offsets node_ptr /
    edge_ptr (left-padded on the fly, no (B, L) target is built).  A kind whose prediction or weights are None is left
    out.  neg_slp, match_loss_w, match_reg_w: float32 device scalars read by the kernels (a captured step follows
    changes to them)."""
    if bp_loss not in MATCH_CRITERIA:
        raise NotImplementedError(bp_loss)
    if isinstance(pred_c, torch.Tensor):
        pred_c = pred_c.contiguous()
    if isinstance(pred_c, torch.Tensor) and pred_c.dim() == 2 and pred_c.size(1) == 1:
        _eval_tensor("match_loss: pred_c", pred_c, torch.float32, 2)
    else:
        _eval_tensor("match_loss: pred_c", pred_c, torch.float32, 1)
    dev = pred_c.device
    B = pred_c.size(0)
    for what, s in (("neg_slp", neg_slp), ("match_loss_w", match_loss_w), ("match_reg_w", match_reg_w)):
        _eval_tensor("match_loss: " + what, s, torch.float32, 0, dev)
    kv = _match_kind("node", pred_v, mask_v, node_weights, node_ptr, B, dev)
    ke = _match_kind("edge", pred_e, mask_e, edge_weights, edge_ptr, B, dev)
    bind_device(dev)
    return _MatchLoss.apply(pred_c, None if kv is None else kv[0], None if ke is None else ke[0], kv, ke,
                            MATCH_CRITERIA[bp_loss], (neg_slp, match_loss_w, match_reg_w))
