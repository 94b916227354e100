"""Kernel-level tests of the counting models' per-edge kernels (dmp.cu K4 / K5, comp.cu), the label-filter gate,
gather_rows and the fixed-order dot product, each against a float64 restatement of the definition in its header comment.

Measures, per element (u = 2^-24, one fp32 rounding):
  - elementwise kernels: |out - ref| <= c u |ref| (c = the roundings on the path), or c u sum|terms| where the value is
    a short sum of terms that may cancel; gathers bit-exact;
  - reductions: |out - ref| <= n u sum|terms|, n = the number of terms;
  - paths that state a summation order (light rows of the node aggregation, the [P|Q] backward, the h-gradient of the
    composition) bit-exact against a sequential fp32 loop in that order;
  - every kernel run twice: bitwise-equal outputs.

The batches hold isolated nodes, self-loops, multi-edges, graphs without edges, in-degrees at the tails of the 4- and
2-edge unrolls (0, 1, 2, 3, 5), the last light row (64 in-edges) and the first heavy one (65), and a hub batch with more
heavy rows than the heavy kernel's grid.  The tests without the gpu mark tie the references to oracle.models."""
import functools

import numpy as np
import pytest
import torch

from conftest import record_error
from helpers import nasty_sub_batch, rel_err

U = 2.0 ** -24
HEAVY = 64          # graph.HEAVY_THRESHOLD: rows with more in-edges go to the CTA-per-row kernel
SUB, MULT = 0, 1    # ops.COMP_SUB, ops.COMP_MULT


# ---------------------------------------------------------------------------------------------------------------------
# batches (flat dicts in the BatchedGraph.from_batch layout)
def _parts_of(b):
    """[(n, src, dst)] per graph, node ids local to the graph."""
    npt, ept = b["node_ptr"], b["edge_ptr"]
    return [(int(npt[i + 1] - npt[i]), b["src"][ept[i]:ept[i + 1]] - npt[i], b["dst"][ept[i]:ept[i + 1]] - npt[i])
            for i in range(len(npt) - 1)]


def _assemble(parts, rng, n_labels=4):
    node_ptr, edge_ptr, src, dst = [0], [0], [np.zeros(0, np.int64)], [np.zeros(0, np.int64)]
    for n, s, d in parts:
        src.append(np.asarray(s, np.int64) + node_ptr[-1])
        dst.append(np.asarray(d, np.int64) + node_ptr[-1])
        node_ptr.append(node_ptr[-1] + n)
        edge_ptr.append(edge_ptr[-1] + len(s))
    N, E = node_ptr[-1], edge_ptr[-1]
    return dict(num_graphs=len(parts), node_ptr=np.asarray(node_ptr, np.int32), edge_ptr=np.asarray(edge_ptr, np.int32),
                src=np.concatenate(src).astype(np.int32), dst=np.concatenate(dst).astype(np.int32),
                vlabel=rng.integers(0, n_labels, N).astype(np.int32), elabel=rng.integers(0, n_labels, E).astype(np.int32))


def _with_in_degrees(rng, degrees, extra):
    """one graph whose first len(degrees) nodes have these in-degrees, sources drawn from all its nodes (self-loops and
    multi-edges included), edge ids shuffled so that a node's in-list is not contiguous in edge-id order."""
    n = len(degrees) + extra
    dst = np.repeat(np.arange(len(degrees)), degrees)
    src = rng.integers(0, n, dst.size)
    perm = rng.permutation(dst.size)
    return n, src[perm], dst[perm]


def _odd_sizes(parts):
    """append tiny graphs until N and E are odd: N is then no multiple of any kernel's rows per CTA, and E * D / 4 no
    multiple of the 256-thread block for every D this file uses."""
    if sum(len(p[1]) for p in parts) % 2 == 0:
        parts.append((2, [0], [1]))
    if sum(p[0] for p in parts) % 2 == 0:
        parts.append((1, [], []))
    return parts


@functools.lru_cache(None)
def _mixed_batch():
    rng = np.random.default_rng(11)
    parts = _parts_of(nasty_sub_batch(rng, 48, 12, 4))
    parts.append(_with_in_degrees(rng, [0, 1, 2, 3, 5, HEAVY, HEAVY + 1, 4, 6, 7, 9, 0, 1], extra=6))
    parts.append((5, [], []))                      # a graph without edges
    parts.append((3, [0, 0, 0], [0, 0, 0]))        # a node with three self-loops next to two isolated nodes
    return _assemble(_odd_sizes(parts), rng)


@functools.lru_cache(None)
def _hub_batch(n_heavy):
    """n_heavy rows with 65..88 in-edges (hubs of graphs of up to 97 hubs and as many leaves) + small graphs."""
    rng = np.random.default_rng(5)
    parts, left = [], n_heavy
    while left > 0:
        k = min(left, 97)
        parts.append(_with_in_degrees(rng, HEAVY + 1 + rng.integers(0, 24, k), extra=k))
        left -= k
    parts += _parts_of(nasty_sub_batch(rng, 16, 12, 4))
    return _assemble(_odd_sizes(parts), rng)


def _with_rev(b, rev):
    """the batch with (rev=True) a seeded random mix of reversed edges in edata["is_reversed"], or without the key."""
    b = dict(b)
    if rev:
        b["e_is_reversed"] = np.random.default_rng(int(b["src"].size)).random(b["src"].size) < 0.5
    return b


def _n_sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _batch(name, rev):
    return _with_rev(_mixed_batch() if name == "mixed" else _hub_batch(4 * _n_sms() + 37), rev)


def _rev(b):
    r = b.get("e_is_reversed")
    return np.zeros(b["src"].size, bool) if r is None else np.asarray(r, bool)


# ---------------------------------------------------------------------------------------------------------------------
# float64 references: (value, magnitude) where the magnitude is sum|terms| per element, the scale of the error bound
def _seg(n, idx, rows):
    """out[k] = sum of rows[i] with idx[i] == k, float64."""
    rows = torch.as_tensor(np.asarray(rows, np.float64))
    out = torch.zeros((n,) + tuple(rows.shape[1:]), dtype=torch.float64)
    return out.index_add_(0, torch.as_tensor(np.asarray(idx, np.int64)), rows).numpy()


def ref_node_agg(ef, dst, rev, N):
    """S[v] = [sum_{e in in(v), rev_e} ef[e] | sum_{e in in(v), !rev_e} ef[e]]  (dmp.cu K4)."""
    ef, r = np.asarray(ef, np.float64), rev[:, None]
    S = np.concatenate([_seg(N, dst, np.where(r, ef, 0.0)), _seg(N, dst, np.where(r, 0.0, ef))], 1)
    mag = np.concatenate([_seg(N, dst, np.where(r, np.abs(ef), 0.0)), _seg(N, dst, np.where(r, 0.0, np.abs(ef)))], 1)
    return S, mag


def ref_node_agg_bwd(gS, dst, rev):
    """gef[e] = gS[dst e, :D] if rev_e else gS[dst e, D:]."""
    D = gS.shape[1] // 2
    return np.where(rev[:, None], gS[dst, :D], gS[dst, D:])


def ref_edge_coeff(out_deg, dst):
    """c_e = 2 (1 + log2(1 + out_deg[dst e]))."""
    return 2.0 * (1.0 + np.log2(1.0 + np.asarray(out_deg, np.float64)[dst]))


def ref_edge_update(PQ, T, bias, src, dst, rev, out_deg):
    """out[e] = T[e,:D] + c_e T[e,D:] + (rev ? P[src]-Q[dst] : P[dst]-Q[src]) + b  (dmp.cu K5)."""
    PQ, T = np.asarray(PQ, np.float64), np.asarray(T, np.float64)
    D = T.shape[1] // 2
    a, b = np.where(rev, src, dst), np.where(rev, dst, src)
    c = ref_edge_coeff(out_deg, dst)[:, None]
    terms = [T[:, :D], c * T[:, D:], PQ[a, :D], -PQ[b, D:]]
    if bias is not None:
        terms.append(np.broadcast_to(np.asarray(bias, np.float64), (len(src), D)))
    return sum(terms), sum(np.abs(t) for t in terms)


def ref_edge_update_bwd(g, src, dst, rev, out_deg, N):
    """(gPQ, gT, gb): gP[v] = sum_{e: a_e = v} g[e], gQ[v] = -sum_{e: b_e = v} g[e], gT = [g | c_e g], gb = sum_e g[e]."""
    g = np.asarray(g, np.float64)
    a, b = np.where(rev, src, dst), np.where(rev, dst, src)
    gPQ = np.concatenate([_seg(N, a, g), -_seg(N, b, g)], 1)
    mag = np.concatenate([_seg(N, a, np.abs(g)), _seg(N, b, np.abs(g))], 1)
    gT = np.concatenate([g, ref_edge_coeff(out_deg, dst)[:, None] * g], 1)
    return gPQ, mag, gT, g.sum(0)


def ref_comp(h, ef, src, op, a):
    """C[e] = a[src e] comp(h[src e], ef[e]),  comp = h - r (sub) | h * r (mult)  (comp.cu)."""
    hs, ef = np.asarray(h, np.float64)[src], np.asarray(ef, np.float64)
    C = hs - ef if op == SUB else hs * ef
    return C if a is None else np.asarray(a, np.float64)[src][:, None] * C


def ref_comp_bwd(gC, h, ef, src, op, a, N):
    """(gh, |gh| terms, gef): the adjoints of ref_comp in h and in ef."""
    gC, h, ef = np.asarray(gC, np.float64), np.asarray(h, np.float64), np.asarray(ef, np.float64)
    s = np.ones(len(src)) if a is None else np.asarray(a, np.float64)[src]
    gef = -s[:, None] * gC if op == SUB else s[:, None] * gC * h[src]
    t = gC if op == SUB else gC * ef
    sa = np.ones(N) if a is None else np.asarray(a, np.float64)
    return sa[:, None] * _seg(N, src, t), np.abs(sa)[:, None] * _seg(N, src, np.abs(t)), gef


def ref_label_gate(g_ptr, g_lab, p_ptr, p_lab, Lp_max, length_clause=True):
    """gate[v] = 1 if label(v) occurs in its pattern's labels, or if label(v) == 0 and the pattern is shorter than
    Lp_max (its zero left-padding then matches, basemodel.py:830-847)."""
    gate = np.zeros(len(g_lab), np.float32)
    for b in range(len(g_ptr) - 1):
        lab, pl = g_lab[g_ptr[b]:g_ptr[b + 1]], p_lab[p_ptr[b]:p_ptr[b + 1]]
        hit = np.isin(lab, pl) | ((len(pl) < Lp_max or not length_clause) & (lab == 0))
        gate[g_ptr[b]:g_ptr[b + 1]] = hit
    return gate


def seq_accumulate(n, keys, rows, negate=False):
    """fp32 acc[k] = 0, then for each item i in array order with keys[i] == k: acc[k] += rows[i] (or -= with negate),
    one separately rounded add at a time -- the fixed order of the kernels' CSR walks."""
    rows = np.asarray(rows, np.float32)
    acc = np.zeros((n,) + rows.shape[1:], np.float32)
    keys = np.asarray(keys, np.int64)
    if keys.size == 0:
        return acc
    order = np.argsort(keys, kind="stable")
    k = keys[order]
    pos = np.arange(k.size) - np.searchsorted(k, k)
    for p in range(int(pos.max()) + 1):
        sel = order[pos == p]                  # at most one item per key: a vectorised step of every key's loop
        acc[keys[sel]] = acc[keys[sel]] - rows[sel] if negate else acc[keys[sel]] + rows[sel]
    return acc


# ---------------------------------------------------------------------------------------------------------------------
# GPU plumbing
def _graph(b, device):
    from dummynode4graphlearning_b200.graph import BatchedGraph
    return BatchedGraph.from_batch(b, device)


def _poison(device, *shapes):
    """free NaN-filled blocks of these shapes: the caching allocator hands them to the next outputs of those sizes, so a
    row a kernel fails to write reads as NaN rather than as what an earlier launch left there."""
    blocks = [torch.full(s, float("nan"), device=device) for s in shapes]
    del blocks


def _np(t):
    return t.detach().cpu().numpy()


def _bits_equal(a, b):
    a, b = np.ascontiguousarray(a, np.float32), np.ascontiguousarray(b, np.float32)
    return a.shape == b.shape and np.array_equal(a.view(np.int32), b.view(np.int32))


def _within(out, ref, bound, test, what):
    """|out - ref| <= bound per element (float64); records the error relative to the largest reference value."""
    out = np.asarray(out, np.float64)
    assert out.shape == ref.shape, (what, out.shape, ref.shape)
    err = np.abs(out - ref)
    bad = ~(err <= bound)                      # NaN fails
    if bad.any():
        i = np.unravel_index(np.flatnonzero(bad)[0], out.shape)
        raise AssertionError("%s: %d of %d elements outside the bound; first at %s: out %r ref %r bound %.3e"
                             % (what, int(bad.sum()), out.size, i, out[i], ref[i], bound[i] if np.ndim(bound) else bound))
    record_error(test, what, err=rel_err(torch.from_numpy(out), torch.from_numpy(ref)))


def _assert_adjoint(lhs, rhs, tol, what):
    assert abs(lhs - rhs) <= tol, "%s: <fwd(x), w> = %.17g but <x, bwd(w)> = %.17g (tolerance %.3e)" % (what, lhs, rhs, tol)


# ---------------------------------------------------------------------------------------------------------------------
# K4: dmp_node_agg
@pytest.mark.gpu
@pytest.mark.parametrize("rev", [False, True], ids=["no_rev", "rev_mix"])
@pytest.mark.parametrize("which", ["mixed", "hub"])
@pytest.mark.parametrize("D", [16, 32, 64, 128, 256])
def test_dmp_node_agg(device, D, which, rev):
    """forward against float64 (n u sum|terms|), light rows bit-exact with the edge-id-order fp32 loop; backward an exact
    gather; the two are adjoint; repeated launches bitwise equal; heavy_count = rows with more than 64 in-edges."""
    from dummynode4graphlearning_b200 import ops

    b = _batch(which, rev)
    g = _graph(b, device)
    N, E, src, dst, r = int(b["node_ptr"][-1]), b["src"].size, b["src"], b["dst"], _rev(b)
    indeg = np.bincount(dst, minlength=N)
    assert g.csr_in.heavy_thr == HEAVY
    assert int(g.csr_in.heavy_count.item()) == int((indeg > HEAVY).sum())
    if which == "hub":
        assert int((indeg > HEAVY).sum()) > 4 * _n_sms()
    rng = np.random.default_rng(D + 2 * rev)
    ef = rng.uniform(-1, 1, (E, D)).astype(np.float32)
    w = rng.uniform(-1, 1, (N, 2 * D)).astype(np.float32)
    eft = torch.from_numpy(ef).to(device).requires_grad_(True)
    runs = []
    for _ in range(2):
        _poison(device, (N, 2 * D))
        S = ops.dmp_node_agg(eft, g)
        _poison(device, (E, D))
        gef, = torch.autograd.grad(S, eft, torch.from_numpy(w).to(device))
        runs.append((_np(S), _np(gef)))
    assert _bits_equal(runs[0][0], runs[1][0]) and _bits_equal(runs[0][1], runs[1][1]), "not deterministic"
    S, gef = runs[0]
    tag = "dmp_node_agg[%s-%d-%s]" % (which, D, rev)

    ref, mag = ref_node_agg(ef, dst, r, N)
    _within(S, ref, np.maximum(indeg, 1)[:, None] * U * mag, tag, "S")
    seq = np.concatenate([seq_accumulate(N, dst[r], ef[r]), seq_accumulate(N, dst[~r], ef[~r])], 1)
    light = indeg <= HEAVY
    assert _bits_equal(S[light], seq[light]), "light rows differ from the edge-id-order fp32 sum"
    assert not S[indeg == 0].any()

    assert _bits_equal(gef, ref_node_agg_bwd(w, dst, r)), "backward is not the gather of the destination's half"
    lhs, rhs = float((S.astype(np.float64) * w).sum()), float((ef.astype(np.float64) * gef).sum())
    tol = float((np.maximum(indeg, 1)[:, None] * U * mag * np.abs(w)).sum()) + 1e-12 * float(np.abs(mag * w).sum())
    _assert_adjoint(lhs, rhs, tol, tag)


@pytest.mark.gpu
@pytest.mark.parametrize("D", [4, 8, 12, 512])
def test_dmp_node_agg_rejects_unsupported_width(device, D):
    """widths without a kernel instance raise before anything is launched."""
    from dummynode4graphlearning_b200 import ops
    from dummynode4graphlearning_b200._lib import Dn4glError, lib

    b = _mixed_batch()
    g = _graph(b, device)
    g.csr_in
    ef = torch.zeros((b["src"].size, D), device=device)
    torch.cuda.synchronize()
    k0 = lib().kernel_launches()
    with pytest.raises(Dn4glError, match="unsupported D"):
        ops.dmp_node_agg(ef, g)
    assert lib().kernel_launches() == k0


# ---------------------------------------------------------------------------------------------------------------------
# K5: dmp_edge_update
@pytest.mark.gpu
@pytest.mark.parametrize("rev", [False, True], ids=["no_rev", "rev_mix"])
@pytest.mark.parametrize("with_bias", [False, True], ids=["no_bias", "bias"])
@pytest.mark.parametrize("D", [4, 16, 64, 256])
def test_dmp_edge_update(device, D, with_bias, rev):
    """forward (c u sum|terms|), gT = [g | c_e g] (the first half exact), gPQ bit-exact with the in-list-then-out-list
    fp32 loop (self-loops appear in both lists; nodes without edges get exact zeros), gb = g.sum(0), adjointness.
    D = 4 has no [P|Q]-backward instance: that backward must raise."""
    from dummynode4graphlearning_b200 import ops
    from dummynode4graphlearning_b200._lib import Dn4glError, lib, ptr
    from dummynode4graphlearning_b200.graph import _stream

    b = _batch("mixed", rev)
    g = _graph(b, device)
    N, E, src, dst, r = int(b["node_ptr"][-1]), b["src"].size, b["src"], b["dst"], _rev(b)
    indeg, outdeg = np.bincount(dst, minlength=N), np.bincount(src, minlength=N)
    rng = np.random.default_rng(100 + D + 2 * with_bias + rev)
    PQ = rng.uniform(-1, 1, (N, 2 * D)).astype(np.float32)
    T = rng.uniform(-1, 1, (E, 2 * D)).astype(np.float32)
    bias = rng.uniform(-1, 1, D).astype(np.float32) if with_bias else None
    w = rng.uniform(-1, 1, (E, D)).astype(np.float32)
    ins = [torch.from_numpy(x).to(device).requires_grad_(True) for x in (PQ, T)]
    bt = torch.from_numpy(bias).to(device).requires_grad_(True) if with_bias else None
    wt = torch.from_numpy(w).to(device)
    has_pq = D >= 16
    runs = []
    for _ in range(2):
        _poison(device, (E, D))
        out = ops.dmp_edge_update(ins[0], ins[1], bt, g)
        if has_pq:
            _poison(device, (E, 2 * D), (N, 2 * D))
            grads = torch.autograd.grad(out, ins + ([bt] if with_bias else []), wt)
        else:
            gT = torch.full((E, 2 * D), float("nan"), device=device)
            out_deg = g.cached("out_deg_i32", lambda: g.out_degrees().to(torch.int32).contiguous())
            lib().call("dn4gl_dmp_edge_update_bwd_T_f32", ptr(g.dst), ptr(out_deg), ptr(wt), ptr(gT), E, D, _stream())
            grads = (None, gT)
        runs.append([_np(out)] + [None if x is None else _np(x) for x in grads])
    for a_, b_ in zip(runs[0], runs[1]):
        assert a_ is None or _bits_equal(a_, b_), "not deterministic"
    out, gPQ, gT = runs[0][:3]
    tag = "dmp_edge_update[%d-%s-%s]" % (D, with_bias, rev)

    ref, mag = ref_edge_update(PQ, T, bias, src, dst, r, outdeg)
    _within(out, ref, 8 * U * mag, tag, "out")
    rgPQ, gmag, rgT, rgb = ref_edge_update_bwd(w, src, dst, r, outdeg, N)
    assert _bits_equal(gT[:, :D], w)
    _within(gT, rgT, 4 * U * np.abs(rgT), tag, "gT")
    if not has_pq:
        with pytest.raises(Dn4glError, match="unsupported D"):
            torch.autograd.grad(ops.dmp_edge_update(ins[0], ins[1], bt, g), ins, wt)
        return

    nterms = (indeg + outdeg)[:, None]
    _within(gPQ, rgPQ, np.maximum(nterms, 1) * U * gmag, tag, "gPQ")
    seq = np.concatenate([seq_accumulate(N, np.concatenate([dst[~r], src[r]]), np.concatenate([w[~r], w[r]])),
                          seq_accumulate(N, np.concatenate([dst[r], src[~r]]), np.concatenate([w[r], w[~r]]), negate=True)], 1)
    assert _bits_equal(gPQ, seq), "gPQ differs from the in-list-then-out-list fp32 sum"
    assert not gPQ[(indeg + outdeg) == 0].any()
    if with_bias:
        gb = runs[0][3]
        _within(gb, rgb, E * U * np.abs(w.astype(np.float64)).sum(0), tag, "gb")

    lhs = float((out.astype(np.float64) * w).sum())
    rhs = float((PQ.astype(np.float64) * gPQ).sum() + (T.astype(np.float64) * gT).sum())
    if with_bias:
        rhs += float((bias.astype(np.float64) * runs[0][3]).sum())
    tol = float((8 * U * mag * np.abs(w)).sum() + (np.maximum(nterms, 1) * U * gmag * np.abs(PQ)).sum()
                + (4 * U * np.abs(rgT * T)).sum() + (E * U * np.abs(w).sum(0) * (np.abs(bias) if with_bias else 0)).sum())
    _assert_adjoint(lhs, rhs, tol, tag)


# ---------------------------------------------------------------------------------------------------------------------
# CompGCN composition
@pytest.mark.gpu
@pytest.mark.parametrize("grads", ["h", "ef", "both"])
@pytest.mark.parametrize("scaled", [False, True], ids=["no_scale", "src_scale"])
@pytest.mark.parametrize("op", [SUB, MULT], ids=["sub", "mult"])
@pytest.mark.parametrize("D", [4, 8, 16, 64, 256])
def test_comp_edge(device, D, op, scaled, grads):
    """C and gef elementwise (<= 3 roundings), gh bit-exact with the out-list fp32 loop in edge-id order (times a[u]),
    zero for nodes without out-edges; only the requested gradients; adjointness; repeated launches bitwise equal."""
    from dummynode4graphlearning_b200 import ops

    b = _mixed_batch()
    g = _graph(b, device)
    N, E, src = int(b["node_ptr"][-1]), b["src"].size, b["src"]
    outdeg = np.bincount(src, minlength=N)
    rng = np.random.default_rng(200 + D + 2 * op + scaled)
    h = rng.uniform(-1, 1, (N, D)).astype(np.float32)
    ef = rng.uniform(-1, 1, (E, D)).astype(np.float32)
    a = rng.uniform(0.1, 1.0, (N, 1)).astype(np.float32) if scaled else None
    w = rng.uniform(-1, 1, (E, D)).astype(np.float32)
    ht = torch.from_numpy(h).to(device).requires_grad_(grads in ("h", "both"))
    eft = torch.from_numpy(ef).to(device).requires_grad_(grads in ("ef", "both"))
    at = None if a is None else torch.from_numpy(a).to(device)
    wrt = [t for t in (ht, eft) if t.requires_grad]
    runs = []
    for _ in range(2):
        _poison(device, (E, D))
        C = ops.comp_edge(ht, eft, g, op, at)
        _poison(device, (E, D), (N, D))
        gs = torch.autograd.grad(C, wrt, torch.from_numpy(w).to(device))
        runs.append([_np(C)] + [_np(x) for x in gs])
    for a_, b_ in zip(runs[0], runs[1]):
        assert _bits_equal(a_, b_), "not deterministic"
    C, gs = runs[0][0], dict(zip([n for n in ("h", "ef") if grads in (n, "both")], runs[0][1:]))
    tag = "comp_edge[%d-%s-%s-%s]" % (D, "sub" if op == SUB else "mult", scaled, grads)
    av = None if a is None else a[:, 0]

    ref = ref_comp(h, ef, src, op, av)
    _within(C, ref, 3 * U * np.abs(ref), tag, "C")
    rgh, ghmag, rgef = ref_comp_bwd(w, h, ef, src, op, av, N)
    if "ef" in gs:
        _within(gs["ef"], rgef, 3 * U * np.abs(rgef), tag, "gef")
    if "h" in gs:
        gh = gs["h"]
        _within(gh, rgh, (outdeg[:, None] + 2) * U * ghmag, tag, "gh")
        seq = seq_accumulate(N, src, w if op == SUB else w * ef)
        if a is not None:
            seq = seq * a
        assert _bits_equal(gh, seq), "gh differs from the out-list fp32 sum in edge-id order"
        assert not gh[outdeg == 0].any()
    lhs = float((C.astype(np.float64) * w).sum())
    x_gx = [(h, rgh, ghmag * (outdeg[:, None] + 2), gs.get("h")), (ef, rgef, 3 * np.abs(rgef), gs.get("ef"))]
    if op == SUB:       # linear in (h, ef): <C, w> = <h, gh> + <ef, gef>
        if grads == "both":
            rhs = sum(float((x.astype(np.float64) * gx).sum()) for x, _, _, gx in x_gx)
            tol = U * float((3 * np.abs(ref * w)).sum() + sum((np.abs(x) * m).sum() for x, _, m, _ in x_gx))
            _assert_adjoint(lhs, rhs, tol, tag)
    else:               # bilinear: <C, w> = <h, gh> = <ef, gef>
        for x, _, m, gx in x_gx:
            if gx is not None:
                tol = U * float((3 * np.abs(ref * w)).sum() + (np.abs(x) * m).sum())
                _assert_adjoint(lhs, float((x.astype(np.float64) * gx).sum()), tol, tag)


# ---------------------------------------------------------------------------------------------------------------------
# ScalarFilter gate
@functools.lru_cache(None)
def _gate_batches():
    """(pattern, graph) batches of B graphs: labels 0..3, patterns mostly shorter than the longest (the zero padding
    leaks label 0), patterns without edges, empty graphs in the graph batch (repeated node_ptr / edge_ptr entries).
    Patterns 0 and B // 2 are the longest of the halves B // 2 splits the batch into, and the last one the longest of
    all; these three have labels 1..3 only, and their graphs some label-0 nodes and edges, which only a shorter
    pattern's padding gates in."""
    rng = np.random.default_rng(3)
    B = 301
    gparts = _parts_of(nasty_sub_batch(rng, B, 10, 4))
    pparts = _parts_of(nasty_sub_batch(rng, B, 5, 4))      # at most 5 nodes and 16 edges
    for i in range(1, B - 1, 7):
        gparts[i] = (0, [], [])
    special = {0: (6, 17), B // 2: (6, 17), B - 1: (9, 20)}
    for i, (n, m) in special.items():
        pparts[i] = (n, rng.integers(0, n, m), rng.integers(0, n, m))
        gparts[i] = (12, rng.integers(0, 12, 30), rng.integers(0, 12, 30))
    pb, gb = _assemble(pparts, rng), _assemble(gparts, rng)
    for key, ptr in (("vlabel", "node_ptr"), ("elabel", "edge_ptr")):
        for i in special:
            lo, hi = pb[ptr][i], pb[ptr][i + 1]
            pb[key][lo:hi] = rng.integers(1, 4, hi - lo)
            lo = gb[ptr][i]
            gb[key][lo:lo + 3] = 0
    return pb, gb


def _slice_batch(b, lo, hi):
    """graphs lo..hi-1 of a flat batch, labels kept."""
    n0, n1, e0, e1 = b["node_ptr"][lo], b["node_ptr"][hi], b["edge_ptr"][lo], b["edge_ptr"][hi]
    return dict(num_graphs=hi - lo, node_ptr=b["node_ptr"][lo:hi + 1] - n0, edge_ptr=b["edge_ptr"][lo:hi + 1] - e0,
                src=b["src"][e0:e1] - n0, dst=b["dst"][e0:e1] - n0, vlabel=b["vlabel"][n0:n1], elabel=b["elabel"][e0:e1])


def _gate_inputs(pb, gb, kind):
    lab, ptr = ("vlabel", "node_ptr") if kind == "node" else ("elabel", "edge_ptr")
    return gb[ptr], gb[lab], pb[ptr], pb[lab]


def _oracle_gate(pb, gb, kind):
    from oracle import models as OM
    g_ptr, g_lab, p_ptr, p_lab = _gate_inputs(pb, gb, kind)
    return OM.scalar_filter_gate(torch.as_tensor(p_lab).long(), [int(x) for x in np.diff(p_ptr)],
                                 torch.as_tensor(g_lab).long(), [int(x) for x in np.diff(g_ptr)]).numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["node", "edge"])
def test_label_filter_gate(device, kind):
    """the gate equals oracle.models.scalar_filter_gate exactly (padding leak included); a shard's gate with the whole
    batch's padded lengths (set_padded_lengths) equals the whole batch's gate on that shard's rows."""
    from dummynode4graphlearning_b200.subgraph_isomorphism.models.filter import ScalarFilter

    pb, gb = _gate_batches()
    pg, gg = _graph(pb, device), _graph(gb, device)
    flt = ScalarFilter()
    _poison(device, (int(gb["node_ptr" if kind == "node" else "edge_ptr"][-1]), 1))
    gate = _np(flt.gate_from_graphs(pg, gg, kind))
    assert _bits_equal(gate, flt.gate_from_graphs(pg, gg, kind).cpu().numpy()), "not deterministic"
    assert _bits_equal(gate, _oracle_gate(pb, gb, kind)), "gate differs from the padded-matrix ScalarFilter"

    B, ptr = pb["num_graphs"], "node_ptr" if kind == "node" else "edge_ptr"
    for lo, hi in ((0, B // 2), (B // 2, B - 1)):     # the longest pattern (the last) is in neither shard
        ps, gs = _graph(_slice_batch(pb, lo, hi), device), _graph(_slice_batch(gb, lo, hi), device)
        ps.set_padded_lengths(nodes=pg.padded_num_nodes(), edges=pg.padded_num_edges())
        shard = _np(flt.gate_from_graphs(ps, gs, kind))
        assert _bits_equal(shard, gate[gb[ptr][lo]:gb[ptr][hi]]), "shard gate with the batch-wide padded lengths"


# ---------------------------------------------------------------------------------------------------------------------
# gather_rows
@pytest.mark.gpu
@pytest.mark.parametrize("n,D", [(0, 16), (1, 4), (777, 4), (4097, 16), (3001, 64), (1023, 256)])
def test_gather_rows_exact(device, n, D):
    from dummynode4graphlearning_b200 import ops

    rng = np.random.default_rng(n + D)
    x = rng.standard_normal((333, D)).astype(np.float32)
    idx = rng.integers(0, 333, n).astype(np.int32)
    xt, it = torch.from_numpy(x).to(device), torch.from_numpy(idx).to(device)
    runs = []
    for _ in range(2):
        _poison(device, (n, D))
        runs.append(_np(ops.gather_rows(xt, it)))
    assert _bits_equal(runs[0], x[idx]) and _bits_equal(runs[1], x[idx])


# ---------------------------------------------------------------------------------------------------------------------
# fixed-order dot
def _dot_n(spec):
    """n of a test case: an int, or "k*grid" = k * 4 SMs * 256 threads * 16 (k times the elements at which every CTA of
    the capped grid runs the unrolled loop), "+r" added."""
    if isinstance(spec, int):
        return spec
    k, _, rest = spec.partition("*grid")
    return int(k) * 4 * _n_sms() * 256 * 16 + (int(rest) if rest else 0)


def _dot_operands(n, offset, seed):
    """a, b with |a_i b_i| >= 1/4 (a dropped term is far above the rounding bound), as views at `offset` floats into
    their allocation: offset 1 takes the kernel's scalar path."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    mk = lambda: (torch.rand(n + offset, device="cuda", generator=g) + 0.5) * (torch.randint(0, 2, (n + offset,), device="cuda", generator=g) * 2 - 1)
    return mk()[offset:], mk()[offset:]


def _dot_bound(a, b):
    """(float64 value, bound): per thread ceil(n / (grid * 256)) fused products, 8 tree levels, the float64 sum of the
    partials and the final rounding -> (terms + 10) u sum|a_i b_i|."""
    n = a.numel()
    a64, b64 = a.double().cpu(), b.double().cpu()
    grid = min(-(-max(n, 1) // 4096), 4 * _n_sms())
    per_thread = -(-n // (grid * 256))
    return float((a64 * b64).sum()), (per_thread + 10) * U * float((a64 * b64).abs().sum())


@pytest.mark.gpu
@pytest.mark.parametrize("offset", [0, 1], ids=["aligned", "offset1"])
@pytest.mark.parametrize("n", [1, 3, 4, 4097, "3*grid", "3*grid+5"])
def test_dot(device, n, offset):
    """dot against float64 within the fixed-order bound, bitwise repeatable; dot_beside + join bitwise equals dot."""
    from dummynode4graphlearning_b200 import ops

    n = _dot_n(n)
    a, b = _dot_operands(n, offset, n)
    assert (a.data_ptr() % 16 == 0) == (offset == 0)
    ref, bound = _dot_bound(a, b)
    outs = []
    for _ in range(2):
        out = torch.full((1,), float("nan"), device=device)
        outs.append(float(ops.dot(a, b, out=out)))
    assert _bits_equal(np.float32(outs[0]), np.float32(outs[1])), "not deterministic"
    assert abs(outs[0] - ref) <= bound, (outs[0], ref, bound)
    record_error("dot[%d-%d]" % (n, offset), "dot", err=abs(outs[0] - ref) / abs(ref))
    side, join = ops.dot_beside(a, b)
    join()
    assert _bits_equal(np.float32(float(side)), np.float32(outs[0])), "dot_beside differs from dot"


@pytest.mark.gpu
def test_dot_back_to_back_calls_reset_the_counter(device):
    """the last CTA resets the ticket counter: each call right after another with a different grid is still right (an
    output left unwritten stays NaN)."""
    from dummynode4graphlearning_b200 import ops

    for stream_side in (False, True):
        for i, n in enumerate(["3*grid+5", 4097, 1, "2*grid", 3, 4 * 4096 + 1, "1*grid"]):
            n = _dot_n(n)
            a, b = _dot_operands(n, i % 2, 1000 + i)
            ref, bound = _dot_bound(a, b)
            if stream_side:
                out, join = ops.dot_beside(a, b)
                join()
            else:
                out = ops.dot(a, b, out=torch.full((1,), float("nan"), device=device))
            assert abs(float(out) - ref) <= bound, (stream_side, n, float(out), ref, bound)


@pytest.mark.gpu
def test_dot_empty_input_is_zero(device):
    from dummynode4graphlearning_b200 import ops
    from dummynode4graphlearning_b200._lib import lib

    a = torch.empty(0, device=device)
    k0 = lib().kernel_launches()
    assert float(ops.dot(a, a)) == 0.0
    assert float(ops.dot(a, a, out=torch.full((1,), float("nan"), device=device))) == 0.0
    out, join = ops.dot_beside(a, a)
    join()
    assert float(out) == 0.0
    assert lib().kernel_launches() == k0
    x = torch.ones(5, device=device)                 # and the next non-empty call is unaffected
    assert float(ops.dot(x, x)) == 5.0


# ---------------------------------------------------------------------------------------------------------------------
# CPU checks of the references and batches themselves (no device needed)
def test_batches_hold_the_cases_the_kernels_branch_on():
    b = _mixed_batch()
    N, E, src, dst = int(b["node_ptr"][-1]), b["src"].size, b["src"], b["dst"]
    indeg, outdeg = np.bincount(dst, minlength=N), np.bincount(src, minlength=N)
    assert {0, 1, 2, 3, 5, HEAVY, HEAVY + 1} <= set(indeg.tolist())
    assert N % 2 == 1 and E % 2 == 1
    assert (src == dst).any() and ((indeg + outdeg) == 0).any() and (np.diff(b["edge_ptr"]) == 0).any()
    assert len(set(zip(src.tolist(), dst.tolist()))) < E                   # multi-edges
    assert not np.all(np.diff(np.argsort(dst, kind="stable")) > 0)         # in-lists are not in storage order
    r = _rev(_with_rev(b, True))
    assert 0.3 < r.mean() < 0.7 and not _rev(_with_rev(b, False)).any()
    for sms in (132, 148, 160):
        h = _hub_batch(4 * sms + 37)
        assert int((np.bincount(h["dst"], minlength=int(h["node_ptr"][-1])) > HEAVY).sum()) == 4 * sms + 37


def test_seq_accumulate_is_the_sequential_loop():
    rng = np.random.default_rng(0)
    keys = rng.integers(0, 7, 60)
    rows = rng.standard_normal((60, 3)).astype(np.float32)
    for negate in (False, True):
        want = np.zeros((7, 3), np.float32)
        for k, x in zip(keys, rows):
            want[k] = want[k] - x if negate else want[k] + x
        assert _bits_equal(seq_accumulate(7, keys, rows, negate), want)


def _adjoint_close(lhs, rhs):
    assert abs(lhs - rhs) <= 1e-12 * max(1.0, abs(lhs)), (lhs, rhs)


@pytest.mark.parametrize("rev", [False, True])
def test_reference_backwards_are_adjoints(rev):
    """<fwd(x), w> = <x, bwd(w)> in float64 for every reference pair."""
    b = _with_rev(_mixed_batch(), rev)
    N, E, src, dst, r = int(b["node_ptr"][-1]), b["src"].size, b["src"], b["dst"], _rev(b)
    outdeg = np.bincount(src, minlength=N)
    rng = np.random.default_rng(7)
    D = 8
    x = rng.standard_normal((E, D))
    w = rng.standard_normal((N, 2 * D))
    _adjoint_close((ref_node_agg(x, dst, r, N)[0] * w).sum(), (x * ref_node_agg_bwd(w, dst, r)).sum())

    PQ, T, bias, g = rng.standard_normal((N, 2 * D)), rng.standard_normal((E, 2 * D)), rng.standard_normal(D), rng.standard_normal((E, D))
    gPQ, _, gT, gb = ref_edge_update_bwd(g, src, dst, r, outdeg, N)
    _adjoint_close((ref_edge_update(PQ, T, bias, src, dst, r, outdeg)[0] * g).sum(),
                   (PQ * gPQ).sum() + (T * gT).sum() + (bias * gb).sum())

    h, ef, a = rng.standard_normal((N, D)), rng.standard_normal((E, D)), rng.uniform(0.1, 1, N)
    for sc in (None, a):
        gh, _, gef = ref_comp_bwd(g, h, ef, src, SUB, sc, N)
        _adjoint_close((ref_comp(h, ef, src, SUB, sc) * g).sum(), (h * gh).sum() + (ef * gef).sum())
        gh, _, gef = ref_comp_bwd(g, h, ef, src, MULT, sc, N)
        lhs = (ref_comp(h, ef, src, MULT, sc) * g).sum()
        _adjoint_close(lhs, (h * gh).sum())
        _adjoint_close(lhs, (ef * gef).sum())


def _ident(D):
    return torch.eye(D, dtype=torch.float64)


@pytest.mark.parametrize("rev", [False, True])
def test_references_compose_to_dmp_layer(rev):
    """node:  h W_nloop + S_rev W_out - S_fwd W_in + nbias,  edge: ref_edge_update(h [W_dst | W_src],
    ef [W_eloop | W_src - W_dst], ebias)  ==  oracle.models.dmp_layer without its MLPs (num_mlp_layers = 0)."""
    from oracle import models as OM

    b = _with_rev(_mixed_batch(), rev)
    N, E, src, dst, r = int(b["node_ptr"][-1]), b["src"].size, b["src"], b["dst"], _rev(b)
    outdeg = np.bincount(src, minlength=N)
    D = 8
    rng = np.random.default_rng(8)
    W = {k: rng.standard_normal((D, D)) for k in ("in", "out", "src", "dst", "nloop", "eloop")}
    nbias, ebias = rng.standard_normal(D), rng.standard_normal(D)
    h, ef = rng.standard_normal((N, D)), rng.standard_normal((E, D))
    sd = {"l.%s_weight" % k: torch.from_numpy(v) for k, v in W.items()}
    sd.update({"l.nbias": torch.from_numpy(nbias), "l.ebias": torch.from_numpy(ebias)})
    T = lambda x: torch.from_numpy(np.asarray(x))
    n_out, e_out = OM.dmp_layer(sd, "l", T(h), T(ef), T(src.astype(np.int64)), T(dst.astype(np.int64)),
                                T(r) if rev else None, T(outdeg), dict(act_func="relu", num_mlp_layers=0))
    S = ref_node_agg(ef, dst, r, N)[0]
    node = h @ W["nloop"] + S[:, :D] @ W["out"] - S[:, D:] @ W["in"] + nbias
    edge = ref_edge_update(h @ np.concatenate([W["dst"], W["src"]], 1), ef @ np.concatenate([W["eloop"], W["src"] - W["dst"]], 1),
                           ebias, src, dst, r, outdeg)[0]
    np.testing.assert_allclose(node, n_out.numpy(), rtol=1e-11, atol=1e-11)
    np.testing.assert_allclose(edge, e_out.numpy(), rtol=1e-11, atol=1e-11)


@pytest.mark.parametrize("edge_norm", ["in", "out", "both"])
@pytest.mark.parametrize("op", [SUB, MULT], ids=["sub", "mult"])
@pytest.mark.parametrize("rev", [False, True])
def test_references_compose_to_compgcn_layer(rev, op, edge_norm):
    """norm_e = a[src] b[dst]: b[v] (S_rev W_out + S_fwd W_in)[v] with S = ref_node_agg(ref_comp(h, ef, src, a)) is the
    message-and-aggregation term of oracle.models.compgcn_layer (act none, no BatchNorm)."""
    from oracle import models as OM

    b = _with_rev(_mixed_batch(), rev)
    N, E, src, dst, r = int(b["node_ptr"][-1]), b["src"].size, b["src"], b["dst"], _rev(b)
    indeg, outdeg = np.bincount(dst, minlength=N), np.bincount(src, minlength=N)
    D = 8
    rng = np.random.default_rng(9)
    Win, Wout, Wloop, Wrel = (rng.standard_normal((D, D)) for _ in range(4))
    loop_rel, bias = rng.standard_normal((1, D)), rng.standard_normal(D)
    h, ef = rng.standard_normal((N, D)), rng.standard_normal((E, D))
    T = lambda x: torch.from_numpy(np.asarray(x))
    sd = {"l.in_weight": T(Win), "l.out_weight": T(Wout), "l.loop_weight": T(Wloop), "l.rel_weight": T(Wrel),
          "l.loop_rel": T(loop_rel), "l.bias": T(bias)}
    out, _ = OM.compgcn_layer(sd, "l", T(h), T(ef), T(src.astype(np.int64)), T(dst.astype(np.int64)), T(r) if rev else None,
                              T(indeg), T(outdeg), dict(act_func="none", comp_opt="sub" if op == SUB else "mult",
                                                        edge_norm=edge_norm))
    innorm, outnorm = 1.0 / (indeg + 1.0), 1.0 / (outdeg + 1.0)
    a, bn = {"in": (None, innorm), "out": (outnorm, np.ones(N)), "both": (np.sqrt(outnorm), np.sqrt(innorm))}[edge_norm]
    S = ref_node_agg(ref_comp(h, ef, src, op, a), dst, r, N)[0]
    agg = bn[:, None] * (S[:, :D] @ Wout + S[:, D:] @ Win)
    loop = (h - loop_rel if op == SUB else h * loop_rel) @ Wloop
    np.testing.assert_allclose((agg + loop) * 0.3333333 + bias, out.numpy(), rtol=1e-11, atol=1e-11)


@pytest.mark.parametrize("kind", ["node", "edge"])
def test_reference_gate_is_scalar_filter(kind):
    """ref_label_gate == oracle.models.scalar_filter_gate on the gate batches, and those batches tell the padding leak,
    the length clause and the shard's padded length apart."""
    pb, gb = _gate_batches()
    g_ptr, g_lab, p_ptr, p_lab = _gate_inputs(pb, gb, kind)
    Lp = int(np.diff(p_ptr).max())
    ref = ref_label_gate(g_ptr, g_lab, p_ptr, p_lab, Lp)
    assert np.array_equal(ref, _oracle_gate(pb, gb, kind)[:, 0])
    assert (np.diff(g_ptr) == 0).any() and (np.diff(p_ptr) < Lp).any()
    assert kind == "node" or (np.diff(p_ptr) == 0).any()
    no_leak = np.zeros_like(ref)
    for bi in range(len(g_ptr) - 1):
        no_leak[g_ptr[bi]:g_ptr[bi + 1]] = np.isin(g_lab[g_ptr[bi]:g_ptr[bi + 1]], p_lab[p_ptr[bi]:p_ptr[bi + 1]])
    assert (ref != no_leak).any(), "no node gated in by the padding leak"
    assert (ref != ref_label_gate(g_ptr, g_lab, p_ptr, p_lab, Lp, length_clause=False)).any(), "length clause never matters"
    B = pb["num_graphs"]
    for lo, hi in ((0, B // 2), (B // 2, B - 1)):
        ps, gs = _slice_batch(pb, lo, hi), _slice_batch(gb, lo, hi)
        sg_ptr, sg_lab, sp_ptr, sp_lab = _gate_inputs(ps, gs, kind)
        own = ref_label_gate(sg_ptr, sg_lab, sp_ptr, sp_lab, int(np.diff(sp_ptr).max()))
        assert (own != ref[g_ptr[lo]:g_ptr[hi]]).any(), "the shard's own padded length gives the same gate"
        assert np.array_equal(ref_label_gate(sg_ptr, sg_lab, sp_ptr, sp_lab, Lp), ref[g_ptr[lo]:g_ptr[hi]])
