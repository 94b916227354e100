"""GPU parity (bit-exact) of the transform kernels against the oracle restatement, through the C ABI."""
import numpy as np
import pytest
import torch

from dummynode4graphlearning_b200 import synth

pytestmark = pytest.mark.gpu

TU_KEYS = ("node_ptr", "edge_ptr", "src", "dst", "vlabel", "elabel", "v_is_dummy", "e_is_dummy", "vid", "eid")
SUB_KEYS = ("node_ptr", "edge_ptr", "src", "dst", "vid", "vlabel", "v_is_dummy", "eid", "elabel", "e_is_dummy",
            "e_is_reversed")


def _eq(dev_batch, ora_batch, keys):
    for k in keys:
        a = dev_batch[k].cpu().numpy()
        b = np.asarray(ora_batch[k])
        assert a.shape == b.shape, (k, a.shape, b.shape)
        assert np.array_equal(a, b), (k, np.flatnonzero(a != b)[:10])


def _empty_graph_batch():
    # ragged edge cases: a graph without edges in the middle, a single-node graph, a 2-cycle
    return dict(num_graphs=4, node_ptr=np.array([0, 3, 4, 6, 9], np.int32), edge_ptr=np.array([0, 4, 4, 6, 10], np.int32),
                src=np.array([0, 1, 1, 2, 4, 5, 6, 7, 7, 8], np.int32), dst=np.array([1, 0, 2, 1, 5, 4, 7, 6, 8, 7], np.int32),
                vlabel=np.array([1, 2, 1, 3, 1, 1, 2, 2, 1], np.int32), elabel=np.array([1, 1, 2, 2, 1, 1, 3, 3, 1, 1], np.int32),
                has_edge_labels=True)


@pytest.mark.parametrize("case", ["appB", "ragged", "mutag", "proteins_small", "proteins_full"])
def test_tu_dummy_and_conjugate(device, case):
    from dummynode4graphlearning_b200 import transforms as T
    from oracle import transforms as O

    if case == "appB":  # SURVEY.md App. B golden vector
        b = dict(num_graphs=2, node_ptr=np.array([0, 3, 5], np.int32), edge_ptr=np.array([0, 4, 6], np.int32),
                 src=np.array([0, 1, 1, 2, 3, 4], np.int32), dst=np.array([1, 0, 2, 1, 4, 3], np.int32),
                 vlabel=np.array([1, 2, 1, 2, 2], np.int32), elabel=np.ones(6, np.int32), has_edge_labels=False)
    elif case == "ragged":
        b = _empty_graph_batch()
    elif case == "mutag":
        b = synth.tu_batch("mutag", seed=0)
    elif case == "proteins_small":
        b = synth.tu_batch("proteins", 64, seed=3)
    else:
        b = synth.tu_batch("proteins", seed=0)   # BASELINE config C2 at full size
    db = T.to_device(b, device)
    o_d = O.tu_add_dummy(b)
    g_d = T.tu_add_dummy(db)
    _eq(g_d, o_d, TU_KEYS)
    o_c = O.tu_conjugate(o_d)
    g_c = T.tu_conjugate(g_d)
    _eq(g_c, o_c, TU_KEYS + ("v_origin", "e_shared"))
    if case == "appB":
        assert g_c["src"].cpu().tolist()[:14] == [1, 4, 0, 3, 4, 0, 3, 4, 2, 4, 1, 0, 3, 2]
        assert g_c["dst"].cpu().tolist()[:14] == [0, 0, 1, 1, 1, 2, 2, 2, 3, 3, 4, 4, 4, 4]
        assert g_c["elabel"].cpu().tolist() == [1, 1, 2, 2, 2, 2, 2, 2, 1, 1, 1, 2, 2, 1, 2, 2, 2, 2, 2, 2]
    # LINE_ graphs (no dummy)
    o_l = O.tu_conjugate(b)
    g_l = T.tu_conjugate(db)
    _eq(g_l, o_l, ("node_ptr", "edge_ptr", "src", "dst", "vlabel", "elabel", "vid", "eid"))
    # closed forms (SURVEY.md App. B): V' = m + 1 per graph with edges, E' = sum in*out + 2m
    n = np.diff(b["node_ptr"]); m = np.diff(b["edge_ptr"])
    indeg = np.bincount(b["dst"], minlength=b["node_ptr"][-1]); outdeg = np.bincount(b["src"], minlength=b["node_ptr"][-1])
    gid = np.repeat(np.arange(len(n)), n)
    prod = np.bincount(gid, weights=(indeg * outdeg).astype(np.float64), minlength=len(n)).astype(np.int64)
    Vc = np.diff(g_c["node_ptr"].cpu().numpy()); Ec = np.diff(g_c["edge_ptr"].cpu().numpy())
    assert np.array_equal(Vc, m + 1)
    assert np.array_equal(Ec, prod + 2 * m)
    torch.cuda.synchronize()
    from dummynode4graphlearning_b200.graph import check_errors
    check_errors()


@pytest.mark.parametrize("shape,bs", [("small", 64), ("small", 512), ("large", 16)])
def test_sub_add_dummy(device, shape, bs):
    from dummynode4graphlearning_b200 import transforms as T
    from oracle import transforms as O

    p, g, _ = synth.counting_batch(shape, bs, seed=1)
    cfg = synth.counting_config(shape)
    for b, (nv, nvl, ne, nel) in ((p, (cfg["max_npv"], cfg["max_npvl"], cfg["max_npe"], cfg["max_npel"])),
                                  (g, (cfg["max_ngv"], cfg["max_ngvl"], cfg["max_nge"], cfg["max_ngel"]))):
        o = O.sub_add_dummy(b, nv, nvl, ne, nel)
        d = T.sub_add_dummy(T.to_device(b, device), nv, nvl, ne, nel)
        _eq(d, o, SUB_KEYS)


def test_sub_add_dummy_golden_appB2(device):
    """SURVEY.md App. B second vector (reference train.py:404-435 executed under the shims)."""
    from dummynode4graphlearning_b200 import transforms as T

    g = dict(num_graphs=1, node_ptr=np.array([0, 3], np.int32), edge_ptr=np.array([0, 3], np.int32),
             src=np.array([0, 1, 1], np.int32), dst=np.array([1, 2, 2], np.int32), vid=np.arange(3, dtype=np.int32),
             vlabel=np.array([0, 1, 0], np.int32), eid=np.arange(3, dtype=np.int32), elabel=np.array([0, 1, 0], np.int32))
    d = T.sub_add_dummy(T.to_device(g, device), 4, 2, 6, 2)
    assert d["src"].cpu().tolist() == [0, 1, 1, 0, 1, 2, 3, 3, 3]
    assert d["dst"].cpu().tolist() == [1, 2, 2, 3, 3, 3, 0, 1, 2]
    assert d["eid"].cpu().tolist() == [0, 1, 2, 6, 6, 6, 7, 7, 7]
    assert d["elabel"].cpu().tolist() == [0, 1, 0, 2, 2, 2, 3, 3, 3]
    assert d["e_is_reversed"].cpu().tolist() == [0, 0, 0, 0, 0, 0, 1, 1, 1]
    assert d["vid"].cpu().tolist() == [0, 1, 2, 4] and d["vlabel"].cpu().tolist() == [0, 1, 0, 2]


SUB_CONJ_KEYS = ("node_ptr", "edge_ptr", "src", "dst", "v_origin", "e_shared", "vid", "vlabel", "v_is_dummy", "v_is_reversed",
                 "eid", "elabel", "e_is_dummy")


@pytest.mark.parametrize("shape,bs,dummy", [("small", 64, True), ("small", 512, True), ("small", 200, False), ("large", 16, True),
                                            ("large", 8, False)])
def test_sub_conjugate(device, shape, bs, dummy):
    """a5: convert_conjugate_graph (utils/graph.py:77-175) on pattern and graph batches, with and without the dummy
    augmentation (whose n^2 equal-key candidates must collapse to one edge), bit-exact incl. edge order."""
    from dummynode4graphlearning_b200 import transforms as T
    from oracle import transforms as O

    p, g, _ = synth.counting_batch(shape, bs, seed=2)
    cfg = synth.counting_config(shape)
    for b, (nv, nvl, ne, nel) in ((p, (cfg["max_npv"], cfg["max_npvl"], cfg["max_npe"], cfg["max_npel"])),
                                  (g, (cfg["max_ngv"], cfg["max_ngvl"], cfg["max_nge"], cfg["max_ngel"]))):
        ob = O.sub_add_dummy(b, nv, nvl, ne, nel) if dummy else b
        db = T.to_device(ob, device)
        keys = [k for k in SUB_CONJ_KEYS if k in O.sub_conjugate(ob)]
        _eq(T.sub_conjugate(db, id_bound=ne + 2), O.sub_conjugate(ob), keys)
        _eq(T.sub_conjugate(db), O.sub_conjugate(ob), keys)       # id bound read from the data


def test_sub_conjugate_duplicate_ids_and_empty_graphs(device):
    """repeated edge ids inside a graph (vertex merge + key dedupe across different shared vertices), a graph without
    edges in the middle of the batch, and the App. B second golden vector (SURVEY.md)."""
    from dummynode4graphlearning_b200 import transforms as T
    from oracle import transforms as O

    rng = np.random.default_rng(5)
    graphs = []
    for n, m in ((6, 14), (3, 0), (9, 30), (1, 0), (5, 12)):
        s = rng.integers(0, n, m); d = rng.integers(0, n, m)
        graphs.append((s, d, rng.integers(0, 2, n), rng.integers(0, 3, m), rng.integers(0, max(m // 3, 1), m)))
    node_ptr = np.cumsum([0] + [len(g[2]) for g in graphs]).astype(np.int32)
    edge_ptr = np.cumsum([0] + [len(g[0]) for g in graphs]).astype(np.int32)
    b = dict(num_graphs=len(graphs), node_ptr=node_ptr, edge_ptr=edge_ptr,
             src=np.concatenate([g[0] + node_ptr[i] for i, g in enumerate(graphs)]).astype(np.int32),
             dst=np.concatenate([g[1] + node_ptr[i] for i, g in enumerate(graphs)]).astype(np.int32),
             vid=np.concatenate([np.arange(len(g[2])) for g in graphs]).astype(np.int32),
             vlabel=np.concatenate([g[2] for g in graphs]).astype(np.int32),
             elabel=np.concatenate([g[3] for g in graphs]).astype(np.int32),
             eid=np.concatenate([g[4] for g in graphs]).astype(np.int32))
    ref = O.sub_conjugate(b)
    _eq(T.sub_conjugate(T.to_device(b, device)), ref, [k for k in SUB_CONJ_KEYS if k in ref])

    g = dict(num_graphs=1, node_ptr=np.array([0, 3], np.int32), edge_ptr=np.array([0, 3], np.int32),
             src=np.array([0, 1, 1], np.int32), dst=np.array([1, 2, 2], np.int32), vid=np.arange(3, dtype=np.int32),
             vlabel=np.array([0, 1, 0], np.int32), eid=np.arange(3, dtype=np.int32), elabel=np.array([0, 1, 0], np.int32))
    c = T.sub_conjugate(T.sub_add_dummy(T.to_device(g, device), 4, 2, 6, 2), id_bound=8)
    assert c["vid"].cpu().tolist() == [0, 1, 2, 6, 7] and c["vlabel"].cpu().tolist() == [0, 1, 0, 2, 3]
    assert list(zip(c["src"].cpu().tolist(), c["dst"].cpu().tolist())) == [(4, 0), (0, 1), (4, 1), (0, 2), (4, 2), (4, 3), (0, 3),
                                                                         (4, 3), (1, 3), (2, 3), (3, 4)]
    assert c["eid"].cpu().tolist() == [0, 1, 1, 1, 1, 0, 1, 1, 2, 2, 4]
    assert c["e_is_dummy"].cpu().tolist() == [0] * 10 + [1] and c["v_is_reversed"].cpu().tolist() == [0, 0, 0, 0, 1]


@pytest.mark.parametrize("case", ["mutag_dummy", "proteins_conj", "dups"])
def test_pyg_canonicalize(device, case):
    from dummynode4graphlearning_b200 import transforms as T
    from oracle import transforms as O

    if case == "mutag_dummy":
        b = O.tu_add_dummy(synth.tu_batch("mutag", seed=0)); b["has_edge_labels"] = True
    elif case == "proteins_conj":
        b = O.tu_conjugate(O.tu_add_dummy(synth.tu_batch("proteins", 200, seed=5))); b["has_edge_labels"] = True
    else:  # self loops + duplicate pairs with different labels
        b = dict(num_graphs=1, node_ptr=np.array([0, 4], np.int32), edge_ptr=np.array([0, 8], np.int32),
                 src=np.array([2, 0, 1, 0, 3, 0, 2, 1], np.int32), dst=np.array([1, 1, 1, 1, 3, 2, 1, 0], np.int32),
                 vlabel=np.array([1, 2, 0, 1], np.int32), elabel=np.array([1, 2, 1, 1, 2, 2, 2, 1], np.int32),
                 has_edge_labels=True)
    d = T.pyg_canonicalize(T.to_device(b, device))
    emin = int(b["elabel"].min()); R = int(b["elabel"].max()) - emin + 1
    o_src, o_dst, o_first, o_mult = O.pyg_coalesce(b["src"], b["dst"], b["elabel"] - emin, R)
    assert np.array_equal(d["edge_index"][0].cpu().numpy(), o_src)
    assert np.array_equal(d["edge_index"][1].cpu().numpy(), o_dst)
    assert np.array_equal(d["first_edge"].cpu().numpy(), o_first)
    assert np.array_equal(d["edge_attr"].cpu().numpy(), o_mult.astype(np.float32))
    vmin = int(b["vlabel"].min())
    onehot = np.eye(int(b["vlabel"].max()) - vmin + 1, dtype=np.float32)[b["vlabel"] - vmin]
    assert np.array_equal(d["x"].cpu().numpy(), onehot)
    # sortedness + no self loops + uniqueness (size-independent properties)
    ei = d["edge_index"].cpu().numpy()
    key = ei[0].astype(np.int64) * (ei.max() + 1) + ei[1]
    assert np.all(np.diff(key) > 0) and np.all(ei[0] != ei[1])


@pytest.mark.parametrize("n,e", [(1, 0), (5, 0), (1000, 5000), (50000, 400000)])
def test_build_csr_stable(device, n, e):
    from dummynode4graphlearning_b200.graph import build_csr, check_errors
    from oracle import transforms as O

    rng = np.random.default_rng(n + e)
    src = rng.integers(0, n, e).astype(np.int32); dst = rng.integers(0, n, e).astype(np.int32)
    if e > 100:   # one very heavy row (exercises the CTA rank sort, both sizes)
        dst[: min(e // 2, 6000)] = 0
        dst[e // 2: e // 2 + 300] = n - 1
    csr = build_csr(torch.from_numpy(dst).to(device), torch.from_numpy(src).to(device), n)
    rp, col, eid = O.csr_by_dst(n, src, dst)
    assert np.array_equal(csr.row_ptr.cpu().numpy(), rp)
    assert np.array_equal(csr.eid.cpu().numpy(), eid)
    assert np.array_equal(csr.col.cpu().numpy(), col)
    if e > 0:
        hv = set(csr.heavy_rows[: int(csr.heavy_count.item())].cpu().tolist())
        assert hv == set(np.flatnonzero(np.diff(rp) > csr.heavy_thr).tolist())
    check_errors()


@pytest.mark.parametrize("n,e", [(1, 0), (7, 0), (9, 3), (1000, 5000), (50000, 400000)])
def test_build_csr_sorted_keys(device, n, e):
    """dn4gl_build_csr_sorted (boundary marking) == the general stable build on non-decreasing keys; an unsorted key
    raises the asynchronous error flag."""
    from dummynode4graphlearning_b200.graph import build_csr, check_errors
    from oracle import transforms as O

    rng = np.random.default_rng(n * 3 + e)
    dst = np.sort(rng.integers(0, n, e)).astype(np.int32)
    if e > 100:
        dst[dst < n // 3] = 0          # a heavy first row and a long run of empty rows behind it
        dst[-50:] = n - 1
    src = rng.integers(0, n, e).astype(np.int32)
    csr = build_csr(torch.from_numpy(dst).to(device), torch.from_numpy(src).to(device), n, sorted_keys=True)
    rp, col, eid = O.csr_by_dst(n, src, dst)
    assert np.array_equal(csr.row_ptr.cpu().numpy(), rp)
    assert np.array_equal(csr.eid.cpu().numpy(), eid)
    assert np.array_equal(csr.col.cpu().numpy(), col)
    check_errors()
    if e > 100:
        bad = dst.copy()
        bad[e // 2] = n - 1            # out of order
        build_csr(torch.from_numpy(bad).to(device), torch.from_numpy(src).to(device), n, sorted_keys=True)
        with pytest.raises(RuntimeError):
            check_errors()
        check_errors()                 # the flag was cleared


@pytest.mark.parametrize("n", [0, 1, 4095, 4096, 4097, 1 << 20, (1 << 22) + 3])
def test_exclusive_scan(device, n):
    from dummynode4graphlearning_b200._lib import lib, ptr

    rng = np.random.default_rng(n)
    a = rng.integers(0, 5, n).astype(np.int32)
    x = torch.from_numpy(a).to(device)
    out = torch.empty(n + 1, dtype=torch.int32, device=device)
    L = lib()
    wsb = L.size("dn4gl_scan_workspace_bytes", n)
    ws = torch.empty(wsb, dtype=torch.uint8, device=device)
    L.call("dn4gl_exclusive_scan_i32", ptr(x), ptr(out), n, ptr(ws), wsb, torch.cuda.current_stream().cuda_stream)
    ref = np.concatenate([[0], np.cumsum(a, dtype=np.int64)]).astype(np.int32)
    assert np.array_equal(out.cpu().numpy(), ref)


@pytest.mark.parametrize("shape", ["small", "large"])
def test_augmentation_flags_match_golden_and_oracle(device, shape):
    """SURVEY.md 8(f) rank 3 on the GPU: remove_loops / add_reversed_edges (+ the dummy augmentation behind it) /
    compute_norm / eigenvalue bounds, bit-exact with the reference-generated goldens."""
    from dummynode4graphlearning_b200 import transforms as T
    from dummynode4graphlearning_b200.graph import BatchedGraph
    from helpers import batches_equal, load_golden

    g = load_golden("transforms")["aug/" + shape]
    cfg = g["cfg"]
    E_KEYS = ("edge_ptr", "src", "dst", "eid", "elabel")
    SUB_KEYS = ("node_ptr", "edge_ptr", "src", "dst", "vid", "vlabel", "v_is_dummy", "eid", "elabel", "e_is_dummy", "e_is_reversed")
    for side, mx in (("pattern", ("max_npv", "max_npvl", "max_npe", "max_npel")), ("graph", ("max_ngv", "max_ngvl", "max_nge", "max_ngel"))):
        batches_equal(T.sub_remove_loops(T.to_device(g[side + "_loops"], device)), g[side + "_noloops"], E_KEYS)
        rev = T.sub_add_reversed(T.to_device(g[side], device), cfg[mx[2]], cfg[mx[3]])
        batches_equal(rev, g[side + "_rev"], E_KEYS + ("e_is_reversed",))
        d = T.sub_add_dummy(rev, cfg[mx[0]], cfg[mx[1]], 2 * cfg[mx[2]], 2 * cfg[mx[3]])
        batches_equal(d, g[side + "_rev_dummy"], SUB_KEYS)
    gd = g["graph_rev_dummy"]
    for sl, key in ((True, "norms_self_loop"), (False, "norms_no_self_loop")):
        bg = BatchedGraph.from_batch(T.to_device(gd, device), device)
        T.calculate_norms(bg, self_loop=sl)
        T.calculate_eigenvalues(bg)
        assert np.array_equal(bg.ndata["norm"].cpu().numpy(), g[key]["node_norm"])
        assert np.array_equal(bg.edata["norm"].cpu().numpy(), g[key]["edge_norm"])
        assert np.array_equal(bg.ndata["node_eigenv"].cpu().numpy(), g[key]["node_eigenv"])
        assert np.array_equal(bg.edata["edge_eigenv"].cpu().numpy(), g[key]["edge_eigenv"])


def test_augmentation_flags_random_against_oracle(device):
    """larger seeded batches (C3 batch size) against the numpy oracle, incl. a graph with no edges left."""
    from dummynode4graphlearning_b200 import synth, transforms as T
    from dummynode4graphlearning_b200.graph import BatchedGraph
    from helpers import batches_equal
    from oracle import transforms as O

    p, g, _ = synth.counting_batch("small", 256, seed=77)
    cfg = synth.counting_config("small")
    g = dict(g)
    g["dst"] = g["dst"].copy()
    g["dst"][::3] = g["src"][::3]
    e0, e1 = int(g["edge_ptr"][5]), int(g["edge_ptr"][6])
    g["dst"][e0:e1] = g["src"][e0:e1]                       # graph 5 loses every edge
    ref = O.sub_remove_loops(g)
    out = T.sub_remove_loops(T.to_device(g, device))
    batches_equal(out, ref, ("edge_ptr", "src", "dst", "eid", "elabel"))
    ref_r = O.sub_add_reversed(ref, cfg["max_nge"], cfg["max_ngel"])
    out_r = T.sub_add_reversed(out, cfg["max_nge"], cfg["max_ngel"])
    batches_equal(out_r, ref_r, ("edge_ptr", "src", "dst", "eid", "elabel", "e_is_reversed"))
    assert T.sub_add_reversed(out_r, 1, 1) is out_r           # already reversed: untouched (train.py:321)
    bg = BatchedGraph.from_batch(out_r, device)
    ne, ee = T.compute_largest_eigenvalues(bg)
    rne, ree = O.compute_largest_eigenvalues(ref_r)
    assert np.array_equal(ne.cpu().numpy(), rne) and np.array_equal(ee.cpu().numpy(), ree)
    assert rne[5] == 0
    for sl in (True, False):
        nn_, en = T.compute_norm(bg, sl)
        rn, re = O.compute_norm(ref_r, sl)
        assert np.array_equal(nn_.cpu().numpy(), rn) and np.array_equal(en.cpu().numpy(), re)


@pytest.mark.parametrize("case", ["small", "large", "runs"])
def test_match_weights_golden(device, case):
    """SURVEY.md 8(f) rank 2 on the GPU: batched node / edge match weights, bit-exact with the reference's numba loops."""
    from dummynode4graphlearning_b200 import transforms as T
    from dummynode4graphlearning_b200.subgraph_isomorphism import matching as M
    from helpers import load_golden
    g = load_golden("transforms")["match/" + case]
    sub = M.pack_subisomorphisms(g["mats"], device)
    pb, gb = T.to_device(g["pattern"], device), T.to_device(g["graph"], device)
    assert np.array_equal(M.node_weights(sub, gb).cpu().numpy(), g["node_weights"])
    assert np.array_equal(M.edge_weights(sub, pb, gb).cpu().numpy(), g["edge_weights"])
    work, conj = M.conjugate_subisomorphisms(sub, pb, gb)
    work, conj = work.cpu().numpy(), conj.cpu().numpy()
    for b, ref in enumerate(g["conj"]):
        assert np.array_equal(conj[work[b]: work[b + 1]].reshape(ref.shape), ref), b


def test_match_weights_batch512_against_oracle(device):
    """C3 batch size, up to 40 subisomorphisms per sample, against the Python oracle; empty samples give zeros."""
    from dummynode4graphlearning_b200 import synth, transforms as T
    from dummynode4graphlearning_b200.subgraph_isomorphism import matching as M
    from oracle import transforms as O
    p, g, _ = synth.counting_batch("small", 512, seed=88)
    mats = synth.random_subisomorphisms(p, g, seed=9, max_rows=40)
    mats[3] = np.zeros((0, mats[3].shape[1]), np.int64)
    sub = M.pack_subisomorphisms(mats, device)
    pb, gb = T.to_device(p, device), T.to_device(g, device)
    nw, ew = M.node_weights(sub, gb), M.edge_weights(sub, pb, gb)
    assert np.array_equal(nw.cpu().numpy(), O.subiso_node_weights(mats, g))
    assert np.array_equal(ew.cpu().numpy(), O.subiso_edge_weights(mats, p, g))
    work, conj = M.conjugate_subisomorphisms(sub, pb, gb)
    work, conj = work.cpu().numpy(), conj.cpu().numpy()
    for b, ref in enumerate(O.subiso_conjugate(mats, p, g)):
        assert np.array_equal(conj[work[b]: work[b + 1]].reshape(ref.shape), ref), b
    n0, n1 = int(g["node_ptr"][3]), int(g["node_ptr"][4])
    assert int(nw[n0:n1].sum()) == 0 and int(ew.sum()) > 0
    empty = M.pack_subisomorphisms([np.zeros((0, m.shape[1]), np.int64) for m in mats], device)
    assert int(M.node_weights(empty, gb).sum()) == 0 and int(M.edge_weights(empty, pb, gb).sum()) == 0


def test_augmentation_and_match_weights_empty_inputs(device):
    """edge cases: graphs without edges inside a batch, a batch without any edge, no subisomorphisms at all."""
    from dummynode4graphlearning_b200 import transforms as T
    from dummynode4graphlearning_b200.graph import BatchedGraph
    from dummynode4graphlearning_b200.subgraph_isomorphism import matching as M
    from helpers import batches_equal
    from oracle import transforms as O

    b = dict(num_graphs=3, node_ptr=np.array([0, 2, 5, 6], np.int32), edge_ptr=np.array([0, 0, 3, 3], np.int32),
             src=np.array([2, 3, 4], np.int32), dst=np.array([3, 3, 2], np.int32), vid=np.array([0, 1, 0, 1, 2, 0], np.int32),
             vlabel=np.zeros(6, np.int32), eid=np.arange(3, dtype=np.int32), elabel=np.array([1, 0, 1], np.int32))
    rev = T.sub_add_reversed(T.to_device(b, device), 7, 3)
    batches_equal(rev, O.sub_add_reversed(b, 7, 3), ("edge_ptr", "src", "dst", "eid", "elabel", "e_is_reversed"))
    batches_equal(T.sub_remove_loops(T.to_device(b, device)), O.sub_remove_loops(b), ("edge_ptr", "src", "dst", "eid", "elabel"))
    empty = dict(b, edge_ptr=np.zeros(4, np.int32), src=np.zeros(0, np.int32), dst=np.zeros(0, np.int32),
                 eid=np.zeros(0, np.int32), elabel=np.zeros(0, np.int32))
    r0 = T.sub_add_reversed(T.to_device(empty, device), 7, 3)
    assert r0["src"].numel() == 0 and r0["edge_ptr"].cpu().tolist() == [0, 0, 0, 0]
    l0 = T.sub_remove_loops(T.to_device(empty, device))
    assert l0["src"].numel() == 0 and l0["edge_ptr"].cpu().tolist() == [0, 0, 0, 0]
    bg = BatchedGraph.from_batch(T.to_device(b, device), device)
    ne, ee = T.compute_largest_eigenvalues(bg)
    rne, ree = O.compute_largest_eigenvalues(b)
    assert np.array_equal(ne.cpu().numpy(), rne) and np.array_equal(ee.cpu().numpy(), ree) and rne[0] == 0 and rne[2] == 0
    sub = M.pack_subisomorphisms([np.zeros((0, 2), np.int64), np.array([[0, 1, 2]], np.int64), np.zeros((0, 1), np.int64)], device)
    gb = T.to_device(b, device)
    assert M.node_weights(sub, gb).cpu().tolist() == [0, 0, 1, 1, 1, 0]
    ew = M.edge_weights(sub, gb, gb)          # the batch as its own pattern: the identity map matches every edge once
    assert ew.cpu().tolist() == O.subiso_edge_weights([np.zeros((0, 2)), np.array([[0, 1, 2]]), np.zeros((0, 1))], b, b).tolist() == [1, 1, 1]


def test_pyg_canonicalize_deferred_count_equals_exact(device):
    """deferred edge count (tail padded with a trash row, no second read-back) == the exact path: same CSRs on the logical
    rows, same lazily materialised edge_index, same GIN output -- on a batch with planted self loops and repeated edges so
    that the padding is really exercised."""
    from argparse import Namespace
    from dummynode4graphlearning_b200 import synth, transforms as T
    from dummynode4graphlearning_b200.graph_classification.data import Batch
    from dummynode4graphlearning_b200.graph_classification.models import GIN

    raw = {k: v for k, v in synth.tu_batch("mutag", 40, seed=3).items() if k != "vattr"}
    raw["dst"] = raw["dst"].copy()
    raw["dst"][::9] = raw["src"][::9]                  # self loops
    raw["src"] = raw["src"].copy()
    for g in range(0, 40, 3):                           # a repeated edge per third graph
        e0 = int(raw["edge_ptr"][g])
        if raw["edge_ptr"][g + 1] - e0 >= 2:
            raw["src"][e0 + 1], raw["dst"][e0 + 1] = raw["src"][e0], raw["dst"][e0]
    b = T.tu_add_dummy(T.to_device(raw, device))
    b["has_edge_labels"] = True
    exact = T.pyg_canonicalize(b, 8, None, node_label_min=0, with_edge_attr=False)
    lazy = T.pyg_canonicalize(b, 8, None, node_label_min=0, with_edge_attr=False, defer_count=True)
    E2 = int(exact["src"].numel())
    assert lazy.get("trash_row") and int(lazy["src"].numel()) > E2, "the test batch must lose edges in coalesce"
    assert torch.equal(lazy["edge_index"], exact["edge_index"]) and torch.equal(lazy["first_edge"], exact["first_edge"])
    N = int(b["vlabel"].numel())
    assert bool((lazy["src"][E2:] == N).all()) and bool((lazy["dst"][E2:] == N).all())
    de, dl = Batch.from_canonical(exact), Batch.from_canonical(lazy)
    for name in ("csr_in", "csr_out"):
        ce, cl = getattr(de.structure, name), getattr(dl.structure, name)
        assert cl.n_rows == ce.n_rows == N
        assert torch.equal(cl.row_ptr[: N + 1], ce.row_ptr) and torch.equal(cl.col[:E2], ce.col)
    args = Namespace(num_features=8, hidden_dim=32, num_classes=2, dropout_ratio=0.0,
                     additional={"train_eps": True, "num_layers": 3, "aggregation": "sum"}, epochs=1, device=str(device))
    torch.manual_seed(0)
    model = GIN(args).to(device).train()
    oe = model(de)
    ol = model(dl)
    assert torch.equal(oe, ol)
    oe.sum().backward()
    ge = [p.grad.clone() for p in model.parameters()]
    model.zero_grad()
    ol.sum().backward()
    for a, c in zip(ge, [p.grad for p in model.parameters()]):
        assert torch.equal(a, c)
