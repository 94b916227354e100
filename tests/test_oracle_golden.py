"""CPU: the standalone oracle restatement (oracle/c/transforms.c, oracle/models.py) against the golden vectors
produced by the UNMODIFIED reference (oracle/gen_golden.py) and against SURVEY.md App. B."""
import numpy as np
import pytest
import torch

from helpers import assert_close_rel, batches_equal, load_golden, oracle_cfg
from oracle import models as OM
from oracle import transforms as OT

TU_KEYS = ("node_ptr", "edge_ptr", "src", "dst", "vlabel", "elabel", "v_is_dummy", "e_is_dummy", "vid", "eid")
SUB_KEYS = ("node_ptr", "edge_ptr", "src", "dst", "vid", "vlabel", "v_is_dummy", "eid", "elabel", "e_is_dummy",
            "e_is_reversed")
CONJ_KEYS = ("node_ptr", "edge_ptr", "src", "dst", "vid", "vlabel", "v_is_dummy", "v_is_reversed", "eid", "elabel",
             "e_is_dummy")


@pytest.fixture(scope="module", autouse=True)
def golden_thread_count():
    """the fp32 goldens carry the reduction order of torch's CPU kernels split over at least 8 intra-op threads (the split
    stops changing there at these sizes); on fewer threads the oracle rounds differently by a few 1e-6, more than the
    1e-6 bars below allow"""
    before = torch.get_num_threads()
    torch.set_num_threads(8)
    yield
    torch.set_num_threads(before)


@pytest.fixture(scope="module")
def gold_t():
    return load_golden("transforms")


@pytest.mark.parametrize("case", ["appB", "mutag12", "proteins8"])
def test_tu_transforms_match_reference_golden(gold_t, case):
    g = gold_t["tu/" + case]
    d = OT.tu_add_dummy(g["inp"])
    batches_equal(d, g["dummy"], TU_KEYS)
    c = OT.tu_conjugate(d)
    batches_equal(c, g["conj"], TU_KEYS)
    line = OT.tu_conjugate(g["inp"])
    batches_equal(line, g["line"], ("node_ptr", "edge_ptr", "src", "dst", "vlabel", "elabel", "vid", "eid"))
    if "vattr" in g["inp"]:
        np.testing.assert_array_equal(d["vattr"], g["dummy"]["vattr"])
        np.testing.assert_array_equal(c["eattr"], g["conj"]["eattr"])
    # the reference's save_graph_data text for the CONJ graphs (tu_data_processing.py:353-414)
    f = g["conj_files"]
    assert f["A"] == ["%d,%d" % (s + 1, t + 1) for s, t in zip(c["src"], c["dst"])]
    assert f["node_labels"] == [str(int(x)) for x in c["vlabel"]]
    assert f["edge_labels"] == [str(int(x)) for x in c["elabel"]]
    assert f["node_ids"] == [str(int(x)) for x in c["vid"]]
    assert f["edge_ids"] == [str(int(x)) for x in c["eid"]]
    assert f["graph_indicator"] == [str(i + 1) for i in range(c["num_graphs"]) for _ in range(c["node_ptr"][i + 1] - c["node_ptr"][i])]


@pytest.mark.parametrize("shape", ["small", "large"])
def test_augmentation_flags_match_reference_golden(gold_t, shape):
    """SURVEY.md 8(f) rank 3: remove_loops / add_reversed_edges / add_dummy after add_rev / norms / eigenvalue bounds."""
    g = gold_t["aug/" + shape]
    cfg = g["cfg"]
    E_KEYS = ("edge_ptr", "src", "dst", "eid", "elabel")
    for side, mx in (("pattern", ("max_npv", "max_npvl", "max_npe", "max_npel")), ("graph", ("max_ngv", "max_ngvl", "max_nge", "max_ngel"))):
        batches_equal(OT.sub_remove_loops(g[side + "_loops"]), g[side + "_noloops"], E_KEYS)
        assert (g[side + "_noloops"]["src"] != g[side + "_noloops"]["dst"]).all()
        rev = OT.sub_add_reversed(g[side], cfg[mx[2]], cfg[mx[3]])
        batches_equal(rev, g[side + "_rev"], E_KEYS + ("e_is_reversed",))
        # the dummy augmentation that follows sees the doubled maxima (process_model_config, train.py:38-47)
        d = OT.sub_add_dummy(rev, cfg[mx[0]], cfg[mx[1]], 2 * cfg[mx[2]], 2 * cfg[mx[3]])
        batches_equal(d, g[side + "_rev_dummy"], SUB_KEYS)
    d = g["graph_rev_dummy"]
    for sl, key in ((True, "norms_self_loop"), (False, "norms_no_self_loop")):
        nn_, en = OT.compute_norm(d, sl)
        np.testing.assert_array_equal(nn_, g[key]["node_norm"])
        np.testing.assert_array_equal(en, g[key]["edge_norm"])
    ne, ee = OT.compute_largest_eigenvalues(d)
    np.testing.assert_array_equal(np.repeat(np.maximum(ne, 1), np.diff(d["node_ptr"])), g["norms_self_loop"]["node_eigenv"].ravel())
    np.testing.assert_array_equal(np.repeat(np.maximum(ee, 1), np.diff(d["edge_ptr"])), g["norms_self_loop"]["edge_eigenv"].ravel())


@pytest.mark.parametrize("case", ["small", "large", "runs"])
def test_match_weights_match_reference_golden(gold_t, case):
    """SURVEY.md 8(f) rank 2: node / edge match weights == the reference's numba loops (dataset.py:54-108)."""
    g = gold_t["match/" + case]
    np.testing.assert_array_equal(OT.subiso_node_weights(g["mats"], g["graph"]), g["node_weights"])
    np.testing.assert_array_equal(OT.subiso_edge_weights(g["mats"], g["pattern"], g["graph"]), g["edge_weights"])
    for a, r in zip(OT.subiso_conjugate(g["mats"], g["pattern"], g["graph"]), g["conj"]):
        assert a.shape == r.shape
        np.testing.assert_array_equal(a, r)
    if case == "runs":      # worked by hand in oracle/gen_golden.py: a later run of the same (u, v) replaces the earlier one
        assert g["edge_weights"].tolist() == [1, 2, 0, 3, 2, 2, 3, 0] and g["node_weights"].tolist() == [3, 3, 2, 1]
        assert g["conj"][0].tolist() == [[6, 4, 5, 1, 1], [6, 4, 5, 1, 1], [0, 6, 1, 1, 1]]


def test_appB_literal_vectors():
    """SURVEY.md App. B, typed in by hand (independent of the generated fixtures)."""
    b = dict(num_graphs=2, node_ptr=np.array([0, 3, 5], np.int32), edge_ptr=np.array([0, 4, 6], np.int32),
             src=np.array([0, 1, 1, 2, 3, 4], np.int32), dst=np.array([1, 0, 2, 1, 4, 3], np.int32),
             vlabel=np.array([1, 2, 1, 2, 2], np.int32), elabel=np.ones(6, np.int32))
    d = OT.tu_add_dummy(b)
    assert list(zip(d["src"][:10], d["dst"][:10])) == [(0, 1), (1, 0), (1, 2), (2, 1), (3, 0), (0, 3), (3, 1), (1, 3), (3, 2), (2, 3)]
    assert d["vlabel"].tolist() == [1, 2, 1, 0, 2, 2, 0] and d["elabel"][:10].tolist() == [1, 1, 1, 1, 0, 0, 0, 0, 0, 0]
    c = OT.tu_conjugate(d)
    assert list(zip(c["src"][:14], c["dst"][:14])) == [(1, 0), (4, 0), (0, 1), (3, 1), (4, 1), (0, 2), (3, 2), (4, 2), (2, 3),
                                                        (4, 3), (1, 4), (0, 4), (3, 4), (2, 4)]
    assert c["vlabel"].tolist() == [1, 1, 1, 1, 0, 1, 1, 0]
    assert c["elabel"].tolist() == [1, 1, 2, 2, 2, 2, 2, 2, 1, 1, 1, 2, 2, 1, 2, 2, 2, 2, 2, 2]
    assert c["eid"].tolist() == [0, 0, 1, 1, 1, 1, 1, 1, 2, 2, 0, 1, 1, 2, 0, 0, 1, 1, 0, 1]
    assert c["v_is_dummy"].tolist() == [0, 0, 0, 0, 1, 0, 0, 1] and not c["e_is_dummy"].any()


@pytest.mark.parametrize("case", ["small", "large", "appB2"])
def test_sub_transforms_match_reference_golden(gold_t, case):
    g = gold_t["sub/" + case]
    cfg = g["cfg"]
    gd = OT.sub_add_dummy(g["graph"], cfg["max_ngv"], cfg["max_ngvl"], cfg["max_nge"], cfg["max_ngel"])
    batches_equal(gd, g["graph_dummy"], SUB_KEYS)
    batches_equal(OT.sub_conjugate(gd), g["graph_conj"], CONJ_KEYS)
    if "pattern" in g:
        pd_ = OT.sub_add_dummy(g["pattern"], cfg["max_npv"], cfg["max_npvl"], cfg["max_npe"], cfg["max_npel"])
        batches_equal(pd_, g["pattern_dummy"], SUB_KEYS)
        batches_equal(OT.sub_conjugate(pd_), g["pattern_conj"], CONJ_KEYS)
    if case == "appB2":   # SURVEY.md App. B second vector, literal
        c = OT.sub_conjugate(gd)
        assert c["vid"].tolist() == [0, 1, 2, 6, 7] and c["vlabel"].tolist() == [0, 1, 0, 2, 3]
        assert list(zip(c["src"], c["dst"])) == [(4, 0), (0, 1), (4, 1), (0, 2), (4, 2), (4, 3), (0, 3), (4, 3), (1, 3), (2, 3), (3, 4)]
        assert c["eid"].tolist() == [0, 1, 1, 1, 1, 0, 1, 1, 2, 2, 4] and c["e_is_dummy"].tolist() == [0] * 10 + [1]


def test_closed_forms_on_random_graphs():
    """count identities: DUMMY V=n+1, E=m+2n (tu_data_processing.py:199-200); CONJ V'=m+1,
    E'=sum_v in(v)out(v)+2m, exactly one label-0 vertex per graph with in = out = m."""
    from dummynode4graphlearning_b200 import synth
    b = synth.tu_batch("proteins", 40, seed=9)
    d = OT.tu_add_dummy(b)
    n, m = np.diff(b["node_ptr"]), np.diff(b["edge_ptr"])
    assert np.array_equal(np.diff(d["node_ptr"]), n + 1) and np.array_equal(np.diff(d["edge_ptr"]), m + 2 * n)
    c = OT.tu_conjugate(d)
    N = int(b["node_ptr"][-1])
    prod = np.bincount(np.repeat(np.arange(len(n)), n), weights=np.bincount(b["dst"], minlength=N) * np.bincount(b["src"], minlength=N)).astype(int)
    assert np.array_equal(np.diff(c["node_ptr"]), m + 1) and np.array_equal(np.diff(c["edge_ptr"]), prod + 2 * m)
    assert (c["elabel"] >= 1).all()
    Vc = int(c["node_ptr"][-1])
    zero = np.flatnonzero(c["vlabel"] == 0)
    assert np.array_equal(zero, c["node_ptr"][1:] - 1)
    assert np.array_equal(np.bincount(c["dst"], minlength=Vc)[zero], m) and np.array_equal(np.bincount(c["src"], minlength=Vc)[zero], m)


@pytest.mark.parametrize("tag", ["RGIN/bdd4", "RGIN/basis_full", "RGIN/basis4_unshared", "DMPNN/node", "DMPNN/node_edge",
                                 "DMPNN/edge_max_nofilter", "RGCN/in_basis", "RGCN/both_bdd4",
                                 "RGCN/none_basis4_bn_unshared", "CompGCN/mult_none", "CompGCN/sub_both_node_edge",
                                 "CompGCN/mult_in_bn_unshared", "CompGCN/corr_out"])
def test_counting_oracle_matches_reference_golden(tag):
    gold = load_golden("counting_models")
    g, b = gold[tag], gold["_batch"]
    sd = {k: v.clone().requires_grad_(v.is_floating_point()) for k, v in g["state_dict"].items()}
    out = OM.counting_model(sd, b["pattern"], b["graph"], oracle_cfg(g["name"], g["kwargs"]))
    for k, ref in g["outputs"].items():
        if ref is None:
            assert out[k] is None, k
        elif ref.dtype == torch.bool:
            assert torch.equal(out[k], ref), k
        elif k in ("pred_v", "pred_e"):
            m = g["outputs"]["g_v_mask" if k == "pred_v" else "g_e_mask"]
            assert_close_rel(out[k].masked_fill(~m, 0), ref.masked_fill(~m, 0), 1e-6, k)
        else:
            assert_close_rel(out[k], ref, 1e-6, k)
    loss = OM.counting_loss(out, torch.from_numpy(b["counts"]), rep_reg_w=1e-3)
    assert_close_rel(loss, g["loss"], 1e-6, "loss")
    loss.backward()
    # shared modules appear under both prefixes in the state_dict; named_parameters() dedupes to the first name.
    # A bias that feeds a BatchNorm has a mathematically zero gradient: only rounding noise is left on both sides (it
    # changes with the BLAS code path of the host), compared against an absolute floor tied to the largest gradient
    gmax = max(float(r.abs().max()) for r in g["grads"].values() if r is not None)
    batch_norm = any(v for k, v in g["kwargs"].items() if k.endswith("_batch_norm"))
    for n, ref in g["grads"].items():
        got = sd[n].grad
        alias = n.replace("g_rep_net", "p_rep_net", 1) if n.startswith("g_rep_net") else None
        if alias in sd and sd[alias].grad is not None and g["kwargs"].get("share_rep_net", True):
            got = got + sd[alias].grad if got is not None else sd[alias].grad
        if ref is None:   # frozen encoder tables / EquivariantEmbedding.row_vec never get a gradient (App. A-13)
            continue
        pre_bn_bias = n.endswith(".bias") and batch_norm and float(ref.abs().max()) <= 1e-6 * gmax
        assert_close_rel(got, ref, 1e-5, "grad " + n, atol=1e-6 * gmax if pre_bn_bias else 0.0)


@pytest.mark.parametrize("tag", ["GIN/mutag_dummy", "GIN/mutag_conj_eps", "RGIN/mutag_dummy"])
def test_classification_oracle_matches_reference_golden(tag):
    import torch.nn.functional as F
    g = load_golden("classification_models.pt")[tag]
    sd = {k: v.clone().requires_grad_(v.is_floating_point()) for k, v in g["state_dict"].items()}
    d, a = g["data"], g["args"]
    nl = a["additional"].get("num_layers", 2)
    B = int(d["node_ptr"].numel()) - 1
    if g["name"] == "GIN":
        out = OM.gin_classifier(sd, d["x"], d["edge_index"], d["batch"], B, nl, a["additional"].get("aggregation", "sum"))
    else:
        out = OM.rgin_classifier(sd, d["x"], d["edge_index"], d["edge_attr"].max(1)[1], d["batch"], B, nl, a["num_relations"])
    assert_close_rel(out, g["out"], 1e-6, "log_softmax")
    loss = F.nll_loss(out, d["y"])
    assert_close_rel(loss, g["loss"], 1e-6, "loss")
    loss.backward()
    for n, ref in g["grads"].items():
        if ref is None:
            continue
        got = sd[n].grad
        # nns.i.* and convs.i.nn.* alias the same parameters (gconv.py:195-197); the oracle reads nns.*
        if got is None and n.startswith("convs.") and ".nn." in n:
            got = sd[n.replace("convs.", "nns.").replace(".nn.", ".")].grad
        assert_close_rel(got, ref, 2e-5, "grad " + n, atol=2e-5)
