"""GPU parity of the drop-in modules (through the C ABI kernels) against
 (1) the golden vectors produced by the UNMODIFIED reference classes (tests/golden/, oracle/gen_golden.py), and
 (2) the oracle restatement on larger seeded batches,
for forward values, loss and every parameter gradient.  Tolerance: 1e-5 relative (BASELINE.json north_star)
measured as max-abs error over max-abs reference value per tensor (SURVEY.md section 2.2's measure)."""
from argparse import Namespace

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import record_error
from helpers import assert_close_rel, load_golden, oracle_cfg, rel_err

pytestmark = pytest.mark.gpu

TOL = 1e-5


def _counting_model(name, kw, state_dict, device):
    from dummynode4graphlearning_b200.subgraph_isomorphism.models import DMPNN, RGCN, RGIN, CompGCN
    model = {"RGIN": RGIN, "DMPNN": DMPNN, "RGCN": RGCN, "CompGCN": CompGCN}[name](**kw)
    missing, unexpected = model.load_state_dict(state_dict, strict=True)   # key compatibility (App. A-12)
    assert not missing and not unexpected
    return model.to(device).train()


def _loss(out, counts, rep_reg_w=1e-3):
    crit = lambda pred, target, slp: F.mse_loss(F.leaky_relu(pred, slp), target)
    loss = crit(out["pred_c"], counts.float().view(-1, 1), 0.01)
    reg = 0.0
    for k in ("p_v_rep", "p_e_rep", "g_v_rep", "g_e_rep"):
        if out[k] is not None:
            reg = reg + crit(out[k], torch.zeros_like(out[k]), 1) * out[k].size(1)
    return loss + rep_reg_w * reg


def _check_outputs(out, ref):
    for k, r in ref.items():
        if r is None:
            assert out[k] is None, k
        elif r.dtype == torch.bool:
            assert torch.equal(out[k].cpu(), r), k
        elif k in ("pred_v", "pred_e"):   # padded / masked positions are don't-care (train.py:783-784 zero them)
            m = ref["g_v_mask" if k == "pred_v" else "g_e_mask"]
            assert_close_rel(out[k].cpu().masked_fill(~m, 0), r.masked_fill(~m, 0), TOL, k)
        else:
            assert_close_rel(out[k], r, TOL, k)


@pytest.mark.parametrize("tag", ["RGIN/bdd4", "RGIN/basis_full", "RGIN/basis4_unshared", "DMPNN/node", "DMPNN/node_edge",
                                 "DMPNN/edge_max_nofilter", "RGCN/in_basis", "RGCN/both_bdd4",
                                 "RGCN/none_basis4_bn_unshared", "CompGCN/mult_none", "CompGCN/sub_both_node_edge",
                                 "CompGCN/mult_in_bn_unshared", "CompGCN/corr_out"])
def test_counting_models_match_reference_golden(device, tag):
    from dummynode4graphlearning_b200.graph import BatchedGraph
    gold = load_golden("counting_models")
    g, b = gold[tag], gold["_batch"]
    model = _counting_model(g["name"], g["kwargs"], g["state_dict"], device)
    pattern = BatchedGraph.from_batch(b["pattern"], device)
    graph = BatchedGraph.from_batch(b["graph"], device)
    out = model(pattern, graph)
    _check_outputs(out, g["outputs"])
    loss = _loss(out, torch.from_numpy(b["counts"]).to(device))
    record_error("counting_golden[%s]" % tag, "loss", err=rel_err(loss, g["loss"]))
    record_error("counting_golden[%s]" % tag, "pred_c", err=rel_err(out["pred_c"], g["outputs"]["pred_c"]))
    assert_close_rel(loss, g["loss"], TOL, "loss")
    loss.backward()
    grads = dict(model.named_parameters())
    assert set(grads) == set(g["grads"])
    # a bias that feeds a BatchNorm (RGCNLayer with batch_norm, rgcn.py:183-186) has a mathematically zero gradient:
    # only rounding noise is left on both sides, compared against an absolute floor tied to the largest gradient
    gmax = max(float(r.abs().max()) for r in g["grads"].values() if r is not None)
    for n, ref in g["grads"].items():
        if ref is None:
            assert grads[n].grad is None, n     # frozen tables / row_vec stay gradient-free
        else:
            record_error("counting_golden[%s]" % tag, "grad " + n, err=rel_err(grads[n].grad, ref) if float(ref.abs().max()) > 1e-6 * gmax else 0.0)
            assert_close_rel(grads[n].grad, ref, TOL, "grad " + n, atol=1e-6 * gmax if n.endswith(".bias") else 0.0)


@pytest.mark.parametrize("name,shape,bs,over", [
    ("RGIN", "small", 64, {}),
    ("RGIN", "small", 512, dict(rep_rgin_regularizer="basis", rep_rgin_num_bases=-1)),   # BASELINE config C3, batch 512
    ("DMPNN", "small", 64, dict(node_pred=True, edge_pred=True, pred_return_weights="node,edge")),
    ("DMPNN", "large", 8, dict(node_pred=True, edge_pred=False)),                        # BASELINE config C4 shapes
    ("RGCN", "small", 64, dict(rep_rgcn_edge_norm="both", rep_rgcn_regularizer="bdd", rep_rgcn_num_bases=4)),   # 8(f) rank 1
    ("CompGCN", "small", 64, dict(rep_compgcn_comp_opt="mult", rep_compgcn_edge_norm="both", node_pred=True, edge_pred=True)),
    ("CompGCN", "large", 8, dict(rep_compgcn_comp_opt="sub", rep_compgcn_edge_norm="in")),
])
def test_counting_models_match_oracle_live(device, name, shape, bs, over):
    from dummynode4graphlearning_b200 import synth, transforms as T
    from dummynode4graphlearning_b200.graph import BatchedGraph
    from dummynode4graphlearning_b200.subgraph_isomorphism.models import DMPNN, RGCN, RGIN, CompGCN
    from oracle import models as OM

    p, g, counts = synth.counting_batch(shape, bs, seed=5)
    cfg = dict(synth.counting_config(shape), add_dummy=True)
    mc = T.process_model_config(cfg)
    # augmentation on the GPU (already bit-exact with the reference, test_transforms_gpu.py)
    pd_ = T.sub_add_dummy(T.to_device(p, device), cfg["max_npv"], cfg["max_npvl"], cfg["max_npe"], cfg["max_npel"])
    gd_ = T.sub_add_dummy(T.to_device(g, device), cfg["max_ngv"], cfg["max_ngvl"], cfg["max_nge"], cfg["max_ngel"])
    kw = dict({k: v for k, v in mc.items() if k.startswith("max_")}, hid_dim=64, rep_num_graph_layers=3,
              rep_num_pattern_layers=3, rep_act_func="leaky_relu", pred_act_func="leaky_relu", pred_net="SumPredictNet",
              pred_hid_dim=64, emb_net="Equivariant", enc_net="Multihot", filter_net="ScalarFilter", pred_with_enc=True,
              pred_with_deg=True, rep_rgin_regularizer="bdd", rep_rgin_num_bases=4, pred_return_weights="node",
              init_neigenv=4.0, init_eeigenv=4.0)
    kw.update(over)
    torch.manual_seed(1)
    model = {"RGIN": RGIN, "DMPNN": DMPNN, "RGCN": RGCN, "CompGCN": CompGCN}[name](**kw)
    with torch.no_grad():
        for n, q in model.named_parameters():
            if "pred_fc2" in n or "weight_fc2" in n:
                q.normal_(0.0, 0.1)
    sd = {k: v.clone().requires_grad_(v.is_floating_point() and "enc_net" not in k) for k, v in model.state_dict().items()}
    model = model.to(device).train()
    pattern, graph = BatchedGraph.from_batch(pd_, device), BatchedGraph.from_batch(gd_, device)
    out = model(pattern, graph)
    loss = _loss(out, torch.from_numpy(counts).to(device))
    loss.backward()

    host = lambda b: {k: (v.cpu().numpy() if isinstance(v, torch.Tensor) else v) for k, v in b.items()}
    ref = OM.counting_model(sd, host(pd_), host(gd_), oracle_cfg(name, kw))
    ref_loss = OM.counting_loss(ref, torch.from_numpy(counts), rep_reg_w=1e-3)
    ref_loss.backward()
    _check_outputs(out, {k: (v.detach() if isinstance(v, torch.Tensor) else None) for k, v in ref.items()})
    # The oracle above is fp32 like the reference, i.e. it carries its own rounding error; the same oracle in float64 is
    # the exact value of the reference's formulas.  A quantity passes if it is within TOL of the fp32 oracle, or at least
    # as close to the exact value as 2x the fp32 oracle's own distance from it (deep sums over 512-node graphs put the
    # fp32 CPU evaluation itself ~1e-5 away from exact).
    sd64 = {k: (v.detach().double().requires_grad_(v.requires_grad) if v.is_floating_point() else v.detach().clone())
            for k, v in sd.items()}
    ref64 = OM.counting_model(sd64, host(pd_), host(gd_), oracle_cfg(name, kw))
    ref64_loss = OM.counting_loss(ref64, torch.from_numpy(counts), rep_reg_w=1e-3)
    ref64_loss.backward()

    tname = "counting_live[%s-%s-%d]" % (name, shape, bs)

    def close(mine, r32, r64, what):
        e32 = rel_err(mine, r32)
        record_error(tname, what, err=e32, err_vs_fp64=rel_err(mine, r64), fp32_oracle_vs_fp64=rel_err(r32, r64))
        if e32 <= TOL:
            return
        e_mine, e_ref = rel_err(mine, r64), rel_err(r32, r64)
        assert e_mine <= max(TOL, 2 * e_ref), "%s: vs fp32 oracle %.2e, vs float64 %.2e (fp32 oracle itself %.2e)" % (
            what, e32, e_mine, e_ref)

    close(loss, ref_loss, ref64_loss, "loss")
    for n, q in model.named_parameters():
        if not q.requires_grad or q.grad is None:
            continue
        r, r64 = sd[n].grad, sd64[n].grad
        alias = n.replace("g_rep_net", "p_rep_net", 1) if n.startswith("g_rep_net") else None
        if alias in sd and sd[alias].grad is not None and kw.get("share_rep_net", True):
            r = r + sd[alias].grad if r is not None else sd[alias].grad
            r64 = r64 + sd64[alias].grad if r64 is not None else sd64[alias].grad
        close(q.grad, r, r64, "grad " + n)


@pytest.mark.parametrize("tag", ["GIN/mutag_dummy", "GIN/mutag_conj_eps", "RGIN/mutag_dummy"])
def test_classifiers_match_reference_golden(device, tag):
    from dummynode4graphlearning_b200.graph_classification.data import Batch
    from dummynode4graphlearning_b200.graph_classification.models import GIN, RGIN
    g = load_golden("classification_models.pt")[tag]
    args = Namespace(**g["args"])
    model = {"GIN": GIN, "RGIN": RGIN}[g["name"]](args)
    missing, unexpected = model.load_state_dict(g["state_dict"], strict=True)
    assert not missing and not unexpected
    model = model.to(device).train()
    d = {k: v.to(device) for k, v in g["data"].items()}
    data = Batch(d["x"], d["edge_index"], d["batch"], d["edge_attr"], d["y"], node_ptr=d["node_ptr"])
    out = model(data)
    assert_close_rel(out, g["out"], TOL, "log_softmax")
    loss = F.nll_loss(out, d["y"])
    assert_close_rel(loss, g["loss"], TOL, "loss")
    loss.backward()
    params = dict(model.named_parameters())
    assert set(params) == set(g["grads"])
    # a bias in front of a BatchNorm has a mathematically zero gradient (only rounding noise on both sides): those are
    # compared against an absolute floor tied to the LARGEST gradient of the model, everything else relatively at 1e-5
    gmax = max(float(r.abs().max()) for r in g["grads"].values() if r is not None)
    record_error("classifier_golden[%s]" % tag, "log_softmax", err=rel_err(out, g["out"]))
    record_error("classifier_golden[%s]" % tag, "loss", err=rel_err(loss, g["loss"]))
    for n, ref in g["grads"].items():
        if ref is not None:
            pre_bn_bias = float(ref.abs().max()) <= 1e-6 * gmax
            if not pre_bn_bias:
                record_error("classifier_golden[%s]" % tag, "grad " + n, err=rel_err(params[n].grad, ref))
            assert_close_rel(params[n].grad, ref, TOL, "grad " + n, atol=1e-6 * gmax if pre_bn_bias else 0.0)


def test_gin_full_size_c2_against_oracle(device):
    """BASELINE config C2 at full size: CONJ transform (GPU) of 1113 PROTEINS-shaped graphs + GIN (hid 32, 4 layers)
    forward/backward.  The synthetic CONJ features are degenerate (two distinct one-hot rows), so several BatchNorm
    channels have ~zero variance and amplify fp32 rounding by 1/sqrt(eps) per layer: two correct fp32
    implementations differ by far more than 1e-5 here.  The size-independent criterion is therefore accuracy against
    exact arithmetic: the float64 oracle is the ground truth, and the CUDA path must be as close to it as the
    fp32 CPU oracle (the reference's own arithmetic) is, within a factor 4."""
    from dummynode4graphlearning_b200 import synth, transforms as T
    from dummynode4graphlearning_b200.graph_classification.data import Batch
    from dummynode4graphlearning_b200.graph_classification.models import GIN
    from oracle import models as OM

    raw = synth.tu_batch("proteins", seed=0)
    conj = T.tu_conjugate(T.tu_add_dummy(T.to_device(raw, device)))
    conj.pop("eattr", None); conj["has_edge_labels"] = True
    can = T.pyg_canonicalize(conj)
    data = Batch.from_canonical(can)
    args = Namespace(num_features=can["x"].size(1), hidden_dim=32, num_classes=2, dropout_ratio=0.0,
                     additional={"train_eps": True, "num_layers": 4, "aggregation": "sum"}, epochs=3, device=str(device))
    torch.manual_seed(0)
    model = GIN(args)
    base = model.state_dict()

    def oracle_run(dtype):
        sd = {k: (v.clone().to(dtype).requires_grad_("running" not in k) if v.is_floating_point() else v.clone())
              for k, v in base.items()}
        ref = OM.gin_classifier(sd, can["x"].cpu().to(dtype), can["edge_index"].cpu(), can["batch"].cpu(),
                                can["num_graphs"], 4, "sum")
        loss = F.nll_loss(ref, can["y"].cpu())
        loss.backward()
        return ref.detach(), loss.detach(), sd

    r64, l64, sd64 = oracle_run(torch.float64)
    r32, l32, sd32 = oracle_run(torch.float32)
    model = model.to(device).train()
    out = model(data)
    loss = F.nll_loss(out, can["y"])
    loss.backward()

    def err(a, b):
        return float((a.detach().double().cpu() - b.double()).abs().max() / (b.double().abs().max() + 1e-30))

    assert err(out, r64) <= 4 * err(r32, r64) + 1e-5, (err(out, r64), err(r32, r64))
    assert err(loss, l64) <= 4 * err(l32, l64) + 1e-5
    for n, q in model.named_parameters():
        key = n if sd64[n].grad is not None else n.replace("convs.", "nns.").replace(".nn.", ".")
        g64, g32 = sd64[key].grad, sd32[key].grad
        scale = float(g64.abs().max())
        e_gpu = float((q.grad.double().cpu() - g64).abs().max())
        e_cpu = float((g32.double() - g64).abs().max())
        assert e_gpu <= 4 * e_cpu + 1e-5 * max(scale, 1e-3), (n, e_gpu, e_cpu, scale)


def _full_size_classification(device, mode, hid, layers, train=True, dropout=0.0, seed=0, graphs=None):
    """PROTEINS-shaped batch -> GPU transform -> (model on the GPU, canonical batch, oracle runner)."""
    from dummynode4graphlearning_b200 import synth, transforms as T
    from dummynode4graphlearning_b200.graph_classification.data import Batch
    from dummynode4graphlearning_b200.graph_classification.models import GIN
    from oracle import models as OM
    raw = synth.tu_batch("proteins", graphs, seed=seed)
    b = T.tu_add_dummy(T.to_device(raw, device))
    if mode == "conj":
        b = T.tu_conjugate(b)
        b.pop("eattr", None)
    b["has_edge_labels"] = True
    can = T.pyg_canonicalize(b)
    data = Batch.from_canonical(can)
    args = Namespace(num_features=can["x"].size(1), hidden_dim=hid, num_classes=2, dropout_ratio=dropout,
                     additional={"train_eps": True, "num_layers": layers, "aggregation": "sum"}, epochs=3, device=str(device))
    torch.manual_seed(0)
    model = GIN(args)
    base = model.state_dict()

    def oracle_run(dtype, training=True):
        sd = {k: (v.clone().to(dtype).requires_grad_("running" not in k) if v.is_floating_point() else v.clone())
              for k, v in base.items()}
        ref = OM.gin_classifier(sd, can["x"].cpu().to(dtype), can["edge_index"].cpu(), can["batch"].cpu(),
                                can["num_graphs"], layers, "sum", training=training)
        loss = F.nll_loss(ref, can["y"].cpu())
        if training:
            loss.backward()
        return ref.detach(), loss.detach(), sd

    return model.to(device), data, can, oracle_run


@pytest.mark.parametrize("hid,layers", [(32, 4), (128, 2)])
def test_gin_full_size_dummy_proteins_meets_1e5(device, hid, layers):
    """The full-size C2-sized batch on NON-degenerate inputs (DUMMY_PROTEINS features: scalar attribute + 3 labels + dummy
    flag; the CONJ features of test_gin_full_size_c2_against_oracle are two one-hot rows): here no BatchNorm channel has
    ~zero variance and the CUDA path is held to the north star's 1e-5 directly against the fp32 CPU oracle, for the
    log-probabilities, the loss and every gradient.  hid 128 = main.py:174's default width (tensor-core GEMM +
    stand-alone fixed-order BatchNorm kernels, ops.gin_mlp_wide; hid 32 = the fused stages)."""
    model, data, can, oracle_run = _full_size_classification(device, "dummy", hid, layers)
    r32, l32, sd32 = oracle_run(torch.float32)
    r64, l64, sd64 = oracle_run(torch.float64)
    model.train()
    out = model(data)
    loss = F.nll_loss(out, can["y"])
    loss.backward()
    tname = "gin_full_size_dummy_proteins[hid%d]" % hid
    record_error(tname, "log_softmax", err=rel_err(out, r32), err_vs_fp64=rel_err(out, r64), fp32_oracle_vs_fp64=rel_err(r32, r64))
    record_error(tname, "loss", err=rel_err(loss, l32), err_vs_fp64=rel_err(loss, l64), fp32_oracle_vs_fp64=rel_err(l32, l64))
    assert_close_rel(out, r32, TOL, "log_softmax")
    assert_close_rel(loss, l32, TOL, "loss")
    gmax = max(float(v.grad.abs().max()) for v in sd32.values() if getattr(v, "grad", None) is not None)
    for n, q in model.named_parameters():
        key = n if sd32[n].grad is not None else n.replace("convs.", "nns.").replace(".nn.", ".")
        ref, ref64 = sd32[key].grad, sd64[key].grad
        pre_bn_bias = float(ref64.abs().max()) <= 1e-6 * gmax          # zero by construction: rounding noise on both sides
        if not pre_bn_bias:
            record_error(tname, "grad " + n, err=rel_err(q.grad, ref), err_vs_fp64=rel_err(q.grad, ref64),
                         fp32_oracle_vs_fp64=rel_err(ref, ref64))
        # Gradients of the BatchNorm parameters and of the weights in front of them are sums over 4.5e4 rows with heavy
        # cancellation: the fp32 CPU oracle itself is 1e-5 .. 2e-4 away from float64 on them (recorded in
        # profiles/*parity_errors*.json).  The bar applies to the distance from the oracle OR, where the oracle's own
        # rounding dominates, to the distance from the exact (float64) value relative to the oracle's own distance
        e32, e64, eref = rel_err(q.grad, ref), rel_err(q.grad, ref64), rel_err(ref, ref64)
        if pre_bn_bias:      # both sides are rounding noise around an exact zero (the fp32 CPU oracle's is ~1e-6 * gmax itself)
            assert float(q.grad.abs().max()) <= 1e-5 * gmax and float(ref.abs().max()) <= 1e-5 * gmax, n
        else:
            assert e32 <= TOL or e64 <= max(TOL, 4 * eref), (n, e32, e64, eref)     # factor as in the C2 test below


def test_gin_eval_mode_and_dropout_paths(device):
    """eval mode (running statistics, no batch statistics: the unfused branch) against the oracle, and dropout > 0 in
    training mode: same mask stream as torch's F.dropout on this device is not required by the reference -- the check is
    that the fused-path switch is taken off and the result is finite, deterministic under a fixed seed and different from
    the dropout-free result."""
    model, data, can, oracle_run = _full_size_classification(device, "dummy", 32, 3, graphs=64, seed=3)
    model.train()
    for _ in range(2):                      # move the running statistics away from their initial values
        model(data)
    sd_after = {k: v.detach().cpu().clone() for k, v in model.state_dict().items()}
    model.eval()
    with torch.no_grad():
        out_eval = model(data)
    from oracle import models as OM
    ref = OM.gin_classifier(sd_after, can["x"].cpu(), can["edge_index"].cpu(), can["batch"].cpu(), can["num_graphs"], 3, "sum",
                            training=False)
    record_error("gin_eval_mode", "log_softmax", err=rel_err(out_eval, ref))
    assert_close_rel(out_eval, ref, TOL, "eval-mode log_softmax")
    model_d, data_d, _, _ = _full_size_classification(device, "dummy", 32, 3, dropout=0.5, graphs=64, seed=3)
    model_d.train()
    torch.manual_seed(7)
    a = model_d(data_d)
    torch.manual_seed(7)
    b = model_d(data_d)
    assert torch.isfinite(a).all() and torch.equal(a, b)
    model.train()
    assert not torch.allclose(a, model(data), atol=1e-3)
