"""GPU: the counting models' full back-propagated loss (count term + representation regulariser + match terms, SURVEY.md
8(a21)) through the product modules and the C-ABI kernels, against the goldens the reference's OWN train_epoch produced
(tests/golden/counting_loss.pt): loss value and every parameter gradient, 1e-5 relative."""
import numpy as np
import pytest
import torch

from conftest import record_error

from helpers import rel_err, assert_close_rel, load_golden

pytestmark = pytest.mark.gpu

CASES = ["DMPNN/node_edge|MSE", "DMPNN/node_edge|MAE", "DMPNN/node_edge|SMSE", "RGIN/bdd4|MSE"]


def _model(name, kw, sd, device):
    from dummynode4graphlearning_b200.subgraph_isomorphism import models as PM
    model = getattr(PM, name)(**kw)
    missing, unexpected = model.load_state_dict(sd, strict=True)
    assert not missing and not unexpected
    return model.to(device).train()


@pytest.mark.parametrize("tag", CASES)
def test_full_bp_loss_matches_reference_train_epoch_golden(device, tag):
    from dummynode4graphlearning_b200.graph import BatchedGraph
    from dummynode4graphlearning_b200.subgraph_isomorphism.losses import counting_bp_loss
    gold, base = load_golden("counting_loss.pt"), load_golden("counting_models")
    g, b = gold[tag], base["_batch"]
    m, c = base[g["model"]], g["conf"]
    model = _model(m["name"], m["kwargs"], g["state_dict"], device)
    pattern, graph = BatchedGraph.from_batch(b["pattern"], device), BatchedGraph.from_batch(b["graph"], device)
    out = model(pattern, graph)
    loss, terms = counting_bp_loss(out, torch.from_numpy(b["counts"]).to(device), gold["_node_weights"].to(device),
                                   gold["_edge_weights"].to(device), model=model, bp_loss=c["bp_loss"],
                                   neg_slp=c["neg_pred_slp"], rep_reg_w=c["rep_reg_w"], match_loss_w=c["match_loss_w"],
                                   match_reg_w=c["match_reg_w"])
    assert abs(float(loss.detach()) - g["loss"]) <= 1e-5 * abs(g["loss"])
    assert float(terms["match_v_loss"]) > 0 and float(terms["match_v_reg"]) > 0
    loss.backward()
    params = dict(model.named_parameters())
    assert set(params) == set(g["grads"])
    if c.get("max_grad_norm", 0) > 0:
        torch.nn.utils.clip_grad_norm_(model.parameters(), c["max_grad_norm"])
    gmax = max(float(r.abs().max()) for r in g["grads"].values() if r is not None)
    for n, ref in g["grads"].items():
        if ref is None:
            assert params[n].grad is None, n
        else:
            # 1e-5 per tensor (max-abs error / max-abs reference), with an absolute floor tied to the LARGEST gradient of the
            # model: a tensor whose own scale is far below that (embedding tables behind three layers) is dominated by the
            # rounding of the sums it is the small difference of -- the reference's fp32 value carries the same noise.  The
            # measured errors are in profiles/*parity_errors*.json (largest: 1.2e-5 on g_emb_net.vl.weight, SMSE case).
            record_error("bp_loss_golden[%s]" % tag, "grad " + n, err=rel_err(params[n].grad, ref),
                         tensor_scale_over_gmax=float(ref.abs().max()) / gmax)
            assert_close_rel(params[n].grad, ref, 1e-5, "grad " + n, atol=2e-6 * gmax)


def test_pipeline_step_with_match_weights(device):
    """CountingPipeline.train_on(..., node_weights=, edge_weights=) == model + match_loss_fn composed by hand, with the
    flat weights produced by the batched match-weight kernels on the augmented batch."""
    from dummynode4graphlearning_b200 import synth, transforms as T
    from dummynode4graphlearning_b200.pipelines import CountingPipeline
    from dummynode4graphlearning_b200.subgraph_isomorphism import matching as M
    from dummynode4graphlearning_b200.subgraph_isomorphism.models import DMPNN
    B = 12
    p, g, counts = synth.counting_batch("small", B, seed=9)
    mats = M.add_dummy_to_subisomorphisms(synth.random_subisomorphisms(p, g, seed=9), g)
    cfg = dict(synth.counting_config("small"), add_dummy=True)
    mc = T.process_model_config(cfg)
    kw = dict({k: v for k, v in mc.items() if k.startswith("max_")}, hid_dim=32, rep_num_graph_layers=2,
              rep_num_pattern_layers=2, pred_hid_dim=32, emb_net="Equivariant", filter_net="ScalarFilter",
              pred_return_weights="node,edge", node_pred=True, edge_pred=True)

    def fresh():
        torch.manual_seed(4)
        model = DMPNN(**kw)
        with torch.no_grad():
            for n, q in model.named_parameters():
                if "fc2" in n:
                    q.normal_(0.0, 0.05)
        model = model.to(device)
        opt = torch.optim.SGD(model.parameters(), lr=0.0)
        return model, CountingPipeline(model, opt, cfg, rep_reg_w=1e-3, max_grad_norm=0.0, cuda_graphs=False,
                                       match_loss_w=0.5, match_reg_w=0.25, share_emb_net=False)   # goldens: per-side maxima

    model, pipe = fresh()
    pattern, graph = pipe.transform(T.to_device(p, device), T.to_device(g, device))
    p_aug = T.sub_add_dummy(T.to_device(p, device), cfg["max_npv"], cfg["max_npvl"], cfg["max_npe"], cfg["max_npel"])
    g_aug = T.sub_add_dummy(T.to_device(g, device), cfg["max_ngv"], cfg["max_ngvl"], cfg["max_nge"], cfg["max_ngel"])
    sub = M.pack_subisomorphisms(mats, device)
    nw, ew = M.node_weights(sub, g_aug), M.edge_weights(sub, p_aug, g_aug)
    assert nw.numel() == graph.number_of_nodes() and ew.numel() == graph.number_of_edges() and int(nw.sum()) > 0
    c_dev = torch.from_numpy(counts).to(device)
    loss = pipe.train_on(pattern, graph, c_dev, node_weights=nw, edge_weights=ew)
    grads = {n: q.grad.clone() for n, q in model.named_parameters() if q.grad is not None}

    model2, pipe2 = fresh()
    pattern2, graph2 = pipe2.transform(T.to_device(p, device), T.to_device(g, device))
    out = model2(pattern2, graph2)
    manual = pipe2.match_loss_fn(out, c_dev, graph2, nw, ew)
    plain = pipe2.loss_fn(model2(pattern2, graph2), c_dev)
    manual.backward()
    assert_close_rel(loss, manual.detach(), 1e-6, "pipeline loss with match terms")
    assert float((manual.detach() - plain.detach()).abs()) > 0, "match terms must contribute"
    for n, q in model2.named_parameters():
        if q.grad is not None:
            assert_close_rel(grads[n], q.grad, 1e-6, "grad " + n)
    assert np.isfinite(float(loss))
