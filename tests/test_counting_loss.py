"""CPU: the full back-propagated loss of the counting path (SURVEY.md 8(a21): count term + representation regulariser
+ match terms, three criteria, clipping) against goldens produced by the reference's OWN ``train_epoch``
(tests/golden/counting_loss.pt, oracle/gen_golden.py::gen_counting_loss).  The forward here is the oracle model; the
loss under test is the product's ``losses.counting_bp_loss`` (pure tensor code)."""
import pytest
import torch

from dummynode4graphlearning_b200.subgraph_isomorphism.losses import bp_criterion, counting_bp_loss, eval_criterion
from helpers import assert_close_rel, load_golden, oracle_cfg
from oracle import models as OM

CASES = ["DMPNN/node_edge|MSE", "DMPNN/node_edge|MAE", "DMPNN/node_edge|SMSE", "RGIN/bdd4|MSE"]


def golden_grads_by_name(sd, names, shared):
    """gradients of the oracle's leaf tensors under the reference's parameter names (shared nets are listed once there)."""
    out = {}
    for n in names:
        g = sd[n].grad
        alias = n.replace("g_rep_net", "p_rep_net", 1) if n.startswith("g_rep_net") else None
        if shared and alias in sd and sd[alias].grad is not None:
            g = sd[alias].grad if g is None else g + sd[alias].grad
        out[n] = g
    return out


@pytest.mark.parametrize("tag", CASES)
def test_bp_loss_matches_reference_train_epoch_golden(tag):
    gold, base = load_golden("counting_loss.pt"), load_golden("counting_models")
    g, b = gold[tag], base["_batch"]
    m, c = base[g["model"]], g["conf"]
    sd = {k: v.clone().requires_grad_(v.is_floating_point()) for k, v in g["state_dict"].items()}
    out = OM.counting_model(sd, b["pattern"], b["graph"], oracle_cfg(m["name"], m["kwargs"]))
    loss, terms = counting_bp_loss(out, torch.from_numpy(b["counts"]), gold["_node_weights"], gold["_edge_weights"], None,
                                   bp_loss=c["bp_loss"], neg_slp=c["neg_pred_slp"], rep_reg_w=c["rep_reg_w"],
                                   match_loss_w=c["match_loss_w"], match_reg_w=c["match_reg_w"])
    assert abs(float(loss.detach()) - g["loss"]) <= 2e-6 * abs(g["loss"])
    assert float(terms["match_v_loss"]) > 0 and float(terms["match_v_reg"]) > 0 and float(terms["rep_reg"]) > 0
    if out["pred_e"] is not None:
        assert float(terms["match_e_loss"]) > 0 and float(terms["match_e_reg"]) > 0
    metric = eval_criterion("MAE")(out["pred_c"].detach(), torch.from_numpy(b["counts"]).float().view(-1, 1))
    assert abs(float(metric) - g["eval_metric"]) <= 2e-6 * abs(g["eval_metric"])
    loss.backward()
    names = [n for n, r in g["grads"].items() if r is not None]
    mine = golden_grads_by_name(sd, names, m["kwargs"].get("share_rep_net", True))
    if c.get("max_grad_norm", 0) > 0:                                    # train.py:833-834, clip_grad_norm_
        total = torch.sqrt(sum((v.double() ** 2).sum() for v in mine.values())).float()
        coef = (c["max_grad_norm"] / (total + 1e-6)).clamp(max=1.0)
        mine = {n: v * coef for n, v in mine.items()}
    for n in names:
        assert_close_rel(mine[n], g["grads"][n], 1e-5, "grad " + n)


def test_criteria_and_missing_heads():
    x, t = torch.tensor([[-2.0], [3.0]]), torch.tensor([[1.0], [1.0]])
    assert float(bp_criterion("MSE")(x, t, 0.5)) == pytest.approx(((-1 - 1) ** 2 + (3 - 1) ** 2) / 2)
    assert float(bp_criterion("MAE")(x, t, 0.0)) == pytest.approx((1 + 2) / 2)
    assert float(eval_criterion("MSE")(x, t)) == pytest.approx((1 + 4) / 2)
    with pytest.raises(NotImplementedError):
        bp_criterion("AUC")
    out = dict(pred_c=x.clone().requires_grad_(True), pred_v=None, pred_e=None, p_v_rep=None, p_e_rep=None, g_v_rep=None,
               g_e_rep=None, g_v_mask=None, g_e_mask=None)
    loss, terms = counting_bp_loss(out, torch.tensor([1, 1]), node_weights=torch.ones(2, 3), match_loss_w=1.0)
    assert float(loss.detach()) == pytest.approx(float(bp_criterion("MSE")(x, t, 0.01))) and float(terms["match_v_loss"]) == 0.0


def test_scheduled_value_known_answers():
    """config.py defaults: the negative slope anneals 1.0 -> 0.01 over the first half of each of two cycles."""
    from dummynode4graphlearning_b200.subgraph_isomorphism.losses import scheduled_value
    spec = "anneal_cosine$1.0$0.01"
    assert scheduled_value(spec, 0, 1000) == 1.0
    assert scheduled_value(spec, 125, 1000) == pytest.approx(1.0 + (0.01 - 1.0) * 0.5)        # quarter of a cycle: midpoint
    assert scheduled_value(spec, 250, 1000) == 0.01 and scheduled_value(spec, 400, 1000) == 0.01
    assert scheduled_value(spec, 500, 1000) == 1.0                                          # second cycle restarts
    assert scheduled_value(spec, 2000, 1000) == 0.01
    assert scheduled_value("cyclical_linear$0.0$1.0", 375, 1000) == pytest.approx(0.5)        # on the way back
    assert scheduled_value(0.3, 5, 10) == 0.3
