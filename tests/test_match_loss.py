"""CPU: the fused match loss of the counting models (csrc/match.cu) restated in float64 in closed form -- value, gradient
of every prediction position and of pred_c -- and tied to ``losses.counting_bp_loss`` under float64 autograd on padded,
masked inputs with negative pred_c and exact ties; the host offsets of the dummy column; argument checks."""
import numpy as np
import pytest
import torch

from dummynode4graphlearning_b200.subgraph_isomorphism.losses import bp_criterion, counting_bp_loss

CRITERIA = ("MAE", "MSE", "SMSE")


def crit_value(crit, d):
    a = np.abs(d)
    if crit == "MAE":
        return a
    if crit == "MSE":
        return d * d
    return np.where(a < 1.0, 0.5 * d * d, a - 0.5)


def crit_grad(crit, d):
    """derivative in d with torch's conventions: sign(0) = 0, smooth-L1 (beta 1) quadratic for |d| < 1."""
    if crit == "MAE":
        return np.sign(d)
    if crit == "MSE":
        return 2.0 * d
    return np.clip(d, -1.0, 1.0)


def pad_left(w, seg_ptr, L):
    """flat per-row weights -> (B, L) left-padded with zeros (pad_match_weights)."""
    B = len(seg_ptr) - 1
    out = np.zeros((B, L))
    for b in range(B):
        n = int(seg_ptr[b + 1] - seg_ptr[b])
        if n:
            out[b, L - n:] = w[seg_ptr[b]:seg_ptr[b + 1]]
    return out


def match_loss_f64(pred_c, kinds, crit, neg_slp, match_loss_w, match_reg_w):
    """float64 restatement of dn4gl_match_loss_f32 / _bwd_f32.  pred_c (B,); kinds: per present kind (pred (B, L),
    mask (B, L) bool, flat weights (N,), seg_ptr (B + 1)).  -> (loss, [gradient of each kind's pred], gradient of pred_c)
    for an upstream gradient of 1."""
    pred_c = np.asarray(pred_c, np.float64).reshape(-1)
    B = pred_c.size
    s_loss = s_reg = 0.0
    g_c = np.zeros(B)
    grads = []
    for pred, mask, w, seg in kinds:
        pred, mask = np.asarray(pred, np.float64), np.asarray(mask, bool)
        p = np.where(mask, pred, 0.0)                              # masked and padded positions: prediction 0 ...
        t = np.where(mask, pad_left(np.asarray(w, np.float64), np.asarray(seg), pred.shape[1]), 0.0)   # ... target 0
        d = np.where(p > 0, p, p * neg_slp) - t
        x = p - pred_c[:, None]
        r = np.maximum(x, 0.0)
        s_loss += crit_value(crit, d).sum()
        s_reg += crit_value(crit, r).sum()
        g_loss = crit_grad(crit, d) * np.where(p > 0, 1.0, neg_slp)
        g_reg = np.where(x > 0, crit_grad(crit, r), 0.0)
        grads.append((match_loss_w * g_loss + match_reg_w * g_reg) / B)
        g_c -= match_reg_w * g_reg.sum(axis=1) / B
    return (match_loss_w * s_loss + match_reg_w * s_reg) / B, grads, g_c


def random_inputs(rng, B=6, Lv=7, Le=9, crit="MSE"):
    """padded, masked predictions with the ties the derivative conventions decide: p - c = 0, |d| = 1, p = 0; pred_c
    negative on some graphs (the regulariser is then live on masked and padded positions)."""
    pred_c = rng.normal(0.0, 2.0, B)
    pred_c[::2] = -np.abs(pred_c[::2]) - 0.5
    kinds = []
    for L in (Lv, Le):
        lens = rng.integers(0, L + 1, B)
        lens[0], lens[-1] = L, 0
        seg = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
        w = rng.integers(0, 4, int(seg[-1]))
        real = np.arange(L)[None, :] >= (L - lens)[:, None]
        mask = real & (rng.random((B, L)) > 0.2)
        pred = rng.normal(0.0, 2.0, (B, L))
        W = pad_left(w, seg, L)
        for b in range(B):
            for j in np.flatnonzero(mask[b]):
                u = rng.random()
                if u < 0.12:
                    pred[b, j] = pred_c[b]                         # p - c = 0
                elif u < 0.24:
                    pred[b, j] = 0.0                               # leaky_relu at 0
                elif u < 0.36:
                    pred[b, j] = W[b, j] + 1.0                     # |d| = 1 (p > 0)
        # float32-representable values: the kernels read fp32
        kinds.append((pred.astype(np.float32).astype(np.float64), mask, w, seg))
    return pred_c.astype(np.float32).astype(np.float64), kinds


def _reference(monkeypatch, pred_c, kinds, crit, neg_slp, mlw, mrw):
    """counting_bp_loss under float64 autograd, its count term (with its gradient) taken out.  counting_bp_loss casts the
    targets with ``.float()``; for the float64 run that cast keeps float64 (the weights are integers either way)."""
    monkeypatch.setattr(torch.Tensor, "float", lambda t: t.double())
    B = pred_c.size
    c = torch.tensor(pred_c).view(B, 1).requires_grad_(True)
    leaves = [torch.tensor(k[0]).requires_grad_(True) for k in kinds]
    out = dict(pred_c=c, pred_v=leaves[0] * 1.0, pred_e=leaves[1] * 1.0,
               g_v_mask=torch.tensor(kinds[0][1]), g_e_mask=torch.tensor(kinds[1][1]))
    nw, ew = (torch.tensor(pad_left(k[2], k[3], k[0].shape[1])) for k in kinds)
    counts = torch.zeros(B)
    loss, _ = counting_bp_loss(out, counts, nw, ew, bp_loss=crit, neg_slp=neg_slp, match_loss_w=mlw, match_reg_w=mrw)
    monkeypatch.undo()
    match = loss - bp_criterion(crit)(c, counts.double().view(-1, 1), neg_slp)
    match.backward()
    return float(match.detach()), [q.grad.numpy() for q in leaves], c.grad.numpy().reshape(-1)


@pytest.mark.parametrize("crit", CRITERIA)
@pytest.mark.parametrize("seed", [0, 1, 2])
def test_closed_form_matches_counting_bp_loss_under_float64_autograd(monkeypatch, crit, seed):
    rng = np.random.default_rng(100 + seed)
    pred_c, kinds = random_inputs(rng, crit=crit)
    slp, mlw, mrw = 0.05, 0.7, 0.3
    loss, grads, g_c = match_loss_f64(pred_c, kinds, crit, slp, mlw, mrw)
    ref, ref_grads, ref_c = _reference(monkeypatch, pred_c, kinds, crit, slp, mlw, mrw)
    assert loss == pytest.approx(ref, rel=1e-12, abs=1e-12)
    for g, r in zip(grads, ref_grads):
        np.testing.assert_allclose(g, r, rtol=1e-12, atol=1e-14)
    np.testing.assert_allclose(g_c, ref_c, rtol=1e-12, atol=1e-14)
    # the inputs exercise what the conventions decide: a live regulariser on masked / padded positions, and ties
    masked_live = any(((~k[1]) & (pred_c[:, None] < 0)).any() for k in kinds)
    assert masked_live and any(np.abs(g[~k[1]]).max() > 0 for g, k in zip(grads, kinds))
    assert any((k[0][k[1]] == 0).any() for k in kinds)


def test_regulariser_depends_on_the_padded_length():
    """padding one more column adds crit(relu(-pred_c)) per graph with negative pred_c to the regulariser."""
    rng = np.random.default_rng(5)
    pred_c, kinds = random_inputs(rng)
    pv, mv, wv, sv = kinds[0]
    wider = (np.concatenate([np.zeros((pv.shape[0], 1)), pv], 1), np.concatenate([np.zeros((pv.shape[0], 1), bool), mv], 1),
             wv, sv)
    a = match_loss_f64(pred_c, [kinds[0]], "MSE", 0.01, 0.0, 1.0)[0]
    b = match_loss_f64(pred_c, [wider], "MSE", 0.01, 0.0, 1.0)[0]
    assert b - a == pytest.approx(np.sum(np.maximum(-pred_c, 0.0) ** 2) / pred_c.size)


def test_dummy_column_offsets_match_the_host_helper():
    from dummynode4graphlearning_b200.subgraph_isomorphism.matching import (add_dummy_to_subisomorphisms,
                                                                            dummy_column_offsets, pack_subisomorphisms)
    rng = np.random.default_rng(3)
    B = 40
    n = rng.integers(1, 20, B)
    graph = dict(node_ptr=np.concatenate([[0], np.cumsum(n)]))
    mats = []
    for b in range(B):
        S = int(rng.integers(0, 4)) if b % 5 else 0                 # samples without rows
        mats.append(rng.integers(0, n[b], (S, int(rng.integers(1, 6)))))
    packed = pack_subisomorphisms(mats)
    want = pack_subisomorphisms(add_dummy_to_subisomorphisms(mats, graph))
    got = dummy_column_offsets(np.diff(packed["val_ptr"]), packed["rows"])
    assert got.dtype == np.int64 and np.array_equal(got, want["val_ptr"])
    assert got[-1] == want["values"].size


def test_argument_checks():
    from dummynode4graphlearning_b200 import ops
    c = torch.zeros(2, 1)
    pv, mv = torch.zeros(2, 3), torch.ones(2, 3, dtype=torch.bool)
    w, seg = torch.zeros(6, dtype=torch.int32), torch.tensor([0, 3, 6], dtype=torch.int32)
    s = torch.zeros(())
    with pytest.raises(NotImplementedError):
        ops.match_loss(c, pv, mv, w, seg, None, None, None, None, "Huber", s, s, s)
    with pytest.raises(ValueError, match="CUDA"):
        ops.match_loss(c, pv, mv, w, seg, None, None, None, None, "MSE", s, s, s)
    with pytest.raises(ValueError, match="float32"):
        ops.match_loss(c.double(), pv, mv, w, seg, None, None, None, None, "MSE", s, s, s)
    i = torch.zeros(3, dtype=torch.int32)
    with pytest.raises(ValueError, match="CUDA"):
        ops.subiso_append_dummy(i, i, i[:2], i, i, 3)
    with pytest.raises(ValueError, match="int32"):
        ops.subiso_append_dummy(i.long(), i, i[:2], i, i, 3)


def _cpu_model(**over):
    from dummynode4graphlearning_b200 import synth, transforms as T
    from dummynode4graphlearning_b200.subgraph_isomorphism.models import DMPNN
    cfg = dict(synth.counting_config("small"), add_dummy=True)
    mc = T.process_model_config(cfg)
    kw = dict({k: v for k, v in mc.items() if k.startswith("max_")}, hid_dim=16, rep_num_graph_layers=1,
              rep_num_pattern_layers=1, pred_hid_dim=16, emb_net="Equivariant", filter_net="ScalarFilter",
              pred_return_weights="node", node_pred=True)
    kw.update(over)
    return DMPNN(**kw), cfg


def test_match_weights_refusals():
    """refused at construction, before anything touches a device."""
    from dummynode4graphlearning_b200.pipelines import CountingPipeline
    from dummynode4graphlearning_b200.subgraph_isomorphism.models import DMPNN
    model, cfg = _cpu_model()
    opt = torch.optim.SGD(model.parameters(), lr=0.0)
    for bad in ("nodes", "node,node", "", "node;edge"):
        with pytest.raises(ValueError, match="match_weights"):
            CountingPipeline(model, opt, cfg, match_weights=bad)
    with pytest.raises(ValueError, match="convert_conj"):
        CountingPipeline(model, opt, cfg, match_weights="node", convert_conj=True)

    class Refined(DMPNN):
        def refine_node_weights(self, weights, use_max=False):
            return weights * 2

    refined, _ = _cpu_model()
    refined.__class__ = Refined
    with pytest.raises(ValueError, match="refine_node_weights"):
        CountingPipeline(refined, opt, cfg, match_weights="node,edge")
