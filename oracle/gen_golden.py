"""Generate tests/golden/* by executing the UNMODIFIED reference under oracle/shims.

Needs a checkout of the original project:   DN4GL_REFERENCE_ROOT=<checkout> python -m oracle.gen_golden
The fixtures pin (a) the transforms' exact index outputs and (b) forward values, loss and every parameter
gradient of the reference's own GIN / RGIN(cls) / RGIN / DMPNN classes on small seeded batches.  They travel
to the GPU box; nothing else of the reference does.
"""
import os
import zlib
from argparse import Namespace

import numpy as np
import torch as th
import torch.nn.functional as F

from dummynode4graphlearning_b200 import synth
from dummynode4graphlearning_b200.transforms import process_model_config

from . import ref_drive as rd
from . import transforms as OT

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def _save(out, name):
    """one file per key under tests/golden/<name>/ (the key's "/" become directories): every file stays small"""
    for k, v in out.items():
        path = os.path.join(OUT, name, k + ".pt")
        os.makedirs(os.path.dirname(path), exist_ok=True)
        th.save(v, path)


def _load(name):
    root = os.path.join(OUT, name)
    return {os.path.relpath(os.path.join(d, f), root)[:-3]: th.load(os.path.join(d, f), weights_only=False)
            for d, _, files in os.walk(root) for f in files if f.endswith(".pt")}


def _np(d):
    return {k: (np.asarray(v) if not isinstance(v, (int, bool)) else v) for k, v in d.items()}


def gen_transforms():
    out = {}
    # SURVEY.md App. B, first vector
    appb = dict(num_graphs=2, node_ptr=np.array([0, 3, 5], np.int32), edge_ptr=np.array([0, 4, 6], np.int32),
                src=np.array([0, 1, 1, 2, 3, 4], np.int32), dst=np.array([1, 0, 2, 1, 4, 3], np.int32),
                vlabel=np.array([1, 2, 1, 2, 2], np.int32), elabel=np.ones(6, np.int32), has_edge_labels=False)
    cases = {"appB": appb, "mutag12": synth.tu_batch("mutag", 12, seed=11), "proteins8": synth.tu_batch("proteins", 8, seed=12)}
    for name, b in cases.items():
        gs = rd.ref_tu_load(b, True)
        conj = rd.ref_tu_conjugate(gs)
        line = rd.ref_tu_conjugate(rd.ref_tu_load(b, False))
        out["tu/" + name] = dict(inp=_np(b), dummy=rd.igraphs_to_batch(gs), conj=rd.igraphs_to_batch(conj),
                                 line=rd.igraphs_to_batch(line), conj_files=rd.ref_tu_save(conj))
    for shape, bs, seed in (("small", 6, 21), ("large", 1, 22)):
        p, g, _ = synth.counting_batch(shape, bs, seed=seed)
        cfg = synth.counting_config(shape)
        rp, rg = rd.ref_sub_add_dummy(p, g, cfg)
        out["sub/%s" % shape] = dict(cfg=cfg, pattern=_np(p), graph=_np(g), pattern_dummy=rp, graph_dummy=rg,
                                     pattern_conj=rd.ref_sub_conjugate(rp), graph_conj=rd.ref_sub_conjugate(rg))
    # SURVEY.md App. B, second vector
    g = dict(num_graphs=1, node_ptr=np.array([0, 3], np.int32), edge_ptr=np.array([0, 3], np.int32),
             src=np.array([0, 1, 1], np.int32), dst=np.array([1, 2, 2], np.int32), vid=np.arange(3, dtype=np.int32),
             vlabel=np.array([0, 1, 0], np.int32), eid=np.arange(3, dtype=np.int32), elabel=np.array([0, 1, 0], np.int32))
    cfg = dict(max_npv=4, max_npvl=2, max_npe=6, max_npel=2, max_ngv=4, max_ngvl=2, max_nge=6, max_ngel=2)
    _, rg = rd.ref_sub_add_dummy(g, g, cfg)
    out["sub/appB2"] = dict(cfg=cfg, graph=_np(g), graph_dummy=rg, graph_conj=rd.ref_sub_conjugate(rg))
    for base in (dict(add_rev=False, add_dummy=True, convert_conj=False), dict(add_rev=True, add_dummy=True, convert_conj=True)):
        c = dict(synth.counting_config("small"), **base)
        out["cfg/%s" % "-".join("%s%d" % (k[:5], v) for k, v in base.items())] = dict(inp=c, out=rd.ref_process_model_config(c))
    _save(out, "transforms")
    print("transforms.pt:", list(out))


def gen_augment():
    """SURVEY.md 8(f) rank 3: the reference's remove_loops / add_reversed_edges / calculate_norms /
    calculate_eigenvalues (train.py:270-345, 500-527) on seeded batches, added to transforms.pt."""
    out = _load("transforms")
    for shape, bs, seed in (("small", 6, 23), ("large", 1, 24)):
        p, g, _ = synth.counting_batch(shape, bs, seed=seed)
        cfg = synth.counting_config(shape)
        loops = {}
        for name, b in (("pattern", p), ("graph", g)):      # plant self loops (the synthetic generator makes none)
            b = dict(b)
            b["dst"] = b["dst"].copy()
            b["dst"][::5] = b["src"][::5]
            loops[name] = b
        lp, lg = rd.ref_sub_remove_loops(loops["pattern"], loops["graph"])
        rp, rg = rd.ref_sub_add_reversed(p, g, cfg)
        dp, dg = rd.ref_sub_add_dummy(rp, rg, process_model_config(dict(cfg, add_rev=True)))
        out["aug/%s" % shape] = dict(
            cfg=cfg, pattern=_np(p), graph=_np(g), pattern_loops=_np(loops["pattern"]), graph_loops=_np(loops["graph"]),
            pattern_noloops=lp, graph_noloops=lg, pattern_rev=rp, graph_rev=rg, pattern_rev_dummy=dp, graph_rev_dummy=dg,
            norms_self_loop=rd.ref_sub_norms_eigen(dg, True), norms_no_self_loop=rd.ref_sub_norms_eigen(dg, False))
    _save(out, "transforms")
    print("transforms.pt:", list(out))


def gen_match_weights():
    """SURVEY.md 8(f) rank 2: the reference's numba loops compute_nodeseq_subisoweights / compute_edgeseq_subisoweights
    (dataset.py:54-108) driven as calculate_node_weights / calculate_edge_weights do (:1491-1520), added to transforms.pt."""
    out = _load("transforms")
    for shape, bs, seed in (("small", 16, 61), ("large", 2, 62)):
        p, g, _ = synth.counting_batch(shape, bs, seed=seed)
        mats = synth.random_subisomorphisms(p, g, seed=seed)
        nw, ew = rd.ref_match_weights(mats, p, g)
        out["match/%s" % shape] = dict(pattern=_np(p), graph=_np(g), mats=mats, node_weights=nw, edge_weights=ew,
                                       conj=rd.ref_conjugate_subisomorphisms(mats, p, g))
    # hand-made: repeated pattern pairs, consecutive (0,1)x2 and NON-consecutive (1,2) ... (1,2): only the last run counts
    p = dict(num_graphs=1, node_ptr=np.array([0, 3], np.int32), edge_ptr=np.array([0, 5], np.int32),
             src=np.array([0, 0, 1, 2, 1], np.int32), dst=np.array([1, 1, 2, 0, 2], np.int32),
             vid=np.arange(3, dtype=np.int32), vlabel=np.zeros(3, np.int32), eid=np.arange(5, dtype=np.int32),
             elabel=np.array([0, 1, 0, 0, 1], np.int32))
    g = dict(num_graphs=1, node_ptr=np.array([0, 4], np.int32), edge_ptr=np.array([0, 8], np.int32),
             src=np.array([3, 0, 1, 0, 1, 2, 0, 1], np.int32), dst=np.array([0, 1, 2, 1, 2, 0, 1, 2], np.int32),
             vid=np.arange(4, dtype=np.int32), vlabel=np.zeros(4, np.int32), eid=np.arange(8, dtype=np.int32),
             elabel=np.array([0, 0, 0, 1, 1, 0, 1, 0], np.int32))
    mats = [np.array([[0, 1, 2], [0, 1, 2], [3, 0, 1]], np.int64)]
    nw, ew = rd.ref_match_weights(mats, p, g)
    out["match/runs"] = dict(pattern=_np(p), graph=_np(g), mats=mats, node_weights=nw, edge_weights=ew,
                             conj=rd.ref_conjugate_subisomorphisms(mats, p, g))
    _save(out, "transforms")
    print("transforms.pt:", list(out), "runs case:", nw.tolist(), ew.tolist())


def _grads(model):
    return {n: (p.grad.clone() if p.grad is not None else None) for n, p in model.named_parameters()}


def gen_counting():
    out = {}
    p, g, counts = synth.counting_batch("small", 8, seed=31)
    cfg = dict(synth.counting_config("small"), add_dummy=True)
    mc = process_model_config(cfg)
    pd_ = OT.sub_add_dummy(p, cfg["max_npv"], cfg["max_npvl"], cfg["max_npe"], cfg["max_npel"])
    gd_ = OT.sub_add_dummy(g, cfg["max_ngv"], cfg["max_ngvl"], cfg["max_nge"], cfg["max_ngel"])
    variants = {
        "RGIN/bdd4": ("RGIN", dict(hid_dim=16, pred_hid_dim=16)),
        "RGIN/basis_full": ("RGIN", dict(hid_dim=16, pred_hid_dim=16, rep_rgin_regularizer="basis", rep_rgin_num_bases=-1,
                                         pred_net="MeanPredictNet", pred_return_weights="none")),
        "RGIN/basis4_unshared": ("RGIN", dict(hid_dim=16, pred_hid_dim=16, rep_rgin_regularizer="basis", rep_rgin_num_bases=4,
                                              share_rep_net=False, rep_act_func="relu")),
        "DMPNN/node": ("DMPNN", dict(hid_dim=16, pred_hid_dim=16, node_pred=True, edge_pred=False)),
        "DMPNN/node_edge": ("DMPNN", dict(hid_dim=16, pred_hid_dim=16, node_pred=True, edge_pred=True,
                                          pred_return_weights="node,edge", init_neigenv=5.0, init_eeigenv=6.0)),
        "DMPNN/edge_max_nofilter": ("DMPNN", dict(hid_dim=16, pred_hid_dim=16, node_pred=False, edge_pred=True,
                                                  pred_net="MaxPredictNet", filter_net="None", rep_residual=False)),
    }
    for tag, (name, over) in variants.items():
        kw = rd.counting_kwargs({k: v for k, v in mc.items() if k.startswith("max_")}, **over)
        model = rd.ref_counting_model(name, kw, seed=zlib.crc32(tag.encode()) % 1000)
        o = model(rd.dgl_batched(pd_), rd.dgl_batched(gd_))
        c = th.from_numpy(counts).float().view(-1, 1)
        crit = lambda pred, target, slp: F.mse_loss(F.leaky_relu(pred, slp), target)   # train.py:624-625
        loss = crit(o["pred_c"], c, 0.01)
        reg = 0.0
        for k in ("p_v_rep", "p_e_rep", "g_v_rep", "g_e_rep"):                          # train.py:801-809
            if o[k] is not None:
                reg = reg + crit(o[k], th.zeros_like(o[k]), 1) * o[k].size(1)
        loss = loss + 1e-3 * reg
        loss.backward()
        out[tag] = dict(name=name, kwargs=kw, state_dict={k: v.clone() for k, v in model.state_dict().items()},
                        outputs={k: (v.detach().clone() if isinstance(v, th.Tensor) else None) for k, v in o.items()},
                        loss=loss.detach().clone(), grads=_grads(model))
    out["_batch"] = dict(pattern=_np(pd_), graph=_np(gd_), counts=counts, cfg=cfg, model_cfg=mc)
    _save(out, "counting_models")
    print("counting_models.pt:", [k for k in out if not k.startswith("_")])


def gen_counting_rgcn():
    """SURVEY.md 8(f) rank 1: the reference's RGCN class, added to counting_models.pt (same batch as gen_counting)."""
    out = _load("counting_models")
    b = out["_batch"]
    pd_, gd_, counts, mc = b["pattern"], b["graph"], b["counts"], b["model_cfg"]
    variants = {
        "RGCN/in_basis": dict(hid_dim=16, pred_hid_dim=16, rep_rgcn_edge_norm="in", rep_rgcn_regularizer="basis",
                              rep_rgcn_num_bases=-1),
        "RGCN/both_bdd4": dict(hid_dim=16, pred_hid_dim=16, rep_rgcn_edge_norm="both", rep_rgcn_regularizer="bdd",
                               rep_rgcn_num_bases=4, pred_net="MeanPredictNet", pred_return_weights="none"),
        "RGCN/none_basis4_bn_unshared": dict(hid_dim=16, pred_hid_dim=16, rep_rgcn_edge_norm="none",
                                             rep_rgcn_regularizer="basis", rep_rgcn_num_bases=4, rep_rgcn_batch_norm=True,
                                             share_rep_net=False, rep_act_func="relu"),
    }
    for tag, over in variants.items():
        kw = rd.counting_kwargs({k: v for k, v in mc.items() if k.startswith("max_")}, **over)
        model = rd.ref_counting_model("RGCN", kw, seed=zlib.crc32(tag.encode()) % 1000)
        o = model(rd.dgl_batched(pd_), rd.dgl_batched(gd_))
        c = th.from_numpy(counts).float().view(-1, 1)
        crit = lambda pred, target, slp: F.mse_loss(F.leaky_relu(pred, slp), target)
        loss = crit(o["pred_c"], c, 0.01)
        reg = 0.0
        for k in ("p_v_rep", "p_e_rep", "g_v_rep", "g_e_rep"):
            if o[k] is not None:
                reg = reg + crit(o[k], th.zeros_like(o[k]), 1) * o[k].size(1)
        loss = loss + 1e-3 * reg
        loss.backward()
        out[tag] = dict(name="RGCN", kwargs=kw, state_dict={k: v.clone() for k, v in model.state_dict().items()},
                        outputs={k: (v.detach().clone() if isinstance(v, th.Tensor) else None) for k, v in o.items()},
                        loss=loss.detach().clone(), grads=_grads(model))
    _save(out, "counting_models")
    print("counting_models.pt:", [k for k in out if not k.startswith("_")])


def gen_counting_compgcn():
    """SURVEY.md 8(f) rank 1: the reference's CompGCN class, added to counting_models.pt (same batch as gen_counting)."""
    out = _load("counting_models")
    b = out["_batch"]
    pd_, gd_, counts, mc = b["pattern"], b["graph"], b["counts"], b["model_cfg"]
    variants = {
        "CompGCN/mult_none": dict(hid_dim=16, pred_hid_dim=16, rep_compgcn_comp_opt="mult", rep_compgcn_edge_norm="none"),
        "CompGCN/sub_both_node_edge": dict(hid_dim=16, pred_hid_dim=16, rep_compgcn_comp_opt="sub",
                                           rep_compgcn_edge_norm="both", node_pred=True, edge_pred=True,
                                           pred_net="MeanPredictNet"),
        "CompGCN/mult_in_bn_unshared": dict(hid_dim=16, pred_hid_dim=16, rep_compgcn_comp_opt="mult",
                                            rep_compgcn_edge_norm="in", rep_compgcn_batch_norm=True, share_rep_net=False),
        "CompGCN/corr_out": dict(hid_dim=16, pred_hid_dim=16, rep_compgcn_comp_opt="corr", rep_compgcn_edge_norm="out"),
    }
    for tag, over in variants.items():
        kw = rd.counting_kwargs({k: v for k, v in mc.items() if k.startswith("max_")}, **over)
        model = rd.ref_counting_model("CompGCN", kw, seed=zlib.crc32(tag.encode()) % 1000)
        o = model(rd.dgl_batched(pd_), rd.dgl_batched(gd_))
        c = th.from_numpy(counts).float().view(-1, 1)
        crit = lambda pred, target, slp: F.mse_loss(F.leaky_relu(pred, slp), target)
        loss = crit(o["pred_c"], c, 0.01)
        reg = 0.0
        for k in ("p_v_rep", "p_e_rep", "g_v_rep", "g_e_rep"):
            if o[k] is not None:
                reg = reg + crit(o[k], th.zeros_like(o[k]), 1) * o[k].size(1)
        loss = loss + 1e-3 * reg
        loss.backward()
        out[tag] = dict(name="CompGCN", kwargs=kw, state_dict={k: v.clone() for k, v in model.state_dict().items()},
                        outputs={k: (v.detach().clone() if isinstance(v, th.Tensor) else None) for k, v in o.items()},
                        loss=loss.detach().clone(), grads=_grads(model))
    _save(out, "counting_models")
    print("counting_models.pt:", [k for k in out if not k.startswith("_")])


def gen_counting_loss():
    """SURVEY.md 8(a21): the full back-propagated loss incl. match terms, produced by the reference's OWN train_epoch
    (train.py:596-1000, executed verbatim on one mini-batch) for the three criteria -> counting_loss.pt."""
    base = _load("counting_models")
    b = base["_batch"]
    Lg = int(np.diff(b["graph"]["node_ptr"]).max())
    Le = int(np.diff(b["graph"]["edge_ptr"]).max())
    B = len(b["counts"])
    gen = th.Generator().manual_seed(77)
    nw, ew = th.randint(0, 4, (B, Lg), generator=gen), th.randint(0, 4, (B, Le), generator=gen)
    out = {"_node_weights": nw, "_edge_weights": ew}
    cases = {
        "DMPNN/node_edge|MSE": dict(bp_loss="MSE", neg_pred_slp=0.01, match_loss_w=0.5, match_reg_w=0.25, rep_reg_w=1e-3),
        "DMPNN/node_edge|MAE": dict(bp_loss="MAE", neg_pred_slp=0.1, match_loss_w=1.0, match_reg_w=1.0, rep_reg_w=0.0),
        "DMPNN/node_edge|SMSE": dict(bp_loss="SMSE", neg_pred_slp=0.05, match_loss_w=0.3, match_reg_w=0.2, rep_reg_w=1e-3,
                                     max_grad_norm=8.0),
        "RGIN/bdd4|MSE": dict(bp_loss="MSE", neg_pred_slp=0.01, match_loss_w=0.7, match_reg_w=0.4, rep_reg_w=1e-3),
    }
    for tag, conf in cases.items():
        mtag = tag.split("|")[0]
        g = base[mtag]
        model = rd.ref_counting_model(g["name"], g["kwargs"], seed=0)
        model.load_state_dict(g["state_dict"])
        th.manual_seed(zlib.crc32(tag.encode()) % 1000)
        with th.no_grad():   # pred_fc2 / weight_fc2 are zero-initialised (App. A-8): make every term of the loss live;
            for n, q in model.named_parameters():   # small pred_c so that relu(pred_v - pred_c) is not identically zero
                if "weight_fc2" in n:
                    q.normal_(0.0, 0.05)
                elif "pred_fc2" in n:
                    q.normal_(0.0, 0.02)
        metric, loss, grads = rd.ref_train_epoch(model, rd.dgl_batched(b["pattern"]), rd.dgl_batched(b["graph"]), b["counts"],
                                                 nw.clone(), ew.clone(), conf)
        out[tag] = dict(model=mtag, conf=conf, state_dict={k: v.clone() for k, v in model.state_dict().items()},
                        loss=float(loss), eval_metric=float(metric), grads=grads)
    th.save(out, os.path.join(OUT, "counting_loss.pt"))
    print("counting_loss.pt:", {k: round(v["loss"], 4) for k, v in out.items() if not k.startswith("_")})


def gen_classification():
    out = {}
    raw = synth.tu_batch("mutag", 10, seed=41)
    dummy = OT.tu_add_dummy(raw)
    conj = OT.tu_conjugate(dummy)
    for tag, b, model_name, add in (("GIN/mutag_dummy", dummy, "GIN", {"train_eps": False, "num_layers": 3, "aggregation": "sum"}),
                                    ("GIN/mutag_conj_eps", conj, "GIN", {"train_eps": True, "num_layers": 2, "aggregation": "mean"}),
                                    ("RGIN/mutag_dummy", dummy, "RGIN", {"num_layers": 2})):
        # PyG read_tu_data view of the saved files (restated: oracle.transforms.pyg_coalesce + one-hot)
        vmin, emin = int(b["vlabel"].min()), int(b["elabel"].min())
        R = int(b["elabel"].max()) - emin + 1
        s, d, first, mult = OT.pyg_coalesce(b["src"], b["dst"], b["elabel"] - emin, R)
        x = th.from_numpy(np.eye(int(b["vlabel"].max()) - vmin + 1, dtype=np.float32)[b["vlabel"] - vmin])
        edge_index = th.from_numpy(np.stack([s, d]).astype(np.int64))
        edge_attr = th.from_numpy(mult.astype(np.float32))
        batch = th.from_numpy(np.repeat(np.arange(b["num_graphs"]), np.diff(b["node_ptr"])).astype(np.int64))
        y = th.from_numpy(raw["y"])
        args = Namespace(num_features=x.size(1), hidden_dim=16, nhid=16, num_classes=2, dropout_ratio=0.0,
                         additional=add, epochs=3, device="cpu", num_relations=R)
        model = rd.ref_classifier(model_name, args, seed=len(tag))
        with th.no_grad():
            for n, p_ in model.named_parameters():
                if n.endswith("eps"):
                    p_.fill_(0.3)
        model.train()
        data = Namespace(x=x, edge_index=edge_index, edge_attr=edge_attr, batch=batch, y=y)
        o = model(data)
        loss = F.nll_loss(o, y)                                                        # main.py:41
        loss.backward()
        out[tag] = dict(name=model_name, args=vars(args), state_dict={k: v.clone() for k, v in model.state_dict().items()},
                        data=dict(x=x, edge_index=edge_index, edge_attr=edge_attr, batch=batch, y=y,
                                  node_ptr=th.from_numpy(b["node_ptr"].astype(np.int32))),
                        out=o.detach().clone(), loss=loss.detach().clone(), grads=_grads(model))
    th.save(out, os.path.join(OUT, "classification_models.pt"))
    print("classification_models.pt:", list(out))


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    gen_transforms()
    gen_augment()
    gen_match_weights()
    gen_counting()
    gen_counting_rgcn()
    gen_counting_compgcn()
    gen_counting_loss()
    gen_classification()
