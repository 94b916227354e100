"""GPU: the matching objective of the counting models -- the dummy column of the subisomorphisms (bit-exact with the host
helper), the fused match loss (csrc/match.cu) per element against its float64 restatement and against the reference's
own train_epoch goldens, ``CountingPipeline(match_weights=...)`` on a resident data set against weights composed by hand,
captured replays that follow the device-scalar weights, device->host reads, refusals, and two ranks."""
import os
import tempfile

import numpy as np
import pytest
import torch

from conftest import record_error
from helpers import assert_close_rel, load_golden, rel_err
from test_match_loss import CRITERIA, match_loss_f64, random_inputs

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")


def _i32(x):
    return torch.from_numpy(np.asarray(x, np.int32)).to(DEV)


# ---- 1. the dummy column -----------------------------------------------------------------------------------------------
def _dummy_cases():
    from dummynode4graphlearning_b200 import synth
    cases = [(k, v["graph"], v["mats"]) for k, v in sorted(load_golden("transforms/match").items())]
    for shape in ("small", "large"):
        p, g, _ = synth.counting_batch(shape, 48, seed=21)
        mats = synth.random_subisomorphisms(p, g, seed=22)
        mats[3] = mats[3][:0]                                   # samples without rows
        cases.append(("synth_" + shape, g, mats))
    return cases


def test_dummy_column_is_bit_exact_with_the_host_helper():
    from dummynode4graphlearning_b200 import transforms as T
    from dummynode4graphlearning_b200.subgraph_isomorphism import matching as M
    for name, g, mats in _dummy_cases():
        want = M.pack_subisomorphisms(M.add_dummy_to_subisomorphisms(mats, g))
        sub = M.pack_subisomorphisms(mats, DEV)
        offs = M.dummy_column_offsets(np.diff(M.pack_subisomorphisms(mats)["val_ptr"]), [np.asarray(m).shape[0] for m in mats])
        assert np.array_equal(offs, want["val_ptr"]), name
        for _ in range(2):
            got = M.append_dummy_column(sub, T.to_device(g, DEV), _i32(offs), int(offs[-1]))
            assert np.array_equal(got["values"].cpu().numpy(), want["values"]), name
            assert np.array_equal(got["val_ptr"].cpu().numpy(), want["val_ptr"]) and torch.equal(got["rows"], sub["rows"])


def test_resident_batch_with_dummy_column_equals_the_host_collation():
    from dummynode4graphlearning_b200 import synth
    from dummynode4graphlearning_b200._lib import lib
    from dummynode4graphlearning_b200.datasets import ResidentCountingDataset
    from dummynode4graphlearning_b200.subgraph_isomorphism import io as sio, matching as M
    samples = synth.counting_samples("small", 40, seed=5, num_patterns=6)
    ds = ResidentCountingDataset(samples, DEV)
    idx = np.random.default_rng(2).integers(0, 40, 33)
    _, g, _, mats = sio.collate([samples[j] for j in idx])
    want = M.pack_subisomorphisms(M.add_dummy_to_subisomorphisms(mats, g))
    k0 = lib().kernel_launches()
    _, _, _, sub = ds.batch(idx, subisomorphisms=True, dummy_column=True)
    assert lib().kernel_launches() - k0 == 7        # the six gathers and the dummy column
    for k in ("val_ptr", "values", "rows"):
        assert np.array_equal(sub[k].cpu().numpy(), want[k]), k


# ---- 2. the loss kernels per element -----------------------------------------------------------------------------------
def _scalars(slp, mlw, mrw):
    return [torch.tensor(v, dtype=torch.float32, device=DEV) for v in (slp, mlw, mrw)]


def _fused(pred_c, kinds, crit, scalars, kind_mask=(True, True)):
    """ops.match_loss on device copies of random_inputs' arrays -> (loss, grads per kind, grad of pred_c)."""
    from dummynode4graphlearning_b200 import ops
    c = torch.tensor(pred_c, dtype=torch.float32, device=DEV).view(-1, 1).requires_grad_(True)
    args, leaves = [], []
    for (pred, mask, w, seg), on in zip(kinds, kind_mask):
        q = torch.tensor(pred, dtype=torch.float32, device=DEV).requires_grad_(True)
        leaves.append(q)
        args += [q, torch.tensor(mask, device=DEV), _i32(w) if on else None, _i32(seg)]
    loss = ops.match_loss(c, *args[:4], *args[4:], crit, *scalars)
    loss.backward()
    return loss.detach(), [q.grad for q in leaves], c.grad.view(-1)


@pytest.mark.parametrize("crit", CRITERIA)
@pytest.mark.parametrize("B,Lv,Le", [(6, 7, 9), (300, 40, 530)])
def test_loss_kernels_match_the_float64_restatement(crit, B, Lv, Le):
    rng = np.random.default_rng(B + Lv)
    pred_c, kinds = random_inputs(rng, B, Lv, Le, crit)
    slp, mlw, mrw = 0.05, 0.7, 0.3
    ref, ref_g, ref_c = match_loss_f64(pred_c, kinds, crit, np.float32(slp), np.float32(mlw), np.float32(mrw))
    runs = [_fused(pred_c, kinds, crit, _scalars(slp, mlw, mrw)) for _ in range(3)]
    loss, grads, gc = runs[0]
    # double sums of the same float64 elements: only the order and the final fp32 rounding differ
    assert abs(float(loss) - ref) <= 2e-7 * abs(ref), (float(loss), ref)
    for g, r in zip(grads, ref_g):
        err = float((g.double().cpu() - torch.from_numpy(r)).abs().max()) / max(float(np.abs(r).max()), 1e-30)
        record_error("match_loss_f64[%s,%d]" % (crit, B), "grad pred", err=err)
        assert err <= 2e-7
        assert torch.equal(g != 0, torch.from_numpy(r != 0).to(DEV))        # ties and masked positions: same zeros
    err_c = float((gc.double().cpu() - torch.from_numpy(ref_c)).abs().max()) / float(np.abs(ref_c).max())
    assert err_c <= 1e-6, err_c
    for other in runs[1:]:                                              # repeated runs: the same bits
        assert torch.equal(other[0], loss) and torch.equal(other[2], gc)
        assert all(torch.equal(a, b) for a, b in zip(other[1], grads))


def test_a_kind_without_weights_contributes_nothing():
    rng = np.random.default_rng(9)
    pred_c, kinds = random_inputs(rng)
    s = _scalars(0.01, 0.5, 0.25)
    loss, grads, gc = _fused(pred_c, kinds, "MSE", s, kind_mask=(True, False))
    ref, ref_g, ref_c = match_loss_f64(pred_c, kinds[:1], "MSE", np.float32(0.01), 0.5, 0.25)
    assert abs(float(loss) - ref) <= 2e-7 * abs(ref)
    assert grads[1] is None
    assert rel_err(gc, torch.from_numpy(ref_c)) <= 1e-6


# ---- 3. the reference's own train_epoch goldens ------------------------------------------------------------------------
@pytest.mark.parametrize("tag", ["DMPNN/node_edge|MSE", "DMPNN/node_edge|MAE", "DMPNN/node_edge|SMSE"])
def test_fused_loss_matches_reference_train_epoch_golden(tag):
    from dummynode4graphlearning_b200 import ops
    from dummynode4graphlearning_b200.graph import BatchedGraph
    from dummynode4graphlearning_b200.subgraph_isomorphism import models as PM
    from dummynode4graphlearning_b200.subgraph_isomorphism.losses import counting_bp_loss
    gold, base = load_golden("counting_loss.pt"), load_golden("counting_models")
    g, b = gold[tag], base["_batch"]
    m, c = base[g["model"]], g["conf"]
    model = getattr(PM, m["name"])(**m["kwargs"])
    model.load_state_dict(g["state_dict"], strict=True)
    model = model.to(DEV).train()
    pattern, graph = BatchedGraph.from_batch(b["pattern"], DEV), BatchedGraph.from_batch(b["graph"], DEV)
    out = model(pattern, graph)

    def flat(padded, ptr):                  # the golden's left-padded (B, L) weights -> flat rows of the graph batch
        lens = (ptr[1:] - ptr[:-1]).cpu().numpy()
        L = padded.size(1)
        return torch.cat([padded[i, L - n:] for i, n in enumerate(lens)]).to(DEV)

    nw, ew = flat(gold["_node_weights"], graph.node_ptr), flat(gold["_edge_weights"], graph.edge_ptr)
    assert gold["_node_weights"].size(1) == graph.padded_num_nodes() and gold["_edge_weights"].size(1) == graph.padded_num_edges()
    rest = counting_bp_loss(out, torch.from_numpy(b["counts"]).to(DEV), bp_loss=c["bp_loss"], neg_slp=c["neg_pred_slp"],
                            rep_reg_w=c["rep_reg_w"])[0]
    match = ops.match_loss(out["pred_c"], out["pred_v"], out["g_v_mask"], nw, graph.node_ptr, out["pred_e"],
                           out["g_e_mask"], ew, graph.edge_ptr, c["bp_loss"],
                           *_scalars(c["neg_pred_slp"], c["match_loss_w"], c["match_reg_w"]))
    loss = rest + match
    assert abs(float(loss.detach()) - g["loss"]) <= 1e-5 * abs(g["loss"]), (float(loss), g["loss"])
    loss.backward()
    params = dict(model.named_parameters())
    if c.get("max_grad_norm", 0) > 0:
        torch.nn.utils.clip_grad_norm_(model.parameters(), c["max_grad_norm"])
    gmax = max(float(r.abs().max()) for r in g["grads"].values() if r is not None)
    for n, ref in g["grads"].items():
        if ref is None:
            assert params[n].grad is None, n
        else:
            record_error("fused_match_loss_golden[%s]" % tag, "grad " + n, err=rel_err(params[n].grad, ref))
            assert_close_rel(params[n].grad, ref, 1e-5, "grad " + n, atol=2e-6 * gmax)


# ---- 4. the pipeline on a resident data set against weights composed by hand -------------------------------------------
def _model(name, cfg, seed=4, device=DEV):
    from dummynode4graphlearning_b200 import transforms as T
    from dummynode4graphlearning_b200.subgraph_isomorphism.models import DMPNN, RGIN
    mc = T.process_model_config(cfg)
    kw = dict({k: v for k, v in mc.items() if k.startswith("max_")}, hid_dim=32, rep_num_graph_layers=2,
              rep_num_pattern_layers=2, pred_hid_dim=32, emb_net="Equivariant", filter_net="ScalarFilter")
    if name == "DMPNN":
        kw.update(pred_return_weights="node,edge", node_pred=True, edge_pred=True)
    else:
        kw.update(pred_return_weights="node", rep_rgin_regularizer="bdd", rep_rgin_num_bases=4)
    torch.manual_seed(seed)
    model = {"DMPNN": DMPNN, "RGIN": RGIN}[name](**kw)
    with torch.no_grad():
        for n, q in model.named_parameters():
            if "fc2" in n:
                q.normal_(0.0, 0.05)
    return model.to(device)


def _pipe(model, cfg, match_weights, opt=None, **kw):
    from dummynode4graphlearning_b200.pipelines import CountingPipeline
    opt = opt or torch.optim.SGD(model.parameters(), lr=0.0)
    kw = dict(dict(rep_reg_w=1e-3, max_grad_norm=0.0, cuda_graphs=False, match_loss_w=0.5, match_reg_w=0.25), **kw)
    return CountingPipeline(model, opt, cfg, match_weights=match_weights, **kw)


def _by_hand(pipe, samples, idx, kinds):
    """the batch, its augmented graphs and its match weights composed from the host helpers."""
    from dummynode4graphlearning_b200 import transforms as T
    from dummynode4graphlearning_b200.subgraph_isomorphism import io as sio, matching as M
    p, g, counts, mats = sio.collate([samples[j] for j in idx])
    if pipe.add_dummy:
        mats = M.add_dummy_to_subisomorphisms(mats, g)
    p_aug, g_aug = pipe.augment(T.to_device(p, DEV), T.to_device(g, DEV))
    sub = M.pack_subisomorphisms(mats, DEV)
    nw = M.node_weights(sub, g_aug) if "node" in kinds else None
    ew = M.edge_weights(sub, p_aug, g_aug) if "edge" in kinds else None
    pattern, graph = pipe.transform(T.to_device(p, DEV), T.to_device(g, DEV))
    return pattern, graph, torch.from_numpy(counts).to(DEV), nw, ew


def _grads(model):
    return {n: q.grad.clone() for n, q in model.named_parameters() if q.grad is not None}


@pytest.mark.parametrize("name,kinds", [("DMPNN", "node,edge"), ("RGIN", "node")])
@pytest.mark.parametrize("prep", [dict(), dict(add_rev=True, remove_loops=True)])
def test_step_indices_equals_train_on_with_weights_by_hand(name, kinds, prep):
    from dummynode4graphlearning_b200 import synth
    from dummynode4graphlearning_b200.datasets import ResidentCountingDataset
    samples = synth.counting_samples("small", 40, seed=17)
    ds = ResidentCountingDataset(samples, DEV)
    cfg = dict(synth.counting_config("small"), add_dummy=True, **prep)
    idx = np.random.default_rng(3).permutation(40)[:29]
    runs = []
    for resident in (True, False):
        model = _model(name, cfg)
        pipe = _pipe(model, cfg, kinds, **prep)
        if resident:
            loss = pipe.step_indices(ds, idx).result()
        else:
            pattern, graph, counts, nw, ew = _by_hand(pipe, samples, idx, kinds)
            assert int(nw.sum()) > 0 and (ew is None or int(ew.sum()) > 0)
            loss = float(pipe.train_on(pattern, graph, counts, node_weights=nw, edge_weights=ew))
        runs.append((loss, _grads(model)))
    (l0, g0), (l1, g1) = runs
    assert abs(l0 - l1) <= 1e-6 * abs(l1), (l0, l1)
    assert set(g0) == set(g1)
    for n in g1:
        assert_close_rel(g0[n], g1[n], 1e-6, "grad " + n)
    # the match terms are in: the same step without them differs
    model = _model(name, cfg)
    plain = _pipe(model, cfg, None, **prep).step_indices(ds, idx).result()
    assert plain != l0


def test_overlapped_matched_step_equals_serial():
    from dummynode4graphlearning_b200 import synth
    from dummynode4graphlearning_b200.datasets import ResidentCountingDataset
    samples = synth.counting_samples("small", 40, seed=17)
    ds = ResidentCountingDataset(samples, DEV)
    cfg = dict(synth.counting_config("small"), add_dummy=True)
    sets = [np.random.default_rng(s).permutation(40)[:24] for s in range(3)]
    runs = []
    for overlap in (False, True):
        model = _model("DMPNN", cfg)
        pipe = _pipe(model, cfg, "node,edge", overlap=overlap)
        runs.append([pipe.step_indices(ds, i).result() for i in sets] + [_grads(model)])
    assert runs[0][:3] == runs[1][:3]
    assert all(torch.equal(runs[0][3][n], runs[1][3][n]) for n in runs[0][3])


# ---- 5. captured replays ---------------------------------------------------------------------------------------------
def test_captured_matched_step_follows_the_device_scalars():
    from dummynode4graphlearning_b200 import synth
    from dummynode4graphlearning_b200.optim import FlatAdam
    samples = synth.counting_samples("small", 32, seed=8)
    cfg = dict(synth.counting_config("small"), add_dummy=True)
    idx = np.arange(32)
    settings = [(0.25, 0.01), (0.25, 0.01), (0.25, 0.01), (0.0625, 0.01), (0.125, 0.3)]     # (match_reg_w, neg_slp)
    runs = {}
    for graphs in (False, True):
        model = _model("DMPNN", cfg)
        pipe = _pipe(model, cfg, "node,edge", opt=FlatAdam(model.parameters(), lr=0.0), cuda_graphs=graphs,
                     overlap=False)
        batch = _by_hand(pipe, samples, idx, "node,edge")
        out = []
        for mrw, slp in settings:
            pipe.match_reg_w, pipe.neg_slp = mrw, slp
            loss = pipe.train_on(*batch[:3], node_weights=batch[3], edge_weights=batch[4]).clone()
            out.append((loss, pipe.bucket.flat.detach().clone()))
        runs[graphs] = (out, pipe)
    pipe = runs[True][1]
    assert pipe.replayed_library_kernels() > 0, "no CUDA graph was replayed"
    for k, ((le, ge), (lg, gg)) in enumerate(zip(runs[False][0], runs[True][0])):
        assert torch.equal(le, lg) and torch.equal(ge, gg), k
    assert not torch.equal(runs[True][0][2][1], runs[True][0][3][1])        # the new match_reg_w was read by the replay
    assert not torch.equal(runs[True][0][3][1], runs[True][0][4][1])


# ---- 6. device->host reads -------------------------------------------------------------------------------------------
def _d2h_copies(pipe, ds, idx):
    from torch.profiler import ProfilerActivity, profile
    pipe.step_indices(ds, idx).result()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        pending = pipe.step_indices(ds, idx)
        torch.cuda.synchronize()
    pending.result()
    return len([e for e in prof.events() if "DtoH" in e.name])


def test_matched_step_reads_back_no_more_than_the_edge_work_total():
    from dummynode4graphlearning_b200 import synth
    from dummynode4graphlearning_b200.datasets import ResidentCountingDataset
    samples = synth.counting_samples("small", 32, seed=12)
    ds = ResidentCountingDataset(samples, DEV)
    cfg = dict(synth.counting_config("small"), add_dummy=True)
    idx = np.arange(24)
    counts = {mw: _d2h_copies(_pipe(_model("DMPNN", cfg), cfg, mw), ds, idx) for mw in (None, "node", "node,edge")}
    assert counts[None] > 0
    assert counts["node"] == counts[None], counts
    assert counts["node,edge"] == counts[None] + 1, counts


# ---- 7. refusals -----------------------------------------------------------------------------------------------------
def test_refusals():
    from dummynode4graphlearning_b200 import synth
    from dummynode4graphlearning_b200.subgraph_isomorphism.models import DMPNN
    cfg = dict(synth.counting_config("small"), add_dummy=True)
    model = _model("DMPNN", cfg)
    with pytest.raises(ValueError, match="convert_conj"):
        _pipe(model, cfg, "node", convert_conj=True)

    class Refined(DMPNN):
        def refine_edge_weights(self, weights, use_max=False):
            return weights + 1

    model.__class__ = Refined
    with pytest.raises(ValueError, match="refine_edge_weights"):
        _pipe(model, cfg, "edge")
    pipe = _pipe(model, cfg, None)             # no match weights asked for: constructed, but weights are refused
    batch = _by_hand(pipe, synth.counting_samples("small", 8, seed=1), np.arange(8), "node")
    with pytest.raises(ValueError, match="refine_edge_weights"):
        pipe.train_on(*batch[:3], node_weights=batch[3])


# ---- 8. two ranks ----------------------------------------------------------------------------------------------------
def _rank_grads(device, idx, total):
    from dummynode4graphlearning_b200 import synth
    from dummynode4graphlearning_b200.datasets import ResidentCountingDataset
    samples = synth.counting_samples("small", 48, seed=19)
    ds = ResidentCountingDataset(samples, device)
    cfg = dict(synth.counting_config("small"), add_dummy=True)
    model = _model("DMPNN", cfg, device=device)
    pipe = _pipe(model, cfg, "node,edge", exact_sharding=True)
    loss = pipe.step_indices(ds, idx, global_batch=total).result()
    return loss, pipe.bucket.flat.detach().cpu().clone()


def _worker(rank, world, port, out_dir, idx):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        n = len(idx)
        _, grad = _rank_grads(dev, idx[rank * n // world:(rank + 1) * n // world], n)
        torch.save(grad, os.path.join(out_dir, "rank%d.pt" % rank))
        dist.barrier()
    finally:
        dist.destroy_process_group()


def test_two_rank_matched_step_equals_single_process():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import torch.multiprocessing as mp
    from test_zz_nccl_gpu import _free_port
    idx = np.random.default_rng(6).permutation(48)[:32]
    with tempfile.TemporaryDirectory() as d:
        mp.spawn(_worker, args=(2, _free_port(), d, idx), nprocs=2, join=True)
        r0, r1 = torch.load(os.path.join(d, "rank0.pt")), torch.load(os.path.join(d, "rank1.pt"))
    assert torch.equal(r0, r1)
    _, ref = _rank_grads(torch.device("cuda:0"), idx, len(idx))
    assert rel_err(r0, ref) <= 1e-5, rel_err(r0, ref)
