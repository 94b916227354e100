"""CPU: what a data-parallel shard must know about the rest of its mini-batch (SURVEY.md 8(e) i, v), established on the
oracle restatement of the reference models: samples of a counting mini-batch are coupled ONLY through the padded
lengths (head bias of padded rows, App. A-7; zero padding of shorter patterns in the label filter, App. A-14).  A shard
that is padded to the batch-wide lengths therefore reproduces the unsharded `pred_c` -- emulated here with the
unmodified oracle by appending the batch's longest pattern / graph samples to each shard ("ghosts") and dropping their
rows.  `BatchedGraph.set_padded_lengths` is the product-side mechanism (tests/test_zz_sharding_gpu.py)."""
import numpy as np
import pytest
import torch

from helpers import assert_close_rel, load_golden, oracle_cfg, rel_err
from oracle import models as OM

NODE_KEYS = ("vid", "vlabel", "v_is_dummy")
EDGE_KEYS = ("eid", "elabel", "e_is_dummy", "e_is_reversed")


def take(b, idx):
    """batch made of the samples idx (repeats allowed) of a flat block-diagonal batch dict."""
    node_ptr, edge_ptr = [0], [0]
    cols = {k: [] for k in ("src", "dst") + NODE_KEYS + EDGE_KEYS if k in b}
    for i in idx:
        n0, n1, e0, e1 = int(b["node_ptr"][i]), int(b["node_ptr"][i + 1]), int(b["edge_ptr"][i]), int(b["edge_ptr"][i + 1])
        for k in ("src", "dst"):
            cols[k].append(b[k][e0:e1] - n0 + node_ptr[-1])
        for k in NODE_KEYS:
            if k in b:
                cols[k].append(b[k][n0:n1])
        for k in EDGE_KEYS:
            if k in b:
                cols[k].append(b[k][e0:e1])
        node_ptr.append(node_ptr[-1] + n1 - n0)
        edge_ptr.append(edge_ptr[-1] + e1 - e0)
    out = {k: np.concatenate(v).astype(b[k].dtype) for k, v in cols.items()}
    out.update(num_graphs=len(idx), node_ptr=np.asarray(node_ptr, np.int32), edge_ptr=np.asarray(edge_ptr, np.int32))
    return out


@pytest.mark.parametrize("tag", ["RGIN/bdd4", "DMPNN/node_edge"])
def test_shard_padded_to_batch_wide_lengths_reproduces_full_batch(tag):
    gold = load_golden("counting_models")
    g, b = gold[tag], gold["_batch"]
    torch.manual_seed(0)
    sd = {k: v.clone() for k, v in g["state_dict"].items()}
    for k in sd:                                    # make the padded rows' bias visible (App. A-7, A-8)
        if "pred_net" in k and (k.endswith("bias") or "fc2" in k):
            sd[k] = torch.randn_like(sd[k]) * 0.1
    cfg = oracle_cfg(g["name"], g["kwargs"])
    P, G = b["pattern"], b["graph"]
    B = int(P["num_graphs"])
    with torch.no_grad():
        full = OM.counting_model(sd, P, G, cfg)["pred_c"]
        ghosts = sorted({int(np.argmax(np.diff(x[k]))) for x in (P, G) for k in ("node_ptr", "edge_ptr")})
        sizes = np.diff(G["node_ptr"])
        cut = 3
        worst = 0.0
        for lo, hi in ((0, cut), (cut, B)):
            own = list(range(lo, hi))
            plain = OM.counting_model(sd, take(P, own), take(G, own), cfg)["pred_c"]
            idx = own + ghosts
            padded = OM.counting_model(sd, take(P, idx), take(G, idx), cfg)["pred_c"][: len(own)]
            assert_close_rel(padded, full[lo:hi], 1e-5, "shard [%d, %d) padded to the batch-wide lengths" % (lo, hi))
            worst = max(worst, rel_err(plain, full[lo:hi]))
        if sizes[:cut].max() != sizes[cut:].max():
            assert worst > 1e-4, "the shard's own padding should have changed pred_c (bias of padded rows)"
