"""Seeded synthetic graph batches of the shapes BASELINE.json names (host side, numpy).

No dataset ships with the reference and there is no network, so every config is realised
as a seed-0 generator (SURVEY.md section 8(d)).  All arrays are int32 / float32 numpy on
the host; ids are GLOBAL (block-diagonal batch), ``node_ptr`` / ``edge_ptr`` give the
per-graph slices.

* ``tu_batch("mutag")``     C1: 188 graphs, n ~ 18, ~20 undirected edges, 7 node / 4 edge labels
* ``tu_batch("proteins")``  C2: 1113 graphs, n ~ 39 (log-normal, <= 620), ~1.86 n undirected edges,
                            3 node labels, one scalar attribute, no edge labels (-> all 1)
* ``counting_batch("small")`` C3: patterns 3-8 nodes, graphs 8-64 nodes / <= 256 edges, <= 16 labels
* ``counting_batch("large")`` C4: graphs 64-512 nodes / <= 2048 edges, <= 64 labels
"""
import numpy as np


def _undirected_graph(rng, n, target_edges, max_deg):
    """random spanning tree + extra edges under a degree cap; returns sorted directed pairs."""
    deg = np.zeros(n, dtype=np.int64)
    pairs = set()
    order = rng.permutation(n)
    for i in range(1, n):
        cand = order[:i]
        ok = cand[deg[cand] < max_deg]
        j = int(ok[rng.integers(len(ok))]) if len(ok) else int(cand[rng.integers(i)])
        a, b = int(order[i]), j
        pairs.add((min(a, b), max(a, b)))
        deg[a] += 1
        deg[b] += 1
    tries = 0
    while len(pairs) < target_edges and tries < 20 * target_edges:
        tries += 1
        a, b = int(rng.integers(n)), int(rng.integers(n))
        if a == b or deg[a] >= max_deg or deg[b] >= max_deg:
            continue
        p = (min(a, b), max(a, b))
        if p in pairs:
            continue
        pairs.add(p)
        deg[a] += 1
        deg[b] += 1
    und = np.array(sorted(pairs), dtype=np.int64).reshape(-1, 2)
    both = np.concatenate([und, und[:, ::-1]], axis=0)
    key = both[:, 0] * n + both[:, 1]
    both = both[np.argsort(key, kind="stable")]
    return both[:, 0], both[:, 1]


def tu_batch(shape="mutag", num_graphs=None, seed=0):
    """Raw TU-shaped batch (what ``load_graph_data_from_TUDatadir(with_dummy=False)`` parses,
    tu_data_processing.py:125-220), labels already shifted so the minimum is 1."""
    rng = np.random.default_rng(seed)
    if shape == "mutag":
        B = 188 if num_graphs is None else num_graphs
        ns = np.clip(np.rint(rng.normal(17.93, 4.6, B)), 10, 28).astype(np.int64)
        ratio, max_deg = 1.104, 4
        vp = np.array([.70, .10, .14, .02, .02, .01, .01])
        n_el = 4
        with_attr = False
    elif shape == "proteins":
        B = 1113 if num_graphs is None else num_graphs
        ns = np.clip(np.rint(rng.lognormal(3.38, 0.75, B)), 4, 620).astype(np.int64)
        ratio, max_deg = 1.864, 8
        vp = np.array([.49, .47, .04])
        n_el = 0
        with_attr = True
    else:
        raise ValueError(shape)
    srcs, dsts, vls, els = [], [], [], []
    node_ptr = np.zeros(B + 1, dtype=np.int64)
    edge_ptr = np.zeros(B + 1, dtype=np.int64)
    for g in range(B):
        n = int(ns[g])
        tgt = max(n - 1, int(round(ratio * n)))
        tgt = min(tgt, n * (n - 1) // 2)
        s, d = _undirected_graph(rng, n, tgt, max_deg)
        srcs.append(s + node_ptr[g])
        dsts.append(d + node_ptr[g])
        vls.append(rng.choice(len(vp), size=n, p=vp) + 1)
        if n_el:
            # the two directions of an undirected edge share a label (as in MUTAG)
            lab = {}
            el = np.empty(len(s), dtype=np.int64)
            for i, (a, b) in enumerate(zip(s, d)):
                k = (min(a, b), max(a, b))
                if k not in lab:
                    lab[k] = int(rng.integers(1, n_el + 1))
                el[i] = lab[k]
            els.append(el)
        else:
            els.append(np.ones(len(s), dtype=np.int64))
        node_ptr[g + 1] = node_ptr[g] + n
        edge_ptr[g + 1] = edge_ptr[g] + len(s)
    out = dict(
        num_graphs=B,
        node_ptr=node_ptr.astype(np.int32), edge_ptr=edge_ptr.astype(np.int32),
        src=np.concatenate(srcs).astype(np.int32), dst=np.concatenate(dsts).astype(np.int32),
        vlabel=np.concatenate(vls).astype(np.int32), elabel=np.concatenate(els).astype(np.int32),
        has_edge_labels=bool(n_el),
        y=rng.integers(0, 2, B).astype(np.int64),
    )
    if with_attr:
        out["vattr"] = rng.normal(0.0, 1.0, int(node_ptr[-1])).astype(np.float32)
    return out


def _directed_multigraph(rng, n, m, n_vl, n_el):
    """connected-ish random directed multigraph with m >= n-1 edges (multi-edges allowed,
    loops excluded), as the upstream NeuralSubgraphCounting generator produces."""
    src = np.empty(m, dtype=np.int64)
    dst = np.empty(m, dtype=np.int64)
    order = rng.permutation(n)
    k = 0
    for i in range(1, n):
        if k >= m:
            break
        a, b = int(order[i]), int(order[rng.integers(i)])
        if rng.integers(2):
            a, b = b, a
        src[k], dst[k] = a, b
        k += 1
    while k < m:
        a, b = int(rng.integers(n)), int(rng.integers(n))
        if a == b:
            continue
        src[k], dst[k] = a, b
        k += 1
    perm = np.argsort(src * n + dst, kind="stable")
    return src[perm], dst[perm], rng.integers(0, n_vl, n), rng.integers(0, n_el, m)


_COUNTING = {
    # C3 ('small', subgraph_isomorphism/README.md:74-97) and C4 ('large', BASELINE.json)
    "small": dict(pn=(3, 4, 8), pm=(2, 4, 8), gn=(8, 16, 32, 64), gm_cap=256, labels=(4, 8, 16),
                  max_npv=8, max_npe=8, max_npvl=8, max_npel=8,
                  max_ngv=64, max_nge=256, max_ngvl=16, max_ngel=16),
    "large": dict(pn=(3, 4, 8, 16), pm=(2, 4, 8, 16), gn=(64, 128, 256, 512), gm_cap=2048, labels=(16, 32, 64),
                  max_npv=16, max_npe=16, max_npvl=16, max_npel=16,
                  max_ngv=512, max_nge=2048, max_ngvl=64, max_ngel=64),
}


def counting_config(shape="small"):
    """the max_* constants of a shape BEFORE augmentation (train.py:38-81 adjusts them)."""
    c = _COUNTING[shape]
    return {k: v for k, v in c.items() if k.startswith("max_")}


def _pack(graphs):
    node_ptr = np.zeros(len(graphs) + 1, dtype=np.int64)
    edge_ptr = np.zeros(len(graphs) + 1, dtype=np.int64)
    for i, (s, d, vl, el) in enumerate(graphs):
        node_ptr[i + 1] = node_ptr[i] + len(vl)
        edge_ptr[i + 1] = edge_ptr[i] + len(s)
    return dict(
        num_graphs=len(graphs),
        node_ptr=node_ptr.astype(np.int32), edge_ptr=edge_ptr.astype(np.int32),
        src=np.concatenate([g[0] + node_ptr[i] for i, g in enumerate(graphs)]).astype(np.int32),
        dst=np.concatenate([g[1] + node_ptr[i] for i, g in enumerate(graphs)]).astype(np.int32),
        vid=np.concatenate([np.arange(len(g[2])) for g in graphs]).astype(np.int32),
        vlabel=np.concatenate([g[2] for g in graphs]).astype(np.int32),
        eid=np.concatenate([np.arange(len(g[0])) for g in graphs]).astype(np.int32),
        elabel=np.concatenate([g[3] for g in graphs]).astype(np.int32),
    )


def counting_batch(shape="small", batch_size=512, seed=0):
    """(pattern batch, graph batch, counts) for the subgraph-counting configs; ids/labels as
    ``train.py:1297-1308`` sets them (NODEID/EDGEID = arange per graph)."""
    c = _COUNTING[shape]
    rng = np.random.default_rng(seed)
    pats, gras = [], []
    for _ in range(batch_size):
        n_l = int(rng.choice(c["labels"]))
        pn = int(rng.choice(c["pn"]))
        pm = int(rng.choice([m for m in c["pm"] if m >= pn - 1]))
        pats.append(_directed_multigraph(rng, pn, pm, min(n_l, c["max_npvl"]), min(n_l, c["max_npel"])))
        gn = int(rng.choice(c["gn"]))
        gm = int(rng.integers(gn, min(c["gm_cap"], 4 * gn) + 1))
        gras.append(_directed_multigraph(rng, gn, gm, n_l, n_l))
    counts = rng.poisson(5.0, batch_size).astype(np.int64)
    return _pack(pats), _pack(gras), counts


def random_subisomorphisms(pattern_b, graph_b, seed=0, max_rows=5):
    """per sample a (S_b, np_b) matrix of graph-local node ids (S_b in 0..max_rows): random maps whose first pattern edge
    is planted on a real graph edge, so that the match-weight targets (dataset.py:54-108) are not all zero.  They are
    inputs for the weight kernels, not true subisomorphisms (the kernels do not care)."""
    rng = np.random.default_rng(seed)
    mats = []
    for b in range(int(pattern_b["num_graphs"])):
        pn0, gn0 = int(pattern_b["node_ptr"][b]), int(graph_b["node_ptr"][b])
        pn, gn = int(pattern_b["node_ptr"][b + 1]) - pn0, int(graph_b["node_ptr"][b + 1]) - gn0
        pe0, pe1 = int(pattern_b["edge_ptr"][b]), int(pattern_b["edge_ptr"][b + 1])
        ge0, ge1 = int(graph_b["edge_ptr"][b]), int(graph_b["edge_ptr"][b + 1])
        S = int(rng.integers(0, max_rows + 1))
        m = np.zeros((S, pn), np.int64)
        for s in range(S):
            m[s] = rng.choice(gn, size=pn, replace=gn < pn)
            if ge1 > ge0 and pe1 > pe0:
                k = int(rng.integers(ge0, ge1))
                j = int(rng.integers(pe0, pe1))
                pu, pv = int(pattern_b["src"][j]) - pn0, int(pattern_b["dst"][j]) - pn0
                m[s, pu] = int(graph_b["src"][k]) - gn0
                if pv != pu:
                    m[s, pv] = int(graph_b["dst"][k]) - gn0
        mats.append(m)
    return mats


def _unpack(b):
    """packed batch -> per-graph dicts of the shape ``subgraph_isomorphism.io.read_gml_graph`` returns (graph-local ids)."""
    out = []
    for i in range(int(b["num_graphs"])):
        n0, n1, e0, e1 = (int(b["node_ptr"][i]), int(b["node_ptr"][i + 1]), int(b["edge_ptr"][i]), int(b["edge_ptr"][i + 1]))
        out.append(dict(num_nodes=n1 - n0, src=b["src"][e0:e1].astype(np.int64) - n0, dst=b["dst"][e0:e1].astype(np.int64) - n0,
                        vid=b["vid"][n0:n1].astype(np.int64), vlabel=b["vlabel"][n0:n1].astype(np.int64),
                        elabel=b["elabel"][e0:e1].astype(np.int64), ekey=np.zeros(e1 - e0, np.int64)))
    return out


def counting_samples(shape="small", num_samples=512, seed=0, num_patterns=None):
    """a counting data set split as ``subgraph_isomorphism.io.load_data`` returns one: a list of ``{id, pattern, graph,
    subisomorphisms, counts}`` dicts.  num_patterns=None: every sample has its own pattern and graph; otherwise
    num_patterns patterns share ceil(num_samples / num_patterns) graphs (one sample per pair, the same graph object in
    every pair that uses it, as in the shared-graph data sets).  Subisomorphisms as ``random_subisomorphisms``."""
    rng = np.random.default_rng(seed)
    if num_patterns is None:
        p, g, counts = counting_batch(shape, num_samples, seed=seed)
        pats, gras = _unpack(p), _unpack(g)
        mats = random_subisomorphisms(p, g, seed=seed)
        return [dict(id="P_%d-G_%d" % (i, i), pattern=pats[i], graph=gras[i], subisomorphisms=mats[i], counts=int(counts[i]))
                for i in range(num_samples)]
    n_g = -(-num_samples // num_patterns)
    p, g, _ = counting_batch(shape, max(num_patterns, n_g), seed=seed)
    pats, gras = _unpack(p)[:num_patterns], _unpack(g)[:n_g]
    out = []
    for k in range(num_samples):
        pi, gi = k % num_patterns, k // num_patterns
        S = int(rng.integers(0, 6))
        m = rng.integers(0, max(gras[gi]["num_nodes"], 1), (S, pats[pi]["num_nodes"]))
        out.append(dict(id="P_%d-G_%d" % (pi, gi), pattern=pats[pi], graph=gras[gi], subisomorphisms=m,
                        counts=int(rng.poisson(5.0))))
    return out
