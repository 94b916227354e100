"""shared test plumbing: golden loading, oracle configuration from constructor kwargs, comparisons."""
import os

import numpy as np
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load_golden(name):
    """a .pt file, or a directory holding one .pt file per key (the larger sets, split to keep every file small):
    {key: value} with the key being the file's path under the directory without ".pt"."""
    path = os.path.join(GOLDEN, name)
    if not os.path.isdir(path):
        return torch.load(path, weights_only=False)
    return {os.path.relpath(os.path.join(d, f), path)[:-3]: torch.load(os.path.join(d, f), weights_only=False)
            for d, _, files in os.walk(path) for f in files if f.endswith(".pt")}


from oracle.models import counting_cfg_from_kwargs as oracle_cfg  # noqa: E402,F401  (kept under its old name for the tests)


def rel_err(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return ((a - b).abs().max() / (b.abs().max() + 1e-30)).item()


def assert_close_rel(a, b, tol, what="", atol=0.0):
    """max-abs error normalised by the max-abs reference value (the survey's parity measure).  `atol` is an
    absolute floor for quantities that are mathematically zero (e.g. the gradient of a Linear bias feeding a
    BatchNorm), where only rounding noise is left on both sides."""
    assert tuple(a.shape) == tuple(b.shape), (what, a.shape, b.shape)
    if b.numel() == 0:
        return
    if atol > 0 and float((a.detach().double().cpu() - b.detach().double().cpu()).abs().max()) <= atol:
        return
    e = rel_err(a, b)
    assert e <= tol, "%s: relative error %.3e > %.1e" % (what, e, tol)


def batches_equal(a, b, keys):
    for k in keys:
        x = a[k].cpu().numpy() if isinstance(a[k], torch.Tensor) else np.asarray(a[k])
        y = b[k].cpu().numpy() if isinstance(b[k], torch.Tensor) else np.asarray(b[k])
        assert x.shape == y.shape, (k, x.shape, y.shape)
        assert np.array_equal(x, y), (k, np.flatnonzero(x != y)[:8])


def oracle_preprocess_chain(p, g, cfg, remove_loops, add_rev, add_dummy, convert_conj):
    """the data-set level switches in the order of train.py:1271-1340, each with the maxima its predecessors leave."""
    npe, npel, nge, ngel = cfg["max_npe"], cfg["max_npel"], cfg["max_nge"], cfg["max_ngel"]
    if remove_loops:
        p, g = _OT().sub_remove_loops(p), _OT().sub_remove_loops(g)
    if add_rev:
        p, g = _OT().sub_add_reversed(p, npe, npel), _OT().sub_add_reversed(g, nge, ngel)
        npe, npel, nge, ngel = 2 * npe, 2 * npel, 2 * nge, 2 * ngel
    if add_dummy:
        p = _OT().sub_add_dummy(p, cfg["max_npv"], cfg["max_npvl"], npe, npel)
        g = _OT().sub_add_dummy(g, cfg["max_ngv"], cfg["max_ngvl"], nge, ngel)
    if convert_conj:
        p, g = _OT().sub_conjugate(p), _OT().sub_conjugate(g)
    return p, g


def _OT():
    from oracle import transforms
    return transforms


def nasty_tu_batch(rng, B):
    """TU-flavoured batch with everything the synthetic shapes avoid: self loops, duplicate edges, isolated nodes,
    single-node graphs, graphs without edges (never the last one: the reference drops those, App. A-2)."""
    node_ptr, edge_ptr, src, dst = [0], [0], [], []
    for g in range(B):
        n = int(rng.integers(1, 7))
        kind = rng.integers(0, 5)
        m = 0 if (kind == 0 and g != B - 1) else int(rng.integers(1, 3 * n + 2))
        s, d = rng.integers(0, n, m), rng.integers(0, n, m)
        if kind == 1 and m:
            d[: m // 2] = s[: m // 2]
        if kind == 2 and m > 1:
            k = len(s[1::2])
            s[1::2], d[1::2] = s[0::2][:k], d[0::2][:k]
        src += list(s + node_ptr[-1])
        dst += list(d + node_ptr[-1])
        node_ptr.append(node_ptr[-1] + n)
        edge_ptr.append(edge_ptr[-1] + m)
    N, E = node_ptr[-1], edge_ptr[-1]
    b = dict(num_graphs=B, node_ptr=np.asarray(node_ptr, np.int32), edge_ptr=np.asarray(edge_ptr, np.int32),
             src=np.asarray(src, np.int32).reshape(E), dst=np.asarray(dst, np.int32).reshape(E),
             vlabel=rng.integers(1, 4, N).astype(np.int32), elabel=rng.integers(1, 3, E).astype(np.int32),
             y=rng.integers(0, 2, B).astype(np.int64))
    b["vlabel"][0] = 1
    if E:
        b["elabel"][0] = 1
    return b


def nasty_sub_batch(rng, B, nmax, lmax):
    """counting-flavoured batch: multi-edges, self loops, isolated nodes, graphs without edges; edges sorted by (src, dst)
    like the generator's."""
    node_ptr, edge_ptr, src, dst = [0], [0], [], []
    for g in range(B):
        n = int(rng.integers(1, nmax + 1))
        kind = rng.integers(0, 5)
        m = 0 if kind == 0 else int(rng.integers(1, 3 * n + 2))
        s, d = rng.integers(0, n, m), rng.integers(0, n, m)
        if kind == 1 and m:
            d[: m // 2] = s[: m // 2]
        order = np.argsort(s * n + d, kind="stable")
        src += list(s[order] + node_ptr[-1])
        dst += list(d[order] + node_ptr[-1])
        node_ptr.append(node_ptr[-1] + n)
        edge_ptr.append(edge_ptr[-1] + m)
    N, E = node_ptr[-1], edge_ptr[-1]
    np_, ep_ = np.asarray(node_ptr), np.asarray(edge_ptr)
    return dict(num_graphs=B, node_ptr=np_.astype(np.int32), edge_ptr=ep_.astype(np.int32),
                src=np.asarray(src, np.int32).reshape(E), dst=np.asarray(dst, np.int32).reshape(E),
                vid=np.concatenate([np.arange(k) for k in np.diff(np_)]).astype(np.int32),
                vlabel=rng.integers(0, lmax, N).astype(np.int32),
                eid=(np.concatenate([np.arange(k) for k in np.diff(ep_)]) if E else np.zeros(0)).astype(np.int32),
                elabel=rng.integers(0, lmax, E).astype(np.int32))


NASTY_CFG = dict(max_npv=8, max_npe=32, max_npvl=8, max_npel=8, max_ngv=8, max_nge=32, max_ngvl=8, max_ngel=8)
