"""Evaluation over a held-out split without a GPU: float64 restatements of the three evaluation kernels' definitions
(csrc/eval.cu), tied here to the torch expressions the reference evaluates with; the fixed evaluation order and its
per-rank slices; argument checks of the ops wrappers, which raise before anything reaches a device."""
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from dummynode4graphlearning_b200 import ops
from dummynode4graphlearning_b200.datasets import EpochSampler
from dummynode4graphlearning_b200.subgraph_isomorphism.losses import eval_criterion

EVAL_THREADS, EVAL_ROWS_PER_THREAD = 256, 4
EVAL_TILE = EVAL_THREADS * EVAL_ROWS_PER_THREAD


# ---- float64 references (imported by test_eval_gpu.py) ---------------------------------------------------------------
def ref_class_rows(logp, y):
    """(B, C) log-probabilities, int64 targets -> (pred int64, nll float64, correct float64) per row, as
    dn4gl_eval_class_rows_f32 defines them: torch.max's arg-max, -logp[y] (0 for a target outside [0, C)), pred == y; a
    row holding a NaN has nll NaN and is never correct."""
    logp = torch.as_tensor(logp).double()
    y = torch.as_tensor(y).long()
    B, C = logp.shape
    pred = logp.max(1)[1] if B else torch.zeros(0, dtype=torch.long)
    ok = (y >= 0) & (y < C)
    nll = torch.zeros(B, dtype=torch.float64)
    nll[ok] = -logp[ok, y[ok]]
    nan_row = torch.isnan(logp).any(1)
    nll[nan_row] = float("nan")
    correct = (ok & (pred == y) & ~nan_row).double()
    return pred, nll, correct


def ref_count_rows(pred_c, counts):
    """per-sample |r - t|, (r - t)^2, smooth-L1(r - t, beta 1) with r = relu(pred_c), t = counts, in float64 (n, 3)."""
    r = torch.relu(torch.as_tensor(pred_c).double().view(-1))
    t = torch.as_tensor(counts).double().view(-1)
    d = r - t
    z = d.abs()
    return torch.stack([z, d * d, torch.where(z < 1, 0.5 * z * z, z - 0.5)], 1)


def ref_reduce(v):
    """dn4gl_eval_reduce_f32's exact order on float32 columns v (n, k), emulated in float64: per tile of 1024 rows,
    thread t adds rows t, t + 256, t + 512, t + 768, then a halving tree over the 256 threads; thread t of the merge adds
    tiles t, t + 256, ..., then the same tree.  -> (k,) float64, bit for bit what the kernel writes."""
    v = np.asarray(v, np.float32)
    v = v.reshape(len(v), -1) if v.ndim == 1 else v
    n, k = v.shape
    if n == 0:
        return np.zeros(k)
    tiles = -(-n // EVAL_TILE)
    x = np.zeros((tiles * EVAL_TILE, k))
    x[:n] = v                                                   # float32 -> float64 is exact; padding adds exact zeros
    x = x.reshape(tiles, EVAL_ROWS_PER_THREAD, EVAL_THREADS, k)
    s = np.zeros((tiles, EVAL_THREADS, k))
    for j in range(EVAL_ROWS_PER_THREAD):
        s = s + x[:, j]
    part = _tree(s)                                             # (tiles, k)
    m = -(-tiles // EVAL_THREADS)
    p = np.zeros((m * EVAL_THREADS, k))
    p[:tiles] = part
    p = p.reshape(m, EVAL_THREADS, k)
    s = np.zeros((EVAL_THREADS, k))
    for j in range(m):
        s = s + p[j]
    return _tree(s[None])[0]


def _tree(s):
    s = s.copy()
    o = EVAL_THREADS // 2
    while o:
        s[:, :o] = s[:, :o] + s[:, o:2 * o]
        o //= 2
    return s[:, 0]


def reduce_bound(v):
    """n * 2^-53 * sum |terms| per column: how far any summation order of v's columns may lie from the exact sum."""
    v = np.abs(np.asarray(v, np.float64))
    v = v.reshape(len(v), -1) if v.ndim == 1 else v
    return len(v) * 2.0 ** -53 * v.sum(0)


# ---- the references against torch -------------------------------------------------------------------------------------
@pytest.mark.parametrize("C", [1, 2, 3, 32])
def test_class_reference_is_torch_max_and_nll_loss(C):
    g = torch.Generator().manual_seed(C)
    B = 257
    logp = torch.log_softmax(torch.randn(B, C, generator=g), 1)
    logp[::5] = logp[::5].round(decimals=0)             # many exact ties
    logp[3] = -1.0                                      # a whole row tied: index 0 wins
    y = torch.randint(0, C, (B,), generator=g)
    pred, nll, correct = ref_class_rows(logp, y)
    assert torch.equal(pred, logp.max(1)[1])
    assert int(pred[3]) == 0
    for r in range(B):                                  # lowest index among the maxima
        assert int(pred[r]) == int(torch.nonzero(logp[r] == logp[r].max())[0])
    assert math.isclose(float(nll.sum()), float(F.nll_loss(logp.double(), y, reduction="sum")), rel_tol=1e-12, abs_tol=1e-12)
    assert float(correct.sum()) == float(logp.max(1)[1].eq(y).sum())


def test_class_reference_nan_rows_and_out_of_range_targets():
    logp = torch.tensor([[-0.1, float("nan"), -3.0], [float("nan"), -0.5, float("nan")], [-1.0, -0.2, -2.0],
                         [-1.0, -0.2, -2.0], [-0.3, -0.3, -5.0]])
    y = torch.tensor([0, 0, 1, 3, -1])
    pred, nll, correct = ref_class_rows(logp, y)
    assert pred.tolist() == logp.max(1)[1].tolist() == [1, 0, 1, 1, 0]    # a NaN is the maximum, the first one wins
    assert torch.isnan(nll[:2]).all() and correct[:2].tolist() == [0.0, 0.0]
    assert nll[2] == -logp[2, 1].double() and correct[2] == 1.0
    assert nll[3] == 0.0 and correct[3] == 0.0 and nll[4] == 0.0 and correct[4] == 0.0


@pytest.mark.parametrize("kind,col", [("MAE", 0), ("MSE", 1), ("SMSE", 2)])
def test_count_reference_is_eval_criterion(kind, col):
    g = torch.Generator().manual_seed(col)
    pred = torch.randn(500, 1, generator=g, dtype=torch.float64) * 6        # about half negative: relu matters
    pred[:50] = -pred[:50].abs()
    counts = torch.randint(0, 8, (500,), generator=g)
    err = ref_count_rows(pred, counts)
    want = eval_criterion(kind)(pred, counts.double().view(-1, 1))
    assert math.isclose(float(err[:, col].mean()), float(want), rel_tol=1e-12)
    # without the relu the negative predictions would score differently
    raw = {"MAE": F.l1_loss, "MSE": F.mse_loss, "SMSE": F.smooth_l1_loss}[kind](pred, counts.double().view(-1, 1))
    assert not math.isclose(float(raw), float(want), rel_tol=1e-6)


@pytest.mark.parametrize("n", [0, 1, 1023, 1024, 1025, 300001])
def test_reduce_reference_is_a_sum(n):
    rng = np.random.default_rng(n)
    v = (rng.normal(size=(n, 3)) * np.exp(rng.uniform(-20, 20, (n, 3)))).astype(np.float32)
    got = ref_reduce(v)
    exact = np.array([math.fsum(v[:, c].astype(np.float64)) for c in range(3)])
    assert (np.abs(got - exact) <= reduce_bound(v)).all()
    if n == 0:
        assert got.tolist() == [0.0, 0.0, 0.0]


# ---- evaluation order and its per-rank slices -------------------------------------------------------------------------
@pytest.mark.parametrize("world", [1, 2, 3, 8])
@pytest.mark.parametrize("n,bs", [(1, 8), (100, 8), (101, 32), (1000, 512), (517, 64), (9, 9)])
def test_evaluation_order_and_rank_slices(world, n, bs):
    """evaluate walks idx in order in batches of bs (last one short); rank r takes the contiguous slice
    [r m // W, (r + 1) m // W) of a batch of m items and writes its records from position pos[0]: over the ranks every
    position of the split is covered exactly once and in order."""
    if bs < world:
        with pytest.raises(ValueError):
            EpochSampler(n, bs, shuffle=False, world_size=world)
        return
    per_rank = [list(EpochSampler(n, bs, shuffle=False, rank=r, world_size=world).batches()) for r in range(world)]
    assert len({len(b) for b in per_rank}) == 1 and len(per_rank[0]) == -(-n // bs)
    seen = []
    for s in range(len(per_rank[0])):
        m = per_rank[0][s][1]
        assert m == min(bs, n - s * bs)
        glob = []
        for r in range(world):
            pos, total = per_rank[r][s]
            assert total == m
            assert pos.tolist() == list(range(s * bs + r * m // world, s * bs + (r + 1) * m // world))
            glob += pos.tolist()
        assert glob == list(range(s * bs, s * bs + m))
        seen += glob
    assert seen == list(range(n))


# ---- argument checks: ValueError before any launch ---------------------------------------------------------------------
def test_wrappers_reject_bad_arguments_before_any_launch():
    f32, i64, i32 = torch.float32, torch.int64, torch.int32
    z = lambda *s, dtype=f32: torch.zeros(*s, dtype=dtype)      # noqa: E731  (host tensors: rejected first)
    with pytest.raises(ValueError, match="CUDA"):
        ops.eval_class_rows(z(4, 2), z(4, dtype=i64), 0, z(4, dtype=i32), z(4), z(4))
    with pytest.raises(ValueError, match="CUDA"):
        ops.eval_count_rows(z(4, 1), z(4, dtype=i64), 0, z(4), z(4, 3))
    with pytest.raises(ValueError, match="CUDA"):
        ops.eval_reduce(z(4, 3))
    with pytest.raises(ValueError, match="tensor"):
        ops.eval_reduce([1.0, 2.0])
    with pytest.raises(ValueError, match="float32"):
        ops.eval_reduce(z(4, dtype=torch.float64))
    with pytest.raises(ValueError, match="2-D"):
        ops.eval_class_rows(z(4), z(4, dtype=i64), 0, z(4, dtype=i32), z(4), z(4))
    with pytest.raises(ValueError, match="span|fit|integer"):
        ops._eval_span("x", 3, 2, 4)
    with pytest.raises(ValueError, match="integer"):
        ops._eval_span("x", 3, 0.5, 4)
    assert ops._eval_span("x", 3, np.int64(1), 4) == 1
