"""Kernel-level tests of the tensor-core MLP stages (mlp_pipe.cu warp-specialised pipelines, mlp_tc.cu phase-serial
kernels, the BatchNorm kernels and their merges) through the C ABI, each against a float64 restatement of the definition
in include/dn4gl.h.  The tests call `ops.lib().call` with buffers they own: every output is NaN-filled and sits between
guard bands, the workspace has exactly the queried size (plus a guard after it), the counters array is private.  After
each call the guards must be unchanged and the counters zero; every case runs twice and must give bitwise-equal outputs.

Tolerances, per element (u = 2^-24, one fp32 rounding):

  GEMM outputs (Y, GX, dW):  |out - ref| <= c u sum_k |a_k| |b_k|   (3xTF32, DESIGN.md section 4 K6)
    - operand split: hi = x rounded to nearest at tf32, so |lo| <= 2^-11 |x|; lo enters the MMA as tf32, rounded (mlp_tc)
      or truncated when read (mlp_pipe): an error <= 2^-10 |lo| <= 2^-21 |x| per operand.  Products of tf32 values are exact
      in fp32, so each product a b is good to 2 * 2^-21 = 16 u; the pipelined weight gradient drops lo * lo (2^-22 = 4 u):
      C_SPLIT = 20.
    - accumulation: every MMA adds into its tensor-memory accumulator with truncation, < 1 ulp <= 2 u of the running sum,
      which is at most the sum of |a b| of its own terms.  The hardware does not document how the 8 products of one k-step
      are summed; they are counted as one more truncation: 4 u per MMA on the longest chain of one accumulator.  The chain
      is at most the KP/8 A_lo k-steps + the KP/8 A_hi k-steps (the A_hi steps may be spread over NACC accumulators;
      counting all of them is an upper bound): C_ACC = 4 * KP/4 = KP (KP = the contraction padded to 32 / 64).
    - epilogue: the [W_hi | W_lo] halves and the NACC <= 4 accumulators added in round-to-nearest, bias, mask: C_EPI = 10.
    - dW: 16 MMAs (k-steps of 8 rows) per 128-row tile into a fresh accumulator, then one fp32 add per tile into the
      CTA's shared-memory copy (T tiles per CTA), the four hi/lo blocks added, double merge, final rounding:
      c = C_SPLIT + 4 * 16 + T + 6.  The 64 x 64 serial kernel keeps accumulating in tensor memory: 4 * 16 * T.
    - prologues: X' = act(bn_in(X)) is 2-3 roundings of |x - mean| |k| + |beta| (C_PRO = 3, magnitudes use that sum);
      gY = k (gm - s1/N - xhat s2/N) with gm = G + Gseg[row2seg]: C_GY = 12 roundings of
      |k| (|gm| + |s1|/N + |xhat| |s2|/N).
  Reductions over values the kernel itself produced are checked against float64 sums of those fp32 values: the record
    from the device's Y, sums_prev from the device's GX, bn_bwd_sums / bn_stats / the pooled rows from their inputs.  The
    bound is n u sum|terms| with n the fp32 adds on the path (per-thread rows + butterflies + warps + the final rounding;
    the merges add in double).  Statistics: shifted sums S1 = sum (y - a), S2 = sum (y - a)^2 with a the CTA's first row,
    so the error scales with the spread s = max |y - mean| of the channel, not with its mean: mean within 2 n u s + u |mean|,
    var within 8 n u s^2 (S2 and the re-centred S1^2 / N), rstd within rstd (var_err / (2 (var + eps)) + 2 u).
  db: n u sum |gY| with n the rows one CTA adds + 16, plus the C_GY error of each term.
  Elementwise kernels: bn_act 3 u (|x - mean| |k| + |beta|), bn_bwd_apply C_GY u of its magnitude.
  ReLU masks: where bn(Y) is within 4 u of its magnitude of 0, the mask is the device's (bn_act's sign, the same fmaf as
    every stage kernel); elsewhere the device's mask must equal the float64 one.
  segment_ids: bit-exact.

The CPU-only tests tie the references to torch: the forward chain to nn.Linear -> nn.BatchNorm1d(training) -> ReLU /
LeakyReLU (running buffers included), each backward reference to float64 autograd of its forward reference."""
import functools
import math
import re
import zlib

import numpy as np
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from conftest import record_error

U = 2.0 ** -24
NONE, RELU, LEAKY = 0, 1, 2          # DN4GL_ACT_*
SLOPE = 1 / 5.5
C_SPLIT, C_EPI, C_PRO, C_GY = 20, 10, 3, 12
GUARD = 64                           # guard floats before and after every output
SENT = 0x7FBADBAD                    # guard bit pattern (a NaN no kernel computes)
LIN_COUNTERS = 64


# ---------------------------------------------------------------------------------------------------------------------
# float64 references: (value, magnitude), the magnitude being the same expression on absolute values
def _f64(a):
    return None if a is None else np.asarray(a, np.float64)


def ref_act(z, act, slope=SLOPE):
    if act == RELU:
        return np.maximum(z, 0.0)
    if act == LEAKY:
        return np.where(z > 0, z, slope * z)
    return z


def ref_dact(pos, act, slope=SLOPE):
    if act == RELU:
        return pos.astype(np.float64)
    if act == LEAKY:
        return np.where(pos, 1.0, slope)
    return np.ones(pos.shape)


def _rec(rec, C):
    r = _f64(rec).reshape(4, C)
    return r[0], r[1], r[2], r[3]          # mean, rstd, k = gamma rstd, beta


def ref_bn_apply(x, rec):
    """(x - mean) k + beta and |x - mean| |k| + |beta|."""
    x = _f64(x)
    mean, _, k, beta = _rec(rec, x.shape[1])
    return (x - mean) * k + beta, np.abs(x - mean) * np.abs(k) + np.abs(beta)


def ref_stage_input(X, in_bn, act, slope=SLOPE):
    """X' = act_in(bn_in(X)) and its magnitude."""
    X = _f64(X)
    z, mag = (X, np.abs(X)) if in_bn is None else ref_bn_apply(X, in_bn)
    return ref_act(z, act, slope), mag


def ref_lin_fwd(X, W, bias, in_bn=None, act=NONE, slope=SLOPE):
    """Y = act_in(bn_in(X)) W^T + bias."""
    Xp, A = ref_stage_input(X, in_bn, act, slope)
    W = _f64(W)
    Y, mag = Xp @ W.T, A @ np.abs(W).T
    if bias is not None:
        Y, mag = Y + _f64(bias), mag + np.abs(_f64(bias))
    return Y, mag


def ref_bn_record(Y, gamma, beta, eps, momentum, running_mean=None, running_var=None):
    """training-mode nn.BatchNorm1d: record {mean, rstd, gamma rstd, beta} of the biased batch variance, and the running
    buffers updated with the unbiased variance (the biased one, 0, at N = 1)."""
    Y = _f64(Y)
    N, M = Y.shape
    mean = Y.mean(0)
    var = ((Y - mean) ** 2).mean(0)
    rstd = 1.0 / np.sqrt(var + eps)
    g = np.ones(M) if gamma is None else _f64(gamma)
    b = np.zeros(M) if beta is None else _f64(beta)
    rec = np.concatenate([mean, rstd, g * rstd, b])
    unb = var * N / (N - 1) if N > 1 else var
    rm = None if running_mean is None else (1 - momentum) * _f64(running_mean) + momentum * mean
    rv = None if running_var is None else (1 - momentum) * _f64(running_var) + momentum * unb
    return rec, rm, rv


def ref_upstream(G, Gseg, row2seg, N, M):
    """G[r] + Gseg[row2seg[r]] and its magnitude."""
    g, mag = np.zeros((N, M)), np.zeros((N, M))
    if G is not None:
        g, mag = g + _f64(G), mag + np.abs(_f64(G))
    if Gseg is not None:
        gs = _f64(Gseg)[np.asarray(row2seg, np.int64)]
        g, mag = g + gs, mag + np.abs(gs)
    return g, mag


def ref_gy(g, gmag, Y, bn, sums, g_masked, pos=None):
    """BatchNorm(+ReLU) backward of the stage output: gm = g [bn(Y) > 0] (not when g_masked),
    gY = k (gm - s1/N - xhat s2/N); bn None: gY = g.  pos: the ReLU mask to use (None: float64's)."""
    if bn is None:
        return g, gmag
    Y = _f64(Y)
    N, M = Y.shape
    mean, rstd, k, _ = _rec(bn, M)
    if not g_masked:
        if pos is None:
            pos = ref_bn_apply(Y, bn)[0] > 0
        g, gmag = g * pos, gmag * pos
    s1, s2 = _f64(sums).reshape(2, M)
    xhat = (Y - mean) * rstd
    return k * (g - s1 / N - xhat * s2 / N), np.abs(k) * (gmag + np.abs(s1) / N + np.abs(xhat) * np.abs(s2) / N)


def ref_lin_bwd(gy, gymag, W, X, in_bn=None, act=NONE, slope=SLOPE, pos_in=None):
    """GX = (gY W) act_in'(bn_in(X)), dW = gY^T X', db = colsum gY, with magnitudes."""
    X, W = _f64(X), _f64(W)
    Xp, A = ref_stage_input(X, in_bn, act, slope)
    if pos_in is None:
        pos_in = (X if in_bn is None else ref_bn_apply(X, in_bn)[0]) > 0
    d = ref_dact(pos_in, act, slope)
    return dict(GX=(gy @ W) * d, GXmag=(gymag @ np.abs(W)) * np.abs(d), dW=gy.T @ Xp, dWmag=gymag.T @ A,
                db=gy.sum(0), dbmag=gymag.sum(0))


def ref_sums_prev(GX, X, in_bn):
    """{sum GX, sum GX xhat_in} (and the sums of absolute terms), xhat_in = (X - mean_in) rstd_in."""
    GX, X = _f64(GX), _f64(X)
    mean, rstd, _, _ = _rec(in_bn, X.shape[1])
    t = GX * ((X - mean) * rstd)
    return np.concatenate([GX.sum(0), t.sum(0)]), np.concatenate([np.abs(GX).sum(0), np.abs(t).sum(0)])


def ref_bn_bwd_sums(G, Gseg, row2seg, Y, rec, act, slope=SLOPE, pos=None):
    """{sum gm, sum gm xhat}, gm = (G + Gseg[row2seg]) act'(bn(Y))."""
    Y = _f64(Y)
    N, M = Y.shape
    g, _ = ref_upstream(G, Gseg, row2seg, N, M)
    if pos is None:
        pos = ref_bn_apply(Y, rec)[0] > 0
    mean, rstd, _, _ = _rec(rec, M)
    gm = g * ref_dact(pos, act, slope)
    t = gm * ((Y - mean) * rstd)
    return np.concatenate([gm.sum(0), t.sum(0)]), np.concatenate([np.abs(gm).sum(0), np.abs(t).sum(0)])


def ref_bn_bwd_apply(G, Y, rec, sums, act, slope=SLOPE, pos=None):
    """GX = k (gm - s1/N - xhat s2/N), gm = G act'(bn(Y))."""
    Y = _f64(Y)
    if pos is None:
        pos = ref_bn_apply(Y, rec)[0] > 0
    d = ref_dact(pos, act, slope)
    return ref_gy(_f64(G) * d, np.abs(_f64(G) * d), Y, rec, sums, True)


def ref_bn_act(Y, rec, act, slope=SLOPE):
    z, mag = (_f64(Y), np.abs(_f64(Y))) if rec is None else ref_bn_apply(Y, rec)
    return ref_act(z, act, slope), mag


def ref_pool(out, seg_ptr, mode):
    """per-segment sum (mode 0) / mean (mode 1, empty segments 0) of the rows of out, and the sum of |rows|."""
    out = _f64(out)
    seg_ptr = np.asarray(seg_ptr, np.int64)
    lens = np.diff(seg_ptr)
    ids = np.repeat(np.arange(len(lens)), lens)
    s = np.zeros((len(lens), out.shape[1]))
    a = np.zeros_like(s)
    np.add.at(s, ids, out)
    np.add.at(a, ids, np.abs(out))
    if mode == 1:
        d = np.maximum(lens, 1)[:, None]
        s, a = s / d, a / d
    return s, a


def ref_segment_ids(seg_ptr, N):
    seg_ptr = np.asarray(seg_ptr, np.int64)
    return np.repeat(np.arange(len(seg_ptr) - 1), np.diff(seg_ptr)).astype(np.int32)[:N]


# ---------------------------------------------------------------------------------------------------------------------
# error model
def c_gemm(kp):
    """C_SPLIT + C_ACC + C_EPI for a contraction padded to kp."""
    return C_SPLIT + kp + C_EPI


def c_dw(T, accw_smem=True):
    return C_SPLIT + (4 * 16 + T if accw_smem else 4 * 16 * T) + 6


def pad32(x):
    return 32 if x <= 32 else 64


def stat_bounds(Yd, n):
    """(mean bound, var bound) per channel for statistics of the fp32 values Yd (n fp32 adds per CTA)."""
    Yd = _f64(Yd)
    mean = Yd.mean(0)
    s = np.abs(Yd - mean).max(0)
    return 2 * n * U * s + U * np.abs(mean), 8 * n * U * s * s


# ---------------------------------------------------------------------------------------------------------------------
# CPU-only: the references against torch
def _t(a):
    return torch.from_numpy(np.asarray(a, np.float64))


@pytest.mark.parametrize("act", [RELU, LEAKY], ids=["relu", "leaky"])
@pytest.mark.parametrize("N", [1, 7, 300])
def test_reference_forward_chain_matches_torch(N, act):
    """Linear -> BatchNorm1d(training) -> act -> Linear in float64 == the stage references: record, running buffers,
    num_batches_tracked, and the second stage with the record folded into its prologue."""
    torch.manual_seed(N + act)
    K, M, M2 = 7, 5, 3
    lin1, bn, lin2 = nn.Linear(K, M).double(), nn.BatchNorm1d(M, momentum=0.3).double(), nn.Linear(M, M2).double()
    with torch.no_grad():
        bn.weight.uniform_(-1.5, 1.5)
        bn.bias.normal_()
        bn.running_mean.normal_()
        bn.running_var.uniform_(0.5, 2.0)
    rm0, rv0 = bn.running_mean.numpy().copy(), bn.running_var.numpy().copy()
    x = torch.randn(N, K, dtype=torch.float64) * 2 + 1
    y = lin1(x)
    if N == 1:                # torch refuses batch statistics of one row; the kernels use the biased variance (0)
        z = (y - y.mean(0)) / torch.sqrt(torch.zeros(M, dtype=torch.float64) + bn.eps) * bn.weight + bn.bias
        bn.running_mean.mul_(0.7).add_(0.3 * y.mean(0).detach())
        bn.running_var.mul_(0.7)
        bn.num_batches_tracked += 1
    else:
        z = bn(y)
    h = F.relu(z) if act == RELU else F.leaky_relu(z, SLOPE)
    out = lin2(h)

    W1, b1, W2, b2 = (p.detach().numpy() for p in (lin1.weight, lin1.bias, lin2.weight, lin2.bias))
    Y, _ = ref_lin_fwd(x.numpy(), W1, b1)
    rec, rm, rv = ref_bn_record(Y, bn.weight.detach().numpy(), bn.bias.detach().numpy(), bn.eps, 0.3, rm0, rv0)
    np.testing.assert_allclose(Y, y.detach().numpy(), rtol=1e-13, atol=1e-13)
    np.testing.assert_allclose(ref_bn_act(Y, rec, act)[0], h.detach().numpy(), rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(rm, bn.running_mean.numpy(), rtol=1e-13, atol=1e-13)
    np.testing.assert_allclose(rv, bn.running_var.numpy(), rtol=1e-13, atol=1e-13)
    assert int(bn.num_batches_tracked) == 1
    Y2, _ = ref_lin_fwd(Y, W2, b2, in_bn=rec, act=act)
    np.testing.assert_allclose(Y2, out.detach().numpy(), rtol=1e-12, atol=1e-12)


@pytest.mark.parametrize("act", [RELU, LEAKY], ids=["relu", "leaky"])
def test_reference_backward_is_autograd(act):
    """two stages Linear, BN, act, Linear, BN, act with a sum readout: the backward references (bn_bwd_sums, the stage
    backward with its BatchNorm prologue, sums_prev, the chained g_masked backward, bn_bwd_apply) == float64 autograd of
    the forward references."""
    torch.manual_seed(act)
    N, K, M, M2, B = 40, 6, 5, 4, 3
    rng = np.random.default_rng(act)
    X = rng.normal(size=(N, K))
    W1, b1 = rng.normal(size=(M, K)), rng.normal(size=M)
    W2, b2 = rng.normal(size=(M2, M)), rng.normal(size=M2)
    g1, be1, g2, be2 = rng.uniform(-1.5, 1.5, M), rng.normal(size=M), rng.uniform(-1.5, 1.5, M2), rng.normal(size=M2)
    row2seg = np.sort(rng.integers(0, B, N))
    G, Gseg = rng.normal(size=(N, M2)), rng.normal(size=(B, M2))
    eps = 1e-5
    fact = (lambda z: F.relu(z)) if act == RELU else (lambda z: F.leaky_relu(z, SLOPE))

    tX, tW1, tb1, tW2, tb2, tg1, tbe1, tg2, tbe2 = (_t(a).requires_grad_(True) for a in (X, W1, b1, W2, b2, g1, be1, g2, be2))
    Y1t = tX @ tW1.T + tb1
    h1 = fact(F.batch_norm(Y1t, None, None, tg1, tbe1, training=True, eps=eps))
    Y1t.retain_grad()
    Y2t = h1 @ tW2.T + tb2
    Y2t.retain_grad()
    h2 = fact(F.batch_norm(Y2t, None, None, tg2, tbe2, training=True, eps=eps))
    pooled = torch.zeros(B, M2, dtype=torch.float64).index_add(0, torch.from_numpy(row2seg), h2)
    ((h2 * _t(G)).sum() + (pooled * _t(Gseg)).sum()).backward()

    Y1, _ = ref_lin_fwd(X, W1, b1)
    rec1, _, _ = ref_bn_record(Y1, g1, be1, eps, 0.1)
    Y2, _ = ref_lin_fwd(Y1, W2, b2, in_bn=rec1, act=act)
    rec2, _, _ = ref_bn_record(Y2, g2, be2, eps, 0.1)
    sums2, _ = ref_bn_bwd_sums(G, Gseg, row2seg, Y2, rec2, act)
    chk = functools.partial(np.testing.assert_allclose, rtol=1e-10, atol=1e-10)
    chk(sums2[:M2], tbe2.grad.numpy())
    chk(sums2[M2:], tg2.grad.numpy())
    g, gmag = ref_upstream(G, Gseg, row2seg, N, M2)
    if act == RELU:
        gy2, _ = ref_gy(g, gmag, Y2, rec2, sums2, False)
    else:                     # LeakyReLU: mask the gradient outside (g_masked), as a LeakyReLU stage hands it over
        pos = ref_bn_apply(Y2, rec2)[0] > 0
        gy2, _ = ref_gy(g * ref_dact(pos, act), gmag, Y2, rec2, sums2, True)
    chk(gy2, Y2t.grad.numpy())
    chk(ref_bn_bwd_apply(g, Y2, rec2, sums2, act)[0], Y2t.grad.numpy())
    r2 = ref_lin_bwd(gy2, gy2, W2, Y1, in_bn=rec1, act=act)
    chk(r2["dW"], tW2.grad.numpy())
    chk(r2["db"], tb2.grad.numpy())
    sp, _ = ref_sums_prev(r2["GX"], Y1, rec1)
    chk(sp[:M], tbe1.grad.numpy())
    chk(sp[M:], tg1.grad.numpy())
    gy1, _ = ref_gy(r2["GX"], r2["GX"], Y1, rec1, sp, True)
    chk(gy1, Y1t.grad.numpy())
    r1 = ref_lin_bwd(gy1, gy1, W1, X)
    chk(r1["GX"], tX.grad.numpy())
    chk(r1["dW"], tW1.grad.numpy())
    chk(r1["db"], tb1.grad.numpy())


def test_reference_pool_and_segment_ids_match_torch():
    rng = np.random.default_rng(3)
    lens = np.array([0, 3, 1, 0, 5, 2])
    seg = np.concatenate([[0], np.cumsum(lens)])
    out = rng.normal(size=(int(seg[-1]), 3))
    ids = torch.repeat_interleave(torch.arange(len(lens)), torch.from_numpy(lens))
    assert np.array_equal(ref_segment_ids(seg, out.shape[0]), ids.numpy())
    s = torch.zeros(len(lens), 3, dtype=torch.float64).index_add(0, ids, _t(out))
    np.testing.assert_allclose(ref_pool(out, seg, 0)[0], s.numpy(), rtol=1e-14)
    np.testing.assert_allclose(ref_pool(out, seg, 1)[0], (s / torch.from_numpy(np.maximum(lens, 1))[:, None]).numpy(), rtol=1e-14)


# ---------------------------------------------------------------------------------------------------------------------
# GPU plumbing
def _lib():
    from dummynode4graphlearning_b200 import ops
    return ops.lib()


def _call(name, *args):
    _lib().call(name, *[a.data_ptr() if isinstance(a, torch.Tensor) else a for a in args])


def _size(name, *args):
    return _lib().size(name, *args)


def _stream():
    return torch.cuda.current_stream().cuda_stream


@functools.lru_cache(None)
def _n_sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _rng(*key):
    return np.random.default_rng(zlib.crc32(repr(key).encode()))


class Buf:
    """a device buffer inside guard bands: `t` is the buffer (NaN-filled, or `init`), offset floats past a 16-byte
    boundary; `check()` asserts the guards still hold SENT."""

    def __init__(self, shape, init=None, offset=0, dtype=torch.float32):
        n = int(np.prod(shape))
        self.lo, self.n = GUARD + offset, n
        self.full = torch.empty(GUARD + offset + n + GUARD, dtype=dtype, device="cuda")
        self.full.view(torch.int32 if dtype != torch.int64 else torch.int64).fill_(SENT)
        self.t = self.full[self.lo:self.lo + n].view(shape)
        if init is not None:
            self.t.copy_(torch.as_tensor(np.asarray(init)).to(dtype))
        elif dtype == torch.float32:
            self.t.fill_(float("nan"))
        else:
            self.t.fill_(-123456)

    def check(self, what):
        g = torch.cat([self.full[:self.lo], self.full[self.lo + self.n:]]).view(torch.int32).cpu()
        assert bool((g == SENT).all()), "%s: a guard band was overwritten" % what

    def np(self):
        return self.t.cpu().numpy()


def _inp(a, offset=0, dtype=torch.float32):
    """input array on the device, offset floats past a 16-byte boundary (None -> None)."""
    if a is None:
        return None
    a = np.ascontiguousarray(a)
    full = torch.empty(a.size + offset + 4, dtype=dtype, device="cuda")
    t = full[offset:offset + a.size].view(a.shape)
    t.copy_(torch.from_numpy(a))
    return t


class Ws:
    """workspace of exactly `nbytes`, followed by a guard."""

    def __init__(self, nbytes):
        self.n = nbytes
        self.full = torch.full((nbytes + 1024,), 0xA5, dtype=torch.uint8, device="cuda")
        self.t = self.full

    def check(self):
        assert bool((self.full[self.n:] == 0xA5).all().cpu()), "written past the queried workspace size"


def _counters():
    return torch.zeros(LIN_COUNTERS, dtype=torch.int32, device="cuda")


def _bits_equal(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.shape == b.shape and a.dtype == b.dtype and a.tobytes() == b.tobytes()


def _twice(fn):
    """run fn() twice (each call allocates its own NaN-filled outputs and checks its guards): bitwise-equal outputs."""
    a, b = fn(), fn()
    for k in a:
        assert _bits_equal(a[k], b[k]), "%s differs between two identical launches" % k
    return a


def _within(out, ref, bound, test, what):
    """|out - ref| <= bound per element; records the worst error relative to the reference and as a fraction of the bound."""
    out, ref = np.asarray(out, np.float64), np.asarray(ref, np.float64)
    bound = np.broadcast_to(np.asarray(bound, np.float64), ref.shape)
    assert out.shape == ref.shape, (what, out.shape, ref.shape)
    err = np.abs(out - ref)
    bad = ~(err <= bound)
    if bad.any():
        i = np.unravel_index(np.flatnonzero(bad)[0], out.shape)
        raise AssertionError("%s: %d of %d elements outside the bound; first at %s: out %r ref %r bound %.3e"
                             % (what, int(bad.sum()), out.size, i, out[i], ref[i], bound[i]))
    if err.size:
        frac = float(np.max(np.where(bound > 0, err / np.where(bound > 0, bound, 1), 0.0)))
        record_error(test, what, err=float(err.max() / max(np.abs(ref).max(), 1e-30)), frac_of_bound=frac)


def _device_pos(z_in, rec):
    """the sign the kernels take for bn(z_in) > 0: dn4gl_bn_act_f32 with ReLU evaluates the same fmaf."""
    z = _inp(np.asarray(z_in, np.float32))
    out = torch.empty_like(z)
    _call("dn4gl_bn_act_f32", z, z.shape[0], z.shape[1], _inp(np.asarray(rec, np.float32)), RELU, 0.0, out, _stream())
    return out.cpu().numpy() > 0


def _mask(z_in, rec, what):
    """the ReLU mask of bn(z_in): float64's, except within rounding of 0 where it is the device's; elsewhere the two
    must agree."""
    z, mag = ref_bn_apply(z_in, rec)
    dev = _device_pos(z_in, rec)
    band = np.abs(z) <= 4 * U * mag
    assert np.array_equal(dev[~band], (z > 0)[~band]), "%s: the device's mask differs from float64 off the kink" % what
    return np.where(band, dev, z > 0)


def _resolve_n(N):
    s = _n_sms()
    return {"sms+1": 128 * s + 1, "multi": 128 * (8 * s + 3) + 77}.get(N, N)


def _tiles_per_cta(N):
    tiles = -(-N // 128)
    return -(-tiles // max(1, min(tiles, _n_sms())))


def _record(M, rng, C_std=1.0):
    """a BatchNorm record {mean, rstd, gamma rstd, beta} (float32) with rstd != 1 and gammas of both signs."""
    mean = rng.normal(size=M) * 0.3
    rstd = rng.uniform(0.5, 1.5, M) / C_std
    gamma = rng.uniform(0.5, 1.5, M) * rng.choice([-1.0, 1.0], M)
    beta = rng.normal(size=M) * 0.3
    return np.concatenate([mean, rstd, gamma * rstd, beta]).astype(np.float32)


def _batch_record(Y, rng, eps=1e-5):
    """the record of Y's own batch statistics (what the stage after a forward receives)."""
    Y = _f64(Y)
    M = Y.shape[1]
    g = rng.uniform(0.5, 1.5, M) * rng.choice([-1.0, 1.0], M)
    rec, _, _ = ref_bn_record(Y, g, rng.normal(size=M) * 0.3, eps, 0.1)
    return rec.astype(np.float32)


# ---------------------------------------------------------------------------------------------------------------------
# lin_fwd: the pipeline with the ring (all four (KP, MP) instances), its x_direct mode, the serial kernel with and without
# the ring
FWD_PATHS = [
    # id, K, M, flags
    ("pipe_k4_m4", 4, 4, ""), ("pipe_k24_m36", 24, 36, ""), ("pipe_k32_m64", 32, 64, ""), ("pipe_k36_m24", 36, 24, ""),
    ("pipe_k64_m32", 64, 32, ""), ("pipe_k36_m36", 36, 36, ""), ("pipe_k64_m64", 64, 64, ""),
    ("xdirect_k1_m32", 1, 32, ""), ("xdirect_k2_m64", 2, 64, ""), ("xdirect_k7_m32", 7, 32, ""),
    ("xdirect_k33_m32", 33, 32, ""), ("xdirect_k63_m64", 63, 64, ""),
    ("xdirect_xoff_k32_m32", 32, 32, "x_off"), ("xdirect_woff_k32_m64", 32, 64, "w_off"),
    ("serial_ring_m1_k32", 32, 1, ""), ("serial_ring_m2_k64", 64, 2, ""), ("serial_noring_m3_k7", 7, 3, ""),
    ("serial_ring_m5_k32", 32, 5, ""), ("serial_ring_m30_k36", 36, 30, ""), ("serial_noring_m33_k7", 7, 33, ""),
    ("serial_ring_m63_k64", 64, 63, ""), ("serial_yoff_k32_m32", 32, 32, "y_off"),
    ("serial_nocounters_k32_m32", 32, 32, "no_counters"), ("serial_nocounters_k64_m64", 64, 64, "no_counters"),
]
FWD_OPTS = [
    dict(stats=True, bias=True, in_bn=True, act=RELU, affine=True, running=True),
    dict(stats=False, bias=False, in_bn=False, act=NONE),
    dict(stats=True, bias=False, in_bn=True, act=LEAKY, affine=False, running=False),
    dict(stats=False, bias=True, in_bn=True, act=NONE),
    dict(stats=True, bias=True, in_bn=False, act=RELU, affine=True, running=True),
    dict(stats=False, bias=True, in_bn=False, act=LEAKY),
]
FWD_NS = [1, 2, 127, 128, 129, "sms+1", "multi"]


def _fwd_inputs(case, N, opt, mean_offset=0.0):
    cid, K, M, flags = case
    rng = _rng("fwd", cid, N, mean_offset)
    X = (rng.normal(size=(N, K)) * 1.5 + 0.2).astype(np.float32)
    W = (rng.normal(size=(M, K)) / (1.5 * math.sqrt(K))).astype(np.float32)
    bias = (rng.normal(size=M) + mean_offset).astype(np.float32) if opt["bias"] else None
    in_bn = None
    if opt["in_bn"]:
        in_bn = _record(K, rng)
        in_bn[:K] += 0.2
    st = None
    if opt["stats"]:
        st = dict(gamma=rng.uniform(-1.5, 1.5, M).astype(np.float32) if opt["affine"] else None,
                  beta=rng.normal(size=M).astype(np.float32) if opt["affine"] else None,
                  eps=1e-5, momentum=0.25,
                  rm=rng.normal(size=M).astype(np.float32) if opt["running"] else None,
                  rv=rng.uniform(0.5, 2.0, M).astype(np.float32) if opt["running"] else None,
                  nbt=opt["running"])
    return dict(X=X, W=W, bias=bias, in_bn=in_bn, act=opt["act"], st=st, flags=flags, K=K, M=M, N=N)


def _run_fwd(inp, counters=True):
    """one dn4gl_lin_fwd_f32 call with owned buffers -> {name: numpy}."""
    N, K, M, fl, st = inp["N"], inp["K"], inp["M"], inp["flags"], inp["st"]
    X = _inp(inp["X"], 1 if "x_off" in fl else 0)
    W = _inp(inp["W"], 1 if "w_off" in fl else 0)
    Y = Buf((N, M), offset=1 if "y_off" in fl else 0)
    bufs = {"Y": Y}
    rec = rm = rv = nbt = None
    if st is not None:
        rec = bufs["rec"] = Buf((4 * M,))
        if st["rm"] is not None:
            rm, rv = bufs["rm"], bufs["rv"] = Buf((M,), st["rm"]), Buf((M,), st["rv"])
        if st["nbt"]:
            nbt = torch.full((1,), 41, dtype=torch.int64, device="cuda")
    wsb = _size("dn4gl_lin_workspace_bytes", N, K, M)
    ws = Ws(wsb)
    cnt = _counters() if counters and "no_counters" not in fl else None
    _call("dn4gl_lin_fwd_f32", X, N, K, _inp(inp["in_bn"]), inp["act"], SLOPE, W, _inp(inp["bias"]), M, Y.t,
          _inp(st and st["gamma"]), _inp(st and st["beta"]), st["eps"] if st else 0.0, st["momentum"] if st else 0.0,
          rec and rec.t, rm and rm.t, rv and rv.t, nbt, ws.t, wsb, cnt, _stream())
    torch.cuda.synchronize()
    for k, b in bufs.items():
        b.check(k)
    ws.check()
    if cnt is not None:
        assert not bool(cnt.any().cpu()), "counters not left at zero"
    out = {k: b.np() for k, b in bufs.items()}
    if nbt is not None:
        out["nbt"] = nbt.cpu().numpy()
    return out


def _check_stats(Y, out, st, n, tag):
    """the record and running buffers of the batch statistics of the fp32 values Y (n fp32 adds per CTA)."""
    N, M = Y.shape
    recd, rmd, rvd = ref_bn_record(Y, st["gamma"], st["beta"], st["eps"], st["momentum"], st["rm"], st["rv"])
    mb, vb = stat_bounds(Y, n)
    Yd = _f64(Y)
    var = ((Yd - Yd.mean(0)) ** 2).mean(0)
    rstd = recd[M:2 * M]
    rb = rstd * (vb / (2 * (var + st["eps"])) + 2 * U)
    g = np.ones(M) if st["gamma"] is None else _f64(st["gamma"])
    rec = out["rec"]
    _within(rec[:M], recd[:M], mb, tag, "record mean")
    _within(rec[M:2 * M], rstd, rb, tag, "record rstd")
    _within(rec[2 * M:3 * M], recd[2 * M:3 * M], np.abs(g) * (rb + U * rstd), tag, "record gamma*rstd")
    assert _bits_equal(rec[3 * M:], np.zeros(M, np.float32) if st["beta"] is None else st["beta"]), "record beta"
    if st["rm"] is not None:
        mom = st["momentum"]
        rm_mag = (1 - mom) * np.abs(_f64(st["rm"])) + mom * np.abs(recd[:M])     # the two terms may cancel
        _within(out["rm"], rmd, mom * mb + 3 * U * rm_mag, tag, "running_mean")
        _within(out["rv"], rvd, mom * vb * (N / (N - 1) if N > 1 else 1.0) + 3 * U * np.abs(rvd), tag, "running_var")


def _check_fwd(inp, out, tag):
    N, K, st = inp["N"], inp["K"], inp["st"]
    ref, mag = ref_lin_fwd(inp["X"], inp["W"], inp["bias"], inp["in_bn"], inp["act"])
    _within(out["Y"], ref, (c_gemm(pad32(K)) + C_PRO) * U * mag, tag, "Y")
    if st is not None:
        _check_stats(out["Y"], out, st, 128 * _tiles_per_cta(N) + 16, tag)
        if st["nbt"]:
            assert int(out["nbt"][0]) == 42, "num_batches_tracked"


@pytest.mark.gpu
@pytest.mark.parametrize("N", FWD_NS)
@pytest.mark.parametrize("case", FWD_PATHS, ids=[c[0] for c in FWD_PATHS])
def test_lin_fwd(case, N):
    """Y, the BatchNorm record and the running buffers against float64, per element; options rotate over the cases."""
    opt = dict(FWD_OPTS[(FWD_PATHS.index(case) + FWD_NS.index(N)) % len(FWD_OPTS)])
    N = _resolve_n(N)
    if "no_counters" in case[3] and not opt["stats"]:
        opt.update(stats=True, affine=True, running=True)     # without statistics a NULL counters array takes the pipeline
    inp = _fwd_inputs(case, N, opt)
    out = _twice(lambda: _run_fwd(inp))
    _check_fwd(inp, out, "lin_fwd[%s-%d]" % (case[0], N))


@pytest.mark.gpu
@pytest.mark.parametrize("N", ["sms+1", "multi", 127])
@pytest.mark.parametrize("case", [c for c in FWD_PATHS if c[0] in (
    "pipe_k32_m64", "pipe_k64_m32", "xdirect_k7_m32", "serial_ring_m30_k36", "serial_nocounters_k64_m64")], ids=lambda c: c[0])
def test_lin_fwd_statistics_of_offset_channels(case, N):
    """channels whose mean is 10^3 times their spread, over several CTAs (what the shifted sums and the K* re-centring
    are for), and a one-tile grid that merges more channels than it has CTAs."""
    N = _resolve_n(N)
    opt = dict(stats=True, bias=True, in_bn=False, act=NONE, affine=True, running=True)
    inp = _fwd_inputs(case, N, opt, mean_offset=1e3)
    out = _twice(lambda: _run_fwd(inp))
    Y = _f64(out["Y"])
    assert np.all(np.abs(Y.mean(0)) > 500 * Y.std(0))
    _check_fwd(inp, out, "lin_fwd_offset[%s-%d]" % (case[0], N))


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["pipe", "serial"])
def test_lin_fwd_one_row_uses_biased_variance(path):
    """N = 1 with statistics: variance 0, rstd = 1/sqrt(eps), and the running variance takes the biased variance (0),
    where nn.BatchNorm1d refuses to train on one row."""
    case = ("n1", 32, 32, "" if path == "pipe" else "no_counters")
    opt = dict(stats=True, bias=True, in_bn=False, act=NONE, affine=True, running=True)
    inp = _fwd_inputs(case, 1, opt)
    out = _twice(lambda: _run_fwd(inp))
    st = inp["st"]
    assert _bits_equal(out["rec"][:32], out["Y"][0])
    assert np.allclose(out["rec"][32:64], 1 / math.sqrt(st["eps"]), rtol=2 * U)
    _within(out["rv"], (1 - st["momentum"]) * _f64(st["rv"]), 3 * U * _f64(st["rv"]), "lin_fwd_n1", "running_var")


# ---------------------------------------------------------------------------------------------------------------------
# lin_bwd: the 32 x 32 pipeline and its x_direct mode, the serial kernel (the three 64-wide instances, M % 4 != 0,
# K % 4 != 0 with GX, misaligned G / Yout / X, counters = NULL)
BWD_PATHS = [
    ("pipe_k32_m32", 32, 32, ""), ("pipe_k4_m8", 4, 8, ""), ("pipe_k24_m32", 24, 32, ""), ("pipe_k32_m4", 32, 4, ""),
    ("pipe_xdirect_k7_m32", 7, 32, "no_gx"), ("pipe_xdirect_xoff_k32_m32", 32, 32, "x_off no_gx"),
    ("serial_k64_m64", 64, 64, ""), ("serial_k32_m64", 32, 64, ""), ("serial_k64_m32", 64, 32, ""),
    ("serial_m30_k32", 32, 30, ""), ("serial_k7_m32_gx", 7, 32, "gx"), ("serial_goff_k32_m32", 32, 32, "g_off"),
    ("serial_yoff_k32_m32", 32, 32, "y_off"), ("serial_xoff_k32_m32_gx", 32, 32, "x_off gx"),
    ("serial_nocounters_k32_m32", 32, 32, "no_counters"),
]
BWD_OPTS = [
    dict(bn=True, g_masked=False, in_bn=True, act=RELU, G=True, Gseg=False, gx=True, dw=True, db=True),
    dict(bn=False, g_masked=False, in_bn=False, act=NONE, G=True, Gseg=False, gx=True, dw=True, db=True),
    dict(bn=True, g_masked=True, in_bn=True, act=LEAKY, G=False, Gseg=True, gx=True, dw=False, db=True),
    dict(bn=True, g_masked=False, in_bn=False, act=LEAKY, G=True, Gseg=True, gx=False, dw=True, db=False),
    dict(bn=False, g_masked=False, in_bn=True, act=NONE, G=True, Gseg=True, gx=True, dw=True, db=False),
    dict(bn=True, g_masked=True, in_bn=False, act=RELU, G=True, Gseg=False, gx=True, dw=False, db=True),
]
BWD_NS = [1, 2, 129, "sms+1", "multi"]


def _bwd_inputs(case, N, opt):
    cid, K, M, flags = case
    rng = _rng("bwd", cid, N, tuple(sorted(opt.items())))
    B = max(1, min(N, 37))
    X = (rng.normal(size=(N, K)) * 1.5 + 0.2).astype(np.float32)
    W = (rng.normal(size=(M, K)) / math.sqrt(M)).astype(np.float32)
    Y = (rng.normal(size=(N, M)) * 1.3 + 0.1).astype(np.float32)
    G = rng.normal(size=(N, M)).astype(np.float32) if opt["G"] else None
    Gseg = rng.normal(size=(B, M)).astype(np.float32) if opt["Gseg"] else None
    row2seg = np.sort(rng.integers(0, B, N)).astype(np.int32) if opt["Gseg"] else None
    bn = sums = None
    if opt["bn"]:
        bn = _batch_record(Y, rng)
        g, _ = ref_upstream(G, Gseg, row2seg, N, M)
        sums = ref_bn_bwd_sums(g, None, None, Y, bn, RELU if not opt["g_masked"] else NONE)[0].astype(np.float32)
    in_bn = _record(K, rng) if opt["in_bn"] else None
    return dict(G=G, Gseg=Gseg, row2seg=row2seg, Y=Y, bn=bn, sums=sums, g_masked=opt["g_masked"], W=W, X=X, in_bn=in_bn,
                act=opt["act"], gx=opt["gx"], dw=opt["dw"], db=opt["db"], flags=flags, K=K, M=M, N=N)


def _run_bwd(inp, counters=True):
    N, K, M, fl = inp["N"], inp["K"], inp["M"], inp["flags"]
    G = _inp(inp["G"], 1 if "g_off" in fl else 0)
    Yo = _inp(inp["Y"], 1 if "y_off" in fl else 0) if inp["bn"] is not None else None
    X = _inp(inp["X"], 1 if "x_off" in fl else 0)
    bufs = {}
    if inp["gx"]:
        bufs["GX"] = Buf((N, K))
        if inp["in_bn"] is not None:
            bufs["sums_prev"] = Buf((2 * K,))
    if inp["dw"]:
        bufs["dW"] = Buf((M, K))
    if inp["db"]:
        bufs["db"] = Buf((M,))
    wsb = _size("dn4gl_lin_workspace_bytes", N, K, M)
    ws = Ws(wsb)
    cnt = _counters() if counters and "no_counters" not in fl else None
    t = lambda k: bufs[k].t if k in bufs else None
    _call("dn4gl_lin_bwd_f32", G, _inp(inp["Gseg"]), _inp(inp["row2seg"], dtype=torch.int32), Yo, N, M, _inp(inp["bn"]),
          _inp(inp["sums"]), 1 if inp["g_masked"] else 0, _inp(inp["W"]), K, X, _inp(inp["in_bn"]), inp["act"], SLOPE,
          t("GX"), t("sums_prev"), t("dW"), t("db"), ws.t, wsb, cnt, _stream())
    torch.cuda.synchronize()
    for k, b in bufs.items():
        b.check(k)
    ws.check()
    if cnt is not None:
        assert not bool(cnt.any().cpu()), "counters not left at zero"
    return {k: b.np() for k, b in bufs.items()}


def _check_bwd(inp, out, tag):
    N, K, M = inp["N"], inp["K"], inp["M"]
    g, gmag = ref_upstream(inp["G"], inp["Gseg"], inp["row2seg"], N, M)
    pos = None
    if inp["bn"] is not None and not inp["g_masked"]:
        pos = _mask(inp["Y"], inp["bn"], tag + " G mask")
    gy, gymag = ref_gy(g, gmag, inp["Y"], inp["bn"], inp["sums"], inp["g_masked"], pos)
    pos_in = None
    if inp["in_bn"] is not None and inp["act"] != NONE:
        pos_in = _mask(inp["X"], inp["in_bn"], tag + " X mask")
    r = ref_lin_bwd(gy, gymag, inp["W"], inp["X"], inp["in_bn"], inp["act"], pos_in=pos_in)
    T = _tiles_per_cta(N)
    if "GX" in out:
        _within(out["GX"], r["GX"], (c_gemm(pad32(M)) + C_GY + 1) * U * r["GXmag"], tag, "GX")
        if "sums_prev" in out:
            sp, spmag = ref_sums_prev(out["GX"], inp["X"], inp["in_bn"])
            _within(out["sums_prev"], sp, (128 * T + 16 + 3) * U * spmag, tag, "sums_prev")
    if "dW" in out:
        accw = not (pad32(K) == 64 and pad32(M) == 64)
        _within(out["dW"], r["dW"], (c_dw(T, accw) + C_GY + C_PRO) * U * r["dWmag"], tag, "dW")
    if "db" in out:
        _within(out["db"], r["db"], (128 * T + 16 + C_GY) * U * r["dbmag"], tag, "db")


@pytest.mark.gpu
@pytest.mark.parametrize("N", BWD_NS)
@pytest.mark.parametrize("case", BWD_PATHS, ids=[c[0] for c in BWD_PATHS])
def test_lin_bwd(case, N):
    """GX, sums_prev, dW and db against float64 per element; options rotate over the cases."""
    Nr = _resolve_n(N)
    opt = dict(BWD_OPTS[(BWD_PATHS.index(case) + BWD_NS.index(N)) % len(BWD_OPTS)])
    fl = case[3]
    if "no_gx" in fl:
        opt["gx"] = False
    if "gx" in fl.split():
        opt["gx"] = True
    if "g_off" in fl:
        opt["G"] = True
    if "y_off" in fl:
        opt["bn"] = True
    inp = _bwd_inputs(case, Nr, opt)
    out = _twice(lambda: _run_bwd(inp))
    _check_bwd(inp, out, "lin_bwd[%s-%s]" % (case[0], N))


@pytest.mark.gpu
@pytest.mark.parametrize("K,M", [(32, 32), (64, 64), (7, 30)])
def test_lin_bwd_empty_batch_writes_zeros(K, M):
    """N = 0: dW, db and sums_prev are zero over NaN-filled buffers, nothing else is written."""
    dW, db, sp = Buf((M, K)), Buf((M,)), Buf((2 * K,))
    wsb = _size("dn4gl_lin_workspace_bytes", 0, K, M)
    ws, cnt = Ws(max(wsb, 1)), _counters()
    dummy = torch.zeros(4, device="cuda")
    _call("dn4gl_lin_bwd_f32", dummy, None, None, None, 0, M, None, None, 0, _inp(np.ones((M, K), np.float32)), K, dummy,
          _inp(_record(K, _rng("n0"))), RELU, 0.0, None, sp.t, dW.t, db.t, ws.t, wsb, cnt, _stream())
    torch.cuda.synchronize()
    for name, b in (("dW", dW), ("db", db), ("sums_prev", sp)):
        b.check(name)
        assert not np.any(b.np()), name


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["fwd", "bwd"])
def test_pipeline_and_serial_both_meet_the_bound(which):
    """one shape both paths accept, forced apart with counters = NULL: each meets the float64 bound on its own."""
    N = _resolve_n("sms+1")
    if which == "fwd":
        opt = dict(stats=True, bias=True, in_bn=True, act=RELU, affine=True, running=True)
        inp = _fwd_inputs(("both", 32, 32, ""), N, opt)
        for counters in (True, False):
            _check_fwd(inp, _run_fwd(inp, counters), "pipe_vs_serial_fwd[%s]" % counters)
    else:
        inp = _bwd_inputs(("both", 32, 32, ""), N, BWD_OPTS[0])
        for counters in (True, False):
            _check_bwd(inp, _run_bwd(inp, counters), "pipe_vs_serial_bwd[%s]" % counters)


# ---------------------------------------------------------------------------------------------------------------------
# path witness: the kernels that ran, by name
def _kernels_of(fn):
    from torch.profiler import ProfilerActivity, profile
    fn()                                          # first launches load the modules outside the profile
    with profile(activities=[ProfilerActivity.CUDA]) as p:
        fn()
        torch.cuda.synchronize()
    return sorted({e.name for e in p.events() if re.search(r"\b(lin|bn)_\w*kernel", e.name)})


WITNESS = [
    # (fwd | bwd, case id, option index, expected kernel name patterns)
    ("fwd", "pipe_k64_m64", 0, [r"lin_fwd_pipe_kernel<64, 64,"]),
    ("fwd", "xdirect_k7_m32", 0, [r"lin_fwd_pipe_kernel<32, 32,"]),
    ("fwd", "serial_ring_m30_k36", 0, [r"lin_fwd_kernel<64, 32, 3,", r"bn_finalize_kernel"]),
    ("fwd", "serial_noring_m33_k7", 1, [r"lin_fwd_kernel<32, 64, 0,"]),
    ("fwd", "serial_yoff_k32_m32", 4, [r"lin_fwd_kernel<32, 32, 3,", r"bn_finalize_kernel"]),
    ("fwd", "serial_nocounters_k64_m64", 0, [r"lin_fwd_kernel<64, 64, 3,", r"bn_finalize_kernel"]),
    ("bwd", "pipe_k32_m32", 0, [r"lin_bwd_pipe_kernel<32, 32,"]),
    ("bwd", "pipe_xdirect_k7_m32", 1, [r"lin_bwd_pipe_kernel<32, 32,"]),
    ("bwd", "serial_k64_m64", 0, [r"lin_bwd_kernel<64, 64, 0,", r"lin_bwd_reduce_kernel"]),
    ("bwd", "serial_k32_m64", 0, [r"lin_bwd_kernel<32, 64, 0,", r"lin_bwd_reduce_kernel"]),
    ("bwd", "serial_k64_m32", 0, [r"lin_bwd_kernel<64, 32, 0,", r"lin_bwd_reduce_kernel"]),
    ("bwd", "serial_m30_k32", 0, [r"lin_bwd_kernel<32, 32, 0,", r"lin_bwd_reduce_kernel"]),
    ("bwd", "serial_k7_m32_gx", 0, [r"lin_bwd_kernel<32, 32, 0,", r"lin_bwd_reduce_kernel"]),
    ("bwd", "serial_nocounters_k32_m32", 0, [r"lin_bwd_kernel<32, 32, 2,", r"lin_bwd_reduce_kernel"]),
]


@pytest.mark.gpu
def test_path_witness():
    """one call per path case under torch.profiler: the kernel names (and the serial kernels' ring depth) are the ones
    the dispatch promises, so the case matrix above cannot quietly collapse onto one path."""
    N = _resolve_n("sms+1")
    lines = []
    for kind, cid, oi, expect in WITNESS:
        if kind == "fwd":
            case = next(c for c in FWD_PATHS if c[0] == cid)
            opt = dict(FWD_OPTS[oi])
            if "no_counters" in case[3]:
                opt.update(stats=True, affine=True, running=True)
            inp = _fwd_inputs(case, N, opt)
            names = _kernels_of(lambda: _run_fwd(inp))
        else:
            case = next(c for c in BWD_PATHS if c[0] == cid)
            opt = dict(BWD_OPTS[oi])
            opt["gx"] = "no_gx" not in case[3]
            inp = _bwd_inputs(case, N, opt)
            names = _kernels_of(lambda: _run_bwd(inp))
        short = [re.search(r"(lin|bn)_\w*kernel(<[^>]*>)?", n).group(0) for n in names]
        lines.append("%s %-28s %s" % (kind, cid, " + ".join(short)))
        for pat in expect:
            assert any(re.search(pat, n) for n in names), (cid, pat, names)
        assert len(names) == len(expect), (cid, names)
    print("\n" + "\n".join(lines))


# ---------------------------------------------------------------------------------------------------------------------
# BatchNorm kernels: bn_stats, bn_act, bn_bwd_sums, bn_bwd_apply, bn_act_pool, segment_ids
BN_MS = [1, 3, 4, 5, 8, 9, 16, 17, 32, 33, 64, 65, 100, 128]
BN_NS = ["1", "rp-1", "rp+1", "8rp-1", "8rp+1", "cap"]


def _chp(M):
    c = 1
    while c < (M + 3) // 4:
        c <<= 1
    return c


def _bn_n(M, key):
    rp = 256 // _chp(M)
    return {"1": 1, "rp-1": rp - 1, "rp+1": rp + 1, "8rp-1": 8 * rp - 1, "8rp+1": 8 * rp + 1,
            "cap": 4 * _n_sms() * 8 * rp + 3}[key]


def _run_stats(Y, M, gamma, beta, rm0, rv0):
    N = Y.shape[0]
    rec, rm, rv = Buf((4 * M,)), Buf((M,), rm0), Buf((M,), rv0)
    nbt = torch.zeros(1, dtype=torch.int64, device="cuda")
    wsb = _size("dn4gl_bn_stats_workspace_bytes", N, M)
    ws = Ws(wsb)
    _call("dn4gl_bn_stats_f32", _inp(Y), N, M, _inp(gamma), _inp(beta), 1e-5, 0.25, rm.t, rv.t, nbt, rec.t, ws.t, wsb,
          _stream())
    torch.cuda.synchronize()
    for k, b in (("rec", rec), ("rm", rm), ("rv", rv)):
        b.check(k)
    ws.check()
    return dict(rec=rec.np(), rm=rm.np(), rv=rv.np(), nbt=nbt.cpu().numpy())


def _run_bn_act(Y, M, rec, act, off=0):
    out = Buf(Y.shape, offset=off)
    _call("dn4gl_bn_act_f32", _inp(Y, off), Y.shape[0], M, _inp(rec), act, SLOPE, out.t, _stream())
    torch.cuda.synchronize()
    out.check("out")
    return dict(out=out.np())


def _run_bwd_sums(G, Gseg, row2seg, Y, M, rec, act):
    N = Y.shape[0]
    sums = Buf((2 * M,))
    wsb = _size("dn4gl_bn_bwd_sums_workspace_bytes", N, M)
    ws, cnt = Ws(wsb), _counters()
    _call("dn4gl_bn_bwd_sums_f32", _inp(G), _inp(Gseg), _inp(row2seg, dtype=torch.int32), _inp(Y), N, M, _inp(rec), act,
          SLOPE, sums.t, ws.t, wsb, cnt, _stream())
    torch.cuda.synchronize()
    sums.check("sums")
    ws.check()
    assert not bool(cnt.any().cpu()), "counters not left at zero"
    return dict(sums=sums.np())


def _run_bwd_apply(G, Y, M, rec, sums, act, off=0):
    GX = Buf(Y.shape, offset=off)
    _call("dn4gl_bn_bwd_apply_f32", _inp(G, off), _inp(Y, off), Y.shape[0], M, _inp(rec), _inp(sums), act, SLOPE, GX.t,
          _stream())
    torch.cuda.synchronize()
    GX.check("GX")
    return dict(GX=GX.np())


def _check_bn_act(Y, rec, act, out, tag):
    pos = _mask(Y, rec, tag)
    z, mag = ref_bn_apply(Y, rec)
    ref = np.where(pos, z, z * (0.0 if act == RELU else SLOPE)) if act != NONE else z
    _within(out, ref, 3 * U * mag, tag, "bn_act")


@pytest.mark.gpu
@pytest.mark.parametrize("Nk", BN_NS)
@pytest.mark.parametrize("M", BN_MS)
def test_bn_kernels(M, Nk):
    """bn_stats (record + running buffers), bn_act (three activations), bn_bwd_sums (G, Gseg or both) and bn_bwd_apply
    at every CHP instance, around the 256/CHP and 8 * 256/CHP row boundaries and at a grid-filling N."""
    N = _bn_n(M, Nk)
    rng = _rng("bn", M, Nk)
    i = BN_MS.index(M) + BN_NS.index(Nk)
    act = (RELU, LEAKY, NONE)[i % 3]
    Y = (rng.normal(size=(N, M)) * rng.uniform(0.5, 3, M) + rng.normal(size=M) * 4).astype(np.float32)
    gamma = rng.uniform(-1.5, 1.5, M).astype(np.float32) if i % 2 else None
    beta = rng.normal(size=M).astype(np.float32) if i % 2 else None
    rm0, rv0 = rng.normal(size=M).astype(np.float32), rng.uniform(0.5, 2, M).astype(np.float32)
    tag = "bn[%d-%s]" % (M, Nk)

    # bn_stats: per-thread rows = row groups per CTA (grid = min(ceil(groups / 8), 4 SMs))
    out = _twice(lambda: _run_stats(Y, M, gamma, beta, rm0, rv0))
    rp = 256 // _chp(M)
    groups = -(-N // rp)
    n = -(-groups // max(1, min(-(-groups // 8), 4 * _n_sms()))) + 16
    st = dict(gamma=gamma, beta=beta, eps=1e-5, momentum=0.25, rm=rm0, rv=rv0, nbt=False)
    _check_stats(Y, out, st, n, tag)
    assert int(out["nbt"][0]) == 1
    rec = out["rec"]

    for a in (NONE, RELU, LEAKY):
        _check_bn_act(Y, rec, a, _twice(lambda: _run_bn_act(Y, M, rec, a))["out"], tag + "-act%d" % a)

    B = max(1, min(N, 29))
    G = rng.normal(size=(N, M)).astype(np.float32) if i % 3 != 1 else None
    Gseg = rng.normal(size=(B, M)).astype(np.float32) if i % 3 != 0 else None
    row2seg = np.sort(rng.integers(0, B, N)).astype(np.int32) if Gseg is not None else None
    pos = _mask(Y, rec, tag + " mask")
    sums = _twice(lambda: _run_bwd_sums(G, Gseg, row2seg, Y, M, rec, act))["sums"]
    ref, mag = ref_bn_bwd_sums(G, Gseg, row2seg, Y, rec, act, pos=pos)
    grid_lb = max(1, min(-(-N // (8 * rp)), _n_sms()))
    n = -(-N // (grid_lb * rp)) + 16
    _within(sums, ref, (n + 4) * U * mag, tag, "bn_bwd_sums")

    Gf = G if G is not None else rng.normal(size=(N, M)).astype(np.float32)
    GX = _twice(lambda: _run_bwd_apply(Gf, Y, M, rec, sums, act))["GX"]
    ref, mag = ref_bn_bwd_apply(Gf, Y, rec, sums, act, pos=pos)
    _within(GX, ref, C_GY * U * mag, tag, "bn_bwd_apply")


@pytest.mark.gpu
@pytest.mark.parametrize("M", [3, 5, 17, 32, 100])
def test_bn_elementwise_misaligned(M):
    """bn_act and bn_bwd_apply on the scalar path: every operand one float past a 16-byte boundary."""
    rng = _rng("mis", M)
    N = 1000 + M
    Y = (rng.normal(size=(N, M)) * 2 + 1).astype(np.float32)
    G = rng.normal(size=(N, M)).astype(np.float32)
    rec = _batch_record(Y, rng)
    for a in (NONE, RELU, LEAKY):
        out = _twice(lambda: _run_bn_act(Y, M, rec, a, off=1))["out"]
        _check_bn_act(Y, rec, a, out, "bn_act_mis[%d-%d]" % (M, a))
        pos = _mask(Y, rec, "mis")
        sums = ref_bn_bwd_sums(G, None, None, Y, rec, a, pos=pos)[0].astype(np.float32)
        GX = _twice(lambda: _run_bwd_apply(G, Y, M, rec, sums, a, off=1))["GX"]
        ref, mag = ref_bn_bwd_apply(G, Y, rec, sums, a, pos=pos)
        _within(GX, ref, C_GY * U * mag, "bn_bwd_apply_mis[%d-%d]" % (M, a), "GX")


def _run_pool(Y, M, rec, act, seg, mode):
    N, B = Y.shape[0], len(seg) - 1
    out, pooled, ids = Buf((N, M)), Buf((B, M)), Buf((N,), dtype=torch.int32)
    segt = _inp(seg, dtype=torch.int32)
    _call("dn4gl_bn_act_pool_f32", _inp(Y), N, M, _inp(rec), act, SLOPE, out.t, segt, B, mode, pooled.t, _stream())
    _call("dn4gl_segment_ids_i32", segt, B, N, ids.t, _stream())
    torch.cuda.synchronize()
    for k, b in (("out", out), ("pooled", pooled), ("ids", ids)):
        b.check(k)
    return dict(out=out.np(), pooled=pooled.np(), ids=ids.np())


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [0, 1], ids=["sum", "mean"])
@pytest.mark.parametrize("M", BN_MS)
def test_bn_act_pool_and_segment_ids(M, mode):
    """segments of 0 and 1 rows, every tail of the 4-row unroll, more than 4 RP rows, and more segments than the grid
    (the grid-stride loop over graphs): out against float64, pooled against float64 sums of the device's out,
    segment_ids bit-exact."""
    rp = 256 // _chp(M)
    rng = _rng("pool", M, mode)
    base = [0, 1, 2, 3, 4, 5, rp - 1, rp, rp + 1, 2 * rp + 3, 3 * rp + 1, 4 * rp - 1, 4 * rp, 4 * rp + 1, 5 * rp + 2,
            9 * rp + 7, 0, 1]
    B = 8 * _n_sms() + 5
    lens = np.array([base[i % len(base)] if i < 2 * len(base) else rng.integers(0, 3) for i in range(B)])
    seg = np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)
    N = int(seg[-1])
    act = (RELU, LEAKY, NONE)[(M + mode) % 3]
    Y = (rng.normal(size=(N, M)) * 2 + 0.5).astype(np.float32)
    rec = _batch_record(Y, rng)
    r = _twice(lambda: _run_pool(Y, M, rec, act, seg, mode))
    tag = "bn_act_pool[%d-%d]" % (M, mode)
    _check_bn_act(Y, rec, act, r["out"], tag)
    ref, mag = ref_pool(r["out"], seg, mode)
    n = np.maximum(-(-lens // rp), 1)[:, None] + 5 + 8 + 3
    _within(r["pooled"], ref, n * U * mag, tag, "pooled")
    assert _bits_equal(r["ids"], ref_segment_ids(seg, N)), "segment_ids"
