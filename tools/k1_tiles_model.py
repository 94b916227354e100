"""CPU model of the aggregation kernel's tile construction (csrc/spmm_tiled.cu: tile_boundary / make_row_tiles_kernel /
collect_cut_heavy_kernel), no GPU: graphs longer than the window are cut -> checked slow path.  Checks on the C2
structure and on random partitions that the tiles stay a partition of [0, N), never exceed the stage, and that the
window search of collect_cut_heavy finds the tile of every row; prints the share of rows left in cut tiles.
Usage: python tools/k1_tiles_model.py [window_rows]"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def boundary(seg_ptr, C, N, k, T):
    """(row, aligned) exactly as the device function computes it."""
    if k >= T:
        return N, True
    target = k * C
    lo = int(np.searchsorted(seg_ptr, target, side="left"))        # first g with seg_ptr[g] >= target
    gs = int(seg_ptr[lo])
    if gs < target + C:
        return gs, True
    return target, False


def make_tiles(seg_ptr, C):
    N = int(seg_ptr[-1])
    T = (N + C - 1) // C
    tiles = []
    for k in range(T):
        r0, a0 = boundary(seg_ptr, C, N, k, T)
        r1, a1 = boundary(seg_ptr, C, N, k + 1, T)
        tiles.append((r0, r1, not (a0 and a1)))
    return tiles


def check(seg_ptr, C):
    N = int(seg_ptr[-1])
    tiles = make_tiles(seg_ptr, C)
    T = len(tiles)
    assert tiles[0][0] == 0 and tiles[-1][1] == N
    for (a0, a1, _), (b0, _, _) in zip(tiles[:-1], tiles[1:]):
        assert a1 == b0 and a0 <= a1
    starts = set(int(x) for x in seg_ptr)
    for r0, r1, cut in tiles:
        if not cut:
            assert r1 - r0 <= 2 * C, (r0, r1)
            assert r0 in starts and r1 in starts          # closed tiles hold whole graphs only
    # the tile of every row, found as collect_cut_heavy_kernel does (window of the row, then one step left)
    x = np.array([t[0] for t in tiles]); y = np.array([t[1] for t in tiles])
    r = np.arange(N)
    k = np.minimum(r // C, T - 1)
    k = np.where(r < x[k], k - 1, k)
    assert ((x[k] <= r) & (r < y[k])).all()
    cut_rows = sum(r1 - r0 for r0, r1, cut in tiles if cut)
    return cut_rows / max(N, 1), max((r1 - r0 for r0, r1, cut in tiles if not cut), default=0)


def main():
    C = int(sys.argv[1]) if len(sys.argv) > 1 else 311
    rng = np.random.default_rng(0)
    for trial in range(300):                                           # random partitions incl. graphs of every length class
        n = rng.integers(1, 4 * C, int(rng.integers(1, 60)))
        if trial % 3 == 0:
            n = np.minimum(n, int(rng.integers(1, 2 * C + 2)))
        seg = np.concatenate([[0], np.cumsum(n)])
        check(seg, C)
    from dummynode4graphlearning_b200 import synth
    from oracle import transforms as OT   # dev tool: the oracle builds the C2 structure on the host
    conj = OT.tu_conjugate(OT.tu_add_dummy(synth.tu_batch("proteins", 1113, seed=0)))
    seg = conj["node_ptr"].astype(np.int64)
    share, biggest = check(seg, C)
    print("C2, window %d: %.1f %% of the rows in cut tiles (checked slow path), largest closed tile %d rows"
          % (C, 100 * share, biggest))


if __name__ == "__main__":
    main()
