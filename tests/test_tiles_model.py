"""CPU: invariants of the aggregation kernel's tile construction on the host model (tools/k1_tiles_model.py restates
csrc/spmm_tiled.cu tile_boundary / make_row_tiles_kernel / collect_cut_heavy_kernel): the tiles partition [0, N), closed
tiles hold whole graphs and fit one stage, and the window search finds every row's tile.  The device code itself is
covered by the GPU aggregation tests (tests/test_agg_gpu.py, every ring size)."""
import importlib.util
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
spec = importlib.util.spec_from_file_location("k1_tiles_model", os.path.join(ROOT, "tools", "k1_tiles_model.py"))
model = importlib.util.module_from_spec(spec)
spec.loader.exec_module(model)


@pytest.mark.parametrize("C", [1, 2, 7, 64, 311])
def test_tiles_partition_rows(C):
    rng = np.random.default_rng(C)
    for trial in range(120):
        n = rng.integers(1, 4 * C + 2, int(rng.integers(1, 40)))
        if trial % 3 == 0:
            n = np.minimum(n, int(rng.integers(1, 2 * C + 2)))
        seg = np.concatenate([[0], np.cumsum(n)])
        _, biggest = model.check(seg, C)
        assert biggest <= 2 * C


def test_a_graph_longer_than_the_window_is_cut():
    # window 10; graphs of 8, 19 (spans window 1 = rows [10, 20)) and 3 rows: the 19-row graph is cut at 10
    seg = np.array([0, 8, 27, 30])
    assert model.make_tiles(seg, 10) == [(0, 10, True), (10, 27, True), (27, 30, False)]
