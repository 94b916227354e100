"""CPU: the on-disk TU reader / writer (SURVEY.md 8(f) rank 4) against the reference-generated goldens, and round trips."""
import os
import tempfile

import numpy as np
import pytest

from dummynode4graphlearning_b200.graph_classification import io as tuio
from helpers import load_golden
from oracle import transforms as OT


@pytest.mark.parametrize("case", ["appB", "mutag12", "proteins8"])
def test_writer_matches_reference_save_graph_data(case):
    """tu_file_lines(CONJ batch) == the text the reference's save_graph_data wrote for the same graphs."""
    g = load_golden("transforms")["tu/" + case]
    conj = OT.tu_conjugate(OT.tu_add_dummy(g["inp"]))
    mine = tuio.tu_file_lines(conj)
    for suffix, lines in g["conj_files"].items():
        assert mine[suffix] == lines, suffix


@pytest.mark.parametrize("case", ["mutag12", "proteins8"])
def test_reader_round_trip_and_reference_loader_equivalence(case):
    """write (reference layout) -> load_tu_dir -> the same batch; and dummy-augmenting the loaded batch gives what the
    reference's load_graph_data_from_TUDatadir(with_dummy=True) built from those files (golden)."""
    g = load_golden("transforms")["tu/" + case]
    b = dict(g["inp"])
    b["vid"] = np.concatenate([np.arange(n) for n in np.diff(b["node_ptr"])]).astype(np.int32)
    b["eid"] = np.concatenate([np.arange(n) for n in np.diff(b["edge_ptr"])]).astype(np.int32)
    with tempfile.TemporaryDirectory() as d:
        raw = os.path.join(d, "DS", "raw")
        tuio.save_tu_dir(b, raw)
        assert sorted(os.listdir(raw))[0].startswith("DS_")
        back = tuio.load_tu_dir(os.path.join(d, "DS"))
    for k in ("node_ptr", "edge_ptr", "src", "dst", "vlabel", "elabel"):
        assert np.array_equal(back[k], b[k]), k
    if "vattr" in b:
        assert np.allclose(back["vattr"], b["vattr"], rtol=0, atol=0)
    dummy = OT.tu_add_dummy(back)
    for k in ("node_ptr", "edge_ptr", "src", "dst", "vlabel", "elabel", "v_is_dummy", "e_is_dummy"):
        assert np.array_equal(dummy[k], g["dummy"][k]), k


def test_label_shift_and_defaults():
    """labels whose minimum is not 1 are shifted to start at 1; missing label files mean all ones (:153-171)."""
    with tempfile.TemporaryDirectory() as d:
        def w(name, lines):
            with open(os.path.join(d, "X_" + name + ".txt"), "w") as f:
                f.write("\n".join(lines) + "\n")
        w("A", ["1, 2", "2, 1", "3, 4", "4, 3"])
        w("graph_indicator", ["1", "1", "2", "2"])
        w("node_labels", ["0", "3", "0", "1"])
        w("graph_labels", ["-1", "1"])
        b = tuio.load_tu_dir(d)
    assert b["vlabel"].tolist() == [1, 4, 1, 2] and b["elabel"].tolist() == [1, 1, 1, 1] and not b["has_edge_labels"]
    assert b["node_ptr"].tolist() == [0, 2, 4] and b["edge_ptr"].tolist() == [0, 2, 4] and b["y"].tolist() == [-1, 1]
    assert b["src"].tolist() == [0, 1, 2, 3] and b["dst"].tolist() == [1, 0, 3, 2]


def _tu_dir_with_decimal_attributes(d, shape="proteins", nb=6, seed=3):
    from dummynode4graphlearning_b200 import synth
    b = synth.tu_batch(shape, nb, seed=seed)
    b["vattr"] = np.round(np.random.default_rng(seed).normal(size=len(b["vlabel"])), 3)   # text that float32 would not keep
    b["vid"] = np.concatenate([np.arange(n) for n in np.diff(b["node_ptr"])]).astype(np.int32)
    b["eid"] = np.concatenate([np.arange(n) for n in np.diff(b["edge_ptr"])]).astype(np.int32)
    raw = os.path.join(d, "PROTEINS", "raw")
    tuio.save_tu_dir(b, raw)
    return raw


@pytest.mark.reference_live
def test_convert_tu_dataset_host_logic_equals_reference_main(monkeypatch):
    """convert_tu_dataset == the body of tu_data_processing.py's __main__ (:431-456) on the same raw directory, file by
    file and byte by byte, attributes included.  The GPU graph construction is replaced by the oracle's here (CPU
    test of the host logic: attribute passthrough, directory naming, labels); tests/test_zzz_convert_gpu.py runs the real
    thing."""
    import dummynode4graphlearning_b200.transforms as T
    from oracle import refload
    monkeypatch.setattr(T, "to_device", lambda b, device: b)
    monkeypatch.setattr(T, "tu_add_dummy", OT.tu_add_dummy)
    monkeypatch.setattr(T, "tu_conjugate", OT.tu_conjugate)
    tu = refload.classification().tu
    with tempfile.TemporaryDirectory() as d:
        raw = _tu_dir_with_decimal_attributes(d)
        out = tuio.convert_tu_dataset(raw, "PROTEINS", "cpu")
        assert sorted(out) == ["CONJ_", "DUMMY_", "LINE_"]
        for prefix, with_dummy, conj in (("DUMMY_", True, False), ("LINE_", False, True), ("CONJ_", True, True)):
            assert out[prefix] == os.path.join(d, prefix + "PROTEINS", "raw")
            graphs = tu.load_graph_data_from_TUDatadir(raw, with_dummy=with_dummy)
            if conj:
                graphs = [tu.convert_conjugate_graph_forward(g) for g in graphs]
            ref_dir = os.path.join(d, "ref", prefix + "PROTEINS", "raw")
            os.makedirs(ref_dir)
            tu.save_graph_data(graphs, ref_dir)
            tu.save_graph_labels(tu.load_graph_labels_from_TUDatadir(raw), ref_dir)
            assert sorted(os.listdir(ref_dir)) == sorted(os.listdir(out[prefix])), prefix
            for name in os.listdir(ref_dir):
                assert open(os.path.join(ref_dir, name)).read() == open(os.path.join(out[prefix], name)).read(), (prefix, name)
            assert any(n.endswith("_attributes.txt") for n in os.listdir(ref_dir))


def _write_tiny(d, A, gi, y):
    for name, lines in (("A", A), ("graph_indicator", gi), ("node_labels", ["1"] * len(gi)), ("graph_labels", y)):
        with open(os.path.join(d, "X_" + name + ".txt"), "w") as f:
            f.write("\n".join(lines) + "\n")


def test_graphs_without_edges():
    """App. A-2: the reference's edge walk never reaches graphs after the last edge's graph (they are dropped, labels kept
    in y_all); graphs without edges before that are produced with m = 0."""
    with tempfile.TemporaryDirectory() as d:
        _write_tiny(d, ["1, 2", "2, 1"], ["1", "1", "2", "2"], ["1", "-1"])
        b = tuio.load_tu_dir(d)
        assert b["num_graphs"] == 1 and b["node_ptr"].tolist() == [0, 2] and b["edge_ptr"].tolist() == [0, 2]
        assert b["vlabel"].tolist() == [1, 1] and b["y"].tolist() == [1] and b["y_all"].tolist() == [1, -1]
        keep = tuio.load_tu_dir(d, keep_trailing_edgeless=True)
        assert keep["num_graphs"] == 2 and keep["node_ptr"].tolist() == [0, 2, 4] and keep["edge_ptr"].tolist() == [0, 2, 2]
    with tempfile.TemporaryDirectory() as d:
        _write_tiny(d, ["1, 2", "2, 1", "5, 6", "6, 5"], ["1", "1", "2", "2", "3", "3"], ["1", "1", "1"])
        b = tuio.load_tu_dir(d)
        assert b["num_graphs"] == 3 and b["edge_ptr"].tolist() == [0, 2, 2, 4] and "y_all" not in b


@pytest.mark.reference_live
@pytest.mark.parametrize("A,gi", [(["1, 2", "2, 1"], ["1", "1", "2", "2"]),
                                  (["1, 2", "2, 1", "5, 6", "6, 5"], ["1", "1", "2", "2", "3", "3"]),
                                  (["3, 4", "4, 3"], ["1", "1", "2", "2"]),
                                  (["1, 2", "2, 1"], ["1", "1", "2", "3", "3", "3"])])
def test_graphs_without_edges_live(A, gi):
    from oracle import ref_drive as rd, refload
    tu = refload.classification().tu
    with tempfile.TemporaryDirectory() as d:
        _write_tiny(d, A, gi, ["1"] * int(gi[-1]))
        ref = rd.igraphs_to_batch(tu.load_graph_data_from_TUDatadir(d, with_dummy=False))
        mine = tuio.load_tu_dir(d)
    assert mine["num_graphs"] == ref["num_graphs"]
    for k in ("node_ptr", "edge_ptr", "src", "dst", "vlabel", "elabel"):
        assert np.array_equal(mine[k], ref[k]), k
