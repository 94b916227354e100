"""Import the UNMODIFIED reference sources from the checkout DN4GL_REFERENCE_ROOT names, under the shims.

TEST SCAFFOLDING.  Works only where such a checkout exists; everything that needs it is guarded by
``available()``.  Used by ``oracle/gen_golden.py`` to produce tests/golden/* and by the ``reference-live`` CPU tests
that re-check the standalone restatement (oracle/transforms.py, oracle/models.py) against the reference.
"""
import ast
import collections.abc
import importlib
import importlib.util
import os
import sys
import types

import numpy as np

REF_ROOT = os.environ.get("DN4GL_REFERENCE_ROOT") or ""
_SUB = os.path.join(REF_ROOT, "subgraph_isomorphism")
_CLS = os.path.join(REF_ROOT, "graph_classification")

_state = {}


def available():
    return os.path.isdir(_SUB) and os.path.isdir(_CLS)


def _install_shims():
    if _state.get("shims"):
        return
    from .shims import fake_dgl, fake_igraph, pyg_stub

    ig = types.ModuleType("igraph")
    ig.Graph = fake_igraph.Graph
    ig.read = fake_igraph.read
    sys.modules["igraph"] = ig

    dgl = types.ModuleType("dgl")
    fn = types.ModuleType("dgl.function")
    fn.sum = fake_dgl.function.sum
    fn.TargetCode = fake_dgl.function.TargetCode                      # dgl 0.4 names used by models/rgcn.py:157-161
    fn.CopyMessageFunction = fake_dgl.function.CopyMessageFunction
    fn.copy_u = fake_dgl.function.copy_u
    dgl.function = fn
    dgl.DGLGraph = fake_dgl.DGLGraph
    dgl.batch = fake_dgl.batch
    dgl.__version__ = fake_dgl.__version__
    sys.modules["dgl"] = dgl
    sys.modules["dgl.function"] = fn

    six = types.ModuleType("torch._six")  # models/container.py:10 (removed in torch 2.x)
    six.container_abcs = collections.abc
    sys.modules["torch._six"] = six

    pyg_stub.install(sys.modules)
    _state["shims"] = True


def subgraph():
    """Namespace with the reference's subgraph_isomorphism objects."""
    if "sub" in _state:
        return _state["sub"]
    _install_shims()
    if _SUB not in sys.path:
        sys.path.insert(0, _SUB)
    ns = types.SimpleNamespace()
    ns.constants = importlib.import_module("constants")
    ns.models = importlib.import_module("models")
    ns.rgin = importlib.import_module("models.rgin")
    ns.dmpnn = importlib.import_module("models.dmpnn")
    ns.rgcn = importlib.import_module("models.rgcn")
    ns.compgcn = importlib.import_module("models.compgcn")
    ns.pred = importlib.import_module("models.pred")
    ns.embed = importlib.import_module("models.embed")
    ns.filter = importlib.import_module("models.filter")
    ns.basemodel = importlib.import_module("models.basemodel")
    ns.graph_utils = importlib.import_module("utils.graph")
    ns.dl = importlib.import_module("utils.dl")
    ns.io = importlib.import_module("utils.io")
    ns.train_funcs = _extract_functions(
        os.path.join(_SUB, "train.py"),
        ["process_model_config", "add_dummy_nodes_edges", "add_reversed_edges", "calculate_degrees", "remove_loops",
         "calculate_norms", "calculate_eigenvalues"],
        extra={"compute_norm": ns.graph_utils.compute_norm,
               "compute_largest_eigenvalues": ns.graph_utils.compute_largest_eigenvalues},
    )
    import numba
    ns.dataset_funcs = _extract_functions(
        os.path.join(_SUB, "dataset.py"),
        ["long_item_bisect_left", "compute_nodeseq_subisoweights", "compute_edgeseq_subisoweights"],
        extra={"numba": numba, "np": np},
    )
    _state["sub"] = ns
    return ns


def _extract_functions(path, names, extra=None):
    """exec selected top-level ``def``s of a reference file verbatim (train.py cannot be
    imported whole: it needs tensorboardX, sklearn metrics, the old-DGL ``dataset.Graph``)."""
    import math
    from copy import deepcopy

    import torch as th

    consts = importlib.import_module("constants")
    src = open(path).read()
    tree = ast.parse(src)
    glb = {"th": th, "math": math, "deepcopy": deepcopy}
    glb.update({k: getattr(consts, k) for k in dir(consts) if not k.startswith("__")})

    class EdgeSeqDataset:  # only used in isinstance() dispatch
        pass

    class GraphAdjDataset(list):
        pass

    glb["EdgeSeqDataset"] = EdgeSeqDataset
    glb["GraphAdjDataset"] = GraphAdjDataset
    glb.update(extra or {})       # names train.py imports from utils.graph
    for node in tree.body:
        if isinstance(node, ast.FunctionDef) and node.name in names:
            code = compile(ast.Module(body=[node], type_ignores=[]), path, "exec")
            exec(code, glb)
    out = types.SimpleNamespace(**{n: glb[n] for n in names})
    out.GraphAdjDataset = GraphAdjDataset
    return out


def _load_by_path(name, path):
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def classification():
    """Namespace with the reference's graph_classification objects (loaded by file path to
    avoid models/__init__.py pulling diffpool/hgpsl and their extra PyG imports)."""
    if "cls" in _state:
        return _state["cls"]
    _install_shims()
    ns = types.SimpleNamespace()
    ns.tu = _load_by_path("_ref_tu_data_processing",
                          os.path.join(_CLS, "data_processing", "tu_data_processing.py"))
    ns.gconv = _load_by_path("_ref_gconv",
                             os.path.join(_CLS, "graph_neural_networks", "models", "gconv.py"))
    ns.rgconv = _load_by_path("_ref_rgconv",
                              os.path.join(_CLS, "graph_neural_networks", "models", "rgconv.py"))
    _state["cls"] = ns
    return ns
