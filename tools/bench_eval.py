"""Evaluation throughput over a resident held-out split (pipelines ``evaluate``) against the loop a user writes without
it (model.eval(), transform, forward, one ``.item()`` per batch), and the device time of the record and reduction
kernels from torch.profiler.

Workloads: GIN as in bench.py's C2 (CONJ_ transform, hidden 32, 4 layers, train_eps, sum pooling) over ~11 k
PROTEINS-shaped graphs, and the counting RGIN of tools/bench_counting.py over 'small' samples.  Every timed pass
ends in a device synchronise (metrics() / the last .item()); medians over --repeats after --warmup passes.  Writes
bench_eval_out/bench_eval.json (or --out) with the GPU name, power limit and clocks read in the same run.

    python tools/bench_eval.py [--graphs 11130] [--samples 11000] [--batch-size 512] [--repeats 7] [--warmup 2]
"""
import argparse
import json
import os
import subprocess
import sys
import time
from argparse import Namespace

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

EVAL_KERNELS = ("eval_class_rows_kernel", "eval_count_rows_kernel", "eval_reduce_kernel")


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm,clocks.mem"
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()
    except (OSError, subprocess.SubprocessError):
        out = []
    return dict(query=q, gpus=out, torch_name=torch.cuda.get_device_name(0))


def timed(fn, repeats, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(repeats):
        t0 = time.perf_counter()
        fn()                    # ends in a host read of the result, i.e. after the device is done
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts)), [float(t) for t in ts]


def kernel_times(fn):
    """device time per evaluation kernel (sum over one call of fn) from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {k: dict(calls=0, us=0.0) for k in EVAL_KERNELS}
    for e in prof.events():
        for k in EVAL_KERNELS:
            if k in e.name and e.device_type == torch.autograd.DeviceType.CUDA:
                out[k]["calls"] += 1
                out[k]["us"] += e.device_time
    return out


def gin_case(a, dev):
    from dummynode4graphlearning_b200 import synth
    from dummynode4graphlearning_b200.datasets import ResidentTUDataset
    from dummynode4graphlearning_b200.graph_classification.models import GIN
    from dummynode4graphlearning_b200.optim import FlatAdam
    from dummynode4graphlearning_b200.pipelines import ClassificationPipeline
    raw = {k: v for k, v in synth.tu_batch("proteins", a.graphs, seed=5).items() if k != "vattr"}
    ds = ResidentTUDataset(raw, dev)
    torch.manual_seed(0)
    args = Namespace(num_features=2, hidden_dim=32, num_classes=2, dropout_ratio=0.0,
                     additional={"train_eps": True, "num_layers": 4, "aggregation": "sum"}, epochs=1, device=str(dev))
    model = GIN(args).to(dev)
    pipe = ClassificationPipeline(model, FlatAdam(model.parameters(), lr=0.01), mode="conj", num_node_labels=2,
                                  node_label_min=0)
    idx = np.arange(len(ds))

    def evaluate():
        return pipe.evaluate(ds, idx, batch_size=a.batch_size).metrics()

    def hand():
        import torch.nn.functional as F
        model.eval()
        correct = loss = 0.0
        with torch.no_grad():
            for s in range(0, len(idx), a.batch_size):
                data = pipe.transform(ds.batch(idx[s:s + a.batch_size]))
                out = model(data)
                correct += out.max(1)[1].eq(data.y).sum().item()
                loss += F.nll_loss(out, data.y, reduction="sum").item()
        model.train()
        return correct / len(idx), loss / len(idx)

    return len(ds), evaluate, hand


def rgin_case(a, dev):
    from bench_counting import build
    from dummynode4graphlearning_b200 import synth
    from dummynode4graphlearning_b200.datasets import ResidentCountingDataset
    from dummynode4graphlearning_b200.optim import FlatAdam
    from dummynode4graphlearning_b200.pipelines import CountingPipeline
    from dummynode4graphlearning_b200.subgraph_isomorphism.losses import eval_criterion
    model, cfg, _ = build("RGIN", "small", dict(rep_rgin_regularizer="bdd", rep_rgin_num_bases=4), dev)
    pipe = CountingPipeline(model, FlatAdam(model.parameters(), lr=1e-3), cfg, add_dummy=True)
    ds = ResidentCountingDataset(synth.counting_samples("small", a.samples, seed=6), dev)
    idx = np.arange(len(ds))
    crit = eval_criterion("MSE")

    def evaluate():
        return pipe.evaluate(ds, idx, batch_size=a.batch_size).metrics()

    def hand():
        model.eval()
        tot = 0.0
        with torch.no_grad():
            for s in range(0, len(idx), a.batch_size):
                sel = idx[s:s + a.batch_size]
                p, g, c = ds.batch(sel)
                out = model(*pipe.transform(p, g))
                tot += crit(out["pred_c"], c.float().view(-1, 1)).item() * len(sel)
        model.train()
        return tot / len(idx)

    return len(ds), evaluate, hand


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--graphs", type=int, default=11130, help="PROTEINS-shaped graphs of the GIN split (10 x 1113)")
    ap.add_argument("--samples", type=int, default=11000, help="'small' counting samples of the RGIN split")
    ap.add_argument("--batch-size", type=int, default=512)
    ap.add_argument("--repeats", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "bench_eval_out"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_eval: needs a CUDA device")
    dev = torch.device("cuda:0")
    res = dict(gpu=gpu_info(), batch_size=a.batch_size, repeats=a.repeats, warmup=a.warmup, statistic="median", cases={})
    for name, case in (("gin_c2_conj", gin_case), ("rgin_small", rgin_case)):
        n, evaluate, hand = case(a, dev)
        t_eval, ts_eval = timed(evaluate, a.repeats, a.warmup)
        t_hand, ts_hand = timed(hand, a.repeats, a.warmup)
        res["cases"][name] = dict(items=n, evaluate_s=t_eval, evaluate_items_per_s=n / t_eval, evaluate_all_s=ts_eval,
                                  hand_loop_s=t_hand, hand_loop_items_per_s=n / t_hand, hand_loop_all_s=ts_hand,
                                  kernels=kernel_times(evaluate), metrics=evaluate())
        print(name, json.dumps({k: v for k, v in res["cases"][name].items() if not k.endswith("all_s")}), flush=True)
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "bench_eval.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(dict(gpu=res["gpu"], out=os.path.join(a.out, "bench_eval.json"))))


if __name__ == "__main__":
    main()
