#!/usr/bin/env python
"""bench_loader.py -- what assembling shuffled mini-batches from a resident data set costs, and what shuffled epochs
train at next to the fixed-batch replay figure.  Everything in one process on one GPU; writes <out>/bench_loader.json
(--out, default ./bench_loader_out) with the card's name and power limit read in the same run.

  assembly        ResidentTUDataset.batch over `--sets` distinct C2-sized index sets (1113 of 11 130 PROTEINS-shaped
                  graphs, with the node attribute): device time per batch (CUDA events), per gather launch (torch.profiler
                  kernel durations), host time of the call, algorithmic bytes
  host_collation  what a user writes today for the same index sets: vectorised numpy collation + conj_sizes hint + pinning
  classification  graphs/s over `--epochs` shuffled epochs of GIN (hidden 32, 4 layers, train_eps) in conj mode:
                  step_indices against host collation + step_async; and the fixed-batch replay of the same pipeline
  counting        the same comparison for RGIN 'small' at batch 512 (host side: io.collate + CountingPipeline.step)
"""
import argparse
import json
import os
import subprocess
import sys
import time
from argparse import Namespace

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.dont_write_bytecode = True

import numpy as np  # noqa: E402
import torch  # noqa: E402


def card():
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        out["power_limit"], out["max_sm_clock"] = [x.strip() for x in q.split(",")[:2]]
    except Exception as e:      # the figures stand without it; say why it is missing
        out["power_limit"] = "not read: %s" % e
    return out


def collate_numpy(raw, idx):
    """vectorised host collation of graphs idx of a raw TU-shaped data set (the layout of synth.tu_batch)."""
    npt, ept = raw["node_ptr"].astype(np.int64), raw["edge_ptr"].astype(np.int64)
    nn_, ne = np.diff(npt)[idx], np.diff(ept)[idx]
    nptr, eptr = np.concatenate([[0], np.cumsum(nn_)]), np.concatenate([[0], np.cumsum(ne)])
    nsel = np.repeat(npt[idx] - nptr[:-1], nn_) + np.arange(nptr[-1])
    esel = np.repeat(ept[idx] - eptr[:-1], ne) + np.arange(eptr[-1])
    shift = np.repeat(nptr[:-1] - npt[idx], ne)
    out = dict(num_graphs=len(idx), node_ptr=nptr.astype(np.int32), edge_ptr=eptr.astype(np.int32),
               src=(raw["src"][esel] + shift).astype(np.int32), dst=(raw["dst"][esel] + shift).astype(np.int32),
               vlabel=raw["vlabel"][nsel], elabel=raw["elabel"][esel], y=raw["y"][idx], has_edge_labels=raw["has_edge_labels"])
    if "vattr" in raw:
        out["vattr"] = raw["vattr"][nsel]
    return out


def batch_bytes(b):
    """algorithmic bytes of one assembled TU batch: every output word read once and written once, plus the staged
    indices / offsets (uploaded, then read by the kernels) and two data-set offsets read per selected graph and level."""
    K = int(b["num_graphs"])
    cols = sum(v.numel() * v.element_size() for k, v in b.items() if isinstance(v, torch.Tensor) and k not in ("node_ptr", "edge_ptr"))
    return 2 * cols + 4 * (4 * K + 3) + 3 * 2 * 4 * K


def assembly(raw, dev, sets, rng):
    from torch.profiler import ProfilerActivity, profile
    from dummynode4graphlearning_b200.datasets import ResidentTUDataset
    ds = ResidentTUDataset(raw, dev)
    idxs = [rng.permutation(len(ds))[:1113] for _ in range(sets)]
    for idx in idxs[:10]:
        ds.batch(idx)
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(sets + 1)]
    host_us, nbytes = [], []
    ev[0].record()
    for i, idx in enumerate(idxs):
        t = time.perf_counter()
        b = ds.batch(idx)
        host_us.append(1e6 * (time.perf_counter() - t))
        ev[i + 1].record()
        nbytes.append(batch_bytes(b))
    torch.cuda.synchronize()
    per_batch = [ev[i].elapsed_time(ev[i + 1]) * 1e3 for i in range(sets)]
    with profile(activities=[ProfilerActivity.CUDA]) as prof:       # kernel durations, separate pass
        for idx in idxs:
            ds.batch(idx)
        torch.cuda.synchronize()
    kern = sorted((e for e in prof.events() if "gather_segments_kernel" in e.name), key=lambda e: e.time_range.start)
    h2d = [e.time_range.elapsed_us() for e in prof.events() if "HtoD" in e.name]
    levels = {}
    for i, e in enumerate(kern):
        levels.setdefault(("nodes", "edges", "graphs")[i % 3], []).append(e.time_range.elapsed_us())
    launch = {k: {"median_us": float(np.median(v)), "mean_us": float(np.mean(v))} for k, v in levels.items()}
    kernel_us = [sum(levels[k][i] for k in levels) for i in range(sets)] if len(kern) == 3 * sets else []
    return {
        "data_set": "synth.tu_batch('proteins', %d, seed=0) with vattr, resident (%d nodes, %d edges); %d distinct index "
                    "sets of 1113 graphs" % (len(ds), int(raw["node_ptr"][-1]), int(raw["edge_ptr"][-1]), sets),
        "per_batch_device_us": {"median": float(np.median(per_batch)), "mean": float(np.mean(per_batch)),
                                "note": "CUDA events between consecutive batch() calls queued back to back: staging copy + "
                                        "3 gathers, and any wait for the host"},
        "per_launch_kernel_us": launch,
        "gather_kernels_per_batch_us": {"median": float(np.median(kernel_us)) if kernel_us else None},
        "staging_copy_us": {"median": float(np.median(h2d)) if h2d else None, "copies": len(h2d)},
        "host_us_per_batch_call": {"median": float(np.median(host_us)), "mean": float(np.mean(host_us))},
        "bytes_per_batch": float(np.mean(nbytes)),
        "gather_GBps_over_kernel_time": float(np.mean(nbytes) / (np.median(kernel_us) * 1e3)) if kernel_us else None,
        "cache": "the resident set (~%.0f MB) fits in the 126 MB L2: warm-cache figures" % (
            (raw["vlabel"].nbytes + raw["vattr"].nbytes + 3 * raw["src"].nbytes) / 1e6),
    }


def host_collation(raw, sets, rng):
    from dummynode4graphlearning_b200 import transforms as T
    from dummynode4graphlearning_b200.pipelines import pin_batch
    t_col, t_hint, t_pin = [], [], []
    for _ in range(sets):
        idx = rng.permutation(int(raw["num_graphs"]))[:1113]
        t0 = time.perf_counter()
        b = collate_numpy(raw, idx)
        t1 = time.perf_counter()
        b["conj_sizes"] = T.tu_conjugate_sizes_ex(b, with_dummy=True)
        t2 = time.perf_counter()
        pin_batch(b)
        t3 = time.perf_counter()
        t_col.append(t1 - t0), t_hint.append(t2 - t1), t_pin.append(t3 - t2)
    ms = lambda v: float(1e3 * np.median(v))      # noqa: E731
    return {"collate_ms": ms(t_col), "hint_ms": ms(t_hint), "pin_ms": ms(t_pin),
            "total_ms": ms(np.add(np.add(t_col, t_hint), t_pin)), "cpu_threads": torch.get_num_threads()}


def _gin_pipe(dev):
    from dummynode4graphlearning_b200.graph_classification.models import GIN
    from dummynode4graphlearning_b200.optim import FlatAdam
    from dummynode4graphlearning_b200.pipelines import ClassificationPipeline
    torch.manual_seed(0)
    args = Namespace(num_features=2, hidden_dim=32, num_classes=2, dropout_ratio=0.0,
                     additional={"train_eps": True, "num_layers": 4, "aggregation": "sum"}, epochs=1, device=str(dev))
    model = GIN(args).to(dev)
    return ClassificationPipeline(model, FlatAdam(model.parameters(), lr=0.01), mode="conj", num_node_labels=2,
                                  node_label_min=0)


def _epochs(sampler, epochs, submit):
    """epoch 0 warms up; epochs 1..`epochs` are timed (host clock to a final synchronise); every loss is read, one step
    late, so that the next step is queued while the previous one runs."""
    out = {}
    for phase, eps in (("warm", [0]), ("timed", range(1, epochs + 1))):
        torch.cuda.synchronize()
        t0, pending, steps, last = time.perf_counter(), None, 0, None
        for e in eps:
            for idx, gb in sampler.batches(e):
                nxt = submit(idx, gb)
                if pending is not None:
                    last = pending.result() if hasattr(pending, "result") else pending
                pending, steps = nxt, steps + 1
        last = pending.result() if hasattr(pending, "result") else pending
        torch.cuda.synchronize()
        out[phase] = (time.perf_counter() - t0, steps, last)
    secs, steps, last = out["timed"]
    return {"graphs_per_s": sampler.num_items * epochs / secs, "ms_per_step": 1e3 * secs / steps, "steps": steps,
            "last_loss": float(last)}


def _fixed(step, dev_batch_size, warm=30, steps=60):
    for _ in range(warm):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    return {"graphs_per_s": dev_batch_size / (ms * 1e-3), "ms_per_step": ms, "steps": steps}


def classification(raw, dev, epochs):
    from dummynode4graphlearning_b200 import transforms as T
    from dummynode4graphlearning_b200.datasets import EpochSampler, ResidentTUDataset
    from dummynode4graphlearning_b200.pipelines import pin_batch
    raw = {k: v for k, v in raw.items() if k != "vattr"}        # GIN on CONJ_ graphs reads labels only (as bench.py)
    ds = ResidentTUDataset(raw, dev)
    sampler = EpochSampler(len(ds), 1113, seed=0)
    pipe = _gin_pipe(dev)
    res = {"resident_step_indices": _epochs(sampler, epochs, lambda idx, gb: pipe.step_indices(ds, idx))}

    def host_step(idx, gb):
        b = collate_numpy(raw, idx)
        b["conj_sizes"] = T.tu_conjugate_sizes_ex(b, with_dummy=True)
        return pipe_h.step_async(pin_batch(b))
    pipe_h = _gin_pipe(dev)
    res["host_collation_step_async"] = _epochs(sampler, epochs, host_step)
    pipe_f = _gin_pipe(dev)
    fixed = ds.batch(np.arange(1113))
    torch.cuda.synchronize()
    res["fixed_batch_replay"] = _fixed(lambda: pipe_f.step_resident(fixed, assume_ready=True), 1113)
    res["fixed_batch_replay"]["how"] = "step_resident on one resident batch of 1113 graphs, replayed CUDA graphs, no L2 flush"
    res["shuffled_over_fixed"] = res["resident_step_indices"]["graphs_per_s"] / res["fixed_batch_replay"]["graphs_per_s"]
    res["workload"] = ("GIN hidden 32, 4 layers, train_eps, conj mode with the size hint, FlatAdam lr 0.01; %d graphs, batch "
                       "1113, %d timed epochs after one warm-up epoch" % (len(ds), epochs))
    return res


def counting(dev, n_samples, bs, epochs):
    from bench_counting import build
    from dummynode4graphlearning_b200 import synth
    from dummynode4graphlearning_b200.datasets import EpochSampler, ResidentCountingDataset
    from dummynode4graphlearning_b200.optim import FlatAdam
    from dummynode4graphlearning_b200.pipelines import CountingPipeline, pin_batch
    from dummynode4graphlearning_b200.subgraph_isomorphism import io as sio
    samples = synth.counting_samples("small", n_samples, seed=0)
    ds = ResidentCountingDataset(samples, dev)
    sampler = EpochSampler(len(ds), bs, seed=0)

    def make():
        model, cfg, _ = build("RGIN", "small", dict(rep_rgin_regularizer="bdd", rep_rgin_num_bases=4), dev)
        opt = FlatAdam(model.parameters(), lr=1e-3, weight_decay=1e-2, amsgrad=True, decoupled_weight_decay=True)
        return CountingPipeline(model, opt, cfg, add_dummy=True, rep_reg_w=1e-3)
    pipe = make()
    res = {"resident_step_indices": _epochs(sampler, epochs, lambda idx, gb: pipe.step_indices(ds, idx))}
    pipe_h = make()

    def host_step(idx, gb):
        p, g, c, _ = sio.collate([samples[j] for j in idx])
        return pipe_h.step(pin_batch(p), pin_batch(g), torch.from_numpy(c))       # blocking: returns the float
    res["host_collate_step"] = _epochs(sampler, epochs, host_step)
    pipe_f = make()
    p, g, c = ds.batch(np.arange(bs))
    torch.cuda.synchronize()
    res["fixed_batch_replay"] = _fixed(lambda: pipe_f.step_resident(p, g, c, assume_ready=True), bs)
    res["shuffled_over_fixed"] = res["resident_step_indices"]["graphs_per_s"] / res["fixed_batch_replay"]["graphs_per_s"]
    res["workload"] = ("RGIN 'small' (bdd, 4 bases, hid 64, 3 layers) + dummy, synth.counting_samples('small', %d), batch %d, "
                       "%d timed epochs after one warm-up epoch; the host arm uses io.collate and the blocking "
                       "CountingPipeline.step, the only host-batch entry point of the counting pipeline" % (n_samples, bs, epochs))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="bench_loader_out", help="directory for bench_loader.json")
    ap.add_argument("--graphs", type=int, default=11130)
    ap.add_argument("--sets", type=int, default=200)
    ap.add_argument("--epochs", type=int, default=3)
    ap.add_argument("--counting-samples", type=int, default=5120)
    ap.add_argument("--counting-batch", type=int, default=512)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_loader.py: no CUDA device (the figures are GPU measurements)")
    from dummynode4graphlearning_b200 import synth
    dev = torch.device("cuda:0")
    rng = np.random.default_rng(0)
    raw = synth.tu_batch("proteins", a.graphs, seed=0)
    res = {"card": card()}
    res["assembly"] = assembly(raw, dev, a.sets, rng)
    res["host_collation"] = host_collation(raw, a.sets, rng)
    res["classification"] = classification(raw, dev, a.epochs)
    res["counting"] = counting(dev, a.counting_samples, a.counting_batch, a.epochs)
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "bench_loader.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
