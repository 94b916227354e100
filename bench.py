#!/usr/bin/env python
"""bench.py -- train graphs/s of the hot path on BASELINE.json's config C2, plus the aggregation roofline.

  python bench.py --gpus N --steps K --warmup W            our arm (libdn4gl.so kernels; one process per GPU)
  python bench.py --impl reference --steps K --warmup W    the reference's CPU path (oracle port) on host cores

Workload "c2": 1113 synthetic PROTEINS-shaped graphs per GPU (seeded), one STEP = dummy-node augmentation +
edge-to-vertex (CONJ) transform + PyG canonicalisation + CSR build + GIN (hidden 32, 4 layers, train_eps,
sum pooling -- hyper_params.py:15) forward + nll_loss + backward [+ gradient all-reduce] + Adam step.
`value`   : inputs (raw graphs) resident in HBM, L2 flushed between steps, device-timed, max over ranks.
`e2e`     : same step through ClassificationPipeline.step(): pinned host buffers -> H2D -> ... -> loss D2H.
`roofline`: the aggregation kernel (dn4gl_spmm_sum_f32 at D=32), algorithmic bytes / CUDA-event duration.
Prints ONE JSON line on rank 0.  `--dump-outputs DIR` also writes what the last timed step handed back (loss, updated
parameters, their gradients, BatchNorm statistics) as DIR/<name>.npy, so that two builds can be compared output for output.
"""
import argparse
import atexit
import json
import os
import statistics
import subprocess
import sys
import time
from argparse import Namespace

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True    # leave the source tree as it is (it may be read-only)

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

HID, LAYERS, CLASSES, LR = 32, 4, 2, 0.01   # hyper_params.py:15 (GIN / PROTEINS)
NUM_NODE_LABELS = 2                          # CONJ graphs: vertex label = original edge label (1) or dummy (0)
L2_FLUSH_BYTES = 192 << 20     # > the 126 MB L2


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--graphs", type=int, default=1113, help="graphs per GPU (C2: 1113)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="only the C2 line (skip the C1 / C3 / C4 / C5 measurements)")
    ap.add_argument("--no-size-hints", dest="size_hints", action="store_false",
                    help="let the transform read its output sizes back from the device (one device->host sync per step) "
                         "instead of taking transforms.tu_conjugate_sizes(raw) from the host batch")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (float32)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs:
        os.makedirs(a.dump_outputs, exist_ok=True)
    return a


def dump_outputs(out_dir, loss, model):
    """what a caller of the timed step holds after it: the returned loss and the model the step updated in place -- every
    parameter, the gradient this step computed for it, the BatchNorm running statistics.  Inputs and initial weights
    are seeded, so the same arguments give the same arrays up to floating-point reordering."""
    arrays = {"loss": loss}
    for n, p in model.named_parameters():
        arrays["param." + n] = p
        if p.grad is not None:
            arrays["grad." + n] = p.grad
    for n, b in model.named_buffers():
        if b.is_floating_point():
            arrays["buffer." + n] = b
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), v.detach().float().cpu().numpy())


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback"


# ---------------------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference path (C transforms + torch-CPU GIN), all host threads
def split_tu_batch(raw, parts):
    """contiguous chunks of whole graphs, balanced by edge count (graphs are independent: block-diagonal batch)."""
    B = int(raw["num_graphs"])
    parts = max(1, min(parts, B))
    ep, npz = raw["edge_ptr"].astype(np.int64), raw["node_ptr"].astype(np.int64)
    cuts = [0] + [int(np.searchsorted(ep, ep[-1] * k / parts)) for k in range(1, parts)] + [B]
    cuts = sorted(set(min(max(c, 0), B) for c in cuts))
    out = []
    for g0, g1 in zip(cuts[:-1], cuts[1:]):
        n0, n1, e0, e1 = int(npz[g0]), int(npz[g1]), int(ep[g0]), int(ep[g1])
        c = dict(num_graphs=g1 - g0, node_ptr=(npz[g0:g1 + 1] - n0).astype(np.int32),
                 edge_ptr=(ep[g0:g1 + 1] - e0).astype(np.int32),
                 src=(raw["src"][e0:e1] - n0).astype(np.int32), dst=(raw["dst"][e0:e1] - n0).astype(np.int32),
                 vlabel=raw["vlabel"][n0:n1], elabel=raw["elabel"][e0:e1])
        if "vattr" in raw:
            c["vattr"] = raw["vattr"][n0:n1]
        if "y" in raw:
            c["y"] = raw["y"][g0:g1]
        out.append(c)
    return out


def cpu_transform(raw, pool, threads):
    """dummy augmentation + CONJ transform + PyG canonicalisation on the host, graphs sharded over `threads` host threads
    (the C restatement releases the GIL).  Chunk results concatenate to exactly the single-thread result because the
    batch is block-diagonal and the canonical (row, col) order is chunk-major.  -> (vlabel, src, dst, nodes per graph)"""
    from oracle import transforms as OT

    def one(c):
        conj = OT.tu_conjugate(OT.tu_add_dummy(c))
        s, d, _, _ = OT.pyg_coalesce(conj["src"], conj["dst"])
        return conj["vlabel"], s, d, np.diff(conj["node_ptr"])

    chunks = split_tu_batch(raw, threads)
    res = list(pool.map(one, chunks)) if pool is not None and len(chunks) > 1 else [one(c) for c in chunks]
    off = np.cumsum([0] + [int(r[3].sum()) for r in res])
    return (np.concatenate([r[0] for r in res]), np.concatenate([r[1] + off[i] for i, r in enumerate(res)]),
            np.concatenate([r[2] + off[i] for i, r in enumerate(res)]), np.concatenate([r[3] for r in res]))


def cpu_transform_dummy(raw, pool, threads):
    """C1: dummy augmentation + PyG canonicalisation on the host (same sharding as cpu_transform)."""
    from oracle import transforms as OT

    def one(c):
        d = OT.tu_add_dummy(c)
        s, dd, _, _ = OT.pyg_coalesce(d["src"], d["dst"])
        return d["vlabel"], s, dd, np.diff(d["node_ptr"])

    chunks = split_tu_batch(raw, threads)
    res = list(pool.map(one, chunks)) if pool is not None and len(chunks) > 1 else [one(c) for c in chunks]
    off = np.cumsum([0] + [int(r[3].sum()) for r in res])
    return (np.concatenate([r[0] for r in res]), np.concatenate([r[1] + off[i] for i, r in enumerate(res)]),
            np.concatenate([r[2] + off[i] for i, r in enumerate(res)]), np.concatenate([r[3] for r in res]))


def cpu_reference_run(raw, steps, warmup, mode="conj", hid=HID, layers=LAYERS, num_labels=NUM_NODE_LABELS):
    from concurrent.futures import ThreadPoolExecutor

    from oracle import models as OM

    torch.set_num_threads(os.cpu_count() or 1)
    from dummynode4graphlearning_b200.graph_classification.models import GIN
    torch.manual_seed(0)
    args = Namespace(num_features=num_labels, hidden_dim=hid, num_classes=CLASSES, dropout_ratio=0.0,
                     additional={"train_eps": True, "num_layers": layers, "aggregation": "sum"}, epochs=1, device="cpu")
    sd = {k: v.clone().requires_grad_(v.is_floating_point() and "running" not in k and "num_batches" not in k)
          for k, v in GIN(args).state_dict().items()}
    params = []
    for k, v in sd.items():   # nns.* / convs.*.nn.* alias: optimise each tensor once
        if v.requires_grad and not (k.startswith("convs.") and ".nn." in k):
            params.append(v)
    opt = torch.optim.Adam(params, lr=LR)
    y = torch.from_numpy(raw["y"])
    B = raw["num_graphs"]
    t_tr, t_md = [], []
    threads = os.cpu_count() or 1
    pool = ThreadPoolExecutor(threads) if threads > 1 else None
    tf = cpu_transform if mode == "conj" else cpu_transform_dummy
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        vlabel, s, d, nodes_per_graph = tf(raw, pool, threads)
        x = torch.from_numpy(np.eye(num_labels, dtype=np.float32)[vlabel])
        ei = torch.from_numpy(np.stack([s, d]).astype(np.int64))
        batch = torch.from_numpy(np.repeat(np.arange(B), nodes_per_graph).astype(np.int64))
        t1 = time.perf_counter()
        opt.zero_grad()
        out = OM.gin_classifier(sd, x, ei, batch, B, layers, "sum")
        loss = F.nll_loss(out, y)
        loss.backward()
        opt.step()
        t2 = time.perf_counter()
        if it >= warmup:
            t_tr.append(t1 - t0)
            t_md.append(t2 - t1)
    total = sum(t_tr) + sum(t_md)
    return dict(graphs_per_s=B * steps / total, ms_per_step=1e3 * total / steps,
                transform_ms=1e3 * statistics.mean(t_tr), train_ms=1e3 * statistics.mean(t_md),
                cores=torch.get_num_threads())


# ---------------------------------------------------------------------------------------------------------
# the other BASELINE.json configurations (C1, C3, C4): same metric (train graphs/s, full step), own CPU leg
COUNTING = {"c3": ("RGIN", "small", 512, dict(rep_rgin_regularizer="bdd", rep_rgin_num_bases=4)),
            "c4": ("DMPNN", "large", 64, dict(node_pred=True, edge_pred=False))}


def counting_kwargs(shape, over):
    from dummynode4graphlearning_b200 import synth, transforms as T
    cfg = dict(synth.counting_config(shape), add_dummy=True)
    mc = T.process_model_config(cfg)
    kw = dict({k: v for k, v in mc.items() if k.startswith("max_")}, hid_dim=64, rep_num_graph_layers=3,
              rep_num_pattern_layers=3, rep_act_func="relu", pred_act_func="relu", pred_net="SumPredictNet",
              pred_hid_dim=64, emb_net="Equivariant", enc_net="Multihot", filter_net="ScalarFilter", pred_with_enc=True,
              pred_with_deg=True, init_neigenv=4.0, init_eeigenv=4.0)
    kw.update(over)
    return cfg, kw


def build_counting_model(name, kw, device):
    from dummynode4graphlearning_b200.subgraph_isomorphism.models import DMPNN, RGIN
    torch.manual_seed(0)
    model = {"RGIN": RGIN, "DMPNN": DMPNN}[name](**kw)
    with torch.no_grad():      # pred_fc2 / weight_fc2 are zero-initialised in the reference (pred.py:50,53): outputs would be 0
        for n, q in model.named_parameters():
            if "pred_fc2" in n or "weight_fc2" in n:
                q.normal_(0.0, 0.1)
    return model.to(device)


def gpu_counting_run(key, dev, world, rank, steps, warmup=20):
    """C3 / C4: augmentation (dummy) + CSR builds + model forward + loss + backward (+ all-reduce) + clip + AdamW(amsgrad)
    per step, inputs resident in HBM, device-timed, max over ranks."""
    from dummynode4graphlearning_b200 import synth, transforms as T
    from dummynode4graphlearning_b200.optim import FlatAdam
    from dummynode4graphlearning_b200.parallel import max_over_ranks
    from dummynode4graphlearning_b200.pipelines import CountingPipeline
    name, shape, bs, over = COUNTING[key]
    cfg, kw = counting_kwargs(shape, over)
    model = build_counting_model(name, kw, dev)
    opt = FlatAdam(model.parameters(), lr=1e-3, weight_decay=1e-2, amsgrad=True, decoupled_weight_decay=True)   # train.py:1408-1411
    pipe = CountingPipeline(model, opt, cfg, add_dummy=True, rep_reg_w=1e-3)
    pipe.global_batch = bs * world
    p, g, counts = synth.counting_batch(shape, bs, seed=rank)
    pd_, gd_ = T.to_device(p, dev), T.to_device(g, dev)
    cd = torch.from_numpy(counts).to(dev)
    for _ in range(warmup):
        loss = pipe.step_resident(pd_, gd_, cd, assume_ready=True)
    if world > 1:
        torch.distributed.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    nmalloc = lambda: int(torch.cuda.memory_stats(dev).get("num_device_alloc", 0))
    m0, t_host = nmalloc(), time.perf_counter()
    e0.record()
    for _ in range(steps):
        loss = pipe.step_resident(pd_, gd_, cd, assume_ready=True)
    e1.record()
    host_ms = 1e3 * (time.perf_counter() - t_host) / steps      # time to SUBMIT a step (the loop throttles on the device)
    if world > 1:
        torch.distributed.barrier()
    torch.cuda.synchronize()
    ms = max_over_ranks(e0.elapsed_time(e1), dev) / steps
    out = {"workload": "%s: %s + dummy, synthetic '%s' shape, batch %d per GPU, hid 64, 3 layers, SumPredictNet; augmentation + "
                       "CSR builds + forward + loss + backward + clip + AdamW(amsgrad) per step" % (key, name, shape, bs),
           "metric": "train graphs/sec", "value": bs * world / (ms * 1e-3), "unit": "graphs/s", "ms_per_step": ms, "steps": steps,
           "n_gpus": world, "graphs_per_gpu": bs, "graph_nodes": int(g["node_ptr"][-1]), "graph_edges": int(g["edge_ptr"][-1]),
           "loss": float(loss.item()), "host_submit_ms_per_step": host_ms, "cudaMalloc_calls_in_timed_region": nmalloc() - m0}
    pipe._graphs.clear()
    return out, (p, g, counts, cfg, kw, name)


def cpu_counting_run(p, g, counts, cfg, kw, name, steps=2, warmup=1):
    """CPU leg of C3 / C4: oracle port (C augmentation + torch-CPU restatement of the reference's per-edge formulation)."""
    from oracle import models as OM, transforms as OT
    torch.set_num_threads(os.cpu_count() or 1)
    model = build_counting_model(name, kw, "cpu")
    sd = {k: v.clone().requires_grad_(v.is_floating_point() and "enc_net" not in k) for k, v in model.state_dict().items()}
    params = [v for k, v in sd.items() if v.requires_grad and not k.startswith("p_")]
    opt = torch.optim.AdamW(params, lr=1e-3, weight_decay=1e-2, amsgrad=True)
    ocfg = OM.counting_cfg_from_kwargs(name, kw)
    ts = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        pa = OT.sub_add_dummy(p, cfg["max_npv"], cfg["max_npvl"], cfg["max_npe"], cfg["max_npel"])
        ga = OT.sub_add_dummy(g, cfg["max_ngv"], cfg["max_ngvl"], cfg["max_nge"], cfg["max_ngel"])
        opt.zero_grad()
        out = OM.counting_model(sd, pa, ga, ocfg)
        loss = OM.counting_loss(out, torch.from_numpy(counts), rep_reg_w=1e-3)
        loss.backward()
        torch.nn.utils.clip_grad_norm_(params, 8.0)
        opt.step()
        if it >= warmup:
            ts.append(time.perf_counter() - t0)
    B = len(counts)
    return {"value": B / statistics.mean(ts), "unit": "graphs/s", "cores": torch.get_num_threads(), "kind": "port",
            "ms_per_step": 1e3 * statistics.mean(ts),
            "sample": "full batch (%d samples), %d timed steps after %d warm-up: oracle/c augmentation + oracle/models.py "
                      "(the reference's per-edge formulation on torch-CPU) + AdamW(amsgrad)" % (B, steps, warmup)}


def gpu_classification_run(shape, graphs, mode, hid, layers, num_labels, dev, steps, warmup=30):
    """C1-style classification step through ClassificationPipeline (inputs resident in HBM, device-timed)."""
    from dummynode4graphlearning_b200 import synth, transforms as T
    from dummynode4graphlearning_b200.graph_classification.models import GIN
    from dummynode4graphlearning_b200.optim import FlatAdam
    from dummynode4graphlearning_b200.pipelines import ClassificationPipeline
    raw = synth.tu_batch(shape, graphs, seed=0)
    dev_batch = T.to_device({k: v for k, v in raw.items() if k != "vattr"}, dev)
    torch.manual_seed(0)
    args = Namespace(num_features=num_labels, hidden_dim=hid, num_classes=CLASSES, dropout_ratio=0.0,
                     additional={"train_eps": True, "num_layers": layers, "aggregation": "sum"}, epochs=1, device=str(dev))
    model = GIN(args).to(dev)
    pipe = ClassificationPipeline(model, FlatAdam(model.parameters(), lr=LR), mode=mode, num_node_labels=num_labels, node_label_min=0)
    for _ in range(warmup):
        pipe.step_resident(dev_batch, assume_ready=True)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    nmalloc = lambda: int(torch.cuda.memory_stats(dev).get("num_device_alloc", 0))
    m0, t_host = nmalloc(), time.perf_counter()
    e0.record()
    for _ in range(steps):
        loss = pipe.step_resident(dev_batch, assume_ready=True)
    e1.record()
    host_ms = 1e3 * (time.perf_counter() - t_host) / steps
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    pipe._graphs.clear()
    return {"metric": "train graphs/sec", "value": graphs / (ms * 1e-3), "unit": "graphs/s", "ms_per_step": ms, "steps": steps,
            "loss": float(loss.item()), "host_submit_ms_per_step": host_ms, "cudaMalloc_calls_in_timed_region": nmalloc() - m0}, raw


def reference_arm(a):
    """rank 0 only: times the reference's CPU implementation (oracle port) on the host cores."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    from dummynode4graphlearning_b200 import synth
    raw = synth.tu_batch("proteins", a.graphs, seed=0)
    r = cpu_reference_run(raw, a.steps, max(a.warmup, 1))
    line = {
        "impl": "reference", "metric": "train graphs/sec", "value": r["graphs_per_s"], "unit": "graphs/s",
        "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": r["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(a.graphs, 1),
        "cpu_baseline": {"value": r["graphs_per_s"], "unit": "graphs/s", "cores": r["cores"], "kind": "port",
                         "sample": "full C2 batch (%d graphs) per step, %d steps; C restatement of the transforms "
                                   "(oracle/c), graphs sharded over all host threads, + torch-CPU restatement of GIN "
                                   "fwd/bwd + Adam (oracle/models.py)" % (a.graphs, a.steps),
                         "transform_ms": r["transform_ms"], "train_ms": r["train_ms"]},
        "e2e": {"value": r["graphs_per_s"], "unit": "graphs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def workload_config(graphs, n_gpus):
    return {"workload": "c2: dummy + edge-to-vertex (CONJ) transform + GIN(hidden 32, 4 layers, train_eps, sum pool) "
                        "train step on synthetic PROTEINS-shaped graphs", "graphs_per_gpu": graphs,
            "global_batch": graphs * n_gpus, "avg_nodes": 39, "optimizer": "Adam(lr=0.01) as one flat-buffer kernel (dn4gl_adam_f32)", "train_step": "CUDA graph replay per batch signature; transform eager on a second stream, overlapping the previous train step",
            "parallelism": "dp%d" % n_gpus, "l2": "flushed between steps (192 MiB write, larger than the 126 MB L2, inside the timed region)"}


# ---------------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock / throttle reasons DURING the timed regions (B200_PROFILING.md clocks line).

    A separate `nvidia-smi -lms 50` process is started before the warm-up (its start-up takes a few hundred ms) and
    its time-stamped rows are filtered to the window between mark_start() and stop().  In-process NVML sampling from a
    thread was tried first: its queries take the driver's lock and stalled single steps of this (host-bound, 1.2 ms)
    loop for 5-130 ms in one run out of four (profiles/README.md, r1f/r1g); the loop without a sampler shows no step
    above 3.1 ms in 4000 (tools/e2e_stall.py).  Falls back to one NVML sample at the end if nvidia-smi is missing."""

    Q = ("timestamp,clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.p, self.t0 = index, None, None
        self.path = "/tmp/dn4gl_clocks_%d_%d.csv" % (os.getpid(), index)
        try:
            uuid = str(torch.cuda.get_device_properties(index).uuid)
            sel = uuid if uuid.startswith("GPU-") else "GPU-" + uuid
        except Exception:   # noqa: BLE001
            sel = str(index)
        try:
            self.f = open(self.path, "w")
            self.p = subprocess.Popen(["nvidia-smi", "-i", sel, "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                       "-lms", "50"], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:   # noqa: BLE001
            self.p = None
        atexit.register(self._kill)      # an exception before stop() must not leave the sampler running

    def _kill(self):
        if self.p is not None and self.p.poll() is None:
            self.p.kill()

    def mark_start(self):
        self.t0 = time.time()

    def _nvml_once(self):
        import pynvml as nv
        nv.nvmlInit()
        h = nv.nvmlDeviceGetHandleByIndex(self.index)
        return {"sm_mhz": float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)),
                "sm_max_mhz": float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)), "samples": 1, "reasons": [],
                "how": "one NVML sample right after the timed regions (nvidia-smi unavailable)"}

    def stop(self):
        import datetime
        t1 = time.time()
        if self.p is None:
            try:
                return self._nvml_once()
            except Exception as e:   # noqa: BLE001
                return {"sm_mhz": None, "sm_max_mhz": None, "samples": 0, "reasons": [], "error": str(e)[:100]}
        time.sleep(0.06)              # let the row that covers the end of the window arrive
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:   # noqa: BLE001
            self.p.kill()
        self.f.close()
        sm, mx, reasons, total = [], [], set(), 0
        for ln in open(self.path):
            c = [x.strip() for x in ln.split(",")]
            if len(c) < 7:
                continue
            total += 1
            try:
                ts = datetime.datetime.strptime(c[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                clk, cmax = float(c[1]), float(c[2])
            except ValueError:
                continue
            if self.t0 is not None and not (self.t0 - 0.05 <= ts <= t1 + 0.05):
                continue
            sm.append(clk); mx.append(cmax)
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        try:
            os.unlink(self.path)
        except OSError:
            pass
        out = {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "samples": len(sm),
               "reasons": sorted(reasons), "how": "nvidia-smi -lms 50 in a separate process, rows inside the timed window",
               "rows_total": total}
        if not sm:
            try:
                out.update(self._nvml_once())
            except Exception:   # noqa: BLE001
                pass
        return out


class EntryPointTimer:
    """CUDA-event pair around every C-ABI call (on the launching stream): per-entry-point device time."""

    def __init__(self):
        self.pending, self.stack = [], []

    def before(self, name, args):
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        self.stack.append(e)

    def after(self, name, args):
        e1 = torch.cuda.Event(enable_timing=True)
        e1.record()
        key = name
        if name in ("dn4gl_spmm_sum_f32", "dn4gl_spmm_tiled_f32"):
            key = "%s[D=%d]" % (name, args[6] if name == "dn4gl_spmm_sum_f32" else args[5])
        self.pending.append((key, self.stack.pop(), e1))

    def summary(self):
        torch.cuda.synchronize()
        agg = {}
        for key, e0, e1 in self.pending:
            agg.setdefault(key, []).append(e0.elapsed_time(e1))
        return {k: {"calls": len(v), "total_ms": sum(v), "avg_us": 1e3 * sum(v) / len(v)} for k, v in agg.items()}


def ours(a):
    import torch.distributed as dist
    from dummynode4graphlearning_b200 import _lib, synth, transforms as T
    from dummynode4graphlearning_b200.graph_classification.models import GIN
    from dummynode4graphlearning_b200.parallel import max_over_ranks
    from dummynode4graphlearning_b200.pipelines import ClassificationPipeline, host_bytes, pin_batch

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the hot path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    L = _lib.lib()

    raw = synth.tu_batch("proteins", a.graphs, seed=rank)      # weak scaling: every rank owns its own 1113 graphs
    host = pin_batch({k: v for k, v in raw.items() if k != "vattr"})
    dev_batch = T.to_device({k: v for k, v in raw.items() if k != "vattr"}, dev)
    if a.size_hints:      # what a loader that sees its batch on the host would attach (computed once here: the batch is fixed)
        host["conj_sizes"] = dev_batch["conj_sizes"] = T.tu_conjugate_sizes_ex(raw, with_dummy=True)
    torch.manual_seed(0)
    args = Namespace(num_features=NUM_NODE_LABELS, hidden_dim=HID, num_classes=CLASSES, dropout_ratio=0.0,
                     additional={"train_eps": True, "num_layers": LAYERS, "aggregation": "sum"}, epochs=1, device=str(dev))
    model = GIN(args).to(dev)
    from dummynode4graphlearning_b200.optim import FlatAdam
    opt = FlatAdam(model.parameters(), lr=LR)   # torch.optim.Adam's update rule as ONE kernel over flat buffers (capturable)
    pipe = ClassificationPipeline(model, opt, mode="conj", num_node_labels=NUM_NODE_LABELS, node_label_min=0)
    pipe.global_batch = a.graphs * world
    flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    clocks = ClockSampler(local) if (rank == 0 and not os.environ.get("DN4GL_NO_CLOCKS")) else None
    n_warm = max(a.warmup, 30)   # first step eager, second captures the CUDA graph, the rest settle the caching allocator
                                 # (two streams, up to two steps in flight: a cudaMalloc inside the timed loop costs 2-10 ms)
    for _ in range(n_warm):
        flush.fill_(1)
        pipe.step_resident(dev_batch, assume_ready=True)   # the raw batch has been resident since before the warm-up
    # long-lived objects (modules, captured graphs, static buffers) leave the cyclic collector's working set: a
    # generation-2 pass over them inside the timed loop showed up as 2-10 ms host stalls (steps are host-bound)
    import gc
    gc.collect()
    gc.freeze()
    # ---- timed region: EXACTLY K steps, device-timed ----------------------------------------------------
    barrier()
    if clocks:
        clocks.mark_start()
    k0 = L.kernel_launches() + pipe.replayed_library_kernels()
    nmalloc = lambda: int(torch.cuda.memory_stats(dev).get("num_device_alloc", 0))   # cudaMalloc calls so far
    m0 = nmalloc()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    trace = [] if os.environ.get("DN4GL_BENCH_TRACE") else None
    for _ in range(a.steps):
        flush.fill_(1)
        loss = pipe.step_resident(dev_batch, assume_ready=True)
        if trace is not None:
            trace.append(time.perf_counter())
    e1.record()
    barrier()
    launches = L.kernel_launches() + pipe.replayed_library_kernels() - k0
    final_loss = float(loss.item())      # read NOW: `loss` is the captured step's static buffer, later steps overwrite it
    m1 = nmalloc()
    ms = max_over_ranks(e0.elapsed_time(e1), dev) / a.steps
    if a.dump_outputs and rank == 0:      # before the loops below step the model again
        dump_outputs(a.dump_outputs, loss, model)
    # what the in-loop L2 flush costs: the same K steps without it, and K flushes alone (informational -- `value` and
    # `ms_per_step` above are the flushed loop, flush included)
    ex0, ex1, ex2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
    barrier()
    ex0.record()
    for _ in range(a.steps):
        pipe.step_resident(dev_batch, assume_ready=True)
    ex1.record()
    for _ in range(a.steps):
        flush.fill_(1)
    ex2.record()
    barrier()
    l2_flush = {"flush_alone_ms_per_step": ex1.elapsed_time(ex2) / a.steps,
                "ms_per_step_without_flush": max_over_ranks(ex0.elapsed_time(ex1), dev) / a.steps,
                "note": "ms_per_step / value are measured WITH the 192 MiB flush write inside the timed loop on the train "
                        "stream; these two figures say how much of the step it is"}
    value = a.graphs * world / (ms * 1e-3)
    if trace:
        print("host ms per step:", " ".join("%.2f" % (1e3 * (b - a_)) for a_, b in zip(trace[:-1], trace[1:])), file=sys.stderr)

    # ---- e2e: host buffers through the public API, copies inside the timed region --------------------------
    pending = None
    for _ in range(15):               # warm-up in the same software-pipelined pattern as the timed loop (two steps in flight)
        nxt = pipe.step_async(host)
        if pending is not None:
            pending.result()
        pending = nxt
    pending.result()
    barrier()
    t0 = time.perf_counter()
    pending = None
    etrace = [] if trace is not None else None
    for _ in range(a.steps):          # software-pipelined: submit step k (H2D, transform, train, D2H of its loss),
        flush.fill_(1)                # then read the loss of step k-1 on the host -- every loss is read, in order
        ta = time.perf_counter()
        nxt = pipe.step_async(host)
        tb = time.perf_counter()
        if pending is not None:
            last = pending.result()
        pending = nxt
        if etrace is not None:
            etrace.append((tb - ta, time.perf_counter() - tb))
    last = pending.result()
    torch.cuda.synchronize()
    t_end = time.perf_counter()
    clk = clocks.stop() if clocks else None      # sampled over both timed regions (+ one sample right at their end)
    e2e_ms = max_over_ranks((t_end - t0) * 1e3, dev) / a.steps
    e2e_value = a.graphs * world / (e2e_ms * 1e-3)
    m2 = nmalloc()
    if etrace:
        print("e2e submit ms:", " ".join("%.2f" % (1e3 * x) for x, _ in etrace), file=sys.stderr)
        print("e2e result ms:", " ".join("%.2f" % (1e3 * y) for _, y in etrace), file=sys.stderr)

    # ---- the transform alone as the pipeline runs it (captured CUDA graph when the loader's size hint is present) ------
    transform_replay = None
    try:
        y0, y1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(3):
            pipe.transform(dev_batch)
        torch.cuda.synchronize()
        th0 = time.perf_counter()
        y0.record()
        for _ in range(20):
            pipe.transform(dev_batch)
        y1.record()
        th1 = time.perf_counter()
        torch.cuda.synchronize()
        transform_replay = {"ms": y0.elapsed_time(y1) / 20, "host_ms": 1e3 * (th1 - th0) / 20,
                            "captured": any(not isinstance(e, str) for e in pipe._tgraphs.values()),
                            "how": "20 pipeline transforms back to back on one stream, no train step in between"}
    except Exception as ex:   # noqa: BLE001
        transform_replay = {"error": str(ex)[:200]}
    # ---- per-entry-point device times + breakdown (instrumented pass, not part of `value`) -----------------
    timer = EntryPointTimer()
    pipe.cuda_graphs = False      # the instrumented pass brackets every C-ABI call with events: eager launches
    pipe.overlap = False          # ... on one stream
    L.profiler = timer
    tr0, tr1, tn1 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
    tr_ms, tn_ms = [], []
    data = None
    for _ in range(min(a.steps, 10)):
        flush.fill_(1)
        tr0.record()
        data = pipe.transform(dev_batch)
        tr1.record()
        pipe.train_on(data)
        tn1.record()
        torch.cuda.synchronize()
        tr_ms.append(tr0.elapsed_time(tr1)); tn_ms.append(tr1.elapsed_time(tn1))
    L.profiler = None
    per_entry = timer.summary()
    # ---- the transform alone (SURVEY.md 8(d): edges/s and GB/s of the builder kernels), eager on one stream ---------
    transform_only = None
    try:
        x0, x1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(3):
            pipe.transform(dev_batch)
        torch.cuda.synchronize()
        x0.record()
        for _ in range(20):
            d_ = pipe.transform(dev_batch)
        x1.record()
        torch.cuda.synchronize()
        t_ms = x0.elapsed_time(x1) / 20
        v_raw, e_raw = int(raw["vlabel"].shape[0]), int(raw["src"].shape[0])
        v_out, e_out = int(d_.structure.num_nodes), int(d_.structure.csr_in.nnz)
        tbytes = 4 * (2 * e_raw + v_raw) + 4 * (2 * e_out + v_out) + 4 * v_out      # in: COO + labels; out: COO + labels
        transform_only = {"ms": t_ms, "raw_edges": e_raw, "conj_edges": e_out, "conj_edges_per_s": e_out / (t_ms * 1e-3),
                          "algorithmic_bytes": tbytes, "gbs": tbytes / (t_ms * 1e-3) / 1e9,
                          "how": "dummy + CONJ + canonicalisation + both CSRs + tilings, 20 eager calls on one stream "
                                 "(host-paced: ~60 small launches and one size read-back per call)"}
    except Exception as ex:   # noqa: BLE001 -- an auxiliary figure must never cost the bench line
        transform_only = {"error": str(ex)[:200]}
    # ---- device duration of the dominant kernel (K1, sum aggregation) ---------------------------------------------
    from dummynode4graphlearning_b200 import ops
    s = data.structure
    N, E = s.num_nodes, int(s.csr_in.nnz)
    peaks, which = measured_peaks()

    def _graph_b2b(fn, nbuf, launches):
        """average device time of one launch: `launches` launches captured in ONE CUDA graph (launch i works on buffer
        i % nbuf), the graph replayed between two events.  The Python -> ctypes call costs 10-15 us per launch, more than
        these kernels take at the small sizes: issued eagerly the loop measured the host, not the kernel."""
        for i in range(min(nbuf, 4)):
            fn(i)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for i in range(launches):
                fn(i % nbuf)
        g.replay()                       # warm
        torch.cuda.synchronize()
        b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        b0.record()
        g.replay()
        b1.record()
        torch.cuda.synchronize()
        return 1e3 * b0.elapsed_time(b1) / launches      # us

    def k1_back_to_back(csr_in, csr_out, n_rows, D, launches=64):
        """`launches` aggregation launches back to back (one CUDA-graph replay between two events on the launching stream),
        each reading a different feature matrix and writing a different output out of a pool larger than L2 (>= 320 MB),
        so every launch finds its operands in HBM, not in L2."""
        per = 2 * 4 * D * n_rows
        nbuf = max(3, -(-(320 << 20) // per))
        xs = [torch.rand((n_rows, D), device=dev) for _ in range(nbuf)]
        outs = [torch.empty((n_rows, D), device=dev) for _ in range(nbuf)]
        t = csr_in.tiles(D) if D in ops._TILED_D and csr_in.seg_ptr is not None else None

        def one(i):
            if t is None:
                ops.spmm_sum(xs[i], csr_in, csr_out, 1.0)
            else:      # the C-ABI call itself, into a preallocated output (no allocation inside the captured region)
                L.call("dn4gl_spmm_tiled_f32", _lib.ptr(csr_in.row_ptr), _lib.ptr(csr_in.col), _lib.ptr(xs[i]), _lib.ptr(outs[i]), n_rows, D,
                       1.0, None, _lib.ptr(t["desc"]), t["T"], _lib.ptr(t["heavy_list"]), _lib.ptr(t["heavy_count"]), t["heavy_cap"],
                       t["smem"], t["stages"], t["npr"], t["warps"], torch.cuda.current_stream().cuda_stream)
        return _graph_b2b(one, nbuf, launches)

    def copy_back_to_back(n_rows, D, launches=64):
        """the same measurement for a plain device copy of one (n_rows, D) matrix into another (read N D 4 + write N D 4
        bytes = the two feature streams of the aggregation): what a kernel with no index work reaches AT THIS SIZE."""
        per = 2 * 4 * D * n_rows
        nbuf = max(3, -(-(320 << 20) // per))
        xs = [torch.rand((n_rows, D), device=dev) for _ in range(nbuf)]
        ys = [torch.empty((n_rows, D), device=dev) for _ in range(nbuf)]
        return _graph_b2b(lambda i: ys[i].copy_(xs[i]), nbuf, launches)

    # (a) one launch at a time behind an L2 flush (CUDA-event resolution ~2 us, includes the launch gap)
    xh = torch.rand((N, HID), device=dev)
    iso = []
    for _ in range(10):
        flush.fill_(1)
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        ops.spmm_sum(xh, s.csr_in, s.csr_out, 1.0)
        a1.record()
        torch.cuda.synchronize()
        iso.append(a0.elapsed_time(a1))
    del xh
    # (b) back to back over operands larger than L2: the number `achieved` is computed from
    b2b_us = k1_back_to_back(s.csr_in, s.csr_out, N, HID)
    agg_bytes = 4 * HID * N * 2 + 4 * E + 4 * (N + 1)        # SURVEY.md section 8(d): compulsory traffic
    agg_name = "dn4gl_spmm_tiled_f32" if ("dn4gl_spmm_tiled_f32[D=%d]" % HID) in per_entry else "dn4gl_spmm_sum_f32"
    in_step = per_entry.get("%s[D=%d]" % (agg_name, HID), {"avg_us": float("nan"), "calls": 0})
    achieved = agg_bytes / (b2b_us * 1e-6) / 1e9
    kern = ("spmm_pipe_kernel<8,1>: producer/consumer ring of cp.async.bulk staged tiles" if agg_name.endswith("tiled_f32")
            else "spmm_rows_kernel<8,1> + spmm_heavy_kernel<8,1>")
    traffic = traffic_src = None
    try:   # dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full` capture
        with open(os.path.join(ROOT, "profiles", "k1_c2_ncu_traffic.json")) as f:
            tj = json.load(f)
        traffic, traffic_src = tj["dram_bytes_read"] + tj["dram_bytes_write"], tj["source"]
    except Exception:   # noqa: BLE001
        pass
    roofline = {"kernel": "%s (%s), D=32, N=%d, E=%d" % (agg_name, kern, N, E),
                "bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                "frac": achieved / peaks["hbm_gbs"], "peak_source": which + " (MEASURED_PEAKS.json hbm_gbs)",
                "algorithmic_bytes_per_launch": agg_bytes,
                "how": "64 launches back to back (captured in one CUDA graph, replayed between two CUDA events on the launching "
                       "stream), operands rotated through a >= 320 MB pool (larger than L2)",
                "avg_launch_us": b2b_us,
                "in_step_eager_us": in_step["avg_us"], "in_step_eager_calls": in_step["calls"],
                "in_step_eager_note": "event pair around each C-ABI call of an eager step: includes the host launch gap",
                "cold_l2_single_launch_us": 1e3 * statistics.median(iso),
                "gather_effective_gbs": (4 * HID * (E + N) + 4 * E + 4 * (N + 1)) / (b2b_us * 1e-6) / 1e9,
                "traffic": traffic, "traffic_source": traffic_src}
    try:   # size-bound reference: a plain copy of the same two matrices, same method (DESIGN.md section 5)
        cus = copy_back_to_back(N, HID)
        roofline["copy_same_size"] = {"avg_launch_us": cus, "gbs": 8 * HID * N / (cus * 1e-6) / 1e9,
                                      "frac_of_peak": 8 * HID * N / (cus * 1e-6) / 1e9 / peaks["hbm_gbs"],
                                      "note": "torch copy_ of one (N, D) fp32 matrix into another, 64 launches back to back over "
                                              "a pool larger than L2: what a kernel without index work reaches at this size"}
        roofline["frac_of_copy_at_same_size"] = achieved / roofline["copy_same_size"]["gbs"]
    except Exception as ex:   # noqa: BLE001
        roofline["copy_same_size"] = {"error": str(ex)[:200]}
    # the same kernel at a C5 sweep point (BASELINE.json configs[4]): 16 384 MUTAG-shaped graphs + dummy, hidden 64
    roofline_c5 = None
    if rank == 0:
        try:
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            from agg_sweep import replicate
            from dummynode4graphlearning_b200.graph import BatchedGraph
            raw5 = replicate(synth.tu_batch("mutag", 1024, seed=0), 16)
            d5 = T.tu_add_dummy(T.to_device({k: v for k, v in raw5.items() if k != "vattr"}, dev))
            g5 = BatchedGraph(d5["src"], d5["dst"], d5["node_ptr"], d5["edge_ptr"])
            g5.host_ptrs()
            N5, E5, D5 = g5.number_of_nodes(), g5.number_of_edges(), 64
            us5 = k1_back_to_back(g5.csr_in, g5.csr_out, N5, D5, launches=32)
            b5 = 4 * D5 * N5 * 2 + 4 * E5 + 4 * (N5 + 1)
            roofline_c5 = {"workload": "c5 point: 16384 MUTAG-shaped graphs + dummy, hidden 64", "N": N5, "E": E5,
                           "algorithmic_bytes_per_launch": b5, "avg_launch_us": us5, "achieved": b5 / (us5 * 1e-6) / 1e9,
                           "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": b5 / (us5 * 1e-6) / 1e9 / peaks["hbm_gbs"]}
            del g5, d5
        except Exception as ex:   # noqa: BLE001
            roofline_c5 = {"error": str(ex)[:200]}
    # ---- C5 sweep (BASELINE.json configs[4]): batches of 1k-64k MUTAG-shaped graphs + dummy, hidden 64-512 ------------
    c5_sweep = None
    if rank == 0 and world == 1 and not a.no_extras:
        c5_sweep = []
        try:
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            from agg_sweep import replicate
            from dummynode4graphlearning_b200.graph import BatchedGraph
            base5 = synth.tu_batch("mutag", 1024, seed=0)
            for B5, dims in ((1024, (64, 512)), (4096, (64, 128, 256)), (16384, (64, 128, 256)), (65536, (64, 128))):
                raw5 = replicate(base5, B5 // 1024)
                d5 = T.tu_add_dummy(T.to_device({k: v for k, v in raw5.items() if k != "vattr"}, dev))
                g5 = BatchedGraph(d5["src"], d5["dst"], d5["node_ptr"], d5["edge_ptr"])
                g5.host_ptrs()
                N5, E5 = g5.number_of_nodes(), g5.number_of_edges()
                for D5 in dims:
                    us5 = k1_back_to_back(g5.csr_in, g5.csr_out, N5, D5, launches=24)
                    cu5 = copy_back_to_back(N5, D5, launches=24)
                    b5 = 4 * D5 * N5 * 2 + 4 * E5 + 4 * (N5 + 1)
                    c5_sweep.append({"graphs": B5, "D": D5, "N": N5, "E": E5, "algorithmic_bytes": b5, "avg_launch_us": round(us5, 2),
                                     "gbs": round(b5 / (us5 * 1e-6) / 1e9, 1), "frac": round(b5 / (us5 * 1e-6) / 1e9 / peaks["hbm_gbs"], 3),
                                     "frac_of_nominal_8tbs": round(b5 / (us5 * 1e-6) / 1e9 / 8000.0, 3),
                                     "graphs_per_s": round(B5 / (us5 * 1e-6)),
                                     "copy_same_size_us": round(cu5, 2), "copy_frac": round(8 * D5 * N5 / (cu5 * 1e-6) / 1e9 / peaks["hbm_gbs"], 3)})
                del g5, d5
                torch.cuda.empty_cache()
        except Exception as ex:   # noqa: BLE001
            c5_sweep.append({"error": str(ex)[:200]})
    # the tensor-core MLP stages of the same step (HBM-bound too, DESIGN.md section 4 K6): algorithmic GB/s from the
    # eager in-step event pairs (upper bound on the duration)
    mlp = {}
    for name, nbytes in (("dn4gl_lin_fwd_f32", 4 * N * (HID + HID)), ("dn4gl_lin_bwd_f32", 4 * N * (2 * HID + 2 * HID))):
        if name in per_entry:
            mlp[name] = {"in_step_eager_us": round(per_entry[name]["avg_us"], 2), "algorithmic_bytes": nbytes,
                         "gbs": round(nbytes / (per_entry[name]["avg_us"] * 1e-6) / 1e9, 1)}

    # ---- fixed global batch (strong scaling): the SAME 1113 graphs split over the ranks, balanced by edge count ----------
    strong = None
    if world > 1 and not a.no_extras:
        try:
            pipe._graphs.clear(); pipe._tgraphs.clear()
            full = synth.tu_batch("proteins", a.graphs, seed=0)
            mine = split_tu_batch({k: v for k, v in full.items() if k != "vattr"}, world)[rank]
            mine["conj_sizes"] = T.tu_conjugate_sizes_ex(mine, with_dummy=True)
            dev_s = T.to_device(mine, dev)
            torch.manual_seed(0)
            model_s = GIN(args).to(dev)
            pipe_s = ClassificationPipeline(model_s, FlatAdam(model_s.parameters(), lr=LR), mode="conj",
                                            num_node_labels=NUM_NODE_LABELS, node_label_min=0)
            pipe_s.global_batch = a.graphs
            for _ in range(30):
                flush.fill_(1)
                pipe_s.step_resident(dev_s, assume_ready=True)
            barrier()
            s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s0.record()
            for _ in range(a.steps):
                flush.fill_(1)
                pipe_s.step_resident(dev_s, assume_ready=True)
            s1.record()
            barrier()
            ms_s = max_over_ranks(s0.elapsed_time(s1), dev) / a.steps
            strong = {"global_batch": a.graphs, "graphs_on_rank0": int(mine["num_graphs"]), "ms_per_step": ms_s,
                      "value": a.graphs / (ms_s * 1e-3), "unit": "graphs/s",
                      "note": "the same C2 mini-batch (1113 graphs) sharded over the ranks by edge count; weak-scaling `value` "
                              "above gives every rank its own 1113 graphs"}
            pipe_s._graphs.clear(); pipe_s._tgraphs.clear()
        except Exception as ex:   # noqa: BLE001
            strong = {"error": str(ex)[:300]}
    # ---- the other BASELINE configurations -------------------------------------------------------------------------
    configs = {}
    if not a.no_extras:
        pipe._graphs.clear()                      # free the C2 graphs' static buffers before the other pipelines capture theirs
        torch.cuda.empty_cache()
        want_cpu = world == 1 and not a.no_cpu_baseline
        try:   # C4 (DMPNN 'large', per-GPU batch 64) runs data-parallel on every rank: the 8-GPU configuration of BASELINE.json
            r4, ctx4 = gpu_counting_run("c4", dev, world, rank, steps=20)
            if want_cpu and rank == 0:
                r4["cpu_baseline"] = cpu_counting_run(*ctx4, steps=2, warmup=1)
            configs["c4_dmpnn_large"] = r4
        except Exception as ex:   # noqa: BLE001
            configs["c4_dmpnn_large"] = {"error": str(ex)[:300]}
        if world == 1:
            try:
                r3, ctx3 = gpu_counting_run("c3", dev, 1, 0, steps=20)
                if want_cpu:
                    r3["cpu_baseline"] = cpu_counting_run(*ctx3, steps=2, warmup=1)
                configs["c3_rgin_small"] = r3
            except Exception as ex:   # noqa: BLE001
                configs["c3_rgin_small"] = {"error": str(ex)[:300]}
            for key, hid1, lay1, note in (("c1_gin_mutag_hid128", 128, 2, "main.py:174 defaults (hidden 128, 2 layers)"),
                                          ("c1_gin_mutag_hid32", 32, 4, "hyper_params.py:15 (hidden 32, 4 layers)")):
                try:
                    r1, raw1 = gpu_classification_run("mutag", 188, "dummy", hid1, lay1, 8, dev, steps=50)
                    r1["workload"] = "c1: dummy augmentation + GIN(%s) train step, 188 MUTAG-shaped graphs" % note
                    if want_cpu:
                        c1 = cpu_reference_run(raw1, 10, 2, mode="dummy", hid=hid1, layers=lay1, num_labels=8)
                        r1["cpu_baseline"] = {"value": c1["graphs_per_s"], "unit": "graphs/s", "cores": c1["cores"], "kind": "port",
                                              "ms_per_step": c1["ms_per_step"], "sample": "full batch (188 graphs) per step, 10 timed steps"}
                    configs[key] = r1
                except Exception as ex:   # noqa: BLE001
                    configs[key] = {"error": str(ex)[:300]}
    # ---- the tensor-core MLP stages alone at the C2 size (graph-captured back to back, operands rotated through > L2) ----
    if rank == 0:
        try:
            nb = 16
            Xs = [torch.randn(N, HID, device=dev) for _ in range(nb)]
            Gs = [torch.randn(N, HID, device=dev) for _ in range(nb)]
            Wm = torch.randn(HID, HID, device=dev) / HID ** 0.5
            bm = torch.randn(HID, device=dev)
            bnp = dict(gamma=torch.ones(HID, device=dev), beta=torch.zeros(HID, device=dev), eps=1e-5, momentum=0.1)
            Y0, rec0 = ops.lin_fwd(Xs[0], Wm, bm, bn=bnp)
            sums0 = ops.bn_bwd_sums(Gs[0], Y0, rec0)
            fwd_us = _graph_b2b(lambda i: ops.lin_fwd(Xs[i], Wm, bm, in_bn=rec0, in_act=1, bn=bnp), nb, 32)
            bwd_us = _graph_b2b(lambda i: ops.lin_bwd(Gs[i], Wm, Xs[i], Yout=Y0, bn=rec0, sums=sums0, in_bn=rec0, in_act=1), nb, 32)
            fb, bb = 4 * N * 2 * HID, 4 * N * 4 * HID
            mlp["back_to_back"] = {
                "rows": N, "D": HID,
                "lin_fwd_bn_stats": {"avg_launch_us": round(fwd_us, 2), "algorithmic_bytes": fb, "gbs": round(fb / (fwd_us * 1e-6) / 1e9, 1),
                                     "frac": round(fb / (fwd_us * 1e-6) / 1e9 / peaks["hbm_gbs"], 3)},
                "lin_bwd_bn": {"avg_launch_us": round(bwd_us, 2), "algorithmic_bytes": bb, "gbs": round(bb / (bwd_us * 1e-6) / 1e9, 1),
                               "frac": round(bb / (bwd_us * 1e-6) / 1e9 / peaks["hbm_gbs"], 3)},
                "how": "32 launches captured in one CUDA graph over 16 rotating input sets (> L2), replayed between two events; "
                       "HBM-bound stages: tensor-pipe utilisation from ncu is in profiles/ (8-14 % at D = 32)"}
            del Xs, Gs
        except Exception as ex:   # noqa: BLE001
            mlp["back_to_back"] = {"error": str(ex)[:200]}
    if rank != 0:
        _finish(pipe, world)
        return
    cpu = None
    if world == 1 and not a.no_cpu_baseline:
        r = cpu_reference_run(raw, 10, 2)
        cpu = {"value": r["graphs_per_s"], "unit": "graphs/s", "cores": r["cores"], "kind": "port",
               "sample": "full C2 batch (%d graphs) per step, 10 timed steps after 2 warm-up" % a.graphs,
               "transform_ms": r["transform_ms"], "train_ms": r["train_ms"]}
    own_ms = sum(v["total_ms"] for v in per_entry.values()) / max(len(tr_ms), 1)
    line = {
        "metric": "train graphs/sec", "value": value, "unit": "graphs/s", "n_gpus": world, "steps": a.steps,
        "warmup": n_warm, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": dict(workload_config(a.graphs, world), **({"size_hints": "the loader attaches the closed-form output sizes of the edge-to-vertex transform "
                       "(transforms.tu_conjugate_sizes_ex of the raw host batch: V', E', largest graph, 'every graph has a node', "
                       "'edges sorted by source'): no device->host read inside a step, the CONJ_ CSR pair is written in closed "
                       "form (dn4gl_tu_conj_direct_*) and the whole transform replays as a CUDA graph"} if a.size_hints else {})),
        "clocks": clk, "gpu_launches": launches, "l2_flush": l2_flush,
        "e2e": {"value": e2e_value, "unit": "graphs/s", "ms_per_step": e2e_ms,
                "h2d_bytes_per_step": host_bytes(host), "d2h_bytes_per_step": 4 + 8 + 4,
                "how": "ClassificationPipeline.step_async(host) per step, loss of step k-1 read on the host after step k "
                       "is submitted (all losses read, last one before the clock stops)"},
        "roofline": roofline, "roofline_c5": roofline_c5, "c5_sweep": c5_sweep, "configs": configs, "strong_scaling": strong,
        "mlp_stages": mlp,
        "transform": transform_only, "transform_as_run": transform_replay, "cpu_baseline": cpu,
        "breakdown": {"how": "instrumented pass AFTER the timed regions: eager launches on one stream with a CUDA-event pair "
                             "around every C-ABI call (medians over %d steps); slower than the measured step by "
                             "construction -- use it for shares, not for totals" % len(tr_ms),
                      "transform_ms": statistics.median(tr_ms), "train_ms": statistics.median(tn_ms),
                      "own_kernels_ms_per_step": own_ms,
                      "cudaMalloc_calls_in_timed_region": m1 - m0, "cudaMalloc_calls_in_e2e_region": m2 - m1, "conj_nodes": N, "conj_edges": E,
                      "final_loss": final_loss, "e2e_last_loss": last,
                      "entry_points": {k: {"calls_per_step": v["calls"] / max(len(tr_ms), 1), "avg_us": round(v["avg_us"], 2)}
                                       for k, v in sorted(per_entry.items(), key=lambda kv: -kv[1]["total_ms"])}},
    }
    print(json.dumps(line))
    _finish(pipe, world)


def _finish(pipe, world):
    """multi-rank teardown: the captured train step holds NCCL work inside live CUDA graphs, and
    destroy_process_group() blocks on that (observed: both ranks hang after the line is printed).  Drop the graphs,
    drain the device and leave the process directly -- the measurement is complete and printed."""
    import sys
    sys.stdout.flush()
    sys.stderr.flush()
    if world > 1:
        pipe._graphs.clear()
        torch.cuda.synchronize()
        os._exit(0)


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        reference_arm(a)
    else:
        ours(a)
