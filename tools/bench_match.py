"""The matching objective on the C4 shape (DMPNN 'large', batch 64, node + edge match weights) against the same model's
unmatched step; figures for DESIGN.md (bench.py reports the C2 line).

  python tools/bench_match.py [--steps 30] [--warmup 5] [--samples 640] [--out FILE.json]

(a) a fixed batch, train step replayed as a CUDA graph: unmatched vs matched (fused match loss);
(b) a fixed batch, eager train step: matched through the tensor composition losses.counting_bp_loss vs the fused loss;
(c) three shuffled epochs of step_indices on a resident data set: unmatched vs match_weights="node,edge";
(d) torch.profiler kernel times of dn4gl_subiso_append_dummy and the two match-loss kernels in eager matched steps.
The card's name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

BS = 64
KERNELS = ("subiso_append_dummy_kernel", "match_loss_kernel", "match_loss_bwd_kernel")


def _card():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], text=True)
        name, power = [s.strip() for s in out.splitlines()[0].split(",")]
    except (OSError, subprocess.CalledProcessError, ValueError, IndexError):
        name, power = torch.cuda.get_device_name(0), "unknown"
    return dict(name=name, power_limit=power)


def _model(dev):
    from bench_counting import build
    return build("DMPNN", "large", dict(node_pred=True, edge_pred=True, pred_return_weights="node,edge"), dev)[:2]


def _pipe(dev, match_weights=None, cuda_graphs=True):
    from dummynode4graphlearning_b200.optim import FlatAdam
    from dummynode4graphlearning_b200.pipelines import CountingPipeline
    model, cfg = _model(dev)
    opt = FlatAdam(model.parameters(), lr=1e-3, weight_decay=1e-2, amsgrad=True, decoupled_weight_decay=True)
    return CountingPipeline(model, opt, cfg, add_dummy=True, rep_reg_w=1e-3, cuda_graphs=cuda_graphs,
                            match_weights=match_weights, match_loss_w=1.0, match_reg_w=0.01)


def _timed(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def _fixed_batch(pipe, samples, dev):
    """one C4 batch (dummy column by the host helper), augmented, with its match weights."""
    from dummynode4graphlearning_b200 import transforms as T
    from dummynode4graphlearning_b200.subgraph_isomorphism import io as sio, matching as M
    p, g, counts, mats = sio.collate(samples[:BS])
    p_aug, g_aug = pipe.augment(T.to_device(p, dev), T.to_device(g, dev))
    sub = M.pack_subisomorphisms(M.add_dummy_to_subisomorphisms(mats, g), dev)
    nw, ew = M.node_weights_i32(sub, g_aug), M.edge_weights_i32(sub, p_aug, g_aug)
    pattern, graph = pipe.transform(T.to_device(p, dev), T.to_device(g, dev))
    return pattern, graph, torch.from_numpy(counts).to(dev), nw, ew


def _eager_composed(pipe, pattern, graph, counts, nw, ew):
    """the eager train step with the match terms of losses.counting_bp_loss (what train_on ran before the fused loss)."""
    pipe.bucket.zero()
    out = pipe.model(pattern, graph)
    loss = pipe.match_loss_fn(out, counts, graph, nw.long(), ew.long())
    loss.backward()
    pipe.bucket.gather()
    flat = pipe.bucket.flat
    flat.mul_((pipe.max_grad_norm / (torch.linalg.vector_norm(flat) + 1e-6)).clamp(max=1.0))
    pipe.opt.step()
    return loss.detach()


def _launch_bytes(graph, B):
    """bytes each match-loss launch must move (from the shapes): per position pred (4) + mask (1), per real row its int32
    weight, per graph pred_c and the two offsets; the backward also writes 4 bytes per position and pred_c's gradient."""
    Lv, Le = graph.padded_num_nodes(), graph.padded_num_edges()
    pos, rows = B * (Lv + Le), graph.number_of_nodes() + graph.number_of_edges()
    fwd = 5 * pos + 4 * rows + B * (4 + 2 * 4)
    return dict(positions=pos, weight_rows=rows, fwd_bytes=fwd, bwd_bytes=fwd + 4 * pos + 4 * B)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--samples", type=int, default=640)
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_match: needs a CUDA device")
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from dummynode4graphlearning_b200 import synth
    from dummynode4graphlearning_b200.datasets import EpochSampler, ResidentCountingDataset
    dev = torch.device("cuda:0")
    res = dict(card=_card(), shape="C4: DMPNN 'large', batch %d, match weights node + edge" % BS)
    samples = synth.counting_samples("large", a.samples, seed=0)

    # (a) captured replay of a fixed batch
    ms = {}
    for tag, mw in (("unmatched", None), ("matched", "node,edge")):
        pipe = _pipe(dev, mw)
        pattern, graph, counts, nw, ew = _fixed_batch(pipe, samples, dev)
        w = (nw, ew) if mw else (None, None)
        ms[tag] = _timed(lambda: pipe.train_on(pattern, graph, counts, *w), a.steps, a.warmup)
        assert pipe.replayed_library_kernels() > 0
    res["replay_ms_per_step"] = ms
    res["launch_bytes"] = _launch_bytes(graph, BS)

    # (b) eager matched step: tensor composition vs fused loss
    pipe = _pipe(dev, "node,edge", cuda_graphs=False)
    batch = _fixed_batch(pipe, samples, dev)
    res["eager_ms_per_step"] = dict(
        composed=_timed(lambda: _eager_composed(pipe, *batch), a.steps, a.warmup),
        fused=_timed(lambda: pipe.train_on(*batch[:3], node_weights=batch[3], edge_weights=batch[4]), a.steps, a.warmup),
        unmatched=_timed(lambda: pipe.train_on(*batch[:3]), a.steps, a.warmup))

    # (c) three shuffled step_indices epochs
    ds = ResidentCountingDataset(samples, dev)
    sampler = EpochSampler(len(ds), BS, seed=1, drop_last=True)
    epochs = {}
    for tag, mw in (("unmatched", None), ("matched", "node,edge")):
        pipe = _pipe(dev, mw)
        for idx, n in sampler.batches(0):          # warm-up epoch: every signature seen and captured
            pipe.step_indices(ds, idx, n)
        pipe.step_indices(ds, idx, n).result()
        t0 = time.perf_counter()
        steps = 0
        for e in range(1, 4):
            for idx, n in sampler.batches(e):
                last = pipe.step_indices(ds, idx, n)
                steps += 1
        last.result()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        epochs[tag] = dict(steps=steps, ms_per_step=1e3 * dt / steps, samples_per_s=steps * BS / dt)
    res["step_indices_3_epochs"] = epochs

    # (d) kernel times inside eager matched step_indices steps (profiled in a run of their own)
    from torch.profiler import ProfilerActivity, profile
    pipe = _pipe(dev, "node,edge", cuda_graphs=False)
    for idx, n in sampler.batches(4):
        pipe.step_indices(ds, idx, n)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for idx, n in sampler.batches(4):
            pipe.step_indices(ds, idx, n)
        torch.cuda.synchronize()
    ker = {}
    for ev in prof.key_averages():
        for k in KERNELS:
            if ev.key.startswith(k + "(") or ev.key == k:
                t = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0)
                ker[k] = dict(calls=ev.count, mean_us=t / max(ev.count, 1))
    res["kernels"] = ker
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
