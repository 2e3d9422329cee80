#!/usr/bin/env python
"""Timeline of one steady-state training step of the bench workload (bench.py's model, data and trainer).

Replays the captured step `--steps` times under torch.profiler (CUDA activities), L2 flushed between steps as in the
bench, writes the Chrome trace to OUT/trace.json and prints, for one step in the middle of the window: every kernel
and copy with its stream, start and end relative to the step's first event, the idle gap before each kernel of the
critical path (pack -> forward x L -> backward x L -> block-1 weight gradient -> step tail; negative: it started before
its predecessor ended) and the step span against the sum of critical-path kernel times.

  python tools/step_timeline.py --out DIR [--batch 4096] [--precision tf32] [--steps 50]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402  (constants, synthetic data and the kernel-name shortener of the bench)


def build_trainer(batch, precision, dev):
    import torch
    from stnf.models import STInterpMLP
    from stnf.dataio import ObservationTable
    from st_dadk_b200.trainer import Trainer
    n_train = max(bench.N_TRAIN, 4 * batch)
    torch.manual_seed(2025)
    model = STInterpMLP(k_spatial_centers=bench.K_SPATIAL, k_temporal_centers=bench.K_TEMPORAL, hidden_dims=bench.HIDDEN,
                        dropout=0.1, layernorm=True, output_dim=1)
    _, coords, t, y = bench.synth_dataset(2025, n_train)
    table = ObservationTable(torch.from_numpy(coords), torch.from_numpy(t), torch.from_numpy(y)).to(dev)
    tr = Trainer(model, dict(bench.CFG, precision=precision), dev, batches_per_epoch=(n_train + batch - 1) // batch,
                 use_cuda_graph=True)
    perm = torch.randperm(n_train, generator=torch.Generator().manual_seed(7)).to(dev)
    n_off = (n_train - batch) // batch
    return lambda i: tr.train_step(table, perm, (i % n_off) * batch, batch, batch)


def critical_path(events):
    """The chain pack -> layer_fwd ... -> layer_bwd ... -> wgrad of block 1 -> fused step tail, in launch order."""
    chain = []
    for e in events:
        n = e["short"]
        if n.startswith(("pack_images_kernel", "layer_fwd_kernel", "layer_bwd_kernel", "adamw_ema_kernel")):
            chain.append(e)
    wg1 = [e for e in events if e["short"].startswith("wgrad_kernel<true")]
    if wg1:
        tail = next((i for i, e in enumerate(chain) if e["short"].startswith("adamw_ema_kernel")), len(chain))
        chain.insert(tail, wg1[-1])
    return chain


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--batch", type=int, default=bench.BATCH)
    ap.add_argument("--precision", default="tf32", choices=["tf32", "tf32x3"])
    ap.add_argument("--steps", type=int, default=50)
    args = ap.parse_args()
    import torch
    from torch.profiler import profile, ProfilerActivity
    dev = torch.device("cuda", 0)
    step = build_trainer(args.batch, args.precision, dev)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
    for i in range(5):                       # the first step captures the graph
        step(i)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for i in range(args.steps):
            flush.fill_(1.0)
            step(5 + i)
        torch.cuda.synchronize()
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "trace.json")
    prof.export_chrome_trace(path)

    with open(path) as f:
        trace = json.load(f)
    evs = [e for e in trace["traceEvents"] if e.get("ph") == "X" and e.get("cat") in ("kernel", "gpu_memcpy", "gpu_memset")]
    evs.sort(key=lambda e: e["ts"])
    for e in evs:
        e["short"] = bench.short_kernel_name(e["name"]) if e["cat"] == "kernel" else e["name"]
        e["stream"] = e.get("args", {}).get("stream", -1)
    # the L2 flush (a fill kernel of 256 MB) opens every step's window
    starts = [i for i, e in enumerate(evs) if e["cat"] == "kernel" and "fill" in e["name"].lower() and e["dur"] > 5]
    if len(starts) < 3:
        raise SystemExit(f"found {len(starts)} step windows in the trace; expected {args.steps}")
    k = len(starts) // 2
    window = evs[starts[k] + 1:starts[k + 1]]
    t0 = window[0]["ts"]
    spans = []
    for a, b in zip(starts[1:-1], starts[2:]):
        w = evs[a + 1:b]
        spans.append(max(e["ts"] + e["dur"] for e in w) - min(e["ts"] for e in w))
    chain = critical_path(window)
    ids = {id(e) for e in chain}

    lines = [f"device: {torch.cuda.get_device_name(0)}; batch {args.batch}, {args.precision}; step {k} of {len(starts)}",
             f"{'start us':>9} {'end us':>9} {'dur us':>8} {'gap us':>8} {'stream':>6}  kernel ('*': critical path)"]
    prev_end = None
    for e in window:
        s, d = e["ts"] - t0, e["dur"]
        gap = ""
        if id(e) in ids:
            if prev_end is not None:
                gap = f"{s - prev_end:8.1f}"
            prev_end = s + d
        lines.append(f"{s:9.1f} {s + d:9.1f} {d:8.1f} {gap:>8} {e['stream']:>6}  {'*' if id(e) in ids else ' '}{e['short']}")
    crit_sum = sum(e["dur"] for e in chain)
    chain_span = chain[-1]["ts"] + chain[-1]["dur"] - chain[0]["ts"] if chain else 0.0
    span = max(e["ts"] + e["dur"] for e in window) - t0
    spans.sort()
    lines += [f"critical path: {len(chain)} kernels, sum of durations {crit_sum:.1f} us, first start -> last end "
              f"{chain_span:.1f} us (idle or overlapped: {chain_span - crit_sum:.1f} us)",
              f"step span (first event -> last end) {span:.1f} us; median over the {len(spans)} traced steps "
              f"{spans[len(spans) // 2]:.1f} us (profiler on)"]
    text = "\n".join(lines)
    print(text)
    with open(os.path.join(args.out, "timeline.txt"), "w") as f:
        f.write(text + "\n")


if __name__ == "__main__":
    main()
