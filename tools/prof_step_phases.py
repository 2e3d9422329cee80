#!/usr/bin/env python
"""Where the time of the training step's forward and backward kernels and fused tail goes around their
programmatic-launch wait.

Needs the profiling build (tools/build_dbg.sh) through STDADK_LIB=st_dadk_b200/libstdadk_dbg.so: its layer_fwd
(FWD_T in layer.cuh), layer_bwd and adamw_ema kernels (STEP_T in common.cuh) stamp globaltimer phases into
stdadk_debug_step_counters.  Two trainers of the
bench workload (bench.py's model, data and batch), one that reads settled inputs before the wait (Executor.prewait,
the default) and one that reads everything after it (the order of the parent commit), replay their captured steps
alternately, L2 flushed between steps as in the bench.  Printed: mean ns per CTA and step of each phase, per kernel.

  STDADK_LIB=st_dadk_b200/libstdadk_dbg.so python tools/prof_step_phases.py [--steps 200] [--out FILE]
"""
import argparse
import ctypes
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

# layer_fwd's counters in phase order (slot, name); slot 8 counts the CTAs
FWD = [(0, "prologue"), (9, "before wait"), (10, "wait"), (1, "operand"), (2, "accumulator"), (3, "epilogue"), (4, "tail")]
BWD = ["prologue", "before wait", "wait", "accumulator", "pass A", "pass B + flush"]
TAIL = ["early loads", "wait", "g + norm partials", "grid barrier", "update"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--out")
    args = ap.parse_args()
    import torch
    import bench
    from step_timeline import build_trainer
    from st_dadk_b200 import _lib as L
    if "dbg" not in L.LIB_PATH:
        raise SystemExit("run with STDADK_LIB pointing at the profiling build (tools/build_dbg.sh)")
    dev = torch.device("cuda", 0)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
    runs = {}
    for mode in ("after wait", "before wait"):
        cnt = torch.zeros(128, dtype=torch.int64, device=dev)
        L.lib().stdadk_debug_step_counters(ctypes.c_void_p(cnt.data_ptr()))   # captured into the graph
        os.environ["STDADK_PREWAIT"] = "1" if mode == "before wait" else "0"
        step = build_trainer(bench.BATCH, "tf32", dev)
        for i in range(5):
            step(i)
        runs[mode] = (step, cnt)
    L.lib().stdadk_debug_step_counters(ctypes.c_void_p(0))
    torch.cuda.synchronize()
    for _, cnt in runs.values():
        cnt.zero_()
    for i in range(args.steps):
        for step, _ in runs.values():
            flush.fill_(1.0)
            step(5 + i)
    torch.cuda.synchronize()
    props = torch.cuda.get_device_properties(0)
    lines = [f"device: {props.name}; batch {bench.BATCH}, tf32; {args.steps} steps per mode, alternating; "
             "mean ns per CTA and step"]
    for mode, (_, cnt) in runs.items():
        v = cnt.cpu().tolist()
        lines.append(f"-- inputs read {mode}")
        for l in range(4):
            c = v[64 + 16 * l + 8]
            if c:
                ph = [v[64 + 16 * l + k] / c for k, _ in FWD]
                lines.append(f"  layer_fwd block {l + 1:d}: " + ", ".join(f"{n} {x:.0f}" for (_, n), x in zip(FWD, ph)) +
                             f" | after wait {sum(ph[3:]):.0f}")
        for l in range(7):
            c = v[8 * l + 7]
            if c:
                ph = [v[8 * l + k] / c for k in range(len(BWD))]
                lines.append(f"  layer_bwd block {l + 1:d}: " + ", ".join(f"{n} {x:.0f}" for n, x in zip(BWD, ph)) +
                             f" | after wait {sum(ph[3:]):.0f}")
        c = v[63]
        if c:
            ph = [v[56 + k] / c for k in range(len(TAIL))]
            lines.append("  adamw_ema tail: " + ", ".join(f"{n} {x:.0f}" for n, x in zip(TAIL, ph)) +
                         f" | after wait {sum(ph[2:]):.0f}")
    text = "\n".join(lines)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
