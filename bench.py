#!/usr/bin/env python
"""Benchmark of the ST-DADK hot path (contract: see the task statement / DESIGN.md section "Measurement").

Workload (BASELINE.json configs[1], the largest single-GPU configuration): the data/2b-shaped problem --
S=10,000 sites x T=100 time steps, 100k observed, 80k training samples, batch 4096 (20 steps/epoch), default
basis resolutions [25,81,121] / [10,15,45], MLP 297-256-256-128-1, LayerNorm, dropout 0.1, AdamW + clip + EMA --
with synthetic targets on synthetic U[0,1]^2 sites (the 2b training blobs are absent upstream and the GPU box has no
copy of the reference tree).

A "step" is one optimisation step over one batch of 4096 samples per GPU (forward with the basis fused into block 1,
fused loss, backward with basis recompute, [one NCCL all-reduce of the flat gradient], grad-norm, fused clip+AdamW+EMA).
`value` = training samples/s over all ranks with the dataset resident in HBM, timed per step with CUDA events on the
launching stream, L2 flushed between steps, max over ranks.  The same JSON line carries the dense-prediction
throughput (1M = T x S points, sharded by point), the end-to-end numbers through the host-buffer API, the roofline of
the dominant kernel and the CPU baseline.

  python bench.py --gpus N --steps K --warmup W            # our arm (torchrun for N > 1)
  python bench.py ... --dump-outputs DIR                   # also write the last timed step's results to DIR/*.npy
  python bench.py --impl reference --gpus N ...            # CPU arm: the reference's own PyTorch path (oracle/_ref, the
                                                           # unmodified `stnf` package) on the host cores, rank 0 only
  python bench.py --config 1|3|4|5 [--gpus N]              # the other BASELINE configs, one JSON line each (profiles/)

The bench compiles nothing and writes nothing into the tree (it may be read-only): it runs the library that
`__graft_entry__.build()` left there, so rebuild after changing a kernel.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

S_SITES, T_STEPS, N_TRAIN, BATCH = 10_000, 100, 80_000, 4096
HIDDEN = [256, 256, 128]
K_SPATIAL, K_TEMPORAL = [25, 81, 121], [10, 15, 45]
CFG = dict(lr=2e-2, weight_decay=5e-4, grad_clip=10.0, regression_type="mean", scheduler="cosine", epochs=500,
           warmup_epochs=10, dropout=0.1, layernorm=True, hidden_dims=HIDDEN, k_spatial_centers=K_SPATIAL,
           k_temporal_centers=K_TEMPORAL)
METRIC, UNIT = "train_samples_per_s", "samples/s"
WORKLOAD = "data/2b-shaped train+predict: S=10000 x T=100, 80k train samples, batch 4096/GPU, default basis [25,81,121]/[10,15,45], MLP 297-256-256-128-1"


def synth_field(coords, t, rng):
    x, y = coords[:, 0], coords[:, 1]
    return (np.sin(2 * np.pi * (x + t)) * np.cos(2 * np.pi * y) + 0.5 * np.sin(6 * np.pi * x * y)
            + 0.1 * rng.standard_normal(len(x))).astype(np.float32)


def synth_dataset(seed, n):
    """n observed (site, time) samples of the S x T problem, sorted by (t, site) like the upstream dataset."""
    rng = np.random.default_rng(seed)
    sites = rng.random((S_SITES, 2)).astype(np.float32)
    flat = np.sort(rng.choice(S_SITES * T_STEPS, size=n, replace=False))
    ti, si = flat // S_SITES, flat % S_SITES
    coords = sites[si]
    t = (ti / (T_STEPS - 1)).astype(np.float32)
    return sites, coords, t, synth_field(coords, t, rng)


# ------------------------------------------------------------------------------------------------ CPU arm
def oracle_model(seed=0):
    from oracle import stdadk_oracle as orc
    rng = np.random.default_rng(seed)
    c, b = orc.uniform_spatial_knots(K_SPATIAL)
    tc, tb = orc.temporal_knots(K_TEMPORAL)
    dims = [c.shape[0] + tc.shape[0], *HIDDEN]
    ws, bs, gs, be = [], [], [], []
    for i in range(len(HIDDEN)):
        bound = 1 / np.sqrt(dims[i])
        ws.append(rng.uniform(-bound, bound, (dims[i + 1], dims[i])).astype(np.float32))
        bs.append(rng.uniform(-bound, bound, dims[i + 1]).astype(np.float32))
        gs.append(np.ones(dims[i + 1], np.float32))
        be.append(np.zeros(dims[i + 1], np.float32))
    bound = 1 / np.sqrt(dims[-1])
    ws.append(rng.uniform(-bound, bound, (1, dims[-1])).astype(np.float32))
    bs.append(rng.uniform(-bound, bound, 1).astype(np.float32))
    return orc.OracleModel(centers=c, bandwidths=b, t_centers=tc, t_bandwidths=tb, weights=ws, biases=bs,
                           ln_gamma=gs, ln_beta=be, dropout=0.1)


def oracle_train_step(m, state, coords, t, y, step):
    """One CPU training step with the oracle port (FP32 numpy on the host BLAS threads): forward with dropout,
    MSE, backward, global-norm clip, AdamW, EMA -- the work of upstream's loop body (train_st_interp.py:608-712)."""
    from oracle import stdadk_oracle as orc
    n = coords.shape[0]
    rng = np.random.default_rng(step)
    masks = [rng.random((n, w.shape[0]), dtype=np.float32) >= 0.1 for w in m.weights[:-1]]
    yh, cache = orc.forward(m, None, coords, t[:, None], dtype=np.float32, train=True, keep_masks=masks,
                            return_cache=True)
    loss, dy = orc.loss_and_grad(yh, y, "mse")
    g = orc.backward(m, cache, dy.astype(np.float32))
    params = m.weights + m.biases + m.ln_gamma + m.ln_beta
    grads = g["weights"] + g["biases"] + g["ln_gamma"] + g["ln_beta"]
    _, coef = orc.clip_coef(grads, 10.0)
    for i, (p, gr) in enumerate(zip(params, grads)):
        st = state.setdefault(i, (np.zeros_like(p), np.zeros_like(p), p.copy()))
        orc.adamw_ema_step(p, gr.astype(np.float32), st[0], st[1], st[2], step, 2e-2, 5e-4, 0.995, clip=coef)
    return loss


def _ref_package():
    """The reference's own `stnf` package, copied unmodified into oracle/_ref by oracle/Makefile (build container) and
    shipped to the GPU box with the snapshot.  Returns the module pair or None when the copy is absent."""
    ref_dir = os.path.join(ROOT, "oracle", "_ref")
    if not os.path.isdir(os.path.join(ref_dir, "stnf")):
        return None
    import importlib.util
    saved = {k: v for k, v in sys.modules.items() if k == "stnf" or k.startswith("stnf.")}
    for k in saved:
        del sys.modules[k]
    sys.path.insert(0, ref_dir)
    try:
        models = importlib.import_module("stnf.models.st_interp")
        ema = importlib.import_module("stnf.utils.ema")
    finally:
        sys.path.remove(ref_dir)
        for k in [k for k in sys.modules if k == "stnf" or k.startswith("stnf.")]:
            del sys.modules[k]        # the reference modules stay referenced by the objects returned below only
        sys.modules.update(saved)
    assert os.path.realpath(models.__file__).startswith(os.path.realpath(ref_dir))
    return models, ema


class ReferenceArm:
    """The reference's CPU PyTorch path for the bench workload: STInterpMLP (st_interp.py:599-882) + nn.MSELoss +
    clip_grad_norm_ + optim.AdamW + ModelEMA, i.e. the loop body of train_model (train_st_interp.py:608-733) on
    pre-batched tensors (its list-of-dict DataLoader, 16.6 ms per 4096-batch, is left out in the reference's favour)."""

    def __init__(self):
        import torch
        mods = _ref_package()
        if mods is None:
            raise RuntimeError("oracle/_ref is absent")
        models, ema = mods
        self.torch = torch
        torch.set_num_threads(os.cpu_count())       # torchrun exports OMP_NUM_THREADS=1: use every host core anyway
        torch.manual_seed(2025)
        self.model = models.STInterpMLP(k_spatial_centers=K_SPATIAL, k_temporal_centers=K_TEMPORAL, hidden_dims=HIDDEN,
                                        dropout=0.1, layernorm=True, output_dim=1)
        self.opt = torch.optim.AdamW(self.model.parameters(), lr=CFG["lr"], weight_decay=CFG["weight_decay"])
        bpe = (N_TRAIN + BATCH - 1) // BATCH
        self.ema = ema.ModelEMA(self.model, decay=1.0 - 1.0 / (10.0 * bpe))
        self.crit = torch.nn.MSELoss()
        _, coords, t, y = synth_dataset(2025, N_TRAIN)
        self.c, self.t, self.y = torch.from_numpy(coords), torch.from_numpy(t)[:, None], torch.from_numpy(y)[:, None]
        self.X = torch.zeros(BATCH, 0)
        self.threads = torch.get_num_threads()

    def step(self, i):
        torch = self.torch
        lo = (i * BATCH) % (N_TRAIN - BATCH)
        self.model.train()
        self.opt.zero_grad()
        pred = self.model(self.X, self.c[lo:lo + BATCH], self.t[lo:lo + BATCH])
        loss = self.crit(pred, self.y[lo:lo + BATCH])
        loss.backward()
        torch.nn.utils.clip_grad_norm_(self.model.parameters(), CFG["grad_clip"])
        self.opt.step()
        self.ema.update(self.model)
        return loss.item()

    def predict_points_per_s(self, n_p=32768):
        torch = self.torch
        self.model.eval()
        g = torch.Generator().manual_seed(1)
        pc, pt = torch.rand(n_p, 2, generator=g), torch.rand(n_p, 1, generator=g)
        with torch.no_grad():
            self.model(torch.zeros(n_p, 0), pc, pt)
            t0 = time.perf_counter()
            self.model(torch.zeros(n_p, 0), pc, pt)
        return n_p / (time.perf_counter() - t0)


def cpu_baseline(seconds=12.0, max_steps=40):
    """Bounded sample of the same workload on the host cores.  The reference's own PyTorch CPU path when oracle/_ref is
    present (kind "reference"); otherwise the numpy oracle port (kind "port")."""
    try:
        arm = ReferenceArm()
    except Exception as e:        # noqa: BLE001 -- no copy of the reference on this box: fall back to the port, say so
        print(f"[bench] reference package unavailable ({e!r}); cpu_baseline uses the oracle port", file=sys.stderr)
        return cpu_baseline_port(seconds)
    for i in range(2):
        arm.step(i)
    times = []
    t_end = time.perf_counter() + seconds
    s = 2
    while len(times) < max_steps and (time.perf_counter() < t_end or len(times) < 3):
        t0 = time.perf_counter()
        arm.step(s)
        times.append(time.perf_counter() - t0)
        s += 1
    per = float(np.median(times))
    return {"value": BATCH / per, "unit": UNIT, "cores": arm.threads, "kind": "reference",
            "sample": f"{len(times)} training steps of batch {BATCH} of the reference's own STInterpMLP + AdamW + clip + "
                      f"ModelEMA on pre-batched CPU tensors (no DataLoader), median; predict sample 32768 points",
            "ms_per_step": per * 1e3, "predict_points_per_s": arm.predict_points_per_s()}


def cpu_baseline_port(seconds=12.0, max_steps=8):
    """Fallback: a few B=4096 training steps of the numpy oracle port."""
    m = oracle_model()
    _, coords, t, y = synth_dataset(2025, N_TRAIN)
    state = {}
    oracle_train_step(m, state, coords[:BATCH], t[:BATCH], y[:BATCH], 1)  # warm-up (BLAS threads, page faults)
    times = []
    t_end = time.perf_counter() + seconds
    s = 1
    while s <= max_steps and (time.perf_counter() < t_end or len(times) < 2):
        lo = (s * BATCH) % (N_TRAIN - BATCH)
        t0 = time.perf_counter()
        oracle_train_step(m, state, coords[lo:lo + BATCH], t[lo:lo + BATCH], y[lo:lo + BATCH], s + 1)
        times.append(time.perf_counter() - t0)
        s += 1
    per = float(np.median(times))
    # prediction sample: forward-only over 32768 points
    n_p = 32768
    pc = np.random.default_rng(1).random((n_p, 2)).astype(np.float32)
    pt = np.random.default_rng(2).random((n_p, 1)).astype(np.float32)
    from oracle import stdadk_oracle as orc
    t0 = time.perf_counter()
    orc.forward(m, None, pc, pt, dtype=np.float32)
    tp = time.perf_counter() - t0
    return {"value": BATCH / per, "unit": UNIT, "cores": os.cpu_count(), "kind": "port",
            "sample": f"{len(times)} oracle (numpy FP32, host BLAS threads) training steps of batch {BATCH}, median; "
                      f"predict sample {n_p} points", "ms_per_step": per * 1e3, "predict_points_per_s": n_p / tp}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    try:
        arm = ReferenceArm()
    except Exception as e:        # noqa: BLE001
        print(f"[bench] reference package unavailable ({e!r}); the reference arm times the oracle port", file=sys.stderr)
        return run_reference_port(args, max(1, min(args.steps, 100)))
    for w in range(max(1, min(args.warmup, 3))):
        arm.step(w)
    # K steps as asked, bounded by wall clock (a step is ~30 ms on 16 cores, ~10x that on a few): the arm stays within
    # minutes on any host; `steps` in the line is what was actually timed
    t0 = time.perf_counter()
    steps = 0
    while steps < max(1, args.steps) and (steps < 20 or time.perf_counter() - t0 < 120.0):
        arm.step(steps + 3)
        steps += 1
    dt = time.perf_counter() - t0
    val = steps * BATCH / dt
    cb = {"value": val, "unit": UNIT, "cores": arm.threads, "kind": "reference",
          "sample": f"{steps} training steps of batch {BATCH}: the reference's own STInterpMLP + MSELoss + clip_grad_norm_ + "
                    f"AdamW + ModelEMA (oracle/_ref, unmodified) on pre-batched CPU tensors, {arm.threads} threads",
          "predict_points_per_s": arm.predict_points_per_s()}
    emit({"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
          "warmup": args.warmup, "ms_per_step": dt / steps * 1e3, "higher_is_better": True, "scaling": "weak",
          "vs_baseline": None, "dtype": "f32", "data": "synthetic",
          "config": {"workload": WORKLOAD, "global_batch": BATCH, "l2": "n/a (CPU)", "cuda_graph": False,
                     "parallelism": "single", "precision": "fp32",
                     "note": "the reference's CPU PyTorch path on the host cores; one rank only (it has no multi-device path)"},
          "cpu_baseline": cb,
          "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})


def run_reference_port(args, steps):
    m = oracle_model()
    _, coords, t, y = synth_dataset(2025, N_TRAIN)
    state = {}
    for w in range(max(1, min(args.warmup, 2))):
        oracle_train_step(m, state, coords[:BATCH], t[:BATCH], y[:BATCH], w + 1)
    t0 = time.perf_counter()
    for s in range(steps):
        lo = (s * BATCH) % (N_TRAIN - BATCH)
        oracle_train_step(m, state, coords[lo:lo + BATCH], t[lo:lo + BATCH], y[lo:lo + BATCH], s + 3)
    dt = time.perf_counter() - t0
    val = steps * BATCH / dt
    cb = {"value": val, "unit": UNIT, "cores": os.cpu_count(), "kind": "port",
          "sample": f"{steps} oracle-port (numpy FP32, host BLAS threads) training steps of batch {BATCH}"}
    emit({"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
                      "steps": steps, "warmup": args.warmup, "ms_per_step": dt / steps * 1e3, "higher_is_better": True,
                      "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                      "config": {"workload": WORKLOAD, "note": "reference CPU path = oracle port on host cores; one "
                                 "rank only (the reference has no multi-device path)"},
                      "cpu_baseline": cb,
          "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})


# ------------------------------------------------------------------------------------------------ GPU arm
class ClockSampler:
    FIELDS = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown," \
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown," \
             "clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def measure_tf32_peak(dev, seconds=1.0):
    """Dense TF32 tensor-core throughput of this GPU measured the way MEASURED_PEAKS.json measures BF16: cuBLAS matmul
    8192^3 with TF32 inputs / FP32 accumulate, best of 10 (burst) and back to back for `seconds` (sustained)."""
    import torch
    n = 8192
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        a = torch.randn(n, n, device=dev)
        b = torch.randn(n, n, device=dev)
        c = torch.empty(n, n, device=dev)
        for _ in range(3):
            torch.matmul(a, b, out=c)
        torch.cuda.synchronize()
        best = 1e9
        for _ in range(10):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            torch.matmul(a, b, out=c)
            e1.record()
            torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        reps = max(10, int(seconds * 1e3 / best))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            torch.matmul(a, b, out=c)
        e1.record()
        torch.cuda.synchronize()
        sus = e0.elapsed_time(e1) / reps
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old
    fl = 2.0 * n ** 3
    del a, b, c
    return {"tf32_tflops": fl / (best * 1e-3) / 1e12, "tf32_tflops_sustained": fl / (sus * 1e-3) / 1e12,
            "how": f"torch.matmul fp32 with allow_tf32 (cuBLAS TF32) {n}^3: best of 10 and {reps} back to back"}


def short_kernel_name(name: str) -> str:
    """stdadk::layer_fwd_kernel<true, 4, 4, 1>(...) -> layer_fwd_kernel<true,4,4,1>"""
    import re
    m = re.search(r"stdadk::([A-Za-z0-9_]+)(<[^(]*>)?", name)
    if m:
        return m.group(1) + (m.group(2) or "").replace(" ", "")
    return name.split("(")[0][-60:]


def profile_kernels(fn, iters):
    """Per-kernel device time of `iters` calls of fn(i) from a CUPTI trace (torch.profiler): the kernels are timed where
    they run -- inside the replayed CUDA graph, back to back -- not with host-side event pairs around eager launches.
    Returns {short name: {"us": average per launch, "per_call": launches per call of fn}} or None if CUPTI is closed."""
    import torch
    try:
        from torch.profiler import profile, ProfilerActivity
        with profile(activities=[ProfilerActivity.CUDA, ProfilerActivity.CPU]) as prof:
            for i in range(iters):
                fn(i)
            torch.cuda.synchronize()
        out = {}
        for ev in prof.key_averages():
            dt = getattr(ev, "device_time_total", None)
            if dt is None:
                dt = getattr(ev, "cuda_time_total", 0.0)
            if dt <= 0 or getattr(ev, "device_type", None) is None:
                continue
            if "DeviceType.CUDA" not in str(ev.device_type):
                continue
            nm = short_kernel_name(ev.key)
            d = out.setdefault(nm, {"us_total": 0.0, "count": 0})
            d["us_total"] += float(dt)
            d["count"] += int(ev.count)
        return {k: {"us": v["us_total"] / max(v["count"], 1), "per_call": v["count"] / iters} for k, v in out.items()} or None
    except Exception as e:        # noqa: BLE001
        print(f"[bench] kernel trace unavailable: {e!r}", file=sys.stderr)
        return None


def dump_outputs(out_dir, tr):
    """Write what the last training step handed its caller as float32 .npy files under out_dir: the step's loss
    (`loss`), the model's state_dict after the step (`model.<key>`) and the EMA weights (`ema.<key>`).  The bench's
    inputs are seeded, so two builds run with the same arguments can be compared file by file.  The backward kernels
    sum gradients with float atomics in a run-dependent order and AdamW at lr 2e-2 amplifies those last bits, so two
    runs of one build differ per array by up to 5e-7 relative L2 after 4 steps, 6e-6 after 23 and 0.4 after 520
    (B200): compare builds at a small --steps."""
    grab = lambda: {k: np.ascontiguousarray(v.detach().cpu().numpy(), dtype=np.float32)
                    for k, v in tr.model.state_dict().items()}
    arrays = {"loss": tr.loss_last.cpu().numpy().astype(np.float32)}
    arrays.update({"model." + k: v for k, v in grab().items()})
    tr.flat.apply_shadow()          # EMA weights swapped into the parameters by value, then swapped back
    try:
        arrays.update({"ema." + k: v for k, v in grab().items()})
    finally:
        tr.flat.restore()
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    return sum(a.nbytes for a in arrays.values())


def run_ours(args):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    log = lambda m: print(f"[bench r{rank}] {m}", file=sys.stderr, flush=True)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        from datetime import timedelta
        dist.init_process_group("nccl", device_id=dev, timeout=timedelta(seconds=180))   # a hang fails fast
        dist.barrier()
    from stnf.models import STInterpMLP
    from stnf.dataio import ObservationTable
    from st_dadk_b200.trainer import Trainer
    from st_dadk_b200.predict import Predictor, shard_range
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    tc_peak = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops", 1590.0)))   # kernels inside a long step
    tc_peak_burst = float(peaks.get("bf16_tflops", tc_peak))                                 # a kernel timed alone
    peak_src = "measured (MEASURED_PEAKS.json)" if peaks else "fallback (B200_PROFILING.md)"

    torch.manual_seed(2025)                    # same initial weights on every rank
    model = STInterpMLP(k_spatial_centers=K_SPATIAL, k_temporal_centers=K_TEMPORAL, hidden_dims=HIDDEN, dropout=0.1,
                        layernorm=True, output_dim=1)
    sites, coords, t, y = synth_dataset(2025 + rank, N_TRAIN)     # weak scaling: each rank owns 80k samples
    host = ObservationTable(torch.from_numpy(coords), torch.from_numpy(t), torch.from_numpy(y)).pin()
    table = host.to(dev)
    bpe = (N_TRAIN + BATCH - 1) // BATCH
    tr = Trainer(model, dict(CFG, precision=args.precision), dev, batches_per_epoch=bpe, use_cuda_graph=not args.no_graph)
    perm = torch.randperm(N_TRAIN, generator=torch.Generator().manual_seed(7 + rank)).to(dev)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)   # 256 MB > 126 MB L2
    global_rows = BATCH * world
    n_off = (N_TRAIN - BATCH) // BATCH

    def one_step(i):
        tr.train_step(table, perm, (i % n_off) * BATCH, BATCH, global_rows)

    log("trainer built; warm-up")
    for i in range(max(args.warmup, 3)):
        one_step(i)
    torch.cuda.synchronize()
    log("warm-up done; timing")
    if world > 1:
        dist.barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    torch.cuda.synchronize()
    wall0 = time.perf_counter()
    for i in range(args.steps):
        flush.fill_(1.0)                        # L2 flush between timed iterations (outside the event pair)
        ev[i][0].record()
        one_step(args.warmup + i)
        ev[i][1].record()
    torch.cuda.synchronize()
    wall = time.perf_counter() - wall0
    if world > 1:
        dist.barrier()
    clocks = sampler.stop() if rank == 0 else None
    dev_ms = sum(a.elapsed_time(b) for a, b in ev)
    tms = torch.tensor([dev_ms], device=dev)
    if world > 1:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    dev_ms = float(tms.item())
    value = args.steps * BATCH * world / (dev_ms * 1e-3)
    final_loss = tr.pop_loss_sum()

    log(f"timed region done: {dev_ms / args.steps:.4f} ms/step")
    if args.dump_outputs and rank == 0:          # data-parallel replicas hold identical weights
        log(f"last step's outputs: {dump_outputs(args.dump_outputs, tr)} bytes written to {args.dump_outputs}")
    # ---- end-to-end through the host-buffer API: per step H2D of the batch from pinned memory + D2H of the loss
    hb = 3 * 4 * BATCH + 4 * BATCH                 # coords (8 B) + t (4 B) + y (4 B) per sample
    # (lagged read-back: every step's batch is copied H2D and every step's loss read D2H inside the timed region; the
    #  host reads step i's loss while step i+1 runs instead of idling the GPU on a per-step synchronisation)
    for i in range(4):
        tr.train_step_host(host, (i % n_off) * BATCH, BATCH, global_rows, lagged=True)
    tr.flush_host_loss()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    e2e_losses = []
    for i in range(args.steps):
        e2e_losses.append(tr.train_step_host(host, ((i + 5) % n_off) * BATCH, BATCH, global_rows, lagged=True))
    e2e_losses.append(tr.flush_host_loss())
    torch.cuda.synchronize()
    e2e_t = torch.tensor([time.perf_counter() - t0], device=dev)
    if world > 1:
        dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
    e2e_lagged = args.steps * BATCH * world / float(e2e_t.item())
    # the same with upstream's semantics: the host waits for EVERY step's loss before it issues the next batch
    # (loss.item() per step, train_st_interp.py:721) -- this is the headline e2e number
    n_sync = min(args.steps, 400)
    for i in range(3):
        tr.train_step_host(host, (i % n_off) * BATCH, BATCH, global_rows, lagged=False)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for i in range(n_sync):
        e2e_losses.append(tr.train_step_host(host, ((i + 9) % n_off) * BATCH, BATCH, global_rows, lagged=False))
    torch.cuda.synchronize()
    e2e_t = torch.tensor([time.perf_counter() - t0], device=dev)
    if world > 1:
        dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
    e2e_val = n_sync * BATCH * world / float(e2e_t.item())

    log("e2e done; prediction")
    # ---- dense prediction: T x S = 1M points (space-time field), sharded by point, no collective
    model.eval()
    pr = Predictor(model, static_weights=True)      # serving: weights are fixed between prediction calls
    sites_d = torch.from_numpy(sites).to(dev)
    n_pred = S_SITES * T_STEPS
    # several GPUs: the field is sharded by SITE (each rank: its sites at every time step), so that the per-site work
    # of the field kernel is done once, as on one GPU; at world 1 the two shardings coincide
    field_fn = (lambda: pr.space_time_field_by_sites(sites_d, T_STEPS, rank, world)) if world > 1 else \
        (lambda: pr.space_time_field(sites_d, T_STEPS, rank, world))
    grid_fn = pr.grid_by_sites if world > 1 else pr.grid
    for _ in range(2):
        field_fn()
    torch.cuda.synchronize()
    reps = 7
    pe = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for i in range(reps):
        flush.fill_(1.0)
        pe[i][0].record()
        out, _ = field_fn()
        pe[i][1].record()
    torch.cuda.synchronize()
    # median of the repetitions on each rank (a launch is 0.2-1 ms: one host hiccup would dominate a mean), max over ranks
    pms = torch.tensor([sorted(a.elapsed_time(b) for a, b in pe)[reps // 2]], device=dev)
    if world > 1:
        dist.all_reduce(pms, op=dist.ReduceOp.MAX)
    pred_pps = n_pred / (float(pms.item()) * 1e-3)
    # 10M-point dense grid (BASELINE configs[2]) generated on the device, sharded by point
    g10 = (1000, 1000, 10)
    grid_fn(*g10, rank, world)
    torch.cuda.synchronize()
    ge_ = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(3)]
    for a, b in ge_:
        flush.fill_(1.0)
        a.record()
        grid_fn(*g10, rank, world)
        b.record()
    torch.cuda.synchronize()
    gms = torch.tensor([sorted(a.elapsed_time(b) for a, b in ge_)[1]], device=dev)
    if world > 1:
        dist.all_reduce(gms, op=dist.ReduceOp.MAX)
    grid_pps = 10_000_000 / (float(gms.item()) * 1e-3)
    # e2e prediction: result copied back to pinned host memory
    rb, re_ = shard_range(n_pred, rank, world)          # the host-delivery path shards the (t, s) rows
    hout = torch.empty(re_ - rb, model.output_dim, dtype=torch.float32).pin_memory()
    pr.space_time_field(sites_d, T_STEPS, rank, world, host_out=hout)       # warm (copy stream, events)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out, _ = pr.space_time_field(sites_d, T_STEPS, rank, world, host_out=hout)   # D2H of each piece overlaps the next
    torch.cuda.synchronize()
    pred_e2e = torch.tensor([time.perf_counter() - t0], device=dev)
    if world > 1:
        dist.all_reduce(pred_e2e, op=dist.ReduceOp.MAX)
    pred_e2e_pps = n_pred / float(pred_e2e.item())

    # ---- rooflines: kernels chosen BY NAME, timed where they run
    log("prediction done; rooflines")
    traffic = {}
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as fh:
            traffic = json.load(fh)      # DRAM bytes per launch from the committed ncu captures (not measured live)
    except OSError:
        pass
    # (a) the kernels of the timed training step, from a CUPTI trace of graph REPLAYS (no eager event pairs)
    ktrace = profile_kernels(lambda i: one_step(i), 20)
    # (b) fused basis + Linear1 + LayerNorm/ReLU forward in the throughput regime: 1M explicit points per launch
    #     (12 B read + 1024 B written per point; the 1 GB it writes is 8x the L2, so no flush is needed between launches)
    n_roof = 1 << 20
    g = torch.Generator().manual_seed(5)
    rc, rt = torch.rand(n_roof, 2, generator=g).to(dev), torch.rand(n_roof, generator=g).to(dev)
    l1 = pr.profile_block1(rc, rt, repeats=5)
    _, fus_generic = pr.profile_fused(1000, 1000, 1)
    fus = pr.profile_field(*g10) or fus_generic       # the kernel dense-grid prediction actually runs
    # the TF32 peak LAST: a second of back-to-back 8192^3 cuBLAS GEMMs leaves some boxes power-limited for a while, and the
    # kernels measured right after it came out 25-40 % slower than in a fresh process (block 1: 1.13 vs 0.79 ms)
    tf32 = measure_tf32_peak(dev) if rank == 0 else None
    roof = roof_gemm = None
    if rank == 0:
        ach = l1["bytes"] / (l1["ms"] * 1e-3) / 1e9
        in_step = None
        if ktrace:
            k1 = [k for k in ktrace if k.startswith("layer_fwd_kernel<true")]
            if k1:
                us = ktrace[k1[0]]["us"]
                in_step = {"kernel": k1[0], "launch_us": us, "rows": BATCH,
                           "GB/s": BATCH * l1["bytes_per_row"] / (us * 1e-6) / 1e9,
                           "note": "the same kernel inside the timed step: 32 tiles on 148 SMs, latency-bound"}
        roof = {"kernel": "layer_fwd_kernel<BASIS> (basis generated in the operand + Linear1 on tcgen05 + LayerNorm/ReLU epilogue)",
                "bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak,
                "traffic": traffic.get("predict", {}).get("layer_fwd[0]"), "traffic_source": traffic.get("source"),
                "rows_per_launch": n_roof, "algorithmic_bytes_per_row": l1["bytes_per_row"],
                "algorithmic_bytes_per_launch": l1["bytes"], "launch_ms": l1["ms"], "peak_source": peak_src,
                "timing": "a CUDA event pair around each of 5 back-to-back launches on the launching stream, after warm-up; "
                          "median", "launch_ms_all": l1.get("ms_all"),
                "in_step": in_step}
        if fus is not None:
            tfl = fus["flops"] / (fus["ms"] * 1e-3) / 1e12
            roof_gemm = {"kernel": f"{fus.get('kernel', 'predict_fused_kernel')} (whole network, {fus['points']} points per launch)",
                         "bound": "tensor", "achieved": tfl, "peak": tf32["tf32_tflops"], "unit": "TFLOP/s",
                         "frac": tfl / tf32["tf32_tflops"], "peak_source": "measured in this run: " + tf32["how"] + " (burst)",
                         "frac_of_sustained_tf32": tfl / tf32["tf32_tflops_sustained"],
                         "executed_flops_per_launch": fus["flops"], "dense_equivalent_flops_per_launch": fus.get("dense_flops"),
                         "traffic": traffic.get("predict", {}).get(
                             "predict_field" if fus.get("kernel") == "predict_field_kernel" else "predict_fused"),
                         "algorithmic_bytes_per_launch": fus["bytes"], "launch_ms": fus["ms"],
                         "tensor_pipe_pct_ncu": traffic.get("tensor_pipe_pct", {}).get(fus.get("kernel")),
                         "points_per_s": fus["points"] / (fus["ms"] * 1e-3),
                         "generic_kernel": None if fus_generic is None else {
                             "kernel": "predict_fused_kernel (arbitrary points)", "points": fus_generic["points"],
                             "launch_ms": fus_generic["ms"],
                             "TFLOP/s": fus_generic["flops"] / (fus_generic["ms"] * 1e-3) / 1e12}}
    x3_ms = None
    if rank == 0 and world == 1 and args.precision == "tf32":
        # the FP32-faithful parity mode (three tensor-core passes per GEMM) on the same step, for the record
        torch.manual_seed(2025)
        m3 = STInterpMLP(k_spatial_centers=K_SPATIAL, k_temporal_centers=K_TEMPORAL, hidden_dims=HIDDEN, dropout=0.1,
                         layernorm=True, output_dim=1)
        t3 = Trainer(m3, dict(CFG, precision="tf32x3"), dev, batches_per_epoch=bpe, use_cuda_graph=not args.no_graph)
        for i in range(5):
            t3.train_step(table, perm, (i % n_off) * BATCH, BATCH, global_rows)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(50):
            t3.train_step(table, perm, ((i + 5) % n_off) * BATCH, BATCH, global_rows)
        e1.record()
        torch.cuda.synchronize()
        x3_ms = e0.elapsed_time(e1) / 50
        del t3, m3
    if rank == 0:
        cb = cpu_baseline() if world == 1 else None
        step_us = {k: round(v["us"] * v["per_call"], 2) for k, v in (ktrace or {}).items()}
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": dev_ms / args.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "tf32" if args.precision == "tf32" else "tf32x3",
                "data": "synthetic",
                "config": {"workload": WORKLOAD, "global_batch": global_rows, "l2": "flushed between timed steps "
                           "(256 MB write)", "cuda_graph": not args.no_graph,
                           "parallelism": f"dp{world}" if world > 1 else "single", "precision": args.precision},
                "clocks": clocks, "gpu_launches": tr.launches_per_step * args.steps,
                "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": hb, "d2h_bytes_per_step": 4,
                        "readback": "every step's loss read by the host before the next batch is issued (upstream's "
                                    "loss.item() per step)", "steps": n_sync,
                        "lagged_value": e2e_lagged, "lagged_readback": "loss read one step behind (double-buffered staging)",
                        "last_loss": e2e_losses[-1]},
                "predict_points_per_s": pred_pps, "grid10M_points_per_s": grid_pps, "predict_e2e_points_per_s": pred_e2e_pps,
                "predict": {"metric": "predict_points_per_s", "value": pred_pps, "unit": "points/s",
                            "workload": f"T x S = {n_pred} space-time points, sharded by point over {world} GPU(s)"
                                        + (" (by site: every rank takes its sites at all time steps)" if world > 1 else ""),
                            "timing": "CUDA events per launch, L2 flushed before each, median of 7 (field) / 3 (10M grid) "
                                      "repetitions per rank, max over ranks",
                            "e2e_value": pred_e2e_pps, "d2h_bytes": int(out.numel() * 4),
                            "grid10M_points_per_s": grid_pps},
                "roofline": roof, "roofline_gemm": roof_gemm, "tf32_peak": tf32,
                "kernel_us_per_step": step_us, "kernel_us_sum": round(sum(step_us.values()), 2),
                "tf32x3_ms_per_step": x3_ms,
                "cpu_baseline": cb, "mean_train_loss": final_loss / max(1, args.steps + max(args.warmup, 3)),
                "wall_s_timed_region": wall}
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


_REAL_STDOUT = None


def _quiet_stdout():
    """Everything libraries print to fd 1 (NCCL's version banner, build logs) goes to stderr; the single JSON line is
    written to the real stdout by emit()."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)


def emit(obj):
    data = (json.dumps(obj) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    global BATCH, N_TRAIN, WORKLOAD
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=BATCH,
                    help="per-GPU batch (default 4096 = the BASELINE config; e.g. 65536 for the throughput regime: the "
                         "resident training set then grows to 4 batches per GPU)")
    ap.add_argument("--precision", default="tf32", choices=["tf32", "tf32x3"],
                    help="tensor-core precision of the measured arm: tf32 = throughput mode, tf32x3 = FP32-faithful parity mode")
    ap.add_argument("--config", type=int, default=2, choices=[1, 2, 3, 4, 5],
                    help="BASELINE.json config (1-based; 2 = the headline workload, the default)")
    ap.add_argument("--no-graph", action="store_true",
                    help="launch every kernel eagerly (for ncu: kernel replay cannot run inside stream capture)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last step's loss, weights and EMA weights to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.config != 2):
        ap.error("--dump-outputs applies to the default workload (--impl ours, --config 2)")
    if args.batch != BATCH:
        WORKLOAD = WORKLOAD.replace(f"batch {BATCH}/GPU", f"batch {args.batch}/GPU").replace(
            "80k train samples", f"{max(N_TRAIN, 4 * args.batch)} train samples")
        BATCH, N_TRAIN = args.batch, max(N_TRAIN, 4 * args.batch)
    _quiet_stdout()
    if args.impl == "reference":
        run_reference(args)
    elif args.config != 2:
        import bench_extra
        bench_extra.run_config(args.config, args, emit)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
