"""Training step time and prediction rate of networks with hidden blocks wider than 256 units, against the same model
in plain PyTorch on the same GPU.

  python tools/bench_wide.py [--steps 30] [--warmup 5] [--out results.jsonl]

For hidden [512, 512, 256] and [384, 384, 192] (the bench's basis, dropout 0.1, LayerNorm, MSE) it prints one JSON line
per (network, batch) with
  * ms_per_step: Trainer.train_step (forward, backward, clip + AdamW + EMA, CUDA graph), CUDA events over `steps` steps;
  * torch_ms_per_step: the same model as nn.Modules (basis evaluated with torch ops, TF32 matmuls), one step of
    forward, backward and torch.optim.AdamW, CUDA events over `steps` steps;
  * predict_points_per_s: Predictor.points on 1,048,576 random points, median of 5 (the per-block chain: the
    whole-network kernel takes blocks of at most 256);
and the card's name and power limit, read in the same process.  Nothing is written to the tree unless --out names a file.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from bench import CFG, K_SPATIAL, K_TEMPORAL, synth_dataset  # noqa: E402

NETS = ([512, 512, 256], [384, 384, 192])
BATCHES = (4096, 65536)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def timed(fn, steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def trainer_ms(hidden, batch, steps, warmup, dev):
    from stnf.dataio import ObservationTable
    from stnf.models import STInterpMLP
    from st_dadk_b200.trainer import Trainer
    n = 4 * batch
    torch.manual_seed(0)
    model = STInterpMLP(k_spatial_centers=K_SPATIAL, k_temporal_centers=K_TEMPORAL, hidden_dims=hidden, dropout=0.1,
                        layernorm=True, output_dim=1)
    _, coords, t, y = synth_dataset(2025, n)
    table = ObservationTable(torch.from_numpy(coords), torch.from_numpy(t), torch.from_numpy(y)).to(dev)
    tr = Trainer(model, dict(CFG, hidden_dims=hidden, precision="tf32"), dev, batches_per_epoch=n // batch,
                 use_cuda_graph=True)
    perm = torch.randperm(n, generator=torch.Generator().manual_seed(7)).to(dev)

    def step(i):
        tr.train_step(table, perm, (i % 4) * batch, batch, batch)
    for i in range(warmup):
        step(i)
    torch.cuda.synchronize()
    return timed(step, steps), model


def predict_pps(model, dev, n=1 << 20, reps=5):
    from st_dadk_b200.predict import Predictor
    model.eval()
    pr = Predictor(model)
    g = torch.Generator().manual_seed(3)
    c, t = torch.rand(n, 2, generator=g).to(dev), torch.rand(n, generator=g).to(dev)
    pr.points(c, t)
    torch.cuda.synchronize()
    ms = sorted(timed(lambda i: pr.points(c, t), 1) for _ in range(reps))
    return n / (ms[reps // 2] * 1e-3), bool(pr.ex.fused_supported())


class TorchNet(torch.nn.Module):
    """The same network in nn.Modules: Wendland spatial and Gaussian temporal basis from torch ops, then
    Linear -> LayerNorm -> ReLU -> Dropout blocks and the head."""

    def __init__(self, hidden, dev):
        super().__init__()
        from st_dadk_b200.knot_init import place_knots, temporal_knots
        c, b = place_knots("uniform", K_SPATIAL, None)
        tc, tb = temporal_knots(K_TEMPORAL)
        self.register_buffer("c", c.float())
        self.register_buffer("th", b.float())
        self.register_buffer("tc", tc.float())
        self.register_buffer("tb", tb.float())
        dims = [c.shape[0] + tc.shape[0], *hidden]
        layers = []
        for i in range(len(hidden)):
            layers += [torch.nn.Linear(dims[i], dims[i + 1]), torch.nn.LayerNorm(dims[i + 1]), torch.nn.ReLU(),
                       torch.nn.Dropout(0.1)]
        layers.append(torch.nn.Linear(dims[-1], 1))
        self.mlp = torch.nn.Sequential(*layers)
        self.to(dev)

    def forward(self, coords, t):
        r = torch.cdist(coords, self.c) / self.th
        u = torch.clamp(1.0 - r, min=0.0)
        phi = u ** 6 * (35.0 / 3.0 * r * r + 6.0 * r + 1.0)
        psi = torch.exp(-0.5 * ((t[:, None] - self.tc) / self.tb) ** 2)
        return self.mlp(torch.cat([phi, psi], 1))


def torch_ms(hidden, batch, steps, warmup, dev):
    torch.backends.cuda.matmul.allow_tf32 = True
    torch.backends.cudnn.allow_tf32 = True
    torch.manual_seed(0)
    net = TorchNet(hidden, dev)
    opt = torch.optim.AdamW(net.parameters(), lr=1e-3, weight_decay=5e-4)
    _, coords, t, y = synth_dataset(2025, batch)
    c, tt, yy = torch.from_numpy(coords).to(dev), torch.from_numpy(t).to(dev), torch.from_numpy(y).to(dev)

    def step(i):
        opt.zero_grad(set_to_none=True)
        loss = torch.nn.functional.mse_loss(net(c, tt)[:, 0], yy)
        loss.backward()
        opt.step()
    for i in range(warmup):
        step(i)
    torch.cuda.synchronize()
    return timed(step, steps)


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_wide: no CUDA device (the numbers are GPU timings)")
    dev = torch.device("cuda")
    gpu = card()
    lines = []
    for hidden in NETS:
        for batch in BATCHES:
            ms, model = trainer_ms(hidden, batch, args.steps, args.warmup, dev)
            rec = {"hidden": hidden, "batch": batch, "ms_per_step": ms, "train_samples_per_s": batch / (ms * 1e-3),
                   "torch_ms_per_step": torch_ms(hidden, batch, args.steps, args.warmup, dev), "gpu": gpu}
            if batch == BATCHES[0]:
                rec["predict_points_per_s"], rec["fused_predict"] = predict_pps(model, dev)
            del model
            torch.cuda.empty_cache()
            lines.append(rec)
            print(json.dumps(rec), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.writelines(json.dumps(r) + "\n" for r in lines)


if __name__ == "__main__":
    main()
