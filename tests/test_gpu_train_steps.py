"""Trainer.train_step, step by step, against the oracle at matched weights.

Every step k of a multi-step run is checked on its own.  Before the step the test snapshots the weights and the flat
p / m / v / shadow buffers; the FP64 oracle then runs the step from that snapshot, with the dropout masks of step k
(k counted by the test) keyed by the row within the batch.  After the step:
  * the gradient the fused tail used is recovered from the moments, g_c = (m' - b1 m) / (1 - b1), and divided by the
    clip factor formed from the tail's own group norms; it must match the oracle's gradient of every parameter, and
    the group norms the oracle's;
  * the loss the tail recorded must match the oracle's loss;
  * v', p' and shadow' must follow AdamW + EMA from the snapshot, with bias correction at step k + 1 and the learning
    rate of each group written out here from the upstream schedule (warm-up written after the step; the basis group
    frozen, then unfrozen at 0.1x and ramped), not read back from the trainer;
  * the device step counter must read k before the step and k + 1 after it, eager or replayed.
Comparing at matched weights keeps the trajectory's drift (TF32, Adam on near-zero gradients) out of the comparison,
so the bounds are those of the single-step tests (test_gpu_regimes).  What this reaches that single steps do not: the
dropout key read from the device step counter (which the previous step's tail advances, and which the one-wave
backward reads before its programmatic-launch wait), per-group hyper-parameters through the pinned ring, graphs of
two batch shapes and their recapture after a workspace eviction, and the delta head's cumsum ops inside the graph."""
from dataclasses import dataclass

import numpy as np
import pytest
import torch

from helpers import oracle_from_state, orc
from test_gpu_kernels import rel_err
from test_gpu_regimes import TF32_TOL, X3_TOL, chunked_oracle, regime_rows

pytestmark = pytest.mark.gpu
DEV = "cuda"

# the moments' constants as Trainer passes them to ops.adamw_ema_step (FP32 on the device)
B1, B2, EPS = np.float64(np.float32(0.9)), np.float64(np.float32(0.999)), 1e-8
OMB1, OMB2 = np.float64(np.float32(1) - np.float32(0.9)), np.float64(np.float32(1) - np.float32(0.999))
ULP = 2.0 ** -24
# A kept pre-activation this close to 0 (a few FP32 roundings of an O(1) LayerNorm output) may land on either side of
# the ReLU in the kernel: that one (row, unit) then moves its block's column sums by the row's share of the batch, up to
# ~1e-3 of the largest gradient at 4,096 rows (measured on a B200: case D step 0, a block-2 pre-activation at 4e-8 of
# zero, d W2 1.3e-3 from FP64 while every other tensor is within 3e-6).  tf32x3 steps with such a unit take this bound;
# at 4,096 rows most steps have one or two.
KINK, X3_KINK_GRAD = 1e-6, 3e-3


@dataclass
class Case:
    model: dict
    cfg: dict
    batches: list                   # per epoch: the batch sizes, in order; they cover the epoch's permutation
    graph: bool = True
    clip_engaged: bool = True       # grad_clip = 0.8x (engaged) or 2x (not engaged) the oracle's step-0 norm
    evict: bool = False             # evaluate between the epochs until the training workspaces are evicted
    control_step: int = -1          # step whose oracle is also run with the masks of steps k - 1 and k + 1
    seed: int = 0
    taus: tuple = ()


def _cases():
    base = dict(lr=2e-3, weight_decay=1e-2, regression_type="mean", epochs=100)
    a = dict(model={}, cfg=dict(base, warmup_epochs=1), batches=[[4096, 4096, 4096, 2176]] * 2, seed=11)
    rows = regime_rows()
    mq3 = dict(base, regression_type="multi-quantile", quantile_levels=[0.1, 0.5, 0.9], non_crossing_weight=0.5,
               non_crossing_power=2, basis_lr_ratio=0.5, basis_unfreeze_epoch=1, basis_lr_rampup_epochs=2)
    mq5 = dict(base, regression_type="multi-quantile", quantile_levels=[0.05, 0.25, 0.5, 0.75, 0.95],
               use_delta_reparameterization=True)
    return {
        "A-tf32x3": Case(**a, control_step=1),
        "A-tf32": Case(**dict(a, cfg=dict(a["cfg"], precision="tf32"))),
        "A-eager": Case(**a, graph=False),
        "A-evict": Case(**a, evict=True),
        "B": Case(model={}, cfg=dict(base, precision="tf32"), batches=[[rows["R128x"]] * 3 + [rows["R128r"]] * 3],
                  seed=12),
        "C": Case(model=dict(spatial_learnable=True, output_dim=3), cfg=mq3, batches=[[4096, 4096]] * 3, seed=13,
                  clip_engaged=False, taus=(0.1, 0.5, 0.9)),
        "D": Case(model=dict(output_dim=5, use_delta_reparameterization=True), cfg=mq5, batches=[[4096] * 3], seed=14,
                  clip_engaged=False, taus=(0.05, 0.25, 0.5, 0.75, 0.95)),
    }


CASE_IDS = ["A-tf32x3", "A-tf32", "A-eager", "A-evict", "B", "C", "D"]


def _table(n, seed):
    rng = np.random.default_rng(seed)
    c = rng.random((n, 2)).astype(np.float32)
    t = (rng.integers(0, 100, n) / 99.0).astype(np.float32)
    y = (np.sin(6 * c[:, 0]) * np.cos(5 * c[:, 1]) + t + 0.1 * rng.standard_normal(n)).astype(np.float32)
    return c, t, y


def _lr_schedule(cs, bpe):
    """Learning rate of each group at every step, from the upstream rules (train_st_interp.py:582-602, :714-718):
    warm-up is written AFTER a step, so step 0 runs at the base lr and step k <= W at base * k / W; the basis group is
    at lr 0 before basis_unfreeze_epoch, at 0.1 x its target in that epoch, then ramps by 0.9 / rampup per epoch."""
    c = cs.cfg
    base, W = c["lr"], c.get("warmup_epochs", 0) * bpe
    out, k = [], 0
    for e, sizes in enumerate(cs.batches):
        for _ in sizes:
            mlp = base * (k / W) if 1 <= k <= W else base
            if "basis_unfreeze_epoch" in c:
                u, r, target = c["basis_unfreeze_epoch"], c["basis_lr_rampup_epochs"], base * c["basis_lr_ratio"]
                basis = 0.0 if e < u else target * min(0.1 + 0.9 * (e - u) / r, 0.1 + 0.9 * (r - 1) / r)
                out.append((mlp, basis))
            else:
                out.append((mlp,))
            k += 1
    return out


def _oracle(model, state, cs, data, idx, seed, step, rnd=None):
    """(yhat, loss, gradients) of the oracle at weights `state` on rows `idx`, dropout masks of `seed` and `step`."""
    c, t, y = data
    m = oracle_from_state(state, dropout=model._dropout_p)
    mq = cs.cfg["regression_type"] == "multi-quantile"
    ncw = 0.0 if cs.cfg.get("use_delta_reparameterization") else cs.cfg.get("non_crossing_weight", 0.0)
    return chunked_oracle(m, None, c[idx], t[idx, None], y[idx], "pinball" if mq else "mse", cs.taus or None, ncw,
                          cs.cfg.get("non_crossing_power", 1), key_offset=0,
                          knot_grads="spatial_basis.log_bandwidths" in state, rnd=rnd, seed=seed, step=step)


def _kinks(model, state, data, idx, seed, step):
    """Kept pre-activations of the step within KINK of the ReLU's kink, from an FP64 forward of the oracle."""
    c, t, _ = data
    m = oracle_from_state(state, dropout=model._dropout_p)
    masks = [orc.dropout_keep_mask(len(idx), w.shape[0], m.dropout, seed, step, l)
             for l, w in enumerate(m.weights[:len(m.ln_gamma)])]
    _, cache = orc.forward(m, None, c[idx], t[idx, None], train=True, keep_masks=masks, return_cache=True)
    n = 0
    for l, rec in enumerate(cache["layers"]):
        pre = rec["xh"] * m.ln_gamma[l] + m.ln_beta[l] if m.ln_gamma[l] is not None else rec["z"]
        n += int(np.sum((np.abs(pre) < KINK) & rec.get("keep", True)))
    return n


def _by_name(model, g):
    """Oracle gradients keyed by the model's parameter names."""
    names = {id(mod): n for n, mod in model.named_modules()}
    out = {}
    for l, (lin, ln) in enumerate(model.hidden_blocks()):
        out[names[id(lin)] + ".weight"], out[names[id(lin)] + ".bias"] = g["weights"][l], g["biases"][l]
        if ln is not None:
            out[names[id(ln)] + ".weight"], out[names[id(ln)] + ".bias"] = g["ln_gamma"][l], g["ln_beta"][l]
    if model.delta_params is not None:
        for j, d in enumerate(g["delta"]):
            out[f"delta_params.{j}"] = d
    else:
        head = names[id(model.mlp[-1])]
        out[head + ".weight"], out[head + ".bias"] = g["weights"][-1], g["biases"][-1]
    if model.spatial_basis.learnable:
        out["spatial_basis.centers"], out["spatial_basis.log_bandwidths"] = g["centers"], g["log_bandwidths"]
    return out


def _split(model, flat64):
    """A flat FP64 array in the FlatState layout -> {parameter name: array of the parameter's (upstream) shape}; the
    Parameters are views into the flat buffer (weights stored transposed), so their strides give the layout."""
    src = torch.from_numpy(flat64)
    return {n: torch.as_strided(src, p.shape, p.stride(), p.storage_offset()).numpy()
            for n, p in model.named_parameters()}


def _grad_errors(kern, ref, tag):
    return {f"{n}/{tag}": rel_err(kern[n], ref[n]) for n in ref}


def _group_norms(ref, names_of_group):
    return [np.sqrt(sum(float(np.sum(np.asarray(ref[n], dtype=np.float64) ** 2)) for n in names))
            for names in names_of_group]


@pytest.mark.parametrize("name", CASE_IDS)
def test_train_steps_vs_oracle_at_matched_weights(name):
    """Every step of a Trainer run against the oracle from that step's snapshot (module docstring).  Cases:
      A   STInterpMLP defaults (297-256-256-128, LN, Wendland, dropout 0.1), MSE, 2 epochs of 3 x 4,096 + 2,176 rows,
          warm-up 1 epoch; tf32x3 and tf32, graphs of two shapes (the bench's step: 64-row tiles, programmatic-launch
          chain, keep bits and x^ before the wait, the fused tail with register-resident state).  A-tf32x3 also runs
          the oracle of step 1 (a replay) with the masks of steps 0 and 2: both must miss by 10x the bounds.
      A-eager  as A, tf32x3, no graphs: row_begin != 0, dropout still keyed by the row within the batch.
      A-evict  as A, tf32x3: between the epochs `evaluate` allocates four workspaces of new batch sizes, which evicts
          the training ones and drops the graphs; the recaptured steps must stay on the oracle.
      B   defaults, tf32, 3 steps of 12,345 rows (128-row tiles, x saved) and 3 of SAVE_X_MAX_ROWS + 1,000 (the
          recompute backward, keep bits after the wait).
      C   learnable knots, Q = 3 pinball with the quadratic non-crossing penalty (weight 0.5), tf32x3, 3 epochs of 2
          steps: the basis group (clip 0.1x) frozen in epoch 0 (centres and log-bandwidths bit-identical across its
          steps), then 0.1x its target lr, then 0.55x; knot gradients.
      D   delta head, Q = 5, tf32x3, 3 steps: delta gradients through the cumsum ops captured in the step graph; the
          scratch head gradient behind the parameters is left zero.
    Bounds: those of test_gpu_regimes (largest measured on a B200, 148 SMs, 1,000 W, in brackets).  tf32x3: gradients
    and group norms 1e-3 of FP64 (1.7e-4; group norms 8.3e-7), 3e-3 on a step with a unit at the ReLU kink (KINK: D
    step 0, 1.3e-3); loss 1e-5 (7.4e-7).  tf32: gradients 3e-3 of the TF32-emulating oracle (5.7e-4) and 2e-2 of FP64
    (5.0e-3); loss 1e-3 (4.9e-5).  Update: v', p', shadow' within a few FP32 roundings, the bias corrections' powf
    3e-4 of the step (at most 0.62 of these bounds).  Negative control: the masks of steps 0 and 2 miss step 1 by
    2.3e-4 / 2.7e-3 in the loss and 5.1e-2 / 4.4e-2 in the gradients.  The clip is engaged on 4 of A's 8 steps (from
    step 0) and on none of C's and D's."""
    from stnf.dataio import ObservationTable
    from stnf.models import STInterpMLP
    from st_dadk_b200.trainer import Trainer

    cs = _cases()[name]
    x3 = cs.cfg.get("precision", "tf32x3") == "tf32x3"
    cfg = dict(cs.cfg, precision="tf32x3" if x3 else "tf32")
    sizes = [b for ep in cs.batches for b in ep]
    bpe = len(cs.batches[0])
    n = sum(cs.batches[0])
    data = _table(n, cs.seed)
    perms = [np.random.default_rng(cs.seed * 100 + e).permutation(n) for e in range(len(cs.batches))]
    torch.manual_seed(cs.seed)
    model = STInterpMLP(**cs.model)
    seed = int(torch.initial_seed() & (2 ** 63 - 1))
    group_names = [[p for p, _ in model.named_parameters() if not p.startswith("spatial_basis.")],
                   [p for p, _ in model.named_parameters() if p.startswith("spatial_basis.")]]
    group_names = [g for g in group_names if g]
    # grad_clip from the oracle's step-0 norm of the mlp group: engaged at step 0, or not
    state0 = {k: v.detach().cpu().numpy().copy() for k, v in model.state_dict().items()}
    ref0 = _oracle(model, state0, cs, data, perms[0][:sizes[0]], seed, 0)
    n0 = _group_norms(_by_name(model, ref0[2]), group_names)[0]
    cfg["grad_clip"] = float((0.8 if cs.clip_engaged else 2.0) * n0)
    clips = [cfg["grad_clip"], 0.1 * cfg["grad_clip"]]
    lrs = _lr_schedule(cs, bpe)
    wd, d32 = cfg["weight_decay"], np.float32(1.0 - 1.0 / (10.0 * bpe))
    d, omd = np.float64(d32), np.float64(np.float32(1) - d32)

    tr = Trainer(model, cfg, DEV, batches_per_epoch=bpe, use_cuda_graph=cs.graph)
    assert tr.seed == seed
    fl = tr.flat
    table = ObservationTable(*(torch.from_numpy(a) for a in data)).to(DEV)
    bounds = X3_TOL if x3 else TF32_TOL
    worst = {}
    engaged = []
    k = 0
    for e, ep_sizes in enumerate(cs.batches):
        tr.begin_epoch(e)
        perm = torch.from_numpy(perms[e]).to(DEV)
        lo = 0
        for B in ep_sizes:
            idx = perms[e][lo:lo + B]
            torch.cuda.synchronize()
            assert int(tr.step_count.item()) == k, (k, int(tr.step_count.item()))
            before = {a: getattr(fl, a).double().cpu().numpy() for a in ("p", "m", "v", "shadow")}
            state = {key: v.detach().cpu().numpy().copy() for key, v in model.state_dict().items()}
            replay = cs.graph and any(key[0] == B for key in tr._graphs)
            tr.train_step(table, perm, lo, B)
            torch.cuda.synchronize()
            after = {a: getattr(fl, a).double().cpu().numpy() for a in ("p", "m", "v", "shadow")}
            assert int(tr.step_count.item()) == k + 1
            assert float(fl.g.abs().max()) == 0.0          # gradient, scratch head gradient and loss slot left zero
            sq = tr.sqnorms.double().cpu().numpy()
            loss = float(tr.loss_last.item())

            # ---- the oracle at this step's weights, masks of step k
            r64 = ref0 if k == 0 else _oracle(model, state, cs, data, idx, seed, k)
            refs = [("64", r64)]
            if not x3:
                refs.append(("emu", _oracle(model, state, cs, data, idx, seed, k, rnd=orc.tf32_round)))

            # ---- the gradient the tail used, unclipped with its own norms
            gc = (after["m"] - B1 * before["m"]) / OMB1
            norms = np.sqrt(sq)
            coef = [min(1.0, clips[gi] / (norms[gi] + 1e-6)) for gi in range(len(group_names))]
            cvec = np.empty_like(gc)
            lrvec = np.empty_like(gc)
            g_lo = 0
            for gi, g_hi in enumerate(fl.group_end):
                cvec[g_lo:g_hi], lrvec[g_lo:g_hi] = coef[gi], lrs[k][gi]
                g_lo = g_hi
            engaged.append(coef[0] < 1.0)
            kern = _split(model, gc / cvec)
            errs = {"loss": abs(loss - r64[1]) / abs(r64[1])}
            for tag, (_, _, gref) in refs:
                byname = _by_name(model, gref)
                errs.update(_grad_errors(kern, byname, tag))
                for gi, nref in enumerate(_group_norms(byname, group_names)):
                    errs[f"norm{gi}/{tag}"] = abs(norms[gi] - nref) / nref

            # ---- the update from the snapshot: v', p' (kernel m', v'), shadow' (kernel p')
            v_ref = B2 * before["v"] + OMB2 * gc * gc
            dg = 2 * ULP * (np.abs(after["m"]) + np.abs(before["m"])) / OMB1       # rounding of the recovered g_c
            v_tol = 4 * ULP * v_ref + 2 * OMB2 * np.abs(gc) * dg + 1e-37
            bc1, bc2 = 1.0 - B1 ** (k + 1), 1.0 - B2 ** (k + 1)
            upd = (lrvec / bc1) * after["m"] / (np.sqrt(after["v"]) / np.sqrt(bc2) + EPS)
            p_ref = before["p"] * (1.0 - lrvec * wd) - upd
            p_tol = 6 * ULP * np.abs(before["p"]) + 3e-4 * np.abs(upd)
            s_ref = d * before["shadow"] + omd * after["p"]
            s_tol = 6 * ULP * (np.abs(d * before["shadow"]) + np.abs(omd * after["p"])) + 1e-37
            upd_errs = {"v": float(np.max(np.abs(after["v"] - v_ref) / v_tol)),
                        "p": float(np.max(np.abs(after["p"] - p_ref) / np.maximum(p_tol, 1e-37))),
                        "shadow": float(np.max(np.abs(after["shadow"] - s_ref) / s_tol))}
            kinks = _kinks(model, state, data, idx, seed, k) if x3 else 0
            step_bounds = dict(bounds, grad64=X3_KINK_GRAD) if kinks else bounds
            bad, summary = [], {}
            for key, v in errs.items():
                kind = "loss" if key == "loss" else ("grad_emu" if key.endswith("/emu") else "grad64")
                what = key if key.startswith(("loss", "norm")) else f"grad/{key.split('/')[-1]}"
                summary[what] = max(summary.get(what, 0.0), v)
                if not v < step_bounds[kind]:
                    bad.append(f"{key}={v:.3e} (bound {step_bounds[kind]:g})")
            summary.update({f"{key}/bound": v for key, v in upd_errs.items()})
            for key, v in summary.items():
                worst[key] = max(worst.get(key, 0.0), v)
            kink_note = f", {kinks} unit(s) at the ReLU kink" if kinks else ""
            print(f"\n{name} step {k} ({B} rows, {'replay' if replay else 'eager or capture'}): lr {lrs[k]}, clip "
                  f"factor {[round(float(c), 4) for c in coef]}, loss {loss:.6f}{kink_note}:",
                  " ".join(f"{key}={v:.2e}" for key, v in summary.items()))
            bad += [f"{key}: {v:.2f} x its bound" for key, v in upd_errs.items() if not v <= 1.0]
            assert not bad, (name, k, bad)
            if len(lrs[k]) > 1 and lrs[k][1] == 0.0:        # frozen basis group: not a bit moves (no 0 * inf either)
                sl = slice(fl.group_end[0], fl.group_end[1])
                assert np.array_equal(after["p"][sl], before["p"][sl]) and np.all(np.isfinite(after["p"][sl]))
            if k == 0:
                assert engaged[0] == cs.clip_engaged, (coef, cfg["grad_clip"])

            # ---- negative control: the masks of the neighbouring steps must be seen
            if k == cs.control_step:
                assert replay
                for kk in (k - 1, k + 1):
                    _, lw, gw = _oracle(model, state, cs, data, idx, seed, kk)
                    le = abs(loss - lw) / abs(lw)
                    ge = max(_grad_errors(kern, _by_name(model, gw), "64").values())
                    print(f"  oracle with the masks of step {kk}: loss {le:.2e}, largest gradient error {ge:.2e}")
                    assert le >= 10 * step_bounds["loss"] and ge >= 10 * step_bounds["grad64"], (kk, le, ge)
            lo += B
            k += 1
        tr.end_epoch(e)
        if cs.evict and e + 1 < len(cs.batches):
            vc, vt, vy = _table(3000, cs.seed + 1)
            val = ObservationTable(torch.from_numpy(vc), torch.from_numpy(vt), torch.from_numpy(vy)).to(DEV)
            assert tr._graphs and len(tr.ex._ws) == 2
            tr.flat.apply_shadow()
            for rows in (700, 1100):               # 700 and 200, 1100 and 800: four new workspaces
                tr.evaluate(val, batch_rows=rows)
            tr.flat.restore()
            assert not tr._graphs and not set(tr.ex._ws) & set(ep_sizes), sorted(tr.ex._ws)
    print(f"\n{name} largest over {k} steps:", " ".join(f"{key}={v:.2e}" for key, v in worst.items()),
          f"clip engaged on {sum(engaged)} of {k} steps")
