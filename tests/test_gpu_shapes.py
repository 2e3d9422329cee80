"""Training and prediction at the network shapes the other step tests never build: one hidden block (block 1 carries
the head and the loss), widths that are not multiples of 32 or of 4, a one-unit block, four and five hidden blocks.

  id   hidden                LN   dropout  head / loss                                 what it reaches
  O1   (64,)                 yes  0.1      Q = 1 MSE                                   block 1 = basis + LN + head + loss;
                                                                                       layer_bwd<BASIS, HEAD>
  O2   (256,)                no   0        Q = 8 pinball, non-crossing (power 2),      widest head epilogue inside the
                                           triangular basis                            basis kernel
  O3   (100,)                yes  0.1      Q = 3 pinball, delta head, learnable knots  knotgrad_kernel fed by the head
                                                                                       block's dz; ragged 4th chunk
  R    (50, 33, 7)           yes  0.1      Q = 2 pinball                               widths not multiples of 4; one
                                                                                       valid column in a chunk; a block
                                                                                       narrower than one chunk
  U    (36, 1)               no   0.1      Q = 1 MSE                                   a one-unit block
  D4   (128, 96, 64, 32)     yes  0.1      Q = 5 pinball                               deepest net of the fused / field
                                                                                       kernels; dropout layer ids 0-3
  D5   (64, 48, 48, 40, 32)  yes  0.1      Q = 1 MSE                                   dropout layer id 4; the fused
                                                                                       kernels decline

All use the golden lattice (227 spatial + 70 temporal knots).  The step tests follow test_gpu_regimes exactly (points
gathered through a permutation, row_begin != 0, dropout keys crossing 2^32, the chunked FP64 oracle and the
TF32-emulating one)."""
from functools import lru_cache

import numpy as np
import pytest
import torch

from helpers import oracle_from_state, orc
from test_gpu_kernels import T, _default_oracle_model, _mods, rel_err, rel_l2, spec_from_oracle
from test_gpu_regimes import P_DROP, TF32_TOL, X3_TOL, Net, _grad_pairs, _rows, _template_args, oracle, regime_rows, \
    train_step
from test_gpu_train_steps import X3_KINK_GRAD, Case, run_case

gpu = pytest.mark.gpu

# name: (hidden, layernorm, dropout, Q, loss, taus, non-crossing weight, basis, delta head, learnable knots)
SHAPES = {
    "O1": ((64,), True, P_DROP, 1, "mse", None, 0.0, "wendland", False, False),
    "O2": ((256,), False, 0.0, 8, "pinball", tuple(np.linspace(0.05, 0.95, 8)), 0.5, "triangular", False, False),
    "O3": ((100,), True, P_DROP, 3, "pinball", (0.1, 0.5, 0.9), 0.0, "wendland", True, True),
    "R": ((50, 33, 7), True, P_DROP, 2, "pinball", (0.3, 0.7), 0.0, "wendland", False, False),
    "U": ((36, 1), False, P_DROP, 1, "mse", None, 0.0, "wendland", False, False),
    "D4": ((128, 96, 64, 32), True, P_DROP, 5, "pinball", (0.05, 0.25, 0.5, 0.75, 0.95), 0.0, "wendland", False, False),
    "D5": ((64, 48, 48, 40, 32), True, P_DROP, 1, "mse", None, 0.0, "wendland", False, False),
}


@lru_cache(maxsize=None)
def shape_net(name):
    """The Net of SHAPES[name], weights drawn like _default_oracle_model (Linear init, perturbed LayerNorm)."""
    hidden, ln, p, q, loss, taus, ncw, fn, delta, learnable = SHAPES[name]
    m = _default_oracle_model(300 + list(SHAPES).index(name), q=q, fn=fn, hidden=hidden)
    m.dropout = p
    if not ln:
        m.ln_gamma = [None] * len(hidden)
        m.ln_beta = [None] * len(hidden)
    if name == "U":
        m.biases[1] = np.float32([0.1])        # keeps the one unit on: an idle unit would train nothing upstream
    if delta:
        # beta_k = sum_{l <= k} delta_l; delta_0 is the first head row, the increments keep the quantiles apart
        W, b = m.weights.pop(), m.biases.pop()
        rng = np.random.default_rng(77)
        d0 = np.concatenate([b[:1], W[0]]).astype(np.float32)
        m.delta = [d0] + [(0.05 + 0.02 * rng.standard_normal(W.shape[1] + 1)).astype(np.float32) for _ in range(q - 1)]
    return Net(m, loss, taus, nc_weight=ncw, learnable=learnable)


# ---------------------------------------------------------------------------------------------------- one step
# (net, precision, kind of error): bound, with the largest value measured on a B200 (148 SMs) and its cause.
SHAPE_EXCEPTIONS = {
    # Q = 2 pinball on a 7-unit last block: few terms average the TF32 rounding of yhat.  Measured 2.7e-3 (R64) of the
    # largest FP64 element, while yhat is 3.3e-5 (relative L2) from the TF32-emulating oracle and every gradient 2.4e-5.
    ("R", "tf32", "yhat64"): 4e-3,
    # Five blocks chain five TF32 roundings: yhat 1.8e-3 of FP64 (9.9e-5 of the emulation), gradients 2.1e-2 (R64,
    # d W0) where the emulation is within 6.7e-5.  test_shapes_the_fused_kernel_does_not_take_fall_back_to_block_kernels
    # measures the same depth at 1.1e-3.
    ("D5", "tf32", "yhat64"): 3e-3,
    ("D5", "tf32", "grad64"): 4e-2,
    # Every batch has kept pre-activations within 1e-5 of the ReLU kink (19 at 12,345 rows, FP64 forward).  The kernel's
    # FP32 sums and the emulation's FP64 sums can put one on opposite sides; the flipped (row, unit) then moves every
    # upstream column sum by that row's share, and five blocks of cancelling sums carry it to block 1.  Measured 1.0e-2
    # (R128x, d W0; d W4, below the flip, 3.0e-5) and 1.6e-3 (R128r); at R64 no unit flipped (6.7e-5).
    ("D5", "tf32", "grad_emu"): 2e-2,
    # The same flip against FP64 in tf32x3: d W0..d W3 1.1e-3 at R128r while d W4 is 1.2e-6 (test_gpu_train_steps.KINK).
    ("D5", "tf32x3", "grad64"): X3_KINK_GRAD,
}

STEP_CASES = ([(s, r, "tf32") for s in SHAPES for r in ("R64", "R128x", "R128r")]
              + [(s, r, "tf32x3") for s in ("O1", "R", "D5", "O3") for r in ("R128x", "R128r")]
              + [("O1", "R128r-feat", "tf32")])


@gpu
@pytest.mark.parametrize("name,regime,precision", STEP_CASES, ids=["-".join(c) for c in STEP_CASES])
def test_shape_training_step_vs_oracle(name, regime, precision):
    """yhat, loss and every gradient of one gathered training step against the chunked FP64 oracle and, in TF32 mode,
    the TF32-emulating oracle, with the bounds of test_gpu_regimes.test_training_step_vs_oracle (TF32_TOL / X3_TOL).
    Delta-head gradients are compared as the cumulative sum of [d head_b | d head_w] (d delta_l = sum_{k >= l} d beta_k).
    Where a reference gradient is identically zero (every unit upstream of a width-1 LayerNorm, a head column behind a
    ReLU that is never on) a relative error means nothing: such a gradient must be at most 1e-6 of max |d head_w|.
    Largest measured on a B200 outside SHAPE_EXCEPTIONS: TF32 yhat 9.6e-4 of FP64 (D4) and 5.4e-5 of the emulation,
    loss 2.7e-5 (R), gradients 6.6e-4 of the emulation (D4, d W1 at R64) and 3.4e-3 of FP64 (R, d W1 at R64), knot
    gradients 1.3e-3 (O3); tf32x3 yhat 2.0e-6, loss 1.0e-6, gradients 1.1e-4 (R, d W1 at R128r)."""
    n = _rows(regime)
    nt = shape_net(name)
    x3 = precision == "tf32x3"
    (y64, l64, g64), (yemu, lemu, gemu) = oracle(nt, n, regime)
    ex, yhat, loss, grads = train_step(nt, n, regime, precision)
    assert np.isfinite(yhat).all()
    errs = {"yhat64": rel_err(yhat, y64), "loss": abs(loss - l64) / abs(l64)}
    if not x3:
        errs["yhat_emu"] = rel_l2(yhat, yemu)
    scale = float(np.abs(grads["head_w"]).max())
    zero = []
    refs = [("64", g64)] + ([] if x3 else [("emu", gemu)])
    for tag, ref in refs:
        for gname, g, r in _grad_pairs(grads, ref, nt):
            if not np.any(r):
                zero.append(f"{gname}/{tag}")
                assert np.abs(g).max() <= 1e-6 * scale, (gname, tag, float(np.abs(g).max()), scale)
                continue
            errs[f"{gname}/{tag}"] = rel_err(g, r)
    print(f"\n{name} {regime} {precision} n={n}:", " ".join(f"{k}={v:.2e}" for k, v in errs.items()),
          f"(identically zero in the reference: {zero})" if zero else "")
    tol = X3_TOL if x3 else TF32_TOL
    bad = []
    for k, v in errs.items():
        kind = k if not k.startswith("d") else ("grad_emu" if k.endswith("/emu") else "grad64")
        bound = SHAPE_EXCEPTIONS.get((name, precision, kind), tol[kind])
        if not v < bound:
            bad.append(f"{k}={v:.3e} (bound {bound:g})")
    assert not bad, bad


# ---------------------------------------------------------------------------------------------------- dispatch
def _step_kernels(nt, n, regime):
    """Template arguments of the layer_fwd_kernel and layer_bwd_kernel launches of one step, in launch order."""
    from torch.profiler import ProfilerActivity, profile
    train_step(nt, n, regime)           # first launches (module load, shared-memory attributes) outside the trace
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        train_step(nt, n, regime)
    kern = sorted((e for e in prof.events() if "DeviceType.CUDA" in str(getattr(e, "device_type", ""))),
                  key=lambda e: e.time_range.start)
    if not kern:
        pytest.skip("the profiler recorded no CUDA kernels (CUPTI unavailable): the instantiations cannot be read")
    fw = [_template_args(e.name, "layer_fwd_kernel") for e in kern if "layer_fwd_kernel" in e.name]
    bw = [_template_args(e.name, "layer_bwd_kernel") for e in kern if "layer_bwd_kernel" in e.name]
    print(f"\n{regime} n={n}: layer_fwd {fw}; layer_bwd {bw}")
    return fw, bw


@gpu
def test_shape_steps_run_the_intended_kernels():
    """The instantiations layer_fwd_kernel<BASIS, TM, CG, NS> and layer_bwd_kernel<BASIS, TM, 2, 4, LNV, HEAD> that the
    step tests above rely on, read from torch.profiler: O1's single block carries the head in both directions (at
    R128r the backward regenerates the basis with the head in the same epilogue, at R64 it reads the saved x); D5's
    five blocks launch five of each, the head on the last and the basis on block 1 only.  If a threshold moves, this
    fails before the step tests silently drift onto another code path."""
    rows = regime_rows()
    fw, bw = _step_kernels(shape_net("O1"), rows["R128r"], "R128r")
    assert fw == [(1, 128, 2, 2)] and bw == [(1, 128, 2, 4, 1, 1)], (fw, bw)
    fw, bw = _step_kernels(shape_net("O1"), rows["R128r-feat"], "R128r-feat")
    assert fw == [(1, 128, 2, 2)] and bw == [(0, 128, 2, 4, 1, 1)], (fw, bw)
    fw, bw = _step_kernels(shape_net("O1"), rows["R64"], "R64")
    assert fw == [(1, 64, 4, 4)] and bw == [(0, 64, 2, 4, 1, 1)], (fw, bw)
    fw, bw = _step_kernels(shape_net("U"), rows["R128r"], "R128r")       # no LayerNorm: LNV = 0
    assert fw == [(1, 128, 2, 2), (0, 128, 2, 2)] and bw == [(0, 128, 2, 4, 0, 1), (1, 128, 2, 4, 0, 0)], (fw, bw)
    for regime, f, tm, regen in (("R128x", (128, 4, 4), 128, 0), ("R128r", (128, 2, 2), 128, 1),
                                 ("R64", (64, 4, 4), 64, 0)):
        fw, bw = _step_kernels(shape_net("D5"), rows[regime], regime)
        assert fw == [(1, *f)] + [(0, *f)] * 4, (regime, fw)
        # backward launches run from block 5 (the head) down to block 1
        assert bw == [(0, tm, 2, 4, 1, 1)] + [(0, tm, 2, 4, 1, 0)] * 3 + [(regen, tm, 2, 4, 1, 0)], (regime, bw)


# ---------------------------------------------------------------------------------------------------- prediction
# Which path forward-only calls take, per net: (whole-network kernel, site-tile x time-loop field kernel).  D5 has more
# blocks than either kernel holds (STDADK_MAX_HIDDEN = 4).  The field kernel declines O2: with the head on a 256-wide
# block and Q = 8 its shared-memory plan (field.cuh plan_field: 192 KB of operand and weight stages, the head's 8 KB,
# 12 KB of head partials of column groups 1-3) is 236,448 B, above 227 KB; O2 then takes the generic per-point kernel.
EXPECTED_PATHS = {"O1": (True, True), "O2": (True, False), "O3": (True, True), "R": (True, True), "U": (True, True),
                  "D4": (True, True), "D5": (False, False)}


def _module(name):
    """STInterpMLP of SHAPES[name] in eval mode (perturbed LayerNorm) and its oracle."""
    from stnf.models import STInterpMLP
    from test_gpu_model import _perturb_ln
    hidden, ln, p, q, loss, taus, ncw, fn, delta, learnable = SHAPES[name]
    seed = 400 + list(SHAPES).index(name)
    torch.manual_seed(seed)
    model = STInterpMLP(hidden_dims=list(hidden), layernorm=ln, dropout=p, output_dim=q, spatial_basis_function=fn,
                        use_delta_reparameterization=delta, spatial_learnable=learnable)
    if ln:
        _perturb_ln(model, seed)
    if name == "U":             # the default initialisation leaves the one unit off for every point: keep it on
        with torch.no_grad():
            model.hidden_blocks()[1][0].bias.fill_(0.5)
    if delta:        # upstream initialises delta at std 0.01: spread the quantiles so the head is not near zero
        with torch.no_grad():
            for d in model.delta_params:
                d.normal_(0.05, 0.1)
    state = {k: v.detach().cpu().numpy().copy() for k, v in model.state_dict().items()}
    return model.to("cuda").eval(), oracle_from_state(state, basis_fn=fn)


def field_chunk(n_sites, n_times, sms):
    """Time steps per work unit that stdadk_predict_field's planner picks: minimise waves x (chunk + 1)."""
    tiles = -(-n_sites // 128)
    best, best_cost = n_times, 1e30
    for chunk in range(1, n_times + 1):
        cost = -(-tiles * -(-n_times // chunk) // sms) * (chunk + 1.0)
        if cost < best_cost - 1e-9 or (cost < best_cost + 1e-9 and chunk > best):
            best, best_cost = chunk, cost
    return best


# FP64 bounds of the prediction paths: 1e-3 relative L2 and 3e-3 of the largest element, as every prediction test;
# five narrow blocks accumulate more TF32 rounding (test_shapes_the_fused_kernel_does_not_take_fall_back_to_block_kernels
# allows 3e-3 relative L2), and their implementation check is the TF32-emulating oracle.
PRED_TOL = {"D5": (3e-3, 1e-2, 5e-4)}          # (relative L2, largest element, relative L2 of the emulation)


@gpu
@pytest.mark.parametrize("name", list(SHAPES))
def test_shape_prediction_paths_vs_oracle(name):
    """Forward-only calls at every shape: 20,000 explicit points (157 tiles: the persistent loop wraps on 148 SMs and the
    last tile is ragged) through the whole-network kernel and the chained block kernels, against each other and the
    oracle; Predictor.space_time_field at S = 20,000 sites and T = 13 (on 148 SMs the planner cuts time into chunks of
    7 steps, the last one ragged) against the generic kernel and the oracle on a row sample.  D4 must take both fused
    kernels, D5 (five blocks) neither; a shape either kernel declines must still match the oracle through the
    fallback (EXPECTED_PATHS).  Largest measured on a B200: 9.4e-4 of FP64 (R, relative L2), field against generic
    7.2e-4 (D4), whole-network against block kernels 1.0e-6."""
    from st_dadk_b200.predict import Predictor
    l2_tol, max_tol, emu_tol = PRED_TOL.get(name, (1e-3, 3e-3, 1e-4))
    model, m = _module(name)
    q = SHAPES[name][3]
    rng = np.random.default_rng(6)
    n = 20000
    coords, t = rng.random((n, 2), dtype=np.float32), rng.random(n, dtype=np.float32)
    pr = Predictor(model)
    fused = pr.points(T(coords), T(t))[0].cpu().numpy()
    fused_ok = bool(pr.ex._fused_ok)
    pr.ex.fused_predict = False
    layered = pr.points(T(coords), T(t))[0].cpu().numpy()
    pr.ex.fused_predict = True
    ref, emu = orc.forward(m, None, coords, t), orc.forward(m, None, coords, t, rnd=orc.tf32_round)
    errs = {"fused/layered": rel_l2(fused, layered), "fused/64": rel_l2(fused, ref), "fused/64max": rel_err(fused, ref),
            "fused/emu": rel_l2(fused, emu), "layered/64": rel_l2(layered, ref), "layered/emu": rel_l2(layered, emu)}

    S, Tn = 20000, 13
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    k_chunk = field_chunk(S, Tn, sms)
    sites = torch.rand(S, 2, generator=torch.Generator().manual_seed(7)).cuda()
    field = pr.space_time_field(sites, Tn)[0]
    field_ok = pr.used_field_kernel
    gen = Predictor(model)
    gen.use_field_kernel = False
    generic = gen.space_time_field(sites, Tn)[0]
    assert not gen.used_field_kernel
    field, generic = field.cpu().numpy(), generic.cpu().numpy()
    rows = np.unique(np.r_[rng.integers(0, S * Tn, 3000), S * Tn - 2000:S * Tn])      # the last time chunk, all sites
    sc = sites.cpu().numpy()[rows % S]
    st = (rows // S).astype(np.float32) / np.float32(Tn - 1)
    fref = orc.forward(m, None, sc, st)
    errs.update({"field/generic": rel_l2(field, generic), "field/64": rel_l2(field[rows], fref),
                 "field/64max": rel_err(field[rows], fref), "generic/64": rel_l2(generic[rows], fref)})
    if not field_ok and len(SHAPES[name][0]) <= 4:        # the reason of the refusal, for the record
        from st_dadk_b200 import _lib as L
        pr.ex._field_ok = None
        assert not pr.ex.field_supported()
        print(f"\n{name}: field kernel declined: {L.lib().stdadk_last_error().decode('utf-8', 'replace')}")
    print(f"\n{name}: whole-network kernel {fused_ok}, field kernel {field_ok} (k_chunk {k_chunk} of T = {Tn} on {sms} "
          f"SMs):", " ".join(f"{k}={v:.2e}" for k, v in errs.items()))
    assert np.isfinite(fused).all() and np.isfinite(field).all() and fused.shape == (n, q)
    assert np.std(fused) > 1e-3 * np.abs(fused).max(), "yhat is constant: the network computes nothing to compare"
    assert (fused_ok, field_ok) == EXPECTED_PATHS[name]
    bad = [f"{k}={v:.3e}" for k, v in errs.items()
           if not v < {"64": l2_tol, "64max": max_tol, "emu": emu_tol}.get(k.split("/")[1], 2e-4 if k == "fused/layered"
                                                                           else 1e-3)]
    assert not bad, bad
    if k_chunk == 1 or Tn % k_chunk == 0:
        pytest.skip(f"on {sms} SMs the field planner takes {k_chunk}-step chunks of T = {Tn}: no multi-step, ragged "
                    "time chunk (the comparisons above passed)")


@gpu
def test_width1_layernorm_known_answer():
    """hidden (16, 1) with LayerNorm, Q = 2.  A LayerNorm over one unit sees mean = x and variance 0, so its output is
    beta for every row and yhat = w_head relu(beta) + b_head is one constant.  The kernels form the normalised value
    as fma(x, rstd, nmr) with rstd = 1/sqrt(eps) = 316.2 and nmr = -round(mean rstd): the exact rounding error e of
    x rstd, |e| <= ulp(x rstd) / 2 <= 316.2 ulp(x).  Then y = round(e gamma + beta), relu, and the head product and
    bias sum in FP32: every output lies within |w_head| (316.2 ulp(x) |gamma| + ulp(beta)) + ulp(w_head beta) +
    ulp(c) of c = w_head beta + b_head, with ulp(x) of the largest |x| over the rows.  Checked through the
    whole-network kernel, the chained block kernels and the field kernel."""
    L, ops, Executor, NetSpec, LossSpec = _mods()
    m = _default_oracle_model(71, q=2, hidden=(16, 1))
    m.ln_gamma[1], m.ln_beta[1] = np.float32([1.3]), np.float32([0.37])
    m.weights[2], m.biases[2] = np.float32([[0.8], [-0.55]]), np.float32([0.1, 0.2])
    ex = Executor(spec_from_oracle(m))
    rng = np.random.default_rng(8)
    S, Tn = 3000, 5
    sites = rng.random((S, 2), dtype=np.float32)
    coords = np.tile(sites, (Tn, 1))
    t = np.repeat(np.arange(Tn, dtype=np.float32) / np.float32(Tn - 1), S)
    pts = ops.make_points(T(coords), T(t))
    outs = {"fused": ex.forward(pts, train=False).clone()}
    assert ex._fused_ok
    ex.fused_predict = False
    outs["layered"] = ex.forward(pts, train=False).clone()
    ex.fused_predict = True
    assert ex.field_supported()
    outs["field"] = torch.empty(S * Tn, 2, device="cuda")
    ex.predict_field(outs["field"], 0, S * Tn, S, Tn, sites=T(sites))
    _, cache = orc.forward(m, None, coords, t, return_cache=True)
    x = np.float32(1.01 * np.abs(cache["layers"][1]["z"]).max())        # 1 %: the kernels' x is TF32-rounded upstream
    assert x > 0
    w, b = m.weights[2][:, 0].astype(np.float64), m.biases[2].astype(np.float64)
    beta, gamma = float(m.ln_beta[1][0]), float(m.ln_gamma[1][0])
    c = w * beta + b
    rstd = 1.0 / np.sqrt(np.float32(m.ln_eps))
    bound = (np.abs(w) * (rstd * float(np.spacing(x)) * abs(gamma) + float(np.spacing(np.float32(beta))))
             + np.spacing(np.abs(w * beta).astype(np.float32)) + np.spacing(np.abs(c).astype(np.float32)))
    for k, v in outs.items():
        dev = np.abs(v.cpu().numpy() - c).max(axis=0)
        print(f"\nwidth-1 LayerNorm, {k}: largest deviation from the constant {dev} (bound {bound})")
        assert np.all(dev <= bound), (k, dev, bound)


# ---------------------------------------------------------------------------------------------------- the trainer
def _trainer_cases():
    base = dict(lr=2e-3, weight_decay=1e-2, regression_type="mean", epochs=100)
    mq3 = dict(base, regression_type="multi-quantile", quantile_levels=[0.1, 0.5, 0.9], non_crossing_weight=0.5,
               non_crossing_power=2)
    return {"h64": Case(model=dict(hidden_dims=[64]), cfg=base, batches=[[4096, 4096]] * 2, seed=21),
            "h50-33-7-q3": Case(model=dict(hidden_dims=[50, 33, 7], output_dim=3), cfg=mq3, batches=[[4096, 4096]] * 2,
                                seed=22, clip_engaged=False, taus=(0.1, 0.5, 0.9))}


@gpu
@pytest.mark.parametrize("name", ["h64", "h50-33-7-q3"])
def test_shape_trainer_steps_vs_oracle(name):
    """Trainer.train_step, tf32x3, graphs replayed, 2 epochs of 2 x 4,096 rows, every step against the oracle at its
    own weights with the per-step assertions of test_gpu_train_steps (gradients recovered from the Adam moments, the
    update, the loss, the device step counter): one hidden block of 64 (head and loss in block 1), and 50-33-7 with
    Q = 3 pinball and the quadratic non-crossing penalty."""
    run_case(name, _trainer_cases()[name])
