"""Training and prediction with hidden blocks wider than 256 units (up to STDADK_MAX_WIDTH = 512), which run the wide
forms of the block kernels: layer_fwd_kernel<BASIS, TM, 4, 2> (two MMAs per K slab into one accumulator of up to 512
tensor-memory columns) and the x-image layer_bwd_kernel<0, TM, 2, 2, LNV, HEAD>.  A wide block keeps its x image at
every batch size; the narrow blocks of a multi-wave batch still recompute theirs.

  id   hidden            LN   dropout  head / loss                      what it reaches
  W1   (512, 512, 256)   yes  0.1      Q = 5 pinball                    a wide block 1 (basis) and block 2 (image); a
                                                                        narrow block below a wide one (K = 512)
  W2   (300,)            no   0        Q = 1 MSE                        the head in a wide block 1; n_pad 320 = 256 + 64
  W3   (384, 257, 64)    yes  0.1      Q = 3 pinball, delta head,       knotgrad_kernel with K = 384; n_pad 288
                                       learnable knots
  W4   (512, 128)        yes  0.1      Q = 1 MSE, 2,496 knots on four   support walk forward / wgrad at 512 columns
                                       lattice levels (cell list)
  W4L  the same knots, learnable                                        knot gradients from the walk

The step tests follow test_gpu_regimes exactly (points gathered through a permutation, row_begin != 0, dropout keys
crossing 2^32, the chunked FP64 oracle and the TF32-emulating one)."""
import ctypes as C
from functools import lru_cache

import numpy as np
import pytest
import torch

from helpers import golden, oracle_from_state, orc
from test_gpu_kernels import T, _default_oracle_model, _mods, rel_err, rel_l2
from test_gpu_regimes import P_DROP, TF32_TOL, X3_TOL, Net, _grad_pairs, _rows, _template_args, oracle, regime_rows, \
    train_step
from test_gpu_train_steps import Case, run_case

gpu = pytest.mark.gpu

# name: (hidden, layernorm, dropout, Q, loss, taus, basis, delta head, learnable knots)
WIDE = {
    "W1": ((512, 512, 256), True, P_DROP, 5, "pinball", (0.05, 0.25, 0.5, 0.75, 0.95), "wendland", False, False),
    "W2": ((300,), False, 0.0, 1, "mse", None, "wendland", False, False),
    "W3": ((384, 257, 64), True, P_DROP, 3, "pinball", (0.1, 0.5, 0.9), "wendland", True, True),
    "W4": ((512, 128), True, P_DROP, 1, "mse", None, "wendland", False, False),
    "W4L": ((512, 128), True, P_DROP, 1, "mse", None, "wendland", False, True),
}
W4_SIDES = (8, 16, 24, 40)          # 64 + 256 + 576 + 1,600 = 2,496 knots: above DENSE_MAX_KNOTS


def _walk_model(seed, hidden):
    """A lattice of 2,496 Wendland knots (the executor walks them) with the golden temporal knots, Linear-init weights."""
    rng = np.random.default_rng(seed)
    cs, bs = [], []
    for s in W4_SIDES:
        g = np.linspace(0.0, 1.0, s)
        cs.append(np.stack(np.meshgrid(g, g, indexing="ij"), -1).reshape(-1, 2))
        bs.append(np.full(s * s, 2.5 / (s - 1)))
    kn = golden("knots")
    c, b = np.concatenate(cs).astype(np.float32), np.concatenate(bs).astype(np.float32)
    dims = [c.shape[0] + kn["t_centers"].shape[0], *hidden]
    ws, bias, gs, be = [], [], [], []
    for i in range(len(hidden)):
        bound = 1 / np.sqrt(dims[i])
        ws.append(rng.uniform(-bound, bound, (dims[i + 1], dims[i])).astype(np.float32))
        bias.append(rng.uniform(-bound, bound, dims[i + 1]).astype(np.float32))
        gs.append((1 + 0.1 * rng.standard_normal(dims[i + 1])).astype(np.float32))
        be.append((0.1 * rng.standard_normal(dims[i + 1])).astype(np.float32))
    bound = 1 / np.sqrt(dims[-1])
    ws.append(rng.uniform(-bound, bound, (1, dims[-1])).astype(np.float32))
    bias.append(rng.uniform(-bound, bound, 1).astype(np.float32))
    return orc.OracleModel(centers=c, bandwidths=b, t_centers=kn["t_centers"], t_bandwidths=kn["t_bandwidths"],
                           weights=ws, biases=bias, ln_gamma=gs, ln_beta=be, basis_fn="wendland")


@lru_cache(maxsize=None)
def wide_net(name):
    hidden, ln, p, q, loss, taus, fn, delta, learnable = WIDE[name]
    if name.startswith("W4"):
        m = _walk_model(900, hidden)
    else:
        m = _default_oracle_model(800 + list(WIDE).index(name), q=q, fn=fn, hidden=hidden)
    m.dropout = p
    if not ln:
        m.ln_gamma = [None] * len(hidden)
        m.ln_beta = [None] * len(hidden)
    if delta:
        W, b = m.weights.pop(), m.biases.pop()
        rng = np.random.default_rng(78)
        d0 = np.concatenate([b[:1], W[0]]).astype(np.float32)
        m.delta = [d0] + [(0.05 + 0.02 * rng.standard_normal(W.shape[1] + 1)).astype(np.float32) for _ in range(q - 1)]
    sizes = [s * s for s in W4_SIDES] if name.startswith("W4") else None     # walked through the cell list
    return Net(m, loss, taus, learnable=learnable, sizes=sizes)


# ---------------------------------------------------------------------------------------------------- one step
# (net, precision, kind of error): bound, with the largest value measured on a B200 and its cause.  (None so far.)
WIDE_EXCEPTIONS = {}

STEP_CASES = ([(s, r, "tf32") for s in WIDE for r in ("R64", "R128x", "R128x-cg2", "R128r")]
              + [(s, r, "tf32x3") for s in ("W1", "W3") for r in ("R64", "R128x", "R128x-cg2", "R128r")])


@gpu
@pytest.mark.parametrize("name,regime,precision", STEP_CASES, ids=["-".join(c) for c in STEP_CASES])
def test_wide_training_step_vs_oracle(name, regime, precision):
    """yhat, loss and every gradient of one gathered training step against the chunked FP64 oracle and, in TF32 mode,
    the TF32-emulating oracle, with the bounds of test_gpu_regimes.test_training_step_vs_oracle (TF32_TOL / X3_TOL).
    The walked nets (W4, W4L) keep the spatial basis in FP32: against the emulation they take the bounds
    test_gpu_regimes allows its walked net N6."""
    n = _rows(regime)
    nt = wide_net(name)
    x3 = precision == "tf32x3"
    (y64, l64, g64), (yemu, lemu, gemu) = oracle(nt, n, regime)
    ex, yhat, loss, grads = train_step(nt, n, regime, precision)
    assert ex.sparse == name.startswith("W4")
    ws = ex._ctx[2]
    # a wide block keeps x at every batch size; a narrow one only in the single-wave regimes
    save_all = n <= ex.SAVE_X_MAX_ROWS
    assert ws.x is not None
    assert [x is not None for x in ws.x] == [save_all or w.shape[0] > 256 for w in ex.spec.weights]
    assert np.isfinite(yhat).all()
    errs = {"yhat64": rel_err(yhat, y64), "loss": abs(loss - l64) / abs(l64)}
    if not x3:
        errs["yhat_emu"] = rel_l2(yhat, yemu)
    refs = [("64", g64)] + ([] if x3 else [("emu", gemu)])
    for tag, ref in refs:
        for gname, g, r in _grad_pairs(grads, ref, nt):
            errs[f"{gname}/{tag}"] = rel_err(g, r)
    print(f"\n{name} {regime} {precision} n={n}:", " ".join(f"{k}={v:.2e}" for k, v in errs.items()))
    tol = X3_TOL if x3 else TF32_TOL
    walked = {"yhat_emu": 1e-3, "dcenters/emu": 5e-2, "dlog_bw/emu": 1e-2, "dcenters/64": 5e-2}
    bad = []
    for k, v in errs.items():
        kind = k if not k.startswith("d") else ("grad_emu" if k.endswith("/emu") else "grad64")
        bound = tol[kind]
        if name.startswith("W4") and not x3:
            bound = walked.get(k, bound)
        bound = WIDE_EXCEPTIONS.get((name, precision, k), bound)
        if not v < bound:
            bad.append(f"{k}={v:.3e} (bound {bound:g})")
    assert not bad, bad


# ---------------------------------------------------------------------------------------------------- dispatch
def _launches(steps):
    """Kernel launches of the training steps `steps` ((net, rows, regime) each), traced in one torch.profiler session
    (every step's first launches, module load and shared-memory attributes, are made before it).  train_step ends in a
    device synchronisation, so sorted by start time the launches fall into the steps in order.  Returns per step
    (layer_fwd template arguments, layer_bwd template arguments, kernel names)."""
    from torch.profiler import ProfilerActivity, profile
    for nt, n, regime in steps:
        train_step(nt, n, regime)
    # The first launches of a session have been missing from its trace (measured: the first step's pack_images of
    # six), so the session opens with one more step whose launches are not read.
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        for nt, n, regime in [steps[0], *steps]:
            train_step(nt, n, regime)
    kern = sorted((e for e in prof.events() if "DeviceType.CUDA" in str(getattr(e, "device_type", ""))),
                  key=lambda e: e.time_range.start)
    if not kern:
        pytest.skip("the profiler recorded no CUDA kernels (CUPTI unavailable): the instantiations cannot be read")
    # every step packs its weight images in one pack_images_kernel launch, before its first layer_fwd
    starts = [i for i, e in enumerate(kern) if "pack_images_kernel" in e.name]
    assert len(starts) >= len(steps), (len(starts), len(steps))
    starts = starts[-len(steps):]
    out = []
    for k, (nt, n, regime) in enumerate(steps):
        part = kern[starts[k]:starts[k + 1] if k + 1 < len(steps) else len(kern)]
        fw = [_template_args(e.name, "layer_fwd_kernel") for e in part if "layer_fwd_kernel" in e.name]
        bw = [_template_args(e.name, "layer_bwd_kernel") for e in part if "layer_bwd_kernel" in e.name]
        print(f"\n{regime} n={n}: layer_fwd {fw}; layer_bwd {bw}")
        out.append((fw, bw, {e.name for e in part}))
    return out


@gpu
def test_wide_steps_run_the_intended_kernels():
    """W1's launches per regime under torch.profiler.  Its wide blocks 1 and 2 take layer_fwd_kernel<B, TM, 4, 2> in
    every regime (never the two-CTA <B, 128, 2, 2>, not even at R128x-cg2 where the narrow block 3 takes it) and the
    x-image backward <0, TM, 2, 2, 1, 0>; block 3 (256, the head) takes the narrow kernels, recomputing x at R128r.
    W2 carries the head in a wide block 1 without LayerNorm; W4 walks its knots with the wide walk kernels."""
    rows = regime_rows()
    L, ops, Executor, *_ = _mods()
    w1 = [(regime, tm, narrow_fwd) for regime, tm, narrow_fwd in
          (("R64", 64, (64, 4, 4)), ("R128x", 128, (128, 4, 4)), ("R128x-cg2", 128, (128, 2, 2)),
           ("R128r", 128, (128, 2, 2)))
          if regime != "R128x-cg2" or rows[regime] <= Executor.SAVE_X_MAX_ROWS]
    steps = ([(wide_net("W1"), rows[r], r) for r, _, _ in w1]
             + [(wide_net("W2"), rows["R128r"], "R128r"), (wide_net("W4"), rows["R128x"], "R128x")])
    got = _launches(steps)
    for (regime, tm, narrow_fwd), (fw, bw, _) in zip(w1, got):
        assert fw == [(1, tm, 4, 2), (0, tm, 4, 2), (0, *narrow_fwd)], (regime, fw)
        assert bw == [(0, tm, 2, 4, 1, 1), (0, tm, 2, 2, 1, 0), (0, tm, 2, 2, 1, 0)], (regime, bw)
    fw, bw, _ = got[len(w1)]            # W2 at R128r: the wide block still reads its x image
    assert fw == [(1, 128, 4, 2)] and bw == [(0, 128, 2, 2, 0, 1)], (fw, bw)
    fw, bw, names = got[len(w1) + 1]    # W4: the walk at 512 columns
    assert fw == [(1, 128, 4, 2), (0, 128, 4, 4)], fw
    assert any("sparse_spatial_fwd_wide_kernel" in s for s in names)
    assert any("sparse_spatial_wgrad_wide_kernel" in s for s in names)


# ---------------------------------------------------------------------------------------------------- the trainer
@gpu
def test_wide_trainer_steps_vs_oracle():
    """Trainer.train_step on [512, 512, 256], tf32x3, graphs replayed and recaptured, 2 epochs of 2 x 4,096 rows, every
    step against the oracle with the per-step assertions of test_gpu_train_steps."""
    base = dict(lr=2e-3, weight_decay=1e-2, regression_type="mean", epochs=100)
    run_case("wide", Case(model=dict(hidden_dims=[512, 512, 256]), cfg=base, batches=[[4096, 4096]] * 2, seed=23))


# ---------------------------------------------------------------------------------------------------- prediction
def _module(name, seed):
    from stnf.models import STInterpMLP
    from test_gpu_model import _perturb_ln
    hidden, ln, p, q, loss, taus, fn, delta, learnable = WIDE[name]
    torch.manual_seed(seed)
    model = STInterpMLP(hidden_dims=list(hidden), layernorm=ln, dropout=p, output_dim=q, spatial_basis_function=fn,
                        use_delta_reparameterization=delta, spatial_learnable=learnable)
    if ln:
        _perturb_ln(model, seed)
    if delta:
        with torch.no_grad():
            for d in model.delta_params:
                d.normal_(0.05, 0.1)
    state = {k: v.detach().cpu().numpy().copy() for k, v in model.state_dict().items()}
    return model.to("cuda").eval(), oracle_from_state(state, basis_fn=fn)


@gpu
@pytest.mark.parametrize("name", ["W1", "W2", "W3"])
def test_wide_prediction_vs_oracle(name):
    """Forward-only calls at 20,000 points through Predictor.points, Predictor.grid and Predictor.space_time_field:
    the whole-network and field kernels report 'unsupported' for a block wider than 256, and the per-block chain
    computes every prediction.  Bounds of test_gpu_shapes: 1e-3 relative L2 and 3e-3 of the largest element of FP64,
    1e-4 relative L2 of the TF32-emulating oracle."""
    from st_dadk_b200 import _lib as L
    from st_dadk_b200.predict import Predictor
    model, m = _module(name, 500 + list(WIDE).index(name))
    rng = np.random.default_rng(9)
    n = 20000
    coords, t = rng.random((n, 2), dtype=np.float32), rng.random(n, dtype=np.float32)
    pr = Predictor(model)
    got = pr.points(T(coords), T(t))[0].cpu().numpy()
    assert not pr.ex.fused_supported()
    assert "at most 256" in L.lib().stdadk_last_error().decode()
    assert not pr.ex.field_supported()
    assert "at most 256" in L.lib().stdadk_last_error().decode()
    ref, emu = orc.forward(m, None, coords, t), orc.forward(m, None, coords, t, rnd=orc.tf32_round)
    errs = {"points/64": rel_l2(got, ref), "points/64max": rel_err(got, ref), "points/emu": rel_l2(got, emu)}
    nx, ny, nt_ = 100, 50, 4                           # 20,000 grid points
    grid = pr.grid(nx, ny, nt_)[0].cpu().numpy().reshape(-1, got.shape[1])
    assert not pr.used_field_kernel
    k, i, j = np.meshgrid(np.arange(nt_), np.arange(nx), np.arange(ny), indexing="ij")
    gc = np.stack([i.ravel() / np.float32(nx - 1), j.ravel() / np.float32(ny - 1)], 1).astype(np.float32)
    gt = (k.ravel() / np.float32(nt_ - 1)).astype(np.float32)
    gref = orc.forward(m, None, gc, gt)
    errs.update({"grid/64": rel_l2(grid, gref), "grid/64max": rel_err(grid, gref)})
    S, Tn = 20000, 3
    sites = torch.rand(S, 2, generator=torch.Generator().manual_seed(7)).cuda()
    field = pr.space_time_field(sites, Tn)[0].cpu().numpy().reshape(-1, got.shape[1])
    assert not pr.used_field_kernel
    rows = np.unique(rng.integers(0, S * Tn, 4000))
    sc = sites.cpu().numpy()[rows % S]
    st = (rows // S).astype(np.float32) / np.float32(Tn - 1)
    fref = orc.forward(m, None, sc, st)
    errs.update({"field/64": rel_l2(field[rows], fref), "field/64max": rel_err(field[rows], fref)})
    print(f"\n{name}:", " ".join(f"{k}={v:.2e}" for k, v in errs.items()))
    assert np.std(got) > 1e-3 * np.abs(got).max(), "yhat is constant: the network computes nothing to compare"
    bad = [f"{k}={v:.3e}" for k, v in errs.items()
           if not v < {"64": 1e-3, "64max": 3e-3, "emu": 1e-4}[k.split("/")[1]]]
    assert not bad, bad


# ---------------------------------------------------------------------------------------------------- capacity
def _wide_block1_launches(ops, L, k_s, k_t_levels, n_out, rows_many):
    """Block 1 of width n_out with k_s scattered knots through every dense launch of a wide block 1: layer_fwd at 1,000
    rows (64-row tiles) and at rows_many rows (128-row tiles), the x-image layer_bwd and the basis-form wgrad.  Returns
    {launch: error or None}; the launches that ran are checked against the FP64 reference."""
    rng = np.random.default_rng(k_s + n_out)
    c = rng.random((k_s, 2)).astype(np.float32)
    b = np.full(k_s, 0.1, np.float32)
    tc, tb = orc.temporal_knots(k_t_levels)
    k_t = tc.shape[0]
    n_in = k_s + k_t
    knots4 = ops.knots_prepare(T(c), T(b), None, "wendland")
    tk = ops.tknots_prepare(T(tc), T(tb))
    basis = ops.make_basis(knots4, tk, k_s, k_t, 0, "wendland")
    W = orc.tf32_round((rng.standard_normal((n_out, n_in)) / 6).astype(np.float32))
    bias = (0.1 * rng.standard_normal(n_out)).astype(np.float32)
    w_img, tbias = ops.pack_image(T(W)), T(bias)        # the layer holds raw pointers: keep the tensors alive
    layer = ops.make_layer(w_img, tbias, None, None, n_in, n_out, 1e-5, 0)
    rows, errs = 1000, {}

    def pts_of(n):
        r = np.random.default_rng(n)
        co, tt = r.random((n, 2)).astype(np.float32), r.random((n, 1)).astype(np.float32)
        return co, tt, ops.make_points(T(co), T(tt))

    def z_ref(co, tt):
        a = np.concatenate([orc.spatial_basis(co, c, b, "wendland"), orc.temporal_basis(tt, tc, tb)], axis=1)
        return a, a @ W.astype(np.float64).T + bias

    def attempt(name, fn):
        try:
            fn()
            torch.cuda.synchronize()
            errs[name] = None
        except RuntimeError as e:
            assert "shared memory" in str(e), e
            errs[name] = str(e)

    x_img = None
    for name, n in (("fwd_tm64", rows), ("fwd_tm128", rows_many)):
        co, tt, pts = pts_of(n)
        out, x = ops.new_image(n, n_out, "cuda"), ops.new_image(n, n_out, "cuda")

        def fwd():
            a = L.FwdArgs()
            a.basis = C.pointer(basis)
            a.pts = pts
            a.layer = layer
            a.drop = L.Dropout(0.0, 0, 0)
            a.out_img, a.x_img = out.data_ptr(), x.data_ptr()
            ops.layer_fwd(a)
        attempt(name, fwd)
        if errs[name] is None:
            idx = np.r_[0:1000, n - 1000:n]
            got = ops.unpack_image(out, n, n_out).cpu().numpy()[idx]
            ref = np.maximum(z_ref(co[idx], tt[idx])[1], 0.0)
            assert rel_l2(got, ref) < 2e-3, (name, rel_l2(got, ref))
            if n == rows:
                x_img = x

    co, tt, pts = pts_of(rows)
    n_next = 32
    Wn = orc.tf32_round((rng.standard_normal((n_next, n_out)) / 6).astype(np.float32))
    dzn = orc.tf32_round(rng.standard_normal((rows, n_next)).astype(np.float32))
    wt_next, dzn_img = ops.pack_image(T(Wn).t()), ops.pack_image(T(dzn))
    dz_img, d_bias = ops.new_image(rows, n_out, "cuda"), torch.zeros(n_out, device="cuda")
    if x_img is not None:           # the wide backward reads the forward's x image: it has no knot tables to hold
        a = L.BwdArgs()
        a.pts = pts
        a.layer = layer
        a.drop = L.Dropout(0.0, 0, 0)
        a.x_img = x_img.data_ptr()
        a.dz_next_img, a.wt_next_img, a.n_next = dzn_img.data_ptr(), wt_next.data_ptr(), n_next
        a.dz_img, a.d_bias = dz_img.data_ptr(), d_bias.data_ptr()
        ops.layer_bwd(a)
        A64, z64 = z_ref(co, tt)
        z_emu = orc.tf32_round(A64.astype(np.float32)).astype(np.float64) @ W.astype(np.float64).T + bias
        ref = (dzn.astype(np.float64) @ Wn.astype(np.float64)) * (z_emu > 0)
        got = ops.unpack_image(dz_img, rows, n_out).cpu().numpy()
        keep = np.abs(z_emu) >= 1e-3
        bad = np.abs(got - ref)[keep] > 2.0 ** -10 * np.abs(ref)[keep] + 1e-5 * np.abs(ref).max()
        assert not bad.any(), int(bad.sum())
        errs["bwd_x"] = None

    dz = orc.tf32_round(rng.standard_normal((rows, n_out)).astype(np.float32))
    dz_w, dw = ops.pack_image(T(dz)), torch.zeros(n_out, n_in, device="cuda")

    def wgrad():
        w = L.WgradArgs()
        w.basis = C.pointer(basis)
        w.pts = pts
        w.dz_img = dz_w.data_ptr()
        w.n_in, w.n_out = n_in, n_out
        w.dw, w.stride_o, w.stride_i = dw.data_ptr(), dw.stride(0), dw.stride(1)
        ops.wgrad(w)
    attempt("wgrad", wgrad)
    if errs["wgrad"] is None:
        ref = dz.astype(np.float64).T @ z_ref(co, tt)[0]
        assert rel_err(dw.cpu().numpy(), ref) < 2e-3, rel_err(dw.cpu().numpy(), ref)
    return errs


@gpu
@pytest.mark.parametrize("k_t_levels", [(10, 15, 45), (10, 15)], ids=["kt70", "kt25"])
def test_wide_capacity_query_equals_the_launch_checks(k_t_levels):
    """Width 512: at the K_s stdadk_dense_max_knots reports every dense block-1 launch runs and matches the FP64
    reference; at K_s + 1 the launch the query names returns its shared-memory error."""
    L, ops, *_ = _mods()
    k_t = sum(k_t_levels)
    K = ops.dense_max_knots(0, k_t, 512, 0)
    S = torch.cuda.get_device_properties(0).multi_processor_count
    at_k = _wide_block1_launches(ops, L, K, k_t_levels, 512, 2 * S * 128)
    assert all(v is None for v in at_k.values()) and "bwd_x" in at_k, at_k
    fits, why = ops.dense_basis_supported(0, K + 1, k_t, 512, 0)
    assert not fits
    above = _wide_block1_launches(ops, L, K + 1, k_t_levels, 512, 2 * S * 128)
    print(f"\nwidth 512, {k_t} temporal knots: K = {K}; at K + 1 the query says {why!r}; launches {above}")
    failed = [v for v in above.values() if v is not None]
    assert failed and any(why in v for v in failed), (why, above)


# ---------------------------------------------------------------------------------------------------- limits
def test_width_above_the_limit_raises():
    """513 units: the model raises on its first forward, naming the limit of 512; the library refuses the block too."""
    from stnf.models import STInterpMLP
    from st_dadk_b200 import _lib as L
    assert L.MAX_WIDTH == 512
    model = STInterpMLP(hidden_dims=[513, 64])
    with pytest.raises(RuntimeError, match=r"513 > 512"):
        model._executor()
    ops = _mods()[1]
    fits, why = ops.dense_basis_supported(0, 227, 70, 513, 0)
    assert not fits, why
    fits, _ = ops.dense_basis_supported(0, 227, 70, 512, 0)
    assert fits
