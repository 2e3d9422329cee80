"""Block 1's dense basis path at large knot counts, and the regime choice at the edge of what its kernels hold.

The parts of block 1 that scale with the number of spatial knots K_s: the chunk-indexed knot tables of layer_fwd /
layer_bwd (64 B per 4-feature chunk of shared memory), the support vote that skips knot groups, wgrad's split of the
block-1 columns into ceil(a_slabs / 8) N tiles (ragged when 8 does not divide the slabs evenly), knotgrad's
ceil(K_s / 128) knot tiles, and the shared-memory fallbacks of the whole-network and field prediction kernels.

Executor._setup_regime keeps the dense path only where stdadk_dense_basis_supported says every block-1 launch fits in
227 KB; above that the knots are walked, or the executor raises at construction when they cannot be.  At first width
256 and 70 temporal knots the recompute layer_bwd binds first (1,626 knots); at widths 128 and 64 the basis-form wgrad
(2,134)."""
import ctypes as C
from functools import lru_cache

import numpy as np
import pytest
import torch

from helpers import orc
from test_gpu_kernels import T, _mods, _small_net, rel_err, rel_l2, spec_from_oracle
from test_gpu_regimes import (EXPECTED, KEY_OFFSET, P_DROP, ROW_BEGIN, SEED, STEP, TF32_TOL, X3_TOL, Net, _grad_pairs,
                              _template_args, chunked_oracle, regime_rows, table)

gpu = pytest.mark.gpu


def _ops():
    import __graft_entry__ as g
    g.build()
    from st_dadk_b200 import ops
    return ops


def _scattered_knots(rng, sizes):
    """Knots that are not a lattice (as _cell_list_knots): per level, clustered centres with per-knot bandwidths in the
    first level after the coarsest, uniform centres (a few outside [0,1]^2) elsewhere."""
    cen, bw = [], []
    for li, k in enumerate(sizes):
        if li == 1:
            c = 0.5 + 0.12 * rng.standard_normal((k, 2))
            b = rng.uniform(0.15, 0.3, k)
        else:
            c = rng.random((k, 2)) * 1.1 - 0.05
            b = rng.uniform(0.6, 1.0, k) * 2.5 / np.sqrt(k)
        cen.append(c)
        bw.append(b)
    return np.concatenate(cen).astype(np.float32), np.concatenate(bw).astype(np.float32)


def _model(rng, c, b, k_t_levels, hidden, q=1, fn="wendland"):
    tc, tb = orc.temporal_knots(k_t_levels)
    ws, bs, gs, be = _small_net(rng, c.shape[0], k_t=tc.shape[0], hidden=hidden)
    ws[-1] = (rng.standard_normal((q, hidden[-1])) / 6).astype(np.float32)
    bs[-1] = np.zeros(q, np.float32)
    return orc.OracleModel(centers=c, bandwidths=b, t_centers=tc, t_bandwidths=tb, weights=ws, biases=bs, ln_gamma=gs,
                           ln_beta=be, basis_fn=fn)


D1_LEVELS = [36, 144, 400, 1024]


@lru_cache(maxsize=None)
def net(name):
    if name == "D1":        # uniform lattice of 1,604 knots: 1,674 block-1 inputs = 53 slabs, wgrad N tiles 7 x 8 + 5
        c, b = orc.uniform_spatial_knots(D1_LEVELS)
        m = _model(np.random.default_rng(71), c, b, [10, 15, 45], (256, 256, 128))
        m.dropout = P_DROP
        return Net(m)
    if name == "D2":        # 900 learnable scattered knots: knotgrad's 8 knot tiles, the last one 4 knots wide
        rng = np.random.default_rng(72)
        c, b = _scattered_knots(rng, [100, 300, 500])
        return Net(_model(rng, c, b, [10, 15], (128, 64), q=3), "pinball", (0.1, 0.5, 0.9), learnable=True)
    if name == "D3":        # one knot more than the dense kernels hold at width 256: the executor must walk
        k_s = _mods()[1].dense_max_knots(0, 70, 256, 0) + 1
        rng = np.random.default_rng(73)
        sizes = [27, 400, k_s - 427]
        c, b = _scattered_knots(rng, sizes)
        return Net(_model(rng, c, b, [10, 15, 45], (256, 256, 128)), sizes=sizes)
    raise KeyError(name)


_ORACLE = {}


def oracle(name, n):
    """FP64 and TF32-emulating chunked oracle of network `name` on the n-row batch; both precisions and the R128r /
    R128r-feat pair share it."""
    key = (name, n)
    if key not in _ORACLE:
        nt = net(name)
        coords, t, y, X, perm = table(n, 0)
        idx = perm[ROW_BEGIN:ROW_BEGIN + n]
        args = (nt.m, None, coords[idx], t[idx], y[idx], nt.loss, nt.taus, nt.nc_weight, 2)
        kw = dict(key_offset=KEY_OFFSET, knot_grads=nt.learnable)
        _ORACLE[key] = (chunked_oracle(*args, **kw), chunked_oracle(*args, rnd=orc.tf32_round, **kw))
    return _ORACLE[key]


def train_step(name, n, regime, precision="tf32"):
    """forward(train, save) + backward of `name` on n gathered rows, the regime left to the executor."""
    L, ops, Executor, NetSpec, LossSpec = _mods()
    nt = net(name)
    spec = spec_from_oracle(nt.m, learnable=nt.learnable, dropout=nt.m.dropout, precision=precision)
    spec.level_sizes = nt.sizes
    ex = Executor(spec)
    assert ex.sparse == (name == "D3")
    ex.store_basis_operand = regime == "R128r-feat"
    coords, t, y, X, perm = table(n, 0)
    pts = ops.make_points(T(coords), T(t), index=torch.tensor(perm, dtype=torch.int64, device="cuda"),
                          row_begin=ROW_BEGIN, n_rows=n)
    ex.loss_acc.zero_()
    yhat = ex.forward(pts, train=True, step=STEP, seed=SEED, y=T(y),
                      loss=LossSpec(nt.loss, nt.taus or (), nt.nc_weight, 2), inv_count=1.0 / (n * nt.q), save=True,
                      key_offset=KEY_OFFSET).clone()
    grads = ex.backward()
    torch.cuda.synchronize()
    grads = {k: ([g.cpu().numpy() if g is not None else None for g in v] if isinstance(v, list) else v.cpu().numpy())
             for k, v in grads.items()}
    return ex, yhat.cpu().numpy(), ex.loss_acc.item(), grads


# ---------------------------------------------------------------------------------------------------- a. the step
# D3 in TF32 mode.  The support walk keeps the spatial basis and W1's spatial columns in FP32, which the TF32-emulating
# oracle rounds, so the emulation is a different computation (test_gpu_regimes N6).  D3's clustered level puts
# hundreds of knots in a support, and that rounding moves the emulation by more than on N6.  Measured on a B200:
# yhat 7.0e-4 from the emulation (relative L2), gradients up to 2.8e-3 from it (head-block bias).  Against FP64, the
# largest of the 9,435 or 38,888 outputs is 1.1e-3 away and the gradients at most 4.7e-3.  The tf32x3 run of the same
# step is within 2.9e-6 (yhat) and 2.7e-5 (gradients) of FP64, so the kernels themselves are exact.
WALK_TF32_TOL = dict(TF32_TOL, yhat64=2e-3, yhat_emu=1e-3, grad_emu=5e-3)

CASES = ([("D1", r, p) for r in ("R64", "R128x", "R128r") for p in ("tf32", "tf32x3")] + [("D1", "R128r-feat", "tf32")]
         + [("D2", r, p) for r in ("R64", "R128r") for p in ("tf32", "tf32x3")]
         + [("D3", r, "tf32") for r in ("R64", "R128r")] + [("D3", "R128r", "tf32x3")])


@gpu
@pytest.mark.parametrize("name,regime,precision", CASES, ids=["-".join(c) for c in CASES])
def test_large_knot_training_step_vs_oracle(name, regime, precision):
    """yhat, loss and every gradient (D2: knot gradients too) of one gathered training step against the FP64 oracle
    and, in TF32 mode, the TF32-emulating oracle, with the bounds of test_gpu_regimes (TF32_TOL, X3_TOL); the walked
    network D3 in TF32 mode has WALK_TF32_TOL, for the reasons given there.  Largest measured on a B200: D1 and D2 in
    TF32 yhat 9.2e-4 of FP64 and 4.1e-5 of the emulation, gradients 1.7e-3 of FP64 (knot gradients 1.5e-2) and 2.1e-4
    of the emulation; in tf32x3 yhat 3.8e-6 and gradients 2.2e-4 of FP64 (knot gradients 8.8e-4)."""
    n = regime_rows()[regime]
    nt = net(name)
    x3 = precision == "tf32x3"
    (y64, l64, g64), (yemu, lemu, gemu) = oracle(name, n)
    ex, yhat, loss, grads = train_step(name, n, regime, precision)
    errs = {"yhat64": rel_err(yhat, y64), "loss": abs(loss - l64) / abs(l64)}
    if not x3:
        errs["yhat_emu"] = rel_l2(yhat, yemu)
    for gname, g, r64 in _grad_pairs(grads, g64, nt):
        errs[f"{gname}/64"] = rel_err(g, r64)
    if not x3:
        for gname, g, re_ in _grad_pairs(grads, gemu, nt):
            errs[f"{gname}/emu"] = rel_err(g, re_)
    print(f"\n{name} K_s={nt.m.centers.shape[0]} {regime} {precision} n={n}:",
          " ".join(f"{k}={v:.2e}" for k, v in errs.items()))
    tol = X3_TOL if x3 else (WALK_TF32_TOL if name == "D3" else TF32_TOL)
    bad = []
    for k, v in errs.items():
        kind = k if not k.startswith("d") else ("grad_emu" if k.endswith("/emu") else "grad64")
        bound = tol[kind]
        if not v < bound:
            bad.append(f"{k}={v:.3e} (bound {bound:g})")
    assert not bad, bad


# ---------------------------------------------------------------------------------------------------- b. ragged N tiles
def _ragged_n_tiles(n_in):
    """wgrad's split of n_in columns into N tiles (stdadk_wgrad): (tiles, slabs per tile, slabs of the last tile)."""
    a_slabs = (n_in + 31) // 32
    n_tiles_n = -(-a_slabs // 8)
    nt_slabs = -(-a_slabs // n_tiles_n)
    return n_tiles_n, nt_slabs, a_slabs - (n_tiles_n - 1) * nt_slabs


@gpu
@pytest.mark.parametrize("rows", [300, 4096, 20000])
@pytest.mark.parametrize("n_in", [257, 288, 544, 1674])
def test_wgrad_mn_major_ragged_n_tile_exact_tf32(rows, n_in):
    """dW = dz^T A from images (test_wgrad_mn_major_exact_tf32) at widths whose last N tile is shorter than the others:
    257 and 288 columns split 5 + 4 slabs, 544 split 6 + 6 + 5, 1,674 split 7 x 8 + 5.  Operands pre-rounded to TF32,
    so only the FP32 summation order differs: 3e-5 of the largest magnitude."""
    L, ops, *_ = _mods()
    n_tiles_n, nt_slabs, last = _ragged_n_tiles(n_in)
    assert n_tiles_n > 1 and last < nt_slabs, (n_in, n_tiles_n, nt_slabs, last)
    n_out = 256
    rng = np.random.default_rng(rows * 11 + n_in)
    A = orc.tf32_round(rng.standard_normal((rows, n_in)).astype(np.float32))
    dz = orc.tf32_round(rng.standard_normal((rows, n_out)).astype(np.float32))
    a_img, dz_img = ops.pack_image(T(A)), ops.pack_image(T(dz))
    ref = dz.astype(np.float64).T @ A.astype(np.float64)
    for transposed_storage in (False, True):
        dw = torch.zeros(n_in, n_out, device="cuda").t() if transposed_storage else torch.zeros(n_out, n_in, device="cuda")
        a = L.WgradArgs()
        a.pts = ops.make_points(grid=None, coords=None, t=None, row_begin=0, n_rows=rows)
        a.a_img, a.dz_img = a_img.data_ptr(), dz_img.data_ptr()
        a.n_in, a.n_out = n_in, n_out
        a.dw, a.stride_o, a.stride_i = dw.data_ptr(), dw.stride(0), dw.stride(1)
        ops.wgrad(a)
        err = np.max(np.abs(dw.cpu().numpy() - ref)) / max(1.0, np.abs(ref).max())
        assert err < 3e-5, (transposed_storage, err)


def _generated_operand(ops, L, basis, pts, rows, n_in):
    """The block-1 operand the forward generates (feat_img of a throwaway 32-wide block), unpacked."""
    rng = np.random.default_rng(n_in)
    w_img = ops.pack_image(T(rng.standard_normal((32, n_in)).astype(np.float32)))
    out, feat = ops.new_image(rows, 32, "cuda"), ops.new_image(rows, n_in, "cuda")
    a = L.FwdArgs()
    a.basis = C.pointer(basis)
    a.pts = pts
    a.layer = ops.make_layer(w_img, torch.zeros(32, device="cuda"), None, None, n_in, 32, 1e-5, 0)
    a.drop = L.Dropout(0.0, 0, 0)
    a.out_img, a.feat_img = out.data_ptr(), feat.data_ptr()
    ops.layer_fwd(a)
    return ops.unpack_image(feat, rows, n_in).cpu().numpy()


@gpu
@pytest.mark.parametrize("rows", [4096, 20000])
def test_wgrad_basis_form_ragged_n_tile_exact_tf32(rows):
    """Block 1's wgrad regenerating D1's basis (1,604 lattice knots + 70 temporal = 1,674 columns, N tiles 7 x 8 + 5)
    for every row tile it walks.  Reference: dz^T A with A the operand the forward generates, itself checked against
    orc.features (test_wgrad_basis_operand_exact_tf32).  3e-5 of the largest magnitude."""
    L, ops, *_ = _mods()
    m = net("D1").m
    k_s, k_t = m.centers.shape[0], m.t_centers.shape[0]
    n_in, n_out = k_s + k_t, 256
    n_tiles_n, nt_slabs, last = _ragged_n_tiles(n_in)
    assert (n_tiles_n, nt_slabs, last) == (7, 8, 5)
    knots4 = ops.knots_prepare(T(m.centers), T(m.bandwidths), None, "wendland")
    tk = ops.tknots_prepare(T(m.t_centers), T(m.t_bandwidths))
    basis = ops.make_basis(knots4, tk, k_s, k_t, 0, "wendland")
    rng = np.random.default_rng(rows + 1)
    coords = rng.random((rows, 2)).astype(np.float32)
    t = rng.random((rows, 1)).astype(np.float32)
    pts = ops.make_points(T(coords), T(t))
    A = _generated_operand(ops, L, basis, pts, rows, n_in)
    a64 = orc.features(m, None, coords, t)
    assert np.array_equal(A, orc.tf32_round(A))
    assert np.all(np.abs(A - a64) <= 2.0 ** -11 * 1.001 * np.abs(a64) + 1e-5 * np.maximum(a64, 1e-2))
    dz = orc.tf32_round(rng.standard_normal((rows, n_out)).astype(np.float32))
    dz_img = ops.pack_image(T(dz))
    ref = dz.astype(np.float64).T @ A.astype(np.float64)
    for transposed_storage in (False, True):
        dw = torch.zeros(n_in, n_out, device="cuda").t() if transposed_storage else torch.zeros(n_out, n_in, device="cuda")
        w = L.WgradArgs()
        w.basis = C.pointer(basis)
        w.pts = pts
        w.dz_img = dz_img.data_ptr()
        w.n_in, w.n_out = n_in, n_out
        w.dw, w.stride_o, w.stride_i = dw.data_ptr(), dw.stride(0), dw.stride(1)
        ops.wgrad(w)
        err = np.max(np.abs(dw.cpu().numpy() - ref)) / max(1.0, np.abs(ref).max())
        print(f"\nwgrad basis form rows={rows} {n_in}x{n_out} transposed={transposed_storage}: {err:.2e}")
        assert err < 3e-5


# ---------------------------------------------------------------------------------------------------- c. dispatch
@gpu
def test_d1_step_runs_the_intended_kernels():
    """One D1 step per regime under torch.profiler (as test_sizes_run_the_intended_kernels): the layer_fwd_kernel /
    layer_bwd_kernel instantiation of every block at 1,604 knots, and what the workspace keeps."""
    from torch.profiler import ProfilerActivity, profile
    rows = regime_rows()
    for regime in ("R64", "R128x", "R128r", "R128r-feat"):
        fwd, bwd_tm, regen, has_x, has_feat = EXPECTED[regime]
        n = rows[regime]
        train_step("D1", n, regime)
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            ex, *_ = train_step("D1", n, regime)
        kern = sorted((e for e in prof.events() if "DeviceType.CUDA" in str(getattr(e, "device_type", ""))),
                      key=lambda e: e.time_range.start)
        if not kern:
            pytest.skip("the profiler recorded no CUDA kernels (CUPTI unavailable): the instantiations cannot be read")
        fw = [_template_args(e.name, "layer_fwd_kernel") for e in kern if "layer_fwd_kernel" in e.name]
        bw = [_template_args(e.name, "layer_bwd_kernel") for e in kern if "layer_bwd_kernel" in e.name]
        print(f"\nD1 {regime} n={n}: layer_fwd {fw}; layer_bwd {bw}")
        assert fw == [(1, *fwd), (0, *fwd), (0, *fwd)], (regime, fw)
        assert bw == [(0, bwd_tm, 2, 4, 1, 1), (0, bwd_tm, 2, 4, 1, 0), (int(regen), bwd_tm, 2, 4, 1, 0)], (regime, bw)
        ws = ex._ctx[2]
        assert (ws.x is not None) == has_x and (ws.feat is not None) == has_feat, regime


def _block1_launches(ops, L, k_s, k_t_levels, n_out, rows_cg2):
    """Block 1 with k_s scattered knots through every dense launch: layer_fwd with 4 column groups (1,000 rows) and 2
    (rows_cg2 rows), the recompute layer_bwd and the basis-form wgrad (1,000 rows).  Returns {launch: error or None};
    the launches that ran are checked against the FP64 reference."""
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
    w_img, tbias = ops.pack_image(T(W)), T(bias)
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

    for name, n in (("fwd_cg4", rows), ("fwd_cg2", rows_cg2)):
        co, tt, pts = pts_of(n)
        out = ops.new_image(n, n_out, "cuda")

        def fwd():
            a = L.FwdArgs()
            a.basis = C.pointer(basis)
            a.pts = pts
            a.layer = layer
            a.drop = L.Dropout(0.0, 0, 0)
            a.out_img = out.data_ptr()
            ops.layer_fwd(a)
        attempt(name, fwd)
        if errs[name] is None:
            idx = np.r_[0:1000, n - 1000:n]
            got = ops.unpack_image(out, n, n_out).cpu().numpy()[idx]
            ref = np.maximum(z_ref(co[idx], tt[idx])[1], 0.0)
            assert rel_l2(got, ref) < 2e-3, (name, rel_l2(got, ref))

    co, tt, pts = pts_of(rows)
    n_next = 32
    Wn = orc.tf32_round((rng.standard_normal((n_next, n_out)) / 6).astype(np.float32))
    dzn = orc.tf32_round(rng.standard_normal((rows, n_next)).astype(np.float32))
    wt_next, dzn_img = ops.pack_image(T(Wn).t()), ops.pack_image(T(dzn))
    dz_img, d_bias = ops.new_image(rows, n_out, "cuda"), torch.zeros(n_out, device="cuda")

    def bwd():
        a = L.BwdArgs()
        a.basis = C.pointer(basis)
        a.pts = pts
        a.layer = layer
        a.drop = L.Dropout(0.0, 0, 0)
        a.dz_next_img, a.wt_next_img, a.n_next = dzn_img.data_ptr(), wt_next.data_ptr(), n_next
        a.dz_img, a.d_bias = dz_img.data_ptr(), d_bias.data_ptr()
        ops.layer_bwd(a)
    attempt("bwd_recompute", bwd)
    A64, z64 = z_ref(co, tt)
    if errs["bwd_recompute"] is None:
        # dz = (dz_next W_next) * relu'(z), z recomputed from the TF32-rounded operand.  Products of the TF32 operands
        # are exact, the dz image is TF32-rounded.  Entries with |z| < 1e-3 are skipped: there the generated basis
        # (FP32, then rounded) may differ from the rounded FP64 basis by one TF32 ulp and flip the ReLU.
        z_emu = orc.tf32_round(A64.astype(np.float32)).astype(np.float64) @ W.astype(np.float64).T + bias
        ref = (dzn.astype(np.float64) @ Wn.astype(np.float64)) * (z_emu > 0)
        got = ops.unpack_image(dz_img, rows, n_out).cpu().numpy()
        keep = np.abs(z_emu) >= 1e-3
        assert keep.mean() > 0.99
        bad = np.abs(got - ref)[keep] > 2.0 ** -10 * np.abs(ref)[keep] + 1e-5 * np.abs(ref).max()
        assert not bad.any(), int(bad.sum())

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
        ref = dz.astype(np.float64).T @ A64
        assert rel_err(dw.cpu().numpy(), ref) < 2e-3, rel_err(dw.cpu().numpy(), ref)
    return errs


CAPACITY = [(w, kt) for w in (256, 128, 64) for kt in ((10, 15, 45), (10, 15))]


@gpu
@pytest.mark.parametrize("n_out,k_t_levels", CAPACITY, ids=[f"w{w}-kt{sum(k)}" for w, k in CAPACITY])
def test_capacity_query_equals_the_launch_checks(n_out, k_t_levels):
    """At the K_s stdadk_dense_max_knots reports, every dense block-1 launch runs (and matches the FP64 reference); at
    K_s + 1 the launch the query names returns its shared-memory error.  So the query and the launchers agree."""
    L, ops, *_ = _mods()
    k_t = sum(k_t_levels)
    K = ops.dense_max_knots(0, k_t, n_out, 0)
    S = torch.cuda.get_device_properties(0).multi_processor_count
    rows_cg2 = 2 * S * 128                      # at least two tiles per SM: 2 column groups
    at_k = _block1_launches(ops, L, K, k_t_levels, n_out, rows_cg2)
    assert all(v is None for v in at_k.values()), at_k
    fits, why = ops.dense_basis_supported(0, K + 1, k_t, n_out, 0)
    assert not fits
    above = _block1_launches(ops, L, K + 1, k_t_levels, n_out, rows_cg2)
    print(f"\nwidth {n_out}, {k_t} temporal knots: K = {K}; at K + 1 the query says {why!r}; launches {above}")
    failed = [v for v in above.values() if v is not None]
    assert failed and any(why in v for v in failed), (why, above)
    fwd_ran = above["fwd_cg4"] is None and above["fwd_cg2"] is None
    assert fwd_ran == ops.dense_basis_supported(0, K + 1, k_t, n_out, 0, training=False)[0]


@gpu
@pytest.mark.parametrize("n_out,k_t_levels", CAPACITY, ids=[f"w{w}-kt{sum(k)}" for w, k in CAPACITY])
def test_executor_regime_at_the_capacity(n_out, k_t_levels):
    """Wendland knots at the capacity K and K + 1: dense at K when K <= DENSE_MAX_KNOTS, walked otherwise; Gaussian and
    covariate models are dense while they fit, and above it raise at construction naming the limit."""
    L, ops, Executor, NetSpec, LossSpec = _mods()
    k_t = sum(k_t_levels)
    K = ops.dense_max_knots(0, k_t, n_out, 0)
    for k_s in (K, K + 1):
        rng = np.random.default_rng(k_s)
        c, b = _scattered_knots(rng, [k_s])
        m = _model(rng, c, b, list(k_t_levels), (n_out, 32))
        spec = spec_from_oracle(m)
        spec.level_sizes = [k_s]
        ex = Executor(spec)
        assert ex.sparse == (k_s > K or k_s > Executor.DENSE_MAX_KNOTS), (k_s, ex.sparse)
        if k_s > K:
            # forced dense above the training limit: predicts (the forward fits) and agrees with the walk, but refuses
            # a training forward before launching anything
            exd = Executor(spec_from_oracle(m), force_dense=True)
            assert not exd.sparse and exd.predict_only
            rng_p = np.random.default_rng(3)
            pts = ops.make_points(T(rng_p.random((700, 2)).astype(np.float32)),
                                  T(rng_p.random((700, 1)).astype(np.float32)))
            yd, yw = exd.forward(pts, train=False).clone(), ex.forward(pts, train=False).clone()
            assert rel_l2(yd.cpu().numpy(), yw.cpu().numpy()) < 1e-3
            with pytest.raises(RuntimeError, match=f"can be predicted but not trained.*at most {K} spatial knots"):
                exd.forward(pts, train=True, save=True)
        m.basis_fn = "gaussian"
        if k_s == K:
            assert not Executor(spec_from_oracle(m)).sparse
        else:
            with pytest.raises(RuntimeError, match=f"at most {K} spatial knots.*gaussian"):
                Executor(spec_from_oracle(m))
    # covariates: three columns in front of the basis widen layer_fwd / layer_bwd's tables (wgrad's are per knot)
    Kp = ops.dense_max_knots(3, k_t, n_out, 0)
    assert Kp < K if n_out == 256 else Kp == K
    for k_s in (Kp, Kp + 1):
        rng = np.random.default_rng(k_s)
        c, b = _scattered_knots(rng, [k_s])
        m = _model(rng, c, b, list(k_t_levels), (n_out, 32))
        m.p = 3
        m.weights[0] = np.concatenate([rng.standard_normal((n_out, 3)).astype(np.float32) / 6, m.weights[0]], axis=1)
        if k_s == Kp:
            assert not Executor(spec_from_oracle(m)).sparse
        else:
            with pytest.raises(RuntimeError, match=f"at most {Kp} spatial knots.*covariates"):
                Executor(spec_from_oracle(m))


def test_regime_rule_raises_at_construction_without_a_gpu():
    """The regime rule runs on the host before any launch: a Gaussian model above what the dense kernels hold, and
    force_dense above what the dense forward holds, raise when the executor is built, naming the knot count, the limit
    and the launch."""
    ops = _ops()
    from st_dadk_b200.executor import Executor
    K = ops.dense_max_knots(0, 70, 256, 0)
    fits, why = ops.dense_basis_supported(0, K + 1, 70, 256, 0)
    assert ops.dense_basis_supported(0, K, 70, 256, 0) == (True, "") and not fits and "layer_bwd" in why
    rng = np.random.default_rng(5)
    c, b = _scattered_knots(rng, [K + 1])
    m = _model(rng, c, b, [10, 15, 45], (256, 64))

    def spec(**kw):
        s = spec_from_oracle_cpu(m)
        for k, v in kw.items():
            setattr(s, k, v)
        return s

    with pytest.raises(RuntimeError, match=f"{K + 1} spatial knots.*at most {K} spatial knots.*layer_bwd.*gaussian"):
        Executor(spec(basis_fn="gaussian"))
    # force_dense: above the training limit the regime rule passes (prediction only) and construction goes on to the
    # device check; above the forward's limit it raises, naming that limit
    with pytest.raises(RuntimeError, match="needs CUDA tensors"):
        Executor(spec(), force_dense=True)
    F = ops.dense_max_knots(0, 70, 256, 0, training=False)
    assert F > K and ops.dense_basis_supported(0, F, 70, 256, 0, training=False) == (True, "")
    c, b = _scattered_knots(rng, [F + 1])
    m = _model(rng, c, b, [10, 15, 45], (256, 64))
    with pytest.raises(RuntimeError,
                       match=f"force_dense: {F + 1} spatial knots do not fit.*forward holds at most {F}.*layer_fwd"):
        Executor(spec(), force_dense=True)
    # a single hidden block carries the head: its bytes lower the limit
    assert ops.dense_max_knots(0, 70, 256, 8) < ops.dense_max_knots(0, 70, 256, 1) < K


def spec_from_oracle_cpu(m):
    """NetSpec of an oracle model on CPU tensors: enough for the regime rule, which runs before the device check."""
    from st_dadk_b200.executor import NetSpec
    t = lambda a: torch.tensor(np.ascontiguousarray(a), dtype=torch.float32)
    Wh, bh = m.head(np.float64)
    nh = len(m.ln_gamma)
    return NetSpec(centers=t(m.centers), bandwidths=t(m.bandwidths), log_bandwidths=None, t_centers=t(m.t_centers),
                   t_bandwidths=t(m.t_bandwidths), weights=[t(w) for w in m.weights[:nh]],
                   biases=[t(b) for b in m.biases[:nh]], gammas=[t(g) for g in m.ln_gamma],
                   betas=[t(b) for b in m.ln_beta], head_w=t(Wh), head_b=t(bh), basis_fn=m.basis_fn, p_cov=m.p)


# ---------------------------------------------------------------------------------------------------- d. prediction
def _fused_capacity(L, hidden, k_t, q):
    """Largest K_s stdadk_predict_supported accepts for this network (host-side shape check; the pointers it is given
    are placeholders, it reads none of them)."""
    ptr = 1 << 12

    def ok(k_s):
        basis = L.Basis(ptr, ptr, k_s, k_t, 0, L.WENDLAND)
        head = L.Head()
        head.w, head.b, head.yhat, head.q = ptr, ptr, ptr, q
        a = L.PredictArgs()
        a.basis = C.pointer(basis)
        a.pts.grid_nx, a.pts.grid_ny, a.pts.grid_nt, a.pts.n_rows = 1, 1, 1, 1
        a.n_layers = len(hidden)
        dims = [k_s + k_t, *hidden]
        for l in range(len(hidden)):
            a.layers[l] = L.Layer(ptr, ptr, ptr, ptr, dims[l], dims[l + 1], 1e-5, l, None)
        a.head = C.pointer(head)
        return bool(L.lib().stdadk_predict_supported(C.byref(a)))

    assert ok(1) and not ok(1 << 14)
    lo, hi = 1, 1 << 14
    while hi - lo > 1:
        mid = (lo + hi) // 2
        lo, hi = (mid, hi) if ok(mid) else (lo, mid)
    return lo


@gpu
def test_fused_prediction_falls_back_above_its_capacity():
    """The whole-network kernel at the largest K_s it takes and one knot above: _fused_ok flips, both outputs are
    within 1e-3 of the FP64 oracle, and at the capacity the fused and layered outputs agree to 2e-4 (one TF32 pass each,
    FP32 sums in different orders)."""
    L, ops, Executor, NetSpec, LossSpec = _mods()
    hidden = (256, 256, 128)
    cap = _fused_capacity(L, hidden, 70, 1)
    rng = np.random.default_rng(81)
    n = 5000
    coords, t = rng.random((n, 2)).astype(np.float32), rng.random((n, 1)).astype(np.float32)
    pts = ops.make_points(T(coords), T(t))
    for k_s in (cap, cap + 1):
        c, b = _scattered_knots(np.random.default_rng(k_s), [k_s // 3, k_s - k_s // 3])
        m = _model(rng, c, b, [10, 15, 45], hidden)
        ex = Executor(spec_from_oracle(m))
        assert not ex.sparse
        out = ex.forward(pts, train=False).clone()
        assert ex._fused_ok is (k_s == cap), (k_s, ex._fused_ok)
        ex.fused_predict = False
        layered = ex.forward(pts, train=False).clone()
        torch.cuda.synchronize()
        ref = orc.forward(m, None, coords, t)
        e_out, e_lay = rel_l2(out.cpu().numpy(), ref), rel_l2(layered.cpu().numpy(), ref)
        print(f"\nK_s={k_s} (capacity {cap}) fused={ex._fused_ok}: vs oracle {e_out:.2e}, layered vs oracle {e_lay:.2e}")
        assert e_out < 1e-3 and e_lay < 1e-3
        if k_s == cap:
            assert rel_l2(out.cpu().numpy(), layered.cpu().numpy()) < 2e-4
        else:
            assert torch.equal(out, layered)        # the fallback is the layered path


@gpu
@pytest.mark.parametrize("levels", [[256], [49, 64, 144]], ids=["256", "257"])
def test_field_kernel_falls_back_above_256_knots(levels):
    """Predictor.space_time_field / grid at 256 knots (8 slabs, the field kernel's resident operand) and 257: the field
    kernel runs at 256 only; both paths match the oracle (1e-3) and shard by site bit for bit."""
    from stnf.models import STInterpMLP
    from st_dadk_b200.predict import Predictor
    from test_gpu_field import _oracle
    from test_gpu_model import _perturb_ln
    torch.manual_seed(9)
    model = STInterpMLP(k_spatial_centers=levels, hidden_dims=[256, 256, 128], dropout=0.0, output_dim=2)
    _perturb_ln(model, 9)
    model = model.to("cuda").eval()
    field_kernel = sum(levels) <= 256
    S, nt = 300, 4
    sites = torch.rand(S, 2, generator=torch.Generator().manual_seed(2)).to("cuda")
    pr = Predictor(model)
    field, _ = pr.space_time_field(sites, nt)
    assert pr.used_field_kernel == field_kernel
    coords = sites.repeat(nt, 1).cpu().numpy()
    t = (torch.arange(nt).repeat_interleave(S).float() / (nt - 1)).numpy()[:, None]
    err = rel_l2(field.cpu().numpy(), _oracle(model, coords, t))
    print(f"\n{sum(levels)} knots, field kernel {pr.used_field_kernel}: vs oracle {err:.2e}")
    assert err < 1e-3
    parts = [pr.space_time_field_by_sites(sites, nt, r, 3)[0] for r in range(3)]
    assert pr.used_field_kernel == field_kernel
    assert torch.equal(torch.cat(parts, dim=1), field.view(nt, S, 2))
    nx, ny = 23, 17
    grid, _ = pr.grid(nx, ny, nt)
    assert pr.used_field_kernel == field_kernel
    gc, gt = orc.grid_points(nx, ny, nt, 0, nx * ny * nt)
    assert rel_l2(grid.cpu().numpy(), _oracle(model, gc, gt)) < 1e-3
    parts = [pr.grid_by_sites(nx, ny, nt, r, 3)[0] for r in range(3)]
    assert torch.equal(torch.cat(parts, dim=1), grid.view(nt, nx * ny, 2))
