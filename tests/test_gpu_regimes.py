"""One training step against the oracle in every row-tile regime of layer_fwd / layer_bwd, not only on 64-row tiles.

stdadk_layer_fwd / stdadk_layer_bwd choose the kernel instantiation from the batch's row count, and Executor._workspace
(SAVE_X_MAX_ROWS, store_basis_operand) decides what the backward reads.  With S SMs and t = ceil(rows / 128):
  * 2 t <= S:               64-row tiles (pairs of CTAs per 128-row image tile), x saved, 64-row backward;
  * 2 t > S, t < 2 S:       128-row tiles, 4 column groups, x saved;
  * t >= 2 S, x saved:      128-row tiles, 2 column groups (up to SAVE_X_MAX_ROWS rows);
  * rows > SAVE_X_MAX_ROWS: 128-row tiles, 2 column groups, the backward recomputes x (block 1 regenerates the basis, or
                            reads the stored operand with store_basis_operand).
Each case runs one forward(train, save) + backward with the points gathered through a permutation of a larger table,
row_begin != 0 and a dropout key offset != row_begin (the form of every trainer step), against an oracle evaluated in
chunks of rows (every forward step is row-local, every gradient a sum over rows)."""
import re
from functools import lru_cache

import numpy as np
import pytest
import torch

from helpers import golden, orc
from test_gpu_kernels import T, _cell_list_knots, _default_oracle_model, _mods, _small_net, rel_err, rel_l2, \
    spec_from_oracle

gpu = pytest.mark.gpu

SEED, STEP, P_DROP = 0x1234567890ABCDEF, 17, 0.1
CHUNK = 8192
TABLE_EXTRA, ROW_BEGIN = 3001, 1717        # table rows beyond the batch; the batch is perm[ROW_BEGIN : ROW_BEGIN + n]
KEY_OFFSET = 2 ** 32 - 3000                 # dropout key of row 0: the keys cross into the high word inside the batch


def regime_rows():
    """Row count of each regime from the device's SM count S and Executor.SAVE_X_MAX_ROWS."""
    L, ops, Executor, NetSpec, LossSpec = _mods()
    S = torch.cuda.get_device_properties(0).multi_processor_count
    save = Executor.SAVE_X_MAX_ROWS
    return {"R64": 128 * (S // 2) - 37,                 # largest 64-row batch minus 37: ragged
            "R128x": 12345,                             # 97 tiles: 128-row, 4 column groups, x saved
            "R128x-cg2": 128 * (2 * S - 1) + 5,         # 2 S - 1 full tiles + 5 rows: 2 column groups, x saved
            "R128r": save + 1000,                       # recompute backward, block 1 regenerates the basis
            "R128r-feat": save + 1000,                  # recompute backward, block 1 reads the stored operand
            "R65536": 65536}                            # the bench's large batch


def _rows(regime):
    rows = regime_rows()
    n = rows[regime]
    if regime == "R128x-cg2":
        L, ops, Executor, NetSpec, LossSpec = _mods()
        if n > Executor.SAVE_X_MAX_ROWS:
            pytest.skip(f"{n} rows (2 column groups on this device's SM count) exceed SAVE_X_MAX_ROWS = "
                        f"{Executor.SAVE_X_MAX_ROWS}: this device has no 2-column-group regime with x saved")
    return n


# ---------------------------------------------------------------------------------------------------- networks
class Net:
    def __init__(self, m, loss="mse", taus=None, nc_weight=0.0, learnable=False, sizes=None):
        self.m, self.loss, self.taus, self.nc_weight, self.learnable, self.sizes = m, loss, taus, nc_weight, learnable, sizes

    @property
    def q(self):
        return len(self.m.delta) if self.m.delta is not None else self.m.weights[-1].shape[0]

    def nc_power(self, regime):
        # N2 takes the linear penalty in the one regime of its own (its row count is not shared with another regime)
        return 1 if regime == "R128x-cg2" else 2


@lru_cache(maxsize=None)
def net(name):
    if name == "N1":        # the bench's step: default widths, MSE, dropout
        m = _default_oracle_model(51)
        m.dropout = P_DROP
        return Net(m)
    if name == "N2":        # STDADK_MAX_Q quantiles with the non-crossing penalty; 160 / 96 columns = 5 / 3 chunks of 32
        m = _default_oracle_model(52, q=8, hidden=(256, 160, 96))
        m.dropout = P_DROP
        return Net(m, "pinball", tuple(np.linspace(0.05, 0.95, 8)), nc_weight=0.5)
    if name == "N3":        # learnable dense knots
        return Net(_default_oracle_model(53, q=3, hidden=(128, 64)), "pinball", (0.1, 0.5, 0.9), learnable=True)
    if name == "N4":        # no LayerNorm, triangular basis, 3 covariates in front of the basis columns, 16-wide last block
        kn = golden("knots")
        rng = np.random.default_rng(54)
        p, hidden, q = 3, (96, 48, 16), 2
        dims = [p + kn["centers"].shape[0] + kn["t_centers"].shape[0], *hidden]
        ws = [rng.uniform(-1, 1, (dims[i + 1], dims[i])).astype(np.float32) / np.float32(np.sqrt(dims[i]))
              for i in range(len(hidden))]
        bs = [rng.uniform(-0.1, 0.1, dims[i + 1]).astype(np.float32) for i in range(len(hidden))]
        ws.append(rng.uniform(-0.25, 0.25, (q, dims[-1])).astype(np.float32))
        bs.append(rng.uniform(-0.1, 0.1, q).astype(np.float32))
        m = orc.OracleModel(centers=kn["centers"], bandwidths=kn["bandwidths"], t_centers=kn["t_centers"],
                            t_bandwidths=kn["t_bandwidths"], weights=ws, biases=bs, ln_gamma=[None] * 3,
                            ln_beta=[None] * 3, basis_fn="triangular", p=p)
        return Net(m, "pinball", (0.3, 0.7))
    if name == "N5":        # Gaussian basis: no compact support anywhere
        return Net(_default_oracle_model(55, fn="gaussian", hidden=(256, 256)))
    if name == "N6":        # support walk over the cell list of a non-lattice knot set (config 4's path)
        rng = np.random.default_rng(33)
        c, b, sizes = _cell_list_knots(rng)
        tc, tb = orc.temporal_knots([10, 15])
        ws, bs, gs, be = _small_net(rng, c.shape[0])
        m = orc.OracleModel(centers=c, bandwidths=b, t_centers=tc, t_bandwidths=tb, weights=ws, biases=bs, ln_gamma=gs,
                            ln_beta=be, basis_fn="wendland")
        return Net(m, learnable=True, sizes=sizes)
    raise KeyError(name)


@lru_cache(maxsize=None)
def table(n, p):
    """Sample table of n + TABLE_EXTRA rows and a permutation of it; the batch is perm[ROW_BEGIN : ROW_BEGIN + n]."""
    rng = np.random.default_rng(n)
    N = n + TABLE_EXTRA
    coords = rng.random((N, 2)).astype(np.float32)
    t = (rng.integers(0, 100, (N, 1)) / 99.0).astype(np.float32)
    y = rng.standard_normal(N).astype(np.float32)
    X = rng.standard_normal((N, p)).astype(np.float32) if p else None
    perm = rng.permutation(N)
    return coords, t, y, X, perm


# ---------------------------------------------------------------------------------------------------- chunked oracle
def _add(a, b):
    if a is None:
        return b
    if isinstance(a, list):
        return [_add(x, y) for x, y in zip(a, b)]
    if isinstance(a, dict):
        return {k: _add(a[k], b[k]) for k in a}
    return a + b


def chunked_oracle(m, X, coords, t, y, loss="mse", taus=None, nc_weight=0.0, nc_power=1, key_offset=0,
                   knot_grads=False, rnd=None, chunk=CHUNK, seed=SEED, step=STEP):
    """(yhat, loss, gradients) of one training step, memory bounded by `chunk` rows: forward per chunk (dropout masks
    of `seed` and `step` keyed from key_offset + chunk start), the loss and dL/dyhat once over all rows (its 1/(n Q) and
    the non-crossing term see the whole batch), then per chunk a forward again and the backward of its slice of
    dL/dyhat, summed."""
    n = coords.shape[0]
    hidden = m.weights[:len(m.ln_gamma)]
    spans = [(lo, min(lo + chunk, n)) for lo in range(0, n, chunk)]

    def fwd(lo, hi, **kw):
        masks = [orc.dropout_keep_mask(hi - lo, w.shape[0], m.dropout, seed, step, l, key_offset + lo)
                 for l, w in enumerate(hidden)]
        return orc.forward(m, None if X is None else X[lo:hi], coords[lo:hi], t[lo:hi], train=True, keep_masks=masks,
                           rnd=rnd, **kw)

    yhat = np.concatenate([fwd(lo, hi) for lo, hi in spans])
    lval, dy = orc.loss_and_grad(yhat, y, loss, taus, nc_weight, nc_power)
    g = None
    for lo, hi in spans:
        _, cache = fwd(lo, hi, return_cache=True)
        g = _add(g, orc.backward(m, cache, dy[lo:hi], coords=coords[lo:hi], want_knot_grads=knot_grads))
    return yhat, lval, g


def test_chunked_oracle_matches_whole_batch():
    """The chunked oracle (3 chunks of at most 1,024 rows, the last ragged) against one whole-batch evaluation of 3,001
    rows: dropout, Q = 3 pinball with the quadratic non-crossing penalty, knot gradients, in FP64 and with the TF32
    operand rounding emulated.  Only the order of the row sums differs: 1e-12."""
    m = _default_oracle_model(61, q=3, hidden=(64, 32))
    m.dropout = P_DROP
    n, k0 = 3001, 12345
    rng = np.random.default_rng(62)
    coords = rng.random((n, 2)).astype(np.float32)
    t = rng.random((n, 1)).astype(np.float32)
    y = rng.standard_normal(n).astype(np.float32)
    taus = (0.2, 0.5, 0.8)
    for rnd in (None, orc.tf32_round):
        masks = [orc.dropout_keep_mask(n, w.shape[0], P_DROP, SEED, STEP, l, k0) for l, w in enumerate(m.weights[:-1])]
        yw, cache = orc.forward(m, None, coords, t, train=True, keep_masks=masks, return_cache=True, rnd=rnd)
        lw, dy = orc.loss_and_grad(yw, y, "pinball", taus, 0.5, 2)
        gw = orc.backward(m, cache, dy, coords=coords, want_knot_grads=True)
        yc, lc, gc = chunked_oracle(m, None, coords, t, y, "pinball", taus, 0.5, 2, key_offset=k0, knot_grads=True,
                                    rnd=rnd, chunk=1024)
        assert rel_err(yc, yw) < 1e-12
        assert abs(lc - lw) <= 1e-12 * abs(lw)
        pairs = [(a, b) for k in ("weights", "biases", "ln_gamma", "ln_beta") for a, b in zip(gc[k], gw[k])]
        pairs += [(gc["centers"], gw["centers"]), (gc["log_bandwidths"], gw["log_bandwidths"])]
        for a, b in pairs:
            assert rel_err(a, b) < 1e-12


_ORACLE = {}


def _as_net(nt):
    """A Net, or the name of one in the net() registry."""
    return net(nt) if isinstance(nt, str) else nt


def oracle(nt, n, regime):
    """FP64 and TF32-emulating oracle results of network `nt` (a Net or a registry name) on the batch of n rows, shared
    by both precisions."""
    nt = _as_net(nt)
    key = (nt, n, nt.nc_power(regime))
    if key not in _ORACLE:
        coords, t, y, X, perm = table(n, nt.m.p)
        idx = perm[ROW_BEGIN:ROW_BEGIN + n]
        args = (nt.m, None if X is None else X[idx], coords[idx], t[idx], y[idx], nt.loss, nt.taus, nt.nc_weight,
                nt.nc_power(regime))
        kw = dict(key_offset=KEY_OFFSET, knot_grads=nt.learnable)
        _ORACLE[key] = (chunked_oracle(*args, **kw), chunked_oracle(*args, rnd=orc.tf32_round, **kw))
    return _ORACLE[key]


# ---------------------------------------------------------------------------------------------------- one step
def train_step(nt, n, regime, precision="tf32"):
    """forward(train, save) + backward of network `nt` (a Net or a registry name) on n gathered rows; returns
    (executor, yhat, loss, grads)."""
    L, ops, Executor, NetSpec, LossSpec = _mods()
    nt = _as_net(nt)
    spec = spec_from_oracle(nt.m, learnable=nt.learnable, dropout=nt.m.dropout, precision=precision)
    if nt.sizes is not None:
        spec.level_sizes = nt.sizes
    ex = Executor(spec, force_sparse=nt.sizes is not None)
    assert ex.sparse == (nt.sizes is not None)
    ex.store_basis_operand = regime == "R128r-feat"
    coords, t, y, X, perm = table(n, nt.m.p)
    pts = ops.make_points(T(coords), T(t), T(X) if X is not None else None,
                          index=torch.tensor(perm, dtype=torch.int64, device="cuda"), row_begin=ROW_BEGIN, n_rows=n)
    ex.loss_acc.zero_()
    yhat = ex.forward(pts, train=True, step=STEP, seed=SEED, y=T(y),
                      loss=LossSpec(nt.loss, nt.taus or (), nt.nc_weight, nt.nc_power(regime)),
                      inv_count=1.0 / (n * nt.q), save=True, key_offset=KEY_OFFSET).clone()
    grads = ex.backward()
    torch.cuda.synchronize()
    grads = {k: ([g.cpu().numpy() if g is not None else None for g in v] if isinstance(v, list) else v.cpu().numpy())
             for k, v in grads.items()}
    return ex, yhat.cpu().numpy(), ex.loss_acc.item(), grads


def _grad_pairs(grads, ref, nt):
    """(name, kernel gradient, oracle gradient) of every parameter of the network."""
    out = []
    for l in range(len(nt.m.ln_gamma)):
        out += [(f"dW{l}", grads["weights"][l], ref["weights"][l]), (f"db{l}", grads["biases"][l], ref["biases"][l])]
        if nt.m.ln_gamma[l] is not None:
            out += [(f"dgamma{l}", grads["gammas"][l], ref["ln_gamma"][l]),
                    (f"dbeta{l}", grads["betas"][l], ref["ln_beta"][l])]
    if nt.m.delta is not None:
        # the kernels give the effective head's gradient; d delta_l = sum_{k >= l} [d head_b | d head_w]_k
        dbeta = np.concatenate([grads["head_b"][:, None], grads["head_w"]], axis=1)
        out.append(("ddelta", np.cumsum(dbeta[::-1], axis=0)[::-1], np.stack(ref["delta"])))
    else:
        out += [("dhead_w", grads["head_w"], ref["weights"][-1]), ("dhead_b", grads["head_b"], ref["biases"][-1])]
    if nt.learnable:
        out += [("dcenters", grads["centers"], ref["centers"]),
                ("dlog_bw", grads["log_bandwidths"], ref["log_bandwidths"])]
    return out


# ---------------------------------------------------------------------------------------------------- the matrix
TF32_TOL = {"yhat64": 1e-3, "yhat_emu": 2e-4, "loss": 1e-3, "grad_emu": 3e-3, "grad64": 2e-2}
X3_TOL = {"yhat64": 2e-5, "loss": 1e-5, "grad64": 1e-3}
# TF32 mode only; the tf32x3 runs of the same networks meet the common bounds (N6: knot gradients 8.8e-5).
TF32_EXCEPTIONS = {
    # Q = 1: d head_b = 2 mean(yhat - y), here -5.8e-3 against a mean |residual| of 0.82.  TF32 rounding of the Gaussian
    # basis shifts yhat by -6.6e-5 on average, so the TF32-emulating oracle is itself 2.3e-2 from FP64.
    # Measured (B200) 2.28e-2 from FP64 and 3.8e-5 from the emulation.
    ("N5", "dhead_b/64"): 3e-2,
    # The support walk keeps the spatial basis and W1's spatial columns in FP32.  The emulation rounds them to TF32,
    # so on N6 it is a different computation: measured yhat 4.0e-4 (relative L2), d centres 2.2e-2, d log-bandwidths
    # 3.8e-3.  Knot gradients are sums of large cancelling terms.  Rounding the dz image to TF32 alone puts the
    # emulating oracle 1.9e-2 from FP64 on d centres.  The kernel is measured 2.2e-2 from FP64
    # (test_cell_list_regime_arbitrary_and_learnable_knots_vs_oracle allows 2e-1 at 600 rows).
    ("N6", "yhat_emu"): 1e-3,
    ("N6", "dcenters/emu"): 5e-2,
    ("N6", "dlog_bw/emu"): 1e-2,
    ("N6", "dcenters/64"): 5e-2,
}

CASES = ([(f"N{i}", r, "tf32") for i in range(1, 6) for r in ("R64", "R128x", "R128r")] + [("N6", "R128r", "tf32")]
         + [(f"N{i}", r, "tf32x3") for i in range(1, 5) for r in ("R128x", "R128r")] + [("N6", "R128r", "tf32x3")]
         + [(f"N{i}", r, "tf32") for i in (1, 2) for r in ("R128x-cg2", "R128r-feat")]
         + [("N1", "R65536", "tf32")])


@gpu
@pytest.mark.parametrize("name,regime,precision", CASES, ids=["-".join(c) for c in CASES])
def test_training_step_vs_oracle(name, regime, precision):
    """yhat, loss and every gradient of one gathered training step against the FP64 oracle and, in TF32 mode, the
    oracle with the kernels' TF32 operand rounding emulated.  Bounds (largest measured on a B200 in brackets):
      * TF32: yhat 1e-3 of FP64, largest element (9.7e-4, N5) and 2e-4 of the emulation, relative L2 (3.8e-5);
        loss 1e-3 (9.2e-5); gradients 3e-3 of the emulation (8.2e-4) and 2e-2 of FP64 (8.0e-3), knot gradients
        included (N3: 1.8e-3 and 8.3e-3).  TF32_EXCEPTIONS lists the five exceptions (N5's head bias, N6) with causes.
      * tf32x3: yhat 2e-5 (1.7e-6); loss 1e-5 (1.4e-6); gradients 1e-3 of FP64 (1.2e-4, N1 dW1 at 12,345 rows), the
        bound of the 9,472-row test (FP32 sums over many row tiles); knot gradients 1e-3 (8.8e-5)."""
    n = _rows(regime)
    nt = net(name)
    x3 = precision == "tf32x3"
    (y64, l64, g64), (yemu, lemu, gemu) = oracle(name, n, regime)
    ex, yhat, loss, grads = train_step(name, n, regime, precision)
    errs = {"yhat64": rel_err(yhat, y64), "loss": abs(loss - l64) / abs(l64)}
    if not x3:
        errs["yhat_emu"] = rel_l2(yhat, yemu)
    for gname, g, r64 in _grad_pairs(grads, g64, nt):
        errs[f"{gname}/64"] = rel_err(g, r64)
    if not x3:
        for gname, g, re_ in _grad_pairs(grads, gemu, nt):
            errs[f"{gname}/emu"] = rel_err(g, re_)
    print(f"\n{name} {regime} {precision} n={n}:", " ".join(f"{k}={v:.2e}" for k, v in errs.items()))
    tol = X3_TOL if x3 else TF32_TOL
    bad = []
    for k, v in errs.items():
        kind = k if not k.startswith("d") else ("grad_emu" if k.endswith("/emu") else "grad64")
        bound = tol[kind] if x3 else TF32_EXCEPTIONS.get((name, k), tol[kind])
        if not v < bound:
            bad.append(f"{k}={v:.3e} (bound {bound:g})")
    assert not bad, bad


# ---------------------------------------------------------------------------------------------------- dispatch
def _template_args(name, kernel):
    """Template arguments of a kernel's instantiation from its (demangled or mangled) name, as integers."""
    m = re.search(kernel + r"<([^>]*)>", name)
    if m:
        args = re.sub(r"\((bool|int)\)", "", m.group(1)).replace(" ", "").split(",")
        return tuple(int({"true": "1", "false": "0"}.get(a, a)) for a in args)
    m = re.search(kernel + r"I((?:L[bi]\d+E)+)E", name)
    return tuple(int(v) for v in re.findall(r"L[bi](\d+)E", m.group(1))) if m else None


# (TM, CG, NS) of layer_fwd_kernel, TM of layer_bwd_kernel, block 1's backward regenerates the basis, x saved, feat stored
EXPECTED = {"R64": ((64, 4, 4), 64, False, True, False),
            "R128x": ((128, 4, 4), 128, False, True, False),
            "R128x-cg2": ((128, 2, 2), 128, False, True, False),
            "R128r": ((128, 2, 2), 128, True, False, False),
            "R128r-feat": ((128, 2, 2), 128, False, False, True),
            "R65536": ((128, 2, 2), 128, True, False, False)}


@gpu
def test_sizes_run_the_intended_kernels():
    """One step of the default network per regime under torch.profiler: the instantiation of layer_fwd_kernel
    <BASIS, TM, CG, NS> and layer_bwd_kernel<BASIS, TM, 2, 4, LNV, HEAD> of every block, and whether the workspace
    keeps x and the block-1 operand.  (cu++filt spells them `layer_fwd_kernel<(bool)1, (int)128, (int)4, (int)4>`.)
    If a threshold moves, this fails before the regime tests silently drift into another regime."""
    from torch.profiler import ProfilerActivity, profile
    rows = regime_rows()
    L, ops, Executor, NetSpec, LossSpec = _mods()
    seen = {}
    for regime, (fwd, bwd_tm, regen, has_x, has_feat) in EXPECTED.items():
        n = rows[regime]
        if regime == "R128x-cg2" and n > Executor.SAVE_X_MAX_ROWS:
            continue
        train_step("N1", n, regime)           # first launches (module load, shared-memory attributes) outside the trace
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            ex, *_ = train_step("N1", n, regime)
        kern = sorted((e for e in prof.events() if "DeviceType.CUDA" in str(getattr(e, "device_type", ""))),
                      key=lambda e: e.time_range.start)
        if not kern:
            pytest.skip("the profiler recorded no CUDA kernels (CUPTI unavailable): the instantiations cannot be read")
        fw = [_template_args(e.name, "layer_fwd_kernel") for e in kern if "layer_fwd_kernel" in e.name]
        bw = [_template_args(e.name, "layer_bwd_kernel") for e in kern if "layer_bwd_kernel" in e.name]
        seen[regime] = (n, fw, bw)
        print(f"\n{regime} n={n}: layer_fwd {fw}; layer_bwd {bw} (blocks 3, 2, 1)")
        assert fw == [(1, *fwd), (0, *fwd), (0, *fwd)], (regime, fw)
        assert bw == [(0, bwd_tm, 2, 4, 1, 1), (0, bwd_tm, 2, 4, 1, 0), (int(regen), bwd_tm, 2, 4, 1, 0)], (regime, bw)
        ws = ex._ctx[2]
        assert (ws.x is not None) == has_x and (ws.feat is not None) == has_feat, regime
    # what the regime tests rely on: a 64-row, a 128-row / 4-group and a 128-row / 2-group forward, both backward forms
    assert {f[0][1:3] for _, f, _ in seen.values()} >= {(64, 4), (128, 4), (128, 2)}
    assert {b[-1][0] for _, _, b in seen.values()} == {0, 1}


# ---------------------------------------------------------------------------------------------------- wgrad, basis form
@gpu
@pytest.mark.parametrize("rows", [20000, 65613])
@pytest.mark.parametrize("n_in,n_out", [(297, 256), (256, 128)])
def test_wgrad_basis_operand_exact_tf32(rows, n_in, n_out):
    """wgrad of block 1 regenerating the basis (wendland, n_in - 70 spatial knots + 70 temporal) for every row tile it
    walks, several tiles per split.  The reference is dz^T A with A the operand the forward generates (feat_img, the
    same generator), itself checked against orc.features after tf32_round: the FP32 basis is within 1e-5 of FP64
    before its TF32 rounding, so some elements round to the neighbouring TF32 value and only a reference built from
    the generated operand is exact.  Bound of test_wgrad_mn_major_exact_tf32: 3e-5 of the largest magnitude (measured
    on a B200: at most 3.6e-6, 65,613 rows, 297 x 256)."""
    import ctypes as C
    L, ops, *_ = _mods()
    kn = golden("knots")
    k_t = kn["t_centers"].shape[0]
    k_s = n_in - k_t
    c, b = kn["centers"][:k_s], kn["bandwidths"][:k_s]
    knots4 = ops.knots_prepare(T(c), T(b), None, "wendland")
    tk = ops.tknots_prepare(T(kn["t_centers"]), T(kn["t_bandwidths"]))
    basis = ops.make_basis(knots4, tk, k_s, k_t, 0, "wendland")
    rng = np.random.default_rng(rows + n_in)
    coords = rng.random((rows, 2)).astype(np.float32)
    t = rng.random((rows, 1)).astype(np.float32)
    pts = ops.make_points(T(coords), T(t))
    # the generated operand, through a throwaway 32-wide forward block
    w_img = ops.pack_image(T(rng.standard_normal((32, n_in)).astype(np.float32)))
    out, feat = ops.new_image(rows, 32, "cuda"), ops.new_image(rows, n_in, "cuda")
    a = L.FwdArgs()
    a.basis = C.pointer(basis)
    a.pts = pts
    a.layer = ops.make_layer(w_img, torch.zeros(32, device="cuda"), None, None, n_in, 32, 1e-5, 0)
    a.drop = L.Dropout(0.0, 0, 0)
    a.out_img, a.feat_img = out.data_ptr(), feat.data_ptr()
    ops.layer_fwd(a)
    A = ops.unpack_image(feat, rows, n_in).cpu().numpy()
    a64 = np.concatenate([orc.spatial_basis(coords, c, b, "wendland"),
                          orc.temporal_basis(t, kn["t_centers"], kn["t_bandwidths"])], axis=1)
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
