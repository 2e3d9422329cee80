"""GPU parity tests (B200): every CUDA kernel, called through the C ABI, against the CPU oracle and the
reference's golden vectors.  Tolerances (stated per test):
  * knot-support index sets, sharding, grid generation, dropout masks: bit-exact;
  * basis values: |err| <= 1e-5 * max(phi, 1e-2) against the FP64 reference;
  * tensor-core GEMMs with operands pre-rounded to TF32: 2e-5 (FP32 accumulation order only);
  * network outputs / loss under TF32: 1e-3 relative (outputs: relative L2 error, and 2e-3 of the largest
    magnitude element-wise; loss: relative); gradients 5e-3 of the largest magnitude of the compared
    tensor; all against the FP64 reference.  (phi: the floor 2e-2 is where FP32's ulp(r) = 6e-8 in 1-r
    stops a 1e-5 relative statement from being meaningful.)
"""
import ctypes as C

import numpy as np
import pytest
import torch

from helpers import golden, kat, oracle_from_state, state_of, c_spatial_basis, orc

pytestmark = pytest.mark.gpu

DEV = "cuda"


def _mods():
    from st_dadk_b200 import _lib as L, ops
    from st_dadk_b200.executor import Executor, NetSpec, LossSpec
    return L, ops, Executor, NetSpec, LossSpec


def T(a):
    return torch.tensor(np.ascontiguousarray(a), dtype=torch.float32, device=DEV)


def rel_l2(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


def rel_err(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-30))


def spec_from_oracle(m, learnable=False, dropout=0.0, precision="tf32"):
    L, ops, Executor, NetSpec, LossSpec = _mods()
    Wh, bh = m.head(np.float64)
    n_hidden = len(m.ln_gamma)
    return NetSpec(
        centers=T(m.centers), bandwidths=None if learnable else T(m.bandwidths),
        log_bandwidths=T(np.log(m.bandwidths.astype(np.float64))) if learnable else None,
        t_centers=T(m.t_centers), t_bandwidths=T(m.t_bandwidths),
        weights=[T(w) for w in m.weights[:n_hidden]], biases=[T(b) for b in m.biases[:n_hidden]],
        gammas=[T(g) if g is not None else None for g in m.ln_gamma],
        betas=[T(b) if b is not None else None for b in m.ln_beta],
        head_w=T(Wh), head_b=T(bh), basis_fn=m.basis_fn, p_cov=m.p, dropout=dropout, ln_eps=m.ln_eps,
        learnable_basis=learnable, precision=precision)


def test_library_loads_on_gpu():
    L, ops, *_ = _mods()
    assert L.lib().stdadk_version() == 100


def test_pack_unpack_roundtrip():
    L, ops, *_ = _mods()
    rng = np.random.default_rng(0)
    for rows, cols in [(1, 1), (128, 32), (130, 33), (300, 297), (256, 256)]:
        a = rng.standard_normal((rows, cols)).astype(np.float32)
        img = ops.pack_image(T(a))
        assert img.numel() == ops.image_floats(rows, cols)
        back = ops.unpack_image(img, rows, cols).cpu().numpy()
        assert np.array_equal(back, orc.tf32_round(a))
        # strided source (transposed view)
        img_t = ops.pack_image(T(a).t())
        back_t = ops.unpack_image(img_t, cols, rows).cpu().numpy()
        assert np.array_equal(back_t, orc.tf32_round(a.T))


@pytest.mark.parametrize("fn", ["wendland", "gaussian", "triangular"])
def test_basis_fwd_values_and_support(fn):
    L, ops, *_ = _mods()
    g = golden("basis_values")
    kn = golden("knots")
    c, b = kn["centers"], kn["bandwidths"]
    rng = np.random.default_rng(3)
    extra = rng.random((5000, 2)).astype(np.float32)
    coords = np.concatenate([g["coords"], extra])
    tt = np.concatenate([g["t"], rng.random((5000, 1)).astype(np.float32)])
    knots4 = ops.knots_prepare(T(c), T(b), None, fn)
    tk = ops.tknots_prepare(T(kn["t_centers"]), T(kn["t_bandwidths"]))
    basis = ops.make_basis(knots4, tk, c.shape[0], kn["t_centers"].shape[0], 0, fn)
    ct, ttt = T(coords), T(tt)
    pts = ops.make_points(ct, ttt)
    phi, psi = ops.basis_fwd(basis, pts, DEV)
    phi, psi = phi.cpu().numpy(), psi.cpu().numpy()
    n0 = g["coords"].shape[0]
    ref = g[f"phi64_{fn}"]
    assert np.max(np.abs(phi[:n0] - ref) / np.maximum(ref, 2e-2)) < 1e-5
    ref_all = orc.spatial_basis(coords, c, b, fn)
    assert np.max(np.abs(phi - ref_all) / np.maximum(ref_all, 2e-2)) < 1e-5
    psi_ref = orc.temporal_basis(tt, kn["t_centers"], kn["t_bandwidths"])
    assert np.max(np.abs(psi - psi_ref) / np.maximum(psi_ref, 1e-2)) < 1e-5
    np.testing.assert_allclose(psi[:n0], g["psi64"], rtol=0, atol=2e-6)
    # knot-support index sets: bit-exact against the C restatement (and the reference's non-zeros)
    thetap = (b * np.float32(orc.CALIBRATION[fn])).astype(np.float32)
    phic, maskc = c_spatial_basis(coords, c, thetap, fn)
    if fn != "gaussian":
        assert np.array_equal(phi > 0, phic > 0)
        assert np.array_equal((phi > 0)[:n0], ref > 0)
    # KAT points of SURVEY 8(c)
    if fn == "wendland":
        for p in kat()["points"]:
            pp = ops.make_points(T([[p["x"], p["y"]]]), T([[p["t"]]]))
            ph, ps = ops.basis_fwd(basis, pp, DEV)
            ph = ph.cpu().numpy()[0]
            assert np.nonzero(ph > 0)[0].tolist() == p["support"]
            assert abs(ph.sum() - p["sum_phi"]) < 1e-5 * p["sum_phi"]
            assert abs(ps.cpu().numpy().sum() - p["sum_psi"]) < 1e-5 * p["sum_psi"]


def test_basis_fwd_grid_generator_bit_exact():
    L, ops, *_ = _mods()
    kn = golden("knots")
    knots4 = ops.knots_prepare(T(kn["centers"]), T(kn["bandwidths"]), None, "wendland")
    tk = ops.tknots_prepare(T(kn["t_centers"]), T(kn["t_bandwidths"]))
    basis = ops.make_basis(knots4, tk, 227, 70, 0, "wendland")
    nx, ny, nt = 37, 29, 5
    begin, end = 1000, 3500
    phi_g, psi_g = ops.basis_fwd(basis, ops.make_points(grid=(nx, ny, nt), row_begin=begin, n_rows=end - begin), DEV)
    coords, t = orc.grid_points(nx, ny, nt, begin, end)
    phi_a, psi_a = ops.basis_fwd(basis, ops.make_points(T(coords), T(t)), DEV)
    assert torch.equal(phi_g, phi_a) and torch.equal(psi_g, psi_a)


def _run_dense(ops, L, A, W, bias, gamma=None, beta=None, eps=1e-5):
    """relu(LN(A W^T + b)) through the image path of layer_fwd; returns the unpacked output."""
    rows, n_in = A.shape
    n_out = W.shape[0]
    a_img = ops.pack_image(T(A))
    w_img = ops.pack_image(T(W))
    out = ops.new_image(rows, n_out, DEV)
    out.fill_(float("nan"))
    tb, tg, tbe = T(bias), (T(gamma) if gamma is not None else None), (T(beta) if beta is not None else None)
    stats = torch.zeros(rows, 2, device=DEV)
    a = L.FwdArgs()
    a.pts = ops.make_points(grid=None, coords=None, t=None, row_begin=0, n_rows=rows)
    a.a_img = a_img.data_ptr()
    a.layer = ops.make_layer(w_img, tb, tg, tbe, n_in, n_out, eps, 0)
    a.drop = L.Dropout(0.0, 0, 0)
    a.out_img = out.data_ptr()
    a.stats = stats.data_ptr()
    ops.layer_fwd(a)
    torch.cuda.synchronize()
    return ops.unpack_image(out, rows, n_out).cpu().numpy(), stats.cpu().numpy()


# Row counts that put layer_fwd on 128-row tiles (148 SMs): 9,473 and 20,000 rows with 4 column groups, 37,765 rows
# (296 tiles, at least two per SM) with 2; all three end in a ragged tile.
ROWS_TM128 = (9473, 20000, 37765)
DENSE_TM128 = [(r, i, o) for r in ROWS_TM128 for i in (32, 297) for o in (16, 48, 96, 160, 256)]


@pytest.mark.parametrize("rows,n_in,n_out", [(128, 32, 32), (128, 64, 128), (200, 96, 48), (384, 256, 256),
                                             (1000, 297, 256), (130, 256, 128), (77, 128, 16), (128, 512, 64)]
                         + DENSE_TM128)
def test_dense_gemm_relu_exact_tf32(rows, n_in, n_out):
    """K-major tcgen05 path: operands pre-rounded to TF32 => products exact, only FP32 summation order differs.
    Up to 1,000 rows the launch runs on 64-row tiles; the ROWS_TM128 sizes run on 128-row tiles (148 SMs)."""
    L, ops, *_ = _mods()
    rng = np.random.default_rng(rows + n_in + n_out)
    A = orc.tf32_round(rng.standard_normal((rows, n_in)).astype(np.float32))
    W = orc.tf32_round((rng.standard_normal((n_out, n_in)) / np.sqrt(n_in)).astype(np.float32))
    bias = rng.standard_normal(n_out).astype(np.float32)
    got, _ = _run_dense(ops, L, A, W, bias)
    ref = np.maximum(A.astype(np.float64) @ W.astype(np.float64).T + bias, 0.0)
    # the stored activation is TF32-rounded: FP32 summation-order noise (2e-5) + one TF32 ulp (2^-11 relative)
    assert np.all(np.abs(got - ref) <= 2e-5 + np.abs(ref) * 2.0 ** -11)


@pytest.mark.parametrize("rows,n_in,n_out", [(256, 256, 256), (300, 96, 48), (128, 297, 128)] + DENSE_TM128)
def test_dense_layernorm_epilogue(rows, n_in, n_out):
    """LayerNorm epilogue: 64-row tiles up to 300 rows, 128-row tiles with 4 and 2 column groups at ROWS_TM128."""
    L, ops, *_ = _mods()
    rng = np.random.default_rng(5)
    A = orc.tf32_round(rng.standard_normal((rows, n_in)).astype(np.float32))
    W = orc.tf32_round((rng.standard_normal((n_out, n_in)) / np.sqrt(n_in)).astype(np.float32))
    bias = (rng.standard_normal(n_out) + 3.0).astype(np.float32)   # non-zero mean stresses the variance
    gamma = (1.0 + 0.2 * rng.standard_normal(n_out)).astype(np.float32)
    beta = (0.1 * rng.standard_normal(n_out)).astype(np.float32)
    got, stats = _run_dense(ops, L, A, W, bias, gamma, beta)
    z = A.astype(np.float64) @ W.astype(np.float64).T + bias
    mu = z.mean(1, keepdims=True)
    var = ((z - mu) ** 2).mean(1, keepdims=True)
    ref = np.maximum((z - mu) / np.sqrt(var + 1e-5) * gamma + beta, 0.0)
    assert np.max(np.abs(got - ref)) < 1e-3 * np.abs(ref).max()          # output image is TF32-rounded
    np.testing.assert_allclose(stats[:, 0], mu[:, 0], rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(stats[:, 1], 1 / np.sqrt(var[:, 0] + 1e-5), rtol=1e-4)


@pytest.mark.parametrize("rows,n_in,n_out", [(128, 32, 32), (256, 256, 256), (1000, 297, 256), (300, 128, 48),
                                             (4096, 256, 128), (130, 40, 16), (20000, 297, 256), (65613, 297, 256),
                                             (20000, 256, 128), (65613, 256, 128)])
def test_wgrad_mn_major_exact_tf32(rows, n_in, n_out):
    """MN-major tcgen05 path: dW = dz^T A with both operands read from the forward's images.  wgrad always reads whole
    128-row tiles and gives each of its row splits every n_split-th tile: up to 4,096 rows (32 tiles) a split gets at most
    one tile; at 20,000 and 65,613 rows (157 and 513 tiles, the last ragged) a split accumulates up to 5 and 14 tiles
    (148 SMs: 37 splits for 297 x 256, 148 for 256 x 128)."""
    L, ops, *_ = _mods()
    rng = np.random.default_rng(rows * 7 + n_in)
    A = orc.tf32_round(rng.standard_normal((rows, n_in)).astype(np.float32))
    dz = orc.tf32_round(rng.standard_normal((rows, n_out)).astype(np.float32))
    a_img, dz_img = ops.pack_image(T(A)), ops.pack_image(T(dz))
    for transposed_storage in (False, True):
        dw = torch.zeros(n_in, n_out, device=DEV).t() if transposed_storage else torch.zeros(n_out, n_in, device=DEV)
        a = L.WgradArgs()
        a.pts = ops.make_points(grid=None, coords=None, t=None, row_begin=0, n_rows=rows)
        a.a_img, a.dz_img = a_img.data_ptr(), dz_img.data_ptr()
        a.n_in, a.n_out = n_in, n_out
        a.dw, a.stride_o, a.stride_i = dw.data_ptr(), dw.stride(0), dw.stride(1)
        ops.wgrad(a)
        ref = dz.astype(np.float64).T @ A.astype(np.float64)
        assert np.max(np.abs(dw.cpu().numpy() - ref)) < 3e-5 * max(1.0, np.abs(ref).max())


CASES = [("small_mse", "wendland", "mse", None), ("small_mq", "wendland", "pinball", [0.1, 0.5, 0.9]),
         ("small_noln_tri", "triangular", "mse", None), ("small_gauss", "gaussian", "mse", None),
         ("small_learnable", "wendland", "pinball", [0.1, 0.5, 0.9]),
         ("small_delta", "wendland", "pinball", [0.1, 0.5, 0.9])]


@pytest.mark.parametrize("precision", ["tf32", "tf32x3"])
@pytest.mark.parametrize("name,fn,loss,taus", CASES)
def test_network_forward_backward_vs_reference(name, fn, loss, taus, precision):
    """Whole chain (basis fused into block 1, tcgen05 blocks, fused head + loss, backward with basis
    recompute, wgrad, knot gradients) against the reference module's FP64 outputs and autograd.
    precision "tf32x3" (three-pass operand split, FP32-faithful products): outputs to 2e-5, every gradient to 5e-4 of
    the FP64 reference (MSE: 1e-4) -- the FP32 reference itself is no closer to its FP64 evaluation."""
    L, ops, Executor, NetSpec, LossSpec = _mods()
    g = golden(name)
    m = oracle_from_state(state_of(g), basis_fn=fn)
    learn = name == "small_learnable"
    x3 = precision == "tf32x3"
    spec = spec_from_oracle(m, learnable=learn, precision=precision)
    ex = Executor(spec)
    ex.SAVE_X_MAX_ROWS = 0 if name in ("small_mq", "small_gauss") else ex.SAVE_X_MAX_ROWS   # also the recompute GEMM
    coords, t, y = T(g["coords"]), T(g["t"]), T(g["y"].reshape(-1))
    n = coords.shape[0]
    pts = ops.make_points(coords, t)
    ex.loss_acc.zero_()
    yhat = ex.forward(pts, train=True, y=y, loss=LossSpec(loss, taus or ()), inv_count=1.0 / (n * spec.q), save=True)
    torch.cuda.synchronize()
    yh = yhat.cpu().numpy()
    print(name, precision, "yhat rel_l2", rel_l2(yh, g["yhat64"]), "loss rel",
          abs(ex.loss_acc.item() - float(g["loss64"])) / abs(float(g["loss64"])))
    assert rel_l2(yh, g["yhat64"]) < (2e-5 if x3 else 1e-3) and rel_err(yh, g["yhat64"]) < (4e-5 if x3 else 2e-3)
    assert abs(ex.loss_acc.item() - float(g["loss64"])) < (1e-5 if x3 else 1e-3) * abs(float(g["loss64"]))
    grads = ex.backward()
    torch.cuda.synchronize()
    ref = {k[5:]: g[k] for k in g.files if k.startswith("grad.")}
    pre = "mlp_trunk." if m.delta is not None else "mlp."
    lin = sorted({int(k.split(".")[1]) for k in ref if k.startswith(pre) and ref[k].ndim == 2})
    # gradients vs the FP64 reference: TF32 operand rounding gives ~5e-3 (measured, profiles/); the check-loss
    # gradient additionally jumps by 1/N when a residual changes sign under a 1e-3 perturbation of yhat
    tol = 4e-2 if loss == "mse" else 6e-2     # networks this narrow (32/16 units) average fewer rounding errors
    if x3:
        tol = 1e-4 if loss == "mse" else 5e-4
    nh = spec.n_hidden
    for li in range(nh):
        k = lin[li]
        assert rel_err(grads["weights"][li].cpu().numpy(), ref[f"{pre}{k}.weight"]) < tol, f"dW{li}"
        assert rel_err(grads["biases"][li].cpu().numpy(), ref[f"{pre}{k}.bias"]) < tol, f"db{li}"
    lns = sorted({int(k.split(".")[1]) for k in ref if k.startswith(pre) and k.endswith("weight") and ref[k].ndim == 1})
    for li, k in enumerate(lns):
        assert rel_err(grads["gammas"][li].cpu().numpy(), ref[f"{pre}{k}.weight"]) < tol, f"dgamma{li}"
        assert rel_err(grads["betas"][li].cpu().numpy(), ref[f"{pre}{k}.bias"]) < tol, f"dbeta{li}"
    if m.delta is not None:
        dbeta = np.concatenate([grads["head_b"].cpu().numpy()[:, None], grads["head_w"].cpu().numpy()], axis=1)
        ddelta = np.cumsum(dbeta[::-1], axis=0)[::-1]
        for j in range(len(m.delta)):
            assert rel_err(ddelta[j], ref[f"delta_params.{j}"]) < tol
    else:
        assert rel_err(grads["head_w"].cpu().numpy(), ref[f"{pre}{lin[-1]}.weight"]) < tol
        assert rel_err(grads["head_b"].cpu().numpy(), ref[f"{pre}{lin[-1]}.bias"]) < tol
    if learn:
        assert rel_err(grads["centers"].cpu().numpy(), ref["spatial_basis.centers"]) < tol
        assert rel_err(grads["log_bandwidths"].cpu().numpy(), ref["spatial_basis.log_bandwidths"]) < tol


def _default_oracle_model(seed, q=1, fn="wendland", hidden=(256, 256, 128)):
    kn = golden("knots")
    rng = np.random.default_rng(seed)
    dims = [kn["centers"].shape[0] + kn["t_centers"].shape[0], *hidden]
    ws, bs, gs, be = [], [], [], []
    for i in range(len(hidden)):
        bound = 1 / np.sqrt(dims[i])
        ws.append(rng.uniform(-bound, bound, (dims[i + 1], dims[i])).astype(np.float32))
        bs.append(rng.uniform(-bound, bound, dims[i + 1]).astype(np.float32))
        gs.append((1 + 0.1 * rng.standard_normal(dims[i + 1])).astype(np.float32))
        be.append((0.1 * rng.standard_normal(dims[i + 1])).astype(np.float32))
    bound = 1 / np.sqrt(dims[-1])
    ws.append(rng.uniform(-bound, bound, (q, dims[-1])).astype(np.float32))
    bs.append(rng.uniform(-bound, bound, q).astype(np.float32))
    return orc.OracleModel(centers=kn["centers"], bandwidths=kn["bandwidths"], t_centers=kn["t_centers"],
                           t_bandwidths=kn["t_bandwidths"], weights=ws, biases=bs, ln_gamma=gs, ln_beta=be,
                           basis_fn=fn)


@pytest.mark.parametrize("q,loss,taus,p,precision", [(1, "mse", None, 0.0, "tf32"),
                                                     (1, "mse", None, 0.1, "tf32"),
                                                     (5, "pinball", [0.05, 0.25, 0.5, 0.75, 0.95], 0.1, "tf32"),
                                                     (1, "mse", None, 0.0, "tf32x3"),
                                                     (1, "mse", None, 0.1, "tf32x3"),
                                                     (5, "pinball", [0.05, 0.25, 0.5, 0.75, 0.95], 0.1, "tf32x3")])
def test_default_size_network_with_dropout_vs_oracle(q, loss, taus, p, precision):
    """Default architecture 297-256-256-128-Q, ragged batch, dropout masks drawn in-kernel (Philox keyed on the
    global row) and replayed by the oracle: outputs, loss and all gradients."""
    L, ops, Executor, NetSpec, LossSpec = _mods()
    m = _default_oracle_model(42 + q, q=q)
    m.dropout = p
    n, row0 = 1000, 0
    rng = np.random.default_rng(9)
    coords = rng.random((n, 2)).astype(np.float32)
    t = (rng.integers(0, 100, (n, 1)) / 99.0).astype(np.float32)
    y = rng.standard_normal(n).astype(np.float32)
    seed, step = 0x1234567890ABCDEF, 17
    masks = [orc.dropout_keep_mask(n, w.shape[0], p, seed, step, l, row0) for l, w in enumerate(m.weights[:-1])]
    yref, cache = orc.forward(m, None, coords, t, train=True, keep_masks=masks, return_cache=True)
    lref, dy = orc.loss_and_grad(yref, y, loss, taus)
    gref = orc.backward(m, cache, dy)
    # second oracle pass with the kernels' operand rounding emulated (TF32 on every tensor-core operand):
    # isolates implementation errors from precision (tolerance 3e-3 instead of 2e-2)
    yemu, cache_e = orc.forward(m, None, coords, t, train=True, keep_masks=masks, return_cache=True, rnd=orc.tf32_round)
    gemu = orc.backward(m, cache_e, orc.loss_and_grad(yemu, y, loss, taus)[1])
    x3 = precision == "tf32x3"        # compared with the FP64 oracle directly (no TF32 emulation)
    spec = spec_from_oracle(m, dropout=p, precision=precision)
    ex = Executor(spec)
    ex.loss_acc.zero_()
    pts = ops.make_points(T(coords), T(t))
    yhat = ex.forward(pts, train=True, step=step, seed=seed, y=T(y), loss=LossSpec(loss, taus or ()),
                      inv_count=1.0 / (n * q), save=True)
    grads = ex.backward()
    torch.cuda.synchronize()
    print("x3" if x3 else "tf32", "yhat err", rel_err(yhat.cpu().numpy(), yref), "dW0 err vs fp64",
          rel_err(grads["weights"][0].cpu().numpy(), gref["weights"][0]))
    assert rel_err(yhat.cpu().numpy(), yref) < (2e-5 if x3 else 1e-3)
    assert abs(ex.loss_acc.item() - lref) < (1e-5 if x3 else 1e-3) * abs(lref)
    assert x3 or rel_l2(yhat.cpu().numpy(), yemu) < 2e-4
    # (pinball: a residual within rounding of zero flips the sign of its gradient, which moves a column sum by ~1/N)
    for ref_g, tol in (((gref, 1e-4 if loss == "mse" else 5e-3),) if x3 else ((gref, 2e-2), (gemu, 3e-3))):
        for l in range(3):
            assert rel_err(grads["weights"][l].cpu().numpy(), ref_g["weights"][l]) < tol, f"dW{l} {tol}"
            assert rel_err(grads["biases"][l].cpu().numpy(), ref_g["biases"][l]) < tol
            assert rel_err(grads["gammas"][l].cpu().numpy(), ref_g["ln_gamma"][l]) < tol
            assert rel_err(grads["betas"][l].cpu().numpy(), ref_g["ln_beta"][l]) < tol
        assert rel_err(grads["head_w"].cpu().numpy(), ref_g["weights"][3]) < tol
        assert rel_err(grads["head_b"].cpu().numpy(), ref_g["biases"][3]) < tol
    # eval mode: no dropout
    ye = ex.forward(pts, train=False).cpu().numpy()
    assert rel_err(ye, orc.forward(m, None, coords, t)) < 1e-3


def test_prediction_sharding_and_grid_bit_exact():
    """Point-sharded dense-grid prediction: contiguous block partition, outputs of the shards concatenated
    are bit-identical to the single-shard run (no cross-row op), and grid == explicit arrays."""
    L, ops, Executor, NetSpec, LossSpec = _mods()
    m = _default_oracle_model(7, q=5)
    ex = Executor(spec_from_oracle(m))
    nx, ny, nt = 50, 40, 3
    n = nx * ny * nt
    full = ex.forward(ops.make_points(grid=(nx, ny, nt)), train=False).clone()
    for world in (2, 3, 8):
        parts = []
        for r in range(world):
            b, e = orc.shard_range(n, r, world)
            parts.append(ex.forward(ops.make_points(grid=(nx, ny, nt), row_begin=b, n_rows=e - b), train=False).clone())
        assert torch.equal(torch.cat(parts), full)
    coords, t = orc.grid_points(nx, ny, nt, 0, n)
    arr = ex.forward(ops.make_points(T(coords), T(t)), train=False)
    assert torch.equal(arr, full)
    assert rel_err(full.cpu().numpy(), orc.forward(m, None, coords, t)) < 1e-3


@pytest.mark.parametrize("fused", [False, True])
def test_adamw_ema_and_sqnorm_vs_oracle(fused):
    """clip_grad_norm_ coefficient + AdamW + EMA (train_st_interp.py:696-718, ema.py:52-66) vs the oracle; `fused`: the
    whole step tail in one launch (norm, step counter, update around a grid barrier) instead of three."""
    L, ops, *_ = _mods()
    rng = np.random.default_rng(1)
    n = 100_003
    ends = [60_001, n]          # group boundary inside a 16-byte vector, n not a multiple of 4
    p0 = rng.standard_normal(n).astype(np.float32)
    p, m, v, sh = T(p0), torch.zeros(n, device=DEV), torch.zeros(n, device=DEV), T(p0)
    pn, mn, vn, shn = p0.astype(np.float64), np.zeros(n), np.zeros(n), p0.astype(np.float64)
    hyper = T([[2e-2, 5e-4, 10.0, 0], [1e-3, 5e-4, 1.0, 0]])
    sq = torch.zeros(2, device=DEV)
    stepc = torch.zeros(1, dtype=torch.int32, device=DEV)
    tail_ws = torch.zeros(148 * 8 + 8, device=DEV)
    for step in range(1, 5):
        gnp = (rng.standard_normal(n) * (3.0 if step == 2 else 0.01)).astype(np.float32)
        g = T(gnp)
        if fused:
            ops.adamw_ema_step(p, g, m, v, sh, ends, hyper, sq, stepc, ema_decay=0.95, norm_ws=tail_ws, zero_grad=True)
            assert float(g.abs().max()) == 0.0
        else:
            ops.grad_sqnorm(g, ends, sq)
            ops.adamw_ema_step(p, g, m, v, sh, ends, hyper, sq, stepc, ema_decay=0.95)
        lo = 0
        for gi, hi in enumerate(ends):
            norm, coef = orc.clip_coef([gnp[lo:hi]], float(hyper[gi, 2]))
            assert abs(np.sqrt(sq[gi].item()) - norm) < 1e-4 * norm
            orc.adamw_ema_step(pn[lo:hi], gnp[lo:hi].astype(np.float64), mn[lo:hi], vn[lo:hi], shn[lo:hi], step,
                               float(hyper[gi, 0]), float(hyper[gi, 1]), 0.95, clip=coef)
            lo = hi
    assert stepc.item() == 4
    np.testing.assert_allclose(p.cpu().numpy(), pn, rtol=2e-5, atol=2e-6)
    np.testing.assert_allclose(sh.cpu().numpy(), shn, rtol=2e-5, atol=2e-6)


def test_errors_are_loud():
    L, ops, *_ = _mods()
    with pytest.raises(RuntimeError):
        ops.pack_image(torch.zeros(4, 4))          # CPU tensor: no CPU path
    a = L.FwdArgs()
    with pytest.raises(RuntimeError, match="libstdadk"):
        ops.layer_fwd(a)                            # NULL weights


@pytest.mark.parametrize("fn,sides", [("wendland", (10, 50)), ("triangular", (4, 37, 64))])
def test_large_knot_regime_support_walk_vs_oracle(fn, sides):
    """Block 1 in the large-K regime: spatial part by walking each point's compact support (gathers of knot-major W1
    rows), temporal part on the tensor cores, joined before LayerNorm; forward, loss and all gradients vs the dense
    FP64 oracle and vs the dense GPU path on the same model."""
    L, ops, Executor, NetSpec, LossSpec = _mods()
    rng = np.random.default_rng(21)
    n_centers = [s * s for s in sides]
    c, b = orc.uniform_spatial_knots(n_centers)
    tc, tb = orc.temporal_knots([10, 15])
    dims = [c.shape[0] + 25, 64, 32]
    ws = [(rng.standard_normal((dims[i + 1], dims[i])) / np.sqrt(40)).astype(np.float32) for i in range(2)]
    bs = [rng.standard_normal(dims[i + 1]).astype(np.float32) * 0.1 for i in range(2)]
    gs = [(1 + 0.1 * rng.standard_normal(dims[i + 1])).astype(np.float32) for i in range(2)]
    be = [(0.1 * rng.standard_normal(dims[i + 1])).astype(np.float32) for i in range(2)]
    ws.append((rng.standard_normal((1, 32)) / 6).astype(np.float32))
    bs.append(np.zeros(1, np.float32))
    m = orc.OracleModel(centers=c, bandwidths=b, t_centers=tc, t_bandwidths=tb, weights=ws, biases=bs, ln_gamma=gs,
                        ln_beta=be, basis_fn=fn)
    n = 700
    coords = rng.random((n, 2)).astype(np.float32)
    coords[:4] = [[0, 0], [1, 1], [0.5, 0.5], [1, 0]]
    t = rng.random((n, 1)).astype(np.float32)
    y = rng.standard_normal(n).astype(np.float32)
    yref, cache = orc.forward(m, None, coords, t, return_cache=True, rnd=orc.tf32_round)
    lref, dy = orc.loss_and_grad(yref, y, "mse")
    gref = orc.backward(m, cache, dy)
    y64 = orc.forward(m, None, coords, t)
    spec = spec_from_oracle(m)
    spec.lattice_sides = list(sides)
    ex = Executor(spec, force_sparse=True)
    assert ex.sparse
    ex.loss_acc.zero_()
    pts = ops.make_points(T(coords), T(t))
    yhat = ex.forward(pts, train=True, y=T(y), loss=LossSpec("mse"), inv_count=1.0 / n, save=True)
    grads = ex.backward()
    torch.cuda.synchronize()
    assert rel_l2(yhat.cpu().numpy(), y64) < 1e-3
    assert abs(ex.loss_acc.item() - lref) < 1e-3 * abs(lref)
    # the spatial contribution is accumulated in FP32 (not TF32): compare with some slack against the TF32 emulation
    for l in range(2):
        assert rel_err(grads["weights"][l].cpu().numpy(), gref["weights"][l]) < 1e-2, f"dW{l}"
        assert rel_err(grads["biases"][l].cpu().numpy(), gref["biases"][l]) < 1e-2
    # dense path on the same model gives the same prediction
    exd = Executor(spec_from_oracle(m), force_dense=True)
    assert not exd.sparse
    yd = exd.forward(pts, train=False).cpu().numpy()
    ys = ex.forward(pts, train=False).cpu().numpy()
    assert rel_l2(ys, yd) < 1e-3
    # rows of W1 outside every support get exactly zero gradient (index sets)
    gw = grads["weights"][0].cpu().numpy()[:, :c.shape[0]]
    mask = orc.support_mask_f32(coords, c, b, fn).any(axis=0)
    assert np.all(gw[:, ~mask] == 0) and np.all(np.abs(gw[:, mask]).sum(axis=0) > 0)


@pytest.mark.parametrize("hidden,q,fn,ln,n", [((256, 256, 128), 5, "wendland", True, 38191),
                                              ((256, 256, 128), 1, "wendland", True, 1000),
                                              ((128, 128), 3, "triangular", True, 20000),
                                              ((64,), 1, "gaussian", False, 777),
                                              ((100, 40), 2, "wendland", True, 5000),
                                              ((256, 192, 96, 32), 8, "wendland", False, 3000)])
def test_fused_prediction_kernel_vs_layered_path_and_oracle(hidden, q, fn, ln, n):
    """stdadk_predict (whole network in one persistent kernel, activations in SMEM/TMEM) against the chained
    layer_fwd path (same TF32 operands, FP32 epilogues: equal up to the rounding of differently ordered FP32 sums and
    the occasional TF32 tie that flips with them) and against the oracle: 1e-3 relative, like every prediction.
    Shapes: more tiles than SMs (the persistent loop wraps), ragged last tile, widths that are not multiples of 32,
    one to four hidden blocks, with and without LayerNorm."""
    L, ops, Executor, NetSpec, LossSpec = _mods()
    m = _default_oracle_model(11, q=q, fn=fn, hidden=hidden)
    if not ln:
        m.ln_gamma = [None] * len(hidden)
        m.ln_beta = [None] * len(hidden)
    ex = Executor(spec_from_oracle(m))
    rng = np.random.default_rng(5)
    coords = rng.random((n, 2), dtype=np.float32)
    t = rng.random(n, dtype=np.float32)
    pts = ops.make_points(T(coords), T(t))
    assert ex.fused_predict
    fused = ex.forward(pts, train=False).clone()
    assert ex._fused_ok is True, "the fused kernel must accept this shape"
    ex.fused_predict = False
    layered = ex.forward(pts, train=False).clone()
    torch.cuda.synchronize()
    f, l = fused.cpu().numpy(), layered.cpu().numpy()
    assert np.isfinite(f).all()
    assert rel_l2(f, l) < 2e-4, rel_l2(f, l)
    idx = np.r_[0:min(n, 400), max(0, n - 400):n]
    ref = orc.forward(m, None, coords[idx], t[idx])
    assert rel_l2(f[idx], ref) < 1e-3 and rel_err(f[idx], ref) < 3e-3
    assert rel_l2(l[idx], ref) < 1e-3
    emu = orc.forward(m, None, coords[idx], t[idx], rnd=orc.tf32_round)
    assert rel_l2(f[idx], emu) < 1e-4, rel_l2(f[idx], emu)


def test_covariates_ragged_single_row_and_empty_inputs():
    """Edge cases of the reference's forward signature (st_interp.py:827-846): X with p > 0 covariates in front of
    the basis columns (first-layer width not a multiple of 4 -> chunks straddling the X|phi and phi|psi boundaries),
    a single row, an empty batch -- through the whole-network kernel, the per-block kernels and a training step."""
    L, ops, Executor, NetSpec, LossSpec = _mods()
    kn = golden("knots")
    rng = np.random.default_rng(21)
    p, hidden, q = 3, (96, 64), 2
    dims = [p + kn["centers"].shape[0] + kn["t_centers"].shape[0], *hidden]
    ws = [rng.uniform(-0.1, 0.1, (dims[i + 1], dims[i])).astype(np.float32) for i in range(len(hidden))]
    bs = [rng.uniform(-0.1, 0.1, dims[i + 1]).astype(np.float32) for i in range(len(hidden))]
    ws.append(rng.uniform(-0.1, 0.1, (q, dims[-1])).astype(np.float32))
    bs.append(rng.uniform(-0.1, 0.1, q).astype(np.float32))
    m = orc.OracleModel(centers=kn["centers"], bandwidths=kn["bandwidths"], t_centers=kn["t_centers"],
                        t_bandwidths=kn["t_bandwidths"], weights=ws, biases=bs,
                        ln_gamma=[(1 + 0.1 * rng.standard_normal(h)).astype(np.float32) for h in hidden],
                        ln_beta=[(0.1 * rng.standard_normal(h)).astype(np.float32) for h in hidden], p=p)
    ex = Executor(spec_from_oracle(m))
    for n in (1, 2, 129, 700):
        X = rng.standard_normal((n, p)).astype(np.float32)
        coords, t = rng.random((n, 2), dtype=np.float32), rng.random(n, dtype=np.float32)
        y = rng.standard_normal(n).astype(np.float32)
        ref = orc.forward(m, X, coords, t)
        pts = ops.make_points(T(coords), T(t), T(X))
        ex.fused_predict = True
        fused = ex.forward(pts, train=False).clone()
        assert ex._fused_ok is True
        ex.fused_predict = False
        layered = ex.forward(pts, train=False).clone()
        assert rel_l2(fused.cpu().numpy(), ref) < 1e-3 and rel_l2(layered.cpu().numpy(), ref) < 1e-3
        # one training forward/backward: gradients of the covariate columns of W1 against the oracle
        yref, cache = orc.forward(m, X, coords, t, return_cache=True, rnd=orc.tf32_round)
        gref = orc.backward(m, cache, orc.loss_and_grad(yref, y, "pinball", [0.3, 0.7])[1])
        ex.loss_acc.zero_()
        ex.forward(pts, train=True, y=T(y), loss=LossSpec("pinball", (0.3, 0.7)), inv_count=1.0 / (n * q), save=True)
        gr = ex.backward()
        torch.cuda.synchronize()
        gw = gr["weights"][0].cpu().numpy()
        assert rel_err(gw[:, :p], gref["weights"][0][:, :p]) < 2e-2, n
        assert rel_err(gw, gref["weights"][0]) < 2e-2, n
    # empty batch: every entry point accepts n_rows = 0 and launches nothing
    e2 = torch.empty(0, 2, device="cuda")
    e1 = torch.empty(0, device="cuda")
    ex.fused_predict = True
    out = ex.forward(ops.make_points(e2, e1, torch.empty(0, p, device="cuda"), n_rows=0), train=False)
    assert out.shape == (0, q)
    ex.fused_predict = False
    out = ex.forward(ops.make_points(e2, e1, torch.empty(0, p, device="cuda"), n_rows=0), train=False)
    assert out.shape[0] == 0


def test_shapes_the_fused_kernel_does_not_take_fall_back_to_block_kernels():
    """Five hidden blocks (> STDADK_MAX_HIDDEN): stdadk_predict_supported says no, the executor chains layer_fwd
    launches instead -- still on the GPU, still within tolerance of the oracle."""
    L, ops, Executor, NetSpec, LossSpec = _mods()
    m = _default_oracle_model(5, q=2, hidden=(64, 64, 48, 32, 32))
    ex = Executor(spec_from_oracle(m))
    rng = np.random.default_rng(2)
    n = 1500
    coords, t = rng.random((n, 2), dtype=np.float32), rng.random(n, dtype=np.float32)
    out = ex.forward(ops.make_points(T(coords), T(t)), train=False)
    assert not ex._fused_ok
    # five narrow blocks accumulate TF32 rounding (measured 1.1e-3 vs FP64): the implementation check is the oracle with
    # the kernels' operand rounding emulated; the FP64 bound is the TF32 budget of this deeper shape
    assert rel_l2(out.cpu().numpy(), orc.forward(m, None, coords, t, rnd=orc.tf32_round)) < 5e-4    # measured 1.4e-4
    assert rel_l2(out.cpu().numpy(), orc.forward(m, None, coords, t)) < 3e-3


def test_large_batch_stored_operand_matches_regenerated_basis():
    """Throughput regime (more rows than one wave of tiles), optional mode `store_basis_operand`: the forward stores
    its generated block-1 operand and the backward / wgrad of block 1 read it back instead of regenerating the basis.  Same TF32 values either way, so the
    gradients agree to the rounding of differently ordered FP32 atomics; outputs are identical."""
    L, ops, Executor, NetSpec, LossSpec = _mods()
    m = _default_oracle_model(13, q=1)
    rng = np.random.default_rng(4)
    n = Executor.SAVE_X_MAX_ROWS + 1000          # 38,888 rows: 304 tiles, ragged
    coords, t = rng.random((n, 2), dtype=np.float32), rng.random(n, dtype=np.float32)
    y = rng.standard_normal(n).astype(np.float32)
    res = []
    for stored in (True, False):
        ex = Executor(spec_from_oracle(m))
        ex.store_basis_operand = stored
        ex.loss_acc.zero_()
        pts = ops.make_points(T(coords), T(t))
        yh = ex.forward(pts, train=True, y=T(y), loss=LossSpec("mse", ()), inv_count=1.0 / n, save=True).clone()
        assert (ex._ctx[2].feat is not None) == stored
        g = ex.backward()
        torch.cuda.synchronize()
        res.append((yh, [w.clone() for w in g["weights"]], [b.clone() for b in g["biases"]], ex.loss_acc.item()))
    (y0, w0, b0, l0), (y1, w1, b1, l1) = res
    assert torch.equal(y0, y1) and abs(l0 - l1) <= 2e-5 * abs(l1)      # the loss: FP32 atomics over 304 tiles
    for a, b in zip(w0 + b0, w1 + b1):
        assert rel_err(a.cpu().numpy(), b.cpu().numpy()) < 2e-5
    # and against the oracle on a subset of rows' worth of statistics: the loss
    yref = orc.forward(m, None, coords[:2000], t[:2000])
    assert rel_l2(y0[:2000].cpu().numpy(), yref) < 1e-3


def _small_net(rng, k_s, k_t=25, hidden=(64, 32)):
    dims = [k_s + k_t, *hidden]
    ws = [(rng.standard_normal((dims[i + 1], dims[i])) / np.sqrt(40)).astype(np.float32) for i in range(len(hidden))]
    bs = [rng.standard_normal(dims[i + 1]).astype(np.float32) * 0.1 for i in range(len(hidden))]
    gs = [(1 + 0.1 * rng.standard_normal(dims[i + 1])).astype(np.float32) for i in range(len(hidden))]
    be = [(0.1 * rng.standard_normal(dims[i + 1])).astype(np.float32) for i in range(len(hidden))]
    ws.append((rng.standard_normal((1, hidden[-1])) / 6).astype(np.float32))
    bs.append(np.zeros(1, np.float32))
    return ws, bs, gs, be


def _cell_list_knots(rng):
    """1,360 knots in three levels (60, 400, 900) that are not a lattice: clustered centres, per-knot bandwidths, some
    centres outside [0,1]^2; the 400-knot level is crowded (wide supports around (0.5, 0.5)).  Returns (c, b, sizes)."""
    sizes = [60, 400, 900]
    cen, bw = [], []
    for li, k in enumerate(sizes):
        if li == 1:      # crowded level: clustered knots with wide supports
            c = 0.5 + 0.08 * rng.standard_normal((k, 2))
            b = rng.uniform(0.25, 0.4, k)
        else:
            c = rng.random((k, 2)) * 1.1 - 0.05             # a few centres outside the unit square
            b = rng.uniform(0.6, 1.0, k) * 2.5 / np.sqrt(k)
        cen.append(c)
        bw.append(b)
    return np.concatenate(cen).astype(np.float32), np.concatenate(bw).astype(np.float32), sizes


@pytest.mark.parametrize("fn,learnable,precision", [("wendland", True, "tf32x3"), ("wendland", True, "tf32"),
                                                   ("triangular", False, "tf32"), ("wendland", False, "tf32")])
def test_cell_list_regime_arbitrary_and_learnable_knots_vs_oracle(fn, learnable, precision):
    """Support walk over a NON-lattice knot set (data-adaptive placement: clustered centres, per-knot bandwidths, some
    knots outside [0,1]^2 as drifted learnable knots are) through the device-built per-level cell list: forward, loss,
    every gradient -- including d centres / d log-bandwidths from the same walk -- vs the FP64 oracle, and the dense
    path on the same model.  One level is crowded on purpose (> 300 knots inside a support): nothing is truncated."""
    L, ops, Executor, NetSpec, LossSpec = _mods()
    rng = np.random.default_rng(33)
    c, b, sizes = _cell_list_knots(rng)
    tc, tb = orc.temporal_knots([10, 15])
    ws, bs, gs, be = _small_net(rng, c.shape[0])
    m = orc.OracleModel(centers=c, bandwidths=b, t_centers=tc, t_bandwidths=tb, weights=ws, biases=bs, ln_gamma=gs,
                        ln_beta=be, basis_fn=fn)
    n = 600
    coords = rng.random((n, 2)).astype(np.float32)
    coords[:4] = [[0, 0], [1, 1], [0.5, 0.5], [1, 0]]
    t = rng.random((n, 1)).astype(np.float32)
    y = rng.standard_normal(n).astype(np.float32)
    y64, cache = orc.forward(m, None, coords, t, return_cache=True)
    lref, dy = orc.loss_and_grad(y64, y, "mse")
    gref = orc.backward(m, cache, dy, coords=coords, want_knot_grads=learnable)
    assert orc.support_mask_f32(coords, c, b, fn).sum(axis=1).max() > 300
    spec = spec_from_oracle(m, learnable=learnable, precision=precision)
    spec.level_sizes = sizes
    x3 = precision == "tf32x3"
    ex = Executor(spec, force_sparse=True)
    assert ex.sparse and ex.lat is None and ex.level_begin == [0, 60, 460, 1360]
    ex.loss_acc.zero_()
    pts = ops.make_points(T(coords), T(t))
    yhat = ex.forward(pts, train=True, y=T(y), loss=LossSpec("mse"), inv_count=1.0 / n, save=True)
    grads = ex.backward()
    torch.cuda.synchronize()
    assert rel_l2(yhat.cpu().numpy(), y64) < (2e-5 if x3 else 1e-3)
    assert abs(ex.loss_acc.item() - lref) < (1e-5 if x3 else 1e-3) * abs(lref)
    # TF32 mode: operand rounding moves pre-activations by ~5e-4, which flips a few ReLUs of this narrow net; knot
    # gradients are sums of large cancelling terms and take that hardest.  tf32x3 shows the kernels themselves are exact.
    tol = 2e-4 if x3 else 2e-2
    for l in range(2):
        assert rel_err(grads["weights"][l].cpu().numpy(), gref["weights"][l]) < tol, f"dW{l}"
        assert rel_err(grads["biases"][l].cpu().numpy(), gref["biases"][l]) < tol
    if learnable:
        ec = rel_err(grads["centers"].cpu().numpy(), gref["centers"])
        eb = rel_err(grads["log_bandwidths"].cpu().numpy(), gref["log_bandwidths"])
        print(precision, "knot gradient errors", ec, eb)
        assert ec < (1e-3 if x3 else 2e-1) and eb < (1e-3 if x3 else 2e-1)
    exd = Executor(spec_from_oracle(m, learnable=learnable, precision=precision), force_dense=True)
    assert not exd.sparse
    assert rel_l2(ex.forward(pts, train=False).cpu().numpy(), exd.forward(pts, train=False).cpu().numpy()) < 1e-3
    gw = grads["weights"][0].cpu().numpy()[:, :c.shape[0]]
    mask = orc.support_mask_f32(coords, c, b, fn).any(axis=0)
    assert np.all(gw[:, ~mask] == 0) and np.all(np.abs(gw[:, mask]).sum(axis=0) > 0)      # index sets


def test_support_walk_at_real_size_99812_knots_vs_oracle():
    """BASELINE config 4 shape at REAL size: 3-level lattice 100^2 + 174^2 + 244^2 = 99,812 knots (W1 = 256 x 99,882,
    102 MB), default hidden widths; 512 rows against the dense FP64 oracle (a 512 x 99,812 basis matrix on the host),
    through both candidate sources -- the closed-form lattice window and the device-built cell list."""
    L, ops, Executor, NetSpec, LossSpec = _mods()
    rng = np.random.default_rng(5)
    n_centers = [10000, 30276, 59536]
    c, b = orc.uniform_spatial_knots(n_centers)
    tc, tb = orc.temporal_knots([10, 15, 45])
    ws, bs, gs, be = _small_net(rng, c.shape[0], k_t=70, hidden=(256, 256, 128))
    m = orc.OracleModel(centers=c, bandwidths=b, t_centers=tc, t_bandwidths=tb, weights=ws, biases=bs, ln_gamma=gs,
                        ln_beta=be, basis_fn="wendland")
    n = 512
    coords = rng.random((n, 2)).astype(np.float32)
    coords[:3] = [[0, 0], [1, 1], [0.5, 0.5]]
    t = rng.random((n, 1)).astype(np.float32)
    y64 = orc.forward(m, None, coords, t)
    spec = spec_from_oracle(m)
    spec.lattice_sides, spec.level_sizes = [100, 174, 244], n_centers
    ex = Executor(spec)
    assert ex.sparse and ex.lat is not None
    pts = ops.make_points(T(coords), T(t))
    ya = ex.forward(pts, train=False).cpu().numpy()
    assert rel_l2(ya, y64) < 1e-3
    spec2 = spec_from_oracle(m)
    spec2.level_sizes = n_centers                     # no lattice information: the cell list takes over
    ex2 = Executor(spec2)
    assert ex2.sparse and ex2.lat is None
    yb = ex2.forward(pts, train=False).cpu().numpy()
    assert rel_l2(yb, y64) < 1e-3 and rel_l2(ya, yb) < 1e-4      # same index sets, different FP32 summation order
