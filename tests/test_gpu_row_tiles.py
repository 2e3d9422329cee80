"""Training batches that fit in one wave of 64-row tiles run layer_fwd / layer_bwd on 64-row CTAs, two per 128-row image
tile (at most 128 x floor(SMs / 2) rows); one row more and they run on 128-row CTAs.  Both sides of that threshold
against the oracle, the two sides against each other on the rows they share, and the padding rows of a batch whose
last image tile is half full."""
import numpy as np
import pytest
import torch

from helpers import orc
from test_gpu_kernels import T, _default_oracle_model, _mods, rel_err, rel_l2, spec_from_oracle

pytestmark = pytest.mark.gpu

SEED, STEP, P_DROP = 0x1234567890ABCDEF, 17, 0.1


def _max64():
    """largest batch on 64-row tiles: one pair of 64-row CTAs per 128-row image tile, one CTA per SM"""
    return 128 * (torch.cuda.get_device_properties(0).multi_processor_count // 2)


def _inputs(n):
    rng = np.random.default_rng(11)
    coords = rng.random((n, 2)).astype(np.float32)
    t = (rng.integers(0, 100, (n, 1)) / 99.0).astype(np.float32)
    y = rng.standard_normal(n).astype(np.float32)
    return coords, t, y


def _train_step(ex, coords, t, y, n, inv_count):
    """forward(save) + backward on the first n rows: yhat, loss, gradients and the dz image of every block (in tf32x3
    mode the sum of its TF32 part and its residual image, i.e. dz to FP32 precision)"""
    L, ops, Executor, NetSpec, LossSpec = _mods()
    ex.loss_acc.zero_()
    pts = ops.make_points(T(coords[:n]), T(t[:n]))
    yhat = ex.forward(pts, train=True, step=STEP, seed=SEED, y=T(y[:n]), loss=LossSpec("mse", ()),
                      inv_count=inv_count, save=True).clone()
    grads = {k: ([g.clone() for g in v] if isinstance(v, list) else v.clone() if v is not None else None)
             for k, v in ex.backward().items()}
    ws = ex._ctx[2]
    dz = [ops.unpack_image(ws.dz[l], n, w.shape[0]) for l, w in enumerate(ex.spec.weights)]
    if ws.dz_lo is not None:
        dz = [d + ops.unpack_image(ws.dz_lo[l], n, w.shape[0]) for l, (d, w) in enumerate(zip(dz, ex.spec.weights))]
    torch.cuda.synchronize()
    return yhat, ex.loss_acc.item(), grads, dz


@pytest.mark.parametrize("size,precision", [("max64", "tf32"), ("ragged64", "tf32"), ("max64+1", "tf32"),
                                            ("max64", "tf32x3")])
def test_row_tile_sizes_with_dropout_vs_oracle(size, precision):
    """Default 297-256-256-128 network with dropout at the largest 64-row batch, a ragged 64-row batch and the smallest
    128-row batch (one row more); tolerances of test_default_size_network_with_dropout_vs_oracle."""
    L, ops, Executor, NetSpec, LossSpec = _mods()
    n = {"max64": _max64(), "ragged64": _max64() - 37, "max64+1": _max64() + 1}[size]
    assert n <= Executor.SAVE_X_MAX_ROWS       # x is saved: the backward takes its 64-row path where the forward does
    m = _default_oracle_model(43)
    m.dropout = P_DROP
    coords, t, y = _inputs(n)
    masks = [orc.dropout_keep_mask(n, w.shape[0], P_DROP, SEED, STEP, l, 0) for l, w in enumerate(m.weights[:-1])]
    yref, cache = orc.forward(m, None, coords, t, train=True, keep_masks=masks, return_cache=True)
    lref, dy = orc.loss_and_grad(yref, y, "mse", None)
    gref = orc.backward(m, cache, dy)
    yemu, cache_e = orc.forward(m, None, coords, t, train=True, keep_masks=masks, return_cache=True, rnd=orc.tf32_round)
    gemu = orc.backward(m, cache_e, orc.loss_and_grad(yemu, y, "mse", None)[1])
    x3 = precision == "tf32x3"
    ex = Executor(spec_from_oracle(m, dropout=P_DROP, precision=precision))
    yhat, loss, grads, _ = _train_step(ex, coords, t, y, n, 1.0 / n)
    yhat = yhat.cpu().numpy()
    assert rel_err(yhat, yref) < (2e-5 if x3 else 1e-3)
    assert abs(loss - lref) < (1e-5 if x3 else 1e-3) * abs(lref)
    assert x3 or rel_l2(yhat, yemu) < 2e-4
    # tf32x3 weight gradients at 9,472 rows: 1.2e-4 (dW0) and 5.5e-4 (dW1) of the FP64 reference, with the 64-row
    # kernels and with the 128-row kernels of the parent commit alike (B200): the FP32 sums over 74 row tiles exceed
    # the 1e-4 that the 1,000-row test meets, so this size gets 1e-3
    for ref_g, tol in (((gref, 1e-3),) if x3 else ((gref, 2e-2), (gemu, 3e-3))):
        for l in range(3):
            assert rel_err(grads["weights"][l].cpu().numpy(), ref_g["weights"][l]) < tol, f"dW{l} {tol}"
            assert rel_err(grads["biases"][l].cpu().numpy(), ref_g["biases"][l]) < tol
            assert rel_err(grads["gammas"][l].cpu().numpy(), ref_g["ln_gamma"][l]) < tol
            assert rel_err(grads["betas"][l].cpu().numpy(), ref_g["ln_beta"][l]) < tol
        assert rel_err(grads["head_w"].cpu().numpy(), ref_g["weights"][3]) < tol
        assert rel_err(grads["head_b"].cpu().numpy(), ref_g["biases"][3]) < tol


def test_row_tiles_64_and_128_agree_on_shared_rows():
    """The same rows through 64-row tiles (the largest such batch) and 128-row tiles (one row more), in tf32x3 mode: the
    GEMM operands are identical and only the order in which a row's LayerNorm partial sums are combined differs (8
    column groups instead of 4 in the forward, 4 instead of 2 in the backward), so yhat and dz agree to FP32 rounding.
    (In TF32 mode the stored activation and dz images are rounded to TF32, and a one-ulp FP32 difference flips that
    rounding now and then: 1.5e-4 on yhat and up to 6.6e-3 on one dz element, measured.)  Bound 1e-5 of the largest
    magnitude; measured on a B200: yhat 4.4e-7, dz of the three blocks 3.4e-7 / 4.8e-7 / 3.8e-7."""
    L, ops, Executor, NetSpec, LossSpec = _mods()
    n = _max64()
    m = _default_oracle_model(44)
    coords, t, y = _inputs(n + 1)
    ex = Executor(spec_from_oracle(m, dropout=P_DROP, precision="tf32x3"))
    inv = 1.0 / (n + 1)         # same per-row loss gradient in both runs
    y64, _, _, dz64 = _train_step(ex, coords, t, y, n, inv)
    y128, _, _, dz128 = _train_step(ex, coords, t, y, n + 1, inv)
    errs = [rel_err(y64.cpu().numpy(), y128[:n].cpu().numpy())]
    errs += [rel_err(a.cpu().numpy(), b[:n].cpu().numpy()) for a, b in zip(dz64, dz128)]
    print("yhat, dz per block: max |64-row - 128-row| / max |128-row| =", errs)
    assert all(e < 1e-5 for e in errs), errs

def test_half_full_last_image_tile_writes_its_padding_rows():
    """187 rows: three 64-row tiles of data, so the last 128-row image tile is half full.  wgrad reads whole 128-row
    tiles and regenerates nonzero basis values for padding rows, so the dz and activation images must hold zeros
    there, as on the 128-row path.  The workspace images are filled with NaN first so that rows no kernel writes
    cannot pass for zeros; the gradients are compared with the TF32-emulating oracle (tolerance 3e-3)."""
    L, ops, Executor, NetSpec, LossSpec = _mods()
    n = 187
    m = _default_oracle_model(45)
    m.dropout = P_DROP
    coords, t, y = _inputs(n)
    masks = [orc.dropout_keep_mask(n, w.shape[0], P_DROP, SEED, STEP, l, 0) for l, w in enumerate(m.weights[:-1])]
    yemu, cache_e = orc.forward(m, None, coords, t, train=True, keep_masks=masks, return_cache=True, rnd=orc.tf32_round)
    gemu = orc.backward(m, cache_e, orc.loss_and_grad(yemu, y, "mse", None)[1])
    ex = Executor(spec_from_oracle(m, dropout=P_DROP))
    ws = ex._workspace(n)
    for img in [*ws.h, *ws.dz, *ws.x]:
        img.fill_(float("nan"))
    yhat, _, grads, _ = _train_step(ex, coords, t, y, n, 1.0 / n)
    assert rel_l2(yhat.cpu().numpy(), yemu) < 2e-4
    for l in range(3):
        assert rel_err(grads["weights"][l].cpu().numpy(), gemu["weights"][l]) < 3e-3, f"dW{l}"
        assert rel_err(grads["biases"][l].cpu().numpy(), gemu["biases"][l]) < 3e-3
    assert rel_err(grads["head_w"].cpu().numpy(), gemu["weights"][3]) < 3e-3
