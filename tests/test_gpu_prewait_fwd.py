"""The one-wave training forward forms its dropout keep bits before its programmatic-launch wait when the step counter
is settled (Executor.prewait, what STDADK_PREWAIT=0 switches off), parks them in shared memory and reads them back in
its epilogue.  Both orders must give the same bits, with the step read from the device counter as in a trainer's step,
at the bench's batch, at a ragged one-wave batch and at a 1,604-knot lattice whose block-1 forward holds 53 slabs of
knot tables."""
import numpy as np
import pytest
import torch

from test_gpu_dense_knots import net
from test_gpu_kernels import T, _default_oracle_model, _mods, rel_err, spec_from_oracle
from test_gpu_row_tiles import P_DROP, SEED, STEP, _inputs

pytestmark = pytest.mark.gpu


def _step(nt, prewait, precision, n):
    L, ops, Executor, NetSpec, LossSpec = _mods()
    coords, t, y = _inputs(n)
    if nt is None:
        spec = spec_from_oracle(_default_oracle_model(45), dropout=P_DROP, precision=precision)
    else:
        spec = spec_from_oracle(nt.m, dropout=P_DROP, precision=precision)
        spec.level_sizes = nt.sizes
    ex = Executor(spec)
    assert not ex.sparse
    ex.prewait = prewait
    step = torch.full((1,), STEP, dtype=torch.int32, device="cuda")
    ex.loss_acc.zero_()
    pts = ops.make_points(T(coords), T(t))
    yhat = ex.forward(pts, train=True, seed=SEED, y=T(y), loss=LossSpec("mse", ()), inv_count=1.0 / n, save=True,
                      step_ptr=step).clone()
    grads = {k: ([g.clone() for g in v] if isinstance(v, list) else v.clone() if v is not None else None)
             for k, v in ex.backward().items()}
    ws = ex._ctx[2]
    assert ws.x is not None, "the step should keep x images (64-row tiles)"
    widths = [w.shape[0] for w in ex.spec.weights]
    x = [ops.unpack_image(ws.x[l], n, w).clone() for l, w in enumerate(widths)]
    h = [ops.unpack_image(ws.h[l], n, widths[l]).clone() for l in range(len(widths) - 1)]
    dz = [ops.unpack_image(ws.dz[l], n, w).clone() for l, w in enumerate(widths)]
    if ws.h_lo is not None:
        h += [ops.unpack_image(ws.h_lo[l], n, widths[l]).clone() for l in range(len(widths) - 1)]
        dz += [ops.unpack_image(ws.dz_lo[l], n, w).clone() for l, w in enumerate(widths)]
    stats = [s.clone() for s in ws.stats if s is not None]
    loss = ex.loss_acc.clone()
    torch.cuda.synchronize()
    return yhat, loss, grads, x + h + stats + dz


CASES = [(net_, n, p) for net_, n in (("default", 4096), ("default", 4001), ("D1", 4096)) for p in ("tf32", "tf32x3")]


@pytest.mark.parametrize("net_name,n,precision", CASES, ids=[f"{a}-{b}-{c}" for a, b, c in CASES])
def test_forward_keep_bits_before_the_wait_are_bit_identical(net_name, n, precision):
    nt = None if net_name == "default" else net(net_name)
    y0, l0, g0, img0 = _step(nt, False, precision, n)
    y1, l1, g1, img1 = _step(nt, True, precision, n)
    assert torch.equal(y0, y1)
    assert len(img0) == len(img1)
    for a, b in zip(img0, img1):
        assert torch.equal(a, b)
    # the loss and the column sums are accumulated with atomics in whatever order the CTAs finish
    assert abs(l0.item() - l1.item()) <= 1e-6 * abs(l0.item())
    for k in ("weights", "biases", "gammas", "betas"):
        for a, b in zip(g0[k], g1[k]):
            if a is not None:
                assert rel_err(a.cpu().numpy(), b.cpu().numpy()) < 1e-5, k
