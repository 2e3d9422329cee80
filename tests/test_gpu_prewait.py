"""The training backward reads settled inputs before its programmatic-launch wait: every block forms its dropout keep
bits there, and the blocks below the head also x^ and the activation bits from the saved x image; the fused step tail
loads the optimizer state there.  Switching that off (Executor.prewait = False, what STDADK_PREWAIT=0 selects; the
tail's state_early) must leave every output bit for bit as it was."""
import numpy as np
import pytest
import torch

from test_gpu_kernels import T, _default_oracle_model, _mods, rel_err, spec_from_oracle
from test_gpu_row_tiles import P_DROP, _inputs, _train_step

pytestmark = pytest.mark.gpu

N = 4096        # the benchmark's batch: one wave of 64-row tiles


def _step(prewait, precision, n=N):
    L, ops, Executor, NetSpec, LossSpec = _mods()
    m = _default_oracle_model(45)
    coords, t, y = _inputs(n)
    ex = Executor(spec_from_oracle(m, dropout=P_DROP, precision=precision))
    ex.prewait = prewait
    yhat, loss, grads, dz = _train_step(ex, coords, t, y, n, 1.0 / n)
    ws = ex._ctx[2]
    assert ws.x is not None, "the step should keep x images (64-row backward)"
    x = [ops.unpack_image(ws.x[l], n, w.shape[0]).clone() for l, w in enumerate(ex.spec.weights)]
    h = [ops.unpack_image(ws.h[l], n, ex.spec.weights[l].shape[0]).clone() for l in range(len(ex.spec.weights) - 1)]
    stats = [s.clone() for s in ws.stats if s is not None]
    torch.cuda.synchronize()
    return yhat, loss, grads, dz, x, h, stats


@pytest.mark.parametrize("precision", ["tf32", "tf32x3"])
def test_prewait_step_is_bit_identical(precision):
    y0, l0, g0, dz0, x0, h0, s0 = _step(False, precision)
    y1, l1, g1, dz1, x1, h1, s1 = _step(True, precision)
    assert torch.equal(y0, y1)
    for a, b in zip(x0 + h0 + s0 + dz0, x1 + h1 + s1 + dz1):
        assert torch.equal(a, b)
    # column sums are accumulated with atomics in whatever order the CTAs finish: rounding-level differences only
    for k in ("weights", "biases", "gammas", "betas"):
        for a, b in zip(g0[k], g1[k]):
            assert rel_err(a.cpu().numpy(), b.cpu().numpy()) < 1e-5, k
    for k in ("head_w", "head_b"):
        assert rel_err(g0[k].cpu().numpy(), g1[k].cpu().numpy()) < 1e-5, k
    assert abs(l0 - l1) <= 1e-6 * abs(l0)


@pytest.mark.parametrize("n", [177_003, 600_001])
def test_tail_state_early_is_bit_identical(n):
    """The fused step tail with its optimizer state loaded before the wait and held in registers across the grid
    barrier (state_early) against the same kernel reading it afterwards, over four steps: p / m / v / shadow and the
    squared norms are the same bits.  177,003 parameters (the bench model's size) use both register slots of a thread
    (44,250 float4 on 148 x 256 threads); 600,001 exceed them and take the streaming loop with the early hyper-parameter
    loads."""
    L, ops, *_ = _mods()
    rng = np.random.default_rng(3)
    ends = [60_001, 150_002, n]
    p0 = rng.standard_normal(n).astype(np.float32)
    hyper = T([[2e-2, 5e-4, 10.0, 0], [1e-3, 5e-4, 1.0, 0], [5e-3, 0.0, 0.5, 0]])
    grads = [(rng.standard_normal(n) * (3.0 if s == 2 else 0.01)).astype(np.float32) for s in range(4)]
    out = []
    for early in (False, True):
        p, m, v, sh = T(p0), torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda"), T(p0)
        sq = torch.zeros(3, device="cuda")
        stepc = torch.zeros(1, dtype=torch.int32, device="cuda")
        ws = torch.zeros(148 * 8 + 8, device="cuda")
        sqs = []
        for gnp in grads:
            g = T(gnp)
            ops.adamw_ema_step(p, g, m, v, sh, ends, hyper, sq, stepc, ema_decay=0.95, norm_ws=ws, zero_grad=True,
                               state_early=early)
            sqs.append(sq.clone())
        torch.cuda.synchronize()
        assert int(stepc.item()) == 4
        out.append([p, m, v, sh] + sqs)
    for a, b in zip(*out):
        assert torch.equal(a, b)
