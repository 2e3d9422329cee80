"""GPU: the drop-in `stnf` module (autograd bridge) and the training engine against the reference's golden outputs.
Tolerances as in test_gpu_kernels.py; loss curves: 1e-3 relative (see test)."""
import copy

import numpy as np
import pytest
import torch

from helpers import golden, orc
from test_gpu_kernels import rel_err, rel_l2, T

pytestmark = pytest.mark.gpu
DEV = "cuda"
DEFAULT = dict(k_spatial_centers=[25, 81, 121], k_temporal_centers=[10, 15, 45], hidden_dims=[256, 256, 128],
               dropout=0.0, layernorm=True)


def _perturb_ln(model, seed):
    g = torch.Generator().manual_seed(seed + 1)
    with torch.no_grad():
        for mod in model.modules():
            if isinstance(mod, torch.nn.LayerNorm):
                mod.weight.add_(0.2 * torch.randn(mod.weight.shape, generator=g))
                mod.bias.add_(0.1 * torch.randn(mod.bias.shape, generator=g))


@pytest.mark.parametrize("name,q,seed,taus", [("default_mse", 1, 0, None),
                                              ("default_mq5", 5, 1, [0.05, 0.25, 0.5, 0.75, 0.95])])
def test_module_forward_backward_matches_reference(name, q, seed, taus):
    """Same seed => same initial weights as upstream (same torch init calls in the same order); forward and
    autograd through the C ABI vs the reference module's FP64 outputs / gradients (default architecture)."""
    from stnf.models import STInterpMLP
    g = golden(name)
    torch.manual_seed(seed)
    model = STInterpMLP(**DEFAULT, output_dim=q)
    _perturb_ln(model, seed)
    for k, v in model.state_dict().items():
        st = g["stat." + k]
        assert abs(float(v.double().sum()) - st[0]) <= 1e-6 * max(1.0, abs(st[0])), k
    model = model.to(DEV).eval()
    coords, t, y = T(g["coords"]), T(g["t"]), T(g["y"])
    X = torch.zeros(coords.shape[0], 0, device=DEV)
    with torch.no_grad():
        y0 = model(X, coords, t)
    assert y0.shape == (coords.shape[0], q)
    assert rel_l2(y0.cpu().numpy(), g["yhat64"]) < 1e-3 and rel_err(y0.cpu().numpy(), g["yhat32"]) < 3e-3
    yp = model(X, coords, t)
    if taus is None:
        loss = torch.nn.functional.mse_loss(yp, y)
    else:
        losses = []
        for qi, tau in enumerate(taus):
            e = y - yp[:, qi:qi + 1]
            losses.append(torch.mean(torch.max((tau - 1) * e, tau * e)))
        loss = torch.mean(torch.stack(losses))
    assert abs(loss.item() - float(g["loss64"])) < 1e-3 * abs(float(g["loss64"]))
    loss.backward()
    # (a) tight: every gradient tensor vs the oracle with the kernels' TF32 operand rounding emulated, built from the
    #     module's own weights (shown above to be the reference's); (b) loose: the reference's FP64 autograd samples.
    #     The gap between (a) and (b) is TF32 itself: a 1e-3 perturbation of a pre-activation flips the ReLU of the
    #     few units sitting at zero, and with only 300 rows one flipped row moves a column sum by several per cent.
    st = {k: v.detach().cpu().numpy() for k, v in model.state_dict().items()}
    m = orc.OracleModel(
        centers=st["spatial_basis.centers"], bandwidths=st["spatial_basis._bandwidths"],
        t_centers=st["temporal_basis.centers"], t_bandwidths=st["temporal_basis.bandwidths"],
        weights=[st[f"mlp.{i}.weight"] for i in (0, 3, 6, 9)], biases=[st[f"mlp.{i}.bias"] for i in (0, 3, 6, 9)],
        ln_gamma=[st[f"mlp.{i}.weight"] for i in (1, 4, 7)], ln_beta=[st[f"mlp.{i}.bias"] for i in (1, 4, 7)])
    yh, cache = orc.forward(m, None, g["coords"], g["t"], return_cache=True, rnd=orc.tf32_round)
    gr = orc.backward(m, cache, orc.loss_and_grad(yh, g["y"], "mse" if taus is None else "pinball", taus)[1])
    emu = {"mlp.0.weight": gr["weights"][0], "mlp.3.weight": gr["weights"][1], "mlp.6.weight": gr["weights"][2],
           "mlp.9.weight": gr["weights"][3], "mlp.1.weight": gr["ln_gamma"][0], "mlp.4.weight": gr["ln_gamma"][1],
           "mlp.7.weight": gr["ln_gamma"][2], "mlp.1.bias": gr["ln_beta"][0], "mlp.4.bias": gr["ln_beta"][1],
           "mlp.7.bias": gr["ln_beta"][2], "mlp.0.bias": gr["biases"][0], "mlp.3.bias": gr["biases"][1],
           "mlp.6.bias": gr["biases"][2], "mlp.9.bias": gr["biases"][3]}
    for k, p in model.named_parameters():
        got = p.grad.detach().cpu().numpy()
        assert rel_err(got, emu[k]) < (2e-2 if taus else 2e-3), (k, rel_err(got, emu[k]))
        gs = g["gsample." + k]
        scale = max(float(np.abs(gs).max()), float(np.sqrt(g["gstat." + k][1] / p.numel())))
        assert float(np.abs(got.reshape(-1)[::97] - gs).max()) / scale < 0.25, k


def test_reference_api_surface():
    """The structural assertions of the reference's own unit tests (tests/stnf/models/
    test_st_interp_delta_reparameterization.py), run on the GPU module."""
    from stnf.models import STInterpMLP, create_model
    cfg = dict(p=0, k_spatial_centers=[9], k_temporal_centers=[5], hidden_dims=[32, 16], dropout=0.0, layernorm=False,
               spatial_learnable=False, spatial_init_method="uniform", spatial_basis_function="wendland", output_dim=5)
    X, coords, t = torch.zeros(4, 0, device=DEV), torch.rand(4, 2, device=DEV), torch.rand(4, 1, device=DEV)
    m = STInterpMLP(use_delta_reparameterization=False, **cfg).to(DEV).eval()
    with torch.no_grad():
        assert m(X, coords, t).shape == (4, 5)
    assert hasattr(m, "mlp") and m.mlp_trunk is None and m.delta_params is None
    md = STInterpMLP(use_delta_reparameterization=True, **cfg).to(DEV)
    assert md.mlp_trunk is not None and len(md.delta_params) == 5
    assert all(d.shape == (17,) and d.requires_grad and not torch.allclose(d, torch.zeros_like(d)) for d in md.delta_params)
    # cumulative beta: delta_k == k+1 everywhere => beta_k[0] = (k+1)(k+2)/2
    with torch.no_grad():
        for k, d in enumerate(md.delta_params):
            d.fill_(float(k + 1))
    w, b = md._effective_head()
    assert [float(v) for v in b.detach()] == [(k + 1) * (k + 2) / 2 for k in range(5)]
    md.eval()
    with torch.no_grad():
        a, bb = md(X, coords, t), md(X, coords, t)
    assert torch.equal(a, bb) and torch.isfinite(a).all()
    md.train()
    out = md(X, coords, t)
    out.sum().backward()
    assert all(d.grad is not None and d.grad.abs().sum() > 0 for d in md.delta_params)
    pen = md.compute_sparsity_penalty("sparse_group", 0.01, 0.01)
    assert set(pen) == {"spatial_penalty", "temporal_penalty", "total_penalty"} and pen["total_penalty"] >= 0
    mc = create_model({"regression_type": "multi-quantile", "quantile_levels": [0.1, 0.5, 0.9],
                       "use_delta_reparameterization": True})
    assert mc.output_dim == 3 and mc.use_delta_reparameterization
    assert sum(p.numel() for p in STInterpMLP().parameters()) == 176385
    m2 = copy.deepcopy(m)
    assert torch.equal(m2(X, coords, t), m(X, coords, t))
    with pytest.raises(RuntimeError):
        STInterpMLP(**cfg)(torch.zeros(4, 0), torch.rand(4, 2), torch.rand(4, 1))   # CPU tensors: no fallback
    # standalone embeddings (values)
    kn = golden("knots")
    sb = STInterpMLP().to(DEV).spatial_basis
    phi = sb(T(golden("basis_values")["coords"]))
    ref = golden("basis_values")["phi64_wendland"]
    assert np.max(np.abs(phi.cpu().numpy() - ref) / np.maximum(ref, 2e-2)) < 1e-5


@pytest.mark.parametrize("precision", ["tf32x3", "tf32"])
def test_training_engine_loss_curve_vs_reference(precision):
    """20 optimisation steps (MSE, AdamW + clip + EMA, warm-up written after the step) on the fixture's data:
    per-step loss and gradient norm vs the reference's FP32 CPU run.

    precision "tf32x3" (the parity mode: three tensor-core passes per GEMM, FP32-faithful products): EVERY one of the
    20 losses within 1e-3 relative of the reference run (measured 2.7e-5), and the final raw and EMA predictions
    within 1e-3 (relative L2) -- the tolerance north_star states for predictions and loss curves.  Gradient norms
    within 3e-3: the reference's own FP32 run differs from its FP64 run by 3e-5 on this loss curve, 1.5e-4 on the EMA
    predictions and up to 1.3e-3 on the gradient norm (step 18, where this path measures 1.4e-3 too).

    precision "tf32" (the throughput mode): at matched weights the loss agrees to <1e-3 (first steps here; 4e-5 in
    the single-step tests), but over many steps at lr=2e-2 TF32 operand rounding (~5e-3 per gradient) moves the
    trajectory: steps 0-3 within 1e-3, every step within 3e-2, the first 8 gradient norms within 3e-2, raw
    predictions within 2e-2."""
    from stnf.models import STInterpMLP
    from stnf.dataio import ObservationTable
    from st_dadk_b200.trainer import Trainer
    g = golden("train_curve")
    n, bs, steps, warm = [int(v) for v in g["meta"]]
    lr, wd, clip = [float(v) for v in g["hyper"]]
    torch.manual_seed(123)
    model = STInterpMLP(**DEFAULT)
    table = ObservationTable(torch.from_numpy(g["coords"]), torch.from_numpy(g["t"].reshape(-1)),
                             torch.from_numpy(g["y"].reshape(-1))).to(DEV)
    bpe = n // bs
    x3 = precision == "tf32x3"
    cfg = dict(lr=lr, weight_decay=wd, grad_clip=clip, warmup_epochs=warm // bpe, epochs=100, regression_type="mean",
               precision=precision)
    for graph in (False, True):
        torch.manual_seed(123)
        model = STInterpMLP(**DEFAULT)
        tr = Trainer(model, cfg, DEV, batches_per_epoch=bpe, use_cuda_graph=graph)
        perm = torch.arange(n, device=DEV)
        losses, norms = [], []
        shadow_host = tr.flat.p.clone()
        for s in range(steps):
            lo = (s % bpe) * bs
            tr.train_step(table, perm, lo, bs)
            shadow_host = tr.ema_decay * shadow_host + (1.0 - tr.ema_decay) * tr.flat.p
            losses.append(tr.pop_loss_sum())
            norms.append(float(tr.sqnorms[0].sqrt().item()))
        losses, norms = np.array(losses), np.array(norms)
        rel = np.abs(losses - g["losses"]) / np.abs(g["losses"])
        nrel = np.abs(norms - g["grad_norms"]) / g["grad_norms"]
        print(precision, "graph", graph, "loss rel", np.array2string(rel, precision=2), "norm rel",
              np.array2string(nrel, precision=2))
        if x3:
            assert rel.max() < 1e-3, (graph, rel)
            assert nrel.max() < 3e-3, (graph, nrel)
        else:
            assert rel[:4].max() < 1e-3 and rel.max() < 3e-2, (graph, rel)
            assert nrel[:8].max() < 3e-2, nrel     # later norms sit on a chaotic trajectory (lr 2e-2): not compared
        model.eval()
        X = torch.zeros(256, 0, device=DEV)
        with torch.no_grad():
            raw = model(X, table.coords[:256], table.t[:256, None]).cpu().numpy()
            tr.flat.apply_shadow()
            st = {k: v.detach().cpu().numpy().copy() for k, v in model.state_dict().items()}
            ema = model(X, table.coords[:256], table.t[:256, None]).cpu().numpy()
            tr.flat.restore()
        print("raw", rel_l2(raw, g["yhat_raw"]), "ema vs reference run", rel_l2(ema, g["yhat_ema"]))
        assert rel_l2(raw, g["yhat_raw"]) < (1e-3 if x3 else 2e-2)
        assert not x3 or rel_l2(ema, g["yhat_ema"]) < 1e-3
        # EMA weights (TF32 mode): the fused kernel's shadow == decay*shadow + (1-decay)*p replayed on the host after every step,
        # and the forward under the swapped-in EMA weights == the oracle on those same weights.  (The reference run's
        # EMA *predictions* are not compared: after 20 steps at lr 2e-2 the averaged model's output is a cancellation
        # that amplifies the 1e-3 weight-trajectory difference to ~1e-1; measured and explained in DESIGN.md.)
        assert float((tr.flat.shadow - shadow_host).abs().max()) < 1e-5
        m = orc.OracleModel(
            centers=st["spatial_basis.centers"], bandwidths=st["spatial_basis._bandwidths"],
            t_centers=st["temporal_basis.centers"], t_bandwidths=st["temporal_basis.bandwidths"],
            weights=[st[f"mlp.{i}.weight"] for i in (0, 3, 6, 9)], biases=[st[f"mlp.{i}.bias"] for i in (0, 3, 6, 9)],
            ln_gamma=[st[f"mlp.{i}.weight"] for i in (1, 4, 7)], ln_beta=[st[f"mlp.{i}.bias"] for i in (1, 4, 7)])
        assert rel_l2(ema, orc.forward(m, None, g["coords"][:256], g["t"][:256])) < 1e-3


def test_space_time_field_equals_explicit_points_any_sharding():
    """Predictor.space_time_field (T x S field of upstream's predictions.npz; sites visited in a space-filling order
    and scattered back) must equal the same points passed explicitly, bit for bit, for whole-step and ragged shards;
    shards concatenated = the single-rank field."""
    from stnf.models import STInterpMLP
    from st_dadk_b200.predict import Predictor
    torch.manual_seed(3)
    model = STInterpMLP(**DEFAULT, output_dim=3)
    _perturb_ln(model, 3)
    model = model.to(DEV).eval()
    S, Tn = 700, 6
    g = torch.Generator().manual_seed(0)
    sites = torch.rand(S, 2, generator=g).to(DEV)
    pr = Predictor(model)
    field, (b, e) = pr.space_time_field(sites, Tn)
    assert (b, e) == (0, S * Tn) and field.shape == (S * Tn, 3)
    coords = sites.repeat(Tn, 1)
    t = torch.arange(Tn, device=DEV).repeat_interleave(S).float() / (Tn - 1)
    explicit, _ = pr.points(coords, t)
    # the field runs the site-tile x time-loop kernel (zs(site) + zt(time), zt in FP32), explicit points the per-point
    # kernel (one TF32 GEMM over [phi | psi]): the same function, equal to TF32 rounding; with the field kernel switched
    # off the two paths are the same kernel and must agree bit for bit
    assert pr.used_field_kernel and rel_l2(field.cpu().numpy(), explicit.cpu().numpy()) < 1e-3
    gen = Predictor(model)
    gen.use_field_kernel = False
    assert torch.equal(gen.space_time_field(sites, Tn)[0], explicit)
    for world in (2, 3, 4):          # 2, 3: whole time steps per rank (ordered path); 4: ragged shards (plain path)
        parts = [pr.space_time_field(sites, Tn, r, world)[0] for r in range(world)]
        assert torch.equal(torch.cat(parts), field)
    again, _ = pr.space_time_field(sites, Tn)      # cached expansion
    assert torch.equal(again, field)
    served = Predictor(model, static_weights=True)  # serving mode: operand images built once
    for _ in range(2):
        assert torch.equal(served.space_time_field(sites, Tn)[0], field)
    # delivered to pinned host memory in pieces, each copy overlapping the next piece's kernel
    hout = torch.empty(S * Tn, 3).pin_memory()
    pr.d2h_chunk_rows = 2 * S + 5                  # -> pieces of two whole time steps
    piecewise, _ = pr.space_time_field(sites, Tn, host_out=hout)
    pr.host_copy_done.synchronize()
    assert torch.equal(piecewise, field) and torch.equal(hout, field.cpu())


def test_step_tail_bookkeeping_gradient_zeroing_and_loss_sum():
    """The fused AdamW kernel leaves the flat gradient (and the loss accumulator that rides at its end) zeroed, and
    an evaluation between two steps must not leak its loss into the running training loss: per-step losses of a run
    with interleaved `evaluate` calls equal those of a run without, and equal the eager (graph-free) run."""
    from stnf.models import STInterpMLP
    from stnf.dataio import ObservationTable
    from st_dadk_b200.trainer import Trainer
    rng = np.random.default_rng(4)
    n, B = 3000, 1000
    c, t = rng.random((n, 2)).astype(np.float32), rng.random(n).astype(np.float32)
    y = (np.sin(5 * c[:, 0]) + t).astype(np.float32)
    table = ObservationTable(torch.from_numpy(c), torch.from_numpy(t), torch.from_numpy(y)).to(DEV)
    perm = torch.arange(n, device=DEV)
    cfg = dict(lr=1e-2, weight_decay=5e-4, grad_clip=5.0, regression_type="mean")

    def run(graph, with_eval):
        torch.manual_seed(2)
        tr = Trainer(STInterpMLP(hidden_dims=[64, 32], dropout=0.1), cfg, DEV, batches_per_epoch=3, use_cuda_graph=graph)
        out = []
        for s in range(6):
            tr.train_step(table, perm, (s % 3) * B, B)
            out.append(tr.pop_loss_sum())
            assert float(tr.flat.g.abs().max()) == 0.0           # gradients and loss slot zeroed by the update
            if with_eval:
                tr.evaluate(table, batch_rows=1024)
        return out, tr.flat.p.clone()

    (l0, p0), (l1, p1), (l2, p2) = run(True, False), run(True, True), run(False, True)
    # Loss and weight-gradient accumulation use floating-point atomics, so runs agree to rounding, not bit for bit --
    # and Adam turns a rounding-level difference of a near-zero gradient entry into an update of order lr, so single
    # parameters may differ by ~1e-2 while the mean stays tiny.  A leaked validation loss would be an O(1) difference.
    close = lambda a, b: float((a - b).abs().mean()) < 2e-4
    assert np.allclose(l0, l1, rtol=2e-3) and close(p0, p1)
    assert np.allclose(l0, l2, rtol=2e-3) and close(p0, p2)


def test_host_buffer_step_sync_and_lagged_match_device_step():
    """Trainer.train_step_host (pinned host batch -> H2D -> step -> D2H loss, double-buffered staging): the
    synchronous form returns each step's loss, the lagged form the previous step's (then flush); both equal the
    device-resident train_step losses and end at the same parameters."""
    from stnf.models import STInterpMLP
    from stnf.dataio import ObservationTable
    from st_dadk_b200.trainer import Trainer
    rng = np.random.default_rng(8)
    n, B, steps = 4000, 1000, 7
    c, t = rng.random((n, 2)).astype(np.float32), rng.random(n).astype(np.float32)
    y = (np.cos(4 * c[:, 1]) - t).astype(np.float32)
    host = ObservationTable(torch.from_numpy(c).pin_memory(), torch.from_numpy(t).pin_memory(),
                            torch.from_numpy(y).pin_memory())
    dev_table = ObservationTable(torch.from_numpy(c), torch.from_numpy(t), torch.from_numpy(y)).to(DEV)
    perm = torch.arange(n, device=DEV)
    cfg = dict(lr=1e-2, weight_decay=5e-4, grad_clip=5.0, regression_type="mean")

    def run(mode):
        torch.manual_seed(6)
        tr = Trainer(STInterpMLP(hidden_dims=[64, 32], dropout=0.1), cfg, DEV, batches_per_epoch=4, use_cuda_graph=True)
        out = []
        for s in range(steps):
            b = (s % 4) * B
            if mode == "device":
                tr.train_step(dev_table, perm, b, B)
                out.append(tr.pop_loss_sum())
            elif mode == "sync":
                out.append(tr.train_step_host(host, b, B))
            else:
                out.append(tr.train_step_host(host, b, B, lagged=True))
        if mode == "lagged":
            assert np.isnan(out[0])
            out = out[1:] + [tr.flush_host_loss()]
        torch.cuda.synchronize()
        return out, tr.flat.p.clone()

    (ld, pd_), (ls, ps), (ll, pl) = run("device"), run("sync"), run("lagged")
    close = lambda a, b: float((a - b).abs().mean()) < 2e-4      # see the note on atomics + Adam above
    assert np.allclose(ld, ls, rtol=2e-3) and np.allclose(ld, ll, rtol=2e-3), (ld, ls, ll)
    assert close(pd_, ps) and close(pd_, pl)


def test_trainer_learnable_knots_cell_list_path_equals_dense_path_and_scales_to_5000():
    """A learnable, data-adaptive (random_site) model trains through the support walk with the per-step device-built
    cell list (knots move every step; knot gradients come from the same walk).  At 1,900 knots -- which the dense kernels
    hold at first width 64 (up to 2,134 with its 70 temporal knots, bound by wgrad's knot table; at width 256 the
    recompute backward holds at most 1,626, test_gpu_dense_knots) -- the same model forced through the dense operand (all columns
    generated, knot gradients on the tensor cores) must follow the same losses and reach the same parameters (tf32x3, so
    operand rounding does not blur the comparison).  The 5,000-knot model (beyond the dense path) must train: finite,
    decreasing loss, moving knots."""
    from stnf.models import STInterpMLP
    from stnf.dataio import ObservationTable
    from st_dadk_b200.trainer import Trainer
    from st_dadk_b200.executor import Executor
    rng = np.random.default_rng(12)
    n, B = 6000, 1500
    c, t = rng.random((n, 2)).astype(np.float32), rng.random(n).astype(np.float32)
    y = (np.sin(6 * c[:, 0]) * np.cos(5 * c[:, 1]) + t).astype(np.float32)
    table = ObservationTable(torch.from_numpy(c), torch.from_numpy(t), torch.from_numpy(y)).to(DEV)
    perm = torch.arange(n, device=DEV)
    cfg = dict(lr=5e-3, basis_lr_ratio=0.5, weight_decay=5e-4, grad_clip=5.0, regression_type="mean", precision="tf32x3",
               gradient_damping=True, damping_threshold=0.0, damping_strength=5.0, domain_penalty_weight=0.01)

    def run(levels, dense, steps=6):
        old = Executor.DENSE_MAX_KNOTS
        Executor.DENSE_MAX_KNOTS = 10 ** 9 if dense else 0
        try:
            torch.manual_seed(4)
            np.random.seed(4)
            model = STInterpMLP(k_spatial_centers=levels, hidden_dims=[64, 32], dropout=0.0,
                                spatial_learnable=True, spatial_init_method="random_site", train_coords=c,
                                gradient_damping=True, damping_threshold=0.0, damping_strength=5.0)
            c_init = model.spatial_basis.centers.detach().clone()
            tr = Trainer(model, cfg, DEV, batches_per_epoch=4, use_cuda_graph=not dense)
            lb = [0]
            for k in levels:
                lb.append(lb[-1] + k)
            assert tr.ex.sparse == (not dense) and (dense or tr.ex.level_begin == lb)
            losses = []
            for s in range(steps):
                tr.train_step(table, perm, (s % 4) * B, B)
                losses.append(tr.pop_loss_sum())
            cen = model.spatial_basis.centers.detach().clone()
            return np.array(losses), tr.flat.p.clone(), cen, float((cen.cpu() - c_init).abs().max())
        finally:
            Executor.DENSE_MAX_KNOTS = old

    small = [300, 700, 900]
    (ls, ps, cs, _), (ld, pd_, cd, _) = run(small, False), run(small, True)
    print("losses", ls, ld, "max |dp|", float((ps - pd_).abs().max()))
    assert np.allclose(ls, ld, rtol=2e-4)
    # (Adam turns a rounding-level difference of a near-zero gradient entry into an update of order lr: single parameters
    #  may differ by ~lr while the mean difference stays at rounding level)
    assert float((ps - pd_).abs().mean()) < 2e-5 and float((ps - pd_).abs().max()) < 3e-2
    assert float((cs - cd).abs().mean()) < 2e-5
    lb, _, _, moved = run([500, 2000, 2500], False, steps=10)
    print("5000 knots: losses", lb, "largest knot movement", moved)
    assert np.all(np.isfinite(lb)) and lb[-1] < 0.7 * lb[0] and moved > 1e-4
