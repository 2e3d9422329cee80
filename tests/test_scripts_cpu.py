"""CPU: host-side pieces of the training driver against fixtures produced by the reference's own script
(oracle/gen_golden.py::masks_fixture) and the known answers of the reference's unit tests."""
import numpy as np
import pytest
import torch

from helpers import golden
from scripts import train_st_interp as drv
from scripts.run_grid_search import generate_config_combinations, DEFAULT_GRID


@pytest.mark.parametrize("tag,om,pat,sm", [("a", "site-wise", "corner", "random"), ("b", "random", "uniform", "site-wise"),
                                           ("c", "site-wise", "uniform", "site-wise"), ("d", "random", "corner", "random")])
def test_masks_and_sample_order_bit_exact(tag, om, pat, sm):
    g = golden("masks_losses")
    z, coords = g["z"], g["coords"]
    fn = drv.create_spatial_obs_prob_fn(pat, 10.0)
    obs, sites = drv.sample_observations(z, coords, om, 0.3, fn, seed=2025)
    tr, va = drv.split_train_valid(obs, sites, sm, 0.8, seed=12025)
    assert np.array_equal(obs, g[f"{tag}_obs"]) and np.array_equal(np.asarray(sites), g[f"{tag}_sites"])
    assert np.array_equal(tr, g[f"{tag}_train"]) and np.array_equal(va, g[f"{tag}_valid"])
    tab = drv.create_dataset_from_mask(z, coords, tr, 0)
    assert np.array_equal(tab.y.numpy(), g[f"{tag}_ds_y"])
    assert np.array_equal(tab.t.numpy(), g[f"{tag}_ds_t"])
    assert np.array_equal(tab.coords.numpy(), g[f"{tag}_ds_c"])


def test_losses_and_penalties_vs_reference():
    g = golden("masks_losses")
    yp, yt = torch.tensor(g["loss_yp"]), torch.tensor(g["loss_yt"])
    assert drv.quantile_loss(yp[:, :1], yt, 0.3).item() == pytest.approx(float(g["pinball_03"]), rel=1e-12)
    assert drv.non_crossing_penalty(yp, "mean", 1).item() == pytest.approx(float(g["nc_p1"]), rel=1e-12)
    assert drv.non_crossing_penalty(yp, "sum", 2).item() == pytest.approx(float(g["nc_p2"]), rel=1e-12)
    deltas = [torch.tensor(d) for d in g["deltas"]]
    assert drv.compute_p_nc_delta_penalty(deltas).item() == pytest.approx(float(g["pnc"]), rel=1e-12)
    assert drv.compute_crps_multi_quantile(g["loss_yp"], g["loss_yt"], [0.1, 0.5, 0.9]) == pytest.approx(float(g["crps"]), rel=1e-12)
    # known answers pinned by the reference's own tests (tests/stnf/models/test_crps_eq_4_6.py:18-44,
    # test_p_nc_delta_penalty.py:51-78)
    one, zero = torch.tensor([[1.0]]), torch.tensor([[0.5]])
    assert drv.quantile_loss(zero, one, 0.5).item() == pytest.approx(0.25)
    assert drv.quantile_loss(one, zero, 0.1).item() == pytest.approx(0.45)
    assert drv.quantile_loss(zero, one, 0.1).item() == pytest.approx(0.05)
    d = [torch.zeros(6), torch.tensor([2.0, 1.0, -0.5, 0.3, -0.2, 0.0])]
    assert drv.compute_p_nc_delta_penalty(d).item() == pytest.approx(0.0)
    assert drv.compute_crps({0.5: np.array([0.5])}, np.array([1.0])) == pytest.approx(0.5)
    assert drv.auto_batch_size(4096, 8000) == 512 and drv.auto_batch_size(4096, 80000) == 4096


def test_grid_of_64_configs():
    cfgs = generate_config_combinations({"epochs": 50, "n_experiments": 1}, DEFAULT_GRID)
    assert len(cfgs) == 64 and len({c["tag"] for c in cfgs}) == 64
    assert {c["config_id"] for c in cfgs} == set(range(1, 65))
    assert sum(c["spatial_learnable"] for c in cfgs) == 32
    for r in range(8):                      # 8 configs per GPU on an 8-GPU box
        assert len(cfgs[r::8]) == 8


def test_yaml_schema_accepted():
    import yaml
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cfg = yaml.safe_load(open(os.path.join(root, "configs", "config_st_interp.yaml")))
    from stnf.models import create_model
    rng = np.random.default_rng(0)
    np.random.seed(0)
    m = create_model(dict(cfg, k_spatial_centers=[4, 9]), train_coords=rng.random((200, 2)).astype(np.float32))
    assert m.output_dim == 5 and m.spatial_basis.learnable and m.spatial_basis.k == 13
    assert m.spatial_basis.centers.shape == (13, 2) and (m.spatial_basis.bandwidths > 0).all()


def test_flat_state_layout_on_cpu():
    """FlatState (host logic, no kernels): parameters re-pointed into one flat buffer with upstream's shapes, Linear
    weights stored (in, out)-contiguous behind a .t() view, gradient views of the same geometry, and -- behind the
    gradients -- the delta head's scratch and the one-float loss slot that lets a data-parallel step use ONE
    all-reduce (n_exchange)."""
    from stnf.models import STInterpMLP
    from st_dadk_b200.trainer import FlatState
    for kw in (dict(output_dim=1), dict(output_dim=3, use_delta_reparameterization=True), dict(spatial_learnable=True)):
        torch.manual_seed(0)
        model = STInterpMLP(k_spatial_centers=[9, 25], k_temporal_centers=[4], hidden_dims=[32, 16], **kw)
        before = {k: v.detach().clone() for k, v in model.state_dict().items()}
        fl = FlatState(model, "cpu")
        n_par = sum(p.numel() for p in model.parameters())
        assert fl.n == n_par and fl.p.numel() == n_par
        assert fl.n_exchange == fl.n + fl.n_scratch + 1 and fl.g.numel() >= fl.n_exchange
        assert fl.loss_slot.data_ptr() == fl.g[fl.n + fl.n_scratch:].data_ptr() and fl.loss_slot.numel() == 1
        for k, v in model.state_dict().items():          # same keys, shapes and values as before the re-pointing
            assert v.shape == before[k].shape and torch.equal(v, before[k]), k
        w = model.hidden_blocks()[0][0].weight
        assert w.shape == (32, 34 + 4) and w.t().is_contiguous()           # (in, out)-contiguous storage
        for p in model.parameters():
            gv = fl.gviews[id(p)]
            assert gv.shape == p.shape
            gv.fill_(1.0)
        assert float(fl.g[:fl.n].sum()) == n_par and float(fl.g[fl.n:].abs().sum()) == 0.0
        # the gradient buffer is padded to whole 16-byte packets for the peer-memory exchange
        assert fl.g.numel() % 4 == 0 and fl.g.numel() - fl.n_exchange < 4


def test_gmm_knot_fit_is_memoised_and_thread_safe():
    """knot_init.gmm_knots: the scikit-learn mixture fit (seconds on the host; upstream fixes random_state=42) is a
    pure function of (sample, k): a sweep's repeated fits come from the per-process cache, identical to a fresh fit."""
    import threading
    import time
    from st_dadk_b200 import knot_init as K
    K._GMM_CACHE.clear()
    rng = np.random.default_rng(5)
    pts = rng.random((600, 2))
    t0 = time.perf_counter()
    c0, b0 = K.gmm_knots([4, 9], pts)
    t_first = time.perf_counter() - t0
    out = []
    ths = [threading.Thread(target=lambda: out.append(K.gmm_knots([4, 9], pts.copy()))) for _ in range(4)]
    t0 = time.perf_counter()
    for th in ths:
        th.start()
    for th in ths:
        th.join()
    t_cached = time.perf_counter() - t0
    assert len(K._GMM_CACHE) == 2 and t_cached < max(0.5 * t_first, 0.05)
    for c, b in out:
        assert torch.equal(c, c0) and torch.equal(b, b0)
    c1, b1 = K.gmm_knots([4, 9], pts + 1e-3)                  # another sample: refit, different result
    assert len(K._GMM_CACHE) == 4 and not torch.equal(c1, c0)
    assert c0.shape == (13, 2) and b0.shape == (13,) and bool((b0 > 0).all())


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` (the reference's own PyTorch CPU path from oracle/_ref when that copy is present,
    else the oracle port) prints ONE JSON line with the contract keys; under torchrun only rank 0 prints and the other
    ranks exit 0 without work."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, RANK="0", WORLD_SIZE="1")
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--gpus", "1", "--steps", "1",
                        "--warmup", "1"], capture_output=True, text=True, timeout=600, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.strip().splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["metric"] == "train_samples_per_s" and d["unit"] == "samples/s"
    assert d["value"] > 0 and d["higher_is_better"] is True and d["vs_baseline"] is None and "workload" in d["config"]
    have_ref = os.path.isdir(os.path.join(root, "oracle", "_ref", "stnf"))
    assert d["cpu_baseline"]["kind"] == ("reference" if have_ref else "port")
    assert d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    other = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                            "--warmup", "1"], capture_output=True, text=True, timeout=600,
                           env=dict(os.environ, RANK="1", WORLD_SIZE="2"))
    assert other.returncode == 0 and other.stdout.strip() == ""


def test_aggregated_artefacts_have_upstream_names_and_columns(tmp_path):
    """summary_statistics.json / all_experiments.csv (upstream train_st_interp.py:2790-2908) and the launch-level
    grid_search_summary.csv / grid_search_detail.csv / grid_search_configs.json|csv (run_grid_search.py:102-237):
    names, keys and column order as upstream writes them, built from per-experiment results.json files."""
    import json
    import pandas as pd
    from scripts.train_st_interp import aggregate_results, collect_experiment_results, METRIC_KEYS
    from scripts.run_grid_search import merge_outputs, generate_config_combinations
    base = dict(n_experiments=3, obs_method="site-wise", obs_ratio=0.1, obs_spatial_pattern="corner")
    cfgs = generate_config_combinations(base, {"lr": [1e-2, 2e-2], "basis_mode": ["uniform-fixed", "gmm-learnable"]})
    rng = np.random.default_rng(0)
    for c in cfgs[:3]:                      # the 4th config "failed": no results on disk
        for e in range(1, 4):
            d = tmp_path / f"config_{c['config_id']:03d}" / f"experiment_{e:03d}"
            d.mkdir(parents=True)
            m = lambda: {k: float(rng.random()) for k in ("mse", "mae", "rmse")}
            json.dump({"experiment_id": e, "experiment_seed": 2024 + e, "metrics": {"train": m(), "valid": m(), "test": m()},
                       "total_time_seconds": float(rng.random())}, open(d / "results.json", "w"))
    assert collect_experiment_results(tmp_path / "config_004", [1, 2, 3]) is None
    df_s, df_d = merge_outputs(cfgs, tmp_path)
    s1 = json.load(open(tmp_path / "config_001" / "summary_statistics.json"))
    assert s1["n_experiments"] == 3 and list(s1["statistics"]) == list(METRIC_KEYS)
    assert list(s1["statistics"]["test_rmse"]) == ["mean", "std", "min", "max", "median", "values"]
    ae = pd.read_csv(tmp_path / "config_001" / "all_experiments.csv")
    assert list(ae.columns) == ["experiment_id", "experiment_seed", *METRIC_KEYS] and len(ae) == 3
    summ = pd.read_csv(tmp_path / "grid_search_summary.csv")
    head = ["config_id", "tag", "spatial_basis_function", "spatial_init_method", "spatial_learnable", "obs_method",
            "obs_ratio", "obs_spatial_pattern", "n_experiments"]
    assert list(summ.columns[:9]) == head and list(summ.columns[9:14]) == [f"test_rmse_{k}" for k in ("mean", "std", "min", "max", "median")]
    assert len(summ) == 3 and len(summ.columns) == 9 + 10 * 5
    det = pd.read_csv(tmp_path / "grid_search_detail.csv")
    assert len(det) == 9 and list(det.columns[:3]) == ["config_id", "tag", "experiment_id"] and "test_rmse" in det.columns
    cj = json.load(open(tmp_path / "grid_search_configs.json"))
    assert sorted(cj) == ["1", "2", "3"] and (tmp_path / "grid_search_configs.csv").exists()
    v = s1["statistics"]["test_mae"]["values"]
    assert abs(summ.loc[summ.config_id == 1, "test_mae_mean"].item() - np.mean(v)) < 1e-12


def test_gmm_fit_is_shared_between_processes_through_files(tmp_path, monkeypatch):
    """Sweeps: every (sample, k) mixture fit is done once per box; other processes read the published file."""
    import numpy as np
    from st_dadk_b200 import knot_init as ki
    monkeypatch.setenv("STDADK_GMM_CACHE_DIR", str(tmp_path))
    ki._GMM_CACHE.clear()
    rng = np.random.default_rng(0)
    sub = rng.random((400, 2))
    m1, c1 = ki._gmm_fit(sub, 9)
    files = sorted(p.name for p in tmp_path.iterdir())
    assert any(f.endswith("_9.npz") for f in files) and any(f.endswith("_9.lock") for f in files)
    ki._GMM_CACHE.clear()                      # "another process": no in-memory memo, must come from the file
    calls = []
    import sklearn.mixture as sm
    orig = sm.GaussianMixture.fit
    monkeypatch.setattr(sm.GaussianMixture, "fit", lambda self, X: calls.append(1) or orig(self, X))
    m2, c2 = ki._gmm_fit(sub, 9)
    assert not calls and np.array_equal(m1, m2) and np.array_equal(c1, c2)
    m3, _ = ki._gmm_fit(sub, 4)                 # a different k is a different fit
    assert calls and m3.shape == (4, 2)


def test_bench_dump_outputs(tmp_path):
    """`bench.py --dump-outputs DIR`: the last step's loss, the model's state_dict and the EMA weights as float32 .npy
    files under the upstream state_dict names, leaving the live weights as they were; the option and --steps are
    checked before any work starts."""
    import os
    import subprocess
    import sys
    import types
    import bench
    from stnf.models import STInterpMLP
    from st_dadk_b200.trainer import FlatState
    torch.manual_seed(0)
    model = STInterpMLP(k_spatial_centers=[9, 25], k_temporal_centers=[4], hidden_dims=[32, 16])
    fl = FlatState(model, "cpu")
    fl.shadow.mul_(0.5)
    p0 = fl.p.clone()
    nbytes = bench.dump_outputs(str(tmp_path), types.SimpleNamespace(model=model, flat=fl, loss_last=torch.tensor([0.25])))
    assert torch.equal(fl.p, p0)
    keys = set(model.state_dict())
    assert {f[:-len(".npy")] for f in os.listdir(tmp_path)} == {"loss"} | {"model." + k for k in keys} | {"ema." + k for k in keys}
    assert nbytes == 4 * (1 + 2 * sum(v.numel() for v in model.state_dict().values()))
    w = np.load(tmp_path / "model.mlp.0.weight.npy")
    assert w.dtype == np.float32 and np.array_equal(w, model.mlp[0].weight.detach().numpy())
    assert np.array_equal(np.load(tmp_path / "ema.mlp.0.weight.npy"), 0.5 * w)
    assert np.load(tmp_path / "loss.npy").tolist() == [0.25]
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for bad in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path / "x")],
                ["--config", "3", "--dump-outputs", str(tmp_path / "x")]):
        r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), *bad], capture_output=True, text=True, timeout=60)
        assert r.returncode == 2 and "error" in r.stderr, (bad, r.stderr)
    assert not (tmp_path / "x").exists()
