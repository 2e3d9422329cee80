"""A Trainer the caller drops is freed at once, with its captured CUDA graphs, rather than whenever the cyclic garbage
collector next runs: a graph freed by the collector inside another capture on the same thread (or any thread, in
global capture mode) invalidates that capture."""
import gc
import weakref

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def test_dropped_trainer_is_freed_without_the_cyclic_collector():
    from stnf.dataio import ObservationTable
    from stnf.models import STInterpMLP
    from st_dadk_b200.trainer import Trainer
    dev = torch.device("cuda", 0)
    torch.manual_seed(5)
    model = STInterpMLP(hidden_dims=[64, 32], dropout=0.1, layernorm=True, output_dim=1)
    rng = np.random.default_rng(5)
    n, batch = 2048, 1024
    table = ObservationTable(torch.from_numpy(rng.random((n, 2), dtype=np.float32)),
                             torch.from_numpy(rng.random(n, dtype=np.float32)),
                             torch.from_numpy(rng.standard_normal(n).astype(np.float32))).to(dev)
    cfg = dict(lr=1e-3, weight_decay=0.0, regression_type="mean", epochs=1, hidden_dims=[64, 32], dropout=0.1)
    tr = Trainer(model, cfg, dev, batches_per_epoch=2, use_cuda_graph=True)
    perm = torch.randperm(n, device=dev)
    for i in range(3):                      # the first call captures the step's graph, the others replay it
        tr.train_step(table, perm, (i % 2) * batch, batch)
    torch.cuda.synchronize()
    assert tr._graphs, "the trainer should hold a captured graph"
    alive = weakref.ref(tr)
    gc_on = gc.isenabled()
    gc.disable()
    try:
        del tr
        assert alive() is None, [type(r).__name__ for r in gc.get_referrers(alive())]
    finally:
        if gc_on:
            gc.enable()
