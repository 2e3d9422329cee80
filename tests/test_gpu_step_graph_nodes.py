"""The captured training step of the bench's model has no copy nodes: the Linear head is read from its parameters in the
flat buffer, with no per-step copy into separate head buffers, so the graph starts at pack_images."""
import ctypes as C

import pytest
import torch

from test_gpu_launch_chain import _check, _graph_edges, _kernel_name

pytestmark = pytest.mark.gpu

MEMCPY_NODE = 1                   # CU_GRAPH_NODE_TYPE_MEMCPY


def test_bench_step_graph_has_no_copies_and_starts_at_pack():
    import numpy as np
    from stnf.models import STInterpMLP
    from stnf.dataio import ObservationTable
    from st_dadk_b200.trainer import Trainer
    dev = torch.device("cuda", 0)
    torch.manual_seed(2025)
    model = STInterpMLP(k_spatial_centers=[25, 81, 121], k_temporal_centers=[10, 15, 45], hidden_dims=[256, 256, 128],
                        dropout=0.1, layernorm=True, output_dim=1)
    rng = np.random.default_rng(0)
    n, batch = 8192, 4096
    coords = torch.from_numpy(rng.random((n, 2), dtype=np.float32))
    t = torch.from_numpy(rng.random(n, dtype=np.float32))
    y = torch.from_numpy(rng.standard_normal(n).astype(np.float32))
    table = ObservationTable(coords, t, y).to(dev)
    cfg = dict(lr=2e-2, weight_decay=5e-4, grad_clip=10.0, regression_type="mean", scheduler="cosine", epochs=10,
               dropout=0.1, layernorm=True, hidden_dims=[256, 256, 128], k_spatial_centers=[25, 81, 121],
               k_temporal_centers=[10, 15, 45])
    tr = Trainer(model, cfg, dev, batches_per_epoch=2, use_cuda_graph=False)
    assert tr.head_w.data_ptr() == model.mlp[-1].weight.data_ptr()
    assert tr.head_b.data_ptr() == model.mlp[-1].bias.data_ptr()
    perm = torch.randperm(n, device=dev)
    tr.train_step(table, perm, 0, batch)          # eager: kernel attributes and workspaces
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph(keep_graph=True)
    with torch.cuda.graph(g):
        tr._step_body(table, perm, batch, batch, batch)
    graph = g.raw_cuda_graph()

    cu = C.CDLL("libcuda.so.1")
    n_nodes = C.c_size_t(0)
    _check(cu.cuGraphGetNodes(C.c_void_p(graph), None, C.byref(n_nodes)), "cuGraphGetNodes")
    nodes = (C.c_void_p * n_nodes.value)()
    _check(cu.cuGraphGetNodes(C.c_void_p(graph), nodes, C.byref(n_nodes)), "cuGraphGetNodes")
    types = {}
    for node in nodes:
        typ = C.c_int(-1)
        _check(cu.cuGraphNodeGetType(C.c_void_p(node), C.byref(typ)), "cuGraphNodeGetType")
        types[node] = typ.value
    assert MEMCPY_NODE not in types.values(), f"node types of the step: {sorted(types.values())}"
    names = {}
    has_pred = {b for _, b, _ in _graph_edges(cu, graph)}
    roots = [_kernel_name(cu, node, names) for node in nodes if node not in has_pred]
    assert len(roots) == 1 and "pack_images_kernel" in roots[0], f"the step starts at {roots}"
