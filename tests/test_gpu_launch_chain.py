"""The training step's kernels are chained by programmatic dependent launch: in the captured graph of a one-wave step
(the bench's model at batch 4,096), pack -> layer_fwd x 3 -> layer_bwd x 3 -> wgrad of block 1 -> fused step tail are
joined by programmatic edges, so each kernel can start while its predecessor runs.  A torch op slipped between two of
them, or a launch without the attribute, breaks the chain."""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

PROGRAMMATIC = 1                  # CU_GRAPH_DEPENDENCY_TYPE_PROGRAMMATIC
KERNEL_NODE = 0                   # CU_GRAPH_NODE_TYPE_KERNEL


class EdgeData(C.Structure):      # CUgraphEdgeData
    _fields_ = [("from_port", C.c_ubyte), ("to_port", C.c_ubyte), ("type", C.c_ubyte), ("reserved", C.c_ubyte * 5)]


def _check(r, what):
    assert r == 0, f"{what}: CUresult {r}"


def _graph_edges(cu, graph):
    n = C.c_size_t(0)
    _check(cu.cuGraphGetEdges_v2(C.c_void_p(graph), None, None, None, C.byref(n)), "cuGraphGetEdges_v2")
    src, dst, data = (C.c_void_p * n.value)(), (C.c_void_p * n.value)(), (EdgeData * n.value)()
    _check(cu.cuGraphGetEdges_v2(C.c_void_p(graph), src, dst, data, C.byref(n)), "cuGraphGetEdges_v2")
    return [(src[i], dst[i], data[i].type) for i in range(n.value)]


def _kernel_name(cu, node, names):
    if node in names:
        return names[node]
    t = C.c_int(-1)
    _check(cu.cuGraphNodeGetType(C.c_void_p(node), C.byref(t)), "cuGraphNodeGetType")
    name = ""
    if t.value == KERNEL_NODE:
        params = (C.c_ubyte * 256)()          # CUDA_KERNEL_NODE_PARAMS_v2: the CUfunction comes first
        _check(cu.cuGraphKernelNodeGetParams_v2(C.c_void_p(node), params), "cuGraphKernelNodeGetParams_v2")
        func = C.c_void_p.from_buffer(params).value
        s = C.c_char_p()
        _check(cu.cuFuncGetName(C.byref(s), C.c_void_p(func)), "cuFuncGetName")
        name = s.value.decode()
    names[node] = name
    return name


# the chain in launch order: (what, substring of the mangled kernel name)
CHAIN = [("pack", "pack_images_kernel")] + [("fwd", "layer_fwd_kernel")] * 3 + [("bwd", "layer_bwd_kernel")] * 3 + \
    [("wgrad block 1", "wgrad_kernelILb1"), ("tail", "adamw_ema_kernelILb1")]


def test_training_step_is_a_programmatic_chain():
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
    perm = torch.randperm(n, device=dev)
    tr.train_step(table, perm, 0, batch)          # eager: kernel attributes and workspaces
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph(keep_graph=True)
    with torch.cuda.graph(g):
        tr._step_body(table, perm, batch, batch, batch)
    graph = g.raw_cuda_graph()

    cu = C.CDLL("libcuda.so.1")
    edges = _graph_edges(cu, graph)
    names = {}
    prog = {}
    for a, b, typ in edges:
        if typ == PROGRAMMATIC:
            prog.setdefault(a, []).append(b)
    starts = sorted({a for a, _, _ in edges if CHAIN[0][1] in _kernel_name(cu, a, names)})
    assert len(starts) == 1, f"expected one pack_images node, found {len(starts)}"
    node, walked = starts[0], [CHAIN[0][0]]
    for what, key in CHAIN[1:]:
        nxt = [b for b in prog.get(node, []) if key in _kernel_name(cu, b, names)]
        assert len(nxt) == 1, (f"no programmatic edge from {walked[-1]} to {what} (chain so far: {walked}; "
                               f"programmatic successors: {[_kernel_name(cu, b, names) for b in prog.get(node, [])]})")
        node = nxt[0]
        walked.append(what)
    assert walked == [w for w, _ in CHAIN]
