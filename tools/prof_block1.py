"""Profiling driver: the fused basis + Linear1 + LayerNorm/ReLU forward kernel (layer_fwd, block 1) alone on 1M explicit
random points (the throughput regime of bench.py's `roofline` entry)."""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from stnf.models import STInterpMLP
from st_dadk_b200.predict import Predictor
torch.manual_seed(0)
model = STInterpMLP(dropout=0.1).to("cuda").eval()
pr = Predictor(model, static_weights=True)
n = int(os.environ.get("ROWS", str(1 << 20)))
g = torch.Generator().manual_seed(5)
c, t = torch.rand(n, 2, generator=g).cuda(), torch.rand(n, generator=g).cuda()
if os.environ.get("SORTED"):
    o = torch.argsort(torch.floor(c[:, 0] * 32.0) * 2.0 + c[:, 1]); c, t = c[o].contiguous(), t[o].contiguous()
r = pr.profile_block1(c, t, repeats=3)
print("block-1 forward", r["rows"], "rows", r["ms"], "ms", r["bytes"] / r["ms"] / 1e6, "GB/s", "frac of 6531.9:", r["bytes"] / r["ms"] / 1e6 / 6531.9)
if os.environ.get("FWD_DBG"):
    # library built with -DSTDADK_PF_DEBUG (tools/build_dbg.sh, STDADK_LIB=...): where a tile's life goes
    import ctypes
    from st_dadk_b200 import _lib as L
    cnt = torch.zeros(16, dtype=torch.int64, device="cuda")
    L.lib().stdadk_debug_counters(ctypes.c_void_p(cnt.data_ptr()))
    pr.profile_block1(c, t, repeats=1)
    torch.cuda.synchronize()
    L.lib().stdadk_debug_counters(ctypes.c_void_p(0))
    v = cnt.cpu().tolist()
    n_cta = max(v[8], 1)
    names = ["prologue", "generate operand (+ stage waits)", "wait accumulator", "epilogue", "tail (barrier, dealloc)"]
    print("CTAs", v[8], "mean ns per CTA:", {k: round(v[i] / n_cta) for i, k in enumerate(names)}, "sum", round(sum(v[:5]) / n_cta),
          "| worker thread 0 waiting for a free stage:", round(v[5] / n_cta), " MMA thread waiting for operands:", round(v[6] / n_cta),
          " producer waiting for a free stage:", round(v[7] / n_cta), "| before / in the launch wait:", round(v[9] / n_cta),
          round(v[10] / n_cta))
