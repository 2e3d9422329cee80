"""Tensor-level wrappers over the C ABI.  PyTorch supplies device memory and the stream; every
arithmetic step runs in libstdadk.so.  All functions require CUDA tensors and raise otherwise."""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence

import torch

from . import _lib as L

TILE_M, SLAB_K, SLAB_FLOATS = 128, 32, 4096


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _ptr(t: Optional[torch.Tensor]):
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("st_dadk_b200: expected a CUDA tensor (there is no CPU path)")
    return t.data_ptr()


def _f32c(t: torch.Tensor, name: str) -> torch.Tensor:
    if not t.is_cuda:
        raise RuntimeError(f"st_dadk_b200: `{name}` must be a CUDA tensor (there is no CPU path)")
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


def pad32(x: int) -> int:
    return (x + 31) & ~31


def image_floats(rows: int, cols: int) -> int:
    return ((rows + TILE_M - 1) // TILE_M) * ((cols + SLAB_K - 1) // SLAB_K) * SLAB_FLOATS


def new_image(rows: int, cols: int, device) -> torch.Tensor:
    return torch.empty(image_floats(rows, cols), dtype=torch.float32, device=device)


def pack_image(src: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """(rows x cols) strided FP32 matrix -> TF32-rounded swizzled operand image."""
    assert src.dim() == 2 and src.dtype == torch.float32
    rows, cols = src.shape
    if out is None:
        out = new_image(rows, cols, src.device)
    L.check(L.lib().stdadk_pack_image(_ptr(src), src.stride(0), src.stride(1), rows, cols, _ptr(out), _stream()),
            "pack_image")
    return out


def pack_images(srcs, outs, parts=None):
    """Pack several strided matrices into their images with one launch; `outs[i]` may be None (allocated).
    parts[i] = 1 asks for the tf32x3 residual image tf32(src - tf32(src)) instead of tf32(src)."""
    res = []
    descs = (L.PackDesc * len(srcs))()
    for i, (src, out) in enumerate(zip(srcs, outs)):
        rows, cols = src.shape
        if out is None:
            out = new_image(rows, cols, src.device)
        descs[i] = L.PackDesc(_ptr(src), src.stride(0), src.stride(1), rows, cols, _ptr(out),
                              int(parts[i]) if parts is not None else 0, 0)
        res.append(out)
    for lo in range(0, len(srcs), 8):
        n = min(8, len(srcs) - lo)
        sub = (L.PackDesc * n)(*descs[lo:lo + n])
        L.check(L.lib().stdadk_pack_images(sub, n, _stream()), "pack_images")
    return res


def unpack_image(img: torch.Tensor, rows: int, cols: int) -> torch.Tensor:
    out = torch.empty(rows, cols, dtype=torch.float32, device=img.device)
    L.check(L.lib().stdadk_unpack_image(_ptr(img), rows, cols, _ptr(out), _stream()), "unpack_image")
    return out


def knots_prepare(centers: torch.Tensor, bandwidths: Optional[torch.Tensor], log_bandwidths: Optional[torch.Tensor],
                  basis_fn: str, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    k = centers.shape[0]
    centers = _f32c(centers, "centers")
    bw = _f32c(bandwidths, "bandwidths") if bandwidths is not None else None
    lbw = _f32c(log_bandwidths, "log_bandwidths") if log_bandwidths is not None else None
    if out is None:
        out = torch.empty(max(k, 1), 4, dtype=torch.float32, device=centers.device)
    L.check(L.lib().stdadk_knots_prepare(_ptr(centers), _ptr(bw), _ptr(lbw), L.CALIBRATION[basis_fn], k, _ptr(out),
                                         _stream()), "knots_prepare")
    return out


def tknots_prepare(centers: torch.Tensor, bandwidths: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    k = centers.shape[0]
    if out is None:
        out = torch.empty(max(k, 1), 2, dtype=torch.float32, device=centers.device)
    L.check(L.lib().stdadk_tknots_prepare(_ptr(_f32c(centers, "t_centers")), _ptr(_f32c(bandwidths, "t_bandwidths")),
                                          k, _ptr(out), _stream()), "tknots_prepare")
    return out


def make_basis(knots4: torch.Tensor, tknots2: torch.Tensor, k_s: int, k_t: int, p_cov: int, basis_fn: str) -> L.Basis:
    return L.Basis(_ptr(knots4), _ptr(tknots2), k_s, k_t, p_cov, L.BASIS_CODE[basis_fn])


class PointsRef(L.Points):
    """stdadk_points plus references that keep the addressed tensors alive as long as the struct is."""
    _keep = None


def make_points(coords: Optional[torch.Tensor] = None, t: Optional[torch.Tensor] = None,
                xcov: Optional[torch.Tensor] = None, grid: Optional[Sequence[int]] = None, row_begin: int = 0,
                n_rows: Optional[int] = None, index: Optional[torch.Tensor] = None) -> L.Points:
    """Array point source (coords (N,2), t (N,1|N)), optionally gathered through `index` (int64 sample ids;
    rows are positions in `index`), or the dense grid (nx, ny, nt)."""
    if grid is not None:
        nx, ny, nt = grid
        if n_rows is None:
            n_rows = nx * ny * nt - row_begin
        return PointsRef(None, None, None, None, nx, ny, nt, 0, row_begin, n_rows)
    if index is not None:
        if index.dtype != torch.int64 or not index.is_cuda or not index.is_contiguous():
            raise RuntimeError("make_points: index must be a contiguous CUDA int64 tensor")
        if n_rows is None:
            n_rows = index.shape[0] - row_begin
    if n_rows is None:
        n_rows = coords.shape[0] - row_begin
    if coords is not None:
        coords, t = _f32c(coords, "coords"), _f32c(t, "t")
    if xcov is not None and xcov.numel() > 0:
        xcov = _f32c(xcov, "X")
    else:
        xcov = None
    pts = PointsRef(_ptr(coords), _ptr(t), _ptr(xcov), _ptr(index), 0, 0, 0, 0, row_begin, n_rows)
    pts._keep = (coords, t, xcov, index)
    return pts


def basis_fwd(basis: L.Basis, pts: L.Points, device) -> tuple:
    n = pts.n_rows
    phi = torch.empty(n, basis.k_s, dtype=torch.float32, device=device)
    psi = torch.empty(n, basis.k_t, dtype=torch.float32, device=device)
    L.check(L.lib().stdadk_basis_fwd(C.byref(basis), C.byref(pts), _ptr(phi), _ptr(psi), _stream()), "basis_fwd")
    return phi, psi


def make_layer(w_img, bias, gamma, beta, n_in, n_out, eps, layer_id, w_img_lo=None) -> L.Layer:
    return L.Layer(_ptr(w_img), _ptr(bias), _ptr(gamma), _ptr(beta), n_in, n_out, eps, layer_id, _ptr(w_img_lo))


def make_head(w, b, q, yhat, loss_type=L.LOSS_NONE, y=None, taus=None, inv_count=0.0, dyhat=None, loss_acc=None,
              nc_weight=0.0, nc_power=1) -> L.Head:
    h = L.Head()
    h.w, h.b, h.q, h.loss_type, h.y = _ptr(w), _ptr(b), q, loss_type, _ptr(y)
    for i, tau in enumerate(taus or []):
        h.taus[i] = float(tau)
    h.inv_count, h.nc_weight, h.nc_power = inv_count, nc_weight, nc_power
    h.yhat, h.dyhat, h.loss_acc = _ptr(yhat), _ptr(dyhat), _ptr(loss_acc)
    return h


def layer_fwd(args: L.FwdArgs):
    L.check(L.lib().stdadk_layer_fwd(C.byref(args), _stream()), "layer_fwd")


def predict_supported(args: L.PredictArgs) -> bool:
    return bool(L.lib().stdadk_predict_supported(C.byref(args)))


def predict(args: L.PredictArgs):
    """Whole-network forward (basis -> hidden blocks -> head) in one persistent kernel."""
    L.check(L.lib().stdadk_predict(C.byref(args), _stream()), "predict")


def predict_field_supported(args: L.FieldArgs) -> bool:
    return bool(L.lib().stdadk_predict_field_supported(C.byref(args)))


def predict_field(args: L.FieldArgs):
    """Space-time field prediction: basis + block 1 once per tile of sites, loop over the time steps."""
    L.check(L.lib().stdadk_predict_field(C.byref(args), _stream()), "predict_field")


def layer_bwd(args: L.BwdArgs):
    L.check(L.lib().stdadk_layer_bwd(C.byref(args), _stream()), "layer_bwd")


def wgrad(args: L.WgradArgs):
    L.check(L.lib().stdadk_wgrad(C.byref(args), _stream()), "wgrad")


def knot_grad(args: L.KnotGradArgs):
    L.check(L.lib().stdadk_knot_grad(C.byref(args), _stream()), "knot_grad")


def dense_basis_supported(p_cov: int, k_s: int, k_t: int, n_out: int, q_head: int, training: bool = True) -> tuple:
    """(fits, reason): whether the dense block-1 launches of a training step (training=True) or of a prediction hold
    this shape in shared memory; reason names the launch that does not."""
    lib = L.lib()
    if lib.stdadk_dense_basis_supported(p_cov + k_s + k_t, n_out, k_s, k_t, q_head, int(training)):
        return True, ""
    return False, lib.stdadk_last_error().decode("utf-8", "replace")


def dense_max_knots(p_cov: int, k_t: int, n_out: int, q_head: int, training: bool = True) -> int:
    """Largest number of spatial knots for which dense_basis_supported holds (-1: none)."""
    return int(L.lib().stdadk_dense_max_knots(p_cov, k_t, n_out, q_head, int(training)))


_sqnorm_ws = {}


def grad_sqnorm(g: torch.Tensor, group_end: Sequence[int], out: torch.Tensor, workspace: Optional[torch.Tensor] = None):
    """Squared L2 norm per parameter group, bitwise deterministic.  `workspace` (zero-initialised, reused across
    calls on one stream) defaults to a per-device buffer."""
    if workspace is None:
        workspace = _sqnorm_ws.get(g.device)
        if workspace is None:
            workspace = _sqnorm_ws[g.device] = torch.zeros(L.lib().stdadk_sqnorm_ws_floats(), device=g.device)
    arr = (C.c_int64 * len(group_end))(*group_end)
    L.check(L.lib().stdadk_grad_sqnorm(_ptr(g), g.numel(), len(group_end), arr, _ptr(out), _ptr(workspace), _stream()),
            "grad_sqnorm")


def adamw_ema_step(p, g, m, v, shadow, group_end: Sequence[int], hyper: torch.Tensor, sqnorms, step_count,
                   beta1=0.9, beta2=0.999, eps=1e-8, ema_decay=0.0, zero_grad=False, loss_acc=None, loss_sum=None,
                   loss_last=None, norm_ws=None, state_early=False):
    """zero_grad: the kernel leaves `g` zeroed (next step's zero_grad); loss_acc/loss_sum: device scalars,
    loss_sum += loss_acc; loss_acc = 0 inside the same launch.  norm_ws (zero-initialised (148*8+8) floats): ONE launch for
    the whole step tail -- the kernel computes the squared gradient norms itself (into `sqnorms`, which stays None when
    clipping is off) and advances the step counter.  state_early (with norm_ws): the kernel launched just before writes
    none of p / m / v / shadow / hyper / step_count, so the tail loads them while that kernel still runs."""
    arr = (C.c_int64 * len(group_end))(*group_end)
    a = L.AdamWArgs(_ptr(p), _ptr(g), _ptr(m), _ptr(v), _ptr(shadow), p.numel(), len(group_end), int(bool(zero_grad)),
                    arr, _ptr(hyper), _ptr(sqnorms), _ptr(step_count), beta1, beta2, eps, ema_decay, _ptr(loss_acc),
                    _ptr(loss_sum), _ptr(loss_last), int(norm_ws is not None), int(bool(state_early)), _ptr(norm_ws))
    L.check(L.lib().stdadk_adamw_ema_step(C.byref(a), _stream()), "adamw_ema_step")


def peer_allreduce(args: L.PeerAllreduceArgs):
    """One-shot sum of the ranks' gradient buffers over peer memory (see st_dadk_b200/peer.py)."""
    L.check(L.lib().stdadk_peer_allreduce(C.byref(args), _stream()), "peer_allreduce")


def make_sparse_args(pts: L.Points, knots4, basis_fn: str, n_out: int, p_cov: int, sides=None, offsets=None,
                     thetaps=None, w1t=None, zs=None, dz_img=None, dw1t=None, celllist=None, n_levels=None,
                     d_centers=None, d_log_bw=None) -> L.SparseArgs:
    """Lattice mode: sides / offsets / thetaps per level.  Cell-list mode: `celllist` (workspace filled by
    celllist_build for these knots) and `n_levels`."""
    a = L.SparseArgs()
    a.pts = pts
    a.knots4 = _ptr(knots4)
    a.basis_fn, a.n_out, a.p_cov = L.BASIS_CODE[basis_fn], n_out, p_cov
    if celllist is not None:
        a.n_levels, a.celllist, a.celllist_k_s = int(n_levels), _ptr(celllist), int(knots4.shape[0])
    else:
        a.n_levels = len(sides)
        for i, (sd, of, th) in enumerate(zip(sides, offsets, thetaps)):
            a.side[i], a.offset[i], a.thetap[i] = int(sd), int(of), float(th)
    a.w1t, a.zs, a.dz_img, a.dw1t = _ptr(w1t), _ptr(zs), _ptr(dz_img), _ptr(dw1t)
    a.d_centers, a.d_log_bw = _ptr(d_centers), _ptr(d_log_bw)
    return a


def celllist_build(knots4: torch.Tensor, level_begin: Sequence[int], ws: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Per-level cell list of an arbitrary knot set (knots4 rows: cx, cy, theta'^2, 1/theta'); levels are the contiguous
    knot ranges level_begin[l] : level_begin[l + 1].  Returns the (reusable) workspace tensor."""
    k_s, nl = int(knots4.shape[0]), len(level_begin) - 1
    need = L.lib().stdadk_celllist_ws_bytes(k_s, nl)
    if need == 0:
        raise RuntimeError(f"celllist_build: unsupported shape (k_s={k_s}, levels={nl})")
    if ws is None or ws.numel() * 4 < need:
        ws = torch.empty((need + 3) // 4, dtype=torch.int32, device=knots4.device)
    arr = (C.c_int32 * (nl + 1))(*[int(v) for v in level_begin])
    L.check(L.lib().stdadk_celllist_build(_ptr(knots4), k_s, arr, nl, _ptr(ws), ws.numel() * 4, _stream()), "celllist_build")
    return ws


def sparse_l1_fwd(args: L.SparseArgs):
    L.check(L.lib().stdadk_sparse_l1_fwd(C.byref(args), _stream()), "sparse_l1_fwd")


def sparse_l1_wgrad(args: L.SparseArgs):
    L.check(L.lib().stdadk_sparse_l1_wgrad(C.byref(args), _stream()), "sparse_l1_wgrad")
