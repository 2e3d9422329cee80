"""Forward / backward chains of the ST-DADK network on libstdadk kernels.

`NetSpec` is a view of the model's tensors (owned by the nn.Module or by the trainer's flat buffer);
`Executor` owns the operand images, activation workspaces and the flat gradient buffer, and issues
the kernel sequence

    forward : layer_fwd(basis -> h1) -> layer_fwd(h1 -> h2) -> ... -> layer_fwd(h_{L-1} -> head [+loss])
    backward: layer_bwd(L) -> ... -> layer_bwd(1), then wgrad(l) for every block, then knot_grad

mirroring STInterpMLP.forward (stnf/models/st_interp.py:827-882) and its autograd.
"""
from __future__ import annotations

import os
import ctypes as C
from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence, Tuple

import torch

from . import _lib as L
from . import ops


@dataclass
class NetSpec:
    centers: torch.Tensor                      # (K_s, 2)
    bandwidths: Optional[torch.Tensor]         # (K_s,) fixed basis
    log_bandwidths: Optional[torch.Tensor]     # (K_s,) learnable basis (theta = exp(.))
    t_centers: torch.Tensor
    t_bandwidths: torch.Tensor
    weights: List[torch.Tensor]                # hidden Linear weights, logical shape (out, in), any strides
    biases: List[torch.Tensor]
    gammas: List[Optional[torch.Tensor]]
    betas: List[Optional[torch.Tensor]]
    head_w: torch.Tensor                       # (Q, d) effective head
    head_b: torch.Tensor                       # (Q,)
    basis_fn: str = "wendland"
    p_cov: int = 0
    dropout: float = 0.0
    ln_eps: float = 1e-5
    learnable_basis: bool = False
    lattice_sides: Optional[List[int]] = None  # knots per axis of each level when the knots are the fixed uniform lattice
    level_sizes: Optional[List[int]] = None    # knots per resolution level (contiguous ranges of `centers`); None = one level
    # "tf32": one tensor-core pass on TF32-rounded operands (throughput mode; outputs within 1e-3 of the FP32 reference).
    # "tf32x3": every operand is split into tf32(x) + tf32(x - tf32(x)) and every GEMM runs hi*hi + hi*lo + lo*hi into
    # the same FP32 accumulator: FP32-faithful products, for runs that must track the reference's FP32 trajectory.
    precision: str = "tf32"

    @property
    def n_hidden(self):
        return len(self.weights)

    @property
    def q(self):
        return self.head_w.shape[0]


@dataclass
class LossSpec:
    kind: str = "mse"                          # "mse" | "pinball"
    taus: Sequence[float] = ()
    nc_weight: float = 0.0
    nc_power: int = 1


class _Workspace:
    def __init__(self, spec: NetSpec, n_rows: int, device, sparse: bool = False, save_x: bool = False,
                 save_feat: bool = False):
        self.n_rows = n_rows
        # block-1 operand [X|phi|psi] as an image, kept for LARGE batches (see Executor.SAVE_FEAT_MIN_ROWS)
        self.feat = ops.new_image(n_rows, spec.weights[0].shape[1], device) if save_feat else None
        self.zs = torch.empty(n_rows, spec.weights[0].shape[0], dtype=torch.float32, device=device) if sparse else None
        self.h = [ops.new_image(n_rows, w.shape[0], device) for w in spec.weights[:-1]]
        self.dz = [ops.new_image(n_rows, w.shape[0], device) for w in spec.weights]
        x3 = spec.precision == "tf32x3"                 # residual images of every activation / dz image
        self.h_lo = [ops.new_image(n_rows, w.shape[0], device) for w in spec.weights[:-1]] if x3 else None
        self.dz_lo = [ops.new_image(n_rows, w.shape[0], device) for w in spec.weights] if x3 else None
        self.stats = [torch.empty(n_rows, 2, dtype=torch.float32, device=device) if g is not None else None
                      for g in spec.gammas]
        # pre-LayerNorm x of every block, kept only for single-wave batches (see Executor.SAVE_X_MAX_ROWS)
        self.x = [ops.new_image(n_rows, w.shape[0], device) for w in spec.weights] if save_x else None
        self.yhat = torch.empty(n_rows, spec.q, dtype=torch.float32, device=device)
        self.dyhat = torch.empty(n_rows, spec.q, dtype=torch.float32, device=device)


class Executor:
    MAX_WORKSPACES = 4
    # Above this many spatial knots block 1 switches from generating every basis column densely in the tensor-core
    # operand to walking each point's compact support (st_dadk_b200/csrc/sparse.cuh): dense work grows with K_s, the
    # walk with the ~20 knots per level inside a support disk.  This is the performance crossover only.  The dense
    # kernels keep block 1's knot tables in shared memory, and below it they may already not hold them: at first
    # width 256 and 70 temporal knots the recompute backward takes at most 1,626 knots
    # (stdadk_dense_basis_supported).  Such networks walk as well, and raise at construction when they cannot.
    DENSE_MAX_KNOTS = 2048
    # Up to this many rows a training forward also stores x = A W^T + b of every block (1 KB/row/block) so that the
    # backward skips its recomputation GEMM (and, for block 1, regenerating the basis for it): a batch this small is at
    # most two CTAs of 128 rows per SM, bound by per-kernel latency, not by HBM.  Larger batches recompute instead.
    # Batches of at most 128 rows per two SMs (9,472 on 148 SMs) run layer_fwd / layer_bwd in one wave of 64-row tiles.
    # (The N x K basis matrix is never stored either way; wgrad regenerates it.)
    SAVE_X_MAX_ROWS = 148 * 2 * 128
    # Beyond that the step is throughput-bound and evaluating the basis three times (forward, the backward's recompute
    # GEMM of block 1, wgrad of block 1) is its largest single cost (batch 65,536: backward 147 us and wgrad 139 us
    # for block 1 against 102 / 47 us for block 2).  OPTIONAL (`store_basis_operand = True`): the forward also writes
    # its generated operand (1.25 KB/row) and the other two read it back through TMA like any activation image:
    # 0.74 -> 0.64 ms per step at 65,536 rows, 2.48 -> 2.12 ms at 262,144.  Off by default: the design point of this
    # path is that the N x K basis matrix is never materialised in HBM and the backward recomputes it.
    SAVE_FEAT_MIN_ROWS = SAVE_X_MAX_ROWS + 1
    store_basis_operand = False

    def __init__(self, spec: NetSpec, force_sparse: bool = False, force_dense: bool = False):
        self.spec = spec
        self.force_sparse = force_sparse
        # keep the dense operand even above DENSE_MAX_KNOTS.  Raises at construction when the dense forward cannot hold
        # the knots; when only the training launches cannot (predict_only), training calls raise before any launch.
        self.force_dense = force_dense
        self._setup_regime(spec)
        dev = spec.centers.device
        if dev.type != "cuda":
            raise RuntimeError("st_dadk_b200.Executor needs CUDA tensors: the hot path has no CPU implementation")
        self.device = dev
        self._ws: Dict[int, _Workspace] = {}
        self.on_evict = None
        self._ctx = None
        self._pack_key = None
        self.w_img: List[torch.Tensor] = [None] * spec.n_hidden
        self.wt_img: List[torch.Tensor] = [None] * spec.n_hidden
        self.w1s_img = None
        self.w_img_lo: List[torch.Tensor] = [None] * spec.n_hidden      # tf32x3 residual images
        self.wt_img_lo: List[torch.Tensor] = [None] * spec.n_hidden
        self.w1s_img_lo = None
        self.knots4 = torch.empty(max(spec.centers.shape[0], 1), 4, dtype=torch.float32, device=dev)
        self.tknots2 = torch.empty(max(spec.t_centers.shape[0], 1), 2, dtype=torch.float32, device=dev)
        self.loss_acc = torch.zeros(1, dtype=torch.float32, device=dev)
        self._grad_flat = None
        self.grads = None
        self._knots_ready = False
        self._side = None
        self.fused_predict = True      # forward-only calls use the whole-network kernel when the shape fits
        # the one-wave backward and the fused step tail read settled inputs (dropout step, saved x images, optimizer
        # state) before their programmatic-launch wait; STDADK_PREWAIT=0 makes them read everything after it (same
        # results, for comparison)
        self.prewait = os.environ.get("STDADK_PREWAIT", "1") != "0"
        self._fused_ok = None
        self._field_ok = None
        self._cell_ws = None
        self._w1sf_img = None
        self._w1sf_key = None
        self._zt_ws = None

    @property
    def x3(self) -> bool:
        return self.spec.precision == "tf32x3"

    def _setup_regime(self, spec: NetSpec):
        if spec.precision not in ("tf32", "tf32x3"):
            raise ValueError(f"precision must be 'tf32' or 'tf32x3', got {spec.precision!r}")
        k_s, k_t = spec.centers.shape[0], spec.t_centers.shape[0]
        n_out = spec.weights[0].shape[0]
        q_head = spec.q if spec.n_hidden == 1 else 0        # a single hidden block carries the head
        fits, why = ops.dense_basis_supported(spec.p_cov, k_s, k_t, n_out, q_head)
        too_big = ""
        self.predict_only = None
        if not fits:
            limit = ops.dense_max_knots(spec.p_cov, k_t, n_out, q_head)
            too_big = (f"the dense path holds at most {limit} spatial knots with a first block of {n_out} outputs "
                       f"and {k_t} temporal knots ({why})")
            if self.force_dense:
                # forced dense: predictions need the forward only; training calls are refused before any launch
                fwd_fits, fwd_why = ops.dense_basis_supported(spec.p_cov, k_s, k_t, n_out, q_head, training=False)
                if not fwd_fits:
                    fwd_limit = ops.dense_max_knots(spec.p_cov, k_t, n_out, q_head, training=False)
                    raise RuntimeError(f"force_dense: {k_s} spatial knots do not fit: the dense forward holds at most "
                                       f"{fwd_limit} spatial knots with a first block of {n_out} outputs and {k_t} "
                                       f"temporal knots ({fwd_why})")
                self.predict_only = f"force_dense: {k_s} spatial knots can be predicted but not trained: {too_big}"
        want = self.force_sparse or (not self.force_dense and (k_s > self.DENSE_MAX_KNOTS or not fits))
        self.sparse = False
        self.lat = None
        self.level_begin = None
        if not want:
            return
        problems = []
        if spec.basis_fn == "gaussian":
            problems.append("the gaussian basis is not compactly supported")
        if spec.p_cov != 0:
            problems.append("covariates are not supported together with the support walk")
        if spec.weights[0].shape[0] % 4:
            problems.append("first hidden width must be a multiple of 4")
        sizes = [int(v) for v in (spec.level_sizes or [k_s])]
        if sum(sizes) != k_s or len(sizes) > 8:
            problems.append("level_sizes must be at most 8 contiguous ranges adding up to the number of knots")
        if problems:
            if self.force_sparse or not fits:
                reason = f" ({too_big})" if too_big else ""
                raise RuntimeError(f"{k_s} spatial knots need the support-walking path{reason}, but " + "; ".join(problems))
            return          # above DENSE_MAX_KNOTS, but the dense kernels still hold the knots
        if spec.lattice_sides is not None and not spec.learnable_basis:
            # fixed uniform lattice: candidate windows in closed form
            sides = [int(v) for v in spec.lattice_sides]
            offs, o = [], 0
            for sd in sides:
                offs.append(o)
                o += sd * sd
            assert o == k_s, "lattice_sides do not add up to the number of knots"
            bw = spec.bandwidths[torch.tensor(offs, device=spec.bandwidths.device)].float().cpu().numpy()
            import numpy as _np
            calib = _np.float32(L.CALIBRATION[spec.basis_fn])
            self.lat = (sides, offs, [float(_np.float32(b) * calib) for b in bw])
        else:
            # any other knot set (gmm / random_site / kmeans_balanced, learnable knots): per-level cell list on the device
            self.level_begin = [0]
            for n in sizes:
                self.level_begin.append(self.level_begin[-1] + n)
        self.sparse = True

    # ------------------------------------------------------------------ operand preparation
    def rebind(self, spec: NetSpec):
        if spec.precision != self.spec.precision:
            self._ws.clear()                       # workspaces carry (or lack) the residual images
            if self.on_evict is not None:
                self.on_evict()
        self.spec = spec
        self._setup_regime(spec)
        self._pack_key = None
        self._knots_ready = False
        self._fused_ok = None
        self._field_ok = None
        self._w1sf_key = None

    def _key(self):
        s = self.spec
        ts = [s.centers, s.bandwidths, s.log_bandwidths, *s.weights]
        return tuple((t.data_ptr(), t._version) for t in ts if t is not None)

    def prepare(self, force: bool = True, for_backward: bool = False):
        """(Re)build knot tables and weight images.  Training calls this every step (weights move);
        evaluation may reuse them while the parameter storage is unchanged."""
        s = self.spec
        key = (self._key(), for_backward)
        if not force and key == self._pack_key:
            return
        if s.learnable_basis or not self._knots_ready:
            ops.knots_prepare(s.centers, s.bandwidths if s.log_bandwidths is None else None, s.log_bandwidths,
                              s.basis_fn, out=self.knots4)
            ops.tknots_prepare(s.t_centers, s.t_bandwidths, out=self.tknots2)   # fixed buffers: only the first time
            if self.sparse and self.level_begin is not None:      # the knots moved (or first use): rebuild the cell list
                self._cell_ws = ops.celllist_build(self.knots4, self.level_begin, self._cell_ws)
            self._knots_ready = True
        srcs, outs, slots, parts = [], [], [], []
        x3 = self.x3

        def add(src, kind, l):
            store = {"w": self.w_img, "wt": self.wt_img, "w1s": None}[kind]
            srcs.append(src); outs.append(store[l] if store is not None else self.w1s_img)
            slots.append((kind, l, 0)); parts.append(0)
            if x3:                                       # residual image of the same matrix
                store = {"w": self.w_img_lo, "wt": self.wt_img_lo, "w1s": None}[kind]
                srcs.append(src); outs.append(store[l] if store is not None else self.w1s_img_lo)
                slots.append((kind, l, 1)); parts.append(1)

        for l, w in enumerate(s.weights):
            if l == 0 and self.sparse:
                k_s = s.centers.shape[0]
                add(w[:, k_s:], "w", l)                  # dense (temporal) columns only; spatial rows are gathered
                wt = w.t()
                self._w1t = wt if wt.is_contiguous() else wt.contiguous()
            else:
                add(w, "w", l)
            if for_backward and l > 0:
                add(w.t(), "wt", l)
        if for_backward and s.learnable_basis and not self.sparse:
            add(s.weights[0][:, s.p_cov:s.p_cov + s.centers.shape[0]].t(), "w1s", 0)   # (K_s, n_out)
        for (kind, l, part), img in zip(slots, ops.pack_images(srcs, outs, parts)):   # one launch per 8 images
            if kind == "w":
                (self.w_img_lo if part else self.w_img)[l] = img
            elif kind == "wt":
                (self.wt_img_lo if part else self.wt_img)[l] = img
            elif part:
                self.w1s_img_lo = img
            else:
                self.w1s_img = img
        self._pack_key = key

    def _workspace(self, n_rows: int) -> _Workspace:
        ws = self._ws.get(n_rows)
        if ws is None:
            if len(self._ws) >= self.MAX_WORKSPACES:
                self._ws.pop(next(iter(self._ws)))
                if self.on_evict is not None:      # whoever captured CUDA graphs over the evicted buffers drops them
                    self.on_evict()
            ws = self._ws[n_rows] = _Workspace(self.spec, n_rows, self.device, self.sparse,
                                               save_x=n_rows <= self.SAVE_X_MAX_ROWS,
                                               save_feat=(self.store_basis_operand and not self.sparse and not self.x3
                                                          and n_rows >= self.SAVE_FEAT_MIN_ROWS))
        return ws

    def _basis(self) -> L.Basis:
        s = self.spec
        k_s = 0 if self.sparse else s.centers.shape[0]     # sparse regime: the tensor-core operand holds [X | psi] only
        return ops.make_basis(self.knots4, self.tknots2, k_s, s.t_centers.shape[0], s.p_cov, s.basis_fn)

    def _n_in(self, l: int) -> int:
        w = self.spec.weights[l]
        return w.shape[1] - (self.spec.centers.shape[0] if (l == 0 and self.sparse) else 0)

    def _layer(self, l: int) -> L.Layer:
        s = self.spec
        w = s.weights[l]
        return ops.make_layer(self.w_img[l], s.biases[l], s.gammas[l], s.betas[l], self._n_in(l), w.shape[0], s.ln_eps, l,
                              self.w_img_lo[l] if self.x3 else None)

    def _sparse_args(self, pts, ws, **kw) -> L.SparseArgs:
        s = self.spec
        if self.lat is not None:
            sides, offs, ths = self.lat
            return ops.make_sparse_args(pts, self.knots4, s.basis_fn, s.weights[0].shape[0], s.p_cov, sides, offs, ths, **kw)
        return ops.make_sparse_args(pts, self.knots4, s.basis_fn, s.weights[0].shape[0], s.p_cov, celllist=self._cell_ws,
                                    n_levels=len(self.level_begin) - 1, **kw)

    # ------------------------------------------------------------------ forward
    def forward(self, pts: L.Points, train: bool = False, step: int = 0, seed: int = 0,
                y: Optional[torch.Tensor] = None, loss: Optional[LossSpec] = None, inv_count: float = 0.0,
                out: Optional[torch.Tensor] = None, save: bool = False, prepared: bool = False,
                step_ptr: Optional[torch.Tensor] = None, key_offset: int = 0):
        """Returns yhat (n_rows, Q).  With `y`/`loss`, also accumulates the loss into self.loss_acc and
        leaves dLoss/dyhat in the workspace for `backward()`.  `save=True` keeps what backward needs."""
        s = self.spec
        n = int(pts.n_rows)
        if n == 0:          # empty batch: nothing to launch (empty tensors have no storage to hand to the library)
            self._ctx = None
            return out if out is not None else torch.empty(0, s.q, dtype=torch.float32, device=self.device)
        if (save or train) and self.predict_only:
            raise RuntimeError(self.predict_only)
        if not prepared:
            # always rebuild the operand images: parameter storage can be rewritten in place by kernels or by
            # an EMA swap without any version counter the executor could observe (5 tiny launches)
            self.prepare(force=True, for_backward=save)
        if not train and not save and loss is None and self.fused_predict and not self.sparse and not self.x3:
            yhat = out if out is not None else torch.empty(n, s.q, dtype=torch.float32, device=self.device)
            if self._predict_fused(pts, yhat):
                return yhat
        ws = self._workspace(n)
        yhat = out if out is not None else ws.yhat
        basis = self._basis()
        drop = L.Dropout(s.dropout if train else 0.0, step & 0xFFFFFFFF, seed,
                         step_ptr.data_ptr() if step_ptr is not None else None, key_offset)
        if self.sparse:
            ops.sparse_l1_fwd(self._sparse_args(pts, ws, w1t=self._w1t, zs=ws.zs))
        for l in range(s.n_hidden):
            a = L.FwdArgs()
            a.pts = pts
            if l == 0:
                a.basis = C.pointer(basis)
                if self.sparse:
                    a.addend = ws.zs.data_ptr()
                if save and ws.feat is not None:
                    a.feat_img = ws.feat.data_ptr()
            else:
                a.a_img = ws.h[l - 1].data_ptr()
                if self.x3:
                    a.a_img_lo = ws.h_lo[l - 1].data_ptr()
            a.layer = self._layer(l)
            a.drop = drop
            if save and ws.stats[l] is not None:
                a.stats = ws.stats[l].data_ptr()
            if save and ws.x is not None:
                a.x_img = ws.x[l].data_ptr()
            if l < s.n_hidden - 1:
                a.out_img = ws.h[l].data_ptr()
                if self.x3:
                    a.out_img_lo = ws.h_lo[l].data_ptr()
            else:
                head = self._make_head(yhat, ws, y, loss, inv_count)
                a.head = C.pointer(head)
            ops.layer_fwd(a)
        if save:
            self._ctx = (pts, drop, ws)
        return yhat

    def _make_head(self, yhat, ws, y, loss, inv_count):
        s = self.spec
        if loss is not None:
            code = L.LOSS_MSE if loss.kind == "mse" else L.LOSS_PINBALL
            return ops.make_head(s.head_w, s.head_b, s.q, yhat, code, y, list(loss.taus), inv_count, ws.dyhat,
                                 self.loss_acc, loss.nc_weight, loss.nc_power)
        return ops.make_head(s.head_w, s.head_b, s.q, yhat)

    def _predict_args(self, pts: L.Points, yhat: torch.Tensor) -> L.PredictArgs:
        """Arguments of the whole-network kernel (stdadk_predict) for this network; needs n_hidden <= MAX_HIDDEN."""
        s = self.spec
        a = L.PredictArgs()
        a.basis = C.pointer(self._basis())
        a.pts = pts
        a.n_layers = s.n_hidden
        for l in range(s.n_hidden):
            a.layers[l] = self._layer(l)
        a.head = C.pointer(ops.make_head(s.head_w, s.head_b, s.q, yhat))
        return a

    def fused_supported(self) -> bool:
        """Whether forward-only calls on this network run through the whole-network kernel (decided once per binding;
        needs the operand images, i.e. prepare() first)."""
        s = self.spec
        if self.sparse or self.x3 or not self.fused_predict or s.n_hidden > L.MAX_HIDDEN:
            return False
        if self._fused_ok is None:
            probe = torch.empty(1, s.q, dtype=torch.float32, device=self.device)
            self._fused_ok = ops.predict_supported(
                self._predict_args(ops.make_points(grid=(1, 1, 1), row_begin=0, n_rows=1), probe))
        return bool(self._fused_ok)

    def _predict_fused(self, pts: L.Points, yhat: torch.Tensor) -> bool:
        """Forward-only path: the whole network in one persistent kernel (stdadk_predict), no activation images.
        Returns False when the shape does not fit the fused kernel; the caller then chains layer_fwd."""
        if self.spec.n_hidden > L.MAX_HIDDEN:
            return False
        a = self._predict_args(pts, yhat)
        if self._fused_ok is None:
            self._fused_ok = ops.predict_supported(a)
        if not self._fused_ok:
            return False
        ops.predict(a)
        return True

    # ------------------------------------------------------------------ space-time field prediction
    def _field_args(self, sites, grid, n_sites, n_times, k0, k1, s0, s1, yhat, row_base, out_k_stride=0) -> L.FieldArgs:
        s = self.spec
        k_s = s.centers.shape[0]
        w1 = s.weights[0]
        key = (w1.data_ptr(), w1._version, self._pack_key)
        if self._w1sf_key != key:      # image of the spatial columns of W1 (forward operand of the site GEMM)
            self._w1sf_img = ops.pack_images([w1[:, s.p_cov:s.p_cov + k_s]], [self._w1sf_img])[0]
            self._w1sf_key = key
        if self._zt_ws is None or self._zt_ws.numel() < n_times * ops.pad32(w1.shape[0]):
            self._zt_ws = torch.empty(n_times * ops.pad32(w1.shape[0]), dtype=torch.float32, device=self.device)
        basis = ops.make_basis(self.knots4, self.tknots2, k_s, s.t_centers.shape[0], 0, s.basis_fn)
        head = ops.make_head(s.head_w, s.head_b, s.q, yhat)
        a = L.FieldArgs()
        a.basis = C.pointer(basis)
        if sites is not None:
            a.sites = sites.data_ptr()
        else:
            a.grid_nx, a.grid_ny = grid
        a.n_sites, a.n_times, a.k_begin, a.k_end = n_sites, n_times, k0, k1
        a.site_begin, a.site_end = s0, s1
        a.n_layers = s.n_hidden
        for l in range(s.n_hidden):
            a.layers[l] = self._layer(l)
        a.layers[0] = ops.make_layer(self._w1sf_img, s.biases[0], s.gammas[0], s.betas[0], k_s, w1.shape[0], s.ln_eps, 0)
        a.w1 = w1.data_ptr()
        a.w1_row_stride, a.w1_col_stride = w1.stride(0), w1.stride(1)
        a.head = C.pointer(head)
        a.row_base = row_base
        a.out_k_stride = out_k_stride
        a.zt_ws = self._zt_ws.data_ptr()
        return a

    def field_supported(self) -> bool:
        """Whether grid / space-time-field predictions of this network run the site-tile x time-loop kernel
        (stdadk_predict_field): dense regime, TF32 mode, no covariates, shape within the kernel's shared memory."""
        s = self.spec
        if self.sparse or self.x3 or not self.fused_predict or s.p_cov != 0 or s.n_hidden > L.MAX_HIDDEN:
            return False
        if self._field_ok is None:
            probe = torch.empty(1, s.q, dtype=torch.float32, device=self.device)
            self._field_ok = ops.predict_field_supported(self._field_args(None, (1, 1), 1, 1, 0, 1, 0, 1, probe, 0))
        return bool(self._field_ok)

    def predict_field(self, yhat: torch.Tensor, begin: int, end: int, n_sites: int, n_times: int,
                      sites: Optional[torch.Tensor] = None, grid: Optional[Tuple[int, int]] = None) -> int:
        """Rows [begin, end) of the (t, s) row-major field (row = k * n_sites + s) into yhat[0 : end - begin].
        The shard is cut into at most three (site range x time range) rectangles -- a partial first time step, whole
        steps, a partial last step -- one launch each.  Returns the number of launches."""
        S = n_sites
        k0, k1 = begin // S, (end - 1) // S if end > begin else begin // S
        rects = []
        if end <= begin:
            return 0
        if k0 == k1:
            rects.append((k0, k0 + 1, begin - k0 * S, end - k0 * S))
        else:
            lo = k0
            if begin > k0 * S:
                rects.append((k0, k0 + 1, begin - k0 * S, S))
                lo = k0 + 1
            hi = k1 + 1
            if end < (k1 + 1) * S:
                hi = k1
            if hi > lo:
                rects.append((lo, hi, 0, S))
            if hi == k1:
                rects.append((k1, k1 + 1, 0, end - k1 * S))
        for (ka, kb, sa, sb) in rects:
            ops.predict_field(self._field_args(sites, grid, S, n_times, ka, kb, sa, sb, yhat, begin))
        return 2 * len(rects)

    def predict_field_sites(self, yhat: torch.Tensor, site_begin: int, site_end: int, n_sites: int, n_times: int,
                            sites: Optional[torch.Tensor] = None, grid: Optional[Tuple[int, int]] = None) -> int:
        """Sites [site_begin, site_end) at ALL n_times steps into yhat viewed as (n_times, site_end - site_begin, Q):
        one rectangle, one launch pair.  The sharding for several GPUs: the per-site work (basis + spatial part of
        block 1) is done once per site on exactly one rank, as on a single GPU."""
        if site_end <= site_begin:
            return 0
        ops.predict_field(self._field_args(sites, grid, n_sites, n_times, 0, n_times, site_begin, site_end, yhat,
                                           site_begin, site_end - site_begin))
        return 2

    # ------------------------------------------------------------------ backward
    def alloc_grads(self, flat: Optional[torch.Tensor] = None, views: Optional[dict] = None):
        """Gradient buffers.  Linear weight gradients are stored (in, out)-contiguous and exposed as
        the transposed (out, in) view so the wgrad epilogue's atomics are coalesced."""
        s = self.spec
        if views is not None:
            self._grad_flat, self.grads = flat, views
            return
        shapes = []
        for w in s.weights:
            shapes.append(w.shape[0] * w.shape[1])
        sizes = shapes + [b.numel() for b in s.biases] + \
            [g.numel() if g is not None else 0 for g in s.gammas] * 2 + \
            [s.head_w.numel(), s.head_b.numel(), s.centers.numel(), s.centers.shape[0]]
        flat = torch.zeros(sum(sizes), dtype=torch.float32, device=self.device)
        o = 0
        g = {"weights": [], "biases": [], "gammas": [], "betas": []}
        for w in s.weights:
            n = w.shape[0] * w.shape[1]
            g["weights"].append(flat[o:o + n].view(w.shape[1], w.shape[0]).t())
            o += n
        for b in s.biases:
            g["biases"].append(flat[o:o + b.numel()])
            o += b.numel()
        for name in ("gammas", "betas"):
            for gm in s.gammas:
                n = gm.numel() if gm is not None else 0
                g[name].append(flat[o:o + n] if n else None)
                o += n
        g["head_w"] = flat[o:o + s.head_w.numel()].view_as(s.head_w)
        o += s.head_w.numel()
        g["head_b"] = flat[o:o + s.head_b.numel()]
        o += s.head_b.numel()
        g["centers"] = flat[o:o + s.centers.numel()].view(-1, 2)
        o += s.centers.numel()
        g["log_bandwidths"] = flat[o:o + s.centers.shape[0]]
        self._grad_flat, self.grads = flat, g

    def _wgrad_block(self, l: int, pts, ws, basis, g):
        """dW_l += dz_l^T A_l (tensor cores; block 1 of the large-knot regime: temporal columns + scattered rows)."""
        s = self.spec
        w = s.weights[l]
        gw = g["weights"][l]
        a = L.WgradArgs()
        a.pts = pts
        if l == 0 and ws.feat is None:
            a.basis = C.pointer(basis)
        else:
            a.a_img = (ws.feat if l == 0 else ws.h[l - 1]).data_ptr()
            if self.x3:
                a.a_img_lo = ws.h_lo[l - 1].data_ptr()
        a.dz_img = ws.dz[l].data_ptr()
        if self.x3:
            a.dz_img_lo = ws.dz_lo[l].data_ptr()
        a.n_in, a.n_out = self._n_in(l), w.shape[0]
        if l == 0 and self.sparse:
            k_s = s.centers.shape[0]
            gd = gw[:, k_s:]                       # dense (temporal) columns on the tensor cores ...
            a.dw = gd.data_ptr()
            a.stride_o, a.stride_i = gd.stride(0), gd.stride(1)
            ops.wgrad(a)
            if gw.stride(0) != 1 or gw.stride(1) != w.shape[0]:
                raise RuntimeError("support-walk wgrad needs the first-layer gradient stored (in, out)-contiguous")
            kg = {}
            if s.learnable_basis:       # knot gradients from the same walk (closed-form chain rule per (point, knot))
                kg = dict(d_centers=g["centers"], d_log_bw=g["log_bandwidths"], w1t=self._w1t)
            ops.sparse_l1_wgrad(self._sparse_args(pts, ws, dz_img=ws.dz[0], dw1t=gw, **kg))   # ... spatial rows scattered
            return
        a.dw = gw.data_ptr()
        a.stride_o, a.stride_i = gw.stride(0), gw.stride(1)
        ops.wgrad(a)

    def backward(self, dyhat: Optional[torch.Tensor] = None, zero: bool = True) -> dict:
        """Gradients of every parameter for the rows of the last `forward(save=True)`.  `dyhat`
        overrides the loss gradient left by the fused loss (used by the autograd bridge)."""
        if self._ctx is None:
            raise RuntimeError("Executor.backward called without a saved forward")
        s = self.spec
        pts, drop, ws = self._ctx
        if self.grads is None:
            self.alloc_grads()
        if zero:
            self._grad_flat.zero_()
        g = self.grads
        if dyhat is not None:
            ws.dyhat.copy_(dyhat)
        basis = self._basis()
        nh = s.n_hidden
        main = torch.cuda.current_stream()
        if self._side is None:
            self._side = torch.cuda.Stream(device=self.device)
        side = self._side
        head = ops.make_head(s.head_w, s.head_b, s.q, ws.yhat, dyhat=ws.dyhat)
        for l in reversed(range(nh)):
            a = L.BwdArgs()
            a.pts = pts
            if l == 0 and ws.feat is None:
                a.basis = C.pointer(basis)
                if self.sparse:
                    a.addend = ws.zs.data_ptr()
            else:
                a.a_img = (ws.feat if l == 0 else ws.h[l - 1]).data_ptr()
                if self.x3:
                    a.a_img_lo = ws.h_lo[l - 1].data_ptr()
            a.layer = self._layer(l)
            a.drop = drop
            if ws.x is not None:
                a.x_img = ws.x[l].data_ptr()
                # The launch just before a backward is another backward (or, for the head, the last forward), and the
                # dropout step counter advances in the previous step's tail.  Below the head x and stats come from the
                # forward, further back.
                if self.prewait:
                    a.settled = L.SETTLED_STEP | (L.SETTLED_X if l < nh - 1 else 0)
            if ws.stats[l] is not None:
                a.stats = ws.stats[l].data_ptr()
                a.d_gamma = g["gammas"][l].data_ptr()
                a.d_beta = g["betas"][l].data_ptr()
            if l == nh - 1:
                a.head = C.pointer(head)
                a.d_head_w = g["head_w"].data_ptr()
                a.d_head_b = g["head_b"].data_ptr()
            else:
                a.dz_next_img = ws.dz[l + 1].data_ptr()
                a.wt_next_img = self.wt_img[l + 1].data_ptr()
                a.n_next = s.weights[l + 1].shape[0]
                if self.x3:
                    a.dz_next_img_lo = ws.dz_lo[l + 1].data_ptr()
                    a.wt_next_img_lo = self.wt_img_lo[l + 1].data_ptr()
            a.dz_img = ws.dz[l].data_ptr()
            if self.x3:
                a.dz_img_lo = ws.dz_lo[l].data_ptr()
            a.d_bias = g["biases"][l].data_ptr()
            ops.layer_bwd(a)
            if l == 0:
                # block 1's dW is the last kernel of the chain and the step waits for it: it follows layer_bwd on the
                # launching stream, where it starts early and regenerates its basis operand while layer_bwd runs
                self._wgrad_block(l, pts, ws, basis, g)
            else:
                # dW_l only needs dz_l: it runs on a second stream, concurrently with the rest of the backward chain
                # (a 4096-row batch is 32 tiles -- one kernel alone leaves most of the 148 SMs idle)
                side.wait_stream(main)
                with torch.cuda.stream(side):
                    self._wgrad_block(l, pts, ws, basis, g)
        main.wait_stream(side)      # join: every weight gradient is complete before the caller continues
        if s.learnable_basis and not self.sparse:
            a = L.KnotGradArgs()
            a.basis = C.pointer(basis)
            a.pts = pts
            a.dz_img = ws.dz[0].data_ptr()
            a.w1s_img = self.w1s_img.data_ptr()
            if self.x3:
                a.dz_img_lo = ws.dz_lo[0].data_ptr()
                a.w1s_img_lo = self.w1s_img_lo.data_ptr()
            a.n_out = s.weights[0].shape[0]
            a.d_centers = g["centers"].data_ptr()
            a.d_log_bw = g["log_bandwidths"].data_ptr()
            ops.knot_grad(a)
        return g
