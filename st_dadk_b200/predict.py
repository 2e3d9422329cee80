"""Dense-grid / point-set kriging prediction, sharded by point across the GPUs of one box.

Upstream runs T sequential forwards of S points each with a D2H copy per time step (plot_spatial_mse,
scripts/train_st_interp.py:1233-1248) or one forward over T*S points (plot_temporal_series, :1380-1394).  Points
are independent (LayerNorm is per row), so rank r of R owns the contiguous block
[floor(r N / R), floor((r+1) N / R)) and there is no data-path collective; the grid itself is generated on the
device from the linear index, so a grid prediction reads 0 bytes of input per point.
"""
from __future__ import annotations

from typing import Optional, Tuple

import torch

from . import ops
from .executor import Executor


def shard_range(n: int, rank: int, world: int) -> Tuple[int, int]:
    return (rank * n) // world, ((rank + 1) * n) // world


class Predictor:
    """Forward-only executor bound to a model; weight images are packed once and reused across chunks."""
    FUSED_CHUNK = 1 << 26      # rows per launch of the whole-network kernel (67M; tiles are counted in 32 bits)

    def __init__(self, model, chunk_rows: int = 1 << 20, static_weights: bool = False):
        """static_weights=True (serving): the model's parameters do not change between calls, so the knot tables and
        weight images are built on the first call only.  The default rebuilds them on every call, because parameter
        storage can be rewritten in place (optimizer kernel, EMA swap) without any version counter changing."""
        self.model = model
        self.chunk = int(chunk_rows)
        self.static_weights = bool(static_weights)
        self._prepared = False
        self.ex: Optional[Executor] = None
        self.launches = 0
        self._field_key = None
        self._field_pts = None
        self.d2h_chunk_rows = 1 << 18      # field predictions delivered to the host: rows per overlapped D2H piece
        self._copy_stream = None
        self.host_copy_done = None
        self.used_field_kernel = False     # the last grid / field call ran the site-tile x time-loop kernel
        self.use_field_kernel = True       # False: grid / field calls go through the generic per-point kernel

    def _prepare(self):
        if self.static_weights and self._prepared:
            return
        m = self.model
        if not next(m.buffers()).is_cuda:
            raise RuntimeError("Predictor: the model must live on a CUDA device (no CPU path)")
        with torch.no_grad():
            spec = m.net_spec()
        if self.ex is None:
            self.ex = Executor(spec)
        else:
            self.ex.rebind(spec)
        self.ex.prepare(force=True, for_backward=False)
        self.launches += 2 + len(spec.weights)
        self._prepared = True

    @property
    def fused(self) -> bool:
        """True when forward-only calls run the whole-network kernel (stdadk_predict)."""
        return bool(self.ex is not None and self.ex.fused_predict and self.ex._fused_ok)

    @torch.no_grad()
    def _run(self, make_pts, begin: int, end: int, out: torch.Tensor):
        n_layers = self.ex.spec.n_hidden
        # the whole-network kernel keeps nothing in HBM per row, so a shard goes in ONE launch; only the per-block
        # fallback (2 KB of activation images per row) needs bounded chunks
        step = self.FUSED_CHUNK if self.ex.fused_supported() else self.chunk
        for b in range(begin, end, step):
            r = min(step, end - b)
            self.ex.forward(make_pts(b, r), train=False, out=out[b - begin:b - begin + r], prepared=True)
            self.launches += 1 if self.fused else n_layers
        return out

    @torch.no_grad()
    def grid(self, nx: int, ny: int, nt: int, rank: int = 0, world: int = 1, out: Optional[torch.Tensor] = None):
        """This rank's block of the (nt, nx, ny) grid prediction: returns (yhat (n_local, Q), (begin, end))."""
        self._prepare()
        n = nx * ny * nt
        begin, end = shard_range(n, rank, world)
        dev = self.ex.device
        if out is None:
            out = torch.empty(end - begin, self.model.output_dim, device=dev)
        self.used_field_kernel = self.use_field_kernel and self.ex.field_supported()
        if self.used_field_kernel:
            # every site of the nx x ny lattice at nt time steps: basis + block 1 once per tile of sites
            self.launches += self.ex.predict_field(out, begin, end, nx * ny, nt, grid=(nx, ny))
            return out, (begin, end)
        self._run(lambda b, r: ops.make_points(grid=(nx, ny, nt), row_begin=b, n_rows=r), begin, end, out)
        return out, (begin, end)

    @torch.no_grad()
    def grid_by_sites(self, nx: int, ny: int, nt: int, rank: int = 0, world: int = 1, out: Optional[torch.Tensor] = None):
        """The same (nt, nx, ny) grid sharded by SITE: this rank's sites [s0, s1) of the nx*ny lattice at all nt time steps;
        returns (yhat (nt, s1 - s0, Q), (s0, s1)) -- concatenating the ranks' results along dim 1 gives the (nt, nx*ny, Q)
        field.  Every point is computed by exactly one rank and has the value `grid` gives it.  With contiguous point
        blocks (`grid`) a rank of an 8-GPU job owns ~nt/8 time steps of every site and repeats the per-site work of
        the field kernel (basis + spatial part of block 1) that a single GPU does once for all nt steps; by sites the
        work per point is the single-GPU one at every world size."""
        self._prepare()
        S = nx * ny
        s0, s1 = shard_range(S, rank, world)
        q = self.model.output_dim
        if out is None:
            out = torch.empty(nt, s1 - s0, q, device=self.ex.device)
        self.used_field_kernel = self.use_field_kernel and self.ex.field_supported()
        if self.used_field_kernel:
            self.launches += self.ex.predict_field_sites(out, s0, s1, S, nt, grid=(nx, ny))
            return out, (s0, s1)
        for k in range(nt):       # generic kernels: one block of rows per time step
            self._run(lambda b, r: ops.make_points(grid=(nx, ny, nt), row_begin=b, n_rows=r), k * S + s0, k * S + s1, out[k])
        return out, (s0, s1)

    @torch.no_grad()
    def points(self, coords: torch.Tensor, t: torch.Tensor, X: Optional[torch.Tensor] = None, rank: int = 0,
               world: int = 1, out: Optional[torch.Tensor] = None):
        """This rank's block of an explicit point set (coords (N,2), t (N,) or (N,1)) resident on the device."""
        self._prepare()
        n = coords.shape[0]
        begin, end = shard_range(n, rank, world)
        coords, t = coords.float().contiguous(), t.reshape(-1).float().contiguous()
        if out is None:
            out = torch.empty(end - begin, self.model.output_dim, device=coords.device)
        self._run(lambda b, r: ops.make_points(coords, t, X, row_begin=b, n_rows=r), begin, end, out)
        return out, (begin, end)

    @torch.no_grad()
    def space_time_field(self, coords: torch.Tensor, T: int, rank: int = 0, world: int = 1,
                         host_out: Optional[torch.Tensor] = None):
        """All T time steps at S sites (the predictions.npz field of upstream, T x S row-major: point n = (t, s)),
        without materialising repeated coordinates: rows gather site n % S through an index.

        `host_out` (pinned (n_local, Q) float32): the field is produced in a few chunks and each chunk is copied to the
        host on a second stream while the next one is computed; the caller synchronises (`torch.cuda.synchronize()` or
        `Predictor.host_copy_done.synchronize()`) before reading it."""
        self._prepare()
        S = coords.shape[0]
        n = S * T
        begin, end = shard_range(n, rank, world)
        dev = coords.device
        # the (site, time) expansion of this shard depends only on the site set: keep it for repeated field predictions
        # (per-epoch plots, evaluation of several checkpoints) instead of rebuilding four 1M-element tensors per call
        key = (coords.data_ptr(), coords._version, S, T, begin, end)
        if self._field_key != key:
            idx = torch.arange(begin, end, device=dev, dtype=torch.int64)
            site = idx % S
            tt = ((idx // S).float() / float(T - 1)) if T > 1 else torch.zeros(end - begin, device=dev)
            cf = coords.float()
            order = None
            if begin % S == 0 and end % S == 0 and S >= 256:
                # whole time steps: visit the sites of each step in a space-filling order (x strips, y inside a strip)
                # so that the 32 rows of a warp are neighbours and share their support -- the kernel then skips most
                # knot chunks with one vote; y_hat is scattered back to the caller's site order below
                order = torch.argsort(torch.floor(cf[:, 0] * 32.0) * 2.0 + cf[:, 1])
                site = order[site]
            cc = cf.index_select(0, site).contiguous()
            # the S sites in the order the field kernel visits them (space-filling when whole steps are owned)
            self._field_sites = (cf.index_select(0, order) if order is not None else cf).contiguous()
            self._field_key, self._field_pts = key, (cc, tt, order)
        cc, tt, order = self._field_pts
        self.used_field_kernel = self.use_field_kernel and self.ex.field_supported()
        out = torch.empty(end - begin, self.model.output_dim, device=dev)
        q = out.shape[1]
        res = torch.empty_like(out) if order is not None else out
        n_local = end - begin
        if host_out is None:
            pieces = [(0, n_local)]
        else:
            if host_out.shape != out.shape or not host_out.is_pinned():
                raise RuntimeError("space_time_field: host_out must be a pinned float32 tensor of shape (n_local, Q)")
            step = max(1, self.d2h_chunk_rows)
            if order is not None:
                step = max(S, step // S * S)            # whole time steps, so that a chunk can be put in site order
            pieces = [(b, min(step, n_local - b)) for b in range(0, n_local, step)]
            if self._copy_stream is None:
                self._copy_stream = torch.cuda.Stream(device=dev)
                self.host_copy_done = torch.cuda.Event()
        main = torch.cuda.current_stream()
        sites_f = None
        if self.used_field_kernel:
            sites_f = self._field_sites
        for b0, r0 in pieces:
            if self.used_field_kernel:
                self.launches += self.ex.predict_field(out[b0:b0 + r0], begin + b0, begin + b0 + r0, S, T, sites=sites_f)
            else:
                self._run(lambda b, r: ops.make_points(cc, tt, None, row_begin=b - begin, n_rows=r), begin + b0,
                          begin + b0 + r0, out[b0:b0 + r0])
            if order is not None:
                res[b0:b0 + r0].view(-1, S, q).index_copy_(1, order, out[b0:b0 + r0].view(-1, S, q))
            if host_out is not None:
                ready = torch.cuda.Event()
                ready.record(main)
                with torch.cuda.stream(self._copy_stream):
                    self._copy_stream.wait_event(ready)
                    host_out[b0:b0 + r0].copy_(res[b0:b0 + r0], non_blocking=True)
        if host_out is not None:
            self.host_copy_done.record(self._copy_stream)
            res.record_stream(self._copy_stream)
        return res, (begin, end)

    @torch.no_grad()
    def space_time_field_by_sites(self, coords: torch.Tensor, T: int, rank: int = 0, world: int = 1):
        """The (T, S) field sharded by SITE: this rank's sites [s0, s1) (in the caller's order) at all T time steps;
        returns (yhat (T, s1 - s0, Q), (s0, s1)); the ranks' results concatenated along dim 1 are the field.  Same values
        as `space_time_field`; the per-site work of the field kernel is not repeated across ranks (see grid_by_sites)."""
        self._prepare()
        S = coords.shape[0]
        s0, s1 = shard_range(S, rank, world)
        n, q, dev = s1 - s0, self.model.output_dim, coords.device
        key = ("by_sites", coords.data_ptr(), coords._version, S, T, s0, s1)
        if self._field_key != key:
            cf = coords[s0:s1].float()
            # neighbours in a warp share their support (one vote skips a knot chunk): visit the sites in x strips
            order = torch.argsort(torch.floor(cf[:, 0] * 32.0) * 2.0 + cf[:, 1]) if n >= 256 else None
            self._field_sites = (cf.index_select(0, order) if order is not None else cf).contiguous()
            self._field_key, self._field_pts = key, (None, None, order)
        order = self._field_pts[2]
        self.used_field_kernel = self.use_field_kernel and self.ex.field_supported()
        out = torch.empty(T, n, q, device=dev)
        if n == 0:
            return out, (s0, s1)
        if self.used_field_kernel:
            self.launches += self.ex.predict_field_sites(out, 0, n, n, T, sites=self._field_sites)
        else:
            cc = self._field_sites.repeat(T, 1)
            tt = (torch.arange(T, device=dev).repeat_interleave(n).float() / float(T - 1)) if T > 1 else \
                torch.zeros(T * n, device=dev)
            self._run(lambda b, r: ops.make_points(cc, tt, None, row_begin=b, n_rows=r), 0, T * n, out.view(T * n, q))
        if order is None:
            return out, (s0, s1)
        res = torch.empty_like(out)
        res.index_copy_(1, order, out)
        return res, (s0, s1)

    @torch.no_grad()
    def profile_layers(self, nx: int, ny: int, nt: int, repeats: int = 3):
        """Per-block kernel time of a grid prediction (CUDA events around each launch on the launching stream) with
        the algorithmic HBM bytes per launch: block 1 reads nothing per point (grid generated on device) and writes
        the h1 image; later blocks read and write images; the last writes y_hat."""
        from . import ops as _ops
        self._prepare()
        n = min(nx * ny * nt, self.chunk)
        rec = []
        orig = _ops.layer_fwd
        fused, self.ex.fused_predict = self.ex.fused_predict, False     # profile the layer-by-layer kernels

        def timed(a):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            orig(a)
            e1.record()
            rec.append((a.layer.layer_id, a.layer.n_in, a.layer.n_out, bool(a.head), e0, e1))

        out = torch.empty(n, self.model.output_dim, device=self.ex.device)
        _ops.layer_fwd = timed
        try:
            for _ in range(repeats + 1):
                self.ex.forward(_ops.make_points(grid=(nx, ny, nt), row_begin=0, n_rows=n), train=False, out=out,
                                prepared=True)
            torch.cuda.synchronize()
        finally:
            _ops.layer_fwd = orig
            self.ex.fused_predict = fused
        res = {}
        nl = self.ex.spec.n_hidden
        for lid, n_in, n_out, has_head, e0, e1 in rec[nl:]:          # first pass = warm-up
            d = res.setdefault(lid, {"ms": 0.0, "n": 0})
            d["ms"] += e0.elapsed_time(e1)
            d["n"] += 1
            pad = lambda c: (c + 31) // 32 * 32
            rd = 0 if lid == 0 else 4 * pad(n_in)
            wr = 4 * self.model.output_dim if has_head else 4 * pad(n_out)
            d["bytes"] = float(n) * (rd + wr)
            d["flops"] = 2.0 * n * n_in * n_out
        for d in res.values():
            d["ms"] /= d["n"]
        return n, res

    @torch.no_grad()
    def profile_block1(self, coords: torch.Tensor, t: torch.Tensor, repeats: int = 5) -> dict:
        """The fused basis + Linear1 + LayerNorm/ReLU forward kernel (layer_fwd, block 1) alone on explicit points:
        median launch time (a CUDA event pair per launch on the launching stream) and its algorithmic HBM bytes, 12 B read (x, y, t) +
        4 * pad32(n_out) B written per row."""
        import ctypes as C
        from . import _lib as L
        self._prepare()
        ex, s = self.ex, self.ex.spec
        n = coords.shape[0]
        ws = ex._workspace(n)
        basis = ex._basis()
        a = L.FwdArgs()
        a.pts = ops.make_points(coords, t)
        a.basis = C.pointer(basis)
        a.layer = ex._layer(0)
        a.drop = L.Dropout(0.0, 0, 0, None, 0)
        a.out_img = ws.h[0].data_ptr()
        if ex.x3:
            a.out_img_lo = ws.h_lo[0].data_ptr()
        ops.layer_fwd(a)
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(repeats)]
        for e0, e1 in ev:
            e0.record()
            ops.layer_fwd(a)
            e1.record()
        torch.cuda.synchronize()
        times = sorted(e0.elapsed_time(e1) for e0, e1 in ev)       # median: one disturbed launch must not move the figure
        per_row = 12 + 4 * ops.pad32(s.weights[0].shape[0]) * (2 if ex.x3 else 1)
        return {"ms": times[len(times) // 2], "ms_all": times, "rows": n, "bytes_per_row": per_row, "bytes": float(n) * per_row,
                "flops": 2.0 * n * s.weights[0].shape[0] * s.weights[0].shape[1]}

    @torch.no_grad()
    def profile_fused(self, nx: int, ny: int, nt: int, repeats: int = 5):
        """Average duration of the whole-network kernel over a grid prediction of min(nx*ny*nt, chunk) points, with
        its algorithmic work: 4Q bytes written per point (nothing read for a generated grid) and the dense FLOPs of
        every block and the head.  Returns (points, {"ms", "bytes", "flops"}) or (points, None) if the fused kernel
        does not take this shape."""
        from . import ops as _ops
        self._prepare()
        n = min(nx * ny * nt, self.chunk)
        out = torch.empty(n, self.model.output_dim, device=self.ex.device)
        pts = _ops.make_points(grid=(nx, ny, nt), row_begin=0, n_rows=n)
        self.ex.forward(pts, train=False, out=out, prepared=True)
        if not self.fused:
            return n, None
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(repeats):
            self.ex.forward(pts, train=False, out=out, prepared=True)
        e1.record()
        torch.cuda.synchronize()
        s = self.ex.spec
        flops = sum(2.0 * w.shape[0] * w.shape[1] for w in s.weights) + 2.0 * s.head_w.shape[0] * s.head_w.shape[1]
        return n, {"ms": e0.elapsed_time(e1) / repeats, "bytes": 4.0 * n * self.model.output_dim, "flops": flops * n,
                   "dense_flops": flops * n, "points": n, "kernel": "predict_fused_kernel"}

    @torch.no_grad()
    def profile_field(self, nx: int, ny: int, nt: int, repeats: int = 3):
        """Median duration of a full (nx, ny, nt) grid prediction through the space-time field kernel with the work it
        EXECUTES (block 1 once per site: 2*k_s*n_1 per site; blocks 2.. and the head per point) next to the dense-equivalent
        FLOPs of the per-point network.  None when the field kernel does not take this network."""
        self._prepare()
        if not (self.use_field_kernel and self.ex.field_supported()):
            return None
        n = nx * ny * nt
        out = torch.empty(n, self.model.output_dim, device=self.ex.device)
        self.grid(nx, ny, nt, out=out)
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(repeats)]
        for e0, e1 in ev:
            e0.record()
            self.grid(nx, ny, nt, out=out)
            e1.record()
        torch.cuda.synchronize()
        ms = sorted(e0.elapsed_time(e1) for e0, e1 in ev)[repeats // 2]       # median of the repetitions
        s = self.ex.spec
        k_s = s.centers.shape[0]
        per_site = 2.0 * k_s * s.weights[0].shape[0]
        per_point = sum(2.0 * w.shape[0] * w.shape[1] for w in s.weights[1:]) + 2.0 * s.head_w.shape[0] * s.head_w.shape[1]
        dense = sum(2.0 * w.shape[0] * w.shape[1] for w in s.weights) + 2.0 * s.head_w.shape[0] * s.head_w.shape[1]
        return {"ms": ms, "bytes": 4.0 * n * self.model.output_dim,
                "flops": per_site * nx * ny + per_point * n, "dense_flops": dense * n, "points": n,
                "kernel": "predict_field_kernel"}
