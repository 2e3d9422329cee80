"""Training / evaluation engine for STInterpMLP on libstdadk.

Replaces the upstream Python loop `train_model` / `evaluate_model` (scripts/train_st_interp.py:463-961):

  * samples live in HBM as a struct-of-arrays `ObservationTable`; a mini-batch is a slice of a device-resident
    permutation that the kernels gather through (no per-sample dict, no collate, no per-step H2D);
  * all trainable parameters, gradients, Adam moments and the EMA shadow live in five flat FP32 buffers; the
    model's nn.Parameters are views into the first, so `state_dict()` / checkpoints keep the upstream keys;
  * one step = forward chain (basis fused into block 1, loss fused into the head) -> backward chain -> [one NCCL
    all-reduce of the flat gradient] -> grad-norm -> fused clip + AdamW + EMA, optionally replayed as a CUDA graph;
  * learning-rate logic (warm-up written after the step, progressive unfreezing, chainable cosine) is the
    upstream host code driving real torch schedulers, so the bug-compatible lr trajectory of SURVEY.md 9.5 holds.
"""
from __future__ import annotations

import gc
import math
import os
import warnings
from dataclasses import dataclass
from typing import Dict, List, Optional

import numpy as np
import torch
import torch.distributed as dist

import threading

from . import _lib as L
from . import ops
from .executor import Executor, LossSpec, NetSpec


def _dist_on() -> bool:
    return dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1


# ------------------------------------------------------------------------------------------------
_CAPTURE_LOCK = threading.Lock()


class FlatState:
    """Flat parameter / gradient / moment / EMA buffers with the model's Parameters re-pointed into them.

    Layout: group 0 ("mlp"): per hidden block W^T (in, out)-contiguous, bias, [gamma, beta]; then the head
    (W (Q, d), b) or the delta vectors; group 1 ("basis", learnable only): centres (K, 2), log-bandwidths (K).
    Linear weights are stored transposed (knot-major for block 1) so that the wgrad kernel's accumulation
    is coalesced; the Parameter seen by PyTorch is the `.t()` view with the upstream (out, in) shape.
    """

    def __init__(self, model, device):
        self.model = model
        blocks = model.hidden_blocks()
        entries = []   # (param, stored_shape, transposed)
        for lin, ln in blocks:
            entries.append((lin.weight, (lin.in_features, lin.out_features), True))
            entries.append((lin.bias, tuple(lin.bias.shape), False))
            if ln is not None:
                entries.append((ln.weight, tuple(ln.weight.shape), False))
                entries.append((ln.bias, tuple(ln.bias.shape), False))
        if model.delta_params is not None:
            for d in model.delta_params:
                entries.append((d, tuple(d.shape), False))
        else:
            head = model.mlp[-1]
            entries.append((head.weight, tuple(head.weight.shape), False))
            entries.append((head.bias, tuple(head.bias.shape), False))
        n_mlp = sum(int(np.prod(s)) for _, s, _ in entries)
        sb = model.spatial_basis
        if sb.learnable:
            entries.append((sb.centers, tuple(sb.centers.shape), False))
            entries.append((sb.log_bandwidths, tuple(sb.log_bandwidths.shape), False))
        n = sum(int(np.prod(s)) for _, s, _ in entries)
        self.n = n
        self.group_end = [n_mlp, n] if sb.learnable else [n]
        q, d = model.output_dim, model.last_hidden_dim
        self.n_scratch = q * d + q if model.delta_params is not None else 0
        mk = lambda extra=0: torch.zeros(n + extra, dtype=torch.float32, device=device)
        # g carries, behind the parameter gradients, the scratch head gradient of the delta parameterisation and ONE
        # more float: the step's loss accumulator, so that a data-parallel step needs a single exchange (the buffer is
        # padded to a multiple of four floats: the peer-memory exchange moves 16-byte packets)
        self.p, self.m, self.v, self.shadow = mk(), mk(), mk(), mk()
        self.n_exchange = n + self.n_scratch + 1
        self.g = mk(self.n_scratch + 1 + (-self.n_exchange) % 4)
        self.loss_slot = self.g[n + self.n_scratch:n + self.n_scratch + 1]
        self.views: Dict[int, torch.Tensor] = {}
        self.gviews: Dict[int, torch.Tensor] = {}
        o = 0
        with torch.no_grad():
            for prm, shape, tr in entries:
                k = int(np.prod(shape))
                pv, gv = self.p[o:o + k].view(*shape), self.g[o:o + k].view(*shape)
                if tr:
                    pv, gv = pv.t(), gv.t()
                pv.copy_(prm.detach().to(device))
                prm.data = pv
                prm.grad = None
                self.views[id(prm)] = pv
                self.gviews[id(prm)] = gv
                o += k
        self.shadow.copy_(self.p)           # ModelEMA starts from the current weights (ema.py:48-50)
        self._backup = None
        # scratch gradient of the effective head for the delta parameterisation (st_interp.py:859-873)
        if self.n_scratch:
            self.g_head_w = self.g[n:n + q * d].view(q, d)
            self.g_head_b = self.g[n + q * d:n + q * d + q]

    def grad_views_for(self, model) -> dict:
        blocks = model.hidden_blocks()
        gv = self.gviews
        out = {"weights": [gv[id(l.weight)] for l, _ in blocks], "biases": [gv[id(l.bias)] for l, _ in blocks],
               "gammas": [gv[id(n.weight)] if n is not None else None for _, n in blocks],
               "betas": [gv[id(n.bias)] if n is not None else None for _, n in blocks]}
        if model.delta_params is not None:
            out["head_w"], out["head_b"] = self.g_head_w, self.g_head_b
        else:
            out["head_w"], out["head_b"] = gv[id(model.mlp[-1].weight)], gv[id(model.mlp[-1].bias)]
        sb = model.spatial_basis
        if sb.learnable:
            out["centers"], out["log_bandwidths"] = gv[id(sb.centers)], gv[id(sb.log_bandwidths)]
        else:
            out["centers"] = out["log_bandwidths"] = None
        return out

    # EMA weight exchange (ema.py:68-89), by value so the Parameter views stay valid
    def apply_shadow(self):
        self._backup = self.p.clone()
        self.p.copy_(self.shadow)

    def restore(self):
        self.p.copy_(self._backup)
        self._backup = None


# ------------------------------------------------------------------------------------------------
@dataclass
class StepStats:
    loss: float
    n_rows: int


class Trainer:
    """One model, one device, optional data-parallel group (torch.distributed, NCCL)."""

    def __init__(self, model, config: dict, device, batches_per_epoch: int = 1, use_cuda_graph: bool = False):
        self.model = model.to(device)
        self.cfg = config
        if config.get("precision") is not None:
            self.model.precision = config["precision"]
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("st_dadk_b200.Trainer runs on CUDA (sm_100) only; there is no CPU training path")
        self.flat = FlatState(self.model, self.device)
        # Data parallel over the GPUs of one box: the per-step gradient exchange is ONE kernel over NVLink peer memory
        # (st_dadk_b200/peer.py: low-latency packets, rank-ordered in-place sum, fused gradient norm), captured inside
        # the step's single CUDA graph.  NCCL's all-reduce between two graphs remains for gradients too large for the
        # receive areas (the 100k-knot model: bandwidth-bound, NCCL's home ground), for non-NCCL groups, when symmetric
        # memory cannot be set up, or on request (STDADK_PEER_ALLREDUCE=0).
        self._peer = None
        if _dist_on() and dist.get_backend() == "nccl" and os.environ.get("STDADK_PEER_ALLREDUCE", "1") != "0":
            ok = torch.ones(1, device=self.device)
            try:
                from .peer import PeerExchange
                self._peer = PeerExchange(self.device, self.flat.n_exchange)
            except Exception as e:       # noqa: BLE001 -- any set-up failure falls back to NCCL, loudly
                if "exceeds the peer-exchange limit" not in str(e):
                    warnings.warn(f"peer-memory gradient exchange unavailable ({e!r}); using the NCCL all-reduce")
                ok.zero_()
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)       # all ranks must agree on the exchange path
            if float(ok.item()) == 0.0:
                self._peer = None
        m = self.model
        self.learnable = bool(m.spatial_basis.learnable)
        self.q = m.output_dim
        # Effective head the kernels read.  The Linear head is read straight from its parameters, which live (Q, d)
        # row-major in the flat buffer and are only ever rewritten in place (AdamW, the EMA swap).  The delta
        # parameterisation has static buffers that _refresh_head recomputes each step.
        if m.delta_params is not None:
            self.head_w = torch.empty(self.q, m.last_hidden_dim, device=self.device)
            self.head_b = torch.empty(self.q, device=self.device)
        else:
            self.head_w, self.head_b = m.mlp[-1].weight.detach(), m.mlp[-1].bias.detach()
        self.ex = Executor(self._spec())
        self.ex.loss_acc = self.flat.loss_slot      # the loss accumulator travels with the gradient all-reduce
        # Captured graphs hold raw pointers into the executor's workspaces: drop them when one is evicted.  The callback
        # holds the graph dictionary, not the trainer: a trainer in a reference cycle with its executor is only freed
        # when the cyclic garbage collector runs, and freeing its graphs then, inside another capture on this thread
        # (a global-mode capture: any thread), invalidates that capture.
        self._graphs: Dict[tuple, torch.cuda.CUDAGraph] = {}
        self.ex.on_evict = self._graphs.clear
        self.ex.alloc_grads(self.flat.g, self.flat.grad_views_for(m))
        self._init_loss()
        self._init_optimizer(batches_per_epoch)
        self.step_count = torch.zeros(1, dtype=torch.int32, device=self.device)   # AdamW step == dropout stream
        self.sqnorms = torch.zeros(len(self.flat.group_end), device=self.device)
        # own reduction workspace (partials + ticket): trainers of different configurations run concurrently on
        # separate streams of one GPU and must not share it
        self._sqnorm_ws = torch.zeros(L.lib().stdadk_sqnorm_ws_floats(), device=self.device)
        self._tail_ws = torch.zeros(148 * 8 + 8, device=self.device)      # fused step tail: norm partials + grid barrier
        self.seed = int(torch.initial_seed() & (2 ** 63 - 1))
        self.loss_sum = torch.zeros(1, device=self.device)      # running sum of per-step losses (one sync / epoch)
        self.loss_last = torch.zeros(1, device=self.device)     # loss of the most recent step (written by AdamW)
        self._g_clean = False     # True while the flat gradient and loss_acc are known to be zero (left so by AdamW)
        self.use_cuda_graph = use_cuda_graph
        self._stage_idx = None
        self._host_stage = None
        self._host_perm = None
        self.world = dist.get_world_size() if _dist_on() else 1
        self.rank = dist.get_rank() if _dist_on() else 0
        c = self.cfg
        self._param_terms_possible = bool(
            self.learnable
            or (c.get("sparsity_penalty_type", "none") != "none"
                and (float(c.get("sparsity_lambda_l1", 0.001)) != 0.0 or float(c.get("sparsity_lambda_group", 0.01)) != 0.0))
            or (c.get("use_delta_reparameterization", False) and float(c.get("non_crossing_lambda", 0.0)) > 0))
        self.kernel_launches = 0

    # ------------------------------------------------------------------ configuration
    def _spec(self) -> NetSpec:
        m = self.model
        self._refresh_head()
        return m.net_spec(self.head_w, self.head_b)

    def _refresh_head(self):
        m = self.model
        if m.delta_params is not None:
            with torch.no_grad():
                beta = torch.cumsum(torch.stack([d.detach() for d in m.delta_params]), dim=0)
                self.head_w.copy_(beta[:, 1:])
                self.head_b.copy_(beta[:, 0])

    def _init_loss(self):
        c = self.cfg
        rt = c.get("regression_type", "mean")
        if rt == "mean":
            self.loss = LossSpec("mse")
        elif rt == "quantile":
            if c.get("current_quantile") is None:
                raise ValueError("current_quantile must be specified for quantile regression")
            self.loss = LossSpec("pinball", [float(c["current_quantile"])])
        elif rt == "multi-quantile":
            taus = [float(x) for x in c.get("quantile_levels", [0.1, 0.5, 0.9])]
            ncw = 0.0 if c.get("use_delta_reparameterization", False) else float(c.get("non_crossing_weight", 0.0))
            self.loss = LossSpec("pinball", taus, ncw, int(c.get("non_crossing_power", 1)))
        else:
            raise ValueError(f"Unknown regression_type: {rt}")

    def _init_optimizer(self, batches_per_epoch: int):
        """Param groups, schedulers and EMA decay exactly as train_st_interp.py:466-541; the torch optimizer
        object only carries the lr state for the schedulers -- the update itself is the fused kernel."""
        c = self.cfg
        self.lr = float(c.get("lr", 1e-3))
        self.wd = float(c.get("weight_decay", 1e-5))
        self.clip = float(c.get("grad_clip", 0) or 0)
        self.unfreeze_epoch = int(c.get("basis_unfreeze_epoch", 0))
        self.rampup_epochs = int(c.get("basis_lr_rampup_epochs", 0))
        dummy = lambda: [torch.nn.Parameter(torch.zeros(1))]
        if self.learnable:
            ratio = c.get("basis_lr_ratio", 0.05)
            init_basis = 0.0 if self.unfreeze_epoch > 0 else self.lr * ratio
            self.opt = torch.optim.AdamW([{"params": dummy(), "lr": self.lr, "name": "mlp"},
                                          {"params": dummy(), "lr": init_basis, "name": "basis"}], weight_decay=self.wd)
            for gq in self.opt.param_groups:
                gq["initial_lr"] = gq["lr"]
                if gq.get("name") == "basis":
                    gq["target_lr"] = self.lr * ratio
        else:
            self.opt = torch.optim.AdamW(dummy(), lr=self.lr, weight_decay=self.wd)
            for gq in self.opt.param_groups:
                gq["initial_lr"] = gq["lr"]
        self.batches_per_epoch = max(1, batches_per_epoch)
        self.warmup_epochs = int(c.get("warmup_epochs", 0))
        self.warmup_steps = self.warmup_epochs * self.batches_per_epoch if self.warmup_epochs > 0 else 0
        self.scheduler = None
        if c.get("scheduler") == "cosine":
            self.scheduler = torch.optim.lr_scheduler.CosineAnnealingLR(self.opt, T_max=c.get("epochs", 100),
                                                                        eta_min=self.lr * 0.5)
        self.ema_decay = 1.0 - 1.0 / (10.0 * self.batches_per_epoch)
        self.global_step = 0
        ng = len(self.opt.param_groups)
        # Per-step hyper-parameters travel host -> device through a RING of pinned slots, each guarded by an event:
        # the host runs many steps ahead of the GPU (graph replay, no per-step sync), so a single pinned buffer would
        # be overwritten while the copy of an earlier step is still pending and that step would then use a later lr.
        self._hyper_ring = [torch.zeros(ng, 4, dtype=torch.float32).pin_memory() for _ in range(self.HYPER_SLOTS)]
        self._hyper_ev = [None] * self.HYPER_SLOTS
        self._hyper_k = 0
        self._hyper_last = None
        self.hyper = torch.zeros(ng, 4, dtype=torch.float32, device=self.device)

    HYPER_SLOTS = 16

    def _hyper_values(self):
        rows = []
        for gq in self.opt.param_groups:
            clip = self.clip * (0.1 if (self.learnable and gq.get("name") == "basis") else 1.0)
            rows.append((float(gq["lr"]), float(self.wd), float(clip)))
        return tuple(rows)

    def _push_hyper(self):
        vals = self._hyper_values()
        if vals == self._hyper_last:           # unchanged since the last step (after warm-up: once per epoch)
            return
        k = self._hyper_k
        self._hyper_k = (k + 1) % self.HYPER_SLOTS
        if self._hyper_ev[k] is not None:
            self._hyper_ev[k].synchronize()    # the copy that last read this slot has completed
        slot = self._hyper_ring[k]
        for i, (lr, wd, clip) in enumerate(vals):
            slot[i, 0], slot[i, 1], slot[i, 2] = lr, wd, clip
        self.hyper.copy_(slot, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream())
        self._hyper_ev[k] = ev
        self._hyper_last = vals

    def begin_epoch(self, epoch: int):
        """Progressive unfreezing of the basis group (train_st_interp.py:582-602)."""
        if not (self.learnable and self.unfreeze_epoch > 0):
            return
        for gq in self.opt.param_groups:
            if gq.get("name") != "basis":
                continue
            if epoch == self.unfreeze_epoch:
                gq["lr"] = gq["target_lr"] * (0.1 if self.rampup_epochs > 0 else 1.0)
            elif self.unfreeze_epoch < epoch < self.unfreeze_epoch + self.rampup_epochs:
                gq["lr"] = gq["target_lr"] * (0.1 + 0.9 * (epoch - self.unfreeze_epoch) / self.rampup_epochs)

    def end_epoch(self, epoch: int):
        """Cosine scheduler advances only after warm-up (train_st_interp.py:820-823)."""
        if self.scheduler is not None and epoch >= self.warmup_epochs:
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                self.scheduler.step()

    # ------------------------------------------------------------------ parameter-only terms (host-side torch)
    def _penalty_terms(self):
        """Domain / movement / sparsity / P_nc(delta) regularisers (train_st_interp.py:636-691).  They depend on
        parameters only, are O(K) or O(K*H), and are skipped when their weight is zero."""
        c, m = self.cfg, self.model
        terms = []
        if self.learnable:
            w = float(c.get("domain_penalty_weight", 0.0))
            if w > 0:
                terms.append(w * m.compute_domain_penalty())
            w = float(c.get("movement_penalty_weight", 0.0))
            if w > 0:
                terms.append(w * m.compute_movement_penalty())
        stype = c.get("sparsity_penalty_type", "none")
        l1, lg = float(c.get("sparsity_lambda_l1", 0.001)), float(c.get("sparsity_lambda_group", 0.01))
        if stype != "none" and (l1 != 0.0 or lg != 0.0):
            pen = m.compute_sparsity_penalty(penalty_type=stype, lambda_l1=l1, lambda_group=lg)
            if c.get("sparsity_apply_to_spatial", True):
                terms.append(pen["spatial_penalty"])
            if c.get("sparsity_apply_to_temporal", True):
                terms.append(pen["temporal_penalty"])
        if c.get("regression_type") == "multi-quantile" and c.get("use_delta_reparameterization", False):
            lam = float(c.get("non_crossing_lambda", 0.0))
            if lam > 0 and m.delta_params is not None and len(m.delta_params) > 1:
                pnc = 0.0
                for d in list(m.delta_params)[1:]:       # J(delta_k) = d0 - max(d0, sum_j max(0, -d_j)), Eq. 3.10
                    pnc = pnc + d[0] - torch.max(d[0], torch.clamp(-d[1:], min=0.0).sum())
                terms.append(lam * pnc)
        return terms

    def _add_penalty_grads(self):
        terms = self._penalty_terms()
        if not terms:
            return None
        total = sum(terms)
        params = [p for p in self.model.parameters() if p.requires_grad]
        # Tensor hooks also fire inside torch.autograd.grad: the damping hook on `centers` is switched off here so the
        # penalty gradient arrives undamped and _damp_center_grads() damps the SUMMED gradient once, as upstream's
        # loss.backward() does (st_interp.py:111-142, train_st_interp.py:661-693).
        sb = self.model.spatial_basis
        sb._hook_enabled = False
        try:
            grads = torch.autograd.grad(total, params, allow_unused=True)
        finally:
            sb._hook_enabled = True
        for p, gr in zip(params, grads):
            if gr is not None:
                self.flat.gviews[id(p)].add_(gr)
        return total.detach()

    def _finish_special_grads(self):
        m = self.model
        if m.delta_params is not None:   # d delta_l = sum_{k>=l} d beta_k
            dbeta = torch.cat([self.flat.g_head_b[:, None], self.flat.g_head_w], dim=1)
            ddelta = torch.flip(torch.cumsum(torch.flip(dbeta, [0]), dim=0), [0])
            for k, d in enumerate(m.delta_params):
                self.flat.gviews[id(d)].copy_(ddelta[k])

    def _damp_center_grads(self):
        sb = self.model.spatial_basis
        if self.learnable and sb.gradient_damping:
            gv = self.flat.gviews[id(sb.centers)]
            gv.copy_(sb._damping_factor() * gv)

    # ------------------------------------------------------------------ one optimisation step
    def _step_compute(self, table, perm, row_begin: int, n_rows: int, global_rows: int, key_offset: int = 0):
        """Local part of a step: forward (fused loss) and backward into the flat gradient."""
        ex, fl = self.ex, self.flat
        if not self._g_clean:          # steady state: the previous step's AdamW kernel left g and loss_acc zeroed
            fl.g.zero_()
            ex.loss_acc.zero_()
        self._g_clean = False
        self._refresh_head()
        ex.prepare(force=True, for_backward=True)
        pts = ops.make_points(table.coords, table.t, table.X, index=perm, row_begin=row_begin, n_rows=n_rows)
        ex.forward(pts, train=True, seed=self.seed, y=table.y, loss=self.loss, inv_count=1.0 / (global_rows * self.q),
                   save=True, prepared=True, step_ptr=self.step_count, key_offset=key_offset)
        ex.backward(zero=False)
        self._finish_special_grads()

    def _step_exchange(self):
        """The one data-parallel exchange of a step: sum of the flat gradient (and of the loss) over ranks."""
        if self.world > 1:
            if self._peer is not None:                               # one kernel over NVLink peer memory (+ the norm)
                fuse = self._norm_fused()
                self._peer.allreduce(self.flat.g, self.step_count, self.flat.group_end if fuse else None, self.sqnorms)
            else:
                dist.all_reduce(self.flat.g[:self.flat.n_exchange])  # gradients + loss accumulator in one call

    def _norm_fused(self) -> bool:
        """The exchange kernel also produces the clip norm when nothing is added to the gradient between the exchange
        and the clip (parameter-only penalties, knot-gradient damping)."""
        return self._peer is not None and self.world > 1 and self.clip > 0 and not self._param_terms_possible

    def _step_update(self):
        """Replicated tail: parameter-only penalties, damping, gradient norm, fused clip + AdamW + EMA."""
        ex, fl = self.ex, self.flat
        pen = self._add_penalty_grads()
        self._damp_center_grads()
        # Step tail.  The exchange kernel of a data-parallel step may already have produced the clip norm; otherwise the
        # update kernel forms it itself (one launch for {norm, step counter, clip + AdamW + EMA}).
        fused_tail = not self._norm_fused()
        scratch_tail = fl.n_scratch > 0          # scratch gradients behind the parameters are not seen by the kernel
        ops.adamw_ema_step(fl.p, fl.g[:fl.n], fl.m, fl.v, fl.shadow, fl.group_end, self.hyper,
                           self.sqnorms if self.clip > 0 else None, self.step_count, ema_decay=self.ema_decay,
                           zero_grad=True, loss_acc=ex.loss_acc, loss_sum=self.loss_sum, loss_last=self.loss_last,
                           norm_ws=self._tail_ws if fused_tail else None, state_early=fused_tail and ex.prewait)
        if scratch_tail:
            fl.g[fl.n:fl.n + fl.n_scratch].zero_()
        self._g_clean = True
        if pen is not None:
            self.loss_sum += pen

    def _step_body(self, table, perm, row_begin: int, n_rows: int, global_rows: int, key_offset: int = 0):
        self._step_compute(table, perm, row_begin, n_rows, global_rows, key_offset)
        self._step_exchange()
        self._step_update()

    def train_step(self, table, perm: torch.Tensor, row_begin: int, n_rows: int, global_rows: Optional[int] = None,
                   key_offset: Optional[int] = None):
        """One step on samples perm[row_begin : row_begin + n_rows] of `table` (this rank's shard of a global batch
        of `global_rows` samples).  Warm-up is written after the step, as upstream (train_st_interp.py:714-718)."""
        if global_rows is None:
            global_rows = n_rows
        if key_offset is None:      # position of this rank's shard inside the global batch (dropout key)
            key_offset = shard_rows(global_rows, self.rank, self.world)[0] if self.world > 1 else 0
        self._push_hyper()
        if self.use_cuda_graph:
            # Kernel arguments (including the gather window) are frozen in a graph, so a replayed step reads its
            # sample ids from a fixed staging buffer that is refreshed with this step's slice of the permutation.
            if self._stage_idx is None or self._stage_idx.shape[0] < n_rows:
                self._stage_idx = torch.zeros(max(n_rows, 1), dtype=torch.int64, device=self.device)
                self._graphs.clear()
            self._stage_idx[:n_rows].copy_(perm[row_begin:row_begin + n_rows])
            gkey = (n_rows, global_rows, table.coords.data_ptr(), table.t.data_ptr(), table.y.data_ptr(),
                    table.X.data_ptr() if table.X is not None else 0, key_offset)
            g = self._graphs.get(gkey)
            if g is None:
                # first use of this shape: run it eagerly once (sets kernel attributes, sizes workspaces) -- that run
                # IS this step; the captures below record the same launch sequence for later steps without executing.
                # Single GPU: one graph for the whole step.  Data parallel: two graphs with the NCCL all-reduce
                # issued between them on the same stream (the collective stays outside stream capture).
                # Captures are serialised across the threads of a process (several configurations train concurrently on
                # separate streams of one GPU, scripts/run_grid_search.py) and use thread-local capture mode, so what
                # the other threads enqueue meanwhile neither enters nor invalidates this capture.
                # The cyclic garbage collector stays off while this thread captures.  Graphs held by any object in a
                # reference cycle are freed whenever the collector happens to run; freeing a graph is not permitted
                # while the same thread captures, and it invalidates the capture.
                with _CAPTURE_LOCK:
                    self._step_body(table, self._stage_idx, 0, n_rows, global_rows, key_offset)
                    torch.cuda.current_stream().synchronize()
                    mode = dict(capture_error_mode="thread_local")
                    # Data parallel: the peer-memory exchange is a plain kernel and is captured with the rest of the
                    # step; an NCCL all-reduce stays between two graphs (the collective outside stream capture).
                    one_graph = self.world == 1 or self._peer is not None
                    gc_on = gc.isenabled()          # read under the lock: no other capture has switched it off
                    gc.disable()
                    try:
                        if one_graph:
                            g1 = torch.cuda.CUDAGraph()
                            with torch.cuda.graph(g1, **mode):
                                self._step_body(table, self._stage_idx, 0, n_rows, global_rows, key_offset)
                            g = (g1, None)
                        else:
                            g1, g2 = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
                            with torch.cuda.graph(g1, **mode):
                                self._step_compute(table, self._stage_idx, 0, n_rows, global_rows, key_offset)
                            with torch.cuda.graph(g2, **mode):
                                self._step_update()
                            g = (g1, g2)
                    finally:
                        if gc_on:
                            gc.enable()
                self._graphs[gkey] = g
            else:
                g[0].replay()
                if g[1] is not None:
                    self._step_exchange()
                    g[1].replay()
        else:
            self._step_body(table, perm, row_begin, n_rows, global_rows, key_offset)
        if self.global_step < self.warmup_steps:
            f = (self.global_step + 1) / self.warmup_steps
            for gq in self.opt.param_groups:
                gq["lr"] = gq["initial_lr"] * f
        self.global_step += 1

    def train_step_host(self, host_table, row_begin: int, n_rows: int, global_rows: Optional[int] = None,
                        lagged: bool = False) -> float:
        """End-to-end step from HOST buffers: the batch host_table[row_begin : row_begin + n_rows] (pinned memory) is
        copied to a device staging table, the step runs, and the step's loss is read back (the shape of upstream's
        loop body: .to(device) per batch and loss.item(), train_st_interp.py:609-612, :721).

        Staging is double-buffered and the H2D copies go through their own stream.  `lagged=False` returns THIS step's
        loss (one host synchronisation per step, like upstream's loss.item()).  `lagged=True` returns the loss of the
        PREVIOUS step (NaN on the first call; `flush_host_loss()` returns the last one): the host then runs one step
        ahead, so the next batch's copy and launch overlap the running step -- every step's inputs are still copied
        and every step's loss still read back."""
        if self._host_stage is None or len(self._host_stage[0]) < n_rows:
            from stnf.dataio import ObservationTable
            z = lambda *sh: torch.zeros(*sh, dtype=torch.float32, device=self.device)
            mk = lambda: ObservationTable(z(n_rows, 2), z(n_rows), z(n_rows),
                                          z(n_rows, self.model.p) if self.model.p > 0 else None)
            self._host_stage = [mk(), mk()]
            self._graphs.clear()               # graphs captured on the previous staging tables point at freed memory
            self._host_perm = torch.arange(n_rows, dtype=torch.int64, device=self.device)
            self._host_copy_stream = torch.cuda.Stream(device=self.device)
            self._host_ready = [torch.cuda.Event(), torch.cuda.Event()]     # staging buffer k filled
            self._host_done = [torch.cuda.Event(), torch.cuda.Event()]      # step that read buffer k finished
            self._host_loss = [torch.full((1,), float("nan")).pin_memory(), torch.full((1,), float("nan")).pin_memory()]
            self._host_k = 0
            self._host_pending = None
            main = torch.cuda.current_stream()
            for e in self._host_done:
                e.record(main)
        k = self._host_k
        self._host_k ^= 1
        st = self._host_stage[k]
        sl = slice(row_begin, row_begin + n_rows)
        main = torch.cuda.current_stream()

        def copy_batch():
            st.coords[:n_rows].copy_(host_table.coords[sl], non_blocking=True)
            st.t[:n_rows].copy_(host_table.t[sl], non_blocking=True)
            st.y[:n_rows].copy_(host_table.y[sl], non_blocking=True)
            if st.X is not None:
                st.X[:n_rows].copy_(host_table.X[sl], non_blocking=True)

        if lagged or self._host_pending is not None:
            with torch.cuda.stream(self._host_copy_stream):
                self._host_copy_stream.wait_event(self._host_done[k])   # the step two calls ago has released buffer k
                copy_batch()
                self._host_ready[k].record(self._host_copy_stream)
            main.wait_event(self._host_ready[k])
        else:
            # one synchronisation per step: nothing can overlap, so the copies go on the launching stream itself (no
            # stream switch, no event pair: ~15 us of host time per step that would sit on the critical path)
            copy_batch()
        self.train_step(st, self._host_perm, 0, n_rows, global_rows)
        self._host_loss[k].copy_(self.loss_last, non_blocking=True)
        self._host_done[k].record(main)
        prev, self._host_pending = self._host_pending, k
        if not lagged:
            self._host_done[k].synchronize()
            self._host_pending = None
            return float(self._host_loss[k].item())
        if prev is None:
            return float("nan")
        self._host_done[prev].synchronize()
        return float(self._host_loss[prev].item())

    def flush_host_loss(self) -> float:
        """Loss of the last `train_step_host(..., lagged=True)` step (waits for it)."""
        if self._host_pending is None:
            return float("nan")
        k, self._host_pending = self._host_pending, None
        self._host_done[k].synchronize()
        return float(self._host_loss[k].item())

    @property
    def launches_per_step(self) -> int:
        """libstdadk kernel launches in one optimisation step (counted from the launch sequence)."""
        nh = self.ex.spec.n_hidden
        n = 1                               # all weight images (W, W^T, W1s) in one pack_images launch
        n += nh + nh + nh                   # layer_fwd, layer_bwd, wgrad per block
        if self.learnable:
            n += 3                          # knot + temporal tables (knots move), knot_grad
        n += 1 if not self._norm_fused() else 2    # fused tail {norm, step counter, clip + AdamW + EMA}; or step counter + update
        if self._peer is not None and self.world > 1:
            n += 1                          # peer-memory exchange kernel
        return n

    def profile_step(self, table, perm, n_rows: int, global_rows: int, repeats: int = 10) -> dict:
        """Eager steps with a CUDA-event pair around every libstdadk launch (on the launching stream): average
        duration, launch count and algorithmic FLOPs per kernel, plus the summed step time."""
        rec: List[tuple] = []
        saved = {}

        def wrap(name, fn, flops_of):
            def inner(*a, **k):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                r = fn(*a, **k)
                e1.record()
                rec.append((name(*a, **k) if callable(name) else name, e0, e1, flops_of(*a, **k)))
                return r
            return inner

        rows = float(n_rows)
        f_fwd = lambda a: 2.0 * rows * a.layer.n_in * a.layer.n_out
        f_bwd = lambda a: 2.0 * rows * a.layer.n_out * (a.layer.n_in + (a.n_next if not a.head else 0))
        f_wg = lambda a: 2.0 * rows * a.n_in * a.n_out
        patches = {
            "layer_fwd": (lambda a: f"layer_fwd[{a.layer.layer_id}]", f_fwd),
            "layer_bwd": (lambda a: f"layer_bwd[{a.layer.layer_id}]", f_bwd),
            "wgrad": (lambda a: f"wgrad[{a.n_in}x{a.n_out}]", f_wg),
            "knot_grad": ("knot_grad", lambda a: 2.0 * rows * a.n_out * self.model.k_spatial),
            "pack_image": ("pack_image", lambda *a, **k: 0.0),
            "pack_images": ("pack_images", lambda *a, **k: 0.0),
            "knots_prepare": ("knots_prepare", lambda *a, **k: 0.0),
            "tknots_prepare": ("knots_prepare", lambda *a, **k: 0.0),
            "grad_sqnorm": ("grad_sqnorm", lambda *a, **k: 0.0),
            "adamw_ema_step": ("adamw_ema_step", lambda *a, **k: 0.0),
        }
        use_graph, self.use_cuda_graph = self.use_cuda_graph, False
        try:
            for fname, (nm, fl) in patches.items():
                saved[fname] = getattr(ops, fname)
                setattr(ops, fname, wrap(nm, saved[fname], fl))
            self.train_step(table, perm, 0, n_rows, global_rows)        # warm
            rec.clear()
            s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s0.record()
            for i in range(repeats):
                self.train_step(table, perm, (i + 1) * n_rows, n_rows, global_rows)
            s1.record()
            torch.cuda.synchronize()
        finally:
            for fname, fn in saved.items():
                setattr(ops, fname, fn)
            self.use_cuda_graph = use_graph
        agg: Dict[str, dict] = {}
        for name, e0, e1, fl in rec:
            d = agg.setdefault(name, {"ms": 0.0, "count": 0, "flops": fl})
            d["ms"] += e0.elapsed_time(e1)
            d["count"] += 1
        for d in agg.values():
            d["count"] = d["count"] / repeats        # launches per step
            d["ms"] = d["ms"] / (d["count"] * repeats)  # average per launch
        return {"kernels": agg, "step_ms": sum(d["ms"] * d["count"] for d in agg.values()),
                "eager_step_ms_wall": s0.elapsed_time(s1) / repeats}

    def pop_loss_sum(self) -> float:
        v = float(self.loss_sum.item())
        self.loss_sum.zero_()
        return v

    # ------------------------------------------------------------------ evaluation
    @torch.no_grad()
    def evaluate(self, table, batch_rows: int = 65536, with_loss: bool = True):
        """Forward over a whole table in chunks; returns (yhat (N, Q) on device, mean of per-batch losses) --
        the batching matters because upstream averages batch losses (train_st_interp.py:741-792)."""
        ex = self.ex
        n = len(table)
        out = torch.empty(n, self.q, device=self.device)
        self._refresh_head()
        ex.prepare(force=True, for_backward=False)
        losses = []
        for b in range(0, n, batch_rows):
            r = min(batch_rows, n - b)
            pts = ops.make_points(table.coords, table.t, table.X, row_begin=b, n_rows=r)
            if with_loss:
                ex.loss_acc.zero_()
                ex.forward(pts, train=False, y=table.y, loss=self.loss, inv_count=1.0 / (r * self.q), out=out[b:b + r],
                           prepared=True)
                losses.append(ex.loss_acc.clone())
            else:
                ex.forward(pts, train=False, out=out[b:b + r], prepared=True)
        loss = float(torch.stack(losses).mean().item()) if losses else float("nan")
        if with_loss:
            ex.loss_acc.zero_()      # training steps rely on the accumulator being zero between steps
        return out, loss

    def state_for_checkpoint(self):
        return {k: v.detach().clone() for k, v in self.model.state_dict().items()}


# ------------------------------------------------------------------------------------------------
def epoch_permutation(n: int, device, shuffle: bool = True) -> torch.Tensor:
    """The order torch's DataLoader(shuffle=True) would visit `n` samples, drawn from the global CPU generator
    with RandomSampler's own calls (seed <- random_(); randperm(n, generator=Generator(seed))) so that a seeded
    run sees the same batches as upstream (SURVEY.md 9.4)."""
    if not shuffle:
        return torch.arange(n, dtype=torch.int64, device=device)
    seed = int(torch.empty((), dtype=torch.int64).random_().item())
    gen = torch.Generator()
    gen.manual_seed(seed)
    return torch.randperm(n, generator=gen).to(device)


def draw_loader_base_seed():
    """DataLoader iterator construction consumes one number from the global generator (dataloader.py); upstream
    builds a train and a validation iterator every epoch, which shifts the stream the sampler seed comes from."""
    torch.empty((), dtype=torch.int64).random_()


def shard_rows(n: int, rank: int, world: int):
    """Contiguous block partition [floor(r n / R), floor((r+1) n / R))."""
    return (rank * n) // world, ((rank + 1) * n) // world


# ------------------------------------------------------------------------------------------------
def fit(model, train_table, val_table, config: dict, device, output_dir=None, batch_size: int = 256,
        val_batch_size: Optional[int] = None, use_cuda_graph: bool = True, verbose: bool = True, shuffle: bool = True):
    """Epoch loop with the semantics of upstream `train_model` (scripts/train_st_interp.py:463-881): per-epoch
    permutation drawn like DataLoader(shuffle=True), EMA-weight validation, cosine/warm-up/unfreeze schedule, best
    checkpoint = EMA weights at the lowest validation loss, early stopping on `patience`, training_history.csv.
    Returns (model, history, basis_centers_history).

    Data parallel: when torch.distributed is initialised (world > 1) every rank holds the tables, draws the SAME
    permutation (same seed => same global-RNG draws) and takes its contiguous block of every global batch of
    `batch_size` samples; one gradient exchange per step; replicas stay bit-identical, so every rank evaluates the
    same validation loss and takes the same early-stopping decision.  Rank 0 alone writes files."""
    dev = torch.device(device)
    train_table, val_table = train_table.to(dev), val_table.to(dev)
    n = len(train_table)
    bpe = max(1, math.ceil(n / batch_size))
    tr = Trainer(model, config, dev, batches_per_epoch=bpe, use_cuda_graph=use_cuda_graph)
    if val_batch_size is None:
        val_batch_size = min(max(batch_size * 16, 32768), max(len(val_table), 1))
    epochs = int(config.get("epochs", 100))
    patience = int(config.get("patience", 15))
    rtype = config.get("regression_type", "mean")
    taus = config.get("quantile_levels", [0.1, 0.5, 0.9])
    history = {"train_loss": [], "val_loss": [], "val_rmse": [], "lr": []}
    centers_hist = []
    best, best_state, bad = float("inf"), None, 0
    best_path = os.path.join(str(output_dir), "model_best.pt") if output_dir is not None else None
    pen_nc = None
    for epoch in range(epochs):
        tr.begin_epoch(epoch)
        model.train()
        draw_loader_base_seed()                       # train DataLoader iterator
        perm = epoch_permutation(n, dev, shuffle)
        for b in range(bpe):
            lo = b * batch_size
            nb = min(batch_size, n - lo)
            if tr.world > 1:       # this rank's block of the global batch (loss and dropout keys are global)
                r0, r1 = shard_rows(nb, tr.rank, tr.world)
                tr.train_step(train_table, perm, lo + r0, r1 - r0, nb, key_offset=r0)
            else:
                tr.train_step(train_table, perm, lo, nb)
        train_loss = tr.pop_loss_sum() / bpe
        if math.isnan(train_loss):
            print(f"\n[WARNING] NaN detected in epoch {epoch + 1}!")
        # validation under EMA weights (train_st_interp.py:737-806)
        model.eval()
        tr.flat.apply_shadow()
        draw_loader_base_seed()                       # validation DataLoader iterator
        yv, val_loss = tr.evaluate(val_table, val_batch_size)
        if rtype == "multi-quantile" and config.get("use_delta_reparameterization", False):
            terms = [t for t in tr._penalty_terms()][-1:] if float(config.get("non_crossing_lambda", 0.0)) > 0 else []
            if terms:
                val_loss += float(terms[0].item())
        tr.flat.restore()
        col = len(taus) // 2 if rtype == "multi-quantile" else 0
        val_rmse = float(torch.sqrt(torch.mean((yv[:, col] - val_table.y) ** 2)).item())
        cur_lr = tr.opt.param_groups[0]["lr"]
        history["train_loss"].append(train_loss)
        history["val_loss"].append(val_loss)
        history["val_rmse"].append(val_rmse)
        history["lr"].append(cur_lr)
        msg = f"Epoch {epoch + 1}/{epochs}: Train={train_loss:.6f}, Val={val_loss:.6f}, RMSE={val_rmse:.6f}"
        if tr.scheduler is not None and epoch >= tr.warmup_epochs:
            tr.end_epoch(epoch)
            msg += f", LR={tr.scheduler.get_last_lr()[0]:.6f}"
        elif epoch < tr.warmup_epochs:
            msg += f", LR={cur_lr:.6f}(warmup)"
        if not math.isnan(val_loss) and val_loss < best:
            best, bad = val_loss, 0
            tr.flat.apply_shadow()
            best_state = tr.state_for_checkpoint()
            if best_path is not None and tr.rank == 0:
                torch.save(best_state, best_path)
            tr.flat.restore()
            msg += " [Best]"
        else:
            bad += 1
            msg += f" ({bad}/{patience})"
        if verbose and tr.rank == 0:
            print(msg)
        if tr.learnable and (epoch + 1) % 100 == 0:
            centers_hist.append((epoch + 1, model.spatial_basis.centers.detach().cpu().numpy().copy()))
        if bad >= patience:      # a NaN epoch never improves `best`, so upstream too runs on until patience is spent
            if verbose and bad >= patience:
                print(f"\nEarly stopping triggered at epoch {epoch + 1}")
            break
    if best_state is not None:
        model.load_state_dict(best_state)
        if verbose:
            print(f"\nTraining Complete! Best Val Loss: {best:.6f} (EMA model)")
    else:
        tr.flat.p.copy_(tr.flat.shadow)
    if output_dir is not None and tr.rank == 0:
        import pandas as pd
        pd.DataFrame({"epoch": list(range(1, len(history["train_loss"]) + 1)), **history}).to_csv(
            os.path.join(str(output_dir), "training_history.csv"), index=False)
    model._trainer = tr
    return model, history, centers_hist
