"""Drop-in `stnf.models.st_interp` on the B200-native kernels.

Same public surface as the upstream module (classes, constructor keywords, attribute and
state_dict names, penalty helpers, `create_model`), but `forward` does not run PyTorch ops: it
hands raw device pointers to libstdadk.so (include/stdadk.h), where block 1 generates the basis
inside the tensor-core operand and every Linear/LayerNorm/ReLU/Dropout block is one tcgen05 kernel.
Upstream references are cited as `st_interp.py:line`.

CUDA (sm_100) only: a CPU tensor raises -- there is no fallback path.
"""
from __future__ import annotations

import math
from typing import List, Optional

import numpy as np
import torch
import torch.nn as nn

from st_dadk_b200 import _lib as _L
from st_dadk_b200 import ops as _ops
from st_dadk_b200.executor import Executor, NetSpec
from st_dadk_b200 import knot_init as _knot_init

__all__ = ["SpatialBasisEmbedding", "TemporalBasisEmbedding", "STInterpMLP", "create_model"]


def _need_cuda(t: torch.Tensor, what: str):
    if not t.is_cuda:
        raise RuntimeError(f"stnf (st_dadk_b200): {what} is on {t.device}; this implementation runs on CUDA "
                           "sm_100 only and has no CPU fallback (move the model and inputs to 'cuda').")


class SpatialBasisEmbedding(nn.Module):
    """phi(s): multi-resolution radial basis on [0,1]^2 (st_interp.py:18-546).

    Knot placement ('uniform' lattice, 'gmm', 'random_site', 'kmeans_balanced') is one-off host work
    (st_dadk_b200.knot_init); evaluation happens on the GPU.  When `learnable`, `centers` and
    `log_bandwidths` are Parameters and their gradients come from the knot-gradient kernel.
    """

    CALIBRATION_FACTORS = dict(_L.CALIBRATION)  # st_interp.py:56-60

    def __init__(self, n_centers: list = [25, 81, 121], learnable: bool = False, init_method: str = "uniform",
                 train_coords: np.ndarray = None, basis_function: str = "wendland", gradient_damping: bool = False,
                 damping_threshold: float = 0.3, damping_strength: float = 1.0):
        super().__init__()
        if basis_function not in self.CALIBRATION_FACTORS:
            raise ValueError(f"Unknown basis function: {basis_function}. "
                             f"Choose from {list(self.CALIBRATION_FACTORS.keys())}")
        self.n_centers = n_centers
        self.learnable = learnable
        self.init_method = init_method
        self.basis_function = basis_function
        self.gradient_damping = gradient_damping
        self.damping_threshold = damping_threshold
        self.damping_strength = damping_strength

        centers, bandwidths = _knot_init.place_knots(init_method, n_centers, train_coords)
        self.k = int(centers.shape[0])
        if learnable:
            self.centers = nn.Parameter(centers)
            self.register_buffer("centers_init", centers.clone())
            self.log_bandwidths = nn.Parameter(bandwidths.log())
            if gradient_damping:
                self.centers.register_hook(self._gradient_damping_hook)
        else:
            self.register_buffer("centers", centers)
            self.register_buffer("_bandwidths", bandwidths)

    # st_interp.py:111-142 -- gradient of a knot that drifted d beyond the threshold is scaled by exp(-strength*d)
    _hook_enabled = True      # the trainer switches the hook off while it differentiates parameter-only penalties

    def _damping_factor(self):
        with torch.no_grad():
            drift = (self.centers - self.centers_init).norm(dim=1, keepdim=True)
            return torch.exp(-self.damping_strength * (drift - self.damping_threshold).clamp_min(0.0))

    def _gradient_damping_hook(self, grad):
        if not self._hook_enabled:
            return grad
        return grad * self._damping_factor()

    @property
    def bandwidths(self):
        return self.log_bandwidths.exp() if self.learnable else self._bandwidths

    def forward(self, coords: torch.Tensor) -> torch.Tensor:
        """Dense phi (N, k) from the unfused parity kernel (values only; gradients with respect to the
        knots flow through STInterpMLP.forward, which never materialises this matrix)."""
        _need_cuda(coords, "coords")
        batched = coords.dim() == 3
        flat = coords.reshape(-1, 2).float().contiguous()
        with torch.no_grad():
            knots4 = _ops.knots_prepare(self.centers.detach(), None if self.learnable else self._bandwidths,
                                        self.log_bandwidths.detach() if self.learnable else None, self.basis_function)
            tk = torch.zeros(1, 2, device=flat.device)
            basis = _ops.make_basis(knots4, tk, self.k, 0, 0, self.basis_function)
            tt = torch.zeros(flat.shape[0], 1, device=flat.device)
            phi, _ = _ops.basis_fwd(basis, _ops.make_points(flat, tt), flat.device)
        return phi.view(*coords.shape[:-1], self.k) if batched else phi

    # st_interp.py:493-546
    def compute_domain_penalty(self, domain_bounds=(0.0, 1.0)):
        if not self.learnable:
            return torch.tensor(0.0, device=self.centers.device)
        lo, hi = domain_bounds
        out = (lo - self.centers).clamp_min(0.0) + (self.centers - hi).clamp_min(0.0)
        return out.square().sum()

    def compute_movement_penalty(self):
        if not self.learnable:
            return torch.tensor(0.0, device=self.centers.device)
        return (self.centers - self.centers_init).square().sum()


class TemporalBasisEmbedding(nn.Module):
    """psi(t): Gaussian bumps on per-level grids linspace(0,1,n), bandwidth 2.5/(n-1) (st_interp.py:549-596)."""

    def __init__(self, n_centers: list = [10, 15, 45]):
        super().__init__()
        self.n_centers = n_centers
        centers, bandwidths = _knot_init.temporal_knots(n_centers)
        self.register_buffer("centers", centers)
        self.register_buffer("bandwidths", bandwidths)
        self.k_time = int(centers.shape[0])

    def forward(self, t: torch.Tensor) -> torch.Tensor:
        _need_cuda(t, "t")
        flat = t.reshape(-1, 1).float().contiguous()
        with torch.no_grad():
            tk = _ops.tknots_prepare(self.centers, self.bandwidths)
            k4 = torch.zeros(1, 4, device=flat.device)
            basis = _ops.make_basis(k4, tk, 0, self.k_time, 0, "wendland")
            cc = torch.zeros(flat.shape[0], 2, device=flat.device)
            _, psi = _ops.basis_fwd(basis, _ops.make_points(cc, flat), flat.device)
        return psi.view(*t.shape[:-1], self.k_time)


class _NetFunction(torch.autograd.Function):
    """Autograd bridge: forward = Executor.forward(save), backward = Executor.backward(dyhat)."""

    @staticmethod
    def forward(ctx, model, coords, t, X, head_w, head_b, *params):
        ex, spec = model._executor(head_w, head_b)
        pts = _ops.make_points(coords, t, X)
        train = model.training
        if train and spec.dropout > 0.0:
            model._dropout_step += 1
        yhat = ex.forward(pts, train=train, step=model._dropout_step, seed=model._dropout_seed(), save=True)
        ctx.model = model
        ctx.keep = (coords, t, X)   # the kernels read these again in backward (basis recompute)
        ctx.n_params = len(params)
        return yhat.clone()

    @staticmethod
    def backward(ctx, dy):
        model = ctx.model
        ex = model._ex
        g = ex.backward(dyhat=dy.contiguous().float())
        out = model._grads_in_param_order(g)
        return (None, None, None, None, g["head_w"].clone(), g["head_b"].clone(), *out)


class STInterpMLP(nn.Module):
    """[X, phi(s), psi(t)] -> (Linear -> LayerNorm -> ReLU -> Dropout) x len(hidden_dims) -> Linear | delta head
    (st_interp.py:599-882)."""

    def __init__(self, p: int = 0, k_spatial_centers: list = [25, 81, 121], k_temporal_centers: list = [10, 15, 45],
                 hidden_dims: list = [256, 256, 128], dropout: float = 0.1, layernorm: bool = True,
                 spatial_learnable: bool = False, spatial_init_method: str = "uniform",
                 spatial_basis_function: str = "wendland", train_coords: np.ndarray = None,
                 gradient_damping: bool = False, damping_threshold: float = 0.3, damping_strength: float = 1.0,
                 output_dim: int = 1, use_delta_reparameterization: bool = False):
        super().__init__()
        self.p = p
        self.k_spatial_centers = k_spatial_centers
        self.spatial_init_method = spatial_init_method
        self.spatial_basis_function = spatial_basis_function
        self.output_dim = output_dim
        self.use_delta_reparameterization = use_delta_reparameterization
        self._dropout_p = float(dropout)
        self._layernorm = bool(layernorm)
        self._hidden_dims = list(hidden_dims)

        self.spatial_basis = SpatialBasisEmbedding(
            n_centers=k_spatial_centers, learnable=spatial_learnable, init_method=spatial_init_method,
            train_coords=train_coords, basis_function=spatial_basis_function, gradient_damping=gradient_damping,
            damping_threshold=damping_threshold, damping_strength=damping_strength)
        self.temporal_basis = TemporalBasisEmbedding(n_centers=k_temporal_centers)
        self.k_spatial = self.spatial_basis.k
        self.k_temporal = self.temporal_basis.k_time

        # Module order (and therefore RNG draw order and state_dict indices) as upstream: st_interp.py:656-692
        stack: List[nn.Module] = []
        width = p + self.k_spatial + self.k_temporal
        for h in hidden_dims:
            stack.append(nn.Linear(width, h))
            if layernorm:
                stack.append(nn.LayerNorm(h))
            stack.append(nn.ReLU())
            if dropout > 0:
                stack.append(nn.Dropout(dropout))
            width = h
        self.last_hidden_dim = width
        if use_delta_reparameterization and output_dim > 1:
            self.mlp_trunk = nn.Sequential(*stack)
            self.delta_params = nn.ParameterList([nn.Parameter(torch.zeros(width + 1)) for _ in range(output_dim)])
            for d in self.delta_params:
                nn.init.normal_(d, mean=0.0, std=0.01)
        else:
            stack.append(nn.Linear(width, output_dim))
            self.mlp = nn.Sequential(*stack)
            self.mlp_trunk = None
            self.delta_params = None
        self._ex: Optional[Executor] = None
        # tensor-core precision of the kernels under this module: "tf32" (throughput) or "tf32x3" (FP32-faithful
        # three-pass split, see NetSpec.precision); `create_model` reads it from the config key `precision`
        self.precision = "tf32"
        self._dropout_step = 0
        self._seed_override: Optional[int] = None

    # ------------------------------------------------------------------ structure helpers
    def _trunk(self) -> nn.Sequential:
        return self.mlp_trunk if self.mlp_trunk is not None else self.mlp

    def hidden_blocks(self):
        """[(Linear, LayerNorm|None)] of the hidden blocks, in order."""
        mods = list(self._trunk())
        if self.mlp_trunk is None:
            mods = mods[:-1]
        blocks, i = [], 0
        while i < len(mods):
            lin = mods[i]
            ln = mods[i + 1] if i + 1 < len(mods) and isinstance(mods[i + 1], nn.LayerNorm) else None
            blocks.append((lin, ln))
            i += 1
            while i < len(mods) and not isinstance(mods[i], nn.Linear):
                i += 1
        return blocks

    def _dropout_seed(self) -> int:
        return self._seed_override if self._seed_override is not None else (torch.initial_seed() & (2 ** 63 - 1))

    def _effective_head(self):
        """(Q, d) weight and (Q,) bias: the Linear head, or beta_k = sum_{l<=k} delta_l (st_interp.py:859-873)."""
        if self.delta_params is not None:
            beta = torch.cumsum(torch.stack(list(self.delta_params)), dim=0)
            return beta[:, 1:], beta[:, 0]
        head = self.mlp[-1]
        return head.weight, head.bias

    def net_spec(self, head_w=None, head_b=None) -> NetSpec:
        sb = self.spatial_basis
        if head_w is None:
            head_w, head_b = self._effective_head()
        blocks = self.hidden_blocks()
        return NetSpec(
            centers=sb.centers.detach(), bandwidths=None if sb.learnable else sb._bandwidths,
            log_bandwidths=sb.log_bandwidths.detach() if sb.learnable else None,
            t_centers=self.temporal_basis.centers, t_bandwidths=self.temporal_basis.bandwidths,
            weights=[lin.weight.detach() for lin, _ in blocks], biases=[lin.bias.detach() for lin, _ in blocks],
            gammas=[ln.weight.detach() if ln is not None else None for _, ln in blocks],
            betas=[ln.bias.detach() if ln is not None else None for _, ln in blocks],
            head_w=head_w.detach().contiguous(), head_b=head_b.detach().contiguous(),
            basis_fn=self.spatial_basis_function, p_cov=self.p, dropout=self._dropout_p,
            ln_eps=blocks[0][1].eps if blocks and blocks[0][1] is not None else 1e-5, learnable_basis=sb.learnable,
            lattice_sides=[int(math.sqrt(k)) for k in sb.n_centers]
            if (sb.init_method == "uniform" and not sb.learnable) else None,
            level_sizes=[int(k) for k in sb.n_centers], precision=getattr(self, "precision", "tf32"))

    def _executor(self, head_w=None, head_b=None):
        spec = self.net_spec(head_w, head_b)
        for hdim in self._hidden_dims:
            if hdim > _L.MAX_WIDTH:
                raise RuntimeError(f"hidden width {hdim} > {_L.MAX_WIDTH} is not supported by the tcgen05 block kernels "
                                   f"(one LayerNorm row per CTA, one of the {_L.MAX_WIDTH} tensor-memory columns per unit)")
        if self._ex is None or self._ex.device != spec.centers.device:
            self._ex = Executor(spec)
        else:
            self._ex.rebind(spec)
        return self._ex, spec

    def _param_inputs(self):
        ps = []
        for lin, ln in self.hidden_blocks():
            ps += [lin.weight, lin.bias]
            if ln is not None:
                ps += [ln.weight, ln.bias]
        if self.spatial_basis.learnable:
            ps += [self.spatial_basis.centers, self.spatial_basis.log_bandwidths]
        return ps

    def _grads_in_param_order(self, g):
        out = []
        for l, (lin, ln) in enumerate(self.hidden_blocks()):
            out += [g["weights"][l].clone(), g["biases"][l].clone()]
            if ln is not None:
                out += [g["gammas"][l].clone(), g["betas"][l].clone()]
        if self.spatial_basis.learnable:
            out += [g["centers"].clone(), g["log_bandwidths"].clone()]
        return out

    # ------------------------------------------------------------------ forward
    def forward(self, X: torch.Tensor, coords: torch.Tensor, t: torch.Tensor) -> torch.Tensor:
        """y_hat (N, Q) for covariates X (N, p) (may be (N, 0)), coords (N, 2), t (N, 1) (st_interp.py:827-882)."""
        _need_cuda(coords, "coords")
        _need_cuda(self.temporal_basis.centers, "the model")
        coords = coords.detach().float().contiguous()
        t = t.detach().float().reshape(-1).contiguous()
        if coords.dim() != 2 or coords.shape[1] != 2 or t.shape[0] != coords.shape[0]:
            raise ValueError(f"expected coords (N, 2) and t (N, 1); got {tuple(coords.shape)} and {tuple(t.shape)}")
        Xc = X.detach().float().contiguous() if (X is not None and X.numel() > 0 and self.p > 0) else None
        if self.p > 0 and Xc is None:
            raise ValueError(f"model has p={self.p} covariates but X is empty")
        head_w, head_b = self._effective_head()
        if coords.shape[0] == 0:
            return torch.zeros(0, self.output_dim, device=coords.device)
        if torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters()):
            return _NetFunction.apply(self, coords, t, Xc, head_w, head_b, *self._param_inputs())
        with torch.no_grad():
            ex, spec = self._executor(head_w, head_b)
            train = self.training
            if train and spec.dropout > 0.0:
                self._dropout_step += 1
            pts = _ops.make_points(coords, t, Xc)
            return ex.forward(pts, train=train, step=self._dropout_step, seed=self._dropout_seed()).clone()

    # ------------------------------------------------------------------ reference helper API
    def compute_domain_penalty(self):
        return self.spatial_basis.compute_domain_penalty()

    def compute_movement_penalty(self):
        return self.spatial_basis.compute_movement_penalty()

    def get_delta_parameters(self):
        if not self.use_delta_reparameterization or self.delta_params is None:
            return None
        return list(self.delta_params)

    def compute_sparsity_penalty(self, penalty_type="element", lambda_l1=0.01, lambda_group=0.01):
        """L1 / group-lasso / sparse-group penalties on the first Linear's spatial and temporal column blocks
        (st_interp.py:724-825); the per-basis norms are one vectorised reduction instead of a Python loop."""
        if penalty_type not in ("element", "group", "sparse_group", "none"):
            raise ValueError(f"Unknown penalty_type: {penalty_type}")
        W = self._trunk()[0].weight
        zero = W.new_zeros(())
        if penalty_type == "none":
            return {"spatial_penalty": zero, "temporal_penalty": zero.clone(), "total_penalty": zero.clone()}

        def block_penalty(block):  # block: (hidden, n_basis) columns of W
            l1 = block.abs().sum()
            grp = block.norm(dim=0).sum()
            if penalty_type == "element":
                return lambda_l1 * l1
            if penalty_type == "group":
                return lambda_group * grp
            return lambda_group * grp + lambda_l1 * l1

        s0 = self.p
        sp = block_penalty(W[:, s0:s0 + self.k_spatial])
        tp = block_penalty(W[:, s0 + self.k_spatial:s0 + self.k_spatial + self.k_temporal])
        return {"spatial_penalty": sp, "temporal_penalty": tp, "total_penalty": sp + tp}

    def __deepcopy__(self, memo):
        import copy
        ex, self._ex = self._ex, None           # the executor's workspaces are not part of the model state
        try:
            cls = self.__class__
            new = cls.__new__(cls)
            memo[id(self)] = new
            for k, v in self.__dict__.items():
                setattr(new, k, copy.deepcopy(v, memo))
        finally:
            self._ex = ex
        return new


def create_model(config: dict, train_coords: np.ndarray = None) -> STInterpMLP:
    """Config dict -> model, with the upstream defaults for every key (st_interp.py:885-919)."""
    multi = config.get("regression_type", "mean") == "multi-quantile"
    q = len(config.get("quantile_levels", [0.1, 0.5, 0.9])) if multi else 1
    get = config.get
    model = STInterpMLP(
        p=get("p_covariates", 0), k_spatial_centers=get("k_spatial_centers", [25, 81, 121]),
        k_temporal_centers=get("k_temporal_centers", [10, 15, 45]), hidden_dims=get("hidden_dims", [256, 256, 128]),
        dropout=get("dropout", 0.1), layernorm=get("layernorm", True), spatial_learnable=get("spatial_learnable", False),
        spatial_init_method=get("spatial_init_method", "uniform"),
        spatial_basis_function=get("spatial_basis_function", "wendland"), train_coords=train_coords,
        gradient_damping=get("gradient_damping", False), damping_threshold=get("damping_threshold", 0.3),
        damping_strength=get("damping_strength", 1.0), output_dim=q,
        use_delta_reparameterization=get("use_delta_reparameterization", False))
    model.precision = get("precision", "tf32")      # not an upstream key: "tf32" | "tf32x3"
    return model
