"""Structured log-posterior specification -- what ``define_model_log_prob`` returns in this engine.

The reference hands hamiltorch an opaque Python closure (``log_prob_func(params) -> scalar``,
Neural_network/VI_HMC/main_VI_HMC.py:96-153).  A CUDA engine cannot call Python once per leapfrog
step, so the same factory signatures return a :class:`LogProbSpec` instead: architecture, data,
prior, likelihood and the VI-HMC split, i.e. everything the closure captured.

Flat parameter layout == ``torch.cat([p.flatten() for p in model.parameters()])`` (util.py:121-122),
row-major per tensor (util.py:125-136).
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch

ACT_TANH, ACT_RELU, ACT_SINE = 0, 1, 2
_ACT_CODES = {"tanh": ACT_TANH, "relu": ACT_RELU, "sine": ACT_SINE}
LOSS_NLL, LOSS_REGRESSION = 0, 1
_LOSS_CODES = {"NLL": LOSS_NLL, "regression": LOSS_REGRESSION}
MODEL_MLP, MODEL_DEEPONET = 0, 1
MAX_LAYERS = 16


def act_code(name: str) -> int:
    if name not in _ACT_CODES:
        raise ValueError("Activation should be relu, sine or tanh")
    return _ACT_CODES[name]


def loss_code(name) -> int:
    if name not in _LOSS_CODES:
        # the reference's classification losses / callables are never used by its shipped configs
        raise NotImplementedError(f"model_loss {name!r}: only 'NLL' and 'regression' are on the hot path")
    return _LOSS_CODES[name]


@dataclass(frozen=True)
class MLPArch:
    """nn.Sequential(Linear(in,w0),act,...,Linear(w_last,out,bias=last_bias)) -- main_VI_HMC.py:297-334."""
    in_dim: int
    widths: Tuple[int, ...]
    out_dim: int = 1
    act: str = "tanh"
    last_bias: bool = True

    @property
    def layer_dims(self) -> List[Tuple[int, int]]:
        dims, prev = [], self.in_dim
        for w in list(self.widths) + [self.out_dim]:
            dims.append((w, prev))
            prev = w
        return dims

    def tensor_numels(self) -> List[int]:
        out = []
        dims = self.layer_dims
        for li, (o, i) in enumerate(dims):
            out.append(o * i)
            if li < len(dims) - 1 or self.last_bias:
                out.append(o)
        return out

    @property
    def num_params(self) -> int:
        return sum(self.tensor_numels())

    @staticmethod
    def from_module(net: torch.nn.Module) -> "MLPArch":
        """Read the architecture off an nn.Sequential built like the reference's get_model()."""
        linears = [m for m in net.modules() if isinstance(m, torch.nn.Linear)]
        if not linears:
            raise ValueError("expected an nn.Sequential of Linear/activation layers")
        acts = [m for m in net.modules() if not isinstance(m, (torch.nn.Linear, torch.nn.Sequential))]
        act = "tanh"
        if acts:
            name = type(acts[0]).__name__.lower()
            act = {"tanh": "tanh", "relu": "relu", "sin": "sine", "sine": "sine"}.get(name)
            if act is None:
                raise ValueError("Activation should be relu, sine or tanh")
        for a, b in zip(linears[:-1], linears[1:]):
            if a.out_features != b.in_features:
                raise ValueError("not a plain MLP")
        if any(l.bias is None for l in linears[:-1]):
            raise ValueError("hidden layers must have a bias")
        return MLPArch(in_dim=linears[0].in_features, widths=tuple(l.out_features for l in linears[:-1]),
                       out_dim=linears[-1].out_features, act=act, last_bias=linears[-1].bias is not None)


@dataclass(frozen=True)
class DeepONetArch:
    """Operator_network/VI_HMC/model.py:11-62.  Flat order: scalar b, branch stack, trunk stack."""
    width_branch: int = 100
    width_trunk: int = 100
    in_branch: int = 101
    in_trunk: int = 5
    depth_branch: int = 9
    depth_trunk: int = 9
    output_neurons: int = 100
    act: str = "tanh"
    impose_bc: bool = True

    def stack_dims(self, which: str) -> List[Tuple[int, int]]:
        in_dim, width, depth = ((self.in_branch, self.width_branch, self.depth_branch) if which == "branch"
                                else (self.in_trunk, self.width_trunk, self.depth_trunk))
        dims, prev = [], in_dim
        for w in [width] * (depth - 1) + [self.output_neurons]:
            dims.append((w, prev))
            prev = w
        return dims

    def tensor_numels(self) -> List[int]:
        out = [1]
        for which in ("branch", "trunk"):
            for o, i in self.stack_dims(which):
                out += [o * i, o]
        return out

    @property
    def num_params(self) -> int:
        return sum(self.tensor_numels())

    @staticmethod
    def from_module(net) -> "DeepONetArch":
        act = type(net.act).__name__.lower()
        return DeepONetArch(width_branch=net.width_branch, width_trunk=net.width_trunk, in_branch=net.in_branch,
                            in_trunk=net.in_trunk, depth_branch=net.depth_branch, depth_trunk=net.depth_trunk,
                            output_neurons=net.output_neurons, act={"tanh": "tanh", "relu": "relu"}[act],
                            impose_bc=getattr(net, "impose_bc", True))


@dataclass
class LogProbSpec:
    """Everything the reference closure captured, as data.

    q (the sampled vector, length d) maps into the full weight vector W (length D) by
    ``W = frozen.clone(); W[sens_ind] = q`` (my_make_func.py:56-57); d == D and no frozen vector
    means plain HMC.  The prior is per coordinate of q: N(prior_mu_i, prior_sigma_i), divided by
    ``prior_scale`` (main_VI_HMC.py:151).  sigma = inf encodes "no prior on this coordinate".
    """
    arch: object                                   # MLPArch | DeepONetArch
    x: torch.Tensor                                # MLP: [N,in]; DeepONet: branch inputs [N,in_branch]
    y: torch.Tensor                                # MLP: [N,out]; DeepONet: [N,P]
    x2: Optional[torch.Tensor] = None              # DeepONet trunk coordinates [P,2] (t, x)
    loss: str = "NLL"
    tau_out: float = 1.0
    prior_mu: Optional[torch.Tensor] = None        # [d] or None (zero mean)
    prior_sigma: Optional[torch.Tensor] = None     # [d] or None (use prior_sigma_scalar)
    prior_sigma_scalar: float = 1.0
    prior_scale: float = 1.0
    frozen: Optional[torch.Tensor] = None          # [D] VI means (my_make_func.py:32) or None
    sens_ind: Optional[np.ndarray] = None          # sorted int64 [d] or None
    vi_sigma: Optional[torch.Tensor] = None        # [D] VI stds, only for the optional redraw hook
    predict: bool = False
    trunk_subsample: Optional[int] = None          # DeepONet: cfg.p trunk points redrawn for every closure call (cfg.sample_data)

    @property
    def model_kind(self) -> int:
        return MODEL_MLP if isinstance(self.arch, MLPArch) else MODEL_DEEPONET

    @property
    def D(self) -> int:
        return self.arch.num_params

    @property
    def d(self) -> int:
        return self.D if self.sens_ind is None else int(len(self.sens_ind))

    @property
    def N(self) -> int:
        return int(self.x.shape[0])

    @property
    def P(self) -> int:
        return int(self.y.shape[1]) if self.model_kind == MODEL_DEEPONET else 1

    def validate(self) -> None:
        if (self.frozen is None) != (self.sens_ind is None):
            raise ValueError("frozen weights and sens_ind must be given together")
        if self.sens_ind is not None:
            ind = np.asarray(self.sens_ind)
            if ind.ndim != 1 or ind.size == 0:
                raise ValueError("sens_ind must be a non-empty 1-D index array")
            if ind.min() < 0 or ind.max() >= self.D:
                raise IndexError("sens_ind out of range")
            if np.unique(ind).size != ind.size:
                raise ValueError("sens_ind must not contain duplicates")
            if int(self.frozen.numel()) != self.D:
                raise ValueError(f"frozen weights have {self.frozen.numel()} entries, architecture has {self.D}")
        for name in ("prior_mu", "prior_sigma"):
            t = getattr(self, name)
            if t is not None and int(t.numel()) != self.d:
                raise ValueError(f"{name} must have d={self.d} entries")
        if self.model_kind == MODEL_DEEPONET:
            if self.x2 is None:
                raise ValueError("DeepONet spec needs trunk coordinates x2")
            if tuple(self.y.shape) != (self.N, int(self.x2.shape[0])):
                raise ValueError("y must be [N, P]")
            # the kernels read x2 with a fixed row stride (2 for the (t, x) pairs of the feature layer, in_trunk for raw
            # trunk inputs): any other width would be read as the wrong numbers, not refused
            cols = 2 if self.arch.impose_bc else self.arch.in_trunk
            if self.x2.dim() != 2 or int(self.x2.shape[1]) != cols:
                what = "(t, x) pairs for the feature layer" if self.arch.impose_bc else f"in_trunk = {cols} raw trunk inputs"
                raise ValueError(f"x2 must be [P, {cols}] ({what}), got {tuple(self.x2.shape)}")
        loss_code(self.loss)
        if self.trunk_subsample is not None:
            if self.model_kind != MODEL_DEEPONET:
                raise ValueError("trunk_subsample is a DeepONet option (cfg.sample_data)")
            if not 1 <= int(self.trunk_subsample) <= self.P:
                raise ValueError("Sample larger than population or is negative")   # random.sample's message


def sliced_prior_sigma(d: int, tensor_numels: Sequence[int], prior_vars: Sequence[float]) -> np.ndarray:
    """Per-coordinate prior std implied by the reference's slice loop (main_VI_HMC.py:107-112).

    The loop walks the REDUCED vector q with the FULL tensors' lengths: coordinate i gets the variance
    of whichever slice [i_prev, i_prev+numel) contains it, and coordinates past the last slice get no
    prior (sigma = inf).  With the shipped equal variances this is an isotropic Gaussian over q.
    """
    sig = np.full(d, np.inf, dtype=np.float64)
    i_prev = 0
    for n, v in zip(tensor_numels, prior_vars):
        hi = min(d, i_prev + n)
        if i_prev < hi:
            sig[i_prev:hi] = float(v) ** 0.5
        i_prev += n
    return sig
