"""TEST INFRASTRUCTURE ONLY -- closures with the SHAPE of the reference's ``log_prob_func``.

``vihmc.closure.spec_from_closure`` recovers a specification from what a reference closure captured
(free-variable names and the functional-model object behind ``fmodel``).  The original project is not part of
this repository, so the tests need closures that capture the same names without importing it.  The factories
below build them on the oracle's restated forward functions; ``tests/test_closure_dropin.py`` checks that they
reproduce, bit for bit, the log-posteriors and gradients the original closures gave (tests/golden/), and, when a
checkout of the original is present, that both yield identical recovered specifications.

Captured names mirrored (reference file:line)
    BNN       x, y, fmodel, dist_list, params_flattened_list, params_shape_list, model, model_loss, tau_out,
              prior_scale, predict, nll_loss       Neural_network/VI_HMC/main_VI_HMC.py:80-153
    object    depth, activation, bias, model, learned_mus, learned_sigmas, sampled_weights, sensitive_ind
                                                    Neural_network/VI_HMC/my_make_func.py:24-43
    DeepONet  tr_data, fmodel, dist_list, model_loss, tau_out, prior_scale, predict, nll_loss
                                                    Operator_network/VI_HMC/main_VI_HMC_burgers.py:67-180
    NUTS      tr_data, fmodel, dist_list, params_flattened_list, model_loss, tau_out, nll_loss
                                                    Operator_network/HMC/NUTS_DeepOnets.py:120-160
    object    depth_branch, depth_trunk, act, impose_bc, model, learned_mus, learned_sigmas, sampled_weights,
              sensitive_ind                         Operator_network/VI_HMC/my_make_func.py:14-31
    globals   cfg.load_prior, cfg.sample_data, cfg.p main_VI_HMC.py:87,104; main_VI_HMC_burgers.py:76,100,127-137 (from random import sample :14)
"""
from __future__ import annotations

import types
from random import sample

import numpy as np
import torch
import torch.nn.functional as F

from . import closures as oc


class Sin(torch.nn.Module):
    def forward(self, x):
        return torch.sin(x)


_ACT_FUNCS = {"tanh": F.tanh, "relu": F.relu}
_ACT_MODULES = {"tanh": torch.nn.Tanh, "relu": torch.nn.ReLU, "sine": Sin}

# the factories read this module-level name exactly as the reference reads ``import config as cfg``
cfg = types.SimpleNamespace(load_prior=False, sample_data=False, p=None)


def mlp_module(in_dim=1, widths=(10, 10), out_dim=1, act="tanh", bias=True) -> torch.nn.Module:
    """An nn.Sequential like the reference's get_model() (main_VI_HMC.py:297-334)."""
    layers, prev = [], in_dim
    for w in widths:
        layers += [torch.nn.Linear(prev, w), _ACT_MODULES[act]()]
        prev = w
    layers.append(torch.nn.Linear(prev, out_dim, bias=bias))
    return torch.nn.Sequential(*layers)


class DeepONetModule(torch.nn.Module):
    """Carries the attributes and the parameter ORDER of the reference's DeepONet (model.py:26,33-34): b, branch, trunk."""

    def __init__(self, width_branch=100, width_trunk=100, in_branch=101, in_trunk=5, depth_branch=9, depth_trunk=9,
                 act="tanh", output_neurons=100):
        super().__init__()
        self.width_branch, self.width_trunk, self.in_branch, self.in_trunk = width_branch, width_trunk, in_branch, in_trunk
        self.depth_branch, self.depth_trunk, self.output_neurons = depth_branch, depth_trunk, output_neurons
        self.act = _ACT_MODULES[act]()
        self.b = torch.nn.Parameter(torch.zeros(1))

        def stack(i, w, depth):
            dims = [i] + [w] * (depth - 1) + [output_neurons]
            return torch.nn.ModuleList([torch.nn.Linear(a, b) for a, b in zip(dims[:-1], dims[1:])])
        self.branch = stack(in_branch, width_branch, depth_branch)
        self.trunk = stack(in_trunk, width_trunk, depth_trunk)


class FunctionalNet:
    def __init__(self, depth, act, bias=True, mus=None, sigmas=None, sensitive_ind=None, model=None):
        self.depth, self.bias, self.model = depth, bias, model
        self.sensitive_ind = sensitive_ind
        self.learned_mus, self.learned_sigmas, self.sampled_weights = mus, sigmas, mus
        self.activation = Sin() if act == "sine" else _ACT_FUNCS[act]
        self._act = act

    def functional_model(self, X, parameters):
        full = oc.scatter_vi(self.sampled_weights, self.sensitive_ind, parameters)
        slots = oc.mlp_layout(X.shape[1], [m.out_features for m in self.model if isinstance(m, torch.nn.Linear)][:-1],
                              [m for m in self.model if isinstance(m, torch.nn.Linear)][-1].out_features, self.bias)
        return oc.mlp_forward(X, oc.unflatten(slots, full), self.depth + 1, self._act, self.bias)


class FunctionalDeepONet:
    def __init__(self, depth_branch=9, depth_trunk=9, mus=None, sigmas=None, activation="relu", sensitive_ind=None,
                 model=None, impose_bc=True):
        self.depth_branch, self.depth_trunk, self.model, self.impose_bc = depth_branch, depth_trunk, model, impose_bc
        self.learned_mus, self.learned_sigmas, self.sampled_weights = mus, sigmas, mus
        self.sensitive_ind = sensitive_ind
        self.act = _ACT_FUNCS[activation]
        self._act = activation

    def functional_model(self, X1, X2, parameters):
        m = self.model
        full = oc.scatter_vi(self.sampled_weights, self.sensitive_ind, parameters)
        slots = oc.deeponet_layout(m.width_branch, m.width_trunk, m.in_branch, m.in_trunk, self.depth_branch,
                                   self.depth_trunk, m.output_neurons)
        return oc.deeponet_forward(X1, X2, oc.unflatten(slots, full), self.depth_branch, self.depth_trunk, self._act,
                                   self.impose_bc)


def _dists(prior_list, load_prior):
    if load_prior:
        return [torch.distributions.Normal(prior_list[0], prior_list[1])]
    return [torch.distributions.Normal(torch.zeros_like(t), t ** 0.5) for t in prior_list]


def bnn_closure(model, model_loss, x, y, params_flattened_list, params_shape_list, prior_list, tau_out, predict=False,
                prior_scale=1.0, params_mu=None, params_std=None, grad_ind=None, depth=1, act="tanh", bias=True):
    """Shape of Neural_network/VI_HMC/main_VI_HMC.py:28-153 (artefacts passed in instead of torch.load'ed)."""
    f_net = FunctionalNet(depth=depth, act=act, bias=bias, mus=params_mu, sigmas=params_std, sensitive_ind=grad_ind, model=model)
    fmodel = f_net.functional_model
    dist_list = _dists(prior_list, cfg.load_prior)
    nll_loss = torch.nn.GaussianNLLLoss(reduction='sum')

    def log_prob_func(params, *args):
        l_prior = torch.zeros_like(params[0], requires_grad=True)
        if cfg.load_prior:
            l_prior = dist_list[0].log_prob(params).sum() + l_prior
        else:
            i_prev = 0
            for weights, index, shape, dist in zip(model.parameters(), params_flattened_list, params_shape_list, dist_list):
                l_prior = dist.log_prob(params[i_prev:index + i_prev]).sum() + l_prior
                i_prev += index
        output = fmodel(x, params)
        if model_loss == 'regression':
            ll = - 0.5 * tau_out * ((output - y) ** 2).sum(0)
        elif model_loss == 'NLL':
            ll = - nll_loss(output, y, tau_out * torch.ones_like(output))
        else:
            raise NotImplementedError()
        return ((ll + l_prior / prior_scale), output) if predict else (ll + l_prior / prior_scale)

    return log_prob_func


def deeponet_closure(model, model_loss, tr_data, tau_list, tau_out, predict=False, prior_scale=1.0, mean_params=None,
                     std_params=None, grad_ind=None, activation="tanh", impose_bc=True):
    """Shape of Operator_network/VI_HMC/main_VI_HMC_burgers.py:27-180 and Operator_network/HMC/main_HMC_splitting.py:79-206."""
    f_deeponet = FunctionalDeepONet(depth_branch=model.depth_branch, depth_trunk=model.depth_trunk, mus=mean_params,
                                    sigmas=std_params, activation=activation, sensitive_ind=grad_ind, model=model,
                                    impose_bc=impose_bc)
    fmodel = f_deeponet.functional_model
    dist_list = _dists(tau_list, cfg.load_prior)
    nll_loss = torch.nn.GaussianNLLLoss(reduction='sum')

    def log_prob_func(params, *args):
        l_prior = dist_list[0].log_prob(params).sum() + torch.zeros_like(params[0], requires_grad=True)
        x1, x2, y = tr_data
        if predict or not cfg.sample_data:
            output = fmodel(x1, x2, parameters=params).squeeze(1)
        else:   # main_VI_HMC_burgers.py:127-137
            ind = sample(range(x2.shape[1]), cfg.p)
            output = fmodel(x1, x2[:, ind], parameters=params).squeeze(1)
            y = y[:, ind]
        assert output.shape == y.shape
        if model_loss == 'NLL':
            ll = - nll_loss(output, y, tau_out * torch.ones_like(output))
        else:
            raise NotImplementedError()
        return ((ll + l_prior / prior_scale), output) if predict else (ll + l_prior / prior_scale)

    return log_prob_func


def deeponet_nuts_closure(model, model_loss, tr_data, params_flattened_list, params_shape_list, tau_list, tau_out,
                          activation="tanh"):
    """Shape of Operator_network/HMC/NUTS_DeepOnets.py:120-160: one prior per parameter tensor, built as Normal(0, tau * 0.5)
    (:132, where every other driver takes tau ** 0.5) and walked by the per-tensor slice loop (:144-150)."""
    f_deeponet = FunctionalDeepONet(depth_branch=model.depth_branch, depth_trunk=model.depth_trunk, activation=activation, model=model)
    fmodel = f_deeponet.functional_model
    dist_list = [torch.distributions.Normal(torch.zeros_like(t), t * 0.5) for t in tau_list]
    nll_loss = torch.nn.GaussianNLLLoss(reduction='sum')

    def log_prob_func(params, *args):
        l_prior = torch.zeros_like(params[0], requires_grad=True)
        i_prev = 0
        for index, shape, dist in zip(params_flattened_list, params_shape_list, dist_list):
            l_prior = dist.log_prob(params[i_prev:index + i_prev]).sum() + l_prior
            i_prev += index
        x1, x2, y = tr_data
        output = fmodel(x1, x2, parameters=params).squeeze(1)
        if model_loss == 'NLL':
            ll = - nll_loss(output, y, tau_out * torch.ones_like(output))
        else:
            raise NotImplementedError()
        return ll + l_prior

    return log_prob_func
