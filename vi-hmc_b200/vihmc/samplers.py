"""Drop-in for the sampler surface the reference uses (``hamiltorch.samplers`` + ``hamiltorch.sample_model``
+ the reference's own ``define_model_log_prob`` factories), backed by the CUDA engine.

Reference call sites mirrored here (argument names and meaning kept):
  samplers.sample(log_prob_func, params_init, num_samples, num_steps_per_sample, step_size, burn, sampler,
                  integrator, debug)              Neural_network/VI_HMC/main_VI_HMC.py:379-380
                                                  Operator_network/VI_HMC/main_VI_HMC_burgers.py:286-287
                                                  Operator_network/HMC/main_HMC_splitting.py:362-369
                                                  Operator_network/HMC/NUTS_DeepOnets.py:289-290
  hamiltorch.sample_model(model, x, y, params_init, model_loss, num_samples, num_steps_per_sample, step_size,
                          tau_out, tau_list, normalizing_const, debug)
                                                  Neural_network/HMC/main_regression_hmc.py:124-127
  define_model_log_prob(...)                      main_VI_HMC.py:28-29, main_VI_HMC_burgers.py:27-28,
                                                  main_HMC_splitting.py:79 and :209-210 (split)

What changes at this boundary: ``log_prob_func`` is a :class:`vihmc.spec.LogProbSpec` (or a list of them
for ``Integrator.SPLITTING``) -- either built by the factories below, or recovered from one of the reference's own
closures by ``vihmc.closure.spec_from_closure`` (so the reference's drivers run unmodified through the ``hamiltorch``
drop-in package) and checked once against that closure at ``params_init``.  New optional keywords: ``num_chains``
(params_init may also be ``[C, d]``), ``seed``, ``chain_offset``, ``return_result``.  hamiltorch's ``inv_mass`` is supported
in its 1-D (diagonal) form.  With one chain the
return value is hamiltorch's list of ``num_samples - burn`` 1-D tensors (so ``np.save`` writes the same
``(S, d)`` array); with C chains it is a ``[S - burn, C, d]`` tensor.
"""
from __future__ import annotations

from typing import List, Optional, Sequence, Union

import numpy as np
import torch

from . import closure, engine
from .spec import DeepONetArch, LogProbSpec, MLPArch, sliced_prior_sigma


class Sampler:
    HMC = 1
    RMHMC = 2
    HMC_NUTS = 3


class Integrator:
    EXPLICIT = 1
    IMPLICIT = 2
    S3 = 3
    SPLITTING = 4
    SPLITTING_RAND = 5
    SPLITTING_KMID = 6


class Metric:
    HESSIAN = 1
    SOFTABS = 2
    JACOBIAN_DIAG = 3


def _initial_states(spec: LogProbSpec, params_init: torch.Tensor, num_chains: Optional[int], seed: int) -> torch.Tensor:
    """[C,d] start points.  A 1-D params_init is replicated; hamiltorch semantics are one chain."""
    q = params_init.detach().to(torch.float32).cpu()
    if q.dim() == 1:
        q = q.unsqueeze(0).repeat(1 if num_chains is None else int(num_chains), 1)
    elif q.dim() != 2:
        raise RuntimeError("params_init must be a 1d tensor.")
    if num_chains is not None and q.shape[0] != num_chains:
        raise ValueError(f"params_init has {q.shape[0]} rows but num_chains={num_chains}")
    if q.shape[1] != spec.d:
        raise ValueError(f"params_init has {q.shape[1]} entries per chain, the log-posterior samples d={spec.d}")
    return q


def check_inv_mass(inv_mass, d: int) -> Optional[torch.Tensor]:
    """hamiltorch's ``inv_mass`` as the engine takes it: None, or a 1-D length-d array of finite, positive entries (a diagonal
    inverse mass shared by all chains), returned as a CPU fp32 tensor.  Checked on the host so that nothing reaches the GPU
    with a mass the kernels cannot use; the dense (2-D) and block-list forms are not implemented."""
    if inv_mass is None:
        return None
    if isinstance(inv_mass, (list, tuple)):
        raise NotImplementedError("inv_mass as a list of blocks is not implemented; pass the diagonal as a 1-D tensor of length d")
    m = inv_mass.detach().cpu() if isinstance(inv_mass, torch.Tensor) else torch.as_tensor(np.asarray(inv_mass))
    if m.dim() == 2:
        raise NotImplementedError("a dense (2-D) inv_mass is not implemented; pass the diagonal as a 1-D tensor of length d")
    if m.dim() != 1 or m.shape[0] != d:
        raise ValueError(f"inv_mass must be a 1-D tensor of length d={d}, got shape {tuple(m.shape)}")
    m = m.to(torch.float32)
    if not bool(torch.isfinite(m).all()) or not bool((m > 0).all()):
        raise ValueError("inv_mass entries must be finite and > 0")
    return m.contiguous()


def sample(log_prob_func, params_init, num_samples=10, num_steps_per_sample=10, step_size=0.1, burn=0, jitter=None,
           inv_mass=None, normalizing_const=1., softabs_const=None, explicit_binding_const=100,
           fixed_point_threshold=1e-5, fixed_point_max_iterations=1000, jitter_max_tries=10, sampler=Sampler.HMC,
           integrator=Integrator.IMPLICIT, metric=Metric.HESSIAN, debug=False, desired_accept_rate=0.8,
           store_on_GPU=True, pass_grad=None, verbose=False, *, num_chains: Optional[int] = None, seed: int = 0,
           chain_offset: int = 0, return_result: bool = False, inject_momenta=None, inject_uniforms=None,
           hamiltorch_fallback_rule: bool = True, verify_closures: bool = True, vi_redraw: bool = False,
           vi_params_uid: Optional[str] = None, inject_vi_normals=None):
    """hamiltorch.samplers.sample on the CUDA engine (see module docstring).

    vi_redraw=True runs the reference's per-sample VI redraw -- what a sampler does that calls ``log_prob_func(params, True)`` once
    per sample (main_VI_HMC.py:96-99 -> my_make_func.py:45-50 ``sample_weights``): every frozen weight is redrawn from its
    variational N(mu, sigma) at the start of each iteration; with ``vi_params_uid`` the draws are written to
    ``vi_params_<uid>.npy`` as the hook does ([num_samples, D] for one chain, [num_samples, C, D] for C chains).

    inv_mass: hamiltorch's diagonal inverse mass, a 1-D tensor or array of length d with finite, positive entries, shared by
    all chains (``check_inv_mass``).  ``params_std[grad_ind] ** 2`` from the VI fit is the natural choice for VI-HMC; the
    step size must then be re-tuned (``Sampler.HMC_NUTS`` does).  Injected momenta are used as given, i.e. already scaled."""
    if sampler == Sampler.RMHMC:
        raise NotImplementedError("RMHMC is not used by the reference and is not on the accelerated path")
    specs = list(log_prob_func) if isinstance(log_prob_func, (list, tuple)) else [log_prob_func]
    closures = {}
    for i, s in enumerate(specs):
        if isinstance(s, (LogProbSpec, engine.Prepared)):
            continue
        if not callable(s):
            raise TypeError("log_prob_func must be a LogProbSpec (vihmc's define_model_log_prob) or one of the reference's "
                            "own log_prob_func closures")
        # one of the reference's closures: read the captured data, prior, likelihood and VI split back out of it
        # (vihmc/closure.py) -- a CUDA engine cannot call Python per leapfrog step, and does not need to
        closures[i] = s
        specs[i] = closure.spec_from_closure(s)
    if integrator in (Integrator.SPLITTING, Integrator.SPLITTING_RAND, Integrator.SPLITTING_KMID):
        if integrator != Integrator.SPLITTING:
            raise NotImplementedError("only Integrator.SPLITTING (the reference's choice) is implemented")
        if len(specs) < 2:
            raise NotImplementedError("splitting needs a list of at least two log-posteriors")
        integ = engine.INTEGRATOR_SPLITTING
    else:
        if len(specs) != 1:
            raise ValueError("a list of log-posteriors requires integrator=Integrator.SPLITTING")
        integ = engine.INTEGRATOR_LEAPFROG
    if burn >= num_samples:
        raise RuntimeError("burn must be less than num_samples.")
    nuts = sampler == Sampler.HMC_NUTS
    if nuts and burn == 0:
        raise RuntimeError("burn must be greater than 0 for NUTS.")
    spec0 = specs[0].spec if isinstance(specs[0], engine.Prepared) else specs[0]
    inv_mass = check_inv_mass(inv_mass, spec0.d)
    single = isinstance(params_init, torch.Tensor) and params_init.dim() == 1 and num_chains in (None, 1)
    q0 = _initial_states(spec0, params_init, num_chains, seed)
    if closures and verify_closures:
        # set-up check, once per closure: the closure's own value and autograd gradient at the first chain's start point
        # must match the engine's for the recovered specification (raises closure.ClosureError otherwise)
        for i, fn in closures.items():
            recovered = specs[i]
            specs[i] = engine.prepare(recovered)
            closure.verify_closure(fn, recovered, q0[0], prepared=specs[i])
    if spec0.trunk_subsample is not None:
        # cfg.sample_data: every closure call redraws its trunk points; composed on the host from the exported building blocks
        if len(specs) != 1 or nuts:
            raise NotImplementedError("trunk sub-sampling (cfg.sample_data) is implemented for plain HMC with one log-posterior")
        res = engine.run_sampler_trunk_subsample(specs[0], q0, num_samples, num_steps_per_sample, float(step_size), burn=burn, seed=seed,
                                                 chain_offset=chain_offset, inject_momenta=inject_momenta,
                                                 inject_uniforms=inject_uniforms, to_host=True, inv_mass=inv_mass)
        if verbose or debug:
            print("Acceptance Rate {:.2f}".format(res.acceptance_rate))
        if return_result:
            return res
        return list(res.samples[:, 0, :].unbind(0)) if single else res.samples
    res = engine.run_sampler(specs, q0, num_samples, num_steps_per_sample, float(step_size), burn=burn, integrator=integ,
                             adapt_step_size=nuts, desired_accept_rate=desired_accept_rate, seed=seed,
                             chain_offset=chain_offset, hamiltorch_fallback_rule=hamiltorch_fallback_rule,
                             inject_momenta=inject_momenta, inject_uniforms=inject_uniforms, to_host=True, vi_redraw=vi_redraw,
                             inject_vi_normals=inject_vi_normals, inv_mass=inv_mass)
    if vi_redraw and vi_params_uid is not None:
        vp = res.vi_params[:, 0] if single else res.vi_params
        np.save(f"vi_params_{vi_params_uid}.npy", vp.clone().detach().cpu())
    if verbose or debug:
        print("Acceptance Rate {:.2f}".format(res.acceptance_rate))
    if return_result:
        return res
    if single:
        out = list(res.samples[:, 0, :].unbind(0))
        if nuts and debug == 2:
            return out, float(res.step_sizes[0])
        if debug == 2:
            return out, res.acceptance_rate
        return out
    return res.samples


# ------------------------------------------------------------------------------------------------
# log-posterior factories with the reference's signatures
# ------------------------------------------------------------------------------------------------


def define_model_log_prob_bnn(model, model_loss, x, y, params_flattened_list, params_shape_list, prior_list, tau_out,
                              predict=False, prior_scale=1.0, device='cpu', dt_string=None, grad_ind=None, *,
                              params_mu=None, params_std=None, load_prior=False) -> LogProbSpec:
    """Neural_network/VI_HMC/main_VI_HMC.py:28-153.

    The reference reads the VI artefacts from ``cfg.prior_file`` inside the factory (:76-79); here they are
    passed in (``params_mu``, ``params_std``, ``grad_ind``).  ``params_mu is None`` gives plain HMC over all
    parameters (my_make_func.py:53-54).  ``load_prior`` selects prior_list = [mu[ind], sigma[ind]] (:87-88,104-105).
    """
    arch = MLPArch.from_module(model) if isinstance(model, torch.nn.Module) else model
    if params_mu is not None and grad_ind is None:
        raise ValueError("grad_ind (gradient_indices_<uid>.npy) is required with VI means")
    d = arch.num_params if params_mu is None else len(grad_ind)
    if load_prior:
        prior_mu, prior_sigma = prior_list[0].detach().float(), prior_list[1].detach().float()
    else:
        vars_ = [float(t) for t in prior_list]
        sig = sliced_prior_sigma(d, list(params_flattened_list), vars_)
        prior_mu, prior_sigma = None, torch.from_numpy(sig.astype(np.float32))
    return LogProbSpec(arch=arch, x=x.detach().float().cpu(), y=y.detach().float().cpu(), loss=model_loss,
                       tau_out=float(tau_out), prior_mu=prior_mu, prior_sigma=prior_sigma, prior_scale=float(prior_scale),
                       frozen=None if params_mu is None else params_mu.detach().float().cpu(),
                       sens_ind=None if params_mu is None else np.asarray(grad_ind, dtype=np.int64),
                       vi_sigma=None if params_std is None else params_std.detach().float().cpu(), predict=predict)


def define_model_log_prob_hamiltorch(model, model_loss, x, y, params_flattened_list, params_shape_list, tau_list, tau_out,
                                     normalizing_const=1., predict=False, prior_scale=1.0, device='cpu') -> LogProbSpec:
    """hamiltorch's own factory (used by sample_model): Gaussian prior N(0, tau^-1/2) per parameter tensor,
    'regression' likelihood -0.5*tau_out*sum((o-y)^2); normalizing_const is accepted and unused, as upstream."""
    arch = MLPArch.from_module(model) if isinstance(model, torch.nn.Module) else model
    sig = np.concatenate([np.full(n, float(t) ** -0.5) for n, t in zip(params_flattened_list, tau_list)])
    return LogProbSpec(arch=arch, x=x.detach().float().cpu(), y=y.detach().float().cpu(), loss=model_loss,
                       tau_out=float(tau_out), prior_sigma=torch.from_numpy(sig.astype(np.float32)),
                       prior_scale=float(prior_scale), predict=predict)


def define_model_log_prob_deeponet(model, model_loss, tr_data, tau_list, tau_out, predict=False, prior_scale=1.0,
                                   device='cpu', *, mean_params=None, std_params=None, grad_ind=None, load_prior=False,
                                   sample_data=False, p=None) -> LogProbSpec:
    """Operator_network/VI_HMC/main_VI_HMC_burgers.py:27-180 and Operator_network/HMC/main_HMC_splitting.py:79-206.

    tr_data = (x1 [N,1,in_branch], x2 [1,P,2], y [N,P]) as util.get_burgers_data returns (util.py:461-473).
    Prior: N(0, sqrt(tau_list[0])) over the sampled vector (:96-102), or N(tau_list[0], tau_list[1]) if load_prior.
    """
    arch = DeepONetArch.from_module(model) if isinstance(model, torch.nn.Module) else model
    x1, x2, y = tr_data
    x1 = x1.detach().float().cpu().reshape(x1.shape[0], -1)
    x2 = x2.detach().float().cpu().reshape(-1, x2.shape[-1])
    if load_prior:
        prior_mu, prior_sigma, scal = tau_list[0].detach().float(), tau_list[1].detach().float(), 1.0
    else:
        prior_mu, prior_sigma, scal = None, None, float(tau_list[0]) ** 0.5
    return LogProbSpec(arch=arch, x=x1, x2=x2, y=y.detach().float().cpu(), loss=model_loss, tau_out=float(tau_out),
                       prior_mu=prior_mu, prior_sigma=prior_sigma, prior_sigma_scalar=scal, prior_scale=float(prior_scale),
                       frozen=None if mean_params is None else mean_params.detach().float().cpu(),
                       sens_ind=None if mean_params is None else np.asarray(grad_ind, dtype=np.int64),
                       vi_sigma=None if std_params is None else std_params.detach().float().cpu(), predict=predict,
                       trunk_subsample=int(p) if (sample_data and not predict) else None)   # cfg.sample_data / cfg.p, :127-137


def define_split_model_log_prob(model, model_loss, train_loader, num_splits, tau_list, tau_out, predict=False,
                                device='cpu', verbose=True, **kw) -> List[LogProbSpec]:
    """main_HMC_splitting.py:209-258: one log-posterior per data block, each with prior_scale = num_splits."""
    out = []
    for batch_idx, data in enumerate(train_loader):
        if batch_idx > num_splits - 1:
            break
        out.append(define_model_log_prob_deeponet(model, model_loss, data, tau_list, tau_out, prior_scale=num_splits,
                                                  predict=predict, device=device, **kw))
    if verbose:
        print('Number of splits: ', len(out), ' , each of batch size ', train_loader[0][0].shape[0], '\n')
    return out


def sample_model(model, x, y, params_init, model_loss='multi_class_linear_output', num_samples=10,
                 num_steps_per_sample=10, step_size=0.1, burn=0, inv_mass=None, jitter=None, normalizing_const=1.,
                 softabs_const=None, explicit_binding_const=100, fixed_point_threshold=1e-5,
                 fixed_point_max_iterations=1000, jitter_max_tries=10, sampler=Sampler.HMC, integrator=Integrator.IMPLICIT,
                 metric=Metric.HESSIAN, debug=False, tau_out=1., tau_list=None, store_on_GPU=True,
                 desired_accept_rate=0.8, verbose=False, **engine_kw):
    """hamiltorch.sample_model as called at Neural_network/HMC/main_regression_hmc.py:124-127 (``inv_mass``: as in ``sample``)."""
    numels = [w.nelement() for w in model.parameters()]
    shapes = [w.shape for w in model.parameters()]
    if tau_list is None:
        tau_list = [torch.tensor(1.) for _ in numels]
    spec = define_model_log_prob_hamiltorch(model, model_loss, x, y, numels, shapes, tau_list, tau_out,
                                            normalizing_const=normalizing_const)
    return sample(spec, params_init, num_samples=num_samples, num_steps_per_sample=num_steps_per_sample,
                  step_size=step_size, burn=burn, inv_mass=inv_mass, sampler=sampler, integrator=integrator, debug=debug,
                  desired_accept_rate=desired_accept_rate, verbose=verbose, **engine_kw)


def predict_model(spec: LogProbSpec, samples, x=None, y=None, data=None):
    """hamiltorch.predict_model / the reference's predict_model (main_VI_HMC.py:156-259,
    main_VI_HMC_burgers.py:183-241): model outputs and log-probability for every sample on validation data.

    samples: list of [d] tensors or a [S,d] tensor.  Returns (pred [S,N,O], list of S log-probabilities)."""
    import dataclasses

    q = torch.stack(list(samples)) if isinstance(samples, (list, tuple)) else samples
    q = q.reshape(-1, spec.d).float()
    if data is not None:
        x1, x2, yv = data
        vspec = dataclasses.replace(spec, x=x1.reshape(x1.shape[0], -1).float().cpu(),
                                    x2=x2.reshape(-1, x2.shape[-1]).float().cpu(), y=yv.float().cpu())
    elif x is not None and y is not None:
        vspec = dataclasses.replace(spec, x=x.float().cpu(), y=y.float().cpu())
    else:
        raise RuntimeError('Val data not defined (i.e. arguments x, y, val_loader are all not defined)')
    prep = engine.prepare(vspec)
    pred = engine.predict(prep, q)
    logp, _ = engine.logp_grad(prep, q, need_grad=False)
    pred = pred.cpu()
    if vspec.model_kind == 0:
        pred = pred.unsqueeze(-1)
    return pred, list(logp.cpu().unbind(0))
