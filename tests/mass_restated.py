"""Restated hamiltorch ``inv_mass`` (a diagonal mass matrix) on top of the identity-mass restatement.

PARITY UNPINNED, like oracle/hamiltorch_restated.py: hamiltorch is not on disk, so its 1-D ``inv_mass`` handling is restated from
its published code, and this restatement is the specification the engine's diagonal-mass paths are tested against.  With
m = inv_mass (one [d] vector shared by all chains) and every operation a separately rounded op in the working dtype:

  mass      hamiltorch ``mass = 1 / inv_mass``                 s_i = sqrt(fl(1 / m_i))
  momentum  ``Normal(0, mass ** 0.5).sample()``                p_i = fl(z_i s_i)
  kinetic   ``0.5 * dot(p, inv_mass * p)``                      0.5 sum_i p_i fl(m_i p_i)
  drift     ``params + step_size * inv_mass * momentum``        q_i = fl(q_i + fl(fl(eps m_i) p_i))
  kick      unchanged

The split integrator drifts with eps / (2 (M - 1)) in place of eps; dual averaging is unchanged.  Injected momenta are used as
p verbatim (already scaled).  With m = 1 every row is exact, so ``inv_mass=None`` and ``inv_mass=ones(d)`` give the same bits;
with ``inv_mass=None`` every function here defers to the pinned identity restatement itself.

``sample`` repeats the bookkeeping of ``oracle.hamiltorch_restated.sample`` (accept/reject, storage rule, dual averaging) line for
line around the three mass-dependent operations above.  ``sample_batched`` is the fp64 many-chain twin for
``oracle.bnn_batched.BatchedBnn``.
"""
from __future__ import annotations

from typing import List, Optional

import numpy as np
import torch

from oracle import hamiltorch_restated as hr


def momentum_scale(inv_mass: torch.Tensor) -> torch.Tensor:
    return (1 / inv_mass) ** 0.5


def gibbs(q: torch.Tensor, inv_mass: Optional[torch.Tensor] = None, generator: Optional[torch.Generator] = None) -> torch.Tensor:
    if inv_mass is None:
        return hr.gibbs(q, generator)
    if generator is None:
        return torch.distributions.Normal(torch.zeros_like(q), momentum_scale(inv_mass)).sample()
    return torch.randn(q.shape, dtype=q.dtype, generator=generator) * momentum_scale(inv_mass)


def hamiltonian(q: torch.Tensor, p: torch.Tensor, log_prob_func, inv_mass: Optional[torch.Tensor] = None) -> torch.Tensor:
    if inv_mass is None:
        return hr.hamiltonian(q, p, log_prob_func)
    with torch.no_grad():
        # -logp from the identity restatement (same LogProbError rule), then the m-weighted kinetic term
        neg_lp = hr.hamiltonian(q, torch.zeros_like(p), log_prob_func)
        return neg_lp + 0.5 * torch.dot(p, inv_mass * p)


def leapfrog(q: torch.Tensor, p: torch.Tensor, log_prob_func, steps: int, step_size: float, integrator: int = hr.Integrator.IMPLICIT,
             inv_mass: Optional[torch.Tensor] = None):
    if inv_mass is None:
        return hr.leapfrog(q, p, log_prob_func, steps, step_size, integrator)
    q = q.detach().clone()
    p = p.clone()
    if integrator != hr.Integrator.SPLITTING:
        g = hr.params_grad(log_prob_func, q)
        p += 0.5 * step_size * g
        for _ in range(steps):
            q = q + (step_size * inv_mass) * p
            g = hr.params_grad(log_prob_func, q)
            p += step_size * g
        p = p - 0.5 * step_size * g
        return q, p
    M = len(log_prob_func)
    if M == 1:
        raise NotImplementedError("splitting needs at least two closures")
    frac = step_size / ((M - 1) * 2)
    for _ in range(steps):
        for m in range(M):
            g = hr.params_grad(log_prob_func[m], q)
            p += 0.5 * step_size * g
            if m < M - 1:
                q += (frac * inv_mass) * p
        for m in reversed(range(M)):
            g = hr.params_grad(log_prob_func[m], q)
            p += 0.5 * step_size * g
            if m > 0:
                q += (frac * inv_mass) * p
    return q, p


def sample(log_prob_func, params_init: torch.Tensor, num_samples: int = 10, num_steps_per_sample: int = 10, step_size: float = 0.1,
           burn: int = 0, sampler: int = hr.Sampler.HMC, integrator: int = hr.Integrator.IMPLICIT, desired_accept_rate: float = 0.8,
           momenta: Optional[torch.Tensor] = None, uniforms: Optional[torch.Tensor] = None,
           generator: Optional[torch.Generator] = None, trace: Optional[dict] = None,
           inv_mass: Optional[torch.Tensor] = None) -> List[torch.Tensor]:
    """``hamiltorch_restated.sample`` with hamiltorch's 1-D ``inv_mass``; ``inv_mass=None`` calls the pinned restatement itself.
    The iteration below is that function's, line for line, with gibbs / hamiltonian / leapfrog taking the mass."""
    if inv_mass is None:
        return hr.sample(log_prob_func, params_init, num_samples, num_steps_per_sample, step_size, burn, sampler, integrator,
                         desired_accept_rate, momenta=momenta, uniforms=uniforms, generator=generator, trace=trace)
    m = torch.as_tensor(inv_mass, dtype=params_init.dtype)
    if params_init.dim() != 1:
        raise RuntimeError("params_init must be a 1d tensor.")
    if burn >= num_samples:
        raise RuntimeError("burn must be less than num_samples.")
    nuts = False
    if sampler == hr.Sampler.HMC_NUTS:
        if burn == 0:
            raise RuntimeError("burn must be greater than 0 for NUTS.")
        nuts, step_size_init, H_t, eps_bar = True, step_size, 0.0, 1.0
    params = params_init.clone()
    param_burn_prev = params_init.clone()
    ret_params = [params.clone()]
    num_rejected = 0
    if trace is not None:
        for k in ("H0", "H1", "accept", "step_size"):
            trace.setdefault(k, [])
    for n in range(num_samples):
        rho = float("nan")
        h0 = h1 = float("nan")
        accepted = False
        if trace is not None:
            trace["step_size"].append(step_size)
        try:
            momentum = momenta[n].clone() if momenta is not None else gibbs(params, m, generator)
            ham = hamiltonian(params, momentum, log_prob_func, m)
            h0 = float(ham)
            q_new, p_new = leapfrog(params, momentum, log_prob_func, num_steps_per_sample, step_size, integrator, m)
            new_ham = hamiltonian(q_new, p_new, log_prob_func, m)
            h1 = float(new_ham)
            rho = min(0.0, float(-new_ham + ham))
            if uniforms is not None:
                log_u = torch.log(uniforms[n].reshape(1).to(torch.float32))
            elif generator is not None:
                log_u = torch.log(torch.rand(1, generator=generator))
            else:
                log_u = torch.log(torch.rand(1))
            if bool(rho >= log_u):
                accepted = True
                params = q_new
                if n > burn:
                    ret_params.append(q_new.clone())
                else:
                    param_burn_prev = q_new.clone()
            else:
                num_rejected += 1
                if n > burn:
                    params = ret_params[-1].clone()
                    ret_params.append(ret_params[-1].clone())
                else:
                    params = param_burn_prev.clone()
            if nuts and n <= burn:
                if n < burn:
                    step_size, eps_bar, H_t = hr.adaptation(rho, n, step_size_init, H_t, eps_bar, desired_accept_rate)
                if n == burn:
                    step_size = eps_bar
        except hr.LogProbError:
            num_rejected += 1
            if n > burn:
                params = ret_params[-1].clone()
                ret_params.append(ret_params[-1].clone())
            else:
                params = param_burn_prev.clone()
            if nuts and n <= burn:
                step_size, eps_bar, H_t = hr.adaptation(float("nan"), n, step_size_init, H_t, eps_bar, desired_accept_rate)
            if nuts and n == burn:
                step_size = eps_bar
        if trace is not None:
            trace["H0"].append(h0)
            trace["H1"].append(h1)
            trace["accept"].append(accepted)
    if trace is not None:
        trace["acceptance_rate"] = 1 - num_rejected / num_samples
        trace["final_step_size"] = step_size
    return [t.detach() for t in ret_params]


def sample_batched(model, q0, num_samples, num_steps, step_size, inv_mass, momenta=None, uniforms=None, rng=None):
    """``oracle.bnn_batched.sample`` with a diagonal mass, numpy fp64, all chains at once: final states, decisions [S, C] and
    (H0, H1) [S, C, 2].  ``momenta`` are used as p verbatim; drawn ones are N(0, 1 / inv_mass)."""
    m = np.asarray(inv_mass, np.float64)
    q = np.array(q0, np.float64)
    C, d = q.shape
    acc = np.zeros((num_samples, C), bool)
    ham = np.zeros((num_samples, C, 2))
    for n in range(num_samples):
        p = np.asarray(momenta[n], np.float64) if momenta is not None else rng.standard_normal((C, d)) * np.sqrt(1.0 / m)
        lp0, g = model.logp_grad(q)
        H0 = -lp0 + 0.5 * (p * (m * p)).sum(1)
        qn = q.copy()
        p = p + 0.5 * step_size * g
        for _ in range(num_steps):
            qn = qn + (step_size * m) * p
            lp1, g = model.logp_grad(qn)
            p = p + step_size * g
        p = p - 0.5 * step_size * g
        H1 = -lp1 + 0.5 * (p * (m * p)).sum(1)
        u = np.asarray(uniforms[n], np.float64) if uniforms is not None else rng.random(C)
        a = np.isfinite(H1) & (np.minimum(0.0, H0 - H1) >= np.log(u))
        q[a] = qn[a]
        acc[n], ham[n, :, 0], ham[n, :, 1] = a, H0, H1
    return q, acc, ham
