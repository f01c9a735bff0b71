"""Device plumbing between LogProbSpec (host description) and the C ABI (libvihmc.so).

torch is used for device memory, streams and host<->device copies only; all arithmetic happens in
the CUDA library.  Every entry point raises if CUDA or the library is unavailable.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import List, Optional, Sequence, Union

import numpy as np
import torch

from . import _lib
from .spec import (LogProbSpec, MLPArch, DeepONetArch, MODEL_DEEPONET, MODEL_MLP, act_code, loss_code)

INTEGRATOR_LEAPFROG, INTEGRATOR_SPLITTING = 0, 1


def _require_cuda(device=None) -> torch.device:
    if not torch.cuda.is_available():
        raise _lib.VihmcError(-2, "no CUDA device: the vihmc engine has no CPU fallback")
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    if dev.type != "cuda":
        raise _lib.VihmcError(-2, f"device {dev} is not a CUDA device: the vihmc engine has no CPU fallback")
    return dev


def _to_dev(t, dev, dtype=torch.float32) -> Optional[torch.Tensor]:
    """Host tensors are staged through pinned memory so the H2D copy is a real async DMA."""
    if t is None:
        return None
    if isinstance(t, np.ndarray):
        t = torch.from_numpy(np.ascontiguousarray(t))
    t = t.detach()
    if t.device.type == "cuda":
        return t.to(device=dev, dtype=dtype).contiguous()
    t = t.to(dtype).contiguous()
    try:
        t = t.pin_memory()
    except RuntimeError:
        pass
    return t.to(dev, non_blocking=True)


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


class Prepared:
    """A LogProbSpec resident on one GPU + its vihmc_problem struct (keeps the tensors alive)."""

    def __init__(self, spec: LogProbSpec, device=None):
        spec.validate()
        self.spec = spec
        self.device = _require_cuda(device)
        dev = self.device
        arch = spec.arch
        p = _lib.Problem()
        p.model_kind = spec.model_kind
        p.act = act_code(arch.act)
        p.loss = loss_code(spec.loss)
        if isinstance(arch, MLPArch):
            dims = [o for o, _ in arch.layer_dims]
            if len(dims) > _lib.MAX_LAYERS:
                raise ValueError("too many layers")
            p.last_bias, p.impose_bc = int(arch.last_bias), 0
            p.n_layers_a, p.n_layers_b, p.in_a, p.in_b = len(dims), 0, arch.in_dim, 0
            for i, w in enumerate(dims):
                p.dims_a[i] = w
            x = spec.x.reshape(spec.N, arch.in_dim)
            y = spec.y.reshape(spec.N, arch.out_dim)
            p.P = 1
        else:
            da = [o for o, _ in arch.stack_dims("branch")]
            db = [o for o, _ in arch.stack_dims("trunk")]
            p.last_bias, p.impose_bc = 1, int(arch.impose_bc)
            p.n_layers_a, p.n_layers_b, p.in_a, p.in_b = len(da), len(db), arch.in_branch, arch.in_trunk
            for i, w in enumerate(da):
                p.dims_a[i] = w
            for i, w in enumerate(db):
                p.dims_b[i] = w
            x = spec.x.reshape(spec.N, arch.in_branch)
            y = spec.y.reshape(spec.N, -1)
            p.P = y.shape[1]
        p.D, p.d, p.N = spec.D, spec.d, spec.N
        p.tau_out, p.prior_scale, p.prior_sigma_scalar = float(spec.tau_out), float(spec.prior_scale), float(spec.prior_sigma_scalar)
        sig_host = None if spec.prior_sigma is None else spec.prior_sigma.detach().cpu().to(torch.float32).contiguous()
        lib = _lib.load()
        p.prior_log_norm = lib.vihmc_prior_log_norm(None if sig_host is None else sig_host.data_ptr(), spec.d,
                                                    float(spec.prior_sigma_scalar))
        self.x = _to_dev(x, dev)
        self.y = _to_dev(y, dev)
        self.x2 = _to_dev(None if spec.x2 is None else spec.x2.reshape(-1, spec.x2.shape[-1]), dev)
        self.frozen = _to_dev(spec.frozen, dev)
        self.sens_ind = _to_dev(None if spec.sens_ind is None else np.asarray(spec.sens_ind, dtype=np.int64), dev, torch.int64)
        self.prior_mu = _to_dev(spec.prior_mu, dev)
        self.prior_sigma = _to_dev(spec.prior_sigma, dev)
        p.x, p.x2, p.y = _ptr(self.x), _ptr(self.x2), _ptr(self.y)
        p.frozen, p.sens_ind = _ptr(self.frozen), _ptr(self.sens_ind)
        p.prior_mu, p.prior_sigma = _ptr(self.prior_mu), _ptr(self.prior_sigma)
        self.problem = p
        self._ws: Optional[torch.Tensor] = None

    @property
    def h2d_bytes(self) -> int:
        ts = (self.x, self.y, self.x2, self.frozen, self.sens_ind, self.prior_mu, self.prior_sigma)
        return sum(t.numel() * t.element_size() for t in ts if t is not None)

    def workspace(self, chains: int) -> torch.Tensor:
        need = int(_lib.load().vihmc_workspace_bytes(C.byref(self.problem), chains))
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(max(need, 256), dtype=torch.uint8, device=self.device)
        return self._ws


def prepare(spec: Union[LogProbSpec, Prepared], device=None) -> Prepared:
    return spec if isinstance(spec, Prepared) else Prepared(spec, device)


def _stream(dev) -> int:
    return torch.cuda.current_stream(dev).cuda_stream


def logp_grad(spec, q: torch.Tensor, need_grad: bool = True):
    """log-posterior [C] and gradient [C,d] for C parameter vectors q[C,d] (device tensors returned)."""
    prep = prepare(spec)
    dev = prep.device
    q2 = _to_dev(q.reshape(-1, prep.spec.d), dev)
    Cn = q2.shape[0]
    logp = torch.empty(Cn, dtype=torch.float32, device=dev)
    grad = torch.empty_like(q2) if need_grad else None
    ws = prep.workspace(Cn)
    with torch.cuda.device(dev):
        _lib.check(_lib.load().vihmc_logp_grad(C.byref(prep.problem), Cn, q2.data_ptr(), logp.data_ptr(), _ptr(grad),
                                               ws.data_ptr(), ws.numel(), _stream(dev)))
    return logp, grad


def predict(spec, q: torch.Tensor) -> torch.Tensor:
    """Model outputs for C parameter vectors: [C,N] (MLP) or [C,N,P] (DeepONet)."""
    prep = prepare(spec)
    dev = prep.device
    q2 = _to_dev(q.reshape(-1, prep.spec.d), dev)
    Cn = q2.shape[0]
    shape = (Cn, prep.spec.N) if prep.spec.model_kind == MODEL_MLP else (Cn, prep.spec.N, int(prep.problem.P))
    out = torch.empty(shape, dtype=torch.float32, device=dev)
    ws = prep.workspace(Cn)
    with torch.cuda.device(dev):
        _lib.check(_lib.load().vihmc_predict(C.byref(prep.problem), Cn, q2.data_ptr(), out.data_ptr(), ws.data_ptr(),
                                             ws.numel(), _stream(dev)))
    return out


def gemm_batched(A: torch.Tensor, B: torch.Tensor, tensor_cores: bool = True) -> torch.Tensor:
    """C[b] = A[b] @ B[b] through vihmc_gemm_batched.  A [batch, M, K] and B [batch, K, N] are CUDA fp32 tensors or
    strided VIEWS of them (e.g. `.transpose(1, 2)`, `.expand(batch, -1, -1)`): the element strides are passed as
    they are, which is how the tests reach every operand staging mode of the tensor-core kernel."""
    assert A.is_cuda and B.is_cuda and A.dtype == torch.float32 and B.dtype == torch.float32
    batch, M, K = A.shape
    _, _, N = B.shape
    dev = A.device
    out = torch.empty(batch, M, N, dtype=torch.float32, device=dev)
    scratch = None
    if tensor_cores and K > 2048:
        scratch = torch.empty(((K + 1023) // 1024) * batch * M * N, dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(_lib.load().vihmc_gemm_batched(A.data_ptr(), A.stride(0), A.stride(1), A.stride(2), B.data_ptr(), B.stride(0),
                                                  B.stride(1), B.stride(2), out.data_ptr(), M * N, N, M, N, K, batch,
                                                  1 if tensor_cores else 0, _ptr(scratch), _stream(dev)))
    return out


@dataclass
class SampleResult:
    samples: torch.Tensor                  # [num_samples - burn, C, d]; row 0 is params_init
    accepted: Optional[torch.Tensor]       # [num_samples, C] uint8
    hamiltonians: Optional[torch.Tensor]   # [num_samples, C, 2]
    logp: Optional[torch.Tensor]           # [num_samples - burn, C]
    step_sizes: Optional[torch.Tensor]     # [C]
    grad_evals_per_chain: int = 0
    gpu_launches: int = 0
    vi_params: Optional[torch.Tensor] = None   # [num_samples, C, D]: the redrawn weight vectors (vi_redraw=True)

    @property
    def acceptance_rate(self) -> float:
        return float(self.accepted.float().mean()) if self.accepted is not None else float("nan")


def run_sampler(specs: Sequence, q0: torch.Tensor, num_samples: int, num_steps: int, step_size: float, burn: int = 0,
                integrator: int = INTEGRATOR_LEAPFROG, adapt_step_size: bool = False, desired_accept_rate: float = 0.8,
                seed: int = 0, chain_offset: int = 0, hamiltorch_fallback_rule: bool = True, diagnostics: bool = True,
                inject_momenta: Optional[torch.Tensor] = None, inject_uniforms: Optional[torch.Tensor] = None,
                to_host: bool = True, force_general: bool = False, vi_redraw: bool = False,
                inject_vi_normals: Optional[torch.Tensor] = None, inv_mass: Optional[torch.Tensor] = None) -> SampleResult:
    """Advance C = q0.shape[0] chains.  specs: one LogProbSpec/Prepared (leapfrog) or several (splitting).

    inv_mass: hamiltorch's 1-D ``inv_mass`` [d], a diagonal inverse mass shared by all chains (finite, > 0; validated by
    ``samplers.sample``): momenta p = z sqrt(1 / m), kinetic energy 0.5 p.(m p), drift q += eps m p.  Injected momenta are used
    as p verbatim.  None is the identity mass.

    vi_redraw: the reference's ``sample_weights`` hook once per iteration (Neural_network/VI_HMC/my_make_func.py:45-50): all D
    frozen weights of every chain are redrawn from N(mu, sigma) (spec.frozen, spec.vi_sigma; Philox stream 2 or
    ``inject_vi_normals`` [num_samples, C, D]) before the momentum draw; the draws come back as ``vi_params``.

    Inputs may be host tensors (they are copied to the GPU here); with ``to_host`` the result tensors are
    copied back, so one call is a complete host-to-host sampling run.
    """
    preps = [prepare(s) for s in specs]
    dev = preps[0].device
    lib = _lib.load()
    d = preps[0].spec.d
    q0d = _to_dev(q0.reshape(-1, d), dev)
    Cn = q0d.shape[0]
    rows = num_samples - burn
    if rows < 1:
        raise RuntimeError("burn must be less than num_samples.")
    cfg = _lib.SamplerCfg(num_samples=num_samples, num_steps=num_steps, burn=burn, integrator=integrator,
                          adapt_step_size=int(adapt_step_size), hamiltorch_fallback_rule=int(hamiltorch_fallback_rule),
                          step_size=step_size, desired_accept_rate=desired_accept_rate, seed=seed, chain_offset=chain_offset)
    samples = torch.empty((rows, Cn, d), dtype=torch.float32, device=dev)
    io = _lib.SamplerIO()
    acc = ham = lp = eps = None
    if diagnostics:
        acc = torch.empty((num_samples, Cn), dtype=torch.uint8, device=dev)
        ham = torch.empty((num_samples, Cn, 2), dtype=torch.float32, device=dev)
        lp = torch.empty((rows, Cn), dtype=torch.float32, device=dev)
        eps = torch.empty(Cn, dtype=torch.float32, device=dev)
        io.accepted, io.hamiltonians, io.logp, io.step_sizes = acc.data_ptr(), ham.data_ptr(), lp.data_ptr(), eps.data_ptr()
    inj_p = _to_dev(inject_momenta, dev)
    inj_u = _to_dev(inject_uniforms, dev)
    if inj_p is not None:
        assert tuple(inj_p.shape) == (num_samples, Cn, d), inj_p.shape
        io.inject_momenta = inj_p.data_ptr()
    if inj_u is not None:
        assert tuple(inj_u.shape) == (num_samples, Cn), inj_u.shape
        io.inject_uniforms = inj_u.data_ptr()
    minv = _to_dev(inv_mass, dev)
    if minv is not None:
        assert tuple(minv.shape) == (d,), minv.shape
        io.inv_mass = minv.data_ptr()
    vip = vsig = inj_v = None
    if vi_redraw:
        sp0 = preps[0].spec
        if sp0.frozen is None or sp0.vi_sigma is None:
            raise ValueError("vi_redraw needs the VI-HMC split: spec.frozen (means), spec.vi_sigma and spec.sens_ind")
        Dn = sp0.D
        vsig = _to_dev(sp0.vi_sigma, dev)
        vip = torch.empty((num_samples, Cn, Dn), dtype=torch.float32, device=dev)
        io.vi_sigma, io.vi_params = vsig.data_ptr(), vip.data_ptr()
        inj_v = _to_dev(inject_vi_normals, dev)
        if inj_v is not None:
            assert tuple(inj_v.shape) == (num_samples, Cn, Dn), inj_v.shape
            io.inject_vi_normals = inj_v.data_ptr()
    M = len(preps)
    evals = num_samples * (num_steps + 1) if integrator == INTEGRATOR_LEAPFROG else num_samples * num_steps * 2 * M
    launches = 0
    with torch.cuda.device(dev):
        small = (M == 1 and integrator == INTEGRATOR_LEAPFROG and not force_general and preps[0].spec.model_kind == MODEL_MLP)
        rc = None
        if small:
            rc = lib.vihmc_mlp_sample(C.byref(preps[0].problem), C.byref(cfg), Cn, q0d.data_ptr(), samples.data_ptr(),
                                      C.byref(io), _stream(dev))
            if rc == 2:  # VIHMC_ERR_UNSUPPORTED: net too large for the persistent small-MLP kernel
                rc = None
            else:
                launches = 1
        if rc is None:
            probs = (_lib.Problem * M)(*[p.problem for p in preps])
            need = max(int(lib.vihmc_workspace_bytes(C.byref(p.problem), Cn)) for p in preps)
            ws = torch.empty(need, dtype=torch.uint8, device=dev)
            rc = lib.vihmc_sample(probs, M, C.byref(cfg), Cn, q0d.data_ptr(), samples.data_ptr(), C.byref(io), ws.data_ptr(),
                                  ws.numel(), _stream(dev))
            launches = -1  # many; counted by the caller from the launch model if needed
        _lib.check(rc)
    res = SampleResult(samples, acc, ham, lp, eps, grad_evals_per_chain=evals, gpu_launches=launches, vi_params=vip)
    if to_host:
        # device -> pinned host buffers (torch's caching host allocator reuses them across calls), all copies queued on the
        # sampler's stream behind the kernel, one synchronisation at the end
        def host(t):
            if t is None:
                return None
            h = torch.empty(t.shape, dtype=t.dtype, device="cpu", pin_memory=True)
            h.copy_(t, non_blocking=True)
            return h
        with torch.cuda.device(dev):
            res = SampleResult(host(samples), host(acc), host(ham), host(lp), host(eps), evals, launches, host(vip))
            torch.cuda.current_stream(dev).synchronize()
    return res


class _TrunkSubset:
    """The problem of a DeepONet spec restricted to a subset of its trunk points: x2 rows and y columns gathered on the device,
    the other pointers shared with the parent Prepared (main_VI_HMC_burgers.py:127-137)."""

    def __init__(self, prep: Prepared, ind):
        self.parent = prep
        # ind: a device int64 tensor (one row of the per-iteration upload) or a host sequence
        idx = ind if isinstance(ind, torch.Tensor) else torch.as_tensor(np.asarray(ind, dtype=np.int64), device=prep.device)
        self.x2 = prep.x2.index_select(0, idx).contiguous()
        self.y = prep.y.index_select(1, idx).contiguous()
        p = _lib.Problem.from_buffer_copy(prep.problem)
        p.x2, p.y, p.P = self.x2.data_ptr(), self.y.data_ptr(), int(idx.numel())
        self.problem = p

    def logp_grad(self, q: torch.Tensor, need_grad: bool = True):
        prep = self.parent
        dev = prep.device
        Cn = q.shape[0]
        logp = torch.empty(Cn, dtype=torch.float32, device=dev)
        grad = torch.empty_like(q) if need_grad else None
        ws = prep.workspace(Cn)   # sized for the full grid: large enough for any subset
        with torch.cuda.device(dev):
            _lib.check(_lib.load().vihmc_logp_grad(C.byref(self.problem), Cn, q.data_ptr(), logp.data_ptr(), _ptr(grad), ws.data_ptr(),
                                                   ws.numel(), _stream(dev)))
        return logp, grad


def run_sampler_trunk_subsample(spec, q0: torch.Tensor, num_samples: int, num_steps: int, step_size: float, burn: int = 0,
                                seed: int = 0, chain_offset: int = 0, inject_momenta: Optional[torch.Tensor] = None,
                                inject_uniforms: Optional[torch.Tensor] = None, to_host: bool = True,
                                inv_mass: Optional[torch.Tensor] = None) -> SampleResult:
    """HMC for a DeepONet closure with cfg.sample_data: EVERY closure call -- the two Hamiltonians and the L + 1 gradients of an
    iteration, L + 3 calls as hamiltorch makes them -- sees a fresh ``random.sample(range(P), p)`` of the trunk points
    (Operator_network/VI_HMC/main_VI_HMC_burgers.py:127-137).  The subsets come from Python's global ``random`` exactly as in the
    reference (seed it for reproducibility); all chains of the call share them.  The iteration is composed on the host from the
    exported building blocks (vihmc_momentum_philox, vihmc_logp_grad on the gathered problem, vihmc_leapfrog_update,
    vihmc_mh_accept): a DeepONet evaluation is milliseconds of GPU work, so the Python loop only enqueues.  ``inv_mass``: diagonal
    inverse mass [d] as in :func:`run_sampler` (the ``_mass`` building blocks)."""
    import random

    prep = prepare(spec)
    sp = prep.spec
    if sp.model_kind != MODEL_DEEPONET or sp.trunk_subsample is None:
        raise ValueError("run_sampler_trunk_subsample needs a DeepONet spec with trunk_subsample set")
    dev, d, P, psub = prep.device, sp.d, sp.P, int(sp.trunk_subsample)
    q = _to_dev(q0.reshape(-1, d), dev).clone()
    Cn = q.shape[0]
    rows = num_samples - burn
    if rows < 1:
        raise RuntimeError("burn must be less than num_samples.")
    samples = torch.empty((rows, Cn, d), dtype=torch.float32, device=dev)
    samples[0].copy_(q)
    acc = torch.empty((num_samples, Cn), dtype=torch.uint8, device=dev)
    ham = torch.empty((num_samples, Cn, 2), dtype=torch.float32, device=dev)
    fb_burn, fb_post = q.clone(), q.clone()   # param_burn_prev / ret_params[-1] of hamiltorch
    inj_p, inj_u = _to_dev(inject_momenta, dev), _to_dev(inject_uniforms, dev)
    m = _to_dev(inv_mass, dev)

    # the L + 3 subsets of an iteration are drawn on the host in the order the closure calls consume them and uploaded ONCE
    # (pinned, non-blocking); the closures then gather from device-resident index rows, so the loop really only enqueues
    calls = num_steps + 3
    subsets = {}

    def closure():
        k = subsets["next"]
        subsets["next"] = k + 1
        return _TrunkSubset(prep, subsets["dev"][k])

    row = 1
    for n in range(num_samples):
        host_idx = torch.tensor([random.sample(range(P), psub) for _ in range(calls)], dtype=torch.int64)
        try:
            host_idx = host_idx.pin_memory()
        except RuntimeError:
            pass
        subsets["dev"], subsets["next"] = host_idx.to(dev, non_blocking=True), 0
        p = inj_p[n].clone() if inj_p is not None else momentum_philox(seed, n, chain_offset, Cn, d, dev, inv_mass=m)
        u = inj_u[n].contiguous() if inj_u is not None else uniform_philox(seed, n, chain_offset, Cn, dev)
        q_prop = q.clone()
        lp0, _ = closure().logp_grad(q_prop, need_grad=False)
        ke0 = kinetic_energy(p, inv_mass=m)
        _, g = closure().logp_grad(q_prop)
        leapfrog_update(q_prop, p, g, step_size, 0.5, 1.0, inv_mass=m)                 # p += eps/2 g ; q += eps p
        for s_ in range(1, num_steps + 1):
            _, g = closure().logp_grad(q_prop)
            if s_ < num_steps:
                leapfrog_update(q_prop, p, g, step_size, 1.0, 1.0, inv_mass=m)         # p += eps g ; q += eps p
            else:
                leapfrog_update(q_prop, p, g, step_size, 1.0, 0.0, inv_mass=m)         # p += eps g
        ke1 = leapfrog_update(q_prop, p, g, step_size, -0.5, 0.0, want_ke=True, inv_mass=m)   # p -= eps/2 g
        lp1, _ = closure().logp_grad(q_prop, need_grad=False)
        H0, H1 = ke0 - lp0, ke1 - lp1
        ham[n, :, 0].copy_(H0)
        ham[n, :, 1].copy_(H1)
        if n > burn:
            mh_accept(H0, H1, u, q_prop, q, fb_post, stored=samples[row], accepted=acc[n])
            row += 1
        else:
            mh_accept(H0, H1, u, q_prop, q, fb_burn, accepted=acc[n])
    res = SampleResult(samples, acc, ham, None, None, grad_evals_per_chain=num_samples * (num_steps + 1), gpu_launches=-1)
    if to_host:
        torch.cuda.current_stream(dev).synchronize()
        res = SampleResult(samples.cpu(), acc.cpu(), ham.cpu(), None, None, res.grad_evals_per_chain, -1)
    return res


def momentum_philox(seed: int, iteration: int, chain0: int, chains: int, d: int, device=None,
                    inv_mass: Optional[torch.Tensor] = None) -> torch.Tensor:
    """p [C, d] ~ N(0, 1) (Philox stream 0); with ``inv_mass`` [d] the same draws times sqrt(1 / inv_mass)."""
    dev = _require_cuda(device)
    p = torch.empty((chains, d), dtype=torch.float32, device=dev)
    m = _to_dev(inv_mass, dev)
    with torch.cuda.device(dev):
        if m is None:
            _lib.check(_lib.load().vihmc_momentum_philox(seed, iteration, chain0, chains, d, p.data_ptr(), _stream(dev)))
        else:
            assert m.numel() == d, m.shape
            _lib.check(_lib.load().vihmc_momentum_philox_mass(seed, iteration, chain0, chains, d, m.data_ptr(), p.data_ptr(),
                                                              _stream(dev)))
    return p


def uniform_philox(seed: int, iteration: int, chain0: int, chains: int, device=None) -> torch.Tensor:
    dev = _require_cuda(device)
    u = torch.empty(chains, dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(_lib.load().vihmc_uniform_philox(seed, iteration, chain0, chains, u.data_ptr(), _stream(dev)))
    return u


def vi_redraw_philox(seed: int, iteration: int, chain0: int, chains: int, mu: torch.Tensor, sigma: torch.Tensor) -> torch.Tensor:
    dev = _require_cuda()
    mu_d, sg_d = _to_dev(mu, dev), _to_dev(sigma, dev)
    D = mu_d.numel()
    W = torch.empty((chains, D), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(_lib.load().vihmc_vi_redraw_philox(seed, iteration, chain0, chains, D, mu_d.data_ptr(), sg_d.data_ptr(),
                                                      W.data_ptr(), _stream(dev)))
    return W


def scatter_vi(frozen: torch.Tensor, sens_ind, q: torch.Tensor) -> torch.Tensor:
    dev = _require_cuda()
    fr = _to_dev(frozen, dev)
    ind = _to_dev(np.asarray(sens_ind, dtype=np.int64), dev, torch.int64)
    qd = _to_dev(q, dev)
    Cn, d = qd.shape
    W = torch.empty((Cn, fr.numel()), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(_lib.load().vihmc_scatter_vi(fr.data_ptr(), ind.data_ptr(), qd.data_ptr(), W.data_ptr(), Cn, fr.numel(), d,
                                                _stream(dev)))
    return W


def leapfrog_update(q: torch.Tensor, p: torch.Tensor, g: torch.Tensor, eps: float, kick: float, drift: float,
                    eps_per_chain: Optional[torch.Tensor] = None, want_ke: bool = False,
                    inv_mass: Optional[torch.Tensor] = None):
    """In-place fused update on device tensors q,p [C,d]; returns ke[C] if requested.  With ``inv_mass`` [d] (a device fp32
    tensor) the drift is q += ((drift eps) inv_mass) p and ke = 0.5 p.(inv_mass p) (vihmc_leapfrog_update_mass)."""
    dev = _require_cuda(q.device)
    Cn, d = q.shape
    lib = _lib.load()
    ke = scratch = None
    if want_ke:
        ke = torch.empty(Cn, dtype=torch.float32, device=dev)
        scratch = torch.empty(Cn * int(lib.vihmc_ke_partials(d)), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        if inv_mass is None:
            _lib.check(lib.vihmc_leapfrog_update(q.data_ptr(), p.data_ptr(), g.data_ptr(), eps, _ptr(eps_per_chain), kick, drift,
                                                 Cn, d, _ptr(ke), _ptr(scratch), _stream(dev)))
        else:
            assert inv_mass.is_cuda and inv_mass.dtype == torch.float32 and inv_mass.numel() == d and inv_mass.is_contiguous()
            _lib.check(lib.vihmc_leapfrog_update_mass(q.data_ptr(), p.data_ptr(), g.data_ptr(), inv_mass.data_ptr(), eps,
                                                      _ptr(eps_per_chain), kick, drift, Cn, d, _ptr(ke), _ptr(scratch), _stream(dev)))
    return ke


def kinetic_energy(p: torch.Tensor, inv_mass: Optional[torch.Tensor] = None) -> torch.Tensor:
    """ke[c] = 0.5 sum p[c]^2 (vihmc_kinetic_energy); with ``inv_mass`` [d] (device fp32) 0.5 sum p[c] (inv_mass p[c])."""
    dev = _require_cuda(p.device)
    Cn, d = p.shape
    lib = _lib.load()
    ke = torch.empty(Cn, dtype=torch.float32, device=dev)
    scratch = torch.empty(Cn * int(lib.vihmc_ke_partials(d)), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        if inv_mass is None:
            _lib.check(lib.vihmc_kinetic_energy(p.data_ptr(), Cn, d, ke.data_ptr(), scratch.data_ptr(), _stream(dev)))
        else:
            assert inv_mass.is_cuda and inv_mass.dtype == torch.float32 and inv_mass.numel() == d and inv_mass.is_contiguous()
            _lib.check(lib.vihmc_kinetic_energy_mass(p.data_ptr(), inv_mass.data_ptr(), Cn, d, ke.data_ptr(), scratch.data_ptr(),
                                                     _stream(dev)))
    return ke


def mh_accept(H0, H1, u, q_prop, q_cur, q_fb, stored=None, accepted=None):
    dev = _require_cuda(q_prop.device)
    Cn, d = q_prop.shape
    with torch.cuda.device(dev):
        _lib.check(_lib.load().vihmc_mh_accept(H0.data_ptr(), H1.data_ptr(), u.data_ptr(), q_prop.data_ptr(), q_cur.data_ptr(),
                                               q_fb.data_ptr(), _ptr(stored), int(stored is not None), _ptr(accepted), None,
                                               None, None, Cn, d, _stream(dev)))
