"""GPU tests of the diagonal mass matrix (hamiltorch's 1-D ``inv_mass``) on every sampler path, against the restated specification
(tests/mass_restated.py) and against the identity-mass engine: ``inv_mass = ones(d)`` must give the identity run's bits."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import cases
import mass_restated as mr
from oracle import hamiltorch_restated as hr
from vihmc import engine, samplers, synth
from vihmc.spec import LogProbSpec, MLPArch

pytestmark = pytest.mark.gpu

RTOL = 1e-5
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bnn(name="d40_nll"):
    g = cases.load_golden("bnn_vi_hmc_logp_grad.npz")
    case = cases.bnn_case(g, name)
    return case, cases.bnn_spec(case)


def _vi_mass(case):
    return (case["sigma"][case["ind"]].float() ** 2).contiguous()


def _same(a, b):
    for k in ("samples", "accepted", "hamiltonians", "logp", "step_sizes"):
        x, y = getattr(a, k), getattr(b, k)
        assert (x is None) == (y is None), k
        if x is not None:
            assert torch.equal(x, y), k


# ------------------------------------------------------------------------------------------------
# 1. ones are the identity, bit for bit, on every path
# ------------------------------------------------------------------------------------------------
_VARIANT_SCRIPT = r"""
import sys, torch
sys.path[:0] = [{root!r}, {root!r} + "/vi-hmc_b200", {root!r} + "/tests"]
import cases
from vihmc import engine
g = cases.load_golden("bnn_vi_hmc_logp_grad.npz")
for name in ("d40_nll", "d141_nll", "d14_nll"):
    case = cases.bnn_case(g, name)
    spec = cases.bnn_spec(case)
    q0 = torch.from_numpy(case["q"][:4]).repeat(3, 1)
    kw = dict(num_samples=6, num_steps=7, step_size=3e-4, burn=1, seed=11)
    a = engine.run_sampler([spec], q0, **kw)
    b = engine.run_sampler([spec], q0, inv_mass=torch.ones(case["d"]), **kw)
    assert a.gpu_launches == b.gpu_launches == 1
    for k in ("samples", "accepted", "hamiltonians", "logp", "step_sizes"):
        assert torch.equal(getattr(a, k), getattr(b, k)), (name, k)
    # and a real mass changes the run
    c = engine.run_sampler([spec], q0, inv_mass=torch.full((case["d"],), 2.0), **kw)
    assert not torch.equal(a.samples, c.samples)
print("VARIANT OK")
"""


@pytest.mark.parametrize("env", [{}, {"VIHMC_SMALL_GENERIC": "1"}, {"VIHMC_SMALL_FAST": "1"}], ids=["default", "generic", "fast1"])
def test_persistent_kernel_ones_mass_is_identity_in_every_variant(env):
    """The persistent kernel's variants are chosen by environment knobs read once per process, so each runs in a subprocess.
    default covers fast v2 with register-resident coordinates (d40, d14) and without (d141)."""
    full = {k: v for k, v in os.environ.items() if not k.startswith("VIHMC_SMALL")}
    full.update(env)
    out = subprocess.run([sys.executable, "-c", _VARIANT_SCRIPT.format(root=ROOT)], env=full, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0 and "VARIANT OK" in out.stdout, out.stdout + out.stderr


def test_general_sampler_ones_mass_is_identity():
    case, spec = _bnn()
    d = case["d"]
    q0 = torch.from_numpy(case["q"][:4])
    ones = torch.ones(d)
    kw = dict(num_samples=6, num_steps=7, step_size=3e-4, burn=2, seed=5)
    _same(engine.run_sampler([spec], q0, force_general=True, **kw), engine.run_sampler([spec], q0, force_general=True, inv_mass=ones, **kw))
    # dual averaging (Sampler.HMC_NUTS)
    kw_nuts = dict(kw, adapt_step_size=True)
    for fg in (False, True):
        _same(engine.run_sampler([spec], q0, force_general=fg, **kw_nuts),
              engine.run_sampler([spec], q0, force_general=fg, inv_mass=ones, **kw_nuts))
    # per-sample VI redraw
    for fg in (False, True):
        _same(engine.run_sampler([spec], q0, force_general=fg, vi_redraw=True, **kw),
              engine.run_sampler([spec], q0, force_general=fg, vi_redraw=True, inv_mass=ones, **kw))
    # split integrator on the small DeepONet (2 closures)
    inp = cases.don_inputs("small")
    specs = cases.don_spec(inp, "split")
    qd = inp["theta"].clone()[None].repeat(2, 1)
    kws = dict(num_samples=4, num_steps=3, step_size=1e-4, burn=1, seed=3, integrator=engine.INTEGRATOR_SPLITTING)
    _same(engine.run_sampler(specs, qd, **kws), engine.run_sampler(specs, qd, inv_mass=torch.ones(qd.shape[1]), **kws))


def test_trunk_subsample_and_data_sharded_ones_mass_is_identity():
    import random

    from vihmc import dist as vd

    inp = cases.don_inputs("small")
    spec = cases.don_spec(inp, "vi")
    import dataclasses
    spec = dataclasses.replace(spec, trunk_subsample=10)
    q0 = inp["mu"][inp["ind"]].clone()[None].repeat(2, 1)
    kw = dict(num_samples=4, num_steps=3, step_size=1e-4, burn=1, seed=4)
    random.seed(0)
    a = engine.run_sampler_trunk_subsample(spec, q0, **kw)
    random.seed(0)
    b = engine.run_sampler_trunk_subsample(spec, q0, inv_mass=torch.ones(q0.shape[1]), **kw)
    assert torch.equal(a.samples, b.samples) and torch.equal(a.accepted, b.accepted) and torch.equal(a.hamiltonians, b.hamiltonians)

    arch = MLPArch(in_dim=1, widths=(64, 64), out_dim=1, act="tanh", last_bias=True)
    x, y = synth.wide_bnn_data(n=500, seed=1)
    wspec = LogProbSpec(arch=arch, x=x, y=y, loss="NLL", tau_out=0.0025, prior_sigma_scalar=1.0)
    q0 = synth.default_linear_init(arch, seed=2).unsqueeze(0).repeat(3, 1)
    kw = dict(num_samples=4, num_steps=5, step_size=2e-5, burn=1, seed=9)
    a = vd.sample_data_sharded(vd.shard_spec_rows(wspec, 0, 1), q0, **kw)
    b = vd.sample_data_sharded(vd.shard_spec_rows(wspec, 0, 1), q0, inv_mass=torch.ones(arch.num_params, device="cuda"), **kw)
    for k in ("samples", "accepted", "hamiltonians"):
        assert torch.equal(a[k], b[k]), k


# ------------------------------------------------------------------------------------------------
# 2./3. building blocks against torch on the device
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("d", [1, 40, 4097, 172401])
def test_momentum_mass_equals_scaled_identity_draws(d):
    rs = np.random.RandomState(d % 1000)
    m = torch.from_numpy(np.exp(rs.uniform(-5, 3, d)).astype(np.float32)).cuda()
    C = 3 if d > 100000 else 9
    z = engine.momentum_philox(77, 5, 11, C, d)
    p = engine.momentum_philox(77, 5, 11, C, d, inv_mass=m)
    assert torch.equal(p, z * torch.sqrt(1 / m))


@pytest.mark.parametrize("d", [1, 40, 4097, 172401])
def test_leapfrog_update_mass_bitwise_vs_torch(d):
    rs = np.random.RandomState(d % 997)
    C = 3 if d > 100000 else 7
    dev = torch.device("cuda")
    m = torch.from_numpy(np.exp(rs.uniform(-5, 3, d)).astype(np.float32)).to(dev)
    eps_pc = torch.from_numpy(rs.uniform(1e-4, 1e-2, C).astype(np.float32)).to(dev)
    for kick, drift in ((0.5, 1.0), (1.0, 1.0), (1.0, 0.0), (-0.5, 0.0)):
        q = torch.from_numpy(rs.randn(C, d).astype(np.float32)).to(dev)
        p = torch.from_numpy(rs.randn(C, d).astype(np.float32)).to(dev)
        g = torch.from_numpy(rs.randn(C, d).astype(np.float32)).to(dev)
        e = eps_pc[:, None]
        p_ref = p + (kick * e) * g
        q_ref = q + ((drift * e) * m) * p_ref if drift != 0.0 else q.clone()
        ke = engine.leapfrog_update(q, p, g, 0.0, kick, drift, eps_per_chain=eps_pc, want_ke=True, inv_mass=m)
        assert torch.equal(p, p_ref) and torch.equal(q, q_ref), (kick, drift)
        ke_ref = 0.5 * (p_ref.double() * (m.double() * p_ref.double())).sum(1)
        np.testing.assert_allclose(ke.cpu().numpy(), ke_ref.cpu().numpy(), rtol=2e-6)
        ke2 = engine.kinetic_energy(p, inv_mass=m)
        np.testing.assert_allclose(ke2.cpu().numpy(), ke_ref.cpu().numpy(), rtol=2e-6)


# ------------------------------------------------------------------------------------------------
# 4./5. trajectories and decisions against the restated oracle
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("force_general", [False, True], ids=["persistent", "general"])
def test_single_trajectory_with_mass_matches_oracle(force_general):
    case, spec = _bnn()
    m = _vi_mass(case)
    d, L, eps = case["d"], 25, 0.02
    rs = np.random.RandomState(11)
    q0 = torch.from_numpy(case["q"][0])
    p = torch.from_numpy((rs.randn(2, 1, d) * np.sqrt(1.0 / m.numpy())).astype(np.float32))
    u = torch.full((2, 1), 1e-30)
    res = engine.run_sampler([spec], q0[None], 2, L, eps, burn=0, inject_momenta=p, inject_uniforms=u, inv_mass=m,
                             force_general=force_general)
    for dtype, tol in ((torch.float32, 2e-5), (torch.float64, 2e-5)):
        closure = cases.bnn_oracle(case, dtype=dtype)
        tr = {}
        out = torch.stack(mr.sample(closure, q0.to(dtype), num_samples=2, num_steps_per_sample=L, step_size=eps,
                                    momenta=p[:, 0].to(dtype), uniforms=u[:, 0], trace=tr, inv_mass=m.to(dtype)))
        np.testing.assert_allclose(res.samples[1, 0].numpy(), out[1].numpy(), rtol=tol, atol=tol * float(out[1].abs().max()))
        np.testing.assert_allclose(res.hamiltonians[:, 0, 0].numpy(), tr["H0"], rtol=RTOL)
        np.testing.assert_allclose(res.hamiltonians[:, 0, 1].numpy(), tr["H1"], rtol=RTOL)


@pytest.mark.parametrize("force_general", [False, True], ids=["persistent", "general"])
def test_accept_reject_with_mass_identical_to_fp64_oracle(force_general):
    """The margin rule of test_gpu_bnn.py::test_accept_reject_identical_over_short_run, with inv_mass = sigma_VI^2 and momenta
    drawn from N(0, 1 / inv_mass) (30 % of them x40 so that trajectories overshoot)."""
    case, spec = _bnn()
    m = _vi_mass(case)
    d, S, L, eps, Cn, burn = case["d"], 40, 5, 0.02, 8, 5
    rs = np.random.RandomState(5)
    mu, sg = case["mu"].numpy()[case["ind"]], case["sigma"].numpy()[case["ind"]]
    q0 = torch.from_numpy((mu[None] + sg[None] * rs.randn(Cn, d)).astype(np.float32))
    p = (rs.randn(S, Cn, d) * np.sqrt(1.0 / m.numpy())).astype(np.float32)
    p[rs.rand(S, Cn) < 0.3] *= 40
    p = torch.from_numpy(p)
    u = torch.from_numpy(rs.uniform(0.01, 1.0, size=(S, Cn)).astype(np.float32))
    res = engine.run_sampler([spec], q0, S, L, eps, burn=burn, inject_momenta=p, inject_uniforms=u, inv_mass=m, force_general=force_general)
    closure = cases.bnn_oracle(case, dtype=torch.float64)
    checked = rejects = 0
    for c in range(Cn):
        tr = {}
        out = torch.stack(mr.sample(closure, q0[c].double(), num_samples=S, num_steps_per_sample=L, step_size=eps, burn=burn,
                                    momenta=p[:, c].double(), uniforms=u[:, c], trace=tr, inv_mass=m.double()))
        acc_ref = np.array(tr["accept"])
        rho = np.minimum(0.0, np.array(tr["H0"]) - np.array(tr["H1"]))
        margin = np.abs(rho - np.log(u[:, c].numpy().astype(np.float64)))
        acc = res.accepted[:, c].numpy().astype(bool)
        diverged = False
        for n in range(S):
            if acc[n] != acc_ref[n]:
                assert margin[n] < 0.1, f"chain {c} iteration {n}: decision differs at margin {margin[n]:.3f}"
                diverged = True
                break
            checked += 1
            rejects += int(not acc[n])
        if not diverged:
            np.testing.assert_allclose(res.samples[:, c].numpy(), out.numpy(), rtol=5e-4, atol=5e-4)
    assert checked >= 150 and rejects >= 20 and checked - rejects >= 20, (checked, rejects)


def test_split_integrator_with_mass_matches_oracle():
    """Small DeepONet, two closures, Integrator.SPLITTING with a mass: H0, H1 and the end point against the fp64 restatement."""
    inp = cases.don_inputs("small")
    specs = cases.don_spec(inp, "split")
    fns = cases.don_oracle(inp, "split", dtype=torch.float64)
    q0 = inp["theta"].clone()
    d = q0.numel()
    rs = np.random.RandomState(2)
    m = torch.from_numpy(np.exp(rs.uniform(-2, 1, d)).astype(np.float32))
    S, L, eps = 3, 4, 1e-4
    p = torch.from_numpy((rs.randn(S, 1, d) * np.sqrt(1.0 / m.numpy())).astype(np.float32))
    u = torch.full((S, 1), 1e-30)
    res = engine.run_sampler(specs, q0[None], S, L, eps, integrator=engine.INTEGRATOR_SPLITTING, inject_momenta=p, inject_uniforms=u,
                             inv_mass=m)
    tr = {}
    out = torch.stack(mr.sample(fns, q0.double(), num_samples=S, num_steps_per_sample=L, step_size=eps, integrator=hr.Integrator.SPLITTING,
                                momenta=p[:, 0].double(), uniforms=u[:, 0], trace=tr, inv_mass=m.double()))
    assert [bool(a) for a in res.accepted[:, 0]] == tr["accept"]
    np.testing.assert_allclose(res.hamiltonians[:, 0, 0].numpy(), tr["H0"], rtol=2e-5)
    np.testing.assert_allclose(res.hamiltonians[:, 0, 1].numpy(), tr["H1"], rtol=2e-5)
    np.testing.assert_allclose(res.samples[-1, 0].numpy(), out[-1].numpy(), rtol=1e-4, atol=1e-4 * float(out[-1].abs().max()))


@pytest.mark.parametrize("force_general", [False, True], ids=["persistent", "general"])
def test_dual_averaging_with_mass_matches_oracle(force_general):
    """Forced decisions (u = 1e-30 accepts, u = 2 rejects) so the recursion itself is compared: the step size of every iteration
    against the oracle's, as in test_gpu_bnn.py::test_dual_averaging_matches_oracle, now with inv_mass = sigma_VI^2."""
    case = dict(_bnn()[0])
    case["tau_out"] = 25.0
    spec = cases.bnn_spec(case)
    m = _vi_mass(case)
    d, S, L, burn, eps0 = case["d"], 9, 6, 7, 0.05
    rs = np.random.RandomState(21)
    q0 = torch.from_numpy(case["q"][0])[None]
    p = torch.from_numpy((rs.randn(S, 1, d) * np.sqrt(1.0 / m.numpy())).astype(np.float32))
    u = torch.full((S, 1), 1e-30)
    u[[2, 5, 6]] = 2.0
    closure = cases.bnn_oracle(case, dtype=torch.float64)
    eps_seen = []
    for k in range(1, burn + 1):
        res = engine.run_sampler([spec], q0, k + 1, L, eps0, burn=k, adapt_step_size=True, inject_momenta=p[:k + 1],
                                 inject_uniforms=u[:k + 1], inv_mass=m, force_general=force_general)
        tr = {}
        mr.sample(closure, q0[0].double(), num_samples=k + 1, num_steps_per_sample=L, step_size=eps0, burn=k, momenta=p[:k + 1, 0].double(),
                  uniforms=u[:k + 1, 0], trace=tr, sampler=hr.Sampler.HMC_NUTS, inv_mass=m.double())
        assert tr["accept"] == [bool(a) for a in res.accepted[:, 0].numpy()]
        assert abs(float(res.step_sizes[0]) - tr["final_step_size"]) <= 3e-3 * tr["final_step_size"], (k, float(res.step_sizes[0]),
                                                                                                         tr["final_step_size"])
        eps_seen.append(tr["final_step_size"])
    assert max(eps_seen) / min(eps_seen) > 1.2


# ------------------------------------------------------------------------------------------------
# 6. exact Gaussian target: stationarity of N(0, diag(sigma^2)) under the mass-preconditioned chain
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("force_general", [False, True], ids=["persistent", "general"])
def test_prior_only_gaussian_is_stationary_with_mass(force_general):
    """loss='regression' with tau_out = 0 makes the likelihood term exactly zero, so the posterior is the prior
    N(0, diag(prior_sigma^2)), prior_sigma over three decades.  4096 chains start from it; 50 iterations later each coordinate's
    mean and variance over the chains still match within 5 standard errors.  eps = 0.3 is fine with inv_mass = prior_sigma^2
    (acceptance > 0.9) and hopeless with the identity mass (< 0.05): it is 30 x the narrowest scale."""
    arch = MLPArch(in_dim=1, widths=(4, 4), out_dim=1, act="tanh", last_bias=True)
    D = arch.num_params
    rs = np.random.RandomState(8)
    sig = torch.from_numpy(np.exp(rs.uniform(np.log(0.01), np.log(10.0), D)).astype(np.float32))
    x = torch.from_numpy(rs.uniform(-1, 1, (20, 1)).astype(np.float32))
    spec = LogProbSpec(arch=arch, x=x, y=torch.zeros(20), loss="regression", tau_out=0.0, prior_sigma=sig)
    Cn = 4096
    q0 = (sig[None] * torch.randn(Cn, D, generator=torch.Generator().manual_seed(1))).float()
    kw = dict(num_samples=50, num_steps=8, step_size=0.3, burn=0, seed=12, force_general=force_general)
    res = engine.run_sampler([spec], q0, inv_mass=sig * sig, **kw)
    assert res.acceptance_rate > 0.9
    qf = res.samples[-1].double()
    s2 = sig.double() ** 2
    mean_se = (s2 / Cn).sqrt()
    var_se = s2 * np.sqrt(2.0 / (Cn - 1))
    assert torch.all(qf.mean(0).abs() < 5 * mean_se)
    assert torch.all((qf.var(0) - s2).abs() < 5 * var_se)
    ident = engine.run_sampler([spec], q0[:256], **dict(kw, num_samples=10))
    assert ident.acceptance_rate < 0.05


# ------------------------------------------------------------------------------------------------
# 7./8. persistent kernel == general sampler; sharding; the data-sharded graphs
# ------------------------------------------------------------------------------------------------
def test_persistent_kernel_matches_general_sampler_with_mass():
    g = cases.load_golden("bnn_vi_hmc_logp_grad.npz")
    for name in ("d40_nll", "d141_nll"):
        case = cases.bnn_case(g, name)
        spec = cases.bnn_spec(case)
        m = _vi_mass(case)
        q0 = torch.from_numpy(case["q"][:4])
        kw = dict(num_samples=5, num_steps=9, step_size=0.02, burn=1, seed=3, inv_mass=m)
        a = engine.run_sampler([spec], q0, **kw)
        b = engine.run_sampler([spec], q0, force_general=True, **kw)
        assert a.gpu_launches == 1
        assert torch.equal(a.accepted, b.accepted)
        np.testing.assert_allclose(a.samples.numpy(), b.samples.numpy(), rtol=1e-5, atol=1e-6)
        np.testing.assert_allclose(a.hamiltonians.numpy(), b.hamiltonians.numpy(), rtol=1e-6)


def test_sharding_invariance_with_mass_and_data_sharded_graph_cache():
    case, spec = _bnn()
    m = _vi_mass(case)
    rs = np.random.RandomState(9)
    mu, sg = case["mu"].numpy()[case["ind"]], case["sigma"].numpy()[case["ind"]]
    q0 = torch.from_numpy((mu[None] + sg[None] * rs.randn(16, case["d"])).astype(np.float32))
    for fg in (False, True):
        kw = dict(num_samples=6, num_steps=7, step_size=0.02, burn=1, seed=42, inv_mass=m, force_general=fg)
        whole = engine.run_sampler([spec], q0, **kw)
        lo = engine.run_sampler([spec], q0[:8], chain_offset=0, **kw)
        hi = engine.run_sampler([spec], q0[8:], chain_offset=8, **kw)
        assert torch.equal(whole.samples[:, :8], lo.samples) and torch.equal(whole.samples[:, 8:], hi.samples)
        assert torch.equal(whole.accepted[:, 8:], hi.accepted)

    from vihmc import dist as vd

    arch = MLPArch(in_dim=1, widths=(64, 64), out_dim=1, act="tanh", last_bias=True)
    x, y = synth.wide_bnn_data(n=500, seed=1)
    wspec = LogProbSpec(arch=arch, x=x, y=y, loss="NLL", tau_out=0.0025, prior_sigma_scalar=1.0)
    q0 = synth.default_linear_init(arch, seed=2).unsqueeze(0).repeat(3, 1)
    kw = dict(num_samples=4, num_steps=5, step_size=2e-5, burn=1, seed=9)
    local = vd.shard_spec_rows(wspec, 0, 1)
    prep = engine.prepare(local)
    for scale in (4.0, 0.25):
        mm = torch.from_numpy(np.exp(rs.uniform(-1, 1, arch.num_params)).astype(np.float32) * scale).cuda()
        a = vd.sample_data_sharded(prep, q0, inv_mass=mm, **kw)
        assert a["graphs"]
        b = engine.run_sampler([wspec], q0, force_general=True, inv_mass=mm, **kw)
        assert torch.equal(a["accepted"].cpu(), b.accepted)
        np.testing.assert_allclose(a["samples"].cpu().numpy(), b.samples.numpy(), rtol=1e-5, atol=1e-6)
        np.testing.assert_allclose(a["hamiltonians"].cpu().numpy(), b.hamiltonians.numpy(), rtol=1e-6)


# ------------------------------------------------------------------------------------------------
# 9. front doors
# ------------------------------------------------------------------------------------------------
def test_front_doors_with_mass_equal_the_device_entry():
    import ctypes as C

    import hamiltorch
    from oracle import reference_shaped as rshape
    from vihmc import _lib, closure

    x, y, _, _ = synth.bnn_data()
    mu, sigma, ind = synth.bnn_vi_artifacts(141, 40, seed=1)
    torch.manual_seed(0)
    net = rshape.mlp_module(1, (10, 10), 1, act="tanh")
    numels = [w.nelement() for w in net.parameters()]
    shapes = [w.shape for w in net.parameters()]
    fn = rshape.bnn_closure(net, "NLL", x, y, numels, shapes, [torch.tensor(1.0) for _ in numels], 0.0025, params_mu=mu,
                            params_std=sigma, grad_ind=ind, depth=1, act="tanh")
    m = (torch.as_tensor(sigma)[ind].float() ** 2).contiguous()
    params_init = mu[ind].clone()
    kw = dict(num_samples=8, num_steps_per_sample=10, step_size=0.02, seed=7)
    out = hamiltorch.samplers.sample(fn, params_init, inv_mass=m, **kw)
    spec = closure.spec_from_closure(fn)
    want = samplers.sample(spec, params_init, inv_mass=m, **kw)
    assert torch.equal(torch.stack(out), torch.stack(want))
    dev = engine.run_sampler([spec], params_init[None], 8, 10, 0.02, seed=7, inv_mass=m)
    assert torch.equal(torch.stack(want), dev.samples[:, 0])
    ident = samplers.sample(spec, params_init, **kw)
    assert not torch.equal(torch.stack(ident), torch.stack(want))

    # hamiltorch.sample_model (hamiltorch's own prior / regression likelihood) forwards inv_mass
    arch = synth.bnn_arch()
    torch.manual_seed(1)
    net2 = rshape.mlp_module(1, (10, 10), 1, act="tanh")
    mm = torch.from_numpy(np.exp(np.random.RandomState(3).uniform(-2, 0, 141)).astype(np.float32))
    q0 = synth.default_linear_init(arch, seed=0)
    a = hamiltorch.sample_model(net2, x, y, q0, model_loss="regression", num_samples=5, num_steps_per_sample=6, step_size=1e-3,
                                tau_out=400.0, inv_mass=mm, seed=3)
    hspec = samplers.define_model_log_prob_hamiltorch(net2, "regression", x, y, numels, shapes, [torch.tensor(1.0)] * 6, 400.0)
    b = engine.run_sampler([hspec], q0[None], 5, 6, 1e-3, seed=3, inv_mass=mm)
    assert torch.equal(torch.stack(a), b.samples[:, 0])

    # vihmc_sample_host uploads io.inv_mass
    prep = engine.prepare(spec)
    lib = _lib.load()
    S, L, Cn, d = 6, 10, 4, 40
    q0h = params_init[None].repeat(Cn, 1).contiguous()
    dev_res = engine.run_sampler([spec], q0h, S, L, 0.02, seed=7, inv_mass=m)
    hp = _lib.Problem.from_buffer_copy(prep.problem)
    keep = {}
    for name, t in (("x", spec.x.reshape(spec.N, -1)), ("y", spec.y.reshape(-1)), ("frozen", spec.frozen),
                    ("prior_sigma", spec.prior_sigma), ("prior_mu", spec.prior_mu)):
        keep[name] = None if t is None else torch.as_tensor(t).detach().float().cpu().contiguous()
        setattr(hp, name, None if t is None else keep[name].data_ptr())
    keep["sens_ind"] = torch.as_tensor(np.asarray(spec.sens_ind, np.int64)).contiguous()
    hp.sens_ind = keep["sens_ind"].data_ptr()
    cfg = _lib.SamplerCfg(num_samples=S, num_steps=L, burn=0, integrator=0, adapt_step_size=0, hamiltorch_fallback_rule=1,
                          step_size=0.02, desired_accept_rate=0.8, seed=7, chain_offset=0)
    io = _lib.SamplerIO()
    acc = torch.zeros((S, Cn), dtype=torch.uint8)
    io.accepted = acc.data_ptr()
    io.inv_mass = m.data_ptr()
    out_h = torch.empty((S, Cn, d), dtype=torch.float32)
    _lib.check(lib.vihmc_sample_host(C.byref(hp), 1, C.byref(cfg), Cn, q0h.data_ptr(), out_h.data_ptr(), C.byref(io)))
    assert torch.equal(out_h, dev_res.samples) and torch.equal(acc, dev_res.accepted)
