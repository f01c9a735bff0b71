"""Diagonal mass matrix (hamiltorch's 1-D ``inv_mass``) on the host: the restated specification (tests/mass_restated.py), the
argument checks of ``samplers.sample``, the forwarding of the hamiltorch front doors and the C ABI layout of the new field."""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest
import torch

import cases
import mass_restated as mr
from oracle import bnn_batched as bb
from oracle import hamiltorch_restated as hr
from vihmc import _lib, samplers, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _gauss_scaled(s):
    return lambda q: -0.5 * (q * q / (s * s)).sum()


def test_ones_mass_is_the_identity_restatement_bit_for_bit():
    """inv_mass = ones(d) reproduces the pinned identity restatement exactly: generator draws, injected streams, the split
    integrator and dual averaging."""
    s = torch.tensor([0.5, 1.0, 2.0, 0.8], dtype=torch.float32)
    f = _gauss_scaled(s)
    ones = torch.ones(4)
    q0 = torch.tensor([0.3, -0.2, 1.0, 0.1])
    for kw in (dict(num_samples=12, num_steps_per_sample=4, step_size=0.3, burn=2),
               dict(num_samples=12, num_steps_per_sample=4, step_size=0.3, burn=4, sampler=hr.Sampler.HMC_NUTS)):
        a_tr, b_tr = {}, {}
        a = hr.sample(f, q0, generator=torch.Generator().manual_seed(3), trace=a_tr, **kw)
        b = mr.sample(f, q0, generator=torch.Generator().manual_seed(3), trace=b_tr, inv_mass=ones, **kw)
        assert all(torch.equal(x, y) for x, y in zip(a, b)) and len(a) == len(b)
        assert a_tr == b_tr
    rs = np.random.RandomState(0)
    p = torch.from_numpy(rs.randn(8, 4).astype(np.float32))
    u = torch.from_numpy(rs.uniform(0.05, 1, 8).astype(np.float32))
    fs = [_gauss_scaled(s * 1.4), _gauss_scaled(s * 1.4)]
    for fn, integ in ((f, hr.Integrator.IMPLICIT), (fs, hr.Integrator.SPLITTING)):
        a_tr, b_tr = {}, {}
        a = hr.sample(fn, q0, num_samples=8, num_steps_per_sample=3, step_size=0.4, integrator=integ, momenta=p, uniforms=u, trace=a_tr)
        b = mr.sample(fn, q0, num_samples=8, num_steps_per_sample=3, step_size=0.4, integrator=integ, momenta=p, uniforms=u, trace=b_tr,
                      inv_mass=ones)
        assert all(torch.equal(x, y) for x, y in zip(a, b)) and a_tr == b_tr


def test_mass_restatement_samples_a_badly_scaled_gaussian():
    """Target N(0, diag(s^2)) with s over three decades: with inv_mass = s^2 the dynamics are those of a unit Gaussian, so a step
    of order one is accepted almost always and every coordinate gets its own variance; with the identity mass the same step is
    rejected.  eps = 0.8, not 1: on a unit Gaussian three leapfrog steps of 1 are exactly q -> -q, a chain that never mixes."""
    s = torch.tensor([0.01, 0.1, 1.0, 10.0], dtype=torch.float64)
    f = _gauss_scaled(s)
    tr = {}
    out = torch.stack(mr.sample(f, torch.zeros(4, dtype=torch.float64), num_samples=3000, num_steps_per_sample=3, step_size=0.8,
                                burn=100, generator=torch.Generator().manual_seed(5), trace=tr, inv_mass=s * s))
    assert tr["acceptance_rate"] > 0.9
    rel = out.var(0) / (s * s)
    assert torch.all((rel - 1).abs() < 0.2), rel           # ~3000 draws of short anti-correlated trajectories: several SE
    assert torch.all((out.mean(0) / s).abs() < 0.15)
    tr_id = {}
    mr.sample(f, torch.zeros(4, dtype=torch.float64), num_samples=200, num_steps_per_sample=3, step_size=0.8,
              generator=torch.Generator().manual_seed(5), trace=tr_id)
    assert tr_id["acceptance_rate"] < 0.05


def test_batched_mass_oracle_matches_the_per_chain_restatement():
    """mass_restated.sample_batched (fp64, all chains) against mass_restated.sample on the pinned BNN closure, with the VI scales as
    the mass and injected (scaled) momenta: same decisions, Hamiltonians to 1e-10."""
    g = cases.load_golden("bnn_vi_hmc_logp_grad.npz")
    case = cases.bnn_case(g, "d40_nll")
    x, y, _, _ = synth.bnn_data()
    model = bb.BatchedBnn(x.numpy(), y.numpy(), case["mu"].numpy(), case["ind"], tau_out=case["tau_out"], prior_var=case["prior_var"])
    closure = cases.bnn_oracle(case, dtype=torch.float64)
    m = (case["sigma"][case["ind"]].double() ** 2).numpy()
    q = case["q"].astype(np.float64)
    S, L, eps, Cn = 6, 7, 0.3, 3
    rs = np.random.RandomState(4)
    p = rs.randn(S, Cn, case["d"]) * np.sqrt(1.0 / m)
    p[2] *= 40.0
    u = rs.uniform(0.05, 1.0, size=(S, Cn))
    qf, acc, ham = mr.sample_batched(model, q[:Cn], S, L, eps, m, momenta=p, uniforms=u)
    for c in range(Cn):
        tr = {}
        mr.sample(closure, torch.from_numpy(q[c]), num_samples=S, num_steps_per_sample=L, step_size=eps,
                  momenta=torch.from_numpy(p[:, c]), uniforms=torch.from_numpy(u[:, c]), trace=tr, inv_mass=torch.from_numpy(m))
        assert tr["accept"] == list(acc[:, c])
        np.testing.assert_allclose(ham[:, c, 0], tr["H0"], rtol=1e-10)
        np.testing.assert_allclose(ham[:, c, 1], tr["H1"], rtol=1e-10)
    assert 0 < acc.sum() < acc.size


def test_inv_mass_argument_errors():
    """Checked on the host before anything reaches the GPU, so these raise without a device."""
    g = cases.load_golden("bnn_vi_hmc_logp_grad.npz")
    spec = cases.bnn_spec(cases.bnn_case(g, "d40_nll"))
    q = torch.zeros(40)
    with pytest.raises(ValueError, match="length d=40"):
        samplers.sample(spec, q, inv_mass=torch.ones(39))
    for bad in (0.0, -1.0, float("nan"), float("inf")):
        m = torch.ones(40)
        m[7] = bad
        with pytest.raises(ValueError, match="finite and > 0"):
            samplers.sample(spec, q, inv_mass=m)
    with pytest.raises(NotImplementedError, match="1-D"):
        samplers.sample(spec, q, inv_mass=torch.eye(40))
    with pytest.raises(NotImplementedError, match="1-D"):
        samplers.sample(spec, q, inv_mass=[torch.ones(20), torch.ones(20)])
    assert torch.equal(samplers.check_inv_mass(np.full(40, 2.0), 40), torch.full((40,), 2.0))
    assert samplers.check_inv_mass(None, 40) is None


def test_front_doors_forward_inv_mass(monkeypatch):
    """samplers.sample_model used to drop inv_mass; it and the hamiltorch shim now hand it to samplers.sample."""
    import hamiltorch

    seen = []
    monkeypatch.setattr(samplers, "sample", lambda *a, **kw: seen.append(kw) or "ran")
    net = torch.nn.Sequential(torch.nn.Linear(1, 4), torch.nn.Tanh(), torch.nn.Linear(4, 1))
    x, y = torch.zeros(5, 1), torch.zeros(5, 1)
    m = torch.full((13,), 0.5)
    assert samplers.sample_model(net, x, y, torch.zeros(13), model_loss="regression", inv_mass=m) == "ran"
    assert hamiltorch.sample_model(net, x, y, torch.zeros(13), model_loss="regression", inv_mass=m, seed=1) == "ran"
    assert hamiltorch.samplers.sample("spec", torch.zeros(13), inv_mass=m, seed=1) == "ran"
    assert len(seen) == 3 and all(kw["inv_mass"] is m for kw in seen)


def test_sampler_io_layout_matches_the_header(tmp_path):
    """ctypes SamplerIO against the C compiler's view of vihmc_sampler_io: size and the offset of every field, inv_mass last."""
    cc = shutil.which("cc") or shutil.which("gcc") or shutil.which("clang")
    if cc is None:
        pytest.skip("no host C compiler")
    fields = [f for f, _ in _lib.SamplerIO._fields_]
    assert fields[-1] == "inv_mass"
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "vihmc.h"\nint main(void) {\n'
                   '  printf("%zu\\n", sizeof(vihmc_sampler_io));\n'
                   + "".join(f'  printf("%zu\\n", offsetof(vihmc_sampler_io, {f}));\n' for f in fields) + "  return 0;\n}\n")
    exe = tmp_path / "layout"
    subprocess.run([cc, "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    vals = [int(v) for v in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    assert vals[0] == ctypes.sizeof(_lib.SamplerIO)
    assert vals[1:] == [getattr(_lib.SamplerIO, f).offset for f in fields]
