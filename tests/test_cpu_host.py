"""CPU-only tests: the C-ABI library loads and exports every symbol include/vihmc.h declares, host-side
validation mirrors the reference's error behaviour, and the oracle sampler behaves as documented."""
import os
import re

import numpy as np
import pytest
import torch

import cases
from oracle import hamiltorch_restated as hr
from oracle import philox_ref
from vihmc import _lib, samplers, synth
from vihmc.spec import DeepONetArch, LogProbSpec, MLPArch, sliced_prior_sigma

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_loads_and_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "vihmc.h")).read()
    declared = set(re.findall(r"VIHMC_API\s+[\w\s\*]+?\b(vihmc_\w+)\s*\(", header))
    assert declared == set(_lib.SYMBOLS), declared ^ set(_lib.SYMBOLS)
    lib = _lib.load()
    for name in declared:
        assert getattr(lib, name) is not None
    assert b"sm_100a" in lib.vihmc_version()


def test_prior_log_norm_host_helper():
    lib = _lib.load()
    sig = torch.tensor([0.5, 2.0, float("inf"), 1.0])
    got = lib.vihmc_prior_log_norm(sig.data_ptr(), 4, 1.0)
    want = sum(-np.log(s) - 0.5 * np.log(2 * np.pi) for s in (0.5, 2.0, 1.0))
    assert abs(got - want) < 1e-12
    assert abs(lib.vihmc_prior_log_norm(None, 3, 0.1) - 3 * (-np.log(np.float32(0.1)) - 0.5 * np.log(2 * np.pi))) < 1e-6


def test_no_cpu_fallback(monkeypatch):
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)   # on a GPU machine too: what a host without one sees
    g = cases.load_golden("bnn_vi_hmc_logp_grad.npz")
    spec = cases.bnn_spec(cases.bnn_case(g, "d40_nll"))
    with pytest.raises(_lib.VihmcError, match="no CPU fallback"):
        samplers.sample(spec, torch.zeros(40), num_samples=2, num_steps_per_sample=2, step_size=1e-3)


def test_layouts_match_torch_modules():
    net = torch.nn.Sequential(torch.nn.Linear(1, 10), torch.nn.Tanh(), torch.nn.Linear(10, 10), torch.nn.Tanh(),
                              torch.nn.Linear(10, 1))
    arch = MLPArch.from_module(net)
    assert arch == MLPArch(1, (10, 10), 1, "tanh", True)
    assert arch.tensor_numels() == [p.nelement() for p in net.parameters()] and arch.num_params == 141
    nobias = torch.nn.Sequential(torch.nn.Linear(1, 4), torch.nn.ReLU(), torch.nn.Linear(4, 1, bias=False))
    assert MLPArch.from_module(nobias) == MLPArch(1, (4,), 1, "relu", False)
    don = DeepONetArch()
    assert don.num_params == 172401 and len(don.tensor_numels()) == 37


def test_sliced_prior_matches_reference_loop():
    # main_VI_HMC.py:107-112 walks q (len d) with the full tensors' lengths [10,10,100,10,10,1]
    sig = sliced_prior_sigma(40, [10, 10, 100, 10, 10, 1], [1.0, 4.0, 9.0, 16.0, 25.0, 36.0])
    assert np.allclose(sig[:10], 1) and np.allclose(sig[10:20], 2) and np.allclose(sig[20:], 3)
    sig = sliced_prior_sigma(150, [10, 10, 100, 10, 10, 1], [1.0] * 6)
    assert np.isinf(sig[141:]).all() and np.allclose(sig[:141], 1)


def test_spec_validation_errors():
    x, y, _, _ = synth.bnn_data()
    arch = synth.bnn_arch()
    mu, sigma, ind = synth.bnn_vi_artifacts()
    with pytest.raises(ValueError, match="together"):
        LogProbSpec(arch=arch, x=x, y=y, frozen=mu).validate()
    with pytest.raises(IndexError):
        LogProbSpec(arch=arch, x=x, y=y, frozen=mu, sens_ind=np.array([0, 141])).validate()
    with pytest.raises(ValueError, match="duplicates"):
        LogProbSpec(arch=arch, x=x, y=y, frozen=mu, sens_ind=np.array([3, 3])).validate()
    with pytest.raises(NotImplementedError):
        LogProbSpec(arch=arch, x=x, y=y, loss="multi_class_linear_output").validate()
    with pytest.raises(ValueError, match="Activation"):
        from vihmc.spec import act_code
        act_code("gelu")


def test_sampler_argument_errors_match_hamiltorch():
    g = cases.load_golden("bnn_vi_hmc_logp_grad.npz")
    spec = cases.bnn_spec(cases.bnn_case(g, "d40_nll"))
    q = torch.zeros(40)
    with pytest.raises(RuntimeError, match="burn must be less than num_samples"):
        samplers.sample(spec, q, num_samples=5, burn=5)
    with pytest.raises(RuntimeError, match="burn must be greater than 0 for NUTS"):
        samplers.sample(spec, q, num_samples=5, sampler=samplers.Sampler.HMC_NUTS)
    with pytest.raises(TypeError, match="LogProbSpec"):
        samplers.sample(lambda p: p.sum(), q)
    with pytest.raises(NotImplementedError):
        samplers.sample([spec], q, integrator=samplers.Integrator.SPLITTING)
    with pytest.raises(ValueError, match="SPLITTING"):
        samplers.sample([spec, spec], q)
    with pytest.raises(RuntimeError, match="1d tensor"):
        samplers.sample(spec, torch.zeros(2, 3, 40))


def test_factories_build_the_same_spec_as_the_cases():
    g = cases.load_golden("bnn_vi_hmc_logp_grad.npz")
    case = cases.bnn_case(g, "d40_nll")
    x, y, _, _ = synth.bnn_data()
    net = torch.nn.Sequential(torch.nn.Linear(1, 10), torch.nn.Tanh(), torch.nn.Linear(10, 10), torch.nn.Tanh(),
                              torch.nn.Linear(10, 1))
    numels = [w.nelement() for w in net.parameters()]
    spec = samplers.define_model_log_prob_bnn(net, "NLL", x, y, numels, None, [torch.tensor(1.0)] * 6, 0.0025,
                                              params_mu=case["mu"], params_std=case["sigma"], grad_ind=case["ind"])
    ref = cases.bnn_spec(case)
    assert spec.d == ref.d == 40 and spec.D == 141
    assert torch.equal(spec.prior_sigma, ref.prior_sigma) and spec.loss == "NLL"
    spec.validate()


# ---------------------------------------------------------------------------------------------
# oracle sampler: bookkeeping + statistical sanity on a closed-form target
# ---------------------------------------------------------------------------------------------

def _gauss(q):
    return -0.5 * (q * q).sum()


def test_oracle_storage_rule():
    g = torch.Generator().manual_seed(0)
    for burn in (0, 3):
        out = hr.sample(_gauss, torch.zeros(3), num_samples=10, num_steps_per_sample=5, step_size=0.3, burn=burn, generator=g)
        assert len(out) == 10 - burn and torch.equal(out[0], torch.zeros(3))
    with pytest.raises(RuntimeError, match="burn must be less"):
        hr.sample(_gauss, torch.zeros(3), num_samples=3, burn=3)
    with pytest.raises(RuntimeError, match="NUTS"):
        hr.sample(_gauss, torch.zeros(3), num_samples=3, sampler=hr.Sampler.HMC_NUTS)


def test_oracle_nan_is_rejected():
    def bad(q):
        return torch.where(q[0] > 0.5, torch.tensor(float("nan"), dtype=q.dtype), -0.5 * (q * q).sum())
    g = torch.Generator().manual_seed(1)
    tr = {}
    out = hr.sample(bad, torch.zeros(2, dtype=torch.float64), num_samples=60, num_steps_per_sample=5, step_size=0.4,
                    generator=g, trace=tr)
    assert all(torch.isfinite(o).all() and o[0] <= 0.5 for o in out)
    assert not all(tr["accept"])


def test_oracle_samples_standard_normal():
    g = torch.Generator().manual_seed(2)
    out = torch.stack(hr.sample(_gauss, torch.zeros(4, dtype=torch.float64), num_samples=1500, num_steps_per_sample=8,
                                step_size=0.35, burn=100, generator=g))
    assert abs(float(out.mean())) < 0.12 and abs(float(out.var()) - 1.0) < 0.15


def test_oracle_split_integrator_is_symmetric_and_sums():
    """With M identical halves of a quadratic target the split integrator is exactly leapfrog-like:
    it must conserve H to O(eps^2) and be time reversible."""
    fs = [lambda q: -0.25 * (q * q).sum(), lambda q: -0.25 * (q * q).sum()]
    q0 = torch.tensor([1.0, -0.5], dtype=torch.float64)
    p0 = torch.tensor([0.3, 0.8], dtype=torch.float64)
    q1, p1 = hr.leapfrog(q0, p0, fs, 20, 0.05, hr.Integrator.SPLITTING)
    h0, h1 = hr.hamiltonian(q0, p0, fs), hr.hamiltonian(q1, p1, fs)
    assert abs(float(h0 - h1)) < 1e-3
    qb, pb = hr.leapfrog(q1, -p1, fs, 20, 0.05, hr.Integrator.SPLITTING)
    assert torch.allclose(qb, q0, atol=1e-12) and torch.allclose(-pb, p0, atol=1e-12)


def test_philox_known_answer_vectors():
    for ctr, key, want in philox_ref.KAT:
        got = philox_ref.philox4x32_10(*ctr, *key)
        assert tuple(int(v) for v in got) == want
    u = philox_ref.uniforms(1, 0, 1000, 0)
    assert u.dtype == np.float32 and (u > 0).all() and (u < 1).all()
    z = philox_ref.normals(1, 0, 64, 0, 101)
    assert z.shape == (64, 101) and abs(z.mean()) < 0.05 and abs(z.std() - 1) < 0.05


def test_artifact_files_have_the_reference_formats(tmp_path):
    """means/stds via torch.save, indices and samples via np.save with the reference's names, dtypes and shapes
    (main_VI_HMC.py:76-79, :381, :418; sensitivity.py:219-234); a single chain's list of draws is saved exactly as
    `np.save(path, params_hmc)` saves hamiltorch's list."""
    from vihmc import artifacts

    D, d, S = 141, 40, 7
    rs = np.random.RandomState(0)
    mu, sg = torch.from_numpy(rs.randn(D).astype(np.float32)), torch.from_numpy(rs.rand(D).astype(np.float32))
    ind = rs.choice(D, d, replace=False)
    artifacts.save_vi_artifacts(str(tmp_path), "uid1", mu, sg, ind, importance=rs.rand(D).astype(np.float32))
    m2, s2, i2 = artifacts.load_vi_artifacts(str(tmp_path), "uid1")
    assert torch.equal(m2, mu) and torch.equal(s2, sg) and m2.dtype == torch.float32
    assert i2.dtype == np.int64 and np.array_equal(i2, np.sort(ind))
    draws = [torch.from_numpy(rs.randn(d).astype(np.float32)) for _ in range(S)]
    (path,) = artifacts.save_hmc_params(str(tmp_path) + "/", "uid1", draws)
    ref = tmp_path / "ref.npy"
    np.save(ref, np.stack([t.numpy() for t in draws]))   # what np.save makes of the reference's list of 1-D tensors
    assert open(path, "rb").read() == open(ref, "rb").read()
    assert artifacts.load_hmc_params(path, burn=2).shape == (S - 2, d)
    paths = artifacts.save_hmc_params(str(tmp_path), "uid2", torch.from_numpy(rs.randn(S, 3, d).astype(np.float32)))
    assert len(paths) == 3 and np.load(paths[1]).shape == (S, d)
