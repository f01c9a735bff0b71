"""GPU side of the ``hamiltorch`` drop-in: closures with the reference's shape (oracle/reference_shaped.py -- the real
reference is not on the GPU box; tests/test_closure_dropin.py shows in the build container that both recover to the
same specification) are handed to ``hamiltorch.samplers.sample`` exactly as the reference's drivers do."""
from __future__ import annotations

import dataclasses

import numpy as np
import pytest
import torch

import cases
from oracle import hamiltorch_restated as hr
from oracle import reference_shaped as rshape
from vihmc import closure, samplers, synth

pytestmark = pytest.mark.gpu


def _bnn_closure(d=40, act="tanh", loss="NLL", tau_out=0.0025):
    x, y, _, _ = synth.bnn_data()
    mu, sigma, ind = synth.bnn_vi_artifacts(141, d, seed=1)
    torch.manual_seed(0)
    net = rshape.mlp_module(1, (10, 10), 1, act=act)
    numels = [w.nelement() for w in net.parameters()]
    shapes = [w.shape for w in net.parameters()]
    prior_list = [torch.tensor(1.0) for _ in numels]
    fn = rshape.bnn_closure(net, loss, x, y, numels, shapes, prior_list, tau_out, params_mu=mu, params_std=sigma, grad_ind=ind,
                            depth=1, act=act)
    return fn, mu, sigma, ind


def test_bnn_closure_through_the_hamiltorch_shim_matches_the_spec_path_bit_for_bit():
    import hamiltorch

    fn, mu, sigma, ind = _bnn_closure()
    params_init = mu[ind].clone()
    out = hamiltorch.samplers.sample(fn, params_init, num_samples=12, num_steps_per_sample=20, step_size=5e-4, debug=False, seed=7)
    assert isinstance(out, list) and len(out) == 12 and out[0].shape == (40,) and out[0].device.type == "cpu"
    spec = closure.spec_from_closure(fn)
    want = samplers.sample(spec, params_init, num_samples=12, num_steps_per_sample=20, step_size=5e-4, seed=7)
    assert torch.equal(torch.stack(out), torch.stack(want))
    # the set-up check itself: closure (torch eager, CPU) vs engine at params_init
    errs = closure.verify_closure(fn, spec, params_init, rtol=1e-5)
    assert errs["logp_rel_err"] <= 1e-5 and errs["grad_rel_err"] <= 1e-5
    # successive calls without a seed draw it from torch's global generator: reproducible under manual_seed, different per call
    torch.manual_seed(3)
    a = torch.stack(hamiltorch.samplers.sample(fn, params_init, num_samples=4, num_steps_per_sample=5, step_size=5e-4))
    b = torch.stack(hamiltorch.samplers.sample(fn, params_init, num_samples=4, num_steps_per_sample=5, step_size=5e-4))
    torch.manual_seed(3)
    a2 = torch.stack(hamiltorch.samplers.sample(fn, params_init, num_samples=4, num_steps_per_sample=5, step_size=5e-4))
    assert torch.equal(a, a2) and not torch.equal(a, b)
    # many chains in one call (extension keyword)
    many = hamiltorch.samplers.sample(fn, params_init, num_samples=4, num_steps_per_sample=5, step_size=5e-4, num_chains=64, seed=1)
    assert many.shape == (4, 64, 40)


def test_a_misread_closure_is_refused_by_the_set_up_check(monkeypatch):
    fn, mu, sigma, ind = _bnn_closure()
    good = closure.spec_from_closure(fn)
    monkeypatch.setattr(closure, "spec_from_closure", lambda f: dataclasses.replace(good, tau_out=good.tau_out * 1.01))
    with pytest.raises(closure.ClosureError, match="does not reproduce"):
        samplers.sample(fn, mu[ind].clone(), num_samples=2, num_steps_per_sample=2, step_size=5e-4)


def test_closure_trajectory_matches_the_restated_sampler_run_on_the_closure_itself():
    """The closure goes to the GPU engine as data; the restated hamiltorch sampler calls the SAME closure on the CPU (fp32,
    injected momenta): end point of every sample agrees."""
    fn, mu, sigma, ind = _bnn_closure(act="relu")
    S, L, eps, d = 3, 10, 5e-4, 40
    rs = np.random.RandomState(2)
    p = torch.from_numpy(rs.randn(S, 1, d).astype(np.float32))
    u = torch.full((S, 1), 1e-30)
    got = samplers.sample(fn, mu[ind].clone(), num_samples=S, num_steps_per_sample=L, step_size=eps, inject_momenta=p,
                          inject_uniforms=u)
    ref = hr.sample(fn, mu[ind].clone(), num_samples=S, num_steps_per_sample=L, step_size=eps, momenta=p[:, 0], uniforms=u[:, 0])
    np.testing.assert_allclose(torch.stack(got).numpy(), torch.stack(ref).numpy(), rtol=1e-4, atol=1e-4)


def _don_closures():
    inp = cases.don_inputs("small")
    arch = inp["arch"]
    net = rshape.DeepONetModule(arch.width_branch, arch.width_trunk, arch.in_branch, arch.in_trunk, arch.depth_branch,
                                arch.depth_trunk, arch.act, arch.output_neurons)
    tr = (inp["x1"].unsqueeze(1), inp["x2"].unsqueeze(0), inp["y"])
    tau_list = [torch.tensor(0.01)]
    return inp, net, tr, tau_list


def test_deeponet_closures_vi_full_and_split_through_the_shim():
    import hamiltorch

    inp, net, tr, tau_list = _don_closures()
    vi = rshape.deeponet_closure(net, "NLL", tr, tau_list, 1.0, mean_params=inp["mu"], std_params=inp["sigma"], grad_ind=inp["ind"])
    q0 = inp["mu"][inp["ind"]].clone()
    out = hamiltorch.samplers.sample(vi, q0, num_samples=5, num_steps_per_sample=4, step_size=1e-4, sampler=hamiltorch.samplers.Sampler.HMC, seed=9)
    want = samplers.sample(cases.don_spec(inp, "vi"), q0, num_samples=5, num_steps_per_sample=4, step_size=1e-4, seed=9)
    assert torch.equal(torch.stack(out), torch.stack(want))

    half = tr[0].shape[0] // 2
    fns = [rshape.deeponet_closure(net, "NLL", (tr[0][i * half:(i + 1) * half], tr[1], tr[2][i * half:(i + 1) * half]), tau_list, 1.0,
                                   prior_scale=2) for i in range(2)]
    out = hamiltorch.samplers.sample(fns, inp["theta"].clone(), num_samples=4, num_steps_per_sample=3, step_size=1e-4,
                                     integrator=hamiltorch.samplers.Integrator.SPLITTING, seed=4)
    want = samplers.sample(cases.don_spec(inp, "split"), inp["theta"].clone(), num_samples=4, num_steps_per_sample=3, step_size=1e-4,
                           integrator=samplers.Integrator.SPLITTING, seed=4)
    assert torch.equal(torch.stack(out), torch.stack(want))
    # NUTS driver call shape (NUTS_DeepOnets.py:289-290): dual-averaged step size during burn, burn draws dropped
    full = rshape.deeponet_closure(net, "NLL", tr, tau_list, 1.0)
    out = hamiltorch.samplers.sample(full, inp["theta"].clone(), num_samples=8, num_steps_per_sample=3, step_size=1e-4,
                                     sampler=hamiltorch.samplers.Sampler.HMC_NUTS, burn=3, debug=False, seed=2)
    assert len(out) == 5 and all(torch.isfinite(o).all() for o in out)


def test_sample_model_and_predict_model_entry_points_of_the_shim():
    """main_regression_hmc.py:115-127,153-155 on the bundled data: hamiltorch.util.flatten, sample_model, predict_model."""
    import hamiltorch

    x, y, xv, yv = synth.bnn_data()
    torch.manual_seed(0)
    net = rshape.mlp_module(1, (10, 10), 1)
    params_init = hamiltorch.util.flatten(net).clone()
    tau_list = torch.tensor([1.0 for _ in net.parameters()])
    out = hamiltorch.sample_model(net, x, y, model_loss='regression', params_init=params_init, num_samples=6, debug=0, step_size=1e-4,
                                  num_steps_per_sample=10, tau_out=400.0, normalizing_const=20, tau_list=tau_list, seed=1)
    assert len(out) == 6 and out[0].shape == (141,)
    samples = torch.stack(out)
    pred, logp = hamiltorch.predict_model(net, x=xv, y=yv, model_loss='regression', samples=samples[2:], tau_out=400.0, tau_list=tau_list)
    assert pred.shape == (4, xv.shape[0], 1) and len(logp) == 4
    oracle = cases.oc.BnnLogProb(x=xv, y=yv, widths=(10, 10), loss="regression", tau_out=400.0, prior=("tau", [1.0] * 6))
    for s, o, lp in zip(samples[2:], pred, logp):
        np.testing.assert_allclose(o.numpy(), oracle.forward(s).detach().numpy(), rtol=1e-5, atol=1e-5)
        assert float(lp) == pytest.approx(float(oracle(s).detach()), rel=1e-5)


def test_subsampling_closure_through_the_shim():
    """cfg.sample_data = True in the reference's config: the closure redraws cfg.p trunk points per call.  Through the shim the
    set-up check replays the closure's subset for the engine (and leaves Python's generator untouched), then the run follows the
    specification path draw for draw."""
    import random

    import hamiltorch

    inp, net, tr, tau_list = _don_closures()
    rshape.cfg.sample_data, rshape.cfg.p = True, 9
    try:
        fn = rshape.deeponet_closure(net, "NLL", tr, tau_list, 1.0, mean_params=inp["mu"], std_params=inp["sigma"], grad_ind=inp["ind"])
        spec = closure.spec_from_closure(fn)
        assert spec.trunk_subsample == 9
        q0 = inp["mu"][inp["ind"]].clone()
        random.seed(21)
        out = hamiltorch.samplers.sample(fn, q0, num_samples=4, num_steps_per_sample=3, step_size=1e-4, seed=6)
        random.seed(21)
        want = samplers.sample(spec, q0, num_samples=4, num_steps_per_sample=3, step_size=1e-4, seed=6)
        assert torch.equal(torch.stack(out), torch.stack(want))
    finally:
        rshape.cfg.sample_data, rshape.cfg.p = False, None


# ------------------------------------------------------------------------------------------------
# the reference's own driver, unmodified, on the GPU (needs a checkout of the original project in oracle/_ref/ or VIHMC_REFERENCE_ROOT --
# its sources are not part of this repository, so without it the test is skipped; the CPU twin of this test,
# tests/test_closure_dropin.py, runs with the oracle standing in for the engine)
# ------------------------------------------------------------------------------------------------
def test_real_reference_driver_main_vi_hmc_on_the_gpu(tmp_path):
    import importlib
    import os
    import sys

    from oracle import ref_loader

    if not ref_loader.reference_available():
        pytest.skip("original project not present (oracle/_ref/ or VIHMC_REFERENCE_ROOT)")
    saved_mods = {k: sys.modules.pop(k, None) for k in ("hamiltorch", "hamiltorch.samplers", "hamiltorch.util")}
    hamiltorch = importlib.import_module("hamiltorch")
    sys.modules["hamiltorch.util"] = hamiltorch.util
    try:
        m = ref_loader.load_script("Neural_network/VI_HMC", "main_VI_HMC", "ref_bnn_vi_hmc_gpu")
        assert m.samplers is hamiltorch.samplers           # the reference imported OUR hamiltorch, nothing was edited
        cfg = m.cfg
        mu, sigma, ind = synth.bnn_vi_artifacts(141, 40, seed=1)
        torch.save(mu, os.path.join(tmp_path, "means_flattened_synthetic"))
        torch.save(sigma, os.path.join(tmp_path, "stds_flattened_synthetic"))
        np.save(os.path.join(tmp_path, "gradient_indices_synthetic.npy"), ind)
        cfg.prior_file, cfg.prior_uid, cfg.out_dir = str(tmp_path), "synthetic", str(tmp_path) + "/"
        cfg.num_samples, cfg.L, cfg.step_size, cfg.load_prior, cfg.init_prior = 30, 20, 5e-4, False, False
        m.device = torch.device("cpu")                      # the closure's tensors stay on the host: the engine reads them out of it
        cwd = os.getcwd()
        os.chdir(os.path.join(ref_loader.REFERENCE_ROOT, "Neural_network", "VI_HMC"))   # get_data() reads ../Data
        try:
            torch.manual_seed(11)
            m.draw_hmc_samples("gpu0")
        finally:
            os.chdir(cwd)
    finally:
        for k, v in saved_mods.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
    out = np.load(tmp_path / "hmc_params_gpu0.npy")         # what the reference's np.save wrote (main_VI_HMC.py:381)
    assert out.shape == (30, 40) and out.dtype == np.float32 and np.isfinite(out).all()
    assert np.abs(out[-1] - out[0]).max() > 0               # the chain moved: the engine, not a stub, produced the samples
