"""The ``hamiltorch`` drop-in: reference drivers run unmodified because ``samplers.sample`` recovers the log-posterior
specification from the reference's OWN closure (vihmc/closure.py).

CPU part: the reference-shaped closures of oracle/reference_shaped.py (what the GPU tests use) give, bit for bit, the
log-posteriors and gradients the original project's closures gave at the stored points (tests/golden/), and the
specification recovered from them equals the one the vihmc factories build, field by field, for the BNN VI-HMC, DeepONet
VI-HMC, DeepONet full / split and NUTS drivers.  With a checkout of the original present (oracle/ref_loader.py), its real
closures recover to the same specifications, and its ``draw_hmc_samples`` runs end to end, unmodified, through the shim
with the oracle standing in for the CUDA engine.
"""
from __future__ import annotations

import dataclasses
import os
import sys
import tempfile

import numpy as np
import pytest
import torch

import cases
from oracle import hamiltorch_restated as hr
from oracle import ref_loader, reference_shaped as rshape
from vihmc import closure, engine, samplers, synth
from vihmc.spec import DeepONetArch, LogProbSpec

needs_reference = pytest.mark.skipif(not ref_loader.reference_available(),
                                     reason="original project not present (oracle/_ref/ or VIHMC_REFERENCE_ROOT)")


def _same(a, b):
    if a is None or b is None:
        return a is None and b is None
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and np.array_equal(a, b)


def assert_specs_equal(got: LogProbSpec, want: LogProbSpec):
    assert got.arch == want.arch
    for f in ("loss", "tau_out", "prior_scale", "predict"):
        assert getattr(got, f) == getattr(want, f), f
    for f in ("x", "x2", "y", "frozen", "sens_ind", "vi_sigma"):
        assert _same(getattr(got, f), getattr(want, f)), f
    # the prior may be stored as a scalar or as a per-coordinate vector: compare what the kernels see
    d = want.d

    def prior(s):
        mu = np.zeros(d, np.float32) if s.prior_mu is None else s.prior_mu.numpy()
        sg = np.full(d, np.float32(s.prior_sigma_scalar)) if s.prior_sigma is None else s.prior_sigma.numpy()
        return mu, sg
    for a, b in zip(prior(got), prior(want)):
        np.testing.assert_array_equal(a, b)


def _write_artifacts(tmp, uid, mu, sigma, ind):
    torch.save(mu, os.path.join(tmp, f"means_flattened_{uid}"))
    torch.save(sigma, os.path.join(tmp, f"stds_flattened_{uid}"))
    np.save(os.path.join(tmp, f"gradient_indices_{uid}.npy"), ind)


def _grad(fn, q):
    p = q.detach().clone().requires_grad_()
    lp = fn(p)
    (g,) = torch.autograd.grad(lp.sum(), p)
    return float(lp.detach().sum()), g.detach()


# ------------------------------------------------------------------------------------------------
# recovered specification == factory-built specification.  Without the original project: the reference-shaped closures
# (oracle/reference_shaped.py) reproduce bit for bit what the original's closures gave at the stored points (tests/golden/,
# produced by oracle/make_golden.py on the original's bundled data, vihmc/data/bnn_regression.npz) and recover to the factory
# spec.  With a checkout of the original present (oracle/ref_loader.py), its live closures are checked as well.
# ------------------------------------------------------------------------------------------------
_BNN_GOLDEN = {(40, "NLL", "tanh", False): "d40_nll", (141, "NLL", "tanh", False): "d141_nll", (70, "regression", "tanh", False): "d70_regression",
               (40, "NLL", "relu", False): "d40_relu", (40, "NLL", "sine", False): "d40_sine", (40, "NLL", "tanh", True): "d40_loadprior"}


def _assert_reproduces(fn, qs, logps, grads):
    """fn gives exactly the stored fp32 log-posteriors and gradients of the original closure."""
    for q, lp_ref, g_ref in zip(qs, logps, grads):
        lp, g = _grad(fn, torch.from_numpy(q))
        assert lp == lp_ref
        np.testing.assert_array_equal(g.numpy(), g_ref)


@pytest.mark.parametrize("d,loss,tau_out,act,load_prior", [(40, "NLL", 0.0025, "tanh", False), (141, "NLL", 0.0025, "tanh", False),
                                                           (70, "regression", 400.0, "tanh", False), (40, "NLL", 0.0025, "relu", False),
                                                           (40, "NLL", 0.0025, "sine", False), (40, "NLL", 0.0025, "tanh", True)])
def test_bnn_reference_closure_recovers_to_the_factory_spec(d, loss, tau_out, act, load_prior):
    case = cases.bnn_case(cases.load_golden("bnn_vi_hmc_logp_grad.npz"), _BNN_GOLDEN[(d, loss, act, load_prior)])
    assert (case["d"], case["tau_out"]) == (d, tau_out)
    x_tr, y_tr, _, _ = synth.bnn_data()
    mu, sigma, ind = case["mu"], case["sigma"], case["ind"]
    torch.manual_seed(0)
    net = rshape.mlp_module(1, (10, 10), 1, act=act)
    shapes = [w.shape for w in net.parameters()]
    numels = [w.nelement() for w in net.parameters()]
    prior_list = [mu[ind], sigma[ind]] if load_prior else [torch.tensor(case["prior_var"]) for _ in numels]
    want = samplers.define_model_log_prob_bnn(net, loss, x_tr, y_tr, numels, shapes, prior_list, tau_out, params_mu=mu,
                                              params_std=sigma, grad_ind=ind, load_prior=load_prior)
    rshape.cfg.load_prior = load_prior
    try:
        fn2 = rshape.bnn_closure(net, loss, x_tr, y_tr, numels, shapes, prior_list, tau_out, params_mu=mu, params_std=sigma,
                                 grad_ind=ind, depth=1, act=act)
        assert_specs_equal(closure.spec_from_closure(fn2), want)
        _assert_reproduces(fn2, case["q"], case["logp"], case["grad"])
        if ref_loader.reference_available():
            _bnn_live(d, loss, tau_out, act, load_prior, fn2)
    finally:
        rshape.cfg.load_prior = False


def _bnn_live(d, loss, tau_out, act, load_prior, fn2):
    """The original's closure recovers to the factory spec and computes what the reference-shaped closure fn2 computes."""
    m = ref_loader.load_bnn_vi_hmc()
    cfg = m.cfg
    x_tr, y_tr, _, _ = ref_loader.load_bnn_data()
    np.testing.assert_array_equal(x_tr.numpy(), synth.bnn_data()[0].numpy())
    mu, sigma, ind = synth.bnn_vi_artifacts(141, d, seed=1)
    saved = (cfg.act, cfg.load_prior, cfg.loss, cfg.tau_out, getattr(cfg, "prior_file", None), getattr(cfg, "prior_uid", None))
    try:
        with tempfile.TemporaryDirectory() as tmp:
            cfg.prior_file, cfg.prior_uid = tmp, "synthetic"
            _write_artifacts(tmp, "synthetic", mu, sigma, ind)
            cfg.act, cfg.load_prior, cfg.loss, cfg.tau_out = act, load_prior, loss, tau_out
            torch.manual_seed(0)
            net = m.get_model(cfg.bias)
            shapes = [w.shape for w in net.parameters()]
            numels = [w.nelement() for w in net.parameters()]
            prior_list = [mu[ind], sigma[ind]] if load_prior else [torch.tensor(cfg.prior_var) for _ in numels]
            fn = m.define_model_log_prob(net, loss, x_tr, y_tr, numels, shapes, prior_list, tau_out, device="cpu", dt_string="t")
            got = closure.spec_from_closure(fn)
            want = samplers.define_model_log_prob_bnn(net, loss, x_tr, y_tr, numels, shapes, prior_list, tau_out, params_mu=mu,
                                                      params_std=sigma, grad_ind=ind, load_prior=load_prior)
            assert_specs_equal(got, want)
            q = mu[ind] + 0.1 * torch.randn(d)
            (l1, g1), (l2, g2) = _grad(fn, q), _grad(fn2, q)
            assert l1 == l2 and torch.equal(g1, g2)
    finally:
        cfg.act, cfg.load_prior, cfg.loss, cfg.tau_out, cfg.prior_file, cfg.prior_uid = saved


def _don_setup(name="small"):
    arch, n_train, n_t, n_x, frac = cases.DON_ARCHS[name]
    x1, x2, y, theta = synth.burgers_like(arch, n_train=n_train, n_t=n_t, n_x=n_x, seed=0)
    mu, sigma, ind = synth.deeponet_vi_artifacts(theta, frac=frac, seed=1)
    return arch, (x1.unsqueeze(1), x2.unsqueeze(0), y), theta, mu, sigma, ind


def _don_net(arch, in_trunk=None):
    return rshape.DeepONetModule(arch.width_branch, arch.width_trunk, arch.in_branch, arch.in_trunk if in_trunk is None else in_trunk,
                                 arch.depth_branch, arch.depth_trunk, arch.act, arch.output_neurons)


def test_deeponet_vi_reference_closure_recovers_to_the_factory_spec():
    import random

    arch, tr_data, theta, mu, sigma, ind = _don_setup()
    g = cases.load_golden("deeponet_logp_grad.npz")
    net = _don_net(arch)
    tau_list = [torch.tensor(float(g["small/vi/prior_var"]))]
    want = samplers.define_model_log_prob_deeponet(net, "NLL", tr_data, tau_list, 1.0, mean_params=mu, std_params=sigma, grad_ind=ind)
    fn2 = rshape.deeponet_closure(net, "NLL", tr_data, tau_list, 1.0, mean_params=mu, std_params=sigma, grad_ind=ind, activation=arch.act)
    assert_specs_equal(closure.spec_from_closure(fn2), want)
    _assert_reproduces(fn2, g["small/vi/q"], g["small/vi/logp"], g["small/vi/grad"])
    q = mu[ind] + 0.01 * torch.randn(len(ind))
    # cfg.sample_data: the recovered specification carries cfg.p, and the closure's value on its random subset equals the oracle's
    # on the same subset (both draw it from Python's global generator)
    rshape.cfg.sample_data, rshape.cfg.p = True, 9
    try:
        sub = closure.spec_from_closure(fn2)
        assert sub.trunk_subsample == 9
        assert_specs_equal(dataclasses.replace(sub, trunk_subsample=None), want)
        oracle = cases.oc.DeepONetLogProb(x1=tr_data[0], x2=tr_data[1], y=tr_data[2], frozen=mu, sens_ind=ind, sample_p=9,
                                          **cases._don_kwargs(arch, torch.float32))
        random.seed(4)
        a = _grad(fn2, q)
        random.seed(4)
        b = _grad(oracle, q)
        assert a[0] == b[0] and torch.equal(a[1], b[1])
        random.seed(5)
        assert _grad(fn2, q)[0] != a[0]          # another subset, another value
    finally:
        rshape.cfg.sample_data, rshape.cfg.p = False, None
    if not ref_loader.reference_available():
        return
    m = ref_loader.load_deeponet_vi_hmc()
    cfg = m.cfg
    cfg.branch_depth, cfg.trunk_depth, cfg.activation = arch.depth_branch, arch.depth_trunk, arch.act
    cfg.sample_data, cfg.load_prior = False, False
    with tempfile.TemporaryDirectory() as tmp:
        cfg.prior_file, cfg.prior_uid = tmp, "synthetic"
        _write_artifacts(tmp, "synthetic", mu, sigma, ind)
        net = m.DeepONet(arch.width_branch, arch.width_trunk, arch.in_branch, arch.in_trunk, arch.depth_branch,
                         arch.depth_trunk, arch.act, arch.output_neurons)
        tau_list = [torch.tensor(cfg.prior_var)]
        fn = m.define_model_log_prob(net, "NLL", tr_data, tau_list, 1.0, device="cpu")
    want = samplers.define_model_log_prob_deeponet(net, "NLL", tr_data, tau_list, 1.0, mean_params=mu, std_params=sigma, grad_ind=ind)
    assert_specs_equal(closure.spec_from_closure(fn), want)
    fn2 = rshape.deeponet_closure(net, "NLL", tr_data, tau_list, 1.0, mean_params=mu, std_params=sigma, grad_ind=ind, activation=arch.act)
    (l1, g1), (l2, g2) = _grad(fn, q), _grad(fn2, q)
    assert l1 == l2 and torch.equal(g1, g2)
    cfg.sample_data, old_p = True, getattr(cfg, "p", None)
    cfg.p = 9
    try:
        sub = closure.spec_from_closure(fn)
        assert sub.trunk_subsample == 9
        assert_specs_equal(dataclasses.replace(sub, trunk_subsample=None), want)
        oracle = cases.oc.DeepONetLogProb(x1=tr_data[0], x2=tr_data[1], y=tr_data[2], frozen=mu, sens_ind=ind, sample_p=9,
                                          **cases._don_kwargs(arch, torch.float32))
        random.seed(4)
        a = _grad(fn, q)
        random.seed(4)
        b = _grad(oracle, q)
        assert a[0] == b[0] and torch.equal(a[1], b[1])
    finally:
        cfg.sample_data, cfg.p = False, old_p


def test_deeponet_full_and_split_reference_closures_recover_to_the_factory_specs():
    arch, tr_data, theta, *_ = _don_setup()
    g = cases.load_golden("deeponet_logp_grad.npz")
    net = _don_net(arch)
    tau_list = [torch.tensor(float(g["small/vi/prior_var"]))]
    full = rshape.deeponet_closure(net, "NLL", tr_data, tau_list, 1.0, activation=arch.act)
    assert_specs_equal(closure.spec_from_closure(full), samplers.define_model_log_prob_deeponet(net, "NLL", tr_data, tau_list, 1.0))
    _assert_reproduces(full, g["small/full/q"], g["small/full/logp"], g["small/full/grad"])
    half = tr_data[0].shape[0] // 2
    split_data = [(tr_data[0][i * half:(i + 1) * half], tr_data[1], tr_data[2][i * half:(i + 1) * half]) for i in range(2)]
    fns = [rshape.deeponet_closure(net, "NLL", sd, tau_list, 1.0, prior_scale=2, activation=arch.act) for sd in split_data]
    wants = samplers.define_split_model_log_prob(net, "NLL", split_data, 2, tau_list, 1.0, verbose=False)
    for si, (fn, want) in enumerate(zip(fns, wants)):
        got = closure.spec_from_closure(fn)
        assert got.prior_scale == 2.0
        assert_specs_equal(got, want)
        _assert_reproduces(fn, g["small/full/q"], g[f"small/split{si}/logp"], g[f"small/split{si}/grad"])
    # a closure without the trunk feature layer (the Cone data set, main_HMC_splitting.py:118) and a 2-input trunk: carried through
    cone = rshape.deeponet_closure(_don_net(arch, in_trunk=2), "NLL", tr_data, tau_list, 1.0, activation=arch.act, impose_bc=False)
    got = closure.spec_from_closure(cone)
    assert got.arch.impose_bc is False and got.arch.in_trunk == 2
    if not ref_loader.reference_available():
        return
    ms = ref_loader.load_deeponet_split_hmc()
    cfg = ms.cfg
    cfg.branch_depth, cfg.trunk_depth, cfg.activation = arch.depth_branch, arch.depth_trunk, arch.act
    cfg.sample_data, cfg.load_prior, cfg.dataset = False, False, "Burgers"
    net = ms.DeepONet(arch.width_branch, arch.width_trunk, arch.in_branch, arch.in_trunk, arch.depth_branch,
                      arch.depth_trunk, arch.act, arch.output_neurons)
    tau_list = [torch.tensor(cfg.prior_var)]
    full = ms.define_model_log_prob(net, "NLL", tr_data, tau_list, 1.0, device="cpu")
    assert_specs_equal(closure.spec_from_closure(full), samplers.define_model_log_prob_deeponet(net, "NLL", tr_data, tau_list, 1.0))
    fns = ms.define_split_model_log_prob(net, "NLL", split_data, 2, tau_list, 1.0, device="cpu", verbose=False)
    wants = samplers.define_split_model_log_prob(net, "NLL", split_data, 2, tau_list, 1.0, verbose=False)
    for fn, want in zip(fns, wants):
        got = closure.spec_from_closure(fn)
        assert got.prior_scale == 2.0
        assert_specs_equal(got, want)
    # the Cone data set switches the trunk feature layer off (main_HMC_splitting.py:118): carried through
    cfg.dataset = "Cone"
    try:
        net5 = ms.DeepONet(arch.width_branch, arch.width_trunk, arch.in_branch, 2, arch.depth_branch, arch.depth_trunk, arch.act,
                           arch.output_neurons)
        cone = ms.define_model_log_prob(net5, "NLL", tr_data, tau_list, 1.0, device="cpu")
        got = closure.spec_from_closure(cone)
        assert got.arch.impose_bc is False and got.arch.in_trunk == 2
    finally:
        cfg.dataset = "Burgers"


def test_nuts_driver_prior_quirk_is_read_from_the_closure():
    """NUTS_DeepOnets.py:132 builds Normal(0, tau * 0.5) where every other driver uses tau ** 0.5: the recovered prior follows
    the closure, not the convention (a closure of the NUTS driver's shape; the original's own when a checkout is present)."""
    arch, tr_data, *_ = _don_setup()
    if ref_loader.reference_available():
        m = ref_loader.load_script("Operator_network/HMC", "NUTS_DeepOnets", "ref_don_nuts")
        cfg = m.cfg
        cfg.branch_depth, cfg.trunk_depth, cfg.activation = arch.depth_branch, arch.depth_trunk, arch.act
        cfg.sample_data, cfg.load_prior = False, False
        net = m.DeepONet(arch.width_branch, arch.width_trunk, arch.in_branch, arch.in_trunk, arch.depth_branch, arch.depth_trunk,
                         arch.act, arch.output_neurons)
        make = lambda *a: m.define_model_log_prob(*a, device="cpu")
    else:
        net = _don_net(arch)
        make = lambda *a: rshape.deeponet_nuts_closure(*a, activation=arch.act)
    numels = [w.nelement() for w in net.parameters()]
    shapes = [w.shape for w in net.parameters()]
    fn = make(net, "NLL", tr_data, numels, shapes, [torch.tensor(0.01) for _ in numels], 1.0)
    got = closure.spec_from_closure(fn)
    np.testing.assert_array_equal(got.prior_sigma.numpy(), np.full(arch.num_params, np.float32(0.005)))
    # value check through the oracle restatement with that prior
    oracle = cases.oc.DeepONetLogProb(x1=tr_data[0], x2=tr_data[1], y=tr_data[2], prior_var=0.005 ** 2,
                                      **{k: v for k, v in cases._don_kwargs(arch, torch.float32).items() if k != "prior_var"})
    q = 0.1 * torch.randn(arch.num_params)
    assert float(fn(q)) == pytest.approx(float(oracle(q)), rel=1e-6)


def test_not_a_reference_closure_is_refused():
    with pytest.raises(closure.ClosureError):
        closure.spec_from_closure(lambda q: -(q ** 2).sum())
    y = torch.zeros(3)

    def f(q):
        return -((q - y) ** 2).sum()
    with pytest.raises(closure.ClosureError, match="fmodel"):
        closure.spec_from_closure(f)
    with pytest.raises(TypeError):
        samplers.sample(3.0, torch.zeros(4))


# ------------------------------------------------------------------------------------------------
# the reference's driver, unmodified, through the shim (oracle stands in for the CUDA engine on this CPU box)
# ------------------------------------------------------------------------------------------------
def _oracle_of(spec: LogProbSpec):
    if spec.model_kind == 0:
        if spec.prior_mu is not None:
            prior = ("loc_scale", spec.prior_mu, spec.prior_sigma)
        else:
            sig = spec.prior_sigma.numpy().astype(np.float64)
            assert np.all(sig == sig[0])
            prior = ("sliced", [float(sig[0]) ** 2] * len(spec.arch.tensor_numels()))
        return cases.oc.BnnLogProb(x=spec.x, y=spec.y, widths=spec.arch.widths, act=spec.arch.act, last_bias=spec.arch.last_bias,
                                   loss=spec.loss, tau_out=spec.tau_out, prior=prior, prior_scale=spec.prior_scale,
                                   frozen=spec.frozen, sens_ind=spec.sens_ind)
    raise NotImplementedError


class _OracleEngine:
    """Monkeypatched over vihmc.engine: prepare / logp_grad / run_sampler answered by the CPU oracle (tests only)."""

    def __init__(self):
        self.calls = []

    def prepare(self, spec, device=None):
        return spec

    def logp_grad(self, spec, q, need_grad=True):
        fn = _oracle_of(spec)
        out = [_grad(fn, row) for row in q.reshape(-1, spec.d)]
        return torch.tensor([o[0] for o in out]), torch.stack([o[1] for o in out])

    def run_sampler(self, specs, q0, num_samples, num_steps, step_size, burn=0, seed=0, **kw):
        self.calls.append(dict(spec=specs[0], q0=q0.clone(), num_samples=num_samples, num_steps=num_steps, step_size=step_size,
                               burn=burn, seed=seed, kw=kw))
        fn = _oracle_of(specs[0])
        torch.manual_seed(seed)
        out = hr.sample(fn, q0[0], num_samples=num_samples, num_steps_per_sample=num_steps, step_size=step_size, burn=burn)
        s = torch.stack(out).unsqueeze(1)
        return engine.SampleResult(s, torch.ones(num_samples, 1, dtype=torch.uint8), None, None, None)


@needs_reference
def test_reference_bnn_vi_hmc_driver_runs_unmodified_through_the_shim(monkeypatch, tmp_path):
    import importlib

    # earlier tests may have left ref_loader's inert hamiltorch stub in sys.modules: import the drop-in package itself
    saved_mods = {k: sys.modules.pop(k, None) for k in ("hamiltorch", "hamiltorch.samplers", "hamiltorch.util")}
    hamiltorch = importlib.import_module("hamiltorch")
    assert os.path.dirname(hamiltorch.__file__).endswith(os.path.join("vi-hmc_b200", "hamiltorch"))
    sys.modules["hamiltorch.util"] = hamiltorch.util
    fake = _OracleEngine()
    for name in ("prepare", "logp_grad", "run_sampler"):
        monkeypatch.setattr(engine, name, getattr(fake, name))
    try:
        m = ref_loader.load_script("Neural_network/VI_HMC", "main_VI_HMC", "ref_bnn_vi_hmc_shim")
        assert m.samplers is hamiltorch.samplers           # the reference imported OUR hamiltorch, nothing was edited
        cfg = m.cfg
        mu, sigma, ind = synth.bnn_vi_artifacts(141, 40, seed=1)
        _write_artifacts(str(tmp_path), "synthetic", mu, sigma, ind)
        cfg.prior_file, cfg.prior_uid, cfg.out_dir = str(tmp_path), "synthetic", str(tmp_path) + "/"
        cfg.num_samples, cfg.L, cfg.step_size, cfg.load_prior, cfg.init_prior = 6, 5, 5e-4, False, False   # shipped: start at the net's own init
        m.device = torch.device("cpu")                      # set under __main__ in the script (main_VI_HMC.py:449)
        cwd = os.getcwd()
        os.chdir(os.path.join(ref_loader.REFERENCE_ROOT, "Neural_network", "VI_HMC"))   # get_data() reads ../Data
        try:
            torch.manual_seed(11)
            m.draw_hmc_samples("run0")
            m.draw_hmc_samples("run1")
        finally:
            os.chdir(cwd)
    finally:
        for k, v in saved_mods.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
    assert len(fake.calls) == 2
    c = fake.calls[0]
    assert (c["num_samples"], c["num_steps"], c["step_size"], c["burn"]) == (6, 5, 5e-4, 0)
    assert c["spec"].d == 40 and c["spec"].D == 141 and c["spec"].loss == cfg.loss and c["spec"].tau_out == cfg.tau_out
    assert c["q0"].shape == (1, 40)
    assert fake.calls[0]["seed"] != fake.calls[1]["seed"]            # successive chains differ, as with the global generator
    out = np.load(tmp_path / "hmc_params_run0.npy")                   # what the reference's np.save wrote (main_VI_HMC.py:381)
    assert out.shape == (6, 40) and out.dtype == np.float32
