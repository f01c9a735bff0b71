"""TEST INFRASTRUCTURE ONLY -- generate tests/golden/* from the REAL reference closures.

Needs a checkout of the original VI-HMC project in oracle/_ref/ (or VIHMC_REFERENCE_ROOT=<checkout>):

    python oracle/make_golden.py

Every fixture stores the inputs that cannot be regenerated from a seed, the evaluation points q, and
the reference closure's log-probability and gradient at each q (fp32, produced by the reference's own
``define_model_log_prob`` + ``torch.autograd.grad``).  Large deterministic inputs (DeepONet data and
VI artefacts) are NOT stored; they are regenerated from ``vihmc.synth`` with the recorded seeds.
Also writes the bundled BNN regression data (data, not code) into the product package.
"""
from __future__ import annotations

import os
import sys
import tempfile

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "vi-hmc_b200"))

from oracle import ref_loader  # noqa: E402
from vihmc import synth  # noqa: E402
from vihmc.spec import DeepONetArch  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")


def _grad(closure, q):
    p = q.detach().clone().requires_grad_()
    lp = closure(p)
    (g,) = torch.autograd.grad(lp.sum(), p)
    return float(lp.sum()), g.detach().numpy().copy()


def _write_artifacts(tmp, uid, mu, sigma, ind):
    torch.save(mu, os.path.join(tmp, f"means_flattened_{uid}"))
    torch.save(sigma, os.path.join(tmp, f"stds_flattened_{uid}"))
    np.save(os.path.join(tmp, f"gradient_indices_{uid}.npy"), ind)


def bnn_data_file():
    x_tr, y_tr, x_va, y_va = ref_loader.load_bnn_data()
    out = os.path.join(ROOT, "vi-hmc_b200", "vihmc", "data", "bnn_regression.npz")
    np.savez(out, x_train=x_tr.numpy(), y_train=y_tr.numpy(), x_val=x_va.numpy(), y_val=y_va.numpy())
    print("wrote", out)


SENS_CASES = [("tanh_10x10", [10, 10], "tanh", 300), ("relu_10x10", [10, 10], "relu", 77), ("sine_16x16", [16, 16], "sine", 50),
              ("tanh_32", [32], "tanh", 31)]


def bnn_sensitivity_cases():
    """Reference eval_std_dydw (Neural_network/VI/sensitivity.py:71-126: jacrev of the functional model) on synthetic VI
    means / standard deviations; stores the inputs and the reference's scores."""
    m = ref_loader.load_script("Neural_network/VI", "sensitivity", "ref_bnn_sens")
    out = {}
    for name, widths, act, n_val in SENS_CASES:
        torch.manual_seed(0)
        model = m.get_model(widths, act, True)
        D = sum(p.numel() for p in model.parameters())
        g = torch.Generator().manual_seed(len(name))
        mu = 0.5 * torch.randn(D, generator=g)
        sg = 0.01 + 0.1 * torch.rand(D, generator=g)
        x = (2 * torch.rand(n_val, 1, generator=g) - 1)
        s = m.eval_std_dydw((x, None), model, mu, sg)
        out[f"{name}/mu"], out[f"{name}/sigma"], out[f"{name}/x"], out[f"{name}/scores"] = mu.numpy(), sg.numpy(), x.numpy(), s
    path = os.path.join(GOLDEN, "bnn_sensitivity.npz")
    np.savez(path, **out)
    print("wrote", path)


DON_SENS_CASES = [
    # name, layer_width, in_branch, depth_branch, depth_trunk, output_neurons, act, [(n functions, p trunk points) per batch]
    ("tanh_small", 16, 12, 3, 4, 8, "tanh", [(6, 35)]),          # n < K: the branch Gram matrix is rank deficient
    ("relu_small", 24, 10, 3, 3, 16, "relu", [(20, 12)]),        # p < K: the trunk Gram matrix is rank deficient
    ("tanh_loader", 16, 12, 3, 4, 8, "tanh", [(1, 9), (1, 9), (1, 9)]),   # the reference's loader: batch size 1, own trunk subset
    ("tanh_shipped", 100, 101, 9, 9, 100, "tanh", [(3, 7)]),     # the shipped 172 401-parameter architecture
]


def deeponet_sensitivity_cases():
    """Reference eval_std_dydw (Operator_network/VI/sensitivity.py:61-126: jacrev of the functional DeepONet) on synthetic VI means /
    standard deviations; stores the inputs and the reference's scores."""
    m = ref_loader.load_script("Operator_network/VI", "sensitivity", "ref_don_sens")
    cfg = m.cfg
    out = {}
    for name, width, in_branch, db, dt, K, act, batches in DON_SENS_CASES:
        cfg.branch_depth, cfg.trunk_depth, cfg.activation, cfg.dataset = db, dt, act, "Burgers"
        torch.manual_seed(0)
        model = m.DeepONet(width, in_branch, 5, db, dt, K, act, impose_bc=True)
        D = sum(p.numel() for p in model.parameters())
        g = torch.Generator().manual_seed(len(name))
        mu = torch.cat([p.detach().flatten() for p in model.parameters()]) + 0.05 * torch.randn(D, generator=g)
        sg = 0.001 + 0.01 * torch.rand(D, generator=g)
        data = [(0.3 * torch.randn(n, 1, in_branch, generator=g), torch.rand(1, p, 2, generator=g)) for n, p in batches]
        s = m.eval_std_dydw(data, model, mu, sg)
        out[f"{name}/mu"], out[f"{name}/sigma"], out[f"{name}/scores"] = mu.numpy(), sg.numpy(), np.asarray(s, np.float32)
        for bi, (xb, xt) in enumerate(data):
            out[f"{name}/xb{bi}"], out[f"{name}/xt{bi}"] = xb.numpy(), xt.numpy()
        print(name, "D", D, "scores max", float(np.max(s)), "nonzero", int(np.count_nonzero(s)))
    path = os.path.join(GOLDEN, "deeponet_sensitivity.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path) // 1024, "KiB")


VI_TRAIN_CASES = [("adam_6x3", 6, 3, 1e-2, 5000), ("plateau_8x2", 8, 2, 0.3, 0)]   # name, epochs, num_ens, lr_start, lr_patience


def bnn_vi_training_cases():
    """The reference's own Bayesian_Net / train_model / validate_model / Adam / ReduceLROnPlateau loop
    (Neural_network/VI/main_regression_VI.py:75-170,:300-335) on the bundled data.  BBBLinear draws eps with
    torch.empty(size).normal_(0, 1) from the global generator, layer by layer (W then bias), draw by draw: reseeding the generator
    and replaying the same calls recovers the eps stream, which is stored next to the reference's results."""
    m = ref_loader.load_script("Neural_network/VI", "main_regression_VI", "ref_bnn_vi_train")
    cfg = m.cfg
    x_tr, y_tr, x_va, y_va = ref_loader.load_bnn_data()
    out = {}
    for name, epochs, num_ens, lr, patience in VI_TRAIN_CASES:
        torch.manual_seed(len(name))
        model = m.Bayesian_Net(cfg.priors, cfg.layer_width, cfg.input_size, cfg.output_size, cfg.activation, cfg.bias_on)
        layers = [l for l in model.net if hasattr(l, "W_mu")]
        flat = lambda attr_w, attr_b: torch.cat([torch.cat([getattr(l, attr_w).detach().flatten(), getattr(l, attr_b).detach().flatten()])
                                                 for l in layers])
        mu0, rho0 = flat("W_mu", "bias_mu").clone(), flat("W_rho", "bias_rho").clone()
        opt = m.Adam(model.parameters(), lr=lr)
        sched = m.lr_scheduler.ReduceLROnPlateau(opt, patience=patience, min_lr=1e-5)
        loss = m.metrics.ELBO()
        noise_param = torch.tensor(cfg.noise ** 2)
        hist, eps_all = [], []
        for ep in range(epochs):
            torch.manual_seed(1000 + ep)
            eps_ep = []
            for j in range(num_ens):
                eps_ep.append(torch.cat([torch.cat([torch.empty(l.W_mu.size()).normal_(0, 1).flatten(),
                                                    torch.empty(l.bias_mu.size()).normal_(0, 1)]) for l in layers]))
            eps_all.append(torch.stack(eps_ep))
            torch.manual_seed(1000 + ep)
            lr_used = opt.param_groups[0]["lr"]
            tl = m.train_model((x_tr, y_tr), model, loss, opt, x_tr.shape[0], 1, num_ens, cfg.beta_type, epoch=ep, num_epochs=None,
                               noise_param=noise_param)
            vl = m.validate_model((x_va, y_va), model, loss, x_va.shape[0], cfg.beta_type, 1, epoch=ep, num_epochs=None,
                                  noise_param=noise_param)
            sched.step(vl)
            hist.append([tl, vl, lr_used])
        out[f"{name}/mu0"], out[f"{name}/rho0"] = mu0.numpy(), rho0.numpy()
        out[f"{name}/eps"] = torch.stack(eps_all).numpy()
        out[f"{name}/mu"], out[f"{name}/rho"] = flat("W_mu", "bias_mu").numpy(), flat("W_rho", "bias_rho").numpy()
        out[f"{name}/history"] = np.asarray(hist, np.float64)
        out[f"{name}/cfg"] = np.asarray([cfg.noise ** 2, cfg.priors["prior_mu"], cfg.priors["prior_sigma"], float(cfg.beta_type), lr, patience],
                                        np.float64)
        print(name, "history", np.asarray(hist)[[0, -1]])
    path = os.path.join(GOLDEN, "bnn_vi_training.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path) // 1024, "KiB")


def deeponet_vi_training_case():
    """The reference's Bayesian_DeepONet / train_model / validate_model / Adam / ReduceLROnPlateau loop
    (Operator_network/VI/main_VI_deeponet.py:24-118,:153-165) on the small synthetic Burgers-shaped problem: two mini-batches of
    functions on a shared trunk grid, loss = NLL(mean) * train_size + beta * KL.  The eps stream is recovered by replaying the global
    generator (branch layers, trunk layers, then the output bias -- the order the forward pass draws them) and stored in the
    flat order of the deterministic net (b first)."""
    m = ref_loader.load_script("Operator_network/VI", "main_VI_deeponet", "ref_don_vi_train")
    cfg = m.cfg
    cfg.dataset, cfg.noise_type, cfg.learn_noise = "Burgers", 0, False
    arch = DeepONetArch(width_branch=16, width_trunk=16, in_branch=12, depth_branch=3, depth_trunk=4, output_neurons=8)
    x1, x2, y, theta = synth.burgers_like(arch, n_train=6, n_t=5, n_x=7, seed=0)
    n, P = x1.shape[0], x2.shape[0]
    half, epochs, num_ens, lr = n // 2, 3, 2, 1e-3
    priors = {"prior_mu": 0, "prior_sigma": 0.1, "posterior_mu_initial": (0, 0.1), "posterior_rho_initial": (-5, 0.1)}
    torch.manual_seed(5)
    model = m.Bayesian_DeepONet(priors, arch.width_branch, arch.width_trunk, arch.in_branch, arch.in_trunk, arch.depth_branch,
                                arch.depth_trunk, arch.output_neurons, arch.act, 0, 0, impose_bc=True)
    layers = [l for l in list(model.b1) + list(model.b2) if hasattr(l, "W_mu")]

    def flat(attr_w, attr_b, battr):
        return torch.cat([getattr(model, battr).detach().flatten()] +
                         [torch.cat([getattr(l, attr_w).detach().flatten(), getattr(l, attr_b).detach().flatten()]) for l in layers])
    mu0, rho0 = flat("W_mu", "bias_mu", "b_mu").clone(), flat("W_rho", "bias_rho", "b_rho").clone()
    batch = lambda lo, hi: (x1[lo:hi].unsqueeze(1), x2.unsqueeze(0).repeat(hi - lo, 1, 1), y[lo:hi])
    train_loader, valid_loader = [batch(0, half), batch(half, n)], [batch(0, n)]
    size = float(n * P)
    opt = m.Adam(model.parameters(), lr=lr)
    sched = m.lr_scheduler.ReduceLROnPlateau(opt, patience=500, min_lr=1e-5)
    loss = m.metrics.ELBO(False, 0)
    noise_param = torch.tensor(1.0)
    hist, eps_all = [], []
    for ep in range(epochs):
        torch.manual_seed(2000 + ep)
        for b in range(2):
            for j in range(num_ens):
                draws = [torch.cat([torch.empty(l.W_mu.size()).normal_(0, 1).flatten(), torch.empty(l.bias_mu.size()).normal_(0, 1)])
                         for l in layers]
                b_eps = torch.empty(model.b_mu.size()).normal_(0, 1)
                eps_all.append(torch.cat([b_eps] + draws))
        torch.manual_seed(2000 + ep)
        lr_used = opt.param_groups[0]["lr"]
        tl = m.train_model(train_loader, model, loss, opt, size, 2, num_ens, 1.0, noise_param=noise_param)
        vl = m.validate_model(valid_loader, model, loss, size, 1.0, 1, noise_param=noise_param)
        sched.step(vl)
        hist.append([tl, vl, lr_used])
    out = {"mu0": mu0.numpy(), "rho0": rho0.numpy(), "eps": torch.stack(eps_all).reshape(epochs * 2, num_ens, -1).numpy(),
           "mu": flat("W_mu", "bias_mu", "b_mu").numpy(), "rho": flat("W_rho", "bias_rho", "b_rho").numpy(),
           "history": np.asarray(hist, np.float64), "cfg": np.asarray([1.0, 0.0, 0.1, 1.0, lr, 500], np.float64)}
    path = os.path.join(GOLDEN, "deeponet_vi_training.npz")
    np.savez_compressed(path, **out)
    print("deeponet VI history", np.asarray(hist), "wrote", path, os.path.getsize(path) // 1024, "KiB")


def bnn_vi_hmc_cases():
    """Reference closure Neural_network/VI_HMC/main_VI_HMC.py:28-153 on the bundled data."""
    m = ref_loader.load_bnn_vi_hmc()
    cfg = m.cfg
    x_tr, y_tr, _, _ = ref_loader.load_bnn_data()
    cases = {}
    with tempfile.TemporaryDirectory() as tmp:
        cfg.prior_file, cfg.prior_uid = tmp, "synthetic"
        for name, d, loss, tau_out, act, load_prior in [
            ("d40_nll", 40, "NLL", 0.0025, "tanh", False),
            ("d141_nll", 141, "NLL", 0.0025, "tanh", False),
            ("d14_nll", 14, "NLL", 0.0025, "tanh", False),
            ("d70_regression", 70, "regression", 400.0, "tanh", False),
            ("d40_relu", 40, "NLL", 0.0025, "relu", False),
            ("d40_sine", 40, "NLL", 0.0025, "sine", False),
            ("d40_loadprior", 40, "NLL", 0.0025, "tanh", True),
        ]:
            mu, sigma, ind = synth.bnn_vi_artifacts(141, d, seed=1)
            _write_artifacts(tmp, "synthetic", mu, sigma, ind)
            cfg.act, cfg.load_prior, cfg.loss, cfg.tau_out = act, load_prior, loss, tau_out
            torch.manual_seed(0)
            net = m.get_model(cfg.bias)
            shapes = [w.shape for w in net.parameters()]
            numels = [w.nelement() for w in net.parameters()]
            if load_prior:
                prior_list = [mu[ind], sigma[ind]]
            else:
                prior_list = [torch.tensor(cfg.prior_var) for _ in numels]
            closure = m.define_model_log_prob(net, loss, x_tr, y_tr, numels, shapes, prior_list, tau_out,
                                              device="cpu", dt_string="golden")
            rs = np.random.RandomState(100 + d)
            qs = (mu.numpy()[ind][None, :] + sigma.numpy()[ind][None, :] * rs.randn(6, d)).astype(np.float32)
            qs[5] = (0.7 * rs.randn(d)).astype(np.float32)  # one far-from-mode point
            lps, grads = zip(*[_grad(closure, torch.from_numpy(q)) for q in qs])
            cases[name] = dict(d=d, loss=loss, tau_out=tau_out, act=act, load_prior=load_prior,
                               prior_var=cfg.prior_var, q=qs, logp=np.array(lps, np.float64),
                               grad=np.stack(grads).astype(np.float32))
    cfg.act, cfg.load_prior, cfg.loss, cfg.tau_out = "tanh", False, "NLL", 0.0025
    flat = {}
    for name, c in cases.items():
        for k, v in c.items():
            flat[f"{name}/{k}"] = np.asarray(v)
    out = os.path.join(GOLDEN, "bnn_vi_hmc_logp_grad.npz")
    np.savez_compressed(out, **flat)
    print("wrote", out, {k: float(v["logp"][0]) for k, v in cases.items()})


def _don_module_cfg(m, arch: DeepONetArch, load_prior=False):
    cfg = m.cfg
    cfg.branch_depth, cfg.trunk_depth, cfg.activation = arch.depth_branch, arch.depth_trunk, arch.act
    cfg.sample_data, cfg.load_prior = False, load_prior
    return cfg


def deeponet_cases():
    """Reference closures Operator_network/VI_HMC/main_VI_HMC_burgers.py:27-180 (VI split) and
    Operator_network/HMC/main_HMC_splitting.py:79-258 (full HMC, M=2 split) on synthetic Burgers-shaped data."""
    flat = {}
    m = ref_loader.load_deeponet_vi_hmc()
    ms = ref_loader.load_deeponet_split_hmc()
    for name, arch, n_train, n_t, n_x, frac in [
        ("small", DeepONetArch(width_branch=16, width_trunk=16, in_branch=12, depth_branch=3, depth_trunk=4,
                               output_neurons=8), 6, 5, 7, 0.25),
        ("full", DeepONetArch(), 8, 3, 11, 0.10),
    ]:
        x1, x2, y, theta = synth.burgers_like(arch, n_train=n_train, n_t=n_t, n_x=n_x, seed=0)
        mu, sigma, ind = synth.deeponet_vi_artifacts(theta, frac=frac, seed=1)
        tr_data = (x1.unsqueeze(1), x2.unsqueeze(0), y)
        # ---- VI-HMC closure (reduced vector) ----
        with tempfile.TemporaryDirectory() as tmp:
            cfg = _don_module_cfg(m, arch)
            cfg.prior_file, cfg.prior_uid = tmp, "synthetic"
            _write_artifacts(tmp, "synthetic", mu, sigma, ind)
            net = m.DeepONet(arch.width_branch, arch.width_trunk, arch.in_branch, arch.in_trunk, arch.depth_branch,
                             arch.depth_trunk, arch.act, arch.output_neurons)
            assert sum(p.nelement() for p in net.parameters()) == arch.num_params
            closure = m.define_model_log_prob(net, "NLL", tr_data, [torch.tensor(cfg.prior_var)], 1.0, device="cpu")
            rs = np.random.RandomState(7)
            d = len(ind)
            qs = (mu.numpy()[ind][None] + sigma.numpy()[ind][None] * rs.randn(3, d)).astype(np.float32)
            lps, grads = zip(*[_grad(closure, torch.from_numpy(q)) for q in qs])
            flat[f"{name}/vi/q"] = qs
            flat[f"{name}/vi/logp"] = np.array(lps, np.float64)
            flat[f"{name}/vi/grad"] = np.stack(grads).astype(np.float32)
            flat[f"{name}/vi/prior_var"] = np.asarray(cfg.prior_var)
        # ---- full-HMC closure + M=2 split closures ----
        cfgs = ms.cfg
        cfgs.branch_depth, cfgs.trunk_depth, cfgs.activation = arch.depth_branch, arch.depth_trunk, arch.act
        cfgs.sample_data, cfgs.load_prior, cfgs.dataset = False, False, "Burgers"
        net = ms.DeepONet(arch.width_branch, arch.width_trunk, arch.in_branch, arch.in_trunk, arch.depth_branch,
                          arch.depth_trunk, arch.act, arch.output_neurons)
        tau_list = [torch.tensor(cfgs.prior_var)]
        full = ms.define_model_log_prob(net, "NLL", tr_data, tau_list, 1.0, device="cpu")
        half = n_train // 2
        split_data = [(tr_data[0][i * half:(i + 1) * half], tr_data[1], tr_data[2][i * half:(i + 1) * half]) for i in range(2)]
        splits = ms.define_split_model_log_prob(net, "NLL", split_data, 2, tau_list, 1.0, device="cpu", verbose=False)
        rs = np.random.RandomState(8)
        qs = (theta.numpy()[None] + 0.01 * rs.randn(2, arch.num_params)).astype(np.float32)
        lps, grads = zip(*[_grad(full, torch.from_numpy(q)) for q in qs])
        flat[f"{name}/full/q"] = qs
        flat[f"{name}/full/logp"] = np.array(lps, np.float64)
        flat[f"{name}/full/grad"] = np.stack(grads).astype(np.float32)
        for si, sc in enumerate(splits):
            lps, grads = zip(*[_grad(sc, torch.from_numpy(q)) for q in qs])
            flat[f"{name}/split{si}/logp"] = np.array(lps, np.float64)
            flat[f"{name}/split{si}/grad"] = np.stack(grads).astype(np.float32)
        flat[f"{name}/meta"] = np.array([n_train, n_t, n_x, int(round(frac * 1000))], np.int64)
        print(name, "D", arch.num_params, "d", len(ind), "logp", flat[f"{name}/vi/logp"], flat[f"{name}/full/logp"])
    out = os.path.join(GOLDEN, "deeponet_logp_grad.npz")
    np.savez_compressed(out, **flat)
    print("wrote", out, os.path.getsize(out) // 1024, "KiB")


def deeponet_fullsize_cases():
    """BASELINE sizes (SURVEY.md 8(d) cfg3 / cfg4): N = 1000 functions, P = 10201 trunk points, D = 172 401.  The REAL reference
    closures -- VI split (Operator_network/VI_HMC/main_VI_HMC_burgers.py:27-180, d = 17 240), full HMC and the M = 2 split closures
    (Operator_network/HMC/main_HMC_splitting.py:79-258) -- evaluated with torch.autograd.grad at two points each.  Inputs come from
    vihmc.synth.burgers_like(seed=0) / deeponet_vi_artifacts(seed=1) and are NOT stored; stored: q, logp (fp64 of the fp32 result),
    grad (fp32), and an fp64 twin (oracle/closures.py at float64) of the full and VI closures at the first point for error attribution."""
    from oracle import closures as oc

    arch = DeepONetArch()
    x1, x2, y, theta = synth.burgers_like(arch, n_train=1000, n_t=101, n_x=101, seed=0)
    mu, sigma, ind = synth.deeponet_vi_artifacts(theta, frac=0.10, seed=1)
    tr_data = (x1.unsqueeze(1), x2.unsqueeze(0), y)
    flat = {}
    m = ref_loader.load_deeponet_vi_hmc()
    ms = ref_loader.load_deeponet_split_hmc()
    torch.set_num_threads(os.cpu_count() or 1)
    kw64 = dict(width_branch=arch.width_branch, width_trunk=arch.width_trunk, in_branch=arch.in_branch, in_trunk=arch.in_trunk,
                depth_branch=arch.depth_branch, depth_trunk=arch.depth_trunk, output_neurons=arch.output_neurons, act=arch.act,
                impose_bc=arch.impose_bc, loss="NLL", tau_out=1.0, prior_var=0.1 ** 2, dtype=torch.float64)
    # ---- VI-HMC closure ----
    with tempfile.TemporaryDirectory() as tmp:
        cfg = _don_module_cfg(m, arch)
        cfg.prior_file, cfg.prior_uid = tmp, "synthetic"
        _write_artifacts(tmp, "synthetic", mu, sigma, ind)
        net = m.DeepONet(arch.width_branch, arch.width_trunk, arch.in_branch, arch.in_trunk, arch.depth_branch, arch.depth_trunk,
                         arch.act, arch.output_neurons)
        closure = m.define_model_log_prob(net, "NLL", tr_data, [torch.tensor(cfg.prior_var)], 1.0, device="cpu")
        rs = np.random.RandomState(17)
        d = len(ind)
        qs = (mu.numpy()[ind][None] + sigma.numpy()[ind][None] * rs.randn(2, d)).astype(np.float32)
        lps, grads = zip(*[_grad(closure, torch.from_numpy(q)) for q in qs])
        flat["vi/q"], flat["vi/logp"], flat["vi/grad"] = qs, np.array(lps, np.float64), np.stack(grads).astype(np.float32)
        twin = oc.DeepONetLogProb(x1=tr_data[0], x2=tr_data[1], y=y, frozen=mu, sens_ind=ind, **kw64)
        lp64, g64 = _grad(twin, torch.from_numpy(qs[0]).double())
        flat["vi/logp_f64"], flat["vi/grad_f64"] = np.array([lp64], np.float64), g64.astype(np.float32)[None]
        print("fullsize vi logp", lps, "fp64 twin", lp64)
    # ---- full-HMC closure + the M = 2 split closures ----
    cfgs = ms.cfg
    cfgs.branch_depth, cfgs.trunk_depth, cfgs.activation = arch.depth_branch, arch.depth_trunk, arch.act
    cfgs.sample_data, cfgs.load_prior, cfgs.dataset = False, False, "Burgers"
    net = ms.DeepONet(arch.width_branch, arch.width_trunk, arch.in_branch, arch.in_trunk, arch.depth_branch, arch.depth_trunk,
                      arch.act, arch.output_neurons)
    tau_list = [torch.tensor(cfgs.prior_var)]
    full = ms.define_model_log_prob(net, "NLL", tr_data, tau_list, 1.0, device="cpu")
    split_data = [(tr_data[0][i * 500:(i + 1) * 500], tr_data[1], tr_data[2][i * 500:(i + 1) * 500]) for i in range(2)]
    splits = ms.define_split_model_log_prob(net, "NLL", split_data, 2, tau_list, 1.0, device="cpu", verbose=False)
    rs = np.random.RandomState(18)
    qs = (theta.numpy()[None] + 0.002 * rs.randn(2, arch.num_params)).astype(np.float32)
    lps, grads = zip(*[_grad(full, torch.from_numpy(q)) for q in qs])
    flat["full/q"], flat["full/logp"], flat["full/grad"] = qs, np.array(lps, np.float64), np.stack(grads).astype(np.float32)
    for si, sc in enumerate(splits):
        lp, g = _grad(sc, torch.from_numpy(qs[0]))
        flat[f"split{si}/logp"], flat[f"split{si}/grad"] = np.array([lp], np.float64), g.astype(np.float32)[None]
    twin = oc.DeepONetLogProb(x1=tr_data[0], x2=tr_data[1], y=y, **kw64)
    lp64, g64 = _grad(twin, torch.from_numpy(qs[0]).double())
    flat["full/logp_f64"], flat["full/grad_f64"] = np.array([lp64], np.float64), g64.astype(np.float32)[None]
    flat["meta"] = np.array([1000, 101, 101, 100], np.int64)
    print("fullsize full logp", lps, "fp64 twin", lp64, "splits", float(flat["split0/logp"][0]), float(flat["split1/logp"][0]))
    out = os.path.join(GOLDEN, "deeponet_fullsize_logp_grad.npz")
    np.savez_compressed(out, **flat)
    print("wrote", out, os.path.getsize(out) // 1024, "KiB")



N1 = dict(chains=64, burn=200, iters=2000, thin=10, L=196, eps=5e-4, tau_out=0.0025, prior_var=1.0)


def n1_start(fit, chains, seed0):
    """q0 = mu[ind] + sigma[ind] z, z from numpy keyed by the chain number (the same rule on the oracle and on the engine side)."""
    mu, sg, ind = fit["mu"].astype(np.float64), fit["sigma"].astype(np.float64), fit["ind"]
    return np.stack([mu[ind] + sg[ind] * np.random.RandomState(seed0 + c).randn(len(ind)) for c in range(chains)])


def n1_chain_statistics(pred):
    """pred [T, C, X] predictions of the thinned draws -> per-chain time averages of f and f^2, [C, X] each."""
    return pred.mean(0), (pred * pred).mean(0)


def bnn_posterior_summary():
    """Long-run reference statistics for the north-star's third correctness tier (posterior predictive mean / variance within Monte
    Carlo standard error): 64 fp64 oracle chains (oracle/bnn_batched.py -- pinned to the reference closure through
    oracle/closures.py) of the BNN VI-HMC problem at the reference's sampler settings (eps 5e-4, L 196: Neural_network/VI_HMC/config.py),
    started from the FITTED variational posterior (tests/golden/bnn_vi_fit.npz, produced on the GPU by tools/make_vi_fit_fixture.py),
    200 burn-in + 2000 iterations; stored: per-chain time averages of the prediction and its square at the 300 validation inputs
    (every 10th draw) and the acceptance decisions."""
    from oracle import bnn_batched as bb

    fit = np.load(os.path.join(GOLDEN, "bnn_vi_fit.npz"))
    x, y, xv, yv = synth.bnn_data()
    model = bb.BatchedBnn(x.numpy(), y.numpy(), fit["mu"], fit["ind"], tau_out=N1["tau_out"], prior_var=N1["prior_var"])
    q0 = n1_start(fit, N1["chains"], 9000)
    rng = np.random.default_rng(123)
    total = N1["burn"] + N1["iters"]
    keep = range(N1["burn"] + N1["thin"] - 1, total, N1["thin"])
    qf, acc, ham, kept = bb.sample(model, q0, total, N1["L"], N1["eps"], rng=rng, keep=keep)
    pred = np.stack([model.forward(k, x=xv.numpy()) for k in kept])          # [T, C, 300]
    m1, m2 = n1_chain_statistics(pred)
    out = os.path.join(GOLDEN, "bnn_posterior_summary.npz")
    np.savez_compressed(out, f_mean=m1.astype(np.float32), f_sq_mean=m2.astype(np.float32), accepted=acc[N1["burn"]:].mean(0).astype(np.float32),
                        cfg=np.array([N1[k] for k in ("chains", "burn", "iters", "thin", "L")], np.int64),
                        logp_last=model.logp_grad(qf, need_grad=False)[0])
    print("bnn posterior summary: acceptance", acc[N1["burn"]:].mean(), "pred mean range", m1.mean(0).min(), m1.mean(0).max(), "wrote", out,
          os.path.getsize(out) // 1024, "KiB")


N1_DON = dict(chains=256, burn=100, iters=1000, thin=10, L=10, eps=0.04, frac=0.25)
N1_DON_ARCH = dict(width_branch=16, width_trunk=16, in_branch=12, depth_branch=3, depth_trunk=4, output_neurons=8)


def n1_don_problem():
    """The small operator-network problem of the long-run test (the 'small' case of tests/cases.py): 6 functions x 35 trunk points,
    D = 1393, VI-HMC split with d = 348."""
    arch = DeepONetArch(**N1_DON_ARCH)
    x1, x2, y, theta = synth.burgers_like(arch, n_train=6, n_t=5, n_x=7, seed=0)
    mu, sigma, ind = synth.deeponet_vi_artifacts(theta, frac=N1_DON["frac"], seed=1)
    return arch, x1, x2, y, mu, sigma, ind


def n1_don_start(mu, sigma, ind, chains, seed0):
    mu, sg = mu.numpy().astype(np.float64), sigma.numpy().astype(np.float64)
    return np.stack([mu[ind] + sg[ind] * np.random.RandomState(seed0 + c).randn(len(ind)) for c in range(chains)])


def _n1_don_worker(c):
    from oracle import closures as oc
    from oracle import hamiltorch_restated as hr

    torch.set_num_threads(1)
    arch, x1, x2, y, mu, sigma, ind = n1_don_problem()
    closure = oc.DeepONetLogProb(x1=x1.unsqueeze(1), x2=x2.unsqueeze(0), y=y, frozen=mu, sens_ind=ind, width_branch=arch.width_branch,
                                 width_trunk=arch.width_trunk, in_branch=arch.in_branch, in_trunk=arch.in_trunk,
                                 depth_branch=arch.depth_branch, depth_trunk=arch.depth_trunk, output_neurons=arch.output_neurons,
                                 act=arch.act, impose_bc=arch.impose_bc, loss="NLL", tau_out=1.0, prior_var=0.1 ** 2, dtype=torch.float64)
    q0 = torch.from_numpy(n1_don_start(mu, sigma, ind, c + 1, 9000)[c])
    total = N1_DON["burn"] + N1_DON["iters"]
    tr = {}
    out = hr.sample(closure, q0, num_samples=total, num_steps_per_sample=N1_DON["L"], step_size=N1_DON["eps"],
                    generator=torch.Generator().manual_seed(5000 + c), trace=tr)
    # out[n] = state after iteration n (out[0] = q0, hamiltorch's storage rule with burn = 0 drops nothing but the last)
    keep = range(N1_DON["burn"] + N1_DON["thin"], total, N1_DON["thin"])
    with torch.no_grad():
        pred = torch.stack([closure.forward(out[k]) for k in keep]).reshape(len(keep), -1).numpy()     # [T, N * P]
    return pred.mean(0), (pred * pred).mean(0), float(np.mean(tr["accept"][N1_DON["burn"]:]))


def deeponet_posterior_summary():
    """The operator-network half of the third correctness tier: 64 fp64 oracle chains (oracle/closures.py::DeepONetLogProb -- pinned
    to the reference's closure by the golden vectors -- under oracle/hamiltorch_restated.py::sample) of a small DeepONet VI-HMC problem,
    100 burn-in + 1000 iterations at eps 0.04 / L 10 (acceptance ~0.85), every 10th draw; stored: per-chain time averages of the
    prediction and its square at the 6 x 35 training outputs and the acceptance rates.  One chain per process, ~3 minutes on 16 cores."""
    import multiprocessing as mp

    with mp.get_context("fork").Pool(min(16, os.cpu_count() or 1)) as pool:
        res = pool.map(_n1_don_worker, range(N1_DON["chains"]))
    m1, m2, acc = (np.stack([r[i] for r in res]) for i in range(3))
    out = os.path.join(GOLDEN, "deeponet_posterior_summary.npz")
    np.savez_compressed(out, f_mean=m1.astype(np.float32), f_sq_mean=m2.astype(np.float32), accepted=acc.astype(np.float32),
                        cfg=np.array([N1_DON[k] for k in ("chains", "burn", "iters", "thin", "L")], np.int64), eps=N1_DON["eps"])
    print("deeponet posterior summary: acceptance", acc.mean(), "wrote", out, os.path.getsize(out) // 1024, "KiB")


if __name__ == "__main__":
    os.makedirs(GOLDEN, exist_ok=True)
    if len(sys.argv) > 1:   # python oracle/make_golden.py deeponet_fullsize_cases  (one generator only)
        for fn in sys.argv[1:]:
            globals()[fn]()
        sys.exit(0)
    bnn_data_file()
    bnn_vi_hmc_cases()
    deeponet_cases()
    bnn_sensitivity_cases()
    deeponet_sensitivity_cases()
    bnn_vi_training_cases()
    deeponet_vi_training_case()
    deeponet_fullsize_cases()
    bnn_posterior_summary()
    deeponet_posterior_summary()
