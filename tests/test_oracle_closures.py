"""CPU: pin the oracle restatement (oracle/closures.py) against golden vectors produced by the
REAL reference closures (oracle/make_golden.py).  Tolerances: the restatement uses the same torch ops
in the same order, so fp32 agreement is to a few ulp of the ~1e5-sized log-probability."""
import os

import numpy as np
import pytest
import torch

import cases
from cases import GOLDEN
from oracle import closures as oc


@pytest.mark.parametrize("name", cases.BNN_CASES)
def test_bnn_closure_matches_reference_golden(name):
    g = cases.load_golden("bnn_vi_hmc_logp_grad.npz")
    case = cases.bnn_case(g, name)
    closure = cases.bnn_oracle(case)
    for q, lp_ref, g_ref in zip(case["q"], case["logp"], case["grad"]):
        lp, grad = oc.value_and_grad(closure, torch.from_numpy(q))
        assert abs(float(lp) - lp_ref) <= 1e-6 * abs(lp_ref)
        np.testing.assert_allclose(grad.numpy(), g_ref, rtol=1e-5, atol=1e-5 * np.abs(g_ref).max())


@pytest.mark.parametrize("name", cases.BNN_CASES)
def test_bnn_fp64_twin_brackets_fp32(name):
    """The fp64 twin attributes error: fp32 reference and fp64 oracle agree to fp32 rounding of a 1e5-sized sum."""
    g = cases.load_golden("bnn_vi_hmc_logp_grad.npz")
    case = cases.bnn_case(g, name)
    closure = cases.bnn_oracle(case, dtype=torch.float64)
    for q, lp_ref, g_ref in zip(case["q"], case["logp"], case["grad"]):
        lp, grad = oc.value_and_grad(closure, torch.from_numpy(q).double())
        assert abs(float(lp) - lp_ref) <= 2e-6 * abs(lp_ref)
        np.testing.assert_allclose(grad.numpy(), g_ref, rtol=2e-4, atol=2e-5 * np.abs(g_ref).max())


@pytest.mark.parametrize("name", ["small", "full"])
def test_deeponet_closures_match_reference_golden(name):
    g = cases.load_golden("deeponet_logp_grad.npz")
    inp = cases.don_inputs(name)
    vi = cases.don_oracle(inp, "vi")
    for q, lp_ref, g_ref in zip(g[f"{name}/vi/q"], g[f"{name}/vi/logp"], g[f"{name}/vi/grad"]):
        lp, grad = oc.value_and_grad(vi, torch.from_numpy(q))
        assert abs(float(lp) - lp_ref) <= 1e-6 * abs(lp_ref)
        np.testing.assert_allclose(grad.numpy(), g_ref, rtol=1e-5, atol=1e-5 * np.abs(g_ref).max())
    full = cases.don_oracle(inp, "full")
    splits = cases.don_oracle(inp, "split")
    for i, q in enumerate(g[f"{name}/full/q"]):
        lp, grad = oc.value_and_grad(full, torch.from_numpy(q))
        lp_ref, g_ref = g[f"{name}/full/logp"][i], g[f"{name}/full/grad"][i]
        assert abs(float(lp) - lp_ref) <= 1e-6 * abs(lp_ref)
        np.testing.assert_allclose(grad.numpy(), g_ref, rtol=1e-5, atol=1e-5 * np.abs(g_ref).max())
        for si, sc in enumerate(splits):
            lp, grad = oc.value_and_grad(sc, torch.from_numpy(q))
            lp_ref, g_ref = g[f"{name}/split{si}/logp"][i], g[f"{name}/split{si}/grad"][i]
            assert abs(float(lp) - lp_ref) <= 1e-6 * abs(lp_ref)
            np.testing.assert_allclose(grad.numpy(), g_ref, rtol=1e-5, atol=1e-5 * np.abs(g_ref).max())


def test_split_closures_sum_to_full():
    """Size-independent property: sum of the M split log-posteriors == the full log-posterior."""
    inp = cases.don_inputs("small")
    full = cases.don_oracle(inp, "full", dtype=torch.float64)
    splits = cases.don_oracle(inp, "split", dtype=torch.float64)
    q = inp["theta"].double()
    lp, grad = oc.value_and_grad(full, q)
    parts = [oc.value_and_grad(s, q) for s in splits]
    assert abs(float(lp) - sum(float(p[0]) for p in parts)) < 1e-8 * abs(float(lp))
    np.testing.assert_allclose(sum(p[1] for p in parts).numpy(), grad.numpy(), rtol=1e-9, atol=1e-9)


def test_reference_still_agrees_when_present():
    """When a checkout of the original project is present (oracle/ref_loader.py), re-run one real reference closure live."""
    from oracle import ref_loader

    if not ref_loader.reference_available():
        pytest.skip("original project not present (oracle/_ref/ or VIHMC_REFERENCE_ROOT)")
    import os
    import tempfile

    m = ref_loader.load_bnn_vi_hmc()
    g = cases.load_golden("bnn_vi_hmc_logp_grad.npz")
    case = cases.bnn_case(g, "d40_nll")
    with tempfile.TemporaryDirectory() as tmp:
        torch.save(case["mu"], os.path.join(tmp, "means_flattened_t"))
        torch.save(case["sigma"], os.path.join(tmp, "stds_flattened_t"))
        np.save(os.path.join(tmp, "gradient_indices_t.npy"), case["ind"])
        m.cfg.prior_file, m.cfg.prior_uid = tmp, "t"
        net = m.get_model(True)
        x, y, _, _ = ref_loader.load_bnn_data()
        numels = [w.nelement() for w in net.parameters()]
        shapes = [w.shape for w in net.parameters()]
        closure = m.define_model_log_prob(net, "NLL", x, y, numels, shapes,
                                          [torch.tensor(1.0)] * 6, 0.0025, device="cpu", dt_string="t")
        q = torch.from_numpy(case["q"][0]).requires_grad_()
        lp = closure(q)
        (gr,) = torch.autograd.grad(lp, q)
    assert abs(float(lp) - case["logp"][0]) <= 1e-6 * abs(case["logp"][0])
    np.testing.assert_allclose(gr.numpy(), case["grad"][0], rtol=1e-6, atol=1e-3)


def test_fullsize_golden_is_self_consistent():
    """BASELINE-size golden vectors (reference closures at N = 1000, P = 10201, D = 172 401): the M = 2 split closures add up to the
    full closure (main_HMC_splitting.py:209-258), the VI gradient is finite, and the reference's fp32 results sit within 1e-5 of the
    fp64 twin of the restatement -- which pins the restatement at this size without re-running it in the CPU suite."""
    g = np.load(os.path.join(GOLDEN, "deeponet_fullsize_logp_grad.npz"))
    full = g["full/grad"][0].astype(np.float64)
    s = g["split0/grad"][0].astype(np.float64) + g["split1/grad"][0]
    assert np.abs(full - s).max() <= 1e-6 * np.abs(full).max()
    assert abs(g["split0/logp"][0] + g["split1/logp"][0] - g["full/logp"][0]) <= 1e-6 * abs(g["full/logp"][0])
    for k in ("vi", "full"):
        a, b = g[f"{k}/grad"][0].astype(np.float64), g[f"{k}/grad_f64"][0].astype(np.float64)
        assert np.linalg.norm(a - b) <= 1e-5 * np.linalg.norm(b)
        assert abs(g[f"{k}/logp"][0] - g[f"{k}/logp_f64"][0]) <= 1e-5 * abs(g[f"{k}/logp_f64"][0])


def test_batched_bnn_oracle_matches_the_pinned_closure():
    """oracle/bnn_batched.py (numpy fp64, all chains at once: the reference statistics of the long-run posterior-parity test) against
    the per-chain torch oracle, which the golden vectors pin to the reference's closure: values, gradients, and a whole sampling run
    with the same momenta and uniforms (decisions identical, states to 1e-9)."""
    from oracle import bnn_batched as bb
    from oracle import hamiltorch_restated as hr
    from vihmc import synth

    g = cases.load_golden("bnn_vi_hmc_logp_grad.npz")
    case = cases.bnn_case(g, "d40_nll")
    x, y, _, _ = synth.bnn_data()
    model = bb.BatchedBnn(x.numpy(), y.numpy(), case["mu"].numpy(), case["ind"], tau_out=case["tau_out"], prior_var=case["prior_var"])
    closure = cases.bnn_oracle(case, dtype=torch.float64)
    q = case["q"].astype(np.float64)
    lp, gr = model.logp_grad(q)
    for i in range(len(q)):
        lp_t, g_t = oc.value_and_grad(closure, torch.from_numpy(q[i]))
        assert abs(lp[i] - float(lp_t)) <= 1e-10 * abs(float(lp_t))
        np.testing.assert_allclose(gr[i], g_t.numpy(), rtol=1e-9, atol=1e-9 * np.abs(g_t.numpy()).max())
        np.testing.assert_allclose(model.forward(q[i:i + 1])[0], closure.forward(torch.from_numpy(q[i]))[:, 0].detach().numpy(), rtol=1e-12)
    # the reference's own fp32 golden values, for good measure
    np.testing.assert_allclose(lp, case["logp"], rtol=2e-6)
    S, L, eps, Cn = 6, 7, 2e-3, 3
    rs = np.random.RandomState(4)
    p = rs.randn(S, Cn, case["d"])
    p[2] *= 40.0                                   # overshooting momenta: a real mix of accepts and rejects
    u = rs.uniform(0.05, 1.0, size=(S, Cn))
    qf, acc, ham, _ = bb.sample(model, q[:Cn], S, L, eps, momenta=p, uniforms=u)
    for c in range(Cn):
        tr = {}
        out = hr.sample(closure, torch.from_numpy(q[c]), num_samples=S, num_steps_per_sample=L, step_size=eps,
                        momenta=torch.from_numpy(p[:, c]), uniforms=torch.from_numpy(u[:, c]), trace=tr)
        assert tr["accept"] == list(acc[:, c])
        np.testing.assert_allclose(ham[:, c, 0], tr["H0"], rtol=1e-10)
        np.testing.assert_allclose(ham[:, c, 1], tr["H1"], rtol=1e-10)
    assert 0 < acc.sum() < acc.size
