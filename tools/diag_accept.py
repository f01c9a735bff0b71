import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "vi-hmc_b200"), os.path.join(ROOT, "tests")]
import numpy as np, torch
import cases
from vihmc import engine
from oracle import bnn_batched as bb
g = cases.load_golden("bnn_vi_hmc_logp_grad.npz")
case = cases.bnn_case(g, "d40_nll")
spec = cases.bnn_spec(case)
x, y, _, _ = cases.synth.bnn_data()
d, S, L, eps, Cn = case["d"], 8, 196, 5e-4, 512
for scale in (6.0, 3.0):
    rs = np.random.RandomState(17)
    mu, sg = case["mu"].numpy()[case["ind"]], case["sigma"].numpy()[case["ind"]]
    q0 = (mu[None] + sg[None] * rs.randn(Cn, d)).astype(np.float32)
    p = rs.randn(S, Cn, d).astype(np.float32)
    big = rs.rand(S, Cn) < 0.33
    p[big] *= scale
    u = rs.uniform(0.01, 1.0, size=(S, Cn)).astype(np.float32)
    res = engine.run_sampler([spec], torch.from_numpy(q0), S, L, eps, burn=0, inject_momenta=torch.from_numpy(p), inject_uniforms=torch.from_numpy(u), hamiltorch_fallback_rule=False)
    model = bb.BatchedBnn(x.numpy(), y.numpy(), case["mu"].numpy(), case["ind"], tau_out=case["tau_out"], prior_var=case["prior_var"])
    _, acc_ref, ham_ref, _ = bb.sample(model, q0.astype(np.float64), S, L, eps, momenta=p.astype(np.float64), uniforms=u.astype(np.float64))
    ham = res.hamiltonians.numpy().astype(np.float64)
    acc = res.accepted.numpy().astype(bool)
    same = np.ones(Cn,bool)
    for n in range(S):
        dH1 = np.abs(ham[n,:,1]-ham_ref[n,:,1])[same]
        dE = np.abs((ham[n,:,0]-ham[n,:,1])-(ham_ref[n,:,0]-ham_ref[n,:,1]))[same]
        print(scale, n, 'chains still identical', same.sum(), 'median |dH1|', np.median(dH1), 'p99', np.percentile(dH1,99), 'max', dH1.max(), '| energy-error diff median', np.median(dE), 'p99', np.percentile(dE,99), 'max', dE.max(), 'rej', (~acc_ref[n]).mean())
        same &= (acc[n]==acc_ref[n])
