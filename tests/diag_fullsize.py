"""Diagnostic (not collected by pytest): per-tensor error of the engine's BASELINE-size DeepONet gradient against the reference
golden vectors and the fp64 twin, for the path selected by the environment (VIHMC_DENSE_SIMT / VIHMC_DENSE_NOFUSE).
    python tests/diag_fullsize.py [full|vi]"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path[:0] = [os.path.dirname(HERE), os.path.join(os.path.dirname(HERE), "vi-hmc_b200"), HERE]
from vihmc import engine, synth  # noqa: E402
from vihmc.spec import DeepONetArch, LogProbSpec  # noqa: E402
from test_gpu_fullsize import _tensor_slices  # noqa: E402


def main():
    which = sys.argv[1] if len(sys.argv) > 1 else "full"
    g = np.load(os.path.join(HERE, "golden", "deeponet_fullsize_logp_grad.npz"))
    arch = DeepONetArch()
    x1, x2, y, theta = synth.burgers_like(arch, n_train=1000, n_t=101, n_x=101, seed=0)
    kw = dict(arch=arch, x=x1, x2=x2, y=y, loss="NLL", tau_out=1.0, prior_sigma_scalar=0.1)
    if which == "vi":
        mu, sigma, ind = synth.deeponet_vi_artifacts(theta, 0.10, seed=1)
        spec = LogProbSpec(frozen=mu, sens_ind=ind, **kw)
    else:
        spec = LogProbSpec(**kw)
    q = torch.from_numpy(g[f"{which}/q"])
    logp, grad = engine.logp_grad(spec, q)
    print("env", {k: v for k, v in os.environ.items() if k.startswith("VIHMC")})
    print("logp ours", logp.double().cpu().numpy(), "reference", g[f"{which}/logp"], "fp64", g[f"{which}/logp_f64"])
    got, ref, f64 = grad[0].cpu().numpy().astype(np.float64), g[f"{which}/grad"][0].astype(np.float64), g[f"{which}/grad_f64"][0].astype(np.float64)
    nr = lambda a, b: np.linalg.norm(a - b) / np.linalg.norm(b)
    print(f"whole vector: ours-vs-ref {nr(got, ref):.2e} ours-vs-f64 {nr(got, f64):.2e} ref-vs-f64 {nr(ref, f64):.2e} "
          f"max-rel {np.abs(got - ref).max() / np.abs(ref).max():.2e}")
    if which == "full":
        for name, sl in _tensor_slices(arch):
            if np.linalg.norm(f64[sl]) > 0:
                print(f"  {name:12s} |g| {np.linalg.norm(f64[sl]):10.3e}  ours-vs-f64 {nr(got[sl], f64[sl]):.2e}  ref-vs-f64 {nr(ref[sl], f64[sl]):.2e}  "
                      f"signed {np.mean(got[sl] - f64[sl]) / np.abs(f64[sl]).max():+.1e}")


if __name__ == "__main__":
    main()
