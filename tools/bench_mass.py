"""Diagonal mass (hamiltorch's 1-D inv_mass) against the identity mass, timed in the same process, alternating the two.

  (a) persistent BNN kernel at cfg2 (1024 chains, d = 40 of D = 141, L = 196, eps 5e-4), inv_mass = sigma_VI[ind]^2:
      chain-gradient-evaluations per second;
  (b) the general sampler's fused leapfrog update at 256 chains x d = 172 401: GB/s of the algorithmic 20 d bytes per chain;
  (c) cfg2 under Sampler.HMC_NUTS (dual averaging over the burn-in) with each mass: adapted step size, acceptance, bulk-ESS/s
      with split-R-hat beside it (an ESS figure means little while R-hat is above 1.05).

One JSON line per measurement on stdout (and appended to --out), each with the GPU name and power limit.
    python tools/bench_mass.py [--out profiles/r03_mass.jsonl]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "vi-hmc_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402  (cfg2 problem and start points)
from vihmc import diagnostics, engine  # noqa: E402


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                            text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        pl = f"unknown ({e})"
    return {"gpu": name, "power_limit": pl}


def timed(fn, reps=1):
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    start.record()
    for _ in range(reps):
        fn()
    end.record()
    torch.cuda.synchronize()
    return start.elapsed_time(end) / 1e3


def emit(rec, out):
    line = json.dumps(rec)
    print(line, flush=True)
    if out:
        with open(out, "a") as f:
            f.write(line + "\n")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()
    info = gpu_info()
    spec, mu, sigma, ind = bench.build_spec()
    prep = engine.prepare(spec)
    m_vi = (torch.as_tensor(sigma)[ind].float() ** 2).cuda()

    # (a) persistent kernel, cfg2
    C, L, eps, S = bench.CHAINS_PER_GPU, bench.L_STEPS, bench.STEP_SIZE, 40
    q0 = bench.initial_states(mu, sigma, ind, C, 0).cuda()
    run = {"identity": lambda: engine.run_sampler([prep], q0, S, L, eps, seed=1, diagnostics=False, to_host=False),
           "mass": lambda: engine.run_sampler([prep], q0, S, L, eps, seed=1, diagnostics=False, to_host=False, inv_mass=m_vi)}
    for f in run.values():
        f()
    times = {k: [] for k in run}
    for _ in range(args.rounds):
        for k, f in run.items():
            times[k].append(timed(f, reps=3) / 3)
    rate = {k: C * S * (L + 1) / float(np.median(v)) for k, v in times.items()}
    emit({**info, "bench": "persistent_cfg2", "chains": C, "d": 40, "L": L, "num_samples": S,
          "chain_grad_evals_per_s": rate, "ratio_mass_over_identity": rate["mass"] / rate["identity"],
          "seconds_per_call": {k: sorted(v) for k, v in times.items()}}, args.out)

    # (b) general fused update at the DeepONet size
    C2, d2, iters = 256, 172401, 200
    g = torch.Generator(device="cuda").manual_seed(0)
    q = torch.randn(C2, d2, device="cuda", generator=g)
    p = torch.randn(C2, d2, device="cuda", generator=g)
    gr = torch.randn(C2, d2, device="cuda", generator=g) * 1e-3
    m = torch.rand(d2, device="cuda", generator=g) + 0.5
    ups = {"identity": lambda: [engine.leapfrog_update(q, p, gr, 1e-6, 1.0, 1.0) for _ in range(iters)],
           "mass": lambda: [engine.leapfrog_update(q, p, gr, 1e-6, 1.0, 1.0, inv_mass=m) for _ in range(iters)]}
    for f in ups.values():
        f()
    ut = {k: [] for k in ups}
    for _ in range(args.rounds):
        for k, f in ups.items():
            ut[k].append(timed(f))
    gbs = {k: 20.0 * d2 * C2 * iters / float(np.median(v)) / 1e9 for k, v in ut.items()}
    emit({**info, "bench": "update_kernel", "chains": C2, "d": d2, "algorithmic_bytes_per_chain_step": 20 * d2, "GB_per_s": gbs,
          "ratio_mass_over_identity": gbs["mass"] / gbs["identity"], "working_set_MB": 3 * C2 * d2 * 4 / 1e6}, args.out)

    # (c) dual averaging with each mass at cfg2
    S3, burn = 600, 200
    for name, mm in (("identity", None), ("mass", m_vi)):
        f = lambda: engine.run_sampler([prep], q0, S3, L, eps, burn=burn, adapt_step_size=True, seed=2, to_host=False, inv_mass=mm)
        torch.cuda.synchronize()
        box = {}
        t = timed(lambda: box.__setitem__("r", f()))
        res = box["r"]
        draws = res.samples[1:].float()
        summ = diagnostics.summarize(draws.cpu())
        acc = float(res.accepted[burn + 1:].float().mean())
        emit({**info, "bench": "nuts_cfg2", "mass": name, "chains": C, "num_samples": S3, "burn": burn, "L": L, "eps0": eps,
              "adapted_step_size_median": float(res.step_sizes.median()), "acceptance_post_burn": acc, "seconds": t,
              "bulk_ess_min": summ["ess_bulk_min"], "bulk_ess_median": summ["ess_bulk_median"],
              "bulk_ess_median_per_s": summ["ess_bulk_median"] / t, "rhat_max": summ["rhat_max"], "rhat_median": summ["rhat_median"]},
             args.out)


if __name__ == "__main__":
    main()
