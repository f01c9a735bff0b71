#!/usr/bin/env python
"""bench.py -- chain-grad-evals/sec and ESS/sec of the VI-HMC hot path on B200 (BASELINE.json metric).

Headline workload (N=1): BASELINE.json configs[1] -- Neural_network/VI_HMC: BNN 1-10-10-1 tanh on the bundled
20-point set, HMC over the VI-selected subset (d=40 of D=141, synthetic artefacts of SURVEY.md 8(d)),
step_size 5e-4, L=196, NLL tau_out=0.0025, 1024 chains per GPU (weak scaling: chains sharded, no
data-path collective).  One STEP = one HMC iteration (momentum draw, H0, L leapfrog steps, H1,
Metropolis test, store) of all chains = L+1 = 197 log-posterior gradient evaluations per chain.
`value` = median over 7 timed launches of `--steps` iterations each.

Further legs in the same JSON line (all independent of --steps):
  ess      ESS/sec, the metric's second half: BNN chains started from a FITTED variational posterior (vihmc.vi.train_bbb ->
           vihmc.sensitivity -> the 40 most sensitive coordinates), burn-in, then a timed run; rank-normalised split-R-hat and
           bulk-ESS over thinned draws, pooled over all ranks' chains (NCCL all-gather of the thinned draws when N > 1)
  configs  cfg3 (N = 1): BASELINE configs[2], DeepONet full HMC, 256 chains, N=1000 x P=10201, D=172401, L=7, eps=1e-4 as
           Operator_network/HMC/config_splitting.py states: device value, e2e, roofline against a MEASURED TF32 peak,
           and the reference's CPU path on this box in both modes BASELINE.md section 3 names
           cfg4 / cfg5 (N > 1): DeepONet VI-HMC sharded over the GPUs incl. the NCCL gather + global split-R-hat in the
           e2e clock, and the data-sharded wide BNN (4x512, 100k rows, gradient all-reduce per evaluation: strong scaling)

  python bench.py [--gpus N] [--steps K] [--warmup W]         our CUDA engine
  python bench.py --impl reference [--steps K] [--warmup W]   the reference's CPU path (oracle port)

Prints ONE JSON line (rank 0).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "vi-hmc_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

METRIC, UNIT = "chain-grad-evals/sec", "chain-grad-evals/s"
_REAL_STDOUT_FD = None               # set when fd 1 is redirected (multi-GPU runs, see run_ours)
CHAINS_PER_GPU = 1024
D_SAMPLED, STEP_SIZE, L_STEPS, TAU_OUT = 40, 5e-4, 196, 0.0025
WAVEFRONTS_PER_EVAL = 213.0   # shared-memory pipe cycles per chain-grad-eval of mlp_small_sample_kernel<10,1,3> (ncu, profiles/r02_summary.md F)
FLOP_PER_GRAD_EVAL = 14_000          # SURVEY.md 8(d): 2*[3*N*sum(in*out) - N*in_1*out_1], N=20, 1-10-10-1
REF_EVALS_PER_STEP = 16              # reference arm: bounded sample = 16 grad-evals per chain per step
REPS = 7                             # timed launches of the headline leg; value = their median
WORKLOAD = "bnn_vi_hmc cfg2: 1-10-10-1 tanh, N=20, d=40 of D=141, L=196, eps=5e-4, NLL v=0.0025, 1024 chains/GPU"
# cfg3: Operator_network/HMC/config_splitting.py (step_size 1e-4, L = int(pi 0.0214^2 / 2e-4) = 7, N_train 1000, p 10201)
DON_CHAINS, DON_N, DON_NT, DON_NX, DON_L, DON_EPS, DON_SAMPLES = 256, 1000, 101, 101, 7, 1e-4, 3
DON_GFLOP = 11.557882                # SURVEY.md 8(d): fwd 3.863 + bwd 7.695 GFLOP per chain-grad-eval
DON_OUT_SCALE = 0.39                 # last branch AND last trunk layer of the teacher scaled by 0.39: targets in the +-0.2 range SURVEY 8(d)
                                     # specifies (rms 0.18); measured (tools/explore_don_stability.py, profiles/r02_summary.md): the
                                     # reference's eps = 1e-4 / L = 7 is then a stable leapfrog (acceptance 0.86), whereas the unscaled
                                     # teacher (outputs of rms 1.3) is stable only below 3e-5
DON_WORKLOAD = ("deeponet_full_hmc cfg3: branch 101-100x8-100, trunk 5-100x8-100 tanh, D=d=172401, N=1000 functions x P=10201 "
                "trunk points (synthetic Burgers-shaped, targets in +-0.2), NLL v=1.0, prior_var 0.01, L=7, eps=1e-4, 256 chains")


def build_spec():
    import numpy as np
    import torch
    from vihmc import synth
    from vihmc.spec import LogProbSpec, sliced_prior_sigma

    x, y, _, _ = synth.bnn_data()
    arch = synth.bnn_arch()
    mu, sigma, ind = synth.bnn_vi_artifacts(arch.num_params, D_SAMPLED, seed=1)
    sig = sliced_prior_sigma(D_SAMPLED, arch.tensor_numels(), [1.0] * 6)
    spec = LogProbSpec(arch=arch, x=x, y=y, loss="NLL", tau_out=TAU_OUT, prior_sigma=torch.from_numpy(sig.astype(np.float32)),
                       frozen=mu, sens_ind=ind, vi_sigma=sigma)
    return spec, mu, sigma, ind


def initial_states(mu, sigma, ind, chains, chain0):
    """q0 = mu[ind] + sigma[ind] * eps_c, eps_c from numpy keyed by the global chain id."""
    import numpy as np
    import torch

    out = np.empty((chains, len(ind)), dtype=np.float32)
    m, s = mu.numpy()[ind], sigma.numpy()[ind]
    for c in range(chains):
        out[c] = m + s * np.random.RandomState(1000 + chain0 + c).randn(len(ind))
    return torch.from_numpy(out)


def don_problem():
    """cfg3 inputs: synthetic Burgers-shaped data (SURVEY 8(d)), the full-HMC spec and start points next to the teacher."""
    import numpy as np
    import torch
    from vihmc import synth
    from vihmc.spec import DeepONetArch, LogProbSpec

    arch = DeepONetArch()
    x1, x2, y, theta = synth.burgers_like(arch, n_train=DON_N, n_t=DON_NT, n_x=DON_NX, seed=0, out_scale=DON_OUT_SCALE, trunk_scale=DON_OUT_SCALE)
    spec = LogProbSpec(arch=arch, x=x1, x2=x2, y=y, loss="NLL", tau_out=1.0, prior_sigma_scalar=0.1)
    return arch, spec, theta


def don_starts(theta, chains, chain0=0):
    import numpy as np
    import torch

    out = np.empty((chains, theta.numel()), dtype=np.float32)
    for c in range(chains):
        out[c] = theta.numpy() + 0.001 * np.random.RandomState(5000 + chain0 + c).randn(theta.numel())
    return torch.from_numpy(out)


# ------------------------------------------------------------------------------------------------
# clocks sampling during the timed region (NVML; falls back to nvidia-smi)
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """NVML is initialised and the first sample taken synchronously in __enter__ (nvmlInit can take longer than the whole
    timed region on a fresh box); the thread then samples every 2 ms until __exit__, which takes a last sample itself."""

    _NAMES = None

    def __init__(self, index):
        self.index, self.samples, self.reasons, self.stop = index, [], set(), threading.Event()
        self.max_mhz = None
        self.nv = self.h = None
        self.thread = threading.Thread(target=self._run, daemon=True)

    def _sample(self):
        nv = self.nv
        self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
        mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
        for bit, nm in self._names.items():
            if mask & bit:
                self.reasons.add(nm)

    def _run(self):
        try:
            while not self.stop.is_set():
                self._sample()
                time.sleep(0.002)
        except Exception as e:  # pragma: no cover
            self.reasons.add(f"clock_sampling_failed:{type(e).__name__}")

    def __enter__(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            self.nv, self.h = nv, nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)
            self._names = {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                           nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                           nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                           nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap"}
            self._sample()
            self.thread.start()
        except Exception as e:  # pragma: no cover
            self.reasons.add(f"clock_sampling_failed:{type(e).__name__}")
        return self

    def __exit__(self, *a):
        self.stop.set()
        if self.thread.is_alive():
            self.thread.join(timeout=2)
        try:
            if self.nv is not None:
                self._sample()
        except Exception:  # pragma: no cover
            pass

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# ------------------------------------------------------------------------------------------------
# reference arm: the reference's CPU path (torch-eager closure + restated hamiltorch leapfrog)
# ------------------------------------------------------------------------------------------------
def _ref_worker(idx, steps, warmup, barrier, out):
    import torch
    torch.set_num_threads(1)
    from oracle import closures as oc
    from oracle import hamiltorch_restated as hr

    spec, mu, sigma, ind = build_spec()
    closure = oc.BnnLogProb(x=spec.x, y=spec.y, widths=(10, 10), act="tanh", loss="NLL", tau_out=TAU_OUT,
                            prior=("sliced", [1.0] * 6), frozen=mu, sens_ind=ind)
    q = initial_states(mu, sigma, ind, 1, idx)[0]
    g = torch.Generator().manual_seed(idx)
    for _ in range(warmup):
        q, _ = hr.leapfrog(q, torch.randn(q.shape, generator=g), closure, REF_EVALS_PER_STEP - 1, STEP_SIZE)
    barrier.wait()
    t0 = time.perf_counter()
    for _ in range(steps):
        q, _ = hr.leapfrog(q, torch.randn(q.shape, generator=g), closure, REF_EVALS_PER_STEP - 1, STEP_SIZE)
    out[idx] = time.perf_counter() - t0
    barrier.wait()


def run_reference(steps, warmup, n_gpus):
    """One chain per host core (torch threads = 1), all cores in parallel -- the better CPU mode for this
    2-3 ms, dispatch-bound closure (BASELINE.md section 3)."""
    if int(os.environ.get("RANK", "0")) != 0:
        return None
    import multiprocessing as mp

    cores = len(os.sched_getaffinity(0))
    ctx = mp.get_context("fork")
    barrier = ctx.Barrier(cores + 1)
    out = ctx.Array("d", cores)
    procs = [ctx.Process(target=_ref_worker, args=(i, steps, warmup, barrier, out)) for i in range(cores)]
    for p in procs:
        p.start()
    barrier.wait()
    t0 = time.perf_counter()
    barrier.wait()
    wall = time.perf_counter() - t0
    for p in procs:
        p.join()
    evals = cores * steps * REF_EVALS_PER_STEP
    value = evals / wall
    sample = (f"{cores} processes x 1 chain x {steps} steps x {REF_EVALS_PER_STEP} grad-evals "
              f"(leapfrog segments of the cfg2 trajectory), torch-eager closure + autograd.grad")
    return {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": n_gpus, "steps": steps, "warmup": warmup,
        "ms_per_step": 1e3 * wall / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": WORKLOAD + f"; reference arm: a step is a bounded sample of the same trajectory -- a {REF_EVALS_PER_STEP}-gradient-"
                               "evaluation leapfrog segment per chain instead of all 197 (throughput per evaluation is what is compared)",
                   "step": f"{REF_EVALS_PER_STEP} grad-evals per chain, one chain per core"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }


def _don_ref_worker(idx, evals, threads, barrier, out):
    """cfg3 on the CPU: the restated DeepONet closure (oracle/closures.py, pinned to the reference's closure by the golden vectors)
    + hamiltorch's params_grad, `evals` gradient evaluations of one chain."""
    import torch
    torch.set_num_threads(threads)
    from oracle import closures as oc

    arch, spec, theta = don_problem()
    closure = oc.DeepONetLogProb(x1=spec.x.unsqueeze(1), x2=spec.x2.unsqueeze(0), y=spec.y)
    q = don_starts(theta, 1, idx)[0]
    oc.value_and_grad(closure, q)          # warm-up (allocator, thread pool)
    barrier.wait()
    t0 = time.perf_counter()
    for _ in range(evals):
        _, g = oc.value_and_grad(closure, q)
        q = q + 1e-4 * g * 1e-6            # keep the arguments changing (no caching anywhere)
    out[idx] = time.perf_counter() - t0
    barrier.wait()


def run_reference_don(mode, evals):
    """The reference's CPU path for cfg3 in the two modes BASELINE.md section 3 names: 'intra' = one chain, all cores as
    intra-op threads; 'procs' = one chain per process with one thread each, all cores."""
    import multiprocessing as mp

    cores = len(os.sched_getaffinity(0))
    nproc, threads = (1, cores) if mode == "intra" else (cores, 1)
    ctx = mp.get_context("fork")
    barrier = ctx.Barrier(nproc + 1)
    out = ctx.Array("d", nproc)
    procs = [ctx.Process(target=_don_ref_worker, args=(i, evals, threads, barrier, out)) for i in range(nproc)]
    for p in procs:
        p.start()
    barrier.wait()
    t0 = time.perf_counter()
    barrier.wait()
    wall = time.perf_counter() - t0
    for p in procs:
        p.join()
    return {"value": nproc * evals / wall, "unit": UNIT, "cores": cores, "kind": "port", "mode": mode,
            "sample": f"{nproc} process(es) x {threads} torch thread(s) x {evals} gradient evaluations of one cfg3 chain each "
                      f"(N=1000, P=10201, D=172401), torch-eager closure + autograd.grad, {wall:.1f} s"}


def _subprocess_json(args, timeout):
    r = subprocess.run([sys.executable, os.path.abspath(__file__)] + args, capture_output=True, text=True, timeout=timeout,
                       env={**os.environ, "RANK": "0", "WORLD_SIZE": "1", "CUDA_VISIBLE_DEVICES": ""})
    return json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])


def cpu_baseline_leg():
    """Bounded CPU sample for our arm's JSON line: run the reference arm in a fresh process (no CUDA context)."""
    try:
        return _subprocess_json(["--impl", "reference", "--steps", "700", "--warmup", "3"], 600)["cpu_baseline"]   # ~10 s of CPU work
    except Exception as e:  # pragma: no cover
        return {"value": None, "unit": UNIT, "cores": None, "kind": "port", "sample": f"failed: {e}"}


def don_cpu_baseline_leg():
    out = {}
    for mode, evals in (("intra", 150), ("procs", 16)):   # ~8 s each on 16 cores
        try:
            out[mode] = _subprocess_json(["--impl", "reference-cfg3", "--mode", mode, "--steps", str(evals)], 900)
        except Exception as e:  # pragma: no cover
            out[mode] = {"value": None, "unit": UNIT, "kind": "port", "mode": mode, "sample": f"failed: {e}"}
    return out


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def measure_tf32_peak(dev, seconds=2.0):
    """cuBLAS TF32 (torch.matmul with allow_tf32) on 8192^3 fp32 operands: best of 10 (burst) and back to back for `seconds`
    (sustained) -- the same recipe MEASURED_PEAKS.json uses for bf16; the denominator of the tensor-pipe rooflines."""
    import torch

    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        n = 8192
        a = torch.randn(n, n, device=dev)
        b = torch.randn(n, n, device=dev)
        c = torch.empty(n, n, device=dev)
        for _ in range(3):
            torch.matmul(a, b, out=c)
        torch.cuda.synchronize()
        best = 1e9
        for _ in range(10):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            torch.matmul(a, b, out=c)
            e1.record()
            torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        reps = max(10, int(seconds * 1e3 / best))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            torch.matmul(a, b, out=c)
        e1.record()
        torch.cuda.synchronize()
        flop = 2.0 * n ** 3
        return {"tf32_tflops_burst": flop / (best * 1e-3) / 1e12, "tf32_tflops_sustained": flop * reps / (e0.elapsed_time(e1) * 1e-3) / 1e12,
                "how": f"torch.matmul fp32 8192^3 with allow_tf32 (cuBLAS): best of 10 / {reps} back to back"}
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old


def ess_leg(dev, rank, world, dist):
    """ESS/sec at the reference's sampler settings (eps 5e-4, L 196) from a fitted start.  See the module docstring."""
    import numpy as np
    import torch
    from vihmc import diagnostics, engine, samplers, sensitivity, synth, vi
    from vihmc.spec import LogProbSpec, MLPArch

    BURN, TIMED, THIN = 2000, 5000, 10
    x, y, xv, yv = synth.bnn_data()
    arch = MLPArch(in_dim=1, widths=(10, 10), out_dim=1, act="tanh", last_bias=True)
    mk = lambda a_, b_: LogProbSpec(arch=arch, x=a_, y=b_, loss="NLL", tau_out=0.05 ** 2, prior_sigma_scalar=1.0)
    t0 = time.perf_counter()
    fit = vi.train_bbb(mk(x, y), mk(xv, yv), epochs=10_000, num_ens=10, lr_start=1e-2, lr_patience=5000, seed=0)
    scores = sensitivity.eval_std_dydw((xv, None), arch, fit.best_mu, fit.best_sigma)
    ind = np.sort(np.argsort(-np.asarray(scores))[:D_SAMPLED]).astype(np.int64)
    mu, sigma = fit.best_mu, fit.best_sigma
    numels = arch.tensor_numels()
    spec = samplers.define_model_log_prob_bnn(arch, "NLL", x, y, numels, None, [torch.tensor(1.0) for _ in numels], TAU_OUT,
                                              params_mu=mu, params_std=sigma, grad_ind=ind)
    fit_s = time.perf_counter() - t0
    chain0 = rank * CHAINS_PER_GPU
    q0 = initial_states(mu, sigma, ind, CHAINS_PER_GPU, chain0).to(dev)
    prep = engine.prepare(spec, dev)
    kw = dict(chain_offset=chain0, diagnostics=True, to_host=False, hamiltorch_fallback_rule=False)
    burn = engine.run_sampler([prep], q0, BURN, L_STEPS, STEP_SIZE, burn=BURN - 2, seed=11, **kw)
    q1 = burn.samples[-1].contiguous()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    res = engine.run_sampler([prep], q1, TIMED, L_STEPS, STEP_SIZE, burn=0, seed=12, **kw)
    e1.record()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1) * 1e-3], device=dev)
    draws, lp = res.samples[::THIN].contiguous(), res.logp[::THIN].contiguous()
    acc = res.accepted.float().mean().reshape(1)
    tg0 = time.perf_counter()
    if world > 1:   # pool the thinned draws of every rank's chains on all ranks (NCCL all-gather), timing = max over ranks
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dl = [torch.empty_like(draws) for _ in range(world)]
        ll = [torch.empty_like(lp) for _ in range(world)]
        dist.all_gather(dl, draws)
        dist.all_gather(ll, lp)
        dist.all_reduce(acc, op=dist.ReduceOp.SUM)
        acc /= world
        draws, lp = torch.cat(dl, 1), torch.cat(ll, 1)
    summ = diagnostics.summarize(draws, logp=lp) if rank == 0 else None
    torch.cuda.synchronize()
    gather_diag_s = time.perf_counter() - tg0
    if rank != 0:
        return None
    secs = float(t.item())
    return {"definition": "bulk-ESS, rank-normalised, split chains (Vehtari et al. 2021); min / median over the d sampled coordinates, chains "
                          "of all ranks pooled; per second of the device-timed sampling run (max over ranks)",
            "start": f"fitted variational posterior: vihmc.vi.train_bbb (10k epochs x 10 draws) -> vihmc.sensitivity scores -> the {D_SAMPLED} "
                     f"most sensitive of 141 weights, q0 = mu + sigma z ({fit_s:.1f} s incl. selection)",
            "chains": int(summ["chains"]), "burn_in_iterations": BURN, "timed_iterations": TIMED, "thin": THIN,
            "post_burn_draws_per_chain": int(summ["draws"]), "seconds": secs, "acceptance_rate": float(acc.item()),
            "rhat_max": float(summ["rhat_max"]), "rhat_median": float(summ["rhat_median"]), "rhat_logp": float(summ["rhat_logp"]),
            "ess_bulk_min": float(summ["ess_bulk_min"]), "ess_bulk_median": float(summ["ess_bulk_median"]),
            "ess_bulk_logp": float(summ["ess_bulk_logp"]),
            "ess_min_per_sec": float(summ["ess_bulk_min"]) / secs, "ess_median_per_sec": float(summ["ess_bulk_median"]) / secs,
            "stationary": bool(summ["rhat_max"] < 1.01),
            "gather_and_diagnostics_seconds": gather_diag_s,
            "note": "the posterior over the selected BNN weights is multi-modal: between 25k and 150k iterations of 1024 chains the "
                    "rank-normalised split-R-hat stays at 2.3-2.6 while the mean log-posterior still drifts (profiles/r02_ess2.log), so no "
                    "budget a bench can afford reaches R-hat < 1.01 at the reference's eps / L; the ESS is reported as measured, with its R-hat"}


def don_leg(dev, peaks_tf32, skip_cpu):
    """cfg3 (BASELINE configs[2]): DeepONet full HMC on one GPU -- device-timed, end to end, roofline, CPU baseline."""
    import torch
    from vihmc import engine, samplers

    arch, spec, theta = don_problem()
    q0_host = don_starts(theta, DON_CHAINS)
    prep = engine.prepare(spec, dev)
    q0 = q0_host.to(dev)
    evals = DON_CHAINS * DON_SAMPLES * (DON_L + 1)
    engine.run_sampler([prep], q0, 1, 1, DON_EPS, to_host=False)             # warm-up: workspace, kernel attributes
    torch.cuda.synchronize()
    runs_ms = []
    for _ in range(3):            # median of three device-timed runs (single runs varied by up to 20 % between boxes / first use)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        res = engine.run_sampler([prep], q0, DON_SAMPLES, DON_L, DON_EPS, burn=0, seed=2, to_host=False)
        e1.record()
        torch.cuda.synchronize()
        runs_ms.append(e0.elapsed_time(e1))
    ms = sorted(runs_ms)[1]
    value = evals / (ms * 1e-3)
    acc = float(res.accepted.float().mean())
    dH = float((res.hamiltonians[..., 0] - res.hamiltonians[..., 1]).abs().median())
    del res
    # a gradient batch alone (what the FLOP count refers to)
    engine.logp_grad(prep, q0)
    torch.cuda.synchronize()
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    g0.record()
    for _ in range(2):
        engine.logp_grad(prep, q0)
    g1.record()
    torch.cuda.synchronize()
    grad_ms = g0.elapsed_time(g1) / 2
    tflops = DON_GFLOP * DON_CHAINS / (grad_ms * 1e-3) / 1e3
    # end to end: host tensors in, host samples out
    # (two full calls, the second is reported: the first one pays the one-off cudaHostAlloc of the 530 MB pinned result buffer and the
    # cudaMalloc of the 37 GB workspace, which torch's caching allocators keep for every later call)
    q0_pinned = q0_host.pin_memory()
    samplers.sample(spec, q0_host[:8], num_samples=1, num_steps_per_sample=1, step_size=DON_EPS)
    e2e_runs = []
    for _ in range(2):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = samplers.sample(spec, q0_pinned, num_samples=DON_SAMPLES, num_steps_per_sample=DON_L, step_size=DON_EPS, seed=3, return_result=True)
        torch.cuda.synchronize()
        e2e_runs.append(time.perf_counter() - t0)
    e2e_s = e2e_runs[-1]
    h2d = sum(t.numel() * t.element_size() for t in (spec.x, spec.x2, spec.y, q0_host))
    d2h = sum(x.numel() * x.element_size() for x in (out.samples, out.accepted, out.hamiltonians, out.logp, out.step_sizes))
    peak = peaks_tf32["tf32_tflops_sustained"]
    leg = {
        "workload": DON_WORKLOAD, "metric": METRIC, "unit": UNIT, "value": value, "ms_per_step": ms / DON_SAMPLES,
        "step": f"one HMC iteration of all {DON_CHAINS} chains = L+1 = {DON_L + 1} grad-evals per chain; {DON_SAMPLES} timed iterations",
        "acceptance_rate": acc, "median_abs_energy_error": dH, "run_ms": runs_ms,
        "e2e": {"value": evals / e2e_s, "unit": UNIT, "seconds": e2e_s, "h2d_bytes_per_step": h2d / DON_SAMPLES,
                "d2h_bytes_per_step": d2h / DON_SAMPLES, "seconds_of_each_call": e2e_runs,
                "timing": "second of two calls of samplers.sample with pinned host tensors (the first pays the one-off pinned / device allocations)"},
        "gradient_batch": {"chains": DON_CHAINS, "ms": grad_ms, "chain_grad_evals_per_s": DON_CHAINS / (grad_ms * 1e-3),
                           "tflops_fp32_equivalent": tflops},
        "roofline": {"bound": "tensor", "achieved": tflops, "peak": peak, "unit": "TFLOP/s", "frac": tflops / peak, "traffic": None,
                     "kernel": "whole gradient batch (launch list and per-kernel ncu: profiles/r02_summary.md section B)",
                     "note": "achieved = 11.56 GFLOP of fp32-equivalent work per chain-grad-eval (SURVEY 8(d)) / CUDA-event time of a "
                             "256-chain gradient batch; peak = cuBLAS TF32 8192^3 sustained, measured in this run (tf32_peak).  The tensor "
                             "core executes 3 tf32 products per fp32 product in the backward pass and 9 bf16 products (exact fixed-point "
                             "accumulation, csrc/xgemm.cuh) in the forward pass, i.e. >= 3x the algorithmic FLOPs"},
        "tf32_peak": peaks_tf32,
        "cpu_baseline": None if skip_cpu else don_cpu_baseline_leg(),
    }
    return leg


def run_ours(steps, warmup, n_gpus, skip_cpu=False, legs="all", dump_dir=None):
    """dump_dir: write the last row of each array the last timed launch returned (rank 0's chains) as <name>.npy there."""
    import statistics

    import numpy as np
    import torch
    import torch.distributed as dist
    from vihmc import engine, samplers

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # the contract is ONE line on stdout, but NCCL writes its "NCCL version ..." banner to file descriptor 1 when the
        # communicator is created: point fd 1 at stderr for the run and keep the real stdout for the JSON line
        global _REAL_STDOUT_FD
        sys.stdout.flush()
        _REAL_STDOUT_FD = os.dup(1)
        os.dup2(2, 1)
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()

    warmup = max(warmup, 3)
    spec, mu, sigma, ind = build_spec()
    chain0 = rank * CHAINS_PER_GPU
    q0_host = initial_states(mu, sigma, ind, CHAINS_PER_GPU, chain0)
    prep = engine.prepare(spec, dev)
    q0 = q0_host.to(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def launch(n_samples, seed):
        return engine.run_sampler([prep], q0, n_samples, L_STEPS, STEP_SIZE, burn=0, seed=seed, chain_offset=chain0,
                                  diagnostics=True, to_host=False)

    # ---- device-timed: inputs resident in HBM; REPS timed launches of `steps` iterations each, value = median ----
    launch(warmup, seed=1)
    torch.cuda.synchronize()
    # the sampler allocates its result tensors with torch.empty: put blocks of those sizes into torch's caching allocator
    # now, so that no cudaMalloc (a host-side, millisecond-scale call) lands between the two timing events
    warm = [torch.empty((steps, CHAINS_PER_GPU, D_SAMPLED), device=dev), torch.empty((steps, CHAINS_PER_GPU, 2), device=dev),
            torch.empty((steps, CHAINS_PER_GPU), device=dev), torch.empty((steps, CHAINS_PER_GPU), dtype=torch.uint8, device=dev),
            torch.empty(CHAINS_PER_GPU, device=dev)]
    del warm
    times, acc_rate = [], 0.0
    with ClockSampler(local_rank) as clk:
        for rep in range(REPS):
            flush.fill_(1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier()
            torch.cuda.synchronize()
            e0.record()
            res = launch(steps, seed=2 + rep)
            e1.record()
            torch.cuda.synchronize()
            barrier()
            t = torch.tensor([e0.elapsed_time(e1)], device=dev)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            times.append(float(t.item()))
            acc_rate = float(res.accepted.float().mean())
            if dump_dir is not None and rep == REPS - 1:
                last_step = {"samples": res.samples[-1], "logp": res.logp[-1], "hamiltonians": res.hamiltonians[-1],
                             "accepted": res.accepted[-1].float(), "step_sizes": res.step_sizes}
                last_step = {k: v.cpu().numpy() for k, v in last_step.items()}
            del res
    ms = statistics.median(times)
    if dump_dir is not None and rank == 0:
        os.makedirs(dump_dir, exist_ok=True)
        for name, arr in last_step.items():
            np.save(os.path.join(dump_dir, f"{name}.npy"), arr)
    evals = world * CHAINS_PER_GPU * steps * (L_STEPS + 1)
    value = evals / (ms * 1e-3)

    # ---- end to end through the public API: host tensors in, host samples out, every call ----
    # warm-up call of the SAME shape as the timed one: the pinned result buffers then come out of torch's caching host allocator
    # instead of a fresh cudaHostAlloc (page-locking tens of MB costs ~0.1 s on a fresh box)
    samplers.sample(spec, q0_host, num_samples=steps, num_steps_per_sample=L_STEPS, step_size=STEP_SIZE, seed=3,
                    chain_offset=chain0)
    e2e_times, out = [], None
    for rep in range(3):
        barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = samplers.sample(spec, q0_host, num_samples=steps, num_steps_per_sample=L_STEPS, step_size=STEP_SIZE, seed=4 + rep,
                              chain_offset=chain0, return_result=True)
        torch.cuda.synchronize()
        t = torch.tensor([time.perf_counter() - t0], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_times.append(float(t.item()))
    e2e_s = statistics.median(e2e_times)
    h2d = prep.h2d_bytes + q0_host.numel() * 4
    d2h = sum(x.numel() * x.element_size() for x in (out.samples, out.accepted, out.hamiltonians, out.logp, out.step_sizes))
    e2e_value = evals / e2e_s
    del out

    # ---- ESS/sec ----
    ess = ess_leg(dev, rank, world, dist) if legs in ("all", "ess") else None

    # ---- the other BASELINE configs ----
    configs = {}
    if legs in ("all", "configs"):
        if world == 1:
            tf32 = measure_tf32_peak(dev)
            configs["cfg3"] = don_leg(dev, tf32, skip_cpu)
            from bench_multi import cfg5_leg
            configs["cfg5"] = cfg5_leg(dev, rank, world, dist if world > 1 else None)   # the N = 1 point of the strong-scaling leg
        else:
            from bench_multi import cfg4_leg, cfg5_leg   # tools-free: lives next to this file
            configs["cfg4"] = cfg4_leg(dev, rank, world, dist)
            configs["cfg5"] = cfg5_leg(dev, rank, world, dist)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return None
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    sm_max_mhz = peaks.get("sm_max_mhz", 1965.0)
    fp32_peak_tflops = 148 * 128 * 2 * sm_max_mhz * 1e6 / 1e12
    achieved_tflops = (CHAINS_PER_GPU * steps * (L_STEPS + 1) * FLOP_PER_GRAD_EVAL) / (ms * 1e-3) / 1e12
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warmup,
        "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": WORKLOAD, "chains_total": world * CHAINS_PER_GPU,
                   "step": "one HMC iteration of all chains = L+1 = 197 grad-evals per chain",
                   "timing": f"median of {REPS} launches of {steps} iterations each (CUDA events, max over ranks per launch); "
                             f"ms of every launch in launch_ms",
                   "l2": "256 MB flush before every timed launch; chain state is shared-memory resident",
                   "parallelism": f"chains sharded {world}x{CHAINS_PER_GPU}, no data-path collective"},
        "launch_ms": times,
        "roofline": {"bound": "fp32", "achieved": achieved_tflops, "peak": fp32_peak_tflops, "unit": "TFLOP/s",
                     "frac": achieved_tflops / fp32_peak_tflops, "traffic": None,
                     "kernel": "mlp_small_sample_kernel<W=10, warps/chain=1, specialised>",
                     "note": "neither hbm nor tensor: 20x10x10 tiles are below any UMMA shape and all state lives in "
                             "shared memory; peak = 148 SM x 128 FMA lanes x 2 x sm_max_mhz (computed, not in "
                             "MEASURED_PEAKS.json); achieved = 14 kFLOP per chain-grad-eval (SURVEY 8(d)) / event time. "
                             "ncu (profiles/r02_ncu_details_mlp_small_sample_v2.csv, profiles/r02_summary.md F): 213 shared-memory "
                             "pipe cycles per evaluation (205 LDS/STS wavefronts + 8 shuffles), 520 warp instructions per "
                             "evaluation, issue slots 43 % busy; the largest stall reason is the fixed-latency dependency wait "
                             "inside a warp (1.7 warps per scheduler at 1024 chains); DRAM traffic negligible"},
        # shared-memory pipe: LDS/STS wavefronts and shuffles share one wavefront per clock per SM (tools/probe_shfl_lds.cu).
        # 213 pipe cycles per chain-grad-eval is a constant of the compiled kernel (ncu: l1tex__data_pipe_lsu_wavefronts_mem_shared
        # 8.30e7 for 1024 chains x 2 iterations x 197 evaluations = 205.6, plus the 8 SHFL of the output layer that metric omits)
        "roofline_binding_unit": {"bound": "shared-memory pipe (l1tex lsu wavefronts + shuffles)", "unit": "Gwavefronts/s",
                                  "achieved": WAVEFRONTS_PER_EVAL * (CHAINS_PER_GPU * steps * (L_STEPS + 1)) / (ms * 1e-3) / 1e9,
                                  "peak": 148 * sm_max_mhz * 1e6 / 1e9,
                                  "frac": WAVEFRONTS_PER_EVAL * (CHAINS_PER_GPU * steps * (L_STEPS + 1)) / (ms * 1e-3) / (148 * sm_max_mhz * 1e6),
                                  "wavefronts_per_chain_grad_eval": WAVEFRONTS_PER_EVAL,
                                  "note": "round 1: 303 wavefronts at 0.78 of the pipe; version 2 of the kernel is bound by "
                                          "dependent-issue latency, not by this pipe any more"},
        "cpu_baseline": cpu_baseline_leg() if (world == 1 and not skip_cpu) else None,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d / steps, "d2h_bytes_per_step": d2h / steps,
                "seconds": e2e_s, "timing": "median of 3 calls of samplers.sample with host tensors"},
        "gpu_launches": 1,
        "clocks": clk.summary(),
        "acceptance_rate": acc_rate,
        "ess": ess,
        "configs": configs,
    }
    if world > 1:
        dist.destroy_process_group()
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "reference-cfg3"])
    ap.add_argument("--mode", default="intra", choices=["intra", "procs"], help="--impl reference-cfg3 only")
    ap.add_argument("--legs", default="all", choices=["all", "main", "ess", "configs"], help="profiling runs: restrict the extra legs")
    ap.add_argument("--skip-cpu-baseline", action="store_true", help="profiling runs only")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last row of each array the last timed launch returned -- samples, logp, hamiltonians, accepted, "
                         "step_sizes (float32, one .npy each) -- to DIR, to compare two builds output for output")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs is not None and a.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours only")
    if a.impl == "reference":
        line = run_reference(a.steps, a.warmup, a.gpus)
    elif a.impl == "reference-cfg3":
        line = run_reference_don(a.mode, a.steps)
    else:
        line = run_ours(a.steps, a.warmup, a.gpus, a.skip_cpu_baseline, a.legs, a.dump_outputs)
    if line is not None:
        if _REAL_STDOUT_FD is not None:
            os.write(_REAL_STDOUT_FD, (json.dumps(line) + "\n").encode())
        else:
            print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
