"""Multi-GPU plumbing: one process per GPU (torchrun), chains sharded, NO collective inside the leapfrog loop.

The reference runs its chains one after another in a Python loop (main_VI_HMC.py:458-460), so chains are
independent by construction: global chain ids [rank*C/G, (rank+1)*C/G) live on GPU `rank`, data and VI
artefacts are replicated, and the Philox streams are keyed on the GLOBAL chain id so the draws do not
depend on the sharding.  Collectives (NCCL on GPUs, gloo in the CPU tests) are used only AFTER sampling:
gather of the stored draws and of per-half-chain moments for split-R-hat.
"""
from __future__ import annotations

from typing import Dict, Optional, Tuple

import torch
import torch.distributed as dist

from . import diagnostics


def world() -> Tuple[int, int]:
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def shard_chains(total_chains: int, rank: Optional[int] = None, world_size: Optional[int] = None) -> Tuple[int, int]:
    """(first global chain id, number of local chains) -- contiguous blocks, remainder spread over the low ranks."""
    r, w = world()
    rank = r if rank is None else rank
    world_size = w if world_size is None else world_size
    if total_chains < world_size:
        raise ValueError(f"{total_chains} chains cannot be sharded over {world_size} ranks")
    base, rem = divmod(total_chains, world_size)
    n = base + (1 if rank < rem else 0)
    start = rank * base + min(rank, rem)
    return start, n


def gather_chains(local: torch.Tensor, total_chains: int, dst: int = 0, chain_dim: int = 1) -> Optional[torch.Tensor]:
    """Gather [.., C_local, ..] shards (ragged allowed) to rank `dst` along `chain_dim`; other ranks get None."""
    rank, w = world()
    if w == 1:
        return local
    counts = [shard_chains(total_chains, r, w)[1] for r in range(w)]
    moved = local.movedim(chain_dim, 0).contiguous()
    cmax = max(counts)
    if moved.shape[0] < cmax:  # pad ragged shards so every rank sends the same shape
        pad = torch.zeros((cmax - moved.shape[0],) + tuple(moved.shape[1:]), dtype=moved.dtype, device=moved.device)
        moved = torch.cat([moved, pad], 0)
    bufs = [torch.empty_like(moved) for _ in range(w)] if rank == dst else None
    dist.gather(moved, bufs, dst=dst)
    if rank != dst:
        return None
    out = torch.cat([b[:c] for b, c in zip(bufs, counts)], 0)
    return out.movedim(0, chain_dim)


def global_split_rhat(local_draws: torch.Tensor) -> torch.Tensor:
    """Split-R-hat over ALL chains of all ranks from per-half-chain moments: each rank contributes
    [2*C_local, d] means and variances (8*C_local*d bytes) instead of its draws.  Same value on every rank."""
    mean, var, S = diagnostics.half_chain_moments(local_draws.reshape(local_draws.shape[0], local_draws.shape[1], -1))
    rank, w = world()
    if w > 1:
        counts = torch.tensor([mean.shape[0]], device=mean.device)
        all_counts = [torch.zeros_like(counts) for _ in range(w)]
        dist.all_gather(all_counts, counts)
        cmax = int(max(int(c) for c in all_counts))
        def pad(t):
            if t.shape[0] == cmax:
                return t.contiguous()
            return torch.cat([t, torch.zeros((cmax - t.shape[0],) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)], 0)
        ms = [torch.empty((cmax,) + tuple(mean.shape[1:]), dtype=mean.dtype, device=mean.device) for _ in range(w)]
        vs = [torch.empty_like(ms[0]) for _ in range(w)]
        dist.all_gather(ms, pad(mean))
        dist.all_gather(vs, pad(var))
        mean = torch.cat([m[:int(c)] for m, c in zip(ms, all_counts)], 0)
        var = torch.cat([v[:int(c)] for v, c in zip(vs, all_counts)], 0)
    return diagnostics.rhat_from_moments(mean, var, S)


def sample_sharded(specs, q0_all: torch.Tensor, total_chains: int, burn_in_draws: int = 0, gather: bool = True, **sampler_kw
                   ) -> Dict[str, object]:
    """Run the local shard of `total_chains` chains on this rank's GPU and gather on rank 0.

    q0_all: [total_chains, d] start points (every rank passes the same tensor; each takes its rows).
    burn_in_draws: stored rows to drop before the diagnostics (the caller-side `params_hmc[cfg.burn:]`).
    Returns {'samples','logp','accepted' (rank 0: full; else None), 'rhat' (all ranks), 'local'}.
    ``sampler_kw`` goes to ``engine.run_sampler`` as it is, including ``inv_mass`` (one [d] diagonal for every chain of every rank)."""
    from . import engine

    chain0, n_local = shard_chains(total_chains)
    res = engine.run_sampler(specs, q0_all[chain0:chain0 + n_local], chain_offset=chain0, to_host=False, **sampler_kw)
    draws = res.samples[burn_in_draws:]
    out = {"local": res, "rhat": global_split_rhat(draws) if draws.shape[0] >= 4 else None}
    if gather:
        out["samples"] = gather_chains(res.samples, total_chains)
        out["logp"] = gather_chains(res.logp, total_chains) if res.logp is not None else None
        out["accepted"] = gather_chains(res.accepted, total_chains) if res.accepted is not None else None
    return out


# ------------------------------------------------------------------------------------------------
# optional second mode (BASELINE.json configs[4]): data-sharded likelihood, gradient all-reduce
# ------------------------------------------------------------------------------------------------
def shard_spec_rows(spec, rank: Optional[int] = None, world_size: Optional[int] = None):
    """Row shard of a LogProbSpec for this rank: training rows [r*N/G, (r+1)*N/G), prior divided by G.

    Summing the shard log-posteriors over ranks gives the full log-posterior -- the same construction as the
    reference's split closures (main_HMC_splitting.py:28-54, 253-254: equal row blocks, prior_scale = num_splits)."""
    import dataclasses

    r, w = world()
    rank = r if rank is None else rank
    world_size = w if world_size is None else world_size
    start, n = shard_chains(spec.N, rank, world_size)   # same contiguous-block rule, applied to rows
    return dataclasses.replace(spec, x=spec.x[start:start + n].contiguous(), y=spec.y[start:start + n].contiguous(),
                               prior_scale=float(spec.prior_scale) * world_size)


def sample_data_sharded(spec_local, q0: torch.Tensor, num_samples: int, num_steps: int, step_size: float, burn: int = 0,
                        seed: int = 0, hamiltorch_fallback_rule: bool = True, use_graphs: bool = True,
                        inv_mass: Optional[torch.Tensor] = None) -> Dict[str, torch.Tensor]:
    """HMC where every rank holds ALL chains and a row shard of the data (spec_local = shard_spec_rows(spec)).

    One exchange step per gradient evaluation: ONE all_reduce(SUM) of a [C, d + 1] buffer (gradients, log-posterior behind them);
    everything else is identical on every rank (same Philox streams), so all ranks make the same accept/reject
    decisions and hold the same samples.  The [C, d] arithmetic runs in the C-ABI building blocks
    (vihmc_logp_grad, vihmc_leapfrog_update, vihmc_momentum_philox, vihmc_mh_accept); torch does the collective
    and the per-chain scalar adds.  Leapfrog order and rounding as in vihmc_sample / hamiltorch.

    ``use_graphs``: the three kinds of leapfrog step (first: H0 + half kick + drift; middle: kick + drift; last: kick, half kick
    back, H1) -- gradient kernels, the packed all-reduce and the update kernels -- are each captured once into a CUDA graph (NCCL
    collectives are capturable) and replayed: with 8 GPUs a step is well under a millisecond of ~40 short launches, and the
    replay removes the launch gaps.  Same kernels, same order, same results as the eager loop
    (tests/test_gpu_deeponet.py::test_data_sharded_sampler_equals_general_sampler compares the two bit for bit).

    ``inv_mass``: diagonal inverse mass [d] as in ``engine.run_sampler``.  The captured graphs read it by address, so the graph
    cache is keyed on the device tensor's ``data_ptr()`` and holds a reference to it: pass the same device tensor again to replay,
    a different one re-captures."""
    from . import engine

    rank, w = world()
    prep = engine.prepare(spec_local)
    dev = prep.device
    d = prep.spec.d
    q0d = q0.reshape(-1, d).to(device=dev, dtype=torch.float32).contiguous()
    C = q0d.shape[0]
    rows = num_samples - burn
    if rows < 1:
        raise RuntimeError("burn must be less than num_samples.")
    if num_steps < 1:
        raise ValueError("num_steps must be at least 1")
    samples = torch.empty((rows, C, d), dtype=torch.float32, device=dev)
    samples[0] = q0d
    accepted = torch.empty((num_samples, C), dtype=torch.uint8, device=dev)
    ham = torch.empty((num_samples, C, 2), dtype=torch.float32, device=dev)
    q_cur, q_fb = q0d.clone(), q0d.clone()
    m = None
    if inv_mass is not None:
        m = inv_mass if isinstance(inv_mass, torch.Tensor) else torch.as_tensor(inv_mass)
        m = m.to(device=dev, dtype=torch.float32).contiguous()
        if m.shape != (d,):
            raise ValueError(f"inv_mass must be a 1-D tensor of length d={d}")

    # Work buffers and graphs are cached on the prepared problem, keyed by what the captured launches depend on: a second call
    # with the same chains / step size (the timed call after a warm-up, the next block of iterations) replays without re-capturing.
    cache = prep.__dict__.setdefault("_data_sharded_cache", {})
    key = (C, d, float(step_size), w, bool(use_graphs), None if m is None else m.data_ptr())
    st = cache.get(key)
    if st is None:
        st = cache[key] = {"q": torch.empty_like(q0d), "p": torch.empty_like(q0d),
                           "inv_mass": m,   # the graphs read it by address: keep it alive as long as they are

                           # ONE collective per evaluation: the [C] log-posteriors ride behind the [C, d] gradients in the same buffer
                           "packed": torch.empty((C, d + 1), dtype=torch.float32, device=dev) if w > 1 else None, "graphs": None}
    q, p, packed, m = st["q"], st["p"], st["packed"], st["inv_mass"]

    def grad(qq):
        lp, g = engine.logp_grad(prep, qq)
        if w > 1:
            packed[:, :d].copy_(g)
            packed[:, d].copy_(lp)
            dist.all_reduce(packed, op=dist.ReduceOp.SUM)
            g.copy_(packed[:, :d])
            lp.copy_(packed[:, d])
        return lp, g

    def step_first():
        lp, g = grad(q)
        ke0 = engine.leapfrog_update(q, p, g, step_size, 0.0, 0.0, want_ke=True, inv_mass=m)   # kinetic energy of the fresh momentum
        h0 = ke0 - lp
        engine.leapfrog_update(q, p, g, step_size, 0.5, 1.0, inv_mass=m)
        return h0

    def step_mid():
        lp, g = grad(q)
        engine.leapfrog_update(q, p, g, step_size, 1.0, 1.0, inv_mass=m)

    def step_last():
        lp, g = grad(q)
        engine.leapfrog_update(q, p, g, step_size, 1.0, 0.0, inv_mass=m)
        ke1 = engine.leapfrog_update(q, p, g, step_size, -0.5, 0.0, want_ke=True, inv_mass=m)
        return ke1 - lp

    # a trajectory of L steps: first, L - 1 middle evaluations, last (L + 1 gradient evaluations)
    if use_graphs and dev.type == "cuda" and st["graphs"] is None:
        q.copy_(q0d)
        p.zero_()
        step_mid()                                  # eager warm-up: lazy kernel attributes, workspace, NCCL channels
        torch.cuda.synchronize(dev)
        side = torch.cuda.Stream(device=dev)
        graphs = {}
        with torch.cuda.device(dev):
            for name, fn in (("first", step_first), ("mid", step_mid), ("last", step_last)):
                q.copy_(q0d)
                p.zero_()
                gr = torch.cuda.CUDAGraph()
                with torch.cuda.graph(gr, stream=side):
                    out = fn()
                graphs[name] = (gr, out)
        torch.cuda.synchronize(dev)
        st["graphs"] = graphs
    graphs = st["graphs"] if use_graphs else None

    def run(name, fn):
        if graphs is None:
            return fn()
        gr, out = graphs[name]
        gr.replay()
        return out

    for n in range(num_samples):
        if hamiltorch_fallback_rule and n == burn + 1:
            q_fb.copy_(q0d)
        p.copy_(engine.momentum_philox(seed, n, 0, C, d, device=dev, inv_mass=m))
        q.copy_(q_cur)
        h0 = run("first", step_first)
        for s in range(1, num_steps):
            run("mid", step_mid)
        h1 = run("last", step_last)
        u = engine.uniform_philox(seed, n, 0, C, device=dev)
        store = n > burn
        engine.mh_accept(h0, h1, u, q, q_cur, q_fb, stored=samples[n - burn] if store else None, accepted=accepted[n])
        ham[n, :, 0], ham[n, :, 1] = h0, h1
    return {"samples": samples, "accepted": accepted, "hamiltonians": ham, "graphs": graphs is not None}
