"""The DeepONet dense path across likelihoods, raw trunk inputs and every route edge, against the fp64 oracle.

Every other DeepONet test uses loss = "NLL" with tau_out = 1, where make_likelihood (csrc/common.cuh) gives ll_const = 0 and
prec = 1: the per-output constant, the precision that scales G = d loglik / d output and the count of outputs on ragged tiles
are all invisible there.  CASES below varies the likelihood (NLL variances 0.01, 4 and 1e-9 -- clamped to 1e-6 as torch's
GaussianNLLLoss does --, regression precisions 100, 10, 4 and 0), the trunk input (the (t, x) feature layer or raw trunk inputs,
impose_bc = False), the VI split, the prior form and the architecture, so that every stack reaches each route make_plan
(csrc/dense.cu) can give it:
    fwd3                    exact-accumulation forward (fused_forward3_kernel) and head3_kernel, fused 3xTF32 backward
    fwd3_fwd+per_layer_bwd  the fwd3 forward, but one GEMM per layer backward (inputs of 105..112: past fused::KPAD, within xg::XK)
    fused                   fused 3xTF32 forward and backward, head product with the EPI_HEAD epilogue
    per_layer               one GEMM per layer both ways, EPI_HEAD epilogue
A Python mirror of make_plan's route rule and of the workspace it sizes from that route (route_of / workspace_bytes) must give
vihmc_workspace_bytes exactly: the fwd3 images and the fused-kernel buffers only enter that count on their route, so equality
confirms the route each row names -- under the default environment and under VIHMC_DENSE_NOFUSE=1 and VIHMC_DENSE_SIMT=1.
Neither switch turns fwd3 off (fwd3_eligible does not read them): fwd3 rows keep their forward and head3_kernel under both, and
only their backward moves to the per-layer GEMMs.

The checker is the one of test_gpu_mlp_range: per parameter tensor (the scalar output bias b0, whose gradient is exactly
sum G, is a tensor of its own) ||g - g64|| <= max(1e-5 ||g64||, C_FP32 ||g32 - g64||); the log-posterior with the scale
N P |ll_const| + half_prec sum r^2 + sum_i |prior_i| / prior_scale; the predictions per output with the scale
sum_k |B_k T_k| + |b0|.  Every row must discriminate (bounds below 1 % of every tensor's norm), and on the CPU the checker must
reject, on every row where they differ from the truth, a gradient without prec, a log-posterior without the N P ll_const term
(regression: with half_prec = 0.5), the padded target columns counted as outputs, and a zeroed b0 gradient.
"""
from __future__ import annotations

import ctypes as C
import functools
import json
import math
import os
import subprocess
import sys
import zlib
from collections import namedtuple

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import closures as oc
from test_gpu_mlp_range import (C_FP32, DISCRIM, REL, assert_grad, compare_with_fp64_chain, grad_violations, loose_tensors,
                                scalar_ok, tensor_groups)
from vihmc import _lib, engine
from vihmc.spec import DeepONetArch, LogProbSpec, act_code, loss_code

KPAD, XK = 104, 112            # fused::KPAD (fused 3xTF32 stack kernels), xg::XK (exact-accumulation forward)
NLL_EPS = float(np.float32(1e-6))
ENVS = (None, "VIHMC_DENSE_NOFUSE", "VIHMC_DENSE_SIMT")

# in_trunk: None = the (t, x) feature layer (impose_bc, 5 features); an integer = that many raw trunk inputs (impose_bc = False)
# split:    "full" | "sorted" / "unsorted" VI subset of half the coordinates (always holding b0)
# prior:    "scalar" sigma | "inf" per-coordinate sigma with +inf entries | "mu" non-zero mean | "scale2" prior_scale = 2
# route:    (branch, trunk), see the module docstring
Case = namedtuple("Case", "id in_branch in_trunk wb db wt dt K act loss tau N P split prior chains route")
F3, F3PL = ("fwd3", "fwd3"), "fwd3_fwd+per_layer_bwd"
CASES = [
    # head3: ll_const, prec, the partial-tile count and the padded copy of the targets (P % 4 = 3)
    Case("nll_v001_ragged", 7, None, 20, 3, 24, 3, 12, "tanh", "NLL", 0.01, 50, 203, "full", "inf", 5, F3),
    # head3 with full tiles only (N % 128 = 0, P % 64 = 0)
    Case("nll_v4_full_tiles", 7, None, 16, 3, 20, 3, 16, "relu", "NLL", 4.0, 128, 128, "sorted", "mu", 5, F3),
    # variance below GaussianNLLLoss's eps: clamped to 1e-6
    Case("nll_clamped", 7, None, 20, 3, 24, 3, 12, "tanh", "NLL", 1e-9, 30, 101, "full", "scalar", 5, F3),
    # regression form, gather through an unsorted sens_ind
    Case("reg_tau100_unsorted", 10, None, 24, 3, 20, 4, 16, "tanh", "regression", 100.0, 60, 150, "unsorted", "scale2", 5, F3),
    # the likelihood contributes nothing: prior-only gradient
    Case("reg_tau0", 7, None, 20, 3, 24, 3, 12, "relu", "regression", 0.0, 40, 90, "full", "inf", 5, F3),
    # K = 10 < 16: the head product on the SIMT kernel's EPI_HEAD epilogue
    Case("head_simt_k10_nll", 7, None, 20, 3, 24, 3, 10, "tanh", "NLL", 0.01, 50, 150, "full", "mu", 5, ("per_layer", "per_layer")),
    # trunk width 22: fused branch only; K = 16, N = 64: the head product on the tensor-core EPI_HEAD epilogue
    Case("head_tc_w22_reg", 7, None, 20, 3, 22, 3, 16, "tanh", "regression", 100.0, 64, 150, "sorted", "inf", 5, ("fused", "per_layer")),
    # raw trunk inputs on the FP32 first layer (in_trunk <= 8)
    Case("raw_trunk2_fwd3", 7, 2, 20, 3, 24, 3, 12, "tanh", "NLL", 0.25, 40, 130, "full", "scalar", 5, F3),
    Case("raw_trunk2_per_layer", 7, 2, 20, 3, 24, 3, 10, "tanh", "regression", 4.0, 40, 130, "unsorted", "mu", 5,
         ("per_layer", "per_layer")),
    # raw trunk inputs on the tensor-core first layer
    Case("raw_trunk12", 7, 12, 20, 3, 24, 3, 12, "tanh", "NLL", 0.01, 40, 97, "sorted", "scale2", 5, F3),
    # branch inputs on each side of MAX_IN0 = 8, KPAD = 104 and XK = 112
    Case("in_branch9", 9, None, 20, 3, 24, 3, 12, "relu", "NLL", 0.01, 45, 77, "full", "inf", 5, F3),
    Case("in_branch104", 104, None, 20, 3, 24, 3, 12, "tanh", "NLL", 0.01, 40, 64, "full", "scalar", 5, F3),
    Case("in_branch108", 108, None, 20, 3, 24, 3, 12, "tanh", "NLL", 0.01, 40, 66, "sorted", "mu", 5, (F3PL, "fwd3")),
    Case("in_branch113", 113, None, 20, 3, 24, 3, 12, "tanh", "NLL", 0.01, 40, 66, "full", "inf", 5, ("per_layer", "fused")),
    # fwd3 at its width edge, the smallest depth the reference's forward accepts
    Case("w104_k104_depth2", 12, None, 104, 2, 104, 2, 104, "tanh", "NLL", 0.01, 40, 70, "full", "mu", 5, F3),
    # per-layer 3xTF32 everywhere (round-1 tanh), tensor-core EPI_HEAD with K = 100
    Case("w108_k100", 12, None, 108, 3, 108, 3, 100, "tanh", "NLL", 0.04, 40, 66, "sorted", "inf", 5, ("per_layer", "per_layer")),
    # VIHMC_MAX_LAYERS, unequal depths
    Case("depth16", 7, None, 16, 16, 16, 16, 16, "tanh", "NLL", 0.01, 30, 50, "full", "scalar", 5, F3),
    Case("depth2_12", 7, None, 20, 2, 24, 12, 12, "relu", "regression", 10.0, 30, 60, "full", "mu", 5, F3),
    # one function, one partial float4
    Case("n1_p3", 7, None, 20, 3, 24, 3, 12, "tanh", "NLL", 0.01, 1, 3, "full", "inf", 5, F3),
    # head3 chunk cap, split-K over P of the trunk weight gradients (trunk width >= 32: tensor cores), 512-deep dBout slices
    Case("long_trunk", 7, None, 20, 3, 32, 3, 12, "tanh", "NLL", 0.01, 40, 2053, "full", "scalar", 2, F3),
]
CASE_BY_ID = {c.id: c for c in CASES}
IDS = [c.id for c in CASES]
SAMPLER_ROWS = ["nll_v001_ragged", "raw_trunk2_per_layer"]


def arch_of(case):
    return DeepONetArch(width_branch=case.wb, width_trunk=case.wt, in_branch=case.in_branch,
                        in_trunk=5 if case.in_trunk is None else case.in_trunk, depth_branch=case.db, depth_trunk=case.dt,
                        output_neurons=case.K, act=case.act, impose_bc=case.in_trunk is None)


def likelihood(case):
    """(ll_const, half_prec, prec) of make_likelihood, in fp64 from the fp32 tau_out the kernels receive."""
    tau = float(np.float32(case.tau))
    if case.loss == "NLL":
        v = max(tau, NLL_EPS)
        return -0.5 * math.log(v), 0.5 / v, 1.0 / v
    return 0.0, 0.5 * tau, tau


def _pad4(v):
    return (v + 3) // 4 * 4


def _cdiv(a, b):
    return -(-a // b)


# ---------------------------------------------------------------------------------------------------------------------
# mirror of make_plan's route rule and workspace (csrc/dense.cu make_plan / dense_workspace_bytes, csrc/api.cu
# vihmc_workspace_bytes / sampler_state_bytes)
# ---------------------------------------------------------------------------------------------------------------------
def _stacks(case):
    a = arch_of(case)
    return [(a.in_branch, [o for o, _ in a.stack_dims("branch")]), (a.in_trunk, [o for o, _ in a.stack_dims("trunk")])]


def _fused_eligible(in_dim, dims, env):
    return (env is None and len(dims) >= 2 and in_dim <= KPAD and all(w % 4 == 0 and w <= KPAD for w in dims))


def _fwd3_eligible(in_dim, dims):
    return len(dims) >= 2 and in_dim <= XK and all(w % 4 == 0 and w <= KPAD for w in dims)


def plan_of(case, env=None):
    """(fwd3, fuse_branch, fuse_trunk) as make_plan decides them."""
    (ia, da), (ib, db) = _stacks(case)
    fwd3 = _fwd3_eligible(ia, da) and _fwd3_eligible(ib, db) and case.K <= XK
    return fwd3, _fused_eligible(ia, da, env), _fused_eligible(ib, db, env)


def route_of(case, env=None):
    fwd3, fa, fb = plan_of(case, env)
    name = lambda fused: ("fwd3" if fused else F3PL) if fwd3 else ("fused" if fused else "per_layer")
    return name(fa), name(fb)


def _splitk_max_slices(K, hint=0):
    chunk = hint or 256
    if K > chunk + chunk // 2:
        return _cdiv(K, chunk)
    if K >= 512:
        return min(K // 128, 8)
    return 1


def workspace_bytes(case, chains, env=None):
    """vihmc_workspace_bytes of the row for `chains` chains, from the route it takes under `env`."""
    pb = problem(case.id)
    N, P, K, D, d = case.N, case.P, case.K, pb["D"], pb["d"]
    Pp = _pad4(P)
    stacks = _stacks(case)
    Dp = 4                                       # the scalar output bias on its own 16-byte slot
    for in_dim, dims in stacks:
        for l, w in enumerate(dims):
            Dp += w * _pad4(in_dim if l == 0 else dims[l - 1]) + _pad4(w)
    (ia, da), (ib, db) = stacks
    R, wmax = max(N, P), max(max(da), max(db))
    head_tiles = _cdiv(P, 128) * _cdiv(N, 128)
    scratch = 0
    for (in_dim, dims), rows in ((stacks[0], N), (stacks[1], P)):
        for l, w in enumerate(dims):
            s = _splitk_max_slices(rows)
            if s > 1:
                scratch = max(scratch, s * w * (in_dim if l == 0 else dims[l - 1]))
    for M, Nn, Kr, hint in ((N, K, P, 512), (P, K, N, 0)):   # dBout = G Tout, dTout = G^T Bout
        s = _splitk_max_slices(Kr, hint)
        if s > 1:
            scratch = max(scratch, s * M * Nn)
    fwd3, fa, fb = plan_of(case, env)
    n_img = max(len(da) if fa else 0, len(db) if fb else 0)
    img = n_img * (2 * 46592 // 4) + 64 if n_img else 0                        # fused::B_TILE = 46 592 B
    dzall = 0
    if fb:
        dzall += (len(db) - 1) * (P * max(db) + 64) + (_cdiv(P, 128) + 16) * max(db) + 64
    if fa:
        dzall += (len(da) - 1) * (N * max(da) + 64) + (_cdiv(N, 128) + 16) * max(da) + 64
    f3 = 0
    if fwd3:
        m_tiles, p_tiles = _cdiv(N, 128), _cdiv(P, 128)
        f3 = (max(len(da), len(db)) * (101248 // 4) + 64                          # xg::XIMG_B = 101 248 B
              + m_tiles * (86016 // 4) + 64 + p_tiles * (86016 // 4) + 64         # xg::XTILE = 86 016 B
              + (m_tiles + p_tiles) * 128 + 128)
    per = (f3 + dzall + img + scratch + 2 * Dp + N * sum(da) + P * sum(db) + N * Pp + 2 * R * wmax + 2 * head_tiles + 8 + 64 * 40
           + P + _cdiv(d, 8192))
    shared = D + 64 + P * 5 + 64 + N * Pp + 64
    cb = min(chains, max(1, (40 << 30) // (per * 4)))
    dense = cb * per * 4 + shared * 4 + 4096
    redraw = D if pb["frozen"] is not None else 0
    sampler = 5 * (chains * d * 4 + 256) + chains * redraw * 4 + 256 + 16 * (chains * 4 + 256) + chains * _cdiv(d, 4096) * 4 + 256
    return dense + sampler + 4096


def abi_problem(case):
    """The vihmc_problem engine.prepare fills for the row, without a device: only sizes are read from it here, so the data
    pointers stay NULL (frozen / sens_ind point at the host copies: their presence decides the sampler-state size)."""
    pb = problem(case.id)
    arch = arch_of(case)
    p = _lib.Problem()
    p.model_kind, p.act, p.loss, p.last_bias, p.impose_bc = 1, act_code(case.act), loss_code(case.loss), 1, int(arch.impose_bc)
    (ia, da), (ib, db) = _stacks(case)
    p.n_layers_a, p.n_layers_b, p.in_a, p.in_b = len(da), len(db), ia, ib
    for i, w in enumerate(da):
        p.dims_a[i] = w
    for i, w in enumerate(db):
        p.dims_b[i] = w
    p.D, p.d, p.N, p.P = pb["D"], pb["d"], case.N, case.P
    p.tau_out, p.prior_scale, p.prior_sigma_scalar = case.tau, pb["prior_scale"], 1.0
    if pb["frozen"] is not None:
        p.frozen, p.sens_ind = pb["frozen"].data_ptr(), pb["ind_np"].ctypes.data
    return p


# ---------------------------------------------------------------------------------------------------------------------
# problems and oracles
# ---------------------------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def problem(case_id):
    """Data, teacher, VI split, prior and the perturbed chains of one row, from a seed fixed by the row id."""
    case = CASE_BY_ID[case_id]
    rs = np.random.RandomState(zlib.crc32(case.id.encode()) % (2 ** 31))
    arch = arch_of(case)
    slots = oc.deeponet_layout(arch.width_branch, arch.width_trunk, arch.in_branch, arch.in_trunk, arch.depth_branch,
                               arch.depth_trunk, arch.output_neurons)
    D = oc.layout_numel(slots)
    assert D == arch.num_params
    x1 = rs.uniform(-1.0, 1.0, size=(case.N, case.in_branch))
    if case.in_trunk is None:
        x2 = np.stack([rs.uniform(0.0, 1.0, case.P), rs.uniform(-1.0, 1.0, case.P)], axis=1)   # (t, x)
    else:
        x2 = rs.uniform(-1.0, 1.0, size=(case.P, case.in_trunk))
    gain = math.sqrt(2.0) if case.act == "relu" else 1.0
    theta = np.empty(D)
    for s in slots:
        if s.name == "b":
            theta[0] = 0.5                                                     # a clearly non-zero output bias
        elif "W" in s.name:
            theta[s.offset:s.offset + s.numel] = gain * rs.randn(s.numel) / math.sqrt(s.shape[1])
        else:
            theta[s.offset:s.offset + s.numel] = 0.3 * rs.randn(s.numel)
    x1 = torch.from_numpy(x1.astype(np.float32))
    x2 = torch.from_numpy(x2.astype(np.float32))
    theta32 = torch.from_numpy(theta.astype(np.float32))
    with torch.no_grad():
        f = oc.deeponet_forward(x1.double().unsqueeze(1), x2.double().unsqueeze(0), oc.unflatten(slots, theta32.double()),
                                case.db, case.dt, case.act, arch.impose_bc).squeeze(1)
    y = (f + 0.1 * torch.from_numpy(rs.randn(case.N, case.P))).float()
    if case.split == "full":
        ind, frozen, d = np.arange(D, dtype=np.int64), None, D
    else:
        d = D // 2
        ind = np.concatenate([[0], 1 + rs.choice(D - 1, d - 1, replace=False)]).astype(np.int64)
        ind = np.sort(ind) if case.split == "sorted" else rs.permutation(ind)
        frozen = theta32.clone()
    q0 = theta[ind]
    prior_mu, prior_scale, scalar, prior_sigma = np.zeros(d, np.float32), 1.0, 0.8, None
    if case.prior == "scale2":
        prior_scale, scalar = 2.0, 1.5
    elif case.prior == "inf":
        prior_sigma = (0.5 + rs.rand(d)).astype(np.float32)
        prior_sigma[rs.rand(d) < 0.2] = np.inf
    elif case.prior == "mu":
        prior_sigma = (0.3 + rs.rand(d)).astype(np.float32)
        prior_mu = (q0 + 0.2 * rs.randn(d)).astype(np.float32)
    sig_np = np.full(d, np.float32(scalar), np.float32) if prior_sigma is None else prior_sigma
    q = torch.from_numpy((q0[None] + 0.02 * rs.randn(case.chains, d)).astype(np.float32))
    spec = LogProbSpec(arch=arch, x=x1, x2=x2, y=y, loss=case.loss, tau_out=case.tau,
                       prior_mu=torch.from_numpy(prior_mu) if case.prior == "mu" else None,
                       prior_sigma=None if prior_sigma is None else torch.from_numpy(prior_sigma), prior_sigma_scalar=scalar,
                       prior_scale=prior_scale, frozen=frozen, sens_ind=None if frozen is None else ind,
                       vi_sigma=None if frozen is None else torch.full((D,), 0.01))
    b0_pos = int(np.nonzero(ind == 0)[0][0])
    return dict(case=case, slots=slots, D=D, d=d, x1=x1, x2=x2, y=y, theta=theta32, frozen=frozen, ind_np=ind,
                ind_or_none=None if frozen is None else ind, prior_mu_np=prior_mu, prior_sigma_np=sig_np, prior_scale=prior_scale,
                q=q, spec=spec, groups=tensor_groups(slots, ind), b0_pos=b0_pos)


class Oracle:
    """DeepONetLogProb's network with the likelihood written out per output (NLL with the clamped variance, or regression)
    and a per-coordinate prior N(mu_i, sigma_i) / prior_scale over the finite sigma_i."""

    def __init__(self, pb, dtype):
        case = pb["case"]
        arch = arch_of(case)
        self.dtype = dtype
        self.net = oc.DeepONetLogProb(x1=pb["x1"].unsqueeze(1), x2=pb["x2"].unsqueeze(0), y=pb["y"], width_branch=case.wb,
                                      width_trunk=case.wt, in_branch=case.in_branch, in_trunk=arch.in_trunk,
                                      depth_branch=case.db, depth_trunk=case.dt, output_neurons=case.K, act=case.act,
                                      impose_bc=arch.impose_bc, loss=case.loss, tau_out=float(np.float32(case.tau)),
                                      frozen=pb["frozen"], sens_ind=pb["ind_or_none"], dtype=dtype)
        self.ll_const, self.half_prec, self.prec = likelihood(case)
        self.fin = torch.from_numpy(np.isfinite(pb["prior_sigma_np"]))
        self.pmu = torch.from_numpy(pb["prior_mu_np"]).to(dtype)[self.fin]
        self.psg = torch.from_numpy(pb["prior_sigma_np"]).to(dtype)[self.fin]
        self.prior_scale = pb["prior_scale"]

    def forward(self, q):
        return self.net.forward(q)

    def loglik_terms(self, q):
        r = self.forward(q) - self.net.y
        return self.ll_const - self.half_prec * r * r

    def prior_terms(self, q):
        return torch.distributions.Normal(self.pmu, self.psg).log_prob(q[self.fin])

    def loglik(self, q):
        return self.loglik_terms(q).sum()

    def __call__(self, q):
        return self.loglik(q) + self.prior_terms(q).sum() / self.prior_scale

    def lp_scale(self, q):
        """N P |ll_const| + half_prec sum r^2 + sum_i |prior_i| / prior_scale: the size of what the log-posterior adds up."""
        with torch.no_grad():
            r = self.forward(q) - self.net.y
            return float(r.numel() * abs(self.ll_const) + self.half_prec * (r * r).sum()
                         + self.prior_terms(q).abs().sum() / self.prior_scale)

    def out_scale(self, q):
        """per output: sum_k |B_k T_k| + |b0|, the size of what the head adds up."""
        n = self.net
        with torch.no_grad():
            ws = oc.unflatten(n.slots, oc.scatter_vi(n.frozen, n.sens_ind, q))
            a, c = oc._ACTS[n.act], 1
            h = n.x1[:, 0]
            for _ in range(n.depth_branch - 1):
                h = a(F.linear(h, ws[c], ws[c + 1]))
                c += 2
            B = F.linear(h, ws[c], ws[c + 1])
            c += 2
            h = oc.trunk_features(n.x2)[0] if n.impose_bc else n.x2[0]
            for _ in range(n.depth_trunk - 1):
                h = a(F.linear(h, ws[c], ws[c + 1]))
                c += 2
            T = F.linear(h, ws[c], ws[c + 1])
            return (B.abs() @ T.abs().T + ws[0].abs()).numpy()


@functools.lru_cache(maxsize=None)
def oracle(case_id, dtype):
    return Oracle(problem(case_id), dtype)


@functools.lru_cache(maxsize=None)
def reference(case_id, c):
    """fp64 and fp32 oracle values, gradients and outputs of chain c, the fp64 likelihood and its gradient, and the scales."""
    pb = problem(case_id)
    q = pb["q"][c]
    o64, o32 = oracle(case_id, torch.float64), oracle(case_id, torch.float32)
    lp64, g64 = oc.value_and_grad(o64, q.double())
    lp32, g32 = oc.value_and_grad(o32, q.float())
    ll64, gl64 = oc.value_and_grad(o64.loglik, q.double())
    with torch.no_grad():
        f64 = o64.forward(q.double()).numpy()
        f32 = o32.forward(q.float()).double().numpy()
    return dict(lp64=float(lp64), g64=g64.numpy(), lp32=float(lp32), g32=g32.double().numpy(), ll64=float(ll64), gl64=gl64.numpy(),
                f64=f64, f32=f32, lp_scale=o64.lp_scale(q.double()), out_scale=o64.out_scale(q.double()))


def report(**kw):
    print("DON_RANGE " + json.dumps(kw, default=float), flush=True)


# ---------------------------------------------------------------------------------------------------------------------
# mutants: what a kernel with one of the blind spots of tau_out = 1 would return
# ---------------------------------------------------------------------------------------------------------------------
def mutants(case_id, c):
    """(name, logp, grad) of the wrong results, in fp64 from the oracle, for the rows where they differ from the truth."""
    case, pb, ref = CASE_BY_ID[case_id], problem(case_id), reference(case_id, c)
    ll_const, half_prec, prec = likelihood(case)
    if prec in (0.0, 1.0):
        return []
    lp, g, b0 = ref["lp64"], ref["g64"], pb["b0_pos"]
    out = [("G without prec", lp, g - ref["gl64"] + ref["gl64"] / prec)]
    if case.loss == "NLL":
        out.append(("no N P ll_const", lp - case.N * case.P * ll_const, g))
    else:
        out.append(("half_prec = 0.5", lp + ref["ll64"] * (0.5 / half_prec - 1.0), g))
    pad = case.N * (_pad4(case.P) - case.P)
    if pad:
        # a padded column has no trunk point: its output is b0 and its target the 0 of the padded copy
        w0 = float(pb["q"][c][b0])
        gm = g.copy()
        gm[b0] += pad * (-prec * w0)
        out.append(("padded columns counted", lp + pad * (ll_const - half_prec * w0 * w0), gm))
    gz = g.copy()
    gz[b0] = 0.0
    out.append(("b0 gradient zeroed", lp, gz))
    return out


def rejected(case_id, c, lp, g):
    ref, pb = reference(case_id, c), problem(case_id)
    ok = scalar_ok(lp, ref["lp64"], ref["lp32"], ref["lp_scale"])[0]
    return (not ok) or bool(grad_violations(g, ref["g64"], ref["g32"], pb["groups"])[0])


# ---------------------------------------------------------------------------------------------------------------------
# checks shared by the tests and the reference-path subprocesses
# ---------------------------------------------------------------------------------------------------------------------
def _stream():
    return torch.cuda.current_stream().cuda_stream


def abi_run(prob, q, N, P, ws_chains):
    """vihmc_logp_grad, the value-only vihmc_logp_grad (grad = NULL) and vihmc_predict for every chain of q with a workspace
    sized for ws_chains chains."""
    lib = _lib.load()
    ws_bytes = int(lib.vihmc_workspace_bytes(C.byref(prob), ws_chains))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
    qd = q.cuda().contiguous()
    Cn = q.shape[0]
    lp = torch.empty(Cn, dtype=torch.float32, device="cuda")
    lpv = torch.empty_like(lp)
    g = torch.empty_like(qd)
    out = torch.empty((Cn, N, P), dtype=torch.float32, device="cuda")
    _lib.check(lib.vihmc_logp_grad(C.byref(prob), Cn, qd.data_ptr(), lp.data_ptr(), g.data_ptr(), ws.data_ptr(), ws_bytes, _stream()))
    _lib.check(lib.vihmc_logp_grad(C.byref(prob), Cn, qd.data_ptr(), lpv.data_ptr(), None, ws.data_ptr(), ws_bytes, _stream()))
    _lib.check(lib.vihmc_predict(C.byref(prob), Cn, qd.data_ptr(), out.data_ptr(), ws.data_ptr(), ws_bytes, _stream()))
    torch.cuda.synchronize()
    return lp.cpu().numpy(), lpv.cpu().numpy(), g.cpu().numpy(), out.cpu().numpy()


def check_row(case, env=None):
    """logp, gradient, value-only logp and predictions of every chain, with the workspace of all chains and with a smaller
    one (chain batches, c0 > 0), against the checker.  Returns the row's statistics."""
    pb = problem(case.id)
    prep = engine.prepare(pb["spec"])
    lib = _lib.load()
    Cn = case.chains
    ws_all = int(lib.vihmc_workspace_bytes(C.byref(prep.problem), Cn))
    assert ws_all == workspace_bytes(case, Cn, env), (case.id, env, ws_all, workspace_bytes(case, Cn, env))
    worst = ratio = lp_worst = pr_worst = 0.0
    for ws_chains in (Cn, 2 if Cn > 2 else 1):
        lp, lpv, g, pred = abi_run(prep.problem, pb["q"], case.N, case.P, ws_chains)
        assert np.array_equal(lp.view(np.uint32), lpv.view(np.uint32)), (case.id, ws_chains, lp, lpv)
        for c in range(Cn):
            ref = reference(case.id, c)
            w, r = assert_grad(g[c], ref["g64"], ref["g32"], pb["groups"], f"{case.id} ws {ws_chains} chain {c}")
            worst, ratio = max(worst, w), max(ratio, r)
            ok, lw = scalar_ok(float(lp[c]), ref["lp64"], ref["lp32"], ref["lp_scale"])
            assert ok, (case.id, ws_chains, c, float(lp[c]), ref["lp64"], ref["lp32"])
            lp_worst = max(lp_worst, lw)
            bound = np.maximum(REL * ref["out_scale"], C_FP32 * np.abs(ref["f32"] - ref["f64"]))
            err = np.abs(pred[c].astype(np.float64) - ref["f64"])
            assert (err <= bound).all(), (case.id, ws_chains, c, np.unravel_index(np.argmax(err / bound), err.shape),
                                          float((err / bound).max()))
            pr_worst = max(pr_worst, float((err / bound).max()))
    return dict(grad_err_over_bound=worst, kernel_over_fp32=ratio, logp_err_over_bound=lp_worst, pred_err_over_bound=pr_worst)


def step_size(case):
    """1 / sqrt(largest |eigenvalue| of the fp64 Hessian at chain 0), by power iteration as test_gpu_mlp_range does."""
    o64 = oracle(case.id, torch.float64)
    q = problem(case.id)["q"][0].double()
    v = torch.from_numpy(np.random.RandomState(0).randn(q.numel()))
    lam = 1.0
    for _ in range(15):
        _, hv = torch.autograd.functional.hvp(o64, q, v / v.norm())
        lam = float(hv.norm())
        v = hv
    return 1.0 / math.sqrt(lam)


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the table, the route mirror and the checker
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_table_routes_follow_the_plan_rule(case):
    assert route_of(case) == case.route
    # the reference paths: neither switch turns fwd3 off, both move every backward to the per-layer GEMMs
    for env in ENVS[1:]:
        assert route_of(case, env) == tuple(F3PL if r in ("fwd3", F3PL) else "per_layer" for r in case.route)


def test_table_reaches_every_edge():
    routes = {r for c in CASES for r in c.route}
    assert routes == {"fwd3", F3PL, "fused", "per_layer"}
    assert {c.split for c in CASES} == {"full", "sorted", "unsorted"}
    assert {c.prior for c in CASES} == {"scalar", "inf", "mu", "scale2"}
    assert {c.act for c in CASES} == {"tanh", "relu"}
    assert {c.in_branch for c in CASES} >= {9, 104, 108, 113}
    assert {c.in_trunk for c in CASES} == {None, 2, 12}
    assert max(max(c.db, c.dt) for c in CASES) == _lib.MAX_LAYERS and min(min(c.db, c.dt) for c in CASES) == 2
    assert any(c.N % 128 == 0 and c.P % 64 == 0 for c in CASES if c.route == F3)            # head3: full tiles only
    assert any(c.P % 4 for c in CASES if c.route == F3) and any(c.P % 4 for c in CASES if "fwd3" not in c.route)
    nll = [likelihood(c) for c in CASES if c.loss == "NLL"]
    assert any(l[2] == 1.0 / NLL_EPS for l in nll) and all(l[0] != 0.0 for l in nll)         # the clamp; ll_const != 0
    assert any(c.loss == "regression" and c.tau == 0.0 for c in CASES)


def test_explicit_likelihood_matches_torch():
    """The oracle's per-output likelihood is GaussianNLLLoss (with its variance clamp) or the regression sum the reference
    closure computes."""
    for case in CASES:
        o64 = oracle(case.id, torch.float64)
        q = problem(case.id)["q"][0].double()
        with torch.no_grad():
            ref = oc.log_likelihood(o64.forward(q), o64.net.y, case.loss, o64.net.tau_out)
            ref = float(ref.sum())
            got = float(o64.loglik(q))
        # torch clamps the variance at 1e-6 in the tensor's dtype, the oracle (as the kernels) at float32(1e-6): 3e-9 apart
        assert abs(got - ref) <= 1e-8 * o64.lp_scale(q), (case.id, got, ref)


@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_every_row_discriminates_and_rejects_the_blind_spots(case):
    """Every tensor's bound is below 1 % of its fp64 norm, the fp32 oracle passes, and on the rows whose prec is neither 0 nor 1
    each mutant is rejected on at least one chain, with the logp bound below the smallest logp mutation."""
    pb = problem(case.id)
    hits = {}
    for c in range(case.chains):
        ref = reference(case.id, c)
        assert not loose_tensors(ref["g64"], ref["g32"], pb["groups"]), (c, loose_tensors(ref["g64"], ref["g32"], pb["groups"]))
        assert not rejected(case.id, c, ref["lp32"], ref["g32"])
        lp_bound = max(REL * ref["lp_scale"], C_FP32 * abs(ref["lp32"] - ref["lp64"]))
        for name, lp, g in mutants(case.id, c):
            hits[name] = hits.get(name, False) or rejected(case.id, c, lp, g)
            if lp != ref["lp64"]:
                assert lp_bound < abs(lp - ref["lp64"]), (name, c, lp_bound, abs(lp - ref["lp64"]))
    assert all(hits.values()), hits
    prec = likelihood(case)[2]
    assert len(hits) == (0 if prec in (0.0, 1.0) else 3 + (case.P % 4 != 0))


_WS_SCRIPT = r"""
import json, sys
sys.path[:0] = [{root!r}, {pkg!r}, {tests!r}]
import ctypes as C
import test_gpu_deeponet_range as t
from vihmc import _lib
lib = _lib.load()
print(json.dumps({{c.id: [int(lib.vihmc_workspace_bytes(C.byref(t.abi_problem(c)), n)) for n in (c.chains, 1)] for c in t.CASES}}))
"""


def _root():
    return os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("env", ENVS, ids=["default", "nofuse", "simt"])
def test_workspace_mirror_confirms_every_route(env):
    """vihmc_workspace_bytes (no device needed) equals the mirror for every row, for all its chains and for one, under the
    default environment and under the two switches (read once per process: a subprocess each)."""
    root = _root()
    script = _WS_SCRIPT.format(root=root, pkg=os.path.join(root, "vi-hmc_b200"), tests=os.path.join(root, "tests"))
    full = {k: v for k, v in os.environ.items() if k not in ENVS[1:]}
    if env is not None:
        full[env] = "1"
    out = subprocess.run([sys.executable, "-c", script], env=full, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-3000:]
    got = json.loads(out.stdout.strip().splitlines()[-1])
    for case in CASES:
        assert got[case.id] == [workspace_bytes(case, case.chains, env), workspace_bytes(case, 1, env)], (case.id, env)


def _spec_with_x2(x2, impose_bc, in_trunk):
    arch = DeepONetArch(width_branch=8, width_trunk=8, in_branch=3, in_trunk=in_trunk, depth_branch=2, depth_trunk=2,
                        output_neurons=4, impose_bc=impose_bc)
    return LogProbSpec(arch=arch, x=torch.zeros(2, 3), x2=x2, y=torch.zeros(2, x2.shape[0]))


def test_validate_checks_the_trunk_input_width():
    """x2 is read with a row stride of 2 (feature layer) or in_trunk (raw inputs): any other width is refused."""
    _spec_with_x2(torch.zeros(6, 2), True, 5).validate()
    _spec_with_x2(torch.zeros(6, 3), False, 3).validate()
    _spec_with_x2(torch.zeros(6, 2), False, 2).validate()
    with pytest.raises(ValueError, match="x2"):
        _spec_with_x2(torch.zeros(6, 5), True, 5).validate()
    with pytest.raises(ValueError, match="x2"):
        _spec_with_x2(torch.zeros(6, 2), False, 3).validate()
    with pytest.raises(ValueError, match="x2"):
        _spec_with_x2(torch.zeros(6, 4), False, 3).validate()


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_logp_grad_predict_vs_fp64_oracle(case):
    stats = check_row(case)
    report(case=case.id, route=list(case.route), N=case.N, P=case.P, loss=case.loss, tau_out=case.tau, **stats)


@pytest.mark.gpu
@pytest.mark.parametrize("row", SAMPLER_ROWS)
def test_short_sampling_run_vs_fp64_hamiltorch(row):
    """S = 3, L = 8 through the general sampler with injected momenta and uniforms, against hamiltorch restated on the fp64
    oracle."""
    case = CASE_BY_ID[row]
    pb = problem(row)
    S, L, Cn, d = 3, 8, 3, pb["d"]
    eps = step_size(case)
    rs = np.random.RandomState(11)
    q0 = pb["q"][:Cn]
    p = torch.from_numpy(rs.randn(S, Cn, d).astype(np.float32))
    u = torch.from_numpy(rs.uniform(0.05, 0.95, size=(S, Cn)).astype(np.float32))
    res = engine.run_sampler([pb["spec"]], q0, S, L, eps, inject_momenta=p, inject_uniforms=u)
    o64, o32 = oracle(row, torch.float64), oracle(row, torch.float32)
    compared = sum(compare_with_fp64_chain(res, c, o64, o32, q0[c], S, L, eps, p[:, c], u[:, c], o64.lp_scale(q0[c].double()))
                   for c in range(Cn))
    report(case=row, eps=eps, decisions_compared=compared, accept_rate=float(res.accepted.float().mean()))
    assert compared >= Cn


_VARIANT_SCRIPT = r"""
import sys
sys.path[:0] = [{root!r}, {pkg!r}, {tests!r}]
import test_gpu_deeponet_range as t
for case in t.CASES:
    stats = t.check_row(case, {env!r})
    t.report(case=case.id, variant={env!r}, route=list(t.route_of(case, {env!r})), **stats)
"""


@pytest.mark.gpu
@pytest.mark.parametrize("env", ENVS[1:])
def test_reference_paths_pass_the_same_checker(env):
    """Every row again with the per-layer backward everywhere (VIHMC_DENSE_NOFUSE=1) and with every GEMM on the FP32-SIMT
    kernel (VIHMC_DENSE_SIMT=1); fwd3 rows keep their forward and head3_kernel under both."""
    root = _root()
    script = _VARIANT_SCRIPT.format(root=root, pkg=os.path.join(root, "vi-hmc_b200"), tests=os.path.join(root, "tests"), env=env)
    full = dict(os.environ, **{env: "1"})
    out = subprocess.run([sys.executable, "-c", script], env=full, capture_output=True, text=True, timeout=1500)
    print(out.stdout)
    assert out.returncode == 0, out.stderr[-3000:]
    assert sum(l.startswith("DON_RANGE") for l in out.stdout.splitlines()) == len(CASES)
