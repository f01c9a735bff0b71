"""The MLP log-posterior kernels across their whole supported architecture range, against the fp64 oracle.

The BNN tests elsewhere pin one network (1-10-10-1 tanh, N = 20).  The small-MLP kernel (csrc/mlp_small.cu) accepts 1-4
hidden layers padded to W = 10 / 16 / 32, in_dim <= 64, tanh / relu / sine, both likelihoods, with or without the output
bias, any N (chunks of NC = 24 / 16 / 8 points) and any sens_ind; everything else goes to the dense path (csrc/dense.cu).
CASES below spans that range.  Each row names the path and kernel variant it is meant to reach; the path is confirmed at
run time (a NULL workspace is accepted by the small path only) and the variant against the selection rule of fill_params.

One checker is used everywhere.  g64 / g32 are the fp64 / fp32 CPU oracle gradients (oracle.closures.BnnLogProb, the
reference's own arithmetic).  For every parameter tensor k (the sampled coordinates that fall in it) and for the whole vector
    ||g - g64||_k <= max(1e-5 ||g64||_k, C_FP32 ||g32 - g64||_k)
The second term lets the kernel be as inexact as fp32 itself where fp32 is ill-conditioned (saturated tanh, cancelling bias
gradients); a bound that is per tensor means a small tensor (the output bias, first-layer biases) cannot hide behind max|g|.
Every case must also discriminate: each tensor's bound is at most 1 % of ||g64||_k (checked on the CPU as well, together
with the checker rejecting a zeroed tensor, two swapped coordinates and the neighbouring chain's gradient).
The log-posterior uses the same rule with the scale sum_n |l_n| + sum_i |prior_i| (NLL sums can cancel towards 0), the
predictions per output with the scale sum_j |W_out,j h_j| + |b_out|.
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

import cases
from oracle import closures as oc
from oracle import hamiltorch_restated as hr
from oracle import sensitivity as osens
from vihmc import _lib, engine
from vihmc.spec import LogProbSpec, MLPArch

REL = 1e-5          # relative floor of every bound
# the kernel may be this many times as inexact as the fp32 oracle.  Measured on one B200 (default power limit), worst
# ||g - g64||_k / ||g32 - g64||_k over every tensor of the 9 chains where that ratio decides (the 1e-5 floor does not):
# 25 on the output bias of w32_fast and 19 on the first-layer biases of saturated (both tanh on the small path, whose
# ex2.approx / rcp.approx tanh has an absolute error of ~1e-7 where torch's is ~0.5 ulp), 21 on dense_vi, 10 on w32_2chunk,
# <= 6.3 elsewhere.  At 32 every case still discriminates (bound <= 1 % of every tensor's norm, asserted below).
C_FP32 = 32.0
DISCRIM = 0.01      # a tensor's bound must stay below this fraction of its fp64 gradient norm
ERR_UNSUPPORTED, ERR_WORKSPACE = 2, 3

# route: ("small", padded width W, variant, chunks of NC points) or ("dense",)
#   variant: "fast1" = eval_fast (1-W-W-1 tanh, N <= NC; default for W = 32 and for last_bias = False),
#            "fast2" = eval_fast2 (W <= 16 with the output bias), "generic" = the runtime-layer-loop evaluation
# prior:  "scalar" sigma | "inf" per-coordinate sigma with +inf (flat) entries | "mu" per-coordinate sigma and non-zero mean
#         | "scale2" scalar sigma with prior_scale = 2
# opts:   "unsorted" sens_ind | "kink" x contains 0 and the first-layer biases are 0 (relu pre-activations exactly 0)
Case = namedtuple("Case", "id in_dim widths act loss last_bias N d prior wscale opts route")
CASES = [
    # never run before this file: last_bias = False on the fast v1 path
    Case("ref_nobias", 1, (10, 10), "tanh", "NLL", False, 20, 40, "inf", 1.0, (), ("small", 10, "fast1", 1)),
    # W = 32 fast v1
    Case("w32_fast", 1, (32, 32), "tanh", "NLL", True, 8, None, "scalar", 1.0, (), ("small", 32, "fast1", 1)),
    # multi-chunk gradient (phase B sums partial gradients over the chunks)
    Case("w32_2chunk", 1, (32, 32), "tanh", "NLL", True, 9, None, "mu", 1.0, (), ("small", 32, "generic", 2)),
    # one hidden layer, 38 chunks
    Case("h1_many", 1, (17,), "relu", "NLL", True, 300, None, "scale2", 1.0, (), ("small", 32, "generic", 38)),
    # three hidden layers, in_dim = 3 (runtime input-width loop), regression loss
    Case("h3_in3", 3, (16, 16, 16), "relu", "regression", True, 17, None, "inf", 1.0, (), ("small", 16, "generic", 2)),
    # unequal zero-padded widths, sine, no output bias
    Case("uneven_sine", 5, (17, 3, 29), "sine", "NLL", False, 50, None, "mu", 1.0, (), ("small", 32, "generic", 7)),
    # four hidden layers, in_dim = 64, unsorted VI subset: 62 KB per chain
    Case("max_in_depth", 64, (32, 32, 32, 32), "relu", "NLL", True, 30, 200, "scalar", 1.0, ("unsorted",),
         ("small", 32, "generic", 4)),
    # 163 kB per chain, close to the 200 KiB limit
    Case("near_limit", 2, (32, 32, 32, 32), "tanh", "NLL", True, 9, None, "scale2", 1.0, (), ("small", 32, "generic", 2)),
    Case("tiny", 1, (1,), "tanh", "NLL", True, 1, None, "scalar", 1.0, (), ("small", 10, "generic", 1)),
    # relu'(0) = 0 as torch takes it
    Case("relu_kink", 1, (10, 10), "relu", "NLL", True, 20, None, "inf", 1.0, ("kink",), ("small", 10, "generic", 1)),
    # |z| up to ~8: fast v2 evaluation, persistent sampler with register-resident coordinates (d <= 64)
    Case("saturated", 1, (16, 16), "tanh", "NLL", True, 16, 64, "mu", 5.0, (), ("small", 16, "fast2", 1)),
    # |z| ~ 50
    Case("sine_large", 1, (10, 10), "sine", "NLL", True, 20, 40, "scale2", 20.0, (), ("small", 10, "generic", 1)),
    # one unit past the small kernel
    Case("dense_edge", 1, (33,), "tanh", "NLL", True, 20, None, "scalar", 1.0, (), ("dense",)),
    # smallk first layer, VI subset, no output bias, regression
    Case("dense_vi", 3, (64, 48), "relu", "regression", False, 333, 120, "mu", 1.0, ("unsorted",), ("dense",)),
    # SIMT first layer
    Case("dense_k12", 12, (40, 40), "tanh", "NLL", True, 300, None, "inf", 1.0, (), ("dense",)),
    # tensor-core first layer, long-K weight gradients
    Case("dense_k40", 40, (64, 64), "relu", "NLL", True, 3000, None, "scale2", 1.0, (), ("dense",)),
    # six hidden layers (> 4)
    Case("deep_narrow", 1, (8, 8, 8, 8, 8, 8), "tanh", "NLL", True, 50, None, "mu", 1.0, (), ("dense",)),
    # max_in_depth with d = D: 245 KB per chain on the small path, so dense
    Case("max_in_depth_full", 64, (32, 32, 32, 32), "relu", "NLL", True, 30, None, "inf", 1.0, (), ("dense",)),
]
CASE_BY_ID = {c.id: c for c in CASES}
SMALL = [c for c in CASES if c.route[0] == "small"]
DENSE = [c for c in CASES if c.route[0] == "dense"]


# ---------------------------------------------------------------------------------------------------------------------
# mirror of the small-path selection (csrc/mlp_small.cu fill_params / pick_geometry, csrc/mlp_small.cuh make_layout)
# ---------------------------------------------------------------------------------------------------------------------
def _round_up(v, m):
    return (v + m - 1) // m * m


def small_chain_bytes(W, nh, in_dim, d, fast=0):
    """Shared memory of one chain (make_layout(...).total * 4)."""
    wsw, off = _round_up(W, 4), 0
    for l in range(nh + 1):
        off += (W if l < nh else 1) * (_round_up(in_dim, 4) if l == 0 else wsw)
        off += wsw if l < nh else 4
        if 1 <= l < nh:
            off += W * wsw
    nc = (32 // W) * 8
    ncs = 64 if fast >= 2 else {10: 52, 16: 20, 32: 12}[W] if fast else nc + 4
    off += in_dim * ncs + nh * W * ncs + (0 if fast else nh * W * ncs) + nh * W * ncs + 2 * ncs
    dp = _round_up(d, 4)
    off += 9 * dp
    if fast:
        off += dp + (2 * W + 9) * 33 + 3 + 64
    return 4 * off


def expected_route(case, d=None, generic=False, fast_version=2):
    """The route fill_params picks for this network (the table states it, this rule and the run-time probe confirm it)."""
    nh, d = len(case.widths), d or case_D(case)
    maxw = max(case.widths)
    W = 10 if maxw <= 10 else 16 if maxw <= 16 else 32 if maxw <= 32 else 0
    if case.act == "sine" and (W == 0 or nh > 4):
        return ("unsupported",)
    if W == 0 or nh > 4 or case.in_dim > 64 or small_chain_bytes(W, nh, case.in_dim, d) > 200 * 1024:
        return ("unsupported",) if case.act == "sine" else ("dense",)
    nc = (32 // W) * 8
    fast = (not generic and nh == 2 and case.in_dim == 1 and case.act == "tanh" and case.N <= nc)
    variant = "generic" if not fast else ("fast2" if W <= 16 and case.last_bias and fast_version == 2 else "fast1")
    return ("small", W, variant, -(-case.N // nc))


def chains_per_cta(chain_bytes, C):
    cpb = 1
    while cpb < 4 and C > 148 * 24 * cpb and chain_bytes * cpb * 2 <= 200 * 1024:
        cpb *= 2
    return cpb


# ---------------------------------------------------------------------------------------------------------------------
# problems and oracles
# ---------------------------------------------------------------------------------------------------------------------
def case_D(case):
    return MLPArch(in_dim=case.in_dim, widths=case.widths, out_dim=1, act=case.act, last_bias=case.last_bias).num_params


def tensor_groups(slots, ind):
    """(tensor name, positions in q of the sampled coordinates that fall in that tensor) for every tensor that has some."""
    ind = np.asarray(ind)
    out = []
    for s in slots:
        sel = np.nonzero((ind >= s.offset) & (ind < s.offset + s.numel))[0]
        if sel.size:
            out.append((s.name, sel))
    return out


class Oracle:
    """BnnLogProb likelihood + a per-coordinate Gaussian prior N(mu_i, sigma_i) / prior_scale over the finite sigma_i
    (sigma = inf: no prior on that coordinate, as vihmc_prior_log_norm and the kernels treat it)."""

    def __init__(self, pb, dtype):
        case = pb["case"]
        self.dtype = dtype
        self.net = oc.BnnLogProb(x=pb["x"], y=pb["y"], widths=case.widths, act=case.act, last_bias=case.last_bias, loss=case.loss,
                                 tau_out=pb["tau_out"], prior=("sliced", []), frozen=pb["frozen"], sens_ind=pb["ind_or_none"],
                                 dtype=dtype)
        self.fin = torch.from_numpy(np.isfinite(pb["prior_sigma_np"]))
        self.pmu = torch.from_numpy(pb["prior_mu_np"]).to(dtype)[self.fin]
        self.psg = torch.from_numpy(pb["prior_sigma_np"]).to(dtype)[self.fin]
        self.prior_scale = pb["prior_scale"]

    def prior_terms(self, q):
        return torch.distributions.Normal(self.pmu, self.psg).log_prob(q[self.fin])

    def loglik_terms(self, q):
        r = self.net.forward(q) - self.net.y
        tau = self.net.tau_out
        return -0.5 * tau * r * r if self.net.loss == "regression" else -0.5 * (math.log(tau) + r * r / tau)

    def __call__(self, q):
        return self.net(q) + self.prior_terms(q).sum() / self.prior_scale

    def forward(self, q, x=None):
        return self.net.forward(q, x)

    def lp_scale(self, q):
        """sum_n |l_n| + sum_i |prior_i| / prior_scale: the size of what the log-posterior adds up."""
        with torch.no_grad():
            return float(self.loglik_terms(q).abs().sum() + self.prior_terms(q).abs().sum() / self.prior_scale)

    def out_scale(self, q):
        """per data point: sum_j |W_out,j h_j| + |b_out|, the size of what the output layer adds up."""
        with torch.no_grad():
            full = oc.scatter_vi(self.net.frozen, self.net.sens_ind, q)
            ws = oc.unflatten(self.net.slots, full)
            h, nh = self.net.x, len(self.net.widths)
            for l in range(nh):
                h = oc._ACTS[self.net.act](F.linear(h, ws[2 * l], ws[2 * l + 1]))
            s = h.abs() @ ws[2 * nh].abs().T
            if self.net.last_bias:
                s = s + ws[2 * nh + 1].abs()
            return s[:, 0].numpy()


@functools.lru_cache(maxsize=None)
def problem(case_id):
    """Data, weights, VI split, prior and 9 perturbed chains of one case, from a seed fixed by the case id."""
    case = CASE_BY_ID[case_id]
    rs = np.random.RandomState(zlib.crc32(case.id.encode()) % (2 ** 31))
    slots = oc.mlp_layout(case.in_dim, case.widths, 1, case.last_bias)
    D = oc.layout_numel(slots)
    x = rs.uniform(-1.5, 1.5, size=(case.N, case.in_dim))
    theta = np.empty(D)
    for s in slots:
        fan_in = s.shape[1] if len(s.shape) == 2 else 1
        if s.name.startswith("W"):
            theta[s.offset:s.offset + s.numel] = case.wscale * rs.randn(s.numel) / math.sqrt(s.shape[1])
        else:
            theta[s.offset:s.offset + s.numel] = 0.5 * case.wscale * rs.randn(s.numel) / math.sqrt(fan_in)
    if "kink" in case.opts:
        x[::4] = 0.0
        theta[slots[1].offset:slots[1].offset + slots[1].numel] = 0.0       # layer-0 biases
    x = torch.from_numpy(x.astype(np.float32))
    theta32 = torch.from_numpy(theta.astype(np.float32))
    with torch.no_grad():
        f = oc.mlp_forward(x.double(), oc.unflatten(slots, theta32.double()), len(case.widths), case.act, case.last_bias)
    y = (f + 0.1 * torch.from_numpy(rs.randn(case.N, 1))).float()
    d = case.d or D
    if d < D:
        ind = rs.choice(D, d, replace=False).astype(np.int64)
        if "unsorted" not in case.opts:
            ind = np.sort(ind)
        frozen = theta32.clone()
    else:
        ind, frozen = np.arange(D, dtype=np.int64), None
    vi_sigma = torch.from_numpy((0.01 + 0.04 * rs.rand(D)).astype(np.float32))
    q0 = theta[ind]
    prior_mu = np.zeros(d, np.float32)
    prior_scale, scalar = 1.0, 0.8
    if case.prior == "scalar":
        prior_sigma = None
    elif case.prior == "scale2":
        prior_sigma, prior_scale, scalar = None, 2.0, 1.5
    elif case.prior == "inf":
        prior_sigma = (0.5 + rs.rand(d)).astype(np.float32)
        prior_sigma[rs.rand(d) < 0.2] = np.inf
    else:
        prior_sigma = (0.3 + rs.rand(d)).astype(np.float32)
        prior_mu = (q0 + 0.2 * rs.randn(d)).astype(np.float32)
    sig_np = np.full(d, np.float32(scalar), np.float32) if prior_sigma is None else prior_sigma
    tau_out = 0.01 if case.loss == "NLL" else 100.0
    q = torch.from_numpy((q0[None] + 0.05 * rs.randn(9, d)).astype(np.float32))
    arch = MLPArch(in_dim=case.in_dim, widths=case.widths, out_dim=1, act=case.act, last_bias=case.last_bias)
    spec = LogProbSpec(arch=arch, x=x, y=y, loss=case.loss, tau_out=tau_out,
                       prior_mu=None if case.prior != "mu" else torch.from_numpy(prior_mu),
                       prior_sigma=None if prior_sigma is None else torch.from_numpy(prior_sigma), prior_sigma_scalar=scalar,
                       prior_scale=prior_scale, frozen=frozen, sens_ind=None if frozen is None else ind, vi_sigma=vi_sigma)
    return dict(case=case, slots=slots, D=D, d=d, x=x, y=y, theta=theta32, frozen=frozen, ind=ind,
                ind_or_none=None if frozen is None else ind, vi_sigma=vi_sigma, prior_mu_np=prior_mu, prior_sigma_np=sig_np,
                prior_scale=prior_scale, tau_out=tau_out, q=q, spec=spec, groups=tensor_groups(slots, ind))


@functools.lru_cache(maxsize=None)
def oracle(case_id, dtype):
    return Oracle(problem(case_id), dtype)


def oracle_grads(orc, q):
    """value and gradient of an oracle closure at the fp32 point q (evaluated in the closure's dtype)."""
    lp, g = oc.value_and_grad(orc, q.to(orc.dtype))
    return float(lp), g.double().numpy()


# ---------------------------------------------------------------------------------------------------------------------
# the checker
# ---------------------------------------------------------------------------------------------------------------------
def grad_violations(g, g64, g32, groups, c=C_FP32, floor=0.0):
    """Per tensor and whole vector: ||g - g64|| <= max(REL ||g64||, c ||g32 - g64||, floor).  Returns (violations, worst
    err / bound, largest ||g - g64|| / ||g32 - g64|| -- the observed kernel-to-fp32 error ratio)."""
    g, g64, g32 = (np.asarray(v, np.float64) for v in (g, g64, g32))
    bad, worst, ratio = [], 0.0, 0.0
    for name, sel in list(groups) + [("all", np.arange(g64.size))]:
        err = float(np.linalg.norm(g[sel] - g64[sel]))
        e32 = float(np.linalg.norm(g32[sel] - g64[sel]))
        bound = max(REL * float(np.linalg.norm(g64[sel])), c * e32, floor)
        if not err <= bound:
            bad.append(f"{name}: |g - g64| = {err:.3e} > bound {bound:.3e} (|g64| {np.linalg.norm(g64[sel]):.3e}, fp32 err {e32:.3e})")
        worst = max(worst, err / bound if bound > 0 else (0.0 if err == 0 else math.inf))
        ratio = max(ratio, err / e32 if e32 > 0 else (0.0 if err == 0 else math.inf))
    return bad, worst, ratio


def loose_tensors(g64, g32, groups, c=C_FP32):
    """Tensors whose bound exceeds DISCRIM of their fp64 gradient norm: the checker could not see an error there."""
    out = []
    for name, sel in groups:
        n64 = float(np.linalg.norm(g64[sel]))
        bound = max(REL * n64, c * float(np.linalg.norm(g32[sel] - g64[sel])))
        if not bound <= DISCRIM * n64:
            out.append((name, bound / n64 if n64 > 0 else math.inf))
    return out


def scalar_ok(v, v64, v32, scale, c=C_FP32):
    bound = max(REL * scale, c * abs(v32 - v64))
    return abs(v - v64) <= bound, abs(v - v64) / bound if bound > 0 else math.inf


def assert_grad(g, g64, g32, groups, what, floor=0.0):
    bad, worst, ratio = grad_violations(g, g64, g32, groups, floor=floor)
    assert not bad, f"{what}: " + "; ".join(bad)
    return worst, ratio


def report(**kw):
    print("MLP_RANGE " + json.dumps(kw, default=float), flush=True)


# ---------------------------------------------------------------------------------------------------------------------
# C ABI helpers
# ---------------------------------------------------------------------------------------------------------------------
def _stream():
    return torch.cuda.current_stream().cuda_stream


def probe_route(prob):
    """vihmc_logp_grad with a NULL workspace: the small path needs none and succeeds, the dense path refuses."""
    dev = torch.device("cuda")
    q = torch.zeros(int(prob.d), dtype=torch.float32, device=dev)
    lp = torch.empty(1, dtype=torch.float32, device=dev)
    rc = _lib.load().vihmc_logp_grad(C.byref(prob), 1, q.data_ptr(), lp.data_ptr(), None, None, 0, _stream())
    torch.cuda.synchronize()
    if rc == 0:
        return "small"
    assert rc == ERR_WORKSPACE, (rc, _lib.load().vihmc_last_error().decode())
    return "dense"


def abi_logp_grad_predict(prob, q, N, ws_chains, P=None):
    """vihmc_logp_grad and vihmc_predict for all chains of q with a workspace sized for ws_chains chains."""
    lib = _lib.load()
    dev = torch.device("cuda")
    Cn = q.shape[0]
    ws_bytes = int(lib.vihmc_workspace_bytes(C.byref(prob), ws_chains))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    qd = q.to(dev).contiguous()
    lp = torch.empty(Cn, dtype=torch.float32, device=dev)
    g = torch.empty_like(qd)
    out = torch.empty((Cn, N) if P is None else (Cn, N, P), dtype=torch.float32, device=dev)
    _lib.check(lib.vihmc_logp_grad(C.byref(prob), Cn, qd.data_ptr(), lp.data_ptr(), g.data_ptr(), ws.data_ptr(), ws_bytes, _stream()))
    _lib.check(lib.vihmc_predict(C.byref(prob), Cn, qd.data_ptr(), out.data_ptr(), ws.data_ptr(), ws_bytes, _stream()))
    torch.cuda.synchronize()
    return lp.cpu().numpy(), g.cpu().numpy(), out.cpu().numpy(), ws_bytes


# ---------------------------------------------------------------------------------------------------------------------
# checks shared by the tests and the variant subprocesses
# ---------------------------------------------------------------------------------------------------------------------
def check_logp_grad_predict(case):
    """logp_grad on the 9 chains and predict, against the checker.  Returns the per-case statistics."""
    pb = problem(case.id)
    o64, o32 = oracle(case.id, torch.float64), oracle(case.id, torch.float32)
    q = pb["q"]
    lp, g = engine.logp_grad(pb["spec"], q)
    lp, g = lp.cpu().numpy(), g.cpu().numpy()
    pred = engine.predict(pb["spec"], q).cpu().numpy()
    worst = ratio = lp_worst = pr_worst = 0.0
    for c in range(q.shape[0]):
        lp64, g64 = oracle_grads(o64, q[c])
        lp32, g32 = oracle_grads(o32, q[c])
        assert not loose_tensors(g64, g32, pb["groups"]), (case.id, c, loose_tensors(g64, g32, pb["groups"]))
        w, r = assert_grad(g[c], g64, g32, pb["groups"], f"{case.id} chain {c}")
        worst, ratio = max(worst, w), max(ratio, r)
        ok, lw = scalar_ok(float(lp[c]), lp64, lp32, o64.lp_scale(q[c].double()))
        assert ok, (case.id, c, float(lp[c]), lp64, lp32)
        lp_worst = max(lp_worst, lw)
        with torch.no_grad():
            f64 = o64.forward(q[c].double())[:, 0].numpy()
            f32 = o32.forward(q[c].float())[:, 0].double().numpy()
        scale = o64.out_scale(q[c].double())
        bound = np.maximum(REL * scale, C_FP32 * np.abs(f32 - f64))
        err = np.abs(pred[c].astype(np.float64) - f64)
        assert (err <= bound).all(), (case.id, c, int(np.argmax(err / bound)), float((err / bound).max()))
        pr_worst = max(pr_worst, float((err / bound).max()))
    return dict(grad_err_over_bound=worst, kernel_over_fp32=ratio, logp_err_over_bound=lp_worst, pred_err_over_bound=pr_worst)


def step_size(case):
    """1 / sqrt(largest |eigenvalue| of the fp64 Hessian at chain 0): stable leapfrog with a real energy error."""
    o64 = oracle(case.id, torch.float64)
    q = problem(case.id)["q"][0].double()
    v = torch.from_numpy(np.random.RandomState(0).randn(q.numel()))
    lam = 1.0
    for _ in range(15):
        _, hv = torch.autograd.functional.hvp(o64, q, v / v.norm())
        lam = float(hv.norm())
        v = hv
    return 1.0 / math.sqrt(lam)


def compare_with_fp64_chain(res, c, orc64, orc32, q0, S, L, eps, p, u, lp_scale):
    """One chain of an engine run against hamiltorch restated in fp64 on the same momenta and uniforms: H0 within
    max(1e-5 of the summed terms, C_FP32 x the fp32 oracle's error), and the same decision wherever the fp64 margin
    |min(0, H0 - H1) - log u| exceeds the difference of the energy errors.  Comparison stops at the first (allowed)
    disagreement.  Returns the number of decisions compared."""
    tr, tr32 = {}, {}
    out = torch.stack(hr.sample(orc64, q0.double(), num_samples=S, num_steps_per_sample=L, step_size=eps, momenta=p.double(),
                                uniforms=u, trace=tr))
    hr.sample(orc32, q0.float(), num_samples=S, num_steps_per_sample=L, step_size=eps, momenta=p.float(), uniforms=u, trace=tr32)
    ham = res.hamiltonians[:, c].numpy().astype(np.float64)
    acc = res.accepted[:, c].numpy().astype(bool)
    h0, h1 = np.array(tr["H0"]), np.array(tr["H1"])
    n_ok = 0
    for n in range(S):
        ke = 0.5 * float((p[n].double() ** 2).sum())
        bound = max(REL * (lp_scale + ke), C_FP32 * abs(tr32["H0"][n] - h0[n]) if tr32["accept"][:n] == tr["accept"][:n] else 0.0)
        assert abs(ham[n, 0] - h0[n]) <= bound, (c, n, ham[n, 0], h0[n], tr32["H0"][n])
        if acc[n] != tr["accept"][n]:
            margin = abs(min(0.0, h0[n] - h1[n]) - math.log(float(u[n])))
            dE = abs((ham[n, 1] - ham[n, 0]) - (h1[n] - h0[n]))
            assert margin <= dE + 1e-9, (c, n, margin, dE)
            return n_ok
        n_ok += 1
        if n >= 1:   # row n of a burn = 0 run is the state after iteration n (row 0 is the initial state)
            ref = out[n].detach().numpy()
            np.testing.assert_allclose(res.samples[n, c].numpy(), ref, rtol=1e-3, atol=1e-4 * float(np.abs(ref).max()))
    return n_ok


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the table itself and the checker
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", CASES, ids=[c.id for c in CASES])
def test_table_routes_follow_the_selection_rule(case):
    """The route each row claims is the one fill_params picks for it (the GPU test confirms small / dense at run time)."""
    assert expected_route(case, d=problem(case.id)["d"]) == case.route


def test_table_reaches_the_variants_it_is_meant_to():
    routes = {c.id: c.route for c in CASES}
    assert {r[1] for r in routes.values() if r[0] == "small"} == {10, 16, 32}
    assert {r[2] for r in routes.values() if r[0] == "small"} == {"fast1", "fast2", "generic"}
    assert routes["ref_nobias"][2] == "fast1" and not CASE_BY_ID["ref_nobias"].last_bias
    assert routes["w32_fast"][1:3] == (32, "fast1")
    assert {len(c.widths) for c in SMALL} == {1, 2, 3, 4} and max(c.in_dim for c in SMALL) == 64
    assert max(r[3] for r in routes.values() if r[0] == "small") > 1
    pb = problem("near_limit")
    assert small_chain_bytes(32, 4, 2, pb["d"]) > 150 * 1024
    assert small_chain_bytes(32, 4, 64, case_D(CASE_BY_ID["max_in_depth_full"])) > 200 * 1024
    assert {c.prior for c in CASES} == {"scalar", "inf", "mu", "scale2"}


@pytest.mark.parametrize("case", CASES, ids=[c.id for c in CASES])
def test_checker_accepts_fp32_and_rejects_wrong_gradients(case):
    """For two chains of every case: the fp32 oracle gradient passes; zeroing any one tensor, swapping two coordinates of one
    tensor, or handing in the neighbouring chain's gradient fails; and every tensor's bound stays below 1 % of its norm."""
    pb = problem(case.id)
    o64, o32 = oracle(case.id, torch.float64), oracle(case.id, torch.float32)
    grads = [(oracle_grads(o64, pb["q"][c])[1], oracle_grads(o32, pb["q"][c])[1]) for c in (0, 1)]
    for c, (g64, g32) in enumerate(grads):
        assert not loose_tensors(g64, g32, pb["groups"]), loose_tensors(g64, g32, pb["groups"])
        assert not grad_violations(g32, g64, g32, pb["groups"])[0]
        for name, sel in pb["groups"]:
            g = g32.copy()
            g[sel] = 0.0
            assert grad_violations(g, g64, g32, pb["groups"])[0], ("zeroed", name)
            if sel.size >= 2:
                a, b = sel[np.argmax(g64[sel])], sel[np.argmin(g64[sel])]
                g = g32.copy()
                g[[a, b]] = g[[b, a]]
                assert grad_violations(g, g64, g32, pb["groups"])[0], ("swapped", name)
        other = grads[1 - c][1]
        assert grad_violations(other, g64, g32, pb["groups"])[0], "neighbouring chain"


# ---------------------------------------------------------------------------------------------------------------------
# GPU: every case
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=[c.id for c in CASES])
def test_logp_grad_predict_and_route(case):
    pb = problem(case.id)
    prep = engine.prepare(pb["spec"])
    path = probe_route(prep.problem)
    assert path == case.route[0], (case.id, path)
    stats = check_logp_grad_predict(case)
    kb = small_chain_bytes(case.route[1], len(case.widths), case.in_dim, pb["d"], {"fast1": 1, "fast2": 2}.get(case.route[2], 0)) \
        / 1024 if path == "small" else None
    report(case=case.id, route=list(case.route), confirmed_path=path, smem_kb_per_chain=kb, **stats)


@pytest.mark.gpu
@pytest.mark.parametrize("case", [c for c in SMALL if c.d is None], ids=[c.id for c in SMALL if c.d is None])
def test_sensitivity_matches_oracle(case):
    """vihmc_mlp_sensitivity (d = D only) against oracle.sensitivity.scores, per tensor with the checker's rule plus a floor of
    1e-5 of the whole score vector: a score many orders below the others (tiny's W1 at 1e-9 of them, from a pre-activation
    that nearly cancels) carries fp32's absolute error, which one fp32 sample does not bound reliably."""
    from vihmc import sensitivity as vs

    pb = problem(case.id)
    arch = pb["spec"].arch
    s = vs.eval_std_dydw((pb["x"], pb["y"]), arch, pb["theta"], pb["vi_sigma"])
    s64 = osens.scores(pb["x"].double(), case.widths, case.act, pb["theta"], pb["vi_sigma"], last_bias=case.last_bias,
                       dtype=torch.float64)
    s32 = osens.scores(pb["x"], case.widths, case.act, pb["theta"], pb["vi_sigma"], last_bias=case.last_bias, dtype=torch.float32)
    worst, ratio = assert_grad(s, s64, s32, pb["groups"], f"{case.id} sensitivity", floor=REL * float(np.linalg.norm(s64)))
    report(case=case.id, sensitivity_err_over_bound=worst, sensitivity_kernel_over_fp32=ratio)


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=[c.id for c in CASES])
def test_short_sampling_run_three_ways(case):
    """S = 3, L = 11 with injected momenta and uniforms: the persistent kernel (small path), the general sampler and
    hamiltorch restated on the fp64 oracle."""
    pb = problem(case.id)
    spec, d, S, L, Cn = pb["spec"], pb["d"], 3, 11, 4
    eps = step_size(case)
    rs = np.random.RandomState(7)
    q0 = pb["q"][:Cn]
    p = torch.from_numpy(rs.randn(S, Cn, d).astype(np.float32))
    u = torch.from_numpy(rs.uniform(0.05, 0.95, size=(S, Cn)).astype(np.float32))
    b = engine.run_sampler([spec], q0, S, L, eps, inject_momenta=p, inject_uniforms=u, force_general=True)
    if case.route[0] == "small":
        a = engine.run_sampler([spec], q0, S, L, eps, inject_momenta=p, inject_uniforms=u)
        assert a.gpu_launches == 1
        assert torch.equal(a.accepted, b.accepted)
        scale = max(oracle(case.id, torch.float64).lp_scale(q0[c].double()) for c in range(Cn))
        np.testing.assert_allclose(a.hamiltonians.numpy(), b.hamiltonians.numpy(), rtol=2e-5, atol=REL * scale)
        np.testing.assert_allclose(a.samples.numpy(), b.samples.numpy(), rtol=1e-4, atol=1e-5 * float(q0.abs().max()))
    o64 = oracle(case.id, torch.float64)
    compared = 0
    for c in range(Cn):
        compared += compare_with_fp64_chain(b, c, o64, oracle(case.id, torch.float32), q0[c], S, L, eps, p[:, c], u[:, c],
                                            o64.lp_scale(q0[c].double()))
    report(case=case.id, eps=eps, decisions_compared=compared, accept_rate=float(b.accepted.float().mean()))
    assert compared >= Cn


@pytest.mark.gpu
@pytest.mark.parametrize("force_general", [False, True])
def test_vi_redraw_through_four_layers_and_64_inputs(force_general):
    """Per-sample VI redraw on max_in_depth (three transposed tables, a 64-wide input layer) against the oracle with
    frozen = mu + sigma z on the same normals."""
    case = CASE_BY_ID["max_in_depth"]
    pb = problem(case.id)
    spec, d, D, S, L, Cn = pb["spec"], pb["d"], pb["D"], 3, 5, 2
    eps = step_size(case)
    rs = np.random.RandomState(31)
    q0 = pb["q"][:Cn]
    p = torch.from_numpy(rs.randn(S, Cn, d).astype(np.float32))
    z = torch.from_numpy(rs.randn(S, Cn, D).astype(np.float32))
    u = torch.full((S, Cn), 1e-30)
    res = engine.run_sampler([spec], q0, S, L, eps, inject_momenta=p, inject_uniforms=u, vi_redraw=True, inject_vi_normals=z,
                             force_general=force_general)
    want = pb["frozen"][None, None] + pb["vi_sigma"][None, None] * z
    np.testing.assert_allclose(res.vi_params.numpy(), want.numpy(), rtol=1e-6, atol=1e-7)
    assert bool(res.accepted.all())
    for c in range(Cn):
        orc = Oracle(pb, torch.float64)
        q = q0[c].double()
        for n in range(S):
            orc.net.frozen = want[n, c].double()
            h0 = float(hr.hamiltonian(q, p[n, c].double(), orc))
            q, p1 = hr.leapfrog(q, p[n, c].double(), orc, L, eps)
            h1 = float(hr.hamiltonian(q, p1, orc))
            scale = orc.lp_scale(q) + 0.5 * float((p[n, c].double() ** 2).sum())
            assert abs(float(res.hamiltonians[n, c, 0]) - h0) <= REL * scale, (c, n)
            assert abs(float(res.hamiltonians[n, c, 1]) - h1) <= 10 * REL * scale, (c, n)
            if n >= 1:   # row n: the state after iteration n
                np.testing.assert_allclose(res.samples[n, c].numpy(), q.detach().numpy(), rtol=1e-4, atol=1e-4)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: several chains per CTA
# ---------------------------------------------------------------------------------------------------------------------
def _geometry_problem(which, Cn):
    rs = np.random.RandomState(Cn)
    if which == "ref":
        g = cases.load_golden("bnn_vi_hmc_logp_grad.npz")
        case = cases.bnn_case(g, "d40_nll")
        spec = cases.bnn_spec(case)
        o64, o32 = cases.bnn_oracle(case, torch.float64), cases.bnn_oracle(case, torch.float32)
        groups = tensor_groups(oc.mlp_layout(1, (10, 10)), case["ind"])
        base, chain_bytes = case["mu"].numpy()[case["ind"]], small_chain_bytes(10, 2, 1, case["d"], 2)
        eps, scale_of = 3e-4, (lambda q: float(abs(o64(q))))
    else:
        pb = problem(which)
        spec, o64, o32, groups = pb["spec"], oracle(which, torch.float64), oracle(which, torch.float32), pb["groups"]
        base, chain_bytes = pb["q"][0].numpy(), small_chain_bytes(32, 1, 1, pb["d"])
        eps, scale_of = step_size(CASE_BY_ID[which]), o64.lp_scale
    q = torch.from_numpy((base[None] + 0.05 * rs.randn(Cn, base.size)).astype(np.float32))
    return spec, o64, o32, groups, q, chain_bytes, eps, scale_of


@pytest.mark.gpu
@pytest.mark.parametrize("which,Cn,cpb", [("ref", 3600, 2), ("ref", 7107, 4), ("h1_many", 7107, 4)])
def test_several_chains_per_cta_vs_fp64(which, Cn, cpb):
    """pick_geometry packs 2 chains into a CTA above 3 552 chains and 4 above 7 104 (7 107 leaves 3 in the last CTA).  Checked
    chain by chain on every slot of the first, second, middle and last two CTAs: logp_grad and a short persistent-kernel run."""
    spec, o64, o32, groups, q, chain_bytes, eps, scale_of = _geometry_problem(which, Cn)
    assert chains_per_cta(chain_bytes, Cn) == cpb
    blocks = -(-Cn // cpb)
    picks = sorted({c for b in (0, 1, blocks // 2, blocks - 2, blocks - 1) for c in range(b * cpb, min(Cn, (b + 1) * cpb))})
    assert {c % cpb for c in picks} == set(range(cpb)) and Cn - 1 in picks
    lp, g = engine.logp_grad(spec, q)
    lp, g = lp.cpu().numpy(), g.cpu().numpy()
    for c in picks:
        lp64, g64 = oracle_grads(o64, q[c])
        lp32, g32 = oracle_grads(o32, q[c])
        assert_grad(g[c], g64, g32, groups, f"{which} C={Cn} chain {c}")
        assert scalar_ok(float(lp[c]), lp64, lp32, abs(lp64) if which == "ref" else scale_of(q[c].double()))[0], (c, lp[c], lp64)
    S, L, d = 2, 4, q.shape[1]
    rs = np.random.RandomState(3)
    p = torch.from_numpy(rs.randn(S, Cn, d).astype(np.float32))
    u = torch.from_numpy(rs.uniform(0.05, 0.95, size=(S, Cn)).astype(np.float32))
    res = engine.run_sampler([spec], q, S, L, eps, inject_momenta=p, inject_uniforms=u)
    assert res.gpu_launches == 1
    for c in picks:
        compare_with_fp64_chain(res, c, o64, o32, q[c], S, L, eps, p[:, c], u[:, c], scale_of(q[c].double()))


# ---------------------------------------------------------------------------------------------------------------------
# GPU: dense chain batches (c0 > 0)
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("frozen_rows", [False, True])
def test_dense_chain_batches_mlp(frozen_rows):
    """vihmc_logp_grad / vihmc_predict for 7 chains with the workspace of 2: dense_run processes the chains in batches, so the
    offsets of q, logp, grad, the predictions and (frozen_chain_stride = D, as the VI redraw sets it) each chain's own row of
    frozen weights are exercised for c0 > 0."""
    case = CASE_BY_ID["dense_vi"]
    pb = problem(case.id)
    prep = engine.prepare(pb["spec"])
    prob = _lib.Problem.from_buffer_copy(prep.problem)
    Cn, D = 7, pb["D"]
    rs = np.random.RandomState(12)
    q = torch.from_numpy((pb["q"][0].numpy()[None] + 0.05 * rs.randn(Cn, pb["d"])).astype(np.float32))
    rows = None
    if frozen_rows:
        rows = (pb["frozen"][None] + pb["vi_sigma"][None] * torch.from_numpy(rs.randn(Cn, D).astype(np.float32))).contiguous()
        rows_dev = rows.cuda()
        prob.frozen, prob.frozen_chain_stride = rows_dev.data_ptr(), D
    lib = _lib.load()
    assert lib.vihmc_workspace_bytes(C.byref(prob), 2) < lib.vihmc_workspace_bytes(C.byref(prob), Cn)
    for ws_chains in (2, 1):
        lp, g, pred, _ = abi_logp_grad_predict(prob, q, case.N, ws_chains)
        for c in range(Cn):
            o64, o32 = Oracle(pb, torch.float64), Oracle(pb, torch.float32)
            if frozen_rows:
                o64.net.frozen, o32.net.frozen = rows[c].double(), rows[c].float()
            lp64, g64 = oracle_grads(o64, q[c])
            lp32, g32 = oracle_grads(o32, q[c])
            assert_grad(g[c], g64, g32, pb["groups"], f"batch chain {c}")
            assert scalar_ok(float(lp[c]), lp64, lp32, o64.lp_scale(q[c].double()))[0], (c, lp[c], lp64)
            with torch.no_grad():
                f64 = o64.forward(q[c].double())[:, 0].numpy()
                f32 = o32.forward(q[c])[:, 0].double().numpy()
            bound = np.maximum(REL * o64.out_scale(q[c].double()), C_FP32 * np.abs(f32 - f64))
            assert (np.abs(pred[c] - f64) <= bound).all(), c


@pytest.mark.gpu
def test_dense_chain_batches_deeponet():
    """The small DeepONet VI case through the same 7-chains-in-batches-of-2 call, against its fp64 oracle."""
    inp = cases.don_inputs("small")
    spec = cases.don_spec(inp, "vi")
    prep = engine.prepare(spec)
    o64, o32 = cases.don_oracle(inp, "vi", torch.float64), cases.don_oracle(inp, "vi", torch.float32)
    arch = inp["arch"]
    slots = oc.deeponet_layout(arch.width_branch, arch.width_trunk, arch.in_branch, arch.in_trunk, arch.depth_branch,
                               arch.depth_trunk, arch.output_neurons)
    groups = tensor_groups(slots, inp["ind"])
    Cn = 7
    rs = np.random.RandomState(2)
    q = torch.from_numpy((inp["mu"].numpy()[inp["ind"]][None] + 0.01 * rs.randn(Cn, spec.d)).astype(np.float32))
    lib = _lib.load()
    assert lib.vihmc_workspace_bytes(C.byref(prep.problem), 2) < lib.vihmc_workspace_bytes(C.byref(prep.problem), Cn)
    lp, g, pred, _ = abi_logp_grad_predict(prep.problem, q, spec.N, 2, P=spec.P)
    for c in range(Cn):
        lp64, g64 = oracle_grads(o64, q[c])
        lp32, g32 = oracle_grads(o32, q[c])
        assert_grad(g[c], g64, g32, groups, f"deeponet batch chain {c}")
        with torch.no_grad():
            qq = q[c].double()
            r = o64.forward(qq) - o64.y
            scale = float((0.5 * (r * r / o64.tau_out)).abs().sum() + o64._dist.log_prob(qq).abs().sum()) + 0.5 * abs(math.log(o64.tau_out)) * r.numel()
            f64 = o64.forward(qq).numpy()
            f32 = o32.forward(q[c]).double().numpy()
        assert scalar_ok(float(lp[c]), lp64, lp32, scale)[0], (c, lp[c], lp64)
        bound = np.maximum(REL * np.abs(f64).max(axis=1, keepdims=True), C_FP32 * np.abs(f32 - f64))
        assert (np.abs(pred[c] - f64) <= bound).all(), c


# ---------------------------------------------------------------------------------------------------------------------
# GPU: kernel variants (environment switches are read once per process) and refusals
# ---------------------------------------------------------------------------------------------------------------------
_VARIANT_SCRIPT = r"""
import sys
sys.path[:0] = [{root!r}, {pkg!r}, {tests!r}]
import test_gpu_mlp_range as t
for cid in sys.argv[1].split(","):
    stats = t.check_logp_grad_predict(t.CASE_BY_ID[cid])
    t.report(case=cid, variant={variant!r}, **stats)
"""


@pytest.mark.gpu
@pytest.mark.parametrize("env", ["VIHMC_SMALL_GENERIC", "VIHMC_SMALL_FAST", "VIHMC_DENSE_SIMT"])
def test_kernel_variants_pass_the_same_checker(env):
    """Every case's logp_grad and predict check again under the generic small evaluation, fast v1 instead of v2 and the
    FP32-SIMT dense GEMMs."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    ids = [c.id for c in (DENSE if env == "VIHMC_DENSE_SIMT" else SMALL)]
    script = _VARIANT_SCRIPT.format(root=root, pkg=os.path.join(root, "vi-hmc_b200"), tests=os.path.join(root, "tests"),
                                    variant=f"{env}=1")
    full = dict(os.environ, **{env: "1"})
    out = subprocess.run([sys.executable, "-c", script, ",".join(ids)], env=full, capture_output=True, text=True, timeout=900)
    print(out.stdout)
    assert out.returncode == 0, out.stderr[-3000:]
    assert sum(l.startswith("MLP_RANGE") for l in out.stdout.splitlines()) == len(ids)


@pytest.mark.gpu
@pytest.mark.parametrize("base", ["dense_edge", "max_in_depth_full"])
def test_sine_outside_the_small_kernel_is_refused(base):
    """The dense path has no sine: such a network must raise VIHMC_ERR_UNSUPPORTED, not return numbers."""
    case = CASE_BY_ID[base]._replace(act="sine")
    assert expected_route(case) == ("unsupported",)
    pb = problem(base)
    arch = MLPArch(in_dim=case.in_dim, widths=case.widths, out_dim=1, act="sine", last_bias=case.last_bias)
    spec = LogProbSpec(arch=arch, x=pb["x"], y=pb["y"], loss=case.loss, tau_out=pb["tau_out"], prior_sigma_scalar=1.0)
    q = pb["q"][:2]
    for call in (lambda: engine.logp_grad(spec, q), lambda: engine.predict(spec, q),
                 lambda: engine.run_sampler([spec], q, 2, 3, 1e-4)):
        with pytest.raises(_lib.VihmcError) as e:
            call()
        assert e.value.code == ERR_UNSUPPORTED
