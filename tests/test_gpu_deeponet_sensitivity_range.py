"""The DeepONet sensitivity kernel (csrc/don_sensitivity.cu, vihmc_deeponet_sensitivity) across its supported architecture
range, against an fp64 Jacobian oracle.

The scores decide which coordinates HMC samples (select_indices -> gradient_indices_<uid>.npy); a wrong score does not fail
a run, it samples the wrong split.  tests/test_sensitivity.py pins four golden architectures (equal widths, the (t, x) feature
layer, tile sizes NB = 1, 2, 7, mostly rank-deficient Gram matrices).  CASES below reaches what those do not:
    every tile size NB = ceil(max(widths, K) / 16) = 1..8 of don_sens_backward_kernel<ACT, NB>, including the 197 KB
    backward and 128 KB Cholesky shared-memory configuration at NB = 8;
    unequal branch / trunk widths (one stack runs padded to the other's tile), K above, below and equal to the widths, K = 1;
    raw trunk inputs (impose_bc = False: the trunk's row stride is in_trunk);
    full-rank branch Gram matrices at the shipped shape and at K = 128, rank-deficient ones, and a zero pivot in the middle of G
    (singular_middle: an exactly zero trunk feature and a duplicated branch feature), where the 1e-12 dmax rule zeroes one
    row of R and the later pivots are not zero;
    in_branch > 128 (the score kernel's gridDim.y > 1) and in_branch = 6145, the first input whose forward row pair exceeds
    the 48 KB of shared memory a launch gets without opting in;
    the per-batch average of the reference's loader with unequal P per batch.
A K above a stack's last hidden width w caps that Gram matrix's rank at w + 1 (its features are an affine image of w numbers):
the `ranks` column says so, and the CPU test confirms every rank and zero pivot from the fp64 Gram matrices.  The branch Gram
matrices of nb7 and nb8_kmax are clearly full rank (smallest pivot 4e-7 and 1e-7 of the largest diagonal entry); their trunk
Gram matrices are not: the trunk's outputs are smooth functions of the two numbers (t, x), so the pivots decay to the
1e-12 dmax rule itself (19 and 33 of them lie within 1e3 of it), and which of those rows the kernel zeroes is a matter of
rounding -- at no visible cost, since such a pivot carries 1e-12 of the sum.

The oracle does not share the kernel's algebra: torch.func.vmap(grad(...)) gives d out[n, p] / d w for every (n, p) pair of
oracle.closures.deeponet_forward, squared and averaged; the fp32 twin of that computation gives the checker's fp32 error.
On the CPU it must equal oracle.sensitivity.deeponet_scores (the per-output autograd loop pinned by the golden vectors), and
an fp64 restatement of the kernel's algorithm (Gram -> PSD Cholesky with the zero-row rule -> seeded back-propagations ->
E h^2 contractions) must equal it to 1e-10 on every row, the singular ones included.

The checker is the one of test_gpu_mlp_range, per parameter tensor (the scalar output bias is a tensor of its own):
    ||s - s64||_k <= max(REL ||s64||_k, C_FP32 ||s32 - s64||_k, REL ||s64||),
the last term a floor of REL times the whole vector, as in its MLP sensitivity test.  Every row must discriminate (each
tensor's bound at most DISCRIM of its norm; the output bias, whose score sigma_b^2 can sit below the floor, is required
bit-exact instead), and the checker must reject, on every row where they are more than DISCRIM away from the truth, the
restatement with the seeds taken from R^T instead of R, with the branch and trunk factors swapped, with sigma shifted by
one coordinate, with act' of layer l in place of layer l - 1, and (feature-layer rows) with the trunk's first-layer scores
computed from the raw (t, x) instead of the five features.
"""
from __future__ import annotations

import ctypes as C
import functools
import json
import math
import zlib
from collections import namedtuple

import numpy as np
import pytest
import torch

from oracle import closures as oc
from oracle import sensitivity as osens
from test_gpu_mlp_range import C_FP32, DISCRIM, ERR_UNSUPPORTED, ERR_WORKSPACE, REL, assert_grad, grad_violations, tensor_groups
from vihmc import _lib
from vihmc.spec import DeepONetArch, act_code

PIVOT_TOL = 1e-12              # don_sens_chol_kernel: a pivot <= PIVOT_TOL * max diag(G) gives a zero row of R
MAX_DIM = 128                  # kMaxDim: widths and output neurons
MAX_FWD_SMEM = 232448          # kMaxForwardSmem: two forward rows of max(input, widths) floats, 227 KB
MAX_INPUT = MAX_FWD_SMEM // 8  # 29 056
DEFAULT_SMEM = 48 * 1024       # what a launch gets without cudaFuncAttributeMaxDynamicSharedMemorySize
RELU_MARGIN = 1e-4             # every relu pre-activation at least this far from the kink
JAC_CHUNK = 1 << 22            # elements of one vmap(grad) chunk of the Jacobian oracle (pairs x D)

# in_trunk: None = the (t, x) feature layer (impose_bc, 5 features); an integer = that many raw trunk inputs (impose_bc = False)
# batches:  None = one batch of N functions x P trunk points; else [(n, p), ...] averaged per batch as the reference's loader
# ranks:    (rank of the branch Gram B^T B, rank of the trunk Gram T^T T), per batch
Case = namedtuple("Case", "id in_branch in_trunk wb db wt dt K act N P batches ranks")
CASES = [
    Case("nb1_full_rank", 7, None, 16, 3, 16, 3, 16, "tanh", 40, 60, None, [(16, 16)]),
    # NB 2 from padding 17 up to 32; out % 4 != 0 in the score kernel
    Case("nb2_odd17", 10, None, 17, 3, 12, 4, 9, "relu", 30, 45, None, [(9, 9)]),
    # NB 3 set by K = 40 above both widths: ranks capped at width + 1
    Case("nb3_k_above_w", 7, None, 20, 3, 24, 3, 40, "tanh", 50, 64, None, [(21, 25)]),
    Case("nb4_k_below_w", 12, 2, 64, 4, 64, 3, 4, "tanh", 20, 30, None, [(4, 4)]),
    # NB 5 set by the trunk only; the branch runs padded to its tile
    Case("nb5_trunk_tile", 7, None, 20, 3, 72, 3, 12, "relu", 30, 40, None, [(12, 12)]),
    Case("nb6_raw12", 9, 12, 96, 3, 40, 3, 33, "relu", 40, 50, None, [(33, 33)]),
    # the shipped architecture with N, P > K: a full-rank branch Gram, trunk pivots down to the zero-row rule
    Case("nb7_shipped_full_rank", 101, None, 100, 9, 100, 9, 100, "tanh", 110, 104, None, [(100, 100)]),
    # 197 KB backward and 128 KB Cholesky shared memory
    Case("nb8_kmax", 7, None, 128, 3, 128, 3, 128, "tanh", 140, 130, None, [(128, 123)]),
    Case("nb8_odd", 33, None, 127, 2, 119, 3, 113, "relu", 30, 25, None, [(30, 25)]),
    Case("n1_p3", 7, None, 16, 3, 20, 3, 16, "tanh", 1, 3, None, [(1, 3)]),
    # trunk last-layer row 5 and its bias zeroed (exact zero pivot at k = 5), branch row 11 a copy of row 3 (a Schur pivot
    # of rounding size at k = 11)
    Case("singular_middle", 7, None, 24, 3, 24, 3, 24, "tanh", 60, 80, None, [(23, 23)]),
    # the smallest depth and VIHMC_MAX_LAYERS
    Case("depth2_16", 7, None, 16, 2, 16, 16, 16, "tanh", 30, 40, None, [(16, 16)]),
    # score kernel gridDim.y = 3, the bias lane on blockIdx.y = 0 only
    Case("in_branch300", 300, None, 24, 3, 24, 3, 12, "relu", 30, 40, None, [(12, 12)]),
    # 2 x 6145 x 4 B = 49 160 B of forward shared memory: past the 48 KB default
    Case("in_branch6145", 6145, None, 16, 2, 16, 2, 8, "tanh", 8, 16, None, [(8, 8)]),
    Case("k1", 7, None, 16, 3, 16, 3, 1, "tanh", 20, 30, None, [(1, 1)]),
    Case("loader_unequal", 12, None, 16, 3, 16, 3, 8, "tanh", None, None, [(1, 9), (1, 13), (4, 40)], [(1, 8), (1, 8), (4, 8)]),
]
CASE_BY_ID = {c.id: c for c in CASES}
IDS = [c.id for c in CASES]
# pivots the fp64 Cholesky zeroes that are not simply the trailing K - rank ones
MIDDLE_ZERO_PIVOTS = {"singular_middle": ([11], [5])}
ORACLE_CHECK_ROWS = ["nb1_full_rank", "nb2_odd17", "nb4_k_below_w", "n1_p3", "depth2_16", "k1", "loader_unequal"]
MUTANTS = ("seeds from R^T", "factors swapped", "sigma shifted", "act' of layer l", "raw (t, x) first-layer scores")


def arch_of(case, **kw):
    a = dict(width_branch=case.wb, width_trunk=case.wt, in_branch=case.in_branch, in_trunk=5 if case.in_trunk is None else case.in_trunk,
             depth_branch=case.db, depth_trunk=case.dt, output_neurons=case.K, act=case.act, impose_bc=case.in_trunk is None)
    a.update(kw)
    return DeepONetArch(**a)


def arch_kwargs(arch):
    return dict(width_branch=arch.width_branch, width_trunk=arch.width_trunk, in_branch=arch.in_branch, in_trunk=arch.in_trunk,
                depth_branch=arch.depth_branch, depth_trunk=arch.depth_trunk, output_neurons=arch.output_neurons, act=arch.act,
                impose_bc=arch.impose_bc)


def batch_shapes(case):
    return case.batches or [(case.N, case.P)]


def tile_nb(case):
    return -(-max(case.wb, case.wt, case.K) // 16)


def report(**kw):
    print("DON_SENS_RANGE " + json.dumps(kw, default=float), flush=True)


# ---------------------------------------------------------------------------------------------------------------------
# problems
# ---------------------------------------------------------------------------------------------------------------------
def _slot(slots, name):
    return next(s for s in slots if s.name == name)


def stack_params(slots, theta, prefix, depth):
    """[(W_l, b_l)] of one stack as views of the flat vector."""
    ws = {s.name: theta[s.offset:s.offset + s.numel].view(s.shape) for s in slots}
    return [(ws[f"{prefix}W{l}"], ws[f"{prefix}b{l}"]) for l in range(depth)]


def stack_forward(x, params, act):
    """Pre-activations and outputs of every layer (the last one linear), in the dtype of x."""
    f = {"tanh": torch.tanh, "relu": torch.relu}[act]
    zs, hs, h = [], [], x
    for l, (W, b) in enumerate(params):
        z = h @ W.T + b
        h = f(z) if l < len(params) - 1 else z
        zs.append(z)
        hs.append(h)
    return zs, hs


def trunk_input(case, x2):
    """What the trunk's first layer reads: the five features of (t, x), or the raw trunk inputs."""
    return x2 if case.in_trunk is not None else oc.trunk_features(x2.unsqueeze(0))[0]


def _draw(case, attempt):
    rs = np.random.RandomState((zlib.crc32(case.id.encode()) + 7919 * attempt) % (2 ** 31))
    arch = arch_of(case)
    slots = oc.deeponet_layout(**{k: v for k, v in arch_kwargs(arch).items() if k not in ("act", "impose_bc")})
    D = oc.layout_numel(slots)
    assert D == arch.num_params
    batches = []
    for n, p in batch_shapes(case):
        x1 = rs.uniform(-1.0, 1.0, size=(n, case.in_branch))
        if case.in_trunk is None:
            x2 = np.stack([rs.uniform(0.0, 1.0, p), rs.uniform(-1.0, 1.0, p)], axis=1)   # (t, x)
        else:
            x2 = rs.uniform(-1.0, 1.0, size=(p, case.in_trunk))
        batches.append((torch.from_numpy(x1.astype(np.float32)), torch.from_numpy(x2.astype(np.float32))))
    theta = np.empty(D)
    for s in slots:
        if s.name == "b":
            theta[0] = 0.5
        else:
            fan_in = (_slot(slots, s.name[:2] + "W" + s.name[3:]) if s.name[2] == "b" else s).shape[1]
            theta[s.offset:s.offset + s.numel] = rs.randn(s.numel) / math.sqrt(fan_in)
    if case.id == "singular_middle":
        Wt, bt = _slot(slots, f"trW{case.dt - 1}"), _slot(slots, f"trb{case.dt - 1}")
        wt = Wt.shape[1]
        theta[Wt.offset + 5 * wt:Wt.offset + 6 * wt] = 0.0
        theta[bt.offset + 5] = 0.0
        Wb, bb = _slot(slots, f"brW{case.db - 1}"), _slot(slots, f"brb{case.db - 1}")
        wb = Wb.shape[1]
        theta[Wb.offset + 11 * wb:Wb.offset + 12 * wb] = theta[Wb.offset + 3 * wb:Wb.offset + 4 * wb]
        theta[bb.offset + 11] = theta[bb.offset + 3]
    sigma = np.exp(rs.uniform(math.log(1e-3), math.log(1e-1), size=D))
    return slots, D, batches, torch.from_numpy(theta.astype(np.float32)), torch.from_numpy(sigma.astype(np.float32))


def relu_margin(case, slots, batches, theta):
    """Smallest |pre-activation| of a hidden layer at the VI means, over every batch (fp64)."""
    th = theta.double()
    m = math.inf
    for x1, x2 in batches:
        for prefix, depth, x in (("br", case.db, x1.double()), ("tr", case.dt, trunk_input(case, x2.double()))):
            zs, _ = stack_forward(x, stack_params(slots, th, prefix, depth), case.act)
            m = min(m, min(float(z.abs().min()) for z in zs[:-1]))
    return m


@functools.lru_cache(maxsize=None)
def problem(case_id):
    """Inputs, VI means and stds of one row from a seed fixed by its id; a relu row is redrawn (next attempt) until every
    hidden pre-activation is at least RELU_MARGIN from 0, so that fp32 and fp64 take the same branch of relu'."""
    case = CASE_BY_ID[case_id]
    for attempt in range(50):
        slots, D, batches, theta, sigma = _draw(case, attempt)
        if case.act != "relu" or relu_margin(case, slots, batches, theta) >= RELU_MARGIN:
            break
    else:
        raise AssertionError(f"{case_id}: no seed with relu pre-activations away from 0")
    return dict(case=case, slots=slots, D=D, batches=batches, theta=theta, sigma=sigma, attempt=attempt,
                groups=tensor_groups(slots, np.arange(D)))


# ---------------------------------------------------------------------------------------------------------------------
# the Jacobian oracle (independent of the kernel's algebra)
# ---------------------------------------------------------------------------------------------------------------------
def jacobian_scores(kw, batches, mu, sigma, dtype):
    """sigma^2 * mean_{n, p} (d out[n, p] / d w)^2 per batch, averaged over the batches: the per-pair gradient of
    oracle.closures.deeponet_forward by torch.func.vmap(grad), in chunks of pairs, summed in `dtype`."""
    slots = oc.deeponet_layout(kw["width_branch"], kw["width_trunk"], kw["in_branch"], kw["in_trunk"], kw["depth_branch"],
                               kw["depth_trunk"], kw["output_neurons"])
    w, sg = mu.to(dtype), sigma.to(dtype)
    D = w.numel()

    def out(w, xb, xt):
        return oc.deeponet_forward(xb.reshape(1, 1, -1), xt.reshape(1, 1, -1), oc.unflatten(slots, w), kw["depth_branch"],
                                   kw["depth_trunk"], kw["act"], kw["impose_bc"]).reshape(())

    per_pair = torch.func.vmap(torch.func.grad(out), in_dims=(None, 0, 0))
    total = torch.zeros(D, dtype=dtype)
    for xb, xt in batches:
        xb, xt = xb.to(dtype).reshape(-1, kw["in_branch"]), xt.to(dtype).reshape(-1, xt.shape[-1])
        n, p = xb.shape[0], xt.shape[0]
        idx = torch.arange(n * p)
        chunk = max(1, JAC_CHUNK // D)
        acc = torch.zeros(D, dtype=dtype)
        with torch.no_grad():
            for s in range(0, n * p, chunk):
                i = idx[s:s + chunk]
                J = per_pair(w, xb[i // p], xt[i % p])
                acc += (J * J).sum(0)
        total += acc / (n * p) * sg * sg
    return (total / len(batches)).double().numpy()


@functools.lru_cache(maxsize=None)
def oracle(case_id, dtype):
    pb = problem(case_id)
    return jacobian_scores(arch_kwargs(arch_of(pb["case"])), pb["batches"], pb["theta"], pb["sigma"], dtype)


# ---------------------------------------------------------------------------------------------------------------------
# fp64 restatement of the kernel's algorithm, with the mutants' switches
# ---------------------------------------------------------------------------------------------------------------------
def chol_psd(G, pivots=False):
    """don_sens_chol_kernel in fp64: upper R with R^T R = G, a pivot <= PIVOT_TOL * max diag(G) gives a zero row.
    Returns (R, indices of the zeroed pivots[, every pivot / max diag(G)])."""
    A = G.clone()
    K = A.shape[0]
    dmax = float(torch.diagonal(A).max())
    tol = PIVOT_TOL * dmax
    zero, piv = [], []
    for k in range(K):
        piv.append(float(A[k, k]) / dmax)
        p = math.sqrt(float(A[k, k])) if float(A[k, k]) > tol else 0.0
        A[k, :k] = 0.0
        if p == 0.0:
            A[k, k:] = 0.0
            zero.append(k)
            continue
        A[k, k] = p
        A[k, k + 1:] /= p
        A[k + 1:, k + 1:] -= torch.outer(A[k, k + 1:], A[k, k + 1:])
    return (A, zero, piv) if pivots else (A, zero)


def _act_deriv(h, act):
    """act' from the layer's output, as act_deriv_from_output."""
    return 1.0 - h * h if act == "tanh" else (h > 0).to(h.dtype)


def restated_scores(case_id, mutant=None):
    """The kernel's algorithm in fp64: forward at the VI means, G = F^T F of both stacks' outputs, PSD Cholesky, K seeded
    back-propagations per row (the branch seeded with the trunk's factor and vice versa), E_l = sum_r delta_l^2 and
    score(W_l[a, b]) = sigma^2 / (N P) sum_rows E_l[a] h_{l-1}[b]^2.  `mutant` names one of MUTANTS."""
    pb = problem(case_id)
    case, slots, D = pb["case"], pb["slots"], pb["D"]
    th = pb["theta"].double()
    sig = pb["sigma"].double()
    if mutant == "sigma shifted":
        sig = torch.roll(sig, -1)
    total = torch.zeros(D, dtype=torch.float64)
    for x1, x2 in pb["batches"]:
        xb, xt = x1.double(), x2.double()
        tin = trunk_input(case, xt)
        stacks = [("br", case.db, xb), ("tr", case.dt, tin)]
        hs = {pre: stack_forward(x, stack_params(slots, th, pre, depth), case.act)[1] for pre, depth, x in stacks}
        RB, _ = chol_psd(hs["br"][-1].T @ hs["br"][-1])
        RT, _ = chol_psd(hs["tr"][-1].T @ hs["tr"][-1])
        if mutant == "factors swapped":
            RB, RT = RT, RB
        if mutant == "seeds from R^T":
            RB, RT = RB.T, RT.T
        n, p = xb.shape[0], xt.shape[0]
        s = torch.zeros(D, dtype=torch.float64)
        s[0] = sig[0] ** 2
        for (pre, depth, x), seed in zip(stacks, (RT, RB)):
            params = stack_params(slots, th, pre, depth)
            h = hs[pre]
            delta = seed.expand(x.shape[0], -1, -1)
            for l in range(depth - 1, -1, -1):
                E = (delta * delta).sum(1)
                inp = x if l == 0 else h[l - 1]
                if mutant == "raw (t, x) first-layer scores" and pre == "tr" and l == 0:
                    inp = torch.cat([xt, torch.zeros(xt.shape[0], 3, dtype=xt.dtype)], 1)
                Ws, bs = _slot(slots, f"{pre}W{l}"), _slot(slots, f"{pre}b{l}")
                s[Ws.offset:Ws.offset + Ws.numel] = (E.T @ (inp * inp)).reshape(-1) / (n * p) * sig[Ws.offset:Ws.offset + Ws.numel]**2
                s[bs.offset:bs.offset + bs.numel] = E.sum(0) / (n * p) * sig[bs.offset:bs.offset + bs.numel] ** 2
                if l == 0:
                    break
                hp = h[l - 1]
                if mutant == "act' of layer l":
                    hp = torch.zeros_like(h[l - 1])
                    m = min(hp.shape[1], h[l].shape[1])
                    hp[:, :m] = h[l][:, :m]
                    ap = _act_deriv(hp, case.act)
                    ap[:, m:] = 0.0
                else:
                    ap = _act_deriv(hp, case.act)
                delta = (delta @ params[l][0]) * ap[:, None, :]
        total += s
    return (total / len(pb["batches"])).numpy()


@functools.lru_cache(maxsize=None)
def restated(case_id, mutant=None):
    return restated_scores(case_id, mutant)


def gram_pivots(case_id):
    """[(branch pivots, trunk pivots)] per batch: the pivots A[k, k] / max diag(G) the fp64 PSD Cholesky meets (before the
    zero-row rule), from the fp64 Gram matrices of the last layer's outputs."""
    pb = problem(case_id)
    case, th = pb["case"], pb["theta"].double()
    out = []
    for x1, x2 in pb["batches"]:
        res = []
        for pre, depth, x in (("br", case.db, x1.double()), ("tr", case.dt, trunk_input(case, x2.double()))):
            F = stack_forward(x, stack_params(pb["slots"], th, pre, depth), case.act)[1][-1]
            _, _, piv = chol_psd(F.T @ F, pivots=True)
            res.append(np.array(piv))
        out.append(tuple(res))
    return out


# ---------------------------------------------------------------------------------------------------------------------
# the checker with the floor of the sensitivity tests
# ---------------------------------------------------------------------------------------------------------------------
def floor_of(s64):
    return REL * float(np.linalg.norm(s64))


def bounds(s64, s32, groups):
    """(name, positions, fp64 norm, bound) per tensor."""
    fl = floor_of(s64)
    return [(name, sel, float(np.linalg.norm(s64[sel])), max(REL * float(np.linalg.norm(s64[sel])),
                                                            C_FP32 * float(np.linalg.norm(s32[sel] - s64[sel])), fl))
            for name, sel in groups]


def rejected(s, s64, s32, groups):
    return bool(grad_violations(s, s64, s32, groups, floor=floor_of(s64))[0])


def differs(s, s64, groups):
    return any(float(np.linalg.norm(s[sel] - s64[sel])) > DISCRIM * float(np.linalg.norm(s64[sel])) for _, sel in groups)


# ---------------------------------------------------------------------------------------------------------------------
# mirror of make_plan's workspace (csrc/don_sensitivity.cu)
# ---------------------------------------------------------------------------------------------------------------------
def _align256(x):
    return (x + 255) // 256 * 256


def workspace_bytes(arch, N, P):
    """vihmc_deeponet_sensitivity_workspace_bytes: 0 for what make_plan refuses."""
    if arch.act not in ("tanh", "relu"):
        return 0
    da = [o for o, _ in arch.stack_dims("branch")]
    db = [o for o, _ in arch.stack_dims("trunk")]
    K = arch.output_neurons
    if max(da + db + [K]) > MAX_DIM:
        return 0
    if 2 * max([arch.in_branch, arch.in_trunk] + da + db) * 4 > MAX_FWD_SMEM:
        return 0
    acts_br, acts_tr = N * sum(da), P * sum(db)
    return (_align256(P * 5 * 4) + 2 * _align256(acts_br * 4) + 2 * _align256(acts_tr * 4) + _align256(2 * K * K * 8)
            + _align256(2 * K * K * 4))


def abi_problem(arch, N, P):
    """The vihmc_problem engine.prepare fills, without a device (the data pointers stay NULL: only sizes are read)."""
    p = _lib.Problem()
    p.model_kind, p.act, p.loss, p.last_bias, p.impose_bc = 1, act_code(arch.act), 0, 1, int(arch.impose_bc)
    da = [o for o, _ in arch.stack_dims("branch")]
    db = [o for o, _ in arch.stack_dims("trunk")]
    p.n_layers_a, p.n_layers_b, p.in_a, p.in_b = len(da), len(db), arch.in_branch, arch.in_trunk
    for i, w in enumerate(da):
        p.dims_a[i] = w
    for i, w in enumerate(db):
        p.dims_b[i] = w
    p.D = p.d = arch.num_params
    p.N, p.P = N, P
    return p


# architectures past the kernel's limits, each one step beyond, with the reason make_plan gives
REFUSED = {
    "width129": (dict(width_branch=129), "widths up to 128"),
    "k129": (dict(output_neurons=129), "widths up to 128"),
    "sine": (dict(act="sine"), "relu or tanh"),
    "in_branch29057": (dict(in_branch=MAX_INPUT + 1), f"inputs up to {MAX_INPUT}"),
    "in_trunk29057": (dict(in_trunk=MAX_INPUT + 1, impose_bc=False), f"inputs up to {MAX_INPUT}"),
}


# ---------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------
def test_table_reaches_every_tile_and_edge():
    assert {tile_nb(c) for c in CASES} == set(range(1, 9))
    nb8 = [c for c in CASES if tile_nb(c) == 8]
    assert (3 * 128 * 128 + 128) * 4 == 197120 and 128 * 128 * 8 == 131072 and any(c.K == 128 for c in nb8)
    assert any(c.wb != c.wt and max(c.wb, c.wt) > max(min(c.wb, c.wt), c.K) for c in CASES)   # one stack padded
    assert any(c.K > max(c.wb, c.wt) for c in CASES) and any(c.K < min(c.wb, c.wt) for c in CASES) and min(c.K for c in CASES) == 1
    assert {c.in_trunk for c in CASES} == {None, 2, 12}
    assert {c.act for c in CASES} == {"tanh", "relu"}
    assert max(c.in_branch for c in CASES) * 8 > DEFAULT_SMEM and any(128 < c.in_branch <= 384 for c in CASES)
    assert min(min(c.db, c.dt) for c in CASES) == 2 and max(max(c.db, c.dt) for c in CASES) == _lib.MAX_LAYERS
    assert len({p for c in CASES if c.batches for _, p in c.batches}) > 1
    # a full-rank branch Gram at the shipped shape and at K = 128, rank-deficient rows, a zero pivot in the middle
    assert {"nb7_shipped_full_rank", "nb8_kmax"} <= {c.id for c in CASES if c.ranks[0][0] == c.K}
    assert any(r[0] < c.K and r[1] < c.K for c in CASES for r in c.ranks) and MIDDLE_ZERO_PIVOTS


@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_ranks_and_zero_pivots_are_as_labelled(case):
    """From the fp64 Gram matrices, per batch and stack: the labelled rank lies between the number of pivots clearly kept
    (> 1e3 PIVOT_TOL) and K minus the number clearly zero (< 1e-3 PIVOT_TOL) -- a pivot between the two may fall on either
    side of the rule with another summation order, in fp64 or in the kernel --; the clearly zero pivots are trailing ones,
    except on singular_middle, where they are exactly k = 11 (branch) and k = 5 (trunk), with every later pivot kept."""
    for ranks, pivs in zip(case.ranks, gram_pivots(case.id)):
        for which, rank, piv in zip((0, 1), ranks, pivs):
            kept, zero = np.nonzero(piv > 1e3 * PIVOT_TOL)[0], np.nonzero(piv < 1e-3 * PIVOT_TOL)[0]
            assert kept.size <= rank <= case.K - zero.size, (which, kept.size, rank, case.K - zero.size)
            if case.id in MIDDLE_ZERO_PIVOTS:
                assert list(zero) == MIDDLE_ZERO_PIVOTS[case.id][which] and kept.size == case.K - 1, (which, zero, kept.size)
            else:
                assert (zero >= rank).all(), (which, zero)


@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_restatement_equals_the_jacobian_oracle(case):
    s64, r = oracle(case.id, torch.float64), restated(case.id)
    pb = problem(case.id)
    for name, sel in pb["groups"] + [("all", np.arange(pb["D"]))]:
        err, ref = float(np.linalg.norm(r[sel] - s64[sel])), float(np.linalg.norm(s64[sel]))
        assert err <= 1e-10 * ref, (name, err, ref)


@pytest.mark.parametrize("row", ORACLE_CHECK_ROWS)
def test_vectorised_oracle_equals_the_autograd_loop(row):
    pb = problem(row)
    kw = arch_kwargs(arch_of(pb["case"]))
    ref = sum(osens.deeponet_scores(x1.unsqueeze(1), x2.unsqueeze(0), kw, pb["theta"], pb["sigma"]) for x1, x2 in pb["batches"])
    ref = ref / len(pb["batches"])
    np.testing.assert_allclose(oracle(row, torch.float64), ref, rtol=1e-12, atol=1e-14 * np.abs(ref).max())


def test_vectorised_oracle_equals_the_autograd_loop_on_the_golden_cases():
    from test_sensitivity import DON_SENS_CASES, _don_case

    for name, width, in_branch, db, dt, K, act in DON_SENS_CASES:
        batches, mu, sigma, _ = _don_case(name)
        kw = dict(width_branch=width, width_trunk=width, in_branch=in_branch, in_trunk=5, depth_branch=db, depth_trunk=dt,
                  output_neurons=K, act=act, impose_bc=True)
        ref = sum(osens.deeponet_scores(xb, xt, kw, mu, sigma) for xb, xt in batches) / len(batches)
        got = jacobian_scores(kw, batches, mu, sigma, torch.float64)
        np.testing.assert_allclose(got, ref, rtol=1e-12, atol=1e-14 * np.abs(ref).max(), err_msg=name)


@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_every_row_discriminates_and_rejects_the_mutants(case):
    """Each tensor's bound is at most DISCRIM of its fp64 norm (a tensor of norm 0 must come back exactly 0, checked on the
    GPU); each mutant that is more than DISCRIM away from the truth in some tensor is rejected by the checker.  The output
    bias b is exempt from the first rule: sigma_b^2 can sit below the floor of REL times the whole vector, and the GPU test
    requires it bit-exact instead."""
    pb = problem(case.id)
    s64, s32 = oracle(case.id, torch.float64), oracle(case.id, torch.float32)
    loose = [(name, b / n64) for name, _, n64, b in bounds(s64, s32, pb["groups"]) if name != "b" and n64 > 0 and b > DISCRIM * n64]
    assert not loose, loose
    assert not rejected(s32, s64, s32, pb["groups"])
    assert not rejected(restated(case.id), s64, s32, pb["groups"])
    for m in MUTANTS:
        if m == "raw (t, x) first-layer scores" and case.in_trunk is not None:
            continue
        s = restated(case.id, m)
        if differs(s, s64, pb["groups"]):
            assert rejected(s, s64, s32, pb["groups"]), m


def test_every_mutant_is_visible_somewhere():
    """Each mutant is more than DISCRIM away from the truth on at least one row (the relu rows and K = 1 hide some)."""
    seen = {m: [] for m in MUTANTS}
    for case in CASES:
        pb = problem(case.id)
        s64 = oracle(case.id, torch.float64)
        for m in MUTANTS:
            if m == "raw (t, x) first-layer scores" and case.in_trunk is not None:
                continue
            if differs(restated(case.id, m), s64, pb["groups"]):
                seen[m].append(case.id)
    assert all(seen.values()), seen
    assert len(seen["sigma shifted"]) == len(CASES)


def test_workspace_mirror_and_refusals():
    """vihmc_deeponet_sensitivity_workspace_bytes (no device needed) equals the mirror for every batch of every row, is 0
    one step past each limit (width or K 129, sine, an input above 29 056) and not 0 at the input limit itself."""
    lib = _lib.load()
    ask = lambda arch, n, p: int(lib.vihmc_deeponet_sensitivity_workspace_bytes(C.byref(abi_problem(arch, n, p))))
    for case in CASES:
        for n, p in batch_shapes(case):
            assert ask(arch_of(case), n, p) == workspace_bytes(arch_of(case), n, p) > 0, case.id
    base = CASE_BY_ID["nb1_full_rank"]
    for what, (kw, _) in REFUSED.items():
        assert workspace_bytes(arch_of(base, **kw), 4, 5) == 0 == ask(arch_of(base, **kw), 4, 5), what
    for kw in (dict(in_branch=MAX_INPUT), dict(in_trunk=MAX_INPUT, impose_bc=False), dict(in_branch=6145)):
        assert ask(arch_of(base, **kw), 4, 5) == workspace_bytes(arch_of(base, **kw), 4, 5) > 0, kw


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
class RefDeepONet:
    """Duck type of the reference's Operator_network/VI/model.py DeepONet: one `neurons` width, an activation module."""

    def __init__(self, arch):
        self.neurons, self.in_branch, self.in_trunk = arch.width_branch, arch.in_branch, arch.in_trunk
        self.depth_branch, self.depth_trunk, self.output_neurons = arch.depth_branch, arch.depth_trunk, arch.output_neurons
        self.act = {"tanh": torch.nn.Tanh, "relu": torch.nn.ReLU}[arch.act]()
        self.impose_bc = arch.impose_bc


def _data(pb, three_d=True):
    bs = [(x1.unsqueeze(1), x2.unsqueeze(0)) if three_d else (x1, x2) for x1, x2 in pb["batches"]]
    return bs[0] if len(bs) == 1 else bs


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_kernel_vs_fp64_jacobian(case):
    from vihmc import sensitivity as vs

    pb = problem(case.id)
    arch = arch_of(case)
    s64, s32 = oracle(case.id, torch.float64), oracle(case.id, torch.float32)
    s = vs.eval_std_dydw(_data(pb), arch, pb["theta"], pb["sigma"])
    worst, ratio = assert_grad(s, s64, s32, pb["groups"], case.id, floor=floor_of(s64))
    for name, sel, n64, _ in bounds(s64, s32, pb["groups"]):
        if n64 == 0.0:
            assert (s[sel] == 0).all(), name
    # d out / d b = 1: every batch gives float32(sigma_b)^2 exactly (the average over several batches is torch's arithmetic)
    sb = _bits(np.float32(pb["sigma"][0]) * np.float32(pb["sigma"][0]))[0]
    one = [s] if len(pb["batches"]) == 1 else [vs.eval_std_dydw(b, arch, pb["theta"], pb["sigma"]) for b in
                                                 (_data(dict(batches=[bt])) for bt in pb["batches"])]
    assert all(_bits(o[:1])[0] == sb for o in one), ([float(o[0]) for o in one], float(pb["sigma"][0]) ** 2)
    assert s[0] == pytest.approx(float(pb["sigma"][0]) ** 2, rel=1e-6)
    # deterministic, and the 2-D forms of the inputs are the same problem
    assert np.array_equal(_bits(s), _bits(vs.eval_std_dydw(_data(pb), arch, pb["theta"], pb["sigma"])))
    assert np.array_equal(_bits(s), _bits(vs.eval_std_dydw(_data(pb, three_d=False), arch, pb["theta"], pb["sigma"])))
    if case.wb == case.wt:
        assert np.array_equal(_bits(s), _bits(vs.eval_std_dydw(_data(pb), RefDeepONet(arch), pb["theta"], pb["sigma"])))
    # the selected split: the same as fp64's except at indices whose fp64 score is within the row's bound of the cut-off
    row_bound = max(b for _, _, _, b in bounds(s64, s32, pb["groups"] + [("all", np.arange(pb["D"]))]))
    sel, sel64 = vs.select_indices(s, 0.9), vs.select_indices(s64, 0.9)
    cut = np.sort(s64)[::-1][len(sel64) - 1]
    moved = np.setxor1d(sel, sel64)
    assert (np.abs(s64[moved] - cut) <= 2 * row_bound).all(), (moved, s64[moved], cut, row_bound)
    report(case=case.id, NB=tile_nb(case), ranks=case.ranks, seed_attempt=pb["attempt"], err_over_bound=worst,
           kernel_over_fp32=ratio, selected=len(sel), selection_moved=len(moved))


@pytest.mark.gpu
@pytest.mark.parametrize("what", list(REFUSED))
def test_unsupported_architectures_raise_with_their_reason(what):
    from vihmc import sensitivity as vs

    kw, reason = REFUSED[what]
    arch = arch_of(CASE_BY_ID["nb1_full_rank"], **kw)
    cols = 2 if arch.impose_bc else arch.in_trunk
    x1, x2 = torch.rand(2, 1, arch.in_branch), torch.rand(1, 3, cols)
    w = torch.full((arch.num_params,), 0.1)
    with pytest.raises(_lib.VihmcError) as e:
        vs.eval_std_dydw((x1, x2), arch, w, w)
    assert e.value.code == ERR_UNSUPPORTED and reason in str(e.value), str(e.value)


@pytest.mark.gpu
def test_a_workspace_one_byte_short_is_refused():
    from vihmc import engine
    from vihmc.spec import LogProbSpec

    pb = problem("nb1_full_rank")
    arch = arch_of(pb["case"])
    x1, x2 = pb["batches"][0]
    prep = engine.prepare(LogProbSpec(arch=arch, x=x1, x2=x2, y=torch.zeros(x1.shape[0], x2.shape[0]), prior_sigma_scalar=1.0))
    lib = _lib.load()
    need = int(lib.vihmc_deeponet_sensitivity_workspace_bytes(C.byref(prep.problem)))
    w, sg = pb["theta"].cuda(), pb["sigma"].cuda()
    out = torch.empty_like(w)
    ws = torch.empty(need, dtype=torch.uint8, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    rc = lib.vihmc_deeponet_sensitivity(C.byref(prep.problem), w.data_ptr(), sg.data_ptr(), out.data_ptr(), ws.data_ptr(), need - 1,
                                        stream)
    assert rc == ERR_WORKSPACE, lib.vihmc_last_error().decode()
    _lib.check(lib.vihmc_deeponet_sensitivity(C.byref(prep.problem), w.data_ptr(), sg.data_ptr(), out.data_ptr(), ws.data_ptr(),
                                              need, stream))
    torch.cuda.synchronize()
