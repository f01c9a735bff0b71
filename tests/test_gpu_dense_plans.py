"""DeepONet dense path on each forward route, in chain batches, against the fp64 oracle; and the split-K scratch that the dense
path and vihmc_gemm_batched size for their products.

Routes: both stacks within the exact-accumulation forward (fwd3 + head3_kernel), only the branch within the fused 3xTF32
forward (a trunk width of 22 is not a multiple of 4), and neither (output_neurons = 10: per-layer GEMMs and the HEAD epilogue)."""
import ctypes as C
import zlib

import numpy as np
import pytest
import torch

from oracle import closures as oc
from vihmc import _lib, engine, synth
from vihmc.spec import DeepONetArch, LogProbSpec

pytestmark = pytest.mark.gpu

VIHMC_ERR_INVALID = 1
ROUTES = {
    "fwd3": dict(width_branch=20, width_trunk=24, output_neurons=12),
    "fused_branch": dict(width_branch=20, width_trunk=22, output_neurons=12),
    "per_layer": dict(width_branch=20, width_trunk=24, output_neurons=10),
}


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _problem(act, n_train, n_t, n_x, chains, **widths):
    arch = DeepONetArch(in_branch=7, depth_branch=3, depth_trunk=3, act=act, **widths)
    x1, x2, y, theta = synth.burgers_like(arch, n_train=n_train, n_t=n_t, n_x=n_x, seed=3)
    spec = LogProbSpec(arch=arch, x=x1, x2=x2, y=y, loss="NLL", tau_out=1.0, prior_sigma_scalar=0.1)
    closure = oc.DeepONetLogProb(x1=x1.unsqueeze(1), x2=x2.unsqueeze(0), y=y, in_branch=7, depth_branch=3, depth_trunk=3, act=act,
                                 dtype=torch.float64, **widths)
    rs = np.random.RandomState(zlib.crc32(repr((act, n_train, n_t, n_x, widths)).encode()))
    q = torch.from_numpy((theta.numpy()[None] + 0.02 * rs.randn(chains, arch.num_params)).astype(np.float32))
    return engine.prepare(spec), closure, q


def _run(prep, q, ws_chains):
    """vihmc_logp_grad and vihmc_predict for every chain of q with the workspace of ws_chains chains."""
    lib = _lib.load()
    prob = prep.problem
    ws_bytes = int(lib.vihmc_workspace_bytes(C.byref(prob), ws_chains))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
    qd = q.cuda().contiguous()
    Cn = q.shape[0]
    lp = torch.empty(Cn, dtype=torch.float32, device="cuda")
    g = torch.empty_like(qd)
    out = torch.empty(Cn, prep.spec.N, int(prob.P), dtype=torch.float32, device="cuda")
    _lib.check(lib.vihmc_logp_grad(C.byref(prob), Cn, qd.data_ptr(), lp.data_ptr(), g.data_ptr(), ws.data_ptr(), ws_bytes, _stream()))
    _lib.check(lib.vihmc_predict(C.byref(prob), Cn, qd.data_ptr(), out.data_ptr(), ws.data_ptr(), ws_bytes, _stream()))
    torch.cuda.synchronize()
    return lp.cpu().numpy(), g.cpu().numpy(), out.cpu().numpy()


def _check_against_oracle(prep, closure, q, ws_chains):
    lp, g, out = _run(prep, q, ws_chains)
    for c in range(q.shape[0]):
        lp64, g64 = oc.value_and_grad(closure, q[c].double())
        assert abs(lp[c] - float(lp64)) <= 1e-5 * abs(float(lp64)), (ws_chains, c, lp[c], float(lp64))
        np.testing.assert_allclose(g[c], g64.numpy(), rtol=2e-5, atol=2e-5 * np.abs(g64.numpy()).max())
        with torch.no_grad():
            ref = closure.forward(q[c].double()).numpy()
        np.testing.assert_allclose(out[c], ref, rtol=2e-5, atol=2e-6)


@pytest.mark.parametrize("act", ["tanh", "relu"])
@pytest.mark.parametrize("route", sorted(ROUTES))
def test_deeponet_routes_in_chain_batches_vs_fp64_oracle(route, act):
    """logp, gradient and predictions of 5 chains, with the workspace of all 5 and with that of 2 (batches 2 + 2 + 1)."""
    prep, closure, q = _problem(act, n_train=131, n_t=13, n_x=11, chains=5, **ROUTES[route])
    for ws_chains in (5, 2):
        _check_against_oracle(prep, closure, q, ws_chains)


@pytest.mark.parametrize("act", ["tanh", "relu"])
def test_deeponet_dbout_fill_split_vs_fp64_oracle(act):
    """P = 600 trunk points: the dBout = G Tout product (512-deep slices, so K = 600 is not a long reduction) is split into
    min(8, 600 / 128) = 4 slices to fill the GPU whenever a batch holds at most 74 chains.  The workspace must hold them."""
    prep, closure, q = _problem(act, n_train=100, n_t=24, n_x=25, chains=6, width_branch=24, width_trunk=24, output_neurons=12)
    assert int(prep.problem.P) == 600
    for ws_chains in (6, 2):
        _check_against_oracle(prep, closure, q, ws_chains)


def test_deeponet_predict_rejects_frozen_without_sens_ind():
    prep, _, q = _problem("tanh", n_train=131, n_t=13, n_x=11, chains=2, **ROUTES["fwd3"])
    lib = _lib.load()
    prob = _lib.Problem.from_buffer_copy(prep.problem)
    frozen = torch.zeros(prep.spec.D, dtype=torch.float32, device="cuda")
    prob.frozen, prob.sens_ind = frozen.data_ptr(), None
    ws_bytes = int(lib.vihmc_workspace_bytes(C.byref(prob), 2))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
    qd = q.cuda().contiguous()
    out = torch.empty(2, prep.spec.N, int(prob.P), dtype=torch.float32, device="cuda")
    rc = lib.vihmc_predict(C.byref(prob), 2, qd.data_ptr(), out.data_ptr(), ws.data_ptr(), ws_bytes, _stream())
    assert rc == VIHMC_ERR_INVALID, (rc, lib.vihmc_last_error())


@pytest.mark.parametrize("shape", [(1, 130, 37, 2500), (2, 100, 130, 3000)])
def test_gemm_batched_split_k_stays_within_its_documented_scratch(shape):
    """vihmc_gemm_batched with splitk_scratch of ceil(K/256) * batch * M * N floats followed by a canary tail in the same
    tensor: the canary is untouched and the product matches fp64.  N = 37 takes the TMEM-A plan, N = 130 the other one."""
    batch, M, N, K = shape
    rs = np.random.RandomState(zlib.crc32(repr(shape).encode()))
    A = torch.from_numpy(rs.randn(batch, M, K).astype(np.float32)).cuda()
    B = torch.from_numpy(rs.randn(batch, K, N).astype(np.float32)).cuda()
    need = (K + 255) // 256 * batch * M * N
    tail = 1 << 16
    scratch = torch.full((need + tail,), 1234.5, dtype=torch.float32, device="cuda")
    out = torch.empty(batch, M, N, dtype=torch.float32, device="cuda")
    lib = _lib.load()
    _lib.check(lib.vihmc_gemm_batched(A.data_ptr(), A.stride(0), A.stride(1), A.stride(2), B.data_ptr(), B.stride(0), B.stride(1),
                                      B.stride(2), out.data_ptr(), M * N, N, M, N, K, batch, 1, scratch.data_ptr(), _stream()))
    torch.cuda.synchronize()
    assert bool((scratch[need:] == 1234.5).all())
    assert not bool((scratch[:need] == 1234.5).all())   # the product did split
    ref = torch.matmul(A.double(), B.double())
    scale = (A.double().abs() @ B.double().abs()).max().item()
    assert (out.double() - ref).abs().max().item() <= 2e-6 * scale
