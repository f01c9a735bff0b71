"""Time vihmc_gemm_batched on the three long-K products of the DeepONet gradient (64 chains): dW = dZ^T H, dxtr = G^T xb, dxb = G xtr."""
import json, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "vi-hmc_b200")]
import torch
from vihmc import engine

def timed(f, reps=5):
    f(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps): f()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps * 1e3

def main():
    C, N, P, K = 64, 1000, 10201, 100
    dev = "cuda"
    dZ = torch.randn(C, P, K, device=dev); H = torch.randn(C, P, K, device=dev)
    Pp = 10204
    G = torch.randn(C, N, Pp, device=dev)[:, :, :P]; xb = torch.randn(C, N, K, device=dev); xtr = torch.randn(C, P, K, device=dev)
    out = {"lib": os.environ.get("VIHMC_LIB_PATH", "default")}
    out["dW_us"] = timed(lambda: engine.gemm_batched(dZ.transpose(1, 2), H))
    out["dxtr_us"] = timed(lambda: engine.gemm_batched(G.transpose(1, 2), xb))
    out["dxb_us"] = timed(lambda: engine.gemm_batched(G, xtr))
    print(json.dumps(out))

if __name__ == "__main__":
    main()
