// Dense path: DeepONet (branch, trunk, dot-product head) and wide-MLP log-posterior + gradient for
// C chains at once, as batched GEMMs with fused epilogues.
//
// Restates, per chain, the reference closures
//   Operator_network/VI_HMC/main_VI_HMC_burgers.py:86-178 (prior :96-102, likelihood :157-163)
//   Operator_network/VI_HMC/my_make_func.py:44-83 (scatter :48-50, branch :53-61, feature layer :33-36,63-65,
//                                                  trunk :69-77, head einsum :79, + scalar bias :81-82)
//   Operator_network/HMC/main_HMC_splitting.py:134-204 (same arithmetic, `reshape` instead of `squeeze`)
// and the autograd backward hamiltorch takes through them.
//
// Round-1 kernels are FP32 SIMT (register-tiled 128x128x8 SGEMM, FP32 accumulate): the correctness
// baseline every later tensor-core kernel is checked against.  Reductions are fixed-order (per-CTA
// partials + a second pass), never float atomics, so accept/reject is reproducible.
//
// Data layout in HBM for one batch of Cb chains (all fp32, row-major):
//   Wf  [Cb, Dp]           full weights (VI scatter of q into the frozen means) in a PADDED layout: every tensor starts
//                          on a 16-byte boundary and weight rows are padded to a multiple of 4 floats, so every GEMM
//                          operand can be staged with float4 loads (flat index -> padded position: pad_map[D])
//   act_a[l] [Cb, N, w]    branch activations after layer l;  act_b[l] [Cb, P, w] trunk activations
//   G   [Cb, N, Pp]        d loglik / d output (the only [N,P]-sized per-chain buffer; rows padded to Pp = 4*ceil(P/4))
//   dz0/dz1 [Cb, R, w]     ping-pong pre-activation gradients, R = max(N, P)
//   dWf [Cb, Dp]           gradient w.r.t. the full weight vector (padded layout); gathered to grad[C, d] at the end
#include <stdlib.h>

#include "common.cuh"
#include "tc_gemm.cuh"
#include "fused_stack.cuh"
#include "xgemm.cuh"
#include "fwd3.cuh"

namespace vihmc {

// =============================================================================================
// batched SGEMM  C[b] = opA(A[b]) (MxK) * opB(B[b]) (KxN), generic element strides, fused epilogues
// =============================================================================================
constexpr int BM = 128, BN = 128, BK = 8, TM = 8, TN = 8, GEMM_THREADS = 256;

template <int EPI>
__global__ void __launch_bounds__(GEMM_THREADS) sgemm_batched_kernel(GemmArgs g) {
  __shared__ __align__(16) float As[2][BK][BM];
  __shared__ __align__(16) float Bs[2][BK][BN];
  const int b = blockIdx.z;
  const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
  const float* __restrict__ A = g.A + (long long)b * g.a_bs;
  const float* __restrict__ B = g.B + (long long)b * g.b_bs;
  const int tid = threadIdx.x;
  const int tx = tid % 16, ty = tid / 16;  // thread's 8x8 micro-tile: rows ty*8.., cols tx*8..

  // loader mapping: make the unit-stride dimension the fastest-varying one across threads
  const bool a_kfast = g.a_sk == 1;
  const bool b_nfast = g.b_sn == 1;
  int a_m[4], a_k[4], b_k[4], b_n[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int e = tid + i * GEMM_THREADS;  // 0..1023 = BM*BK
    if (a_kfast) { a_k[i] = e % BK; a_m[i] = e / BK; } else { a_m[i] = e % BM; a_k[i] = e / BM; }
    if (b_nfast) { b_n[i] = e % BN; b_k[i] = e / BN; } else { b_k[i] = e % BK; b_n[i] = e / BK; }
  }
  float ra[4], rb[4];
  auto fetch = [&](int k0) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int m = m0 + a_m[i], k = k0 + a_k[i];
      ra[i] = (m < g.M && k < g.K) ? __ldg(A + (long long)m * g.a_sm + (long long)k * g.a_sk) : 0.0f;
      const int kk = k0 + b_k[i], n = n0 + b_n[i];
      rb[i] = (kk < g.K && n < g.N) ? __ldg(B + (long long)kk * g.b_sk + (long long)n * g.b_sn) : 0.0f;
    }
  };
  auto stash = [&](int buf) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      As[buf][a_k[i]][a_m[i]] = ra[i];
      Bs[buf][b_k[i]][b_n[i]] = rb[i];
    }
  };

  float acc[TM][TN];
#pragma unroll
  for (int i = 0; i < TM; ++i)
#pragma unroll
    for (int j = 0; j < TN; ++j) acc[i][j] = 0.0f;

  const int nk = (g.K + BK - 1) / BK;
  fetch(0);
  stash(0);
  __syncthreads();
  for (int kt = 0; kt < nk; ++kt) {
    const int buf = kt & 1;
    if (kt + 1 < nk) fetch((kt + 1) * BK);
#pragma unroll
    for (int k = 0; k < BK; ++k) {
      float av[TM], bv[TN];
      const float4 a0 = *reinterpret_cast<const float4*>(&As[buf][k][ty * TM]);
      const float4 a1 = *reinterpret_cast<const float4*>(&As[buf][k][ty * TM + 4]);
      const float4 b0 = *reinterpret_cast<const float4*>(&Bs[buf][k][tx * TN]);
      const float4 b1 = *reinterpret_cast<const float4*>(&Bs[buf][k][tx * TN + 4]);
      av[0] = a0.x; av[1] = a0.y; av[2] = a0.z; av[3] = a0.w; av[4] = a1.x; av[5] = a1.y; av[6] = a1.z; av[7] = a1.w;
      bv[0] = b0.x; bv[1] = b0.y; bv[2] = b0.z; bv[3] = b0.w; bv[4] = b1.x; bv[5] = b1.y; bv[6] = b1.z; bv[7] = b1.w;
#pragma unroll
      for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
    if (kt + 1 < nk) {
      stash(buf ^ 1);
      __syncthreads();
    }
  }

  // ---------------- epilogue ----------------
  float* __restrict__ Cb = g.C + (long long)b * g.c_bs;
  float ll_acc = 0.0f, g_acc = 0.0f;
  const float bias0 = (EPI == EPI_HEAD) ? __ldg(g.bias + (long long)b * g.bias_bs) : 0.0f;
#pragma unroll
  for (int i = 0; i < TM; ++i) {
    const int m = m0 + ty * TM + i;
    if (m >= g.M) continue;
#pragma unroll
    for (int j = 0; j < TN; ++j) {
      const int n = n0 + tx * TN + j;
      if (n >= g.N) continue;
      float v = acc[i][j];
      if (EPI == EPI_BIAS_ACT) {
        v += __ldg(g.bias + (long long)b * g.bias_bs + n);
        if (g.act == VIHMC_ACT_TANH) v = tanhf(v);
        else if (g.act == VIHMC_ACT_RELU) v = v > 0.0f ? v : 0.0f;
      } else if (EPI == EPI_DACT) {
        const float a = __ldg(g.aux + (long long)b * g.aux_bs + (long long)m * g.ld_aux + n);
        v *= (g.act == VIHMC_ACT_TANH) ? (1.0f - a * a) : (a > 0.0f ? 1.0f : 0.0f);
      } else if (EPI == EPI_HEAD) {
        const float r = v + bias0 - __ldg(g.aux + (long long)b * g.aux_bs + (long long)m * g.ld_aux + n);
        ll_acc += g.ll_const - g.half_prec * r * r;
        v = -g.prec * r;
        g_acc += v;
      }
      Cb[(long long)m * g.ldc + n] = v;
    }
  }
  if (EPI == EPI_HEAD) {
    __shared__ float red[2][GEMM_THREADS / 32];
    ll_acc = warp_sum(ll_acc);
    g_acc = warp_sum(g_acc);
    if ((tid & 31) == 0) { red[0][tid >> 5] = ll_acc; red[1][tid >> 5] = g_acc; }
    __syncthreads();
    if (tid == 0) {
      float s0 = 0.0f, s1 = 0.0f;
      for (int w = 0; w < GEMM_THREADS / 32; ++w) { s0 += red[0][w]; s1 += red[1][w]; }
      const long long tiles = (long long)gridDim.x * gridDim.y;
      const long long t = (long long)blockIdx.y * gridDim.x + blockIdx.x;
      g.part_ll[(long long)b * tiles + t] = s0;
      g.part_g[(long long)b * tiles + t] = s1;
    }
  }
}

// Products with a reduction of at most 8 terms (the wide BNN's first layer, in_dim = 1: z = x W^T + b over 100 000 rows x 512 units,
// and the backward product through its output layer, K = out_dim = 1) are outer-product-like and memory-bound: one thread per
// (row, 4 consecutive columns), 16-byte loads / stores where the operands allow.  The tiled SIMT kernel spent 1.7 / 1.2 ms per
// evaluation on them writing 8 x 8 blocks with scalar stores (1.6 GB: 0.25 ms at HBM speed).  Same arithmetic in the same order
// (fmaf over k ascending, tanhf) as sgemm_batched_kernel: bit-identical results.
constexpr int SMALLK_MAX = 8;
template <int EPI>
__global__ void __launch_bounds__(256) smallk_gemm_kernel(GemmArgs g) {
  const int b = blockIdx.y;
  const int nq = (g.N + 3) / 4;
  const long long t = (long long)blockIdx.x * 256 + threadIdx.x;
  if (t >= (long long)g.M * nq) return;
  const int m = (int)(t / nq), n = (int)(t % nq) * 4;
  const float* __restrict__ A = g.A + (long long)b * g.a_bs + (long long)m * g.a_sm;
  const float* __restrict__ B = g.B + (long long)b * g.b_bs + (long long)n * g.b_sn;
  const int nv = g.N - n < 4 ? g.N - n : 4;
  float acc[4] = {0.0f, 0.0f, 0.0f, 0.0f};
  const bool bvec = g.b_sn == 1 && nv == 4 && (g.b_sk & 3) == 0 && (g.b_bs & 3) == 0 && ((reinterpret_cast<uintptr_t>(g.B) & 15u) == 0);
  for (int k = 0; k < g.K; ++k) {
    const float av = __ldg(A + (long long)k * g.a_sk);
    float bv[4] = {0.0f, 0.0f, 0.0f, 0.0f};
    const float* bk = B + (long long)k * g.b_sk;
    if (bvec) {
      const float4 v = __ldg(reinterpret_cast<const float4*>(bk));
      bv[0] = v.x; bv[1] = v.y; bv[2] = v.z; bv[3] = v.w;
    } else {
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (j < nv) bv[j] = __ldg(bk + (long long)j * g.b_sn);
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[j] = fmaf(av, bv[j], acc[j]);
  }
  float aux[4] = {0.0f, 0.0f, 0.0f, 0.0f};
  if (EPI == EPI_DACT) {
    const float* ar = g.aux + (long long)b * g.aux_bs + (long long)m * g.ld_aux + n;
    if (nv == 4 && (g.ld_aux & 3) == 0 && (g.aux_bs & 3) == 0 && ((reinterpret_cast<uintptr_t>(g.aux) & 15u) == 0)) {
      const float4 v = __ldg(reinterpret_cast<const float4*>(ar));
      aux[0] = v.x; aux[1] = v.y; aux[2] = v.z; aux[3] = v.w;
    } else {
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (j < nv) aux[j] = __ldg(ar + j);
    }
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    if (j >= nv) break;
    float v = acc[j];
    if (EPI == EPI_BIAS_ACT) {
      v += __ldg(g.bias + (long long)b * g.bias_bs + n + j);
      if (g.act == VIHMC_ACT_TANH) v = tanhf(v);
      else if (g.act == VIHMC_ACT_RELU) v = v > 0.0f ? v : 0.0f;
    } else if (EPI == EPI_DACT) {
      v *= (g.act == VIHMC_ACT_TANH) ? (1.0f - aux[j] * aux[j]) : (aux[j] > 0.0f ? 1.0f : 0.0f);
    }
    acc[j] = v;
  }
  float* cr = g.C + (long long)b * g.c_bs + (long long)m * g.ldc + n;
  if (nv == 4 && (g.ldc & 3) == 0 && (g.c_bs & 3) == 0 && ((reinterpret_cast<uintptr_t>(g.C) & 15u) == 0)) {
    *reinterpret_cast<float4*>(cr) = make_float4(acc[0], acc[1], acc[2], acc[3]);
  } else {
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (j < nv) cr[j] = acc[j];
  }
}

// VIHMC_DENSE_SIMT=1 keeps every GEMM on the FP32-SIMT kernel (A/B runs and the baseline the
// tensor-core kernel is checked against)
static bool tensor_cores_enabled() {
  static const bool on = []() {
    const char* e = getenv("VIHMC_DENSE_SIMT");
    return !(e != nullptr && e[0] == '1');
  }();
  return on;
}

template <int EPI>
static int launch_gemm(const GemmArgs& g, int batch, cudaStream_t st, float* scratch = nullptr, long long scratch_floats = 0,
                       int force = -1, float* rowsum_part = nullptr, float* rowsum_out = nullptr, long long rowsum_bs = 0,
                       int* rowsum_done = nullptr) {
  if (g.M < 1 || g.N < 1 || g.K < 1 || batch < 1) return fail(VIHMC_ERR_INVALID, "gemm: empty problem");
  if (batch > 65535) return fail(VIHMC_ERR_UNSUPPORTED, "gemm: batch > 65535");
  const bool tc = force < 0 ? tensor_cores_enabled() && tc_gemm_eligible(g) : force == 1;
  if (tc) return launch_tc_gemm<EPI>(g, batch, st, scratch, scratch_floats, rowsum_part, rowsum_out, rowsum_bs, rowsum_done);
  if (EPI == EPI_STORE && force < 0 && tensor_cores_enabled() && g.M == 1) {
    // A single output row over a long reduction (the output layer's weight gradient dW[1, in] = dz^T[1, R] a[R, in] of the
    // wide-BNN config: 22 ms per evaluation on the SIMT kernel, a third of the whole gradient): run the transposed problem
    // C^T[in, 1] = a^T dz on the tensor-core kernel instead.  C^T's rows are one element long, so it is the same memory as C.
    GemmArgs t = g;
    t.A = g.B; t.a_bs = g.b_bs; t.a_sm = g.b_sn; t.a_sk = g.b_sk;
    t.B = g.A; t.b_bs = g.a_bs; t.b_sk = g.a_sk; t.b_sn = g.a_sm;
    t.M = g.N; t.N = 1; t.ldc = 1;
    if (tc_gemm_eligible(t)) return launch_tc_gemm<EPI>(t, batch, st, scratch, scratch_floats);   // no fused row sums: opA is not dz any more
  }
  if (EPI != EPI_HEAD && force < 0 && g.K <= SMALLK_MAX && g.N >= 16) {
    const long long threads = (long long)g.M * ((g.N + 3) / 4);
    if ((threads + 255) / 256 < 0x7fffffffLL) {
      dim3 sgrid((unsigned)((threads + 255) / 256), batch);
      smallk_gemm_kernel<EPI><<<sgrid, 256, 0, st>>>(g);
      VIHMC_LAUNCH_OK("smallk_gemm_kernel");
      return VIHMC_OK;
    }
  }
  dim3 grid((g.N + BN - 1) / BN, (g.M + BM - 1) / BM, batch);
  sgemm_batched_kernel<EPI><<<grid, GEMM_THREADS, 0, st>>>(g);
  VIHMC_LAUNCH_OK("sgemm_batched_kernel");
  return VIHMC_OK;
}

// =============================================================================================
// small helper kernels
// =============================================================================================
// trunk features [t, sin 2pi x, sin 4pi x, cos 2pi x, cos 4pi x]  (my_make_func.py:33-36,63-65)
__global__ void trunk_features_kernel(const float* __restrict__ x2, long long P, float* __restrict__ F) {
  const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  const float t = x2[2 * p], x = x2[2 * p + 1];
  const float two_pi = 6.283185307179586f;   // float32(2*np.pi) as torch computes 2*np.pi*x in fp32
  const float four_pi = 12.566370614359172f;
  F[5 * p + 0] = t;
  F[5 * p + 1] = sinf(two_pi * x);
  F[5 * p + 2] = sinf(four_pi * x);
  F[5 * p + 3] = cosf(two_pi * x);
  F[5 * p + 4] = cosf(four_pi * x);
}

// out[b, n] = sum_r Z[b, r, n]   (bias gradients), two fixed-order passes so that the [R, n] slab of every chain is
// streamed by R/128 CTAs instead of one: pass 1, grid (slabs, batch), block (32, 8): part[b, slab, n] = sum of the
// slab's 128 rows; pass 2 (colsum_finish_kernel): out[b, n] = sum_slab part[b, slab, n].
constexpr int kColsumRows = 128;
__global__ void __launch_bounds__(256) colsum_kernel(const float* __restrict__ Z, long long z_bs, long long R, int ncols, long long ldz,
                                                     float* __restrict__ part) {
  __shared__ float red[8][33];
  const int b = blockIdx.y, slab = blockIdx.x;
  const long long r_lo = (long long)slab * kColsumRows, r_hi = r_lo + kColsumRows < R ? r_lo + kColsumRows : R;
  const float* Zb = Z + (long long)b * z_bs;
  for (int col0 = 0; col0 < ncols; col0 += 32) {
    const int col = col0 + threadIdx.x;
    float s = 0.0f;
    if (col < ncols)
      for (long long r = r_lo + threadIdx.y; r < r_hi; r += 8) s += Zb[r * ldz + col];
    red[threadIdx.y][threadIdx.x] = s;
    __syncthreads();
    if (threadIdx.y == 0 && col < ncols) {
      float t = 0.0f;
      for (int i = 0; i < 8; ++i) t += red[i][threadIdx.x];
      part[((long long)b * gridDim.x + slab) * ncols + col] = t;
    }
    __syncthreads();
  }
}
__global__ void colsum_finish_kernel(const float* __restrict__ part, int slabs, int ncols, float* __restrict__ out, long long out_bs) {
  const int b = blockIdx.x;
  for (int col = threadIdx.x; col < ncols; col += blockDim.x) {
    float s = 0.0f;
    for (int i = 0; i < slabs; ++i) s += part[((long long)b * slabs + i) * ncols + col];
    out[(long long)b * out_bs + col] = s;
  }
}
// `part` needs batch * ceil(R/128) * ncols floats
static int launch_colsum(const float* Z, long long z_bs, long long R, int ncols, long long ldz, float* part, float* out,
                         long long out_bs, int batch, cudaStream_t st) {
  const int slabs = (int)((R + kColsumRows - 1) / kColsumRows);
  colsum_kernel<<<dim3(slabs, batch), dim3(32, 8), 0, st>>>(Z, z_bs, R, ncols, ldz, part);
  VIHMC_LAUNCH_OK("colsum_kernel");
  colsum_finish_kernel<<<batch, 128, 0, st>>>(part, slabs, ncols, out, out_bs);
  VIHMC_LAUNCH_OK("colsum_finish_kernel");
  return VIHMC_OK;
}

// fixed-order sum of per-tile partials: out[b] = sum_t part[b, t]  (one warp per batch row)
__global__ void reduce_partials_kernel(const float* __restrict__ part, long long tiles, long long batch, float* __restrict__ out,
                                       long long out_stride) {
  const long long b = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (b >= batch) return;
  float s = 0.0f;
  for (long long t = threadIdx.x & 31; t < tiles; t += 32) s += part[b * tiles + t];
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) out[b * out_stride] = s;
}

// MLP likelihood on the output column: G[b,n] = -prec (o - y); per-CTA partial loglik.  grid (ceil(N/256), batch)
__global__ void mlp_loss_kernel(const float* __restrict__ O, const float* __restrict__ y, long long N, float ll_const,
                                float half_prec, float prec, float* __restrict__ G, float* __restrict__ part_ll) {
  const int b = blockIdx.y;
  const long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  float ll = 0.0f;
  if (n < N) {
    const float r = O[(long long)b * N + n] - __ldg(y + n);
    ll = ll_const - half_prec * r * r;
    G[(long long)b * N + n] = -prec * r;
  }
  __shared__ float red[8];
  ll = warp_sum(ll);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = ll;
  __syncthreads();
  if (threadIdx.x == 0) {
    float s = 0.0f;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += red[w];
    part_ll[(long long)b * gridDim.x + blockIdx.x] = s;
  }
}

// grad[c,i] = dWf[c, ind[i]] - (q - mu) / sigma^2 / prior_scale, plus this slab's share of the prior
// sum_i -0.5 (q-mu)^2 / sigma^2.  grid (slabs, chains): every CTA streams kFinSlab coordinates of one chain and
// writes one partial; logp_kernel then adds the partials in fixed order (no float atomics).
constexpr int kFinSlab = 8192;
__global__ void __launch_bounds__(256) finalize_kernel(const float* __restrict__ dWf, const long long* __restrict__ ind,
                                                        const float* __restrict__ q, const float* __restrict__ prior_mu,
                                                        const float* __restrict__ prior_sigma, float sigma_scalar,
                                                        float inv_scale, long long Dp, long long d, const int* __restrict__ pad_map,
                                                        float* __restrict__ prior_part, float* __restrict__ grad) {
  const long long c = blockIdx.y;
  const long long lo = (long long)blockIdx.x * kFinSlab, hi = lo + kFinSlab < d ? lo + kFinSlab : d;
  float lp = 0.0f;
  for (long long i = lo + threadIdx.x; i < hi; i += blockDim.x) {
    const float sg = prior_sigma ? __ldg(prior_sigma + i) : sigma_scalar;
    const float iv = isinf(sg) ? 0.0f : 1.0f / (sg * sg);
    const float dq = q[c * d + i] - (prior_mu ? __ldg(prior_mu + i) : 0.0f);
    lp = fmaf(-0.5f * dq * dq, iv, lp);
    if (grad != nullptr) {
      const long long f = ind ? __ldg(ind + i) : i;
      grad[c * d + i] = fmaf(-dq * iv, inv_scale, dWf[c * Dp + __ldg(pad_map + f)]);
    }
  }
  __shared__ float red[8];
  lp = warp_sum(lp);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = lp;
  __syncthreads();
  if (threadIdx.x == 0) {
    float s = 0.0f;
    for (int w = 0; w < 8; ++w) s += red[w];
    prior_part[c * gridDim.x + blockIdx.x] = s;
  }
}

// logp[c] = loglik[c] + (sum_slabs prior_part[c, :] + log_norm) / prior_scale
__global__ void logp_kernel(const float* __restrict__ prior_part, int slabs, const float* __restrict__ loglik, float inv_scale,
                            float log_norm, long long C, float* __restrict__ logp) {
  const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  float s = 0.0f;
  for (int i = 0; i < slabs; ++i) s += prior_part[c * slabs + i];
  logp[c] = loglik[c] + (s + log_norm) * inv_scale;
}

// ---- padded weight layout ----
// one tensor of the flat parameter vector: flat [flat0, flat0+numel) viewed as rows of `in` floats -> pad0 + row*ld + col
struct PadSeg { long long flat0, numel, pad0; int in, ld; };
struct PadTable { int n; PadSeg seg[4 * VIHMC_MAX_LAYERS + 1]; };

__global__ void pad_map_kernel(PadTable t, long long D, int* __restrict__ pad_map) {
  const long long f = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= D) return;
  for (int s = 0; s < t.n; ++s) {
    const PadSeg& g = t.seg[s];
    if (f < g.flat0 + g.numel) {
      const long long r = f - g.flat0;
      pad_map[f] = (int)(g.pad0 + (r / g.in) * g.ld + (r % g.in));
      return;
    }
  }
}

// Wf[c, pad_map[f]] = src[f]  (src = frozen means shared by every chain, or -- full HMC -- the chain's own q row)
__global__ void __launch_bounds__(256) scatter_fill_padded_kernel(const float* __restrict__ src, long long src_cs,
                                                                  const int* __restrict__ pad_map, float* __restrict__ Wf,
                                                                  long long D, long long Dp) {
  const long long c = blockIdx.y;
  for (long long f = (long long)blockIdx.x * blockDim.x + threadIdx.x; f < D; f += (long long)gridDim.x * blockDim.x)
    Wf[c * Dp + __ldg(pad_map + f)] = src[c * src_cs + f];
}
// Wf[c, pad_map[ind[i]]] = q[c, i]   (my_make_func.py:56-57; ind sorted ascending => near-coalesced)
__global__ void __launch_bounds__(256) scatter_put_padded_kernel(const long long* __restrict__ ind, const float* __restrict__ q,
                                                                 const int* __restrict__ pad_map, float* __restrict__ Wf,
                                                                 long long d, long long Dp) {
  const long long c = blockIdx.y;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < d; i += (long long)gridDim.x * blockDim.x)
    Wf[c * Dp + __ldg(pad_map + __ldg(ind + i))] = q[c * d + i];
}

// =============================================================================================
// host orchestration
// =============================================================================================
struct Stack {
  int n_layers, in_dim;
  int dims[VIHMC_MAX_LAYERS];
  long long w_off[VIHMC_MAX_LAYERS], b_off[VIHMC_MAX_LAYERS];   // offsets in the PADDED layout
  int ldw[VIHMC_MAX_LAYERS];                                     // padded weight row stride
  bool has_bias[VIHMC_MAX_LAYERS];
  int in_of(int l) const { return l == 0 ? in_dim : dims[l - 1]; }
  int max_width() const {
    int w = 0;
    for (int l = 0; l < n_layers; ++l) w = dims[l] > w ? dims[l] : w;
    return w;
  }
};

static inline long long pad4(long long v) { return (v + 3) / 4 * 4; }

// lays one stack out after flat offset `off` / padded offset `poff`; appends its tensors to the pad table
static void build_stack(Stack& s, int n_layers, int in_dim, const int32_t* dims, long long& off, long long& poff, bool last_bias,
                        PadTable& tbl) {
  s.n_layers = n_layers;
  s.in_dim = in_dim;
  for (int l = 0; l < n_layers; ++l) {
    s.dims[l] = dims[l];
    const int in = s.in_of(l);
    s.ldw[l] = (int)pad4(in);
    s.w_off[l] = poff;
    tbl.seg[tbl.n++] = PadSeg{off, (long long)dims[l] * in, poff, in, s.ldw[l]};
    off += (long long)dims[l] * in;
    poff += (long long)dims[l] * s.ldw[l];
    s.has_bias[l] = (l < n_layers - 1) || last_bias;
    s.b_off[l] = poff;
    if (s.has_bias[l]) {
      tbl.seg[tbl.n++] = PadSeg{off, dims[l], poff, dims[l], dims[l]};
      off += dims[l];
      poff += pad4(dims[l]);
    }
  }
}

struct DensePlan {
  bool deeponet;
  Stack a, b;       // MLP: a only
  long long D, Dp, N, P, Pp, R;   // Dp, Pp: padded parameter count / padded trunk-point row length
  PadTable tbl;
  int K;            // DeepONet: output_neurons
  long long head_tiles, loss_tiles;
  // per-chain float counts
  long long act_a_floats, act_b_floats, per_chain_floats, scratch_per_chain;
  bool fuse_a, fuse_b;       // the branch / trunk stack runs through the fused kernels
  long long img_floats;      // pre-split weight images of the fused kernels (0 when no stack is eligible)
  long long dzall_floats;    // fused trunk backward: dz of every layer below the top one + bias-gradient partials
  long long shared_floats;  // trunk features
  // exact-accumulation forward (fwd3.cuh): weight blobs, operand images of Bout / Tout and their row scales
  bool fwd3;
  int m_tiles, p_tiles128;
  long long wimg3_floats, ximg_a_floats, ximg_b_floats, xsc_floats;
};

// VIHMC_DENSE_NOFUSE=1 keeps every stack on the per-layer GEMMs (A/B baseline of the fused kernel)
static bool fused_enabled() {
  static const bool on = []() {
    const char* e = getenv("VIHMC_DENSE_NOFUSE");
    return !(e != nullptr && e[0] == '1');
  }();
  return on && tensor_cores_enabled();
}

// shapes the fused kernels take: every width a multiple of 4 and <= 104, input at most 104 wide, bias everywhere
static bool fused_eligible(const Stack& s) {
  if (!fused_enabled() || s.n_layers < 2 || s.in_dim > fused::KPAD) return false;
  for (int l = 0; l < s.n_layers; ++l)
    if (s.dims[l] % 4 != 0 || s.dims[l] > fused::KPAD || !s.has_bias[l]) return false;
  return true;
}

// forward of one stack in ONE kernel (fused_stack.cuh); img: Cb * (n_layers-1) * 2 * B_TILE bytes of scratch
static int stack_forward_fused(const Stack& s, const float* input, long long R, const float* Wf, long long Dp, float* const* acts,
                               int act, int Cb, float* img, cudaStream_t st) {
  fused::ImgTable t{};
  const int l0 = s.in_dim > fused::MAX_IN0 ? 0 : 1;   // a wide input makes the first layer a tensor-core layer too
  t.n = s.n_layers - l0;
  for (int l = l0; l < s.n_layers; ++l) t.L[l - l0] = fused::ImgLayer{s.w_off[l], s.dims[l], s.in_of(l), s.ldw[l], 1};
  fused::weight_image_kernel<<<dim3(t.n, Cb), 256, 0, st>>>(Wf, Dp, t, img);
  VIHMC_LAUNCH_OK("weight_image_kernel");
  fused::FusedFwdArgs a{};
  a.input = input; a.in_dim = s.in_dim; a.Wf = Wf; a.Dp = Dp; a.w0_off = s.w_off[0]; a.ldw0 = s.ldw[0];
  for (int l = 0; l < s.n_layers; ++l) { a.b_off[l] = s.b_off[l]; a.dims[l] = s.dims[l]; a.acts[l] = acts[l]; }
  a.n_layers = s.n_layers; a.img = img; a.R = R; a.act = act;
  const dim3 grid((unsigned)((R + tc::BM - 1) / tc::BM), Cb);
  auto launch = [&](auto kernel) -> int {
    VIHMC_CUDA_OK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, fused::F_SMEM));
    kernel<<<grid, fused::F_THREADS, fused::F_SMEM, st>>>(a);
    return VIHMC_OK;
  };
  if (act == VIHMC_ACT_TANH) { if (int rc = launch(fused::fused_forward_kernel<VIHMC_ACT_TANH>)) return rc; }
  else { if (int rc = launch(fused::fused_forward_kernel<VIHMC_ACT_RELU>)) return rc; }
  VIHMC_LAUNCH_OK("fused_forward_kernel");
  return VIHMC_OK;
}

// weight gradient of layer l, dW[o,i] = sum_r dz[r,o] * a_in[r,i], and its bias gradient = column sums of dz = row sums of
// opA: the tensor-core GEMM reads them off its operand stream when it can (MN-major A), launch_colsum sums them otherwise;
// `part` holds the bias partials either way
static int layer_weight_grad(const Stack& s, int l, const float* input, long long R, float* const* acts, const float* dz, float* dWf,
                             long long Dp, float* part, int Cb, float* scratch, long long scratch_floats, cudaStream_t st) {
  const int in = s.in_of(l), out = s.dims[l];
  GemmArgs g{};
  g.A = dz; g.a_bs = R * out; g.a_sm = 1; g.a_sk = out;            // opA[m=o,k=r] = dz[r,o]
  g.B = l == 0 ? input : acts[l - 1]; g.b_bs = l == 0 ? 0 : R * in; g.b_sk = in; g.b_sn = 1;
  g.C = dWf + s.w_off[l]; g.c_bs = Dp; g.ldc = s.ldw[l];
  g.M = out; g.N = in; g.K = (int)R;
  float* bias = s.has_bias[l] ? dWf + s.b_off[l] : nullptr;
  int bias_done = 0;
  if (int rc = launch_gemm<EPI_STORE>(g, Cb, st, scratch, scratch_floats, -1, bias ? part : nullptr, bias, Dp, &bias_done)) return rc;
  if (bias != nullptr && !bias_done)
    if (int rc = launch_colsum(dz, R * out, R, out, out, part, bias, Dp, Cb, st)) return rc;
  return VIHMC_OK;
}

// backward of one stack with the data pass in ONE kernel (fused_stack.cuh): dzs[top] holds d/d(pre-activation of the last
// layer) on entry, dzs[l < top] are written by the kernel; the weight / bias gradients follow as one GEMM per layer.
static int stack_backward_fused(const Stack& s, const float* input, long long R, const float* Wf, float* dWf, long long Dp,
                                float* const* acts, float* const* dzs, int act, int Cb, float* img, float* bias_part, float* scratch,
                                long long scratch_floats, cudaStream_t st) {
  fused::ImgTable t{};
  t.n = s.n_layers - 1;
  for (int l = 1; l < s.n_layers; ++l) t.L[l - 1] = fused::ImgLayer{s.w_off[l], s.in_of(l), s.dims[l], 1, s.ldw[l]};   // W_l^T
  fused::weight_image_kernel<<<dim3(t.n, Cb), 256, 0, st>>>(Wf, Dp, t, img);
  VIHMC_LAUNCH_OK("weight_image_kernel");
  fused::FusedBwdArgs a{};
  for (int l = 0; l < s.n_layers; ++l) { a.dims[l] = s.dims[l]; a.acts[l] = acts[l]; a.dz[l] = dzs[l]; }
  a.n_layers = s.n_layers; a.img = img; a.R = R;
  const dim3 grid((unsigned)((R + tc::BM - 1) / tc::BM), Cb);
  auto launch = [&](auto kernel) -> int {
    VIHMC_CUDA_OK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, fused::F_SMEM));
    kernel<<<grid, fused::F_THREADS, fused::F_SMEM, st>>>(a);
    return VIHMC_OK;
  };
  if (act == VIHMC_ACT_TANH) { if (int rc = launch(fused::fused_backward_kernel<VIHMC_ACT_TANH>)) return rc; }
  else { if (int rc = launch(fused::fused_backward_kernel<VIHMC_ACT_RELU>)) return rc; }
  VIHMC_LAUNCH_OK("fused_backward_kernel");
  for (int l = s.n_layers - 1; l >= 0; --l)
    if (int rc = layer_weight_grad(s, l, input, R, acts, dzs[l], dWf, Dp, bias_part, Cb, scratch, scratch_floats, st)) return rc;
  return VIHMC_OK;
}

static bool fwd3_eligible(const Stack& s) {
  if (s.n_layers < 2 || s.in_dim > xg::XK) return false;
  for (int l = 0; l < s.n_layers; ++l)
    if (s.dims[l] % 4 != 0 || s.dims[l] > fused::KPAD || !s.has_bias[l]) return false;
  return true;
}

// forward of one stack through fused_forward3_kernel; out_img / out_scales (optional): operand image of the last layer's output
static int stack_forward3(const Stack& s, const float* input, long long R, const float* Wf, long long Dp, float* const* acts, int act,
                          int Cb, unsigned char* wimg, unsigned char* out_img, float* out_scales, cudaStream_t st) {
  xg::Img3Table t{};
  const int l0 = s.in_dim > xg::MAX_IN0 ? 0 : 1;
  t.n = s.n_layers - l0;
  for (int l = l0; l < s.n_layers; ++l) t.L[l - l0] = xg::Img3Layer{s.w_off[l], s.b_off[l], s.dims[l], s.in_of(l), s.ldw[l], 1};
  xg::weight_image3_kernel<<<dim3(t.n, Cb), 256, 0, st>>>(Wf, Dp, t, wimg);
  VIHMC_LAUNCH_OK("weight_image3_kernel");
  xg::Fwd3Args a{};
  a.input = input; a.in_dim = s.in_dim; a.Wf = Wf; a.Dp = Dp; a.w0_off = s.w_off[0]; a.b0_off = s.b_off[0]; a.ldw0 = s.ldw[0];
  for (int l = 0; l < s.n_layers; ++l) { a.dims[l] = s.dims[l]; a.acts[l] = acts[l]; }
  a.n_layers = s.n_layers; a.wimg = wimg; a.R = R; a.out_img = out_img; a.out_scales = out_scales;
  const dim3 grid((unsigned)((R + 127) / 128), Cb);
  auto launch = [&](auto kernel) -> int {
    VIHMC_CUDA_OK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, xg::F3_SMEM));
    kernel<<<grid, xg::F3_THREADS, xg::F3_SMEM, st>>>(a);
    return VIHMC_OK;
  };
  if (act == VIHMC_ACT_TANH) { if (int rc = launch(xg::fused_forward3_kernel<VIHMC_ACT_TANH>)) return rc; }
  else { if (int rc = launch(xg::fused_forward3_kernel<VIHMC_ACT_RELU>)) return rc; }
  VIHMC_LAUNCH_OK("fused_forward3_kernel");
  return VIHMC_OK;
}

// head product + Gaussian residual (likelihood mode) or plain outputs (predict mode) through head3_kernel
static int launch_head3(const DensePlan& pl, int Cb, const unsigned char* a_img, const float* a_sc, const unsigned char* b_img,
                        const float* b_sc, const float* bias, long long bias_bs, const float* Y, long long ldy, float* G, long long g_bs,
                        long long ldg, const Likelihood& lik, float* part_ll, float* part_g, int* parts_out, cudaStream_t st) {
  xg::Head3Args a{};
  a.a_img = a_img; a.a_sc = a_sc; a.b_img = b_img; a.b_sc = b_sc;
  a.M = (int)pl.N; a.P = (int)pl.P; a.K = pl.K;
  a.bias = bias; a.bias_bs = bias_bs; a.Y = Y; a.ldy = ldy; a.G = G; a.g_bs = g_bs; a.ldg = ldg;
  a.ll_const = lik.ll_const; a.half_prec = lik.half_prec; a.prec = lik.prec;
  a.part_ll = part_ll; a.part_g = part_g;
  a.Cb = Cb; a.m_tiles = pl.m_tiles; a.p_tiles128 = pl.p_tiles128;
  a.p_tiles = (int)((pl.P + xg::H3_BN - 1) / xg::H3_BN);
  // trunk-point chunks: enough work items to balance the persistent CTAs, at least four tiles per item, and no more
  // partial-sum slots per chain than the workspace holds (head_tiles)
  const int sms = tc_num_sms();
  long long want = (6LL * sms + (long long)Cb * a.m_tiles - 1) / ((long long)Cb * a.m_tiles);
  long long cap = a.p_tiles / 4 > 1 ? a.p_tiles / 4 : 1;
  if (cap > pl.head_tiles / a.m_tiles) cap = pl.head_tiles / a.m_tiles;
  if (want > cap) want = cap;
  if (want < 1) want = 1;
  a.tiles_per_chunk = (int)((a.p_tiles + want - 1) / want);
  a.p_chunks = (a.p_tiles + a.tiles_per_chunk - 1) / a.tiles_per_chunk;
  a.parts = a.m_tiles * a.p_chunks;
  static const int ahead = []() { const char* e = getenv("VIHMC_HEAD_PREFETCH"); return e != nullptr ? atoi(e) : 0; }();
  a.prefetch_ahead = ahead;
  a.n_items = (long long)Cb * a.parts;
  if (parts_out != nullptr) *parts_out = a.parts;
  const unsigned grid = (unsigned)(a.n_items < sms ? a.n_items : sms);
  if (Y == nullptr) {
    VIHMC_CUDA_OK(cudaFuncSetAttribute(xg::head3_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, xg::H3_SMEM));
    xg::head3_kernel<true><<<grid, xg::H3_THREADS, xg::H3_SMEM, st>>>(a);
  } else {
    VIHMC_CUDA_OK(cudaFuncSetAttribute(xg::head3_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, xg::H3_SMEM));
    xg::head3_kernel<false><<<grid, xg::H3_THREADS, xg::H3_SMEM, st>>>(a);
  }
  VIHMC_LAUNCH_OK("head3_kernel");
  return VIHMC_OK;
}

// dBout = G Tout writes 400 KB per slice and chain: 512-deep slices halve that traffic (their share of the BASELINE-size
// gradient error stays below 2e-6, tests/diag_fullsize.py)
constexpr int kDBoutChunk = 512;

static int make_plan(const vihmc_problem* p, DensePlan& pl) {
  pl.deeponet = p->model_kind == VIHMC_MODEL_DEEPONET;
  pl.N = p->N;
  pl.P = pl.deeponet ? p->P : 1;
  if (p->n_layers_a < 1 || p->n_layers_a > VIHMC_MAX_LAYERS || p->n_layers_b < 0 || p->n_layers_b > VIHMC_MAX_LAYERS)
    return fail(VIHMC_ERR_INVALID, "layer counts out of range");
  pl.Pp = pad4(pl.P);
  pl.tbl.n = 0;
  long long off = 0, poff = 0;
  if (pl.deeponet) {
    pl.tbl.seg[pl.tbl.n++] = PadSeg{0, 1, 0, 1, 1};   // scalar output bias b0 = W[0] (my_make_func.py:52)
    off = 1;
    poff = 4;
    build_stack(pl.a, p->n_layers_a, p->in_a, p->dims_a, off, poff, true, pl.tbl);
    build_stack(pl.b, p->n_layers_b, p->in_b, p->dims_b, off, poff, true, pl.tbl);
    pl.K = p->dims_a[p->n_layers_a - 1];
    if (p->dims_b[p->n_layers_b - 1] != pl.K) return fail(VIHMC_ERR_INVALID, "branch and trunk output widths differ");
    if (p->impose_bc && p->in_b != 5) return fail(VIHMC_ERR_INVALID, "impose_bc needs in_trunk = 5");
  } else {
    build_stack(pl.a, p->n_layers_a, p->in_a, p->dims_a, off, poff, p->last_bias != 0, pl.tbl);
    pl.b.n_layers = 0;
    pl.K = 1;
    if (p->dims_a[p->n_layers_a - 1] != 1) return fail(VIHMC_ERR_UNSUPPORTED, "dense MLP path needs out_dim = 1");
  }
  if (off != p->D) return fail(VIHMC_ERR_INVALID, "D=%lld does not match the architecture (%lld)", (long long)p->D, off);
  if (poff > 0x7fffffffLL) return fail(VIHMC_ERR_UNSUPPORTED, "more than 2^31 parameters per chain");
  pl.D = p->D;
  pl.Dp = poff;
  pl.R = pl.N > pl.P ? pl.N : pl.P;
  pl.act_a_floats = 0;
  for (int l = 0; l < pl.a.n_layers; ++l) pl.act_a_floats += pl.N * pl.a.dims[l];
  pl.act_b_floats = 0;
  for (int l = 0; l < pl.b.n_layers; ++l) pl.act_b_floats += pl.P * pl.b.dims[l];
  const int wmax = pl.a.max_width() > pl.b.max_width() ? pl.a.max_width() : pl.b.max_width();
  pl.head_tiles = ((pl.P + BN - 1) / BN) * ((pl.N + BM - 1) / BM);
  pl.loss_tiles = (pl.N + 255) / 256;
  const long long tiles = pl.deeponet ? pl.head_tiles : pl.loss_tiles;
  const long long G = pl.deeponet ? pl.N * pl.Pp : pl.N;
  pl.scratch_per_chain = 0;   // split-K partials of the largest product that can be split, at the most slices it can take
  auto budget = [&](int M, int N, long long K, int kc_hint) {
    const long long slices = splitk_max_slices((int)K, kc_hint);
    if (slices > 1 && slices * M * N > pl.scratch_per_chain) pl.scratch_per_chain = slices * M * N;
  };
  for (int l = 0; l < pl.a.n_layers; ++l) budget(pl.a.dims[l], pl.a.in_of(l), pl.N, 0);   // weight gradients
  for (int l = 0; l < pl.b.n_layers; ++l) budget(pl.b.dims[l], pl.b.in_of(l), pl.P, 0);
  if (pl.deeponet) {   // dBout = G Tout reduces over the P trunk points, dTout = G^T Bout over the N functions
    budget((int)pl.N, pl.K, pl.P, kDBoutChunk);
    budget((int)pl.P, pl.K, pl.N, 0);
  }
  // fused kernels (DeepONet stacks): weight images (the two stacks use the buffer one after the other), dz of every layer
  pl.fuse_a = pl.deeponet && fused_eligible(pl.a);
  pl.fuse_b = pl.deeponet && fused_eligible(pl.b);
  const int n_img = (pl.fuse_a ? pl.a.n_layers : 0) > (pl.fuse_b ? pl.b.n_layers : 0) ? pl.a.n_layers : (pl.fuse_b ? pl.b.n_layers : 0);
  pl.img_floats = n_img > 0 ? (long long)n_img * (2 * fused::B_TILE / 4) + 64 : 0;
  pl.dzall_floats = 0;
  if (pl.fuse_b) {
    const long long wb = pl.b.max_width();
    pl.dzall_floats += (long long)(pl.b.n_layers - 1) * (pl.P * wb + 64) + ((pl.P + 127) / 128 + 16) * wb + 64;
  }
  if (pl.fuse_a) {
    const long long wa = pl.a.max_width();
    pl.dzall_floats += (long long)(pl.a.n_layers - 1) * (pl.N * wa + 64) + ((pl.N + 127) / 128 + 16) * wa + 64;
  }
  pl.fwd3 = pl.deeponet && fwd3_eligible(pl.a) && fwd3_eligible(pl.b) && pl.K <= xg::XK;
  pl.m_tiles = (int)((pl.N + 127) / 128);
  pl.p_tiles128 = (int)((pl.P + 127) / 128);
  pl.wimg3_floats = pl.ximg_a_floats = pl.ximg_b_floats = pl.xsc_floats = 0;
  if (pl.fwd3) {
    const int n_blobs = pl.a.n_layers > pl.b.n_layers ? pl.a.n_layers : pl.b.n_layers;
    pl.wimg3_floats = (long long)n_blobs * (xg::XIMG_B / 4) + 64;
    pl.ximg_a_floats = (long long)pl.m_tiles * (xg::XTILE / 4) + 64;
    pl.ximg_b_floats = (long long)pl.p_tiles128 * (xg::XTILE / 4) + 64;
    pl.xsc_floats = ((long long)pl.m_tiles + pl.p_tiles128) * 128 + 128;
  }
  pl.per_chain_floats = pl.wimg3_floats + pl.ximg_a_floats + pl.ximg_b_floats + pl.xsc_floats + pl.dzall_floats + pl.img_floats + pl.scratch_per_chain + 2 * pl.Dp + pl.act_a_floats + pl.act_b_floats + G + 2 * pl.R * wmax + 2 * tiles + 8 + 64 * 40 + pl.P + (p->d + 8191) / 8192;
  // shared by every chain: pad map, trunk features, padded copy of the targets
  pl.shared_floats = pl.D + 64 + (pl.deeponet ? pl.P * 5 + 64 + pl.N * pl.Pp + 64 : 0);
  return VIHMC_OK;
}

bool dense_supported(const vihmc_problem* p) {
  if (p->act == VIHMC_ACT_SINE) return false;  // the dense path stores activations only; cos(z) would need z
  DensePlan pl;
  return make_plan(p, pl) == VIHMC_OK;
}

static const long long kMaxBatchBytes = 40LL << 30;  // cap one chain batch at 40 GB of workspace

static long long chains_per_batch(const DensePlan& pl, long long C, size_t avail_bytes) {
  const long long per = pl.per_chain_floats * 4;
  long long cb = (long long)(avail_bytes / (size_t)per);
  if (cb > C) cb = C;
  if (cb > 65535) cb = 65535;
  return cb;
}

size_t dense_workspace_bytes(const vihmc_problem* p, long long C) {
  DensePlan pl;
  if (make_plan(p, pl) != VIHMC_OK) return 0;
  const long long per = pl.per_chain_floats * 4;
  long long cb = kMaxBatchBytes / per;
  if (cb < 1) cb = 1;
  if (cb > C) cb = C;
  return (size_t)(cb * per + pl.shared_floats * 4 + 4096);
}

namespace {
struct Bump {
  float* base;
  long long off = 0;
  explicit Bump(float* b) : base(b) {}
  float* take(long long n) {
    off = (off + 63) / 64 * 64;
    float* r = base + off;
    off += n;
    return r;
  }
};
}  // namespace

// forward of one stack for Cb chains: in [R, in_dim] shared -> acts[l] [Cb, R, dims[l]]   (D = padded per-chain stride of Wf);
// no activation on the last layer
static int stack_forward(const Stack& s, const float* input, long long R, const float* Wf, long long D, float* const* acts,
                         int act, int Cb, cudaStream_t st) {
  for (int l = 0; l < s.n_layers; ++l) {
    GemmArgs g{};
    const int in = s.in_of(l), out = s.dims[l];
    g.A = l == 0 ? input : acts[l - 1];
    g.a_bs = l == 0 ? 0 : R * in; g.a_sm = in; g.a_sk = 1;
    g.B = Wf + s.w_off[l]; g.b_bs = D; g.b_sk = 1; g.b_sn = s.ldw[l];   // opB[k,n] = W[n,k]
    g.C = acts[l]; g.c_bs = R * out; g.ldc = out;
    g.M = (int)R; g.N = out; g.K = in;
    if (s.has_bias[l]) {
      g.bias = Wf + s.b_off[l]; g.bias_bs = D;
      g.act = l == s.n_layers - 1 ? -1 : act;
      if (int rc = launch_gemm<EPI_BIAS_ACT>(g, Cb, st)) return rc;
    } else {
      if (int rc = launch_gemm<EPI_STORE>(g, Cb, st)) return rc;
    }
  }
  return VIHMC_OK;
}

// backward of one stack: dz holds d/d(pre-activation of the last layer) [Cb, R, dims[last]] on entry.
static int stack_backward(const Stack& s, const float* input, long long R, const float* Wf, float* dWf, long long D,
                          float* const* acts, float* dz_cur, float* dz_other, int act, int Cb, float* scratch, long long scratch_floats,
                          cudaStream_t st) {
  for (int l = s.n_layers - 1; l >= 0; --l) {
    const int in = s.in_of(l), out = s.dims[l];
    // dz_other is free until the dX GEMM below writes it: it holds the bias partials
    if (int rc = layer_weight_grad(s, l, input, R, acts, dz_cur, dWf, D, dz_other, Cb, scratch, scratch_floats, st)) return rc;
    if (l > 0) {
      // dz_prev[r,i] = (sum_o dz[r,o] W[o,i]) * act'(a_{l-1}[r,i])
      GemmArgs h{};
      h.A = dz_cur; h.a_bs = R * out; h.a_sm = out; h.a_sk = 1;
      h.B = Wf + s.w_off[l]; h.b_bs = D; h.b_sk = s.ldw[l]; h.b_sn = 1;   // opB[k=o,n=i] = W[o,i]
      h.C = dz_other; h.c_bs = R * in; h.ldc = in;
      h.M = (int)R; h.N = in; h.K = out;
      h.aux = acts[l - 1]; h.aux_bs = R * in; h.ld_aux = in; h.act = act;
      if (int rc = launch_gemm<EPI_DACT>(h, Cb, st)) return rc;
      float* t = dz_cur; dz_cur = dz_other; dz_other = t;
    }
  }
  return VIHMC_OK;
}

// forward of one stack of the plan: through fused_forward3_kernel when the plan runs both DeepONet stacks there (with the
// operand image and row scales of the last layer's output for head3_kernel), else through the fused 3xTF32 kernel when this
// stack is eligible (`fused`), else one GEMM per layer
static int stack_forward_any(const DensePlan& pl, const Stack& s, bool fused, const float* input, long long R, const float* Wf,
                             float* const* acts, int act, int Cb, float* img, unsigned char* wimg3, unsigned char* out_img,
                             float* out_scales, cudaStream_t st) {
  if (pl.fwd3) return stack_forward3(s, input, R, Wf, pl.Dp, acts, act, Cb, wimg3, out_img, out_scales, st);
  if (fused) return stack_forward_fused(s, input, R, Wf, pl.Dp, acts, act, Cb, img, st);
  return stack_forward(s, input, R, Wf, pl.Dp, acts, act, Cb, st);
}

// chain-independent buffers at the head of the workspace: pad map, trunk features, the targets the DeepONet head reads
struct SharedBufs {
  const int* pad_map;
  const float* trunk_in;
  const float* y_pad;   // log-posterior: [N, Pp] (DeepONet) or p->y; predict: a zero row (HEAD epilogue) or null (head3_kernel)
  long long ld_y;       // row stride of y_pad: Pp, or 0 for the zero row
  float* batch_base;
};

static int prepare_shared(const vihmc_problem* p, const DensePlan& pl, void* ws, bool predict, cudaStream_t st, SharedBufs& sb) {
  Bump bump(static_cast<float*>(ws));
  int* map = reinterpret_cast<int*>(bump.take(pl.D));
  pad_map_kernel<<<(unsigned)((pl.D + 255) / 256), 256, 0, st>>>(pl.tbl, pl.D, map);
  VIHMC_LAUNCH_OK("pad_map_kernel");
  sb.pad_map = map;
  sb.trunk_in = nullptr;
  sb.y_pad = predict ? nullptr : p->y;
  sb.ld_y = pl.Pp;
  if (pl.deeponet) {
    if (p->impose_bc) {
      float* feats = bump.take(pl.P * 5);
      trunk_features_kernel<<<(unsigned)((pl.P + 255) / 256), 256, 0, st>>>(p->x2, pl.P, feats);
      VIHMC_LAUNCH_OK("trunk_features_kernel");
      sb.trunk_in = feats;
    } else {
      sb.trunk_in = p->x2;
    }
    if (!predict && pl.Pp != pl.P) {   // rows of the targets on 16-byte boundaries: the head epilogue reads them with float4 loads
      float* yp = bump.take(pl.N * pl.Pp);
      VIHMC_CUDA_OK(cudaMemsetAsync(yp, 0, sizeof(float) * pl.N * pl.Pp, st));
      VIHMC_CUDA_OK(cudaMemcpy2DAsync(yp, sizeof(float) * pl.Pp, p->y, sizeof(float) * pl.P, sizeof(float) * pl.P, (size_t)pl.N,
                                      cudaMemcpyDeviceToDevice, st));
      sb.y_pad = yp;
    } else if (predict && !pl.fwd3) {   // the HEAD epilogue with prec = -1 against zero targets computes the outputs themselves
      float* zero_row = bump.take(pl.Pp);
      VIHMC_CUDA_OK(cudaMemsetAsync(zero_row, 0, sizeof(float) * pl.Pp, st));
      sb.y_pad = zero_row;
      sb.ld_y = 0;
    }
  }
  sb.batch_base = bump.take(0);
  return VIHMC_OK;
}

// Wf[c] = padded(frozen with q scattered at sens_ind)   (my_make_func.py:48-50 / :56-57)
static int scatter_padded(const vihmc_problem* p, const DensePlan& pl, const int* pad_map, const float* qb, float* Wf, int Cb,
                          cudaStream_t st, long long c0 = 0) {
  const long long D = pl.D, d = p->d;
  const unsigned gx = (unsigned)((D + 1023) / 1024 < 148 * 4 ? (D + 1023) / 1024 : 148 * 4);
  if (p->frozen == nullptr) {
    scatter_fill_padded_kernel<<<dim3(gx, Cb), 256, 0, st>>>(qb, D, pad_map, Wf, D, pl.Dp);
    VIHMC_LAUNCH_OK("scatter_fill_padded_kernel");
    return VIHMC_OK;
  }
  // frozen_chain_stride != 0: every chain has its own row of frozen weights (per-sample VI redraw)
  scatter_fill_padded_kernel<<<dim3(gx, Cb), 256, 0, st>>>(p->frozen + c0 * p->frozen_chain_stride, p->frozen_chain_stride, pad_map, Wf, D, pl.Dp);
  VIHMC_LAUNCH_OK("scatter_fill_padded_kernel");
  const unsigned gd = (unsigned)((d + 1023) / 1024 < 148 * 4 ? (d + 1023) / 1024 : 148 * 4);
  scatter_put_padded_kernel<<<dim3(gd, Cb), 256, 0, st>>>(reinterpret_cast<const long long*>(p->sens_ind), qb, pad_map, Wf, d, pl.Dp);
  VIHMC_LAUNCH_OK("scatter_put_padded_kernel");
  return VIHMC_OK;
}

// Log-posterior (out == NULL: logp[C], and grad[C, d] unless grad is NULL) or predict (out != NULL: MLP out[C, N]; DeepONet
// out[C, N, P] = Bout Tout^T + b0) for C chains, in batches of as many chains as the workspace holds.
int dense_run(const vihmc_problem* p, long long C, const float* q, float* logp, float* grad, float* out, void* ws, size_t ws_bytes,
              cudaStream_t st) {
  DensePlan pl;
  if (int rc = make_plan(p, pl)) return rc;
  const bool predict = out != nullptr;
  if (p->act == VIHMC_ACT_SINE) return fail(VIHMC_ERR_UNSUPPORTED, "dense path implements tanh and relu (the DeepONet reference's set)");
  if (p->x == nullptr || (pl.deeponet && p->x2 == nullptr)) return fail(VIHMC_ERR_INVALID, "x and x2 must be device pointers");
  if ((p->frozen == nullptr) != (p->sens_ind == nullptr)) return fail(VIHMC_ERR_INVALID, "frozen and sens_ind must be given together");
  if (p->sens_ind == nullptr && p->d != p->D) return fail(VIHMC_ERR_INVALID, "d != D requires sens_ind");
  if (!predict && p->y == nullptr) return fail(VIHMC_ERR_INVALID, "y must be a device pointer");
  if (!predict && p->prior_scale == 0.0f) return fail(VIHMC_ERR_INVALID, "prior_scale must be non-zero");
  if (ws == nullptr) return fail(VIHMC_ERR_WORKSPACE, "dense path needs a workspace");
  const size_t shared_bytes = (size_t)pl.shared_floats * 4 + 2048;
  if (ws_bytes <= shared_bytes) return fail(VIHMC_ERR_WORKSPACE, "workspace too small");
  const long long cb_max = chains_per_batch(pl, C, ws_bytes - shared_bytes);
  if (cb_max < 1) return fail(VIHMC_ERR_WORKSPACE, "workspace too small for one chain: need %lld bytes", pl.per_chain_floats * 4 + (long long)shared_bytes);
  const Likelihood lik = predict ? Likelihood{0.0f, 0.0f, -1.0f} : make_likelihood(p->loss, p->tau_out);
  const long long Dp = pl.Dp, d = p->d, N = pl.N, P = pl.P, Pp = pl.Pp;
  const int wmax = pl.a.max_width() > pl.b.max_width() ? pl.a.max_width() : pl.b.max_width();

  SharedBufs sb;
  if (int rc = prepare_shared(p, pl, ws, predict, st, sb)) return rc;
  const float* trunk_in = sb.trunk_in;
  if (!predict && pl.fwd3 && (reinterpret_cast<uintptr_t>(sb.y_pad) & 15u) != 0) return fail(VIHMC_ERR_INVALID, "targets must be 16-byte aligned");

  for (long long c0 = 0; c0 < C; c0 += cb_max) {
    const int Cb = (int)((C - c0) < cb_max ? (C - c0) : cb_max);
    Bump bb(sb.batch_base);
    float* Wf = bb.take((long long)Cb * Dp);
    float* dWf = bb.take((long long)Cb * Dp);
    float* acts_a[VIHMC_MAX_LAYERS];
    float* acts_b[VIHMC_MAX_LAYERS];
    for (int l = 0; l < pl.a.n_layers; ++l) acts_a[l] = bb.take((long long)Cb * N * pl.a.dims[l]);
    for (int l = 0; l < pl.b.n_layers; ++l) acts_b[l] = bb.take((long long)Cb * P * pl.b.dims[l]);
    const long long tiles = pl.deeponet ? pl.head_tiles : pl.loss_tiles;
    float* G = bb.take((long long)Cb * (pl.deeponet ? N * Pp : N));
    float* dz0 = bb.take((long long)Cb * pl.R * wmax);
    float* dz1 = bb.take((long long)Cb * pl.R * wmax);
    float* part_ll = bb.take((long long)Cb * tiles);
    float* part_g = bb.take((long long)Cb * tiles);
    float* loglik = bb.take(Cb);
    float* prior_part = bb.take((long long)Cb * ((d + kFinSlab - 1) / kFinSlab));
    const long long scratch_floats = (long long)Cb * pl.scratch_per_chain;
    float* scratch = scratch_floats > 0 ? bb.take(scratch_floats) : nullptr;
    float* img = pl.img_floats > 0 ? bb.take((long long)Cb * pl.img_floats) : nullptr;
    float* dzs_a[VIHMC_MAX_LAYERS] = {nullptr};
    float* dzs_b[VIHMC_MAX_LAYERS] = {nullptr};
    float* bias_part_a = nullptr;
    float* bias_part_b = nullptr;
    if (pl.fuse_b) {   // the fused backward keeps dz of every layer for the weight gradients
      const long long wb = pl.b.max_width();
      for (int l = 0; l < pl.b.n_layers - 1; ++l) dzs_b[l] = bb.take((long long)Cb * P * wb);
      dzs_b[pl.b.n_layers - 1] = dz0;
      bias_part_b = bb.take((long long)Cb * (((P + 127) / 128 + 16) * wb));
    }
    if (pl.fuse_a) {
      const long long wa = pl.a.max_width();
      for (int l = 0; l < pl.a.n_layers - 1; ++l) dzs_a[l] = bb.take((long long)Cb * N * wa);
      dzs_a[pl.a.n_layers - 1] = dz0;
      bias_part_a = bb.take((long long)Cb * (((N + 127) / 128 + 16) * wa));
    }
    unsigned char *wimg3 = nullptr, *ximg_a = nullptr, *ximg_b = nullptr;
    float *xsc_a = nullptr, *xsc_b = nullptr;
    if (pl.fwd3) {
      wimg3 = reinterpret_cast<unsigned char*>(bb.take((long long)Cb * pl.wimg3_floats));
      ximg_a = reinterpret_cast<unsigned char*>(bb.take((long long)Cb * pl.ximg_a_floats));
      ximg_b = reinterpret_cast<unsigned char*>(bb.take((long long)Cb * pl.ximg_b_floats));
      xsc_a = bb.take((long long)Cb * pl.m_tiles * 128);
      xsc_b = bb.take((long long)Cb * pl.p_tiles128 * 128);
    }
    const float* qb = q + c0 * d;

    if (int rc = scatter_padded(p, pl, sb.pad_map, qb, Wf, Cb, st, c0)) return rc;
    if (int rc = stack_forward_any(pl, pl.a, pl.fuse_a, p->x, N, Wf, acts_a, p->act, Cb, img, wimg3, ximg_a, xsc_a, st)) return rc;
    if (pl.deeponet)
      if (int rc = stack_forward_any(pl, pl.b, pl.fuse_b, trunk_in, P, Wf, acts_b, p->act, Cb, img, wimg3, ximg_b, xsc_b, st)) return rc;

    if (pl.deeponet) {
      // head: O = Bout * Tout^T + b0 into out (predict), or G = d loglik / dO with fused loglik partials
      const float* Bout = acts_a[pl.a.n_layers - 1];
      const float* Tout = acts_b[pl.b.n_layers - 1];
      const int K = pl.K;
      float* O = predict ? out + c0 * N * P : G;
      const long long ldo = predict ? P : Pp;   // G and the padded targets have Pp floats per row
      long long parts = tiles;
      if (pl.fwd3) {
        int np = 0;
        if (int rc = launch_head3(pl, Cb, ximg_a, xsc_a, ximg_b, xsc_b, Wf, Dp, sb.y_pad, sb.ld_y, O, N * ldo, ldo, lik, part_ll, part_g, &np, st)) return rc;
        parts = np;
      } else {
        GemmArgs g{};
        g.A = Bout; g.a_bs = N * K; g.a_sm = K; g.a_sk = 1;
        g.B = Tout; g.b_bs = P * K; g.b_sk = 1; g.b_sn = K;
        g.M = (int)N; g.N = (int)P; g.K = K;
        g.C = O; g.c_bs = N * ldo; g.ldc = ldo; g.row_pad_ok = !predict;
        g.bias = Wf; g.bias_bs = Dp;                   // scalar output bias is W[0] (my_make_func.py:52)
        g.aux = sb.y_pad; g.aux_bs = 0; g.ld_aux = sb.ld_y;
        g.ll_const = lik.ll_const; g.half_prec = lik.half_prec; g.prec = lik.prec;
        g.part_ll = part_ll; g.part_g = part_g;
        if (int rc = launch_gemm<EPI_HEAD>(g, Cb, st)) return rc;
      }
      if (predict) continue;
      reduce_partials_kernel<<<(Cb + 3) / 4, 128, 0, st>>>(part_ll, parts, Cb, loglik, 1);
      if (grad != nullptr) {
        reduce_partials_kernel<<<(Cb + 3) / 4, 128, 0, st>>>(part_g, parts, Cb, dWf, Dp);  // d/d b0 = sum G
        // dBout[n,k] = sum_p G[n,p] Tout[p,k]
        GemmArgs h{};
        h.A = G; h.a_bs = N * Pp; h.a_sm = Pp; h.a_sk = 1;
        h.B = Tout; h.b_bs = P * K; h.b_sk = K; h.b_sn = 1;
        h.C = dz0; h.c_bs = N * K; h.ldc = K; h.M = (int)N; h.N = K; h.K = (int)P;
        h.kc_hint = kDBoutChunk;
        if (int rc = launch_gemm<EPI_STORE>(h, Cb, st, scratch, scratch_floats)) return rc;
        if (bias_part_a != nullptr) {
          if (int rc = stack_backward_fused(pl.a, p->x, N, Wf, dWf, Dp, acts_a, dzs_a, p->act, Cb, img, bias_part_a, scratch, scratch_floats, st)) return rc;
        } else {
          if (int rc = stack_backward(pl.a, p->x, N, Wf, dWf, Dp, acts_a, dz0, dz1, p->act, Cb, scratch, scratch_floats, st)) return rc;
        }
        // dTout[p,k] = sum_n G[n,p] Bout[n,k]
        GemmArgs t{};
        t.A = G; t.a_bs = N * Pp; t.a_sm = 1; t.a_sk = Pp;
        t.B = Bout; t.b_bs = N * K; t.b_sk = K; t.b_sn = 1;
        t.C = dz0; t.c_bs = P * K; t.ldc = K; t.M = (int)P; t.N = K; t.K = (int)N;
        if (int rc = launch_gemm<EPI_STORE>(t, Cb, st, scratch, scratch_floats)) return rc;
        if (bias_part_b != nullptr) {
          if (int rc = stack_backward_fused(pl.b, trunk_in, P, Wf, dWf, Dp, acts_b, dzs_b, p->act, Cb, img, bias_part_b, scratch, scratch_floats, st)) return rc;
        } else {
          if (int rc = stack_backward(pl.b, trunk_in, P, Wf, dWf, Dp, acts_b, dz0, dz1, p->act, Cb, scratch, scratch_floats, st)) return rc;
        }
      }
    } else {
      const float* O = acts_a[pl.a.n_layers - 1];
      if (predict) {
        VIHMC_CUDA_OK(cudaMemcpyAsync(out + c0 * N, O, sizeof(float) * Cb * N, cudaMemcpyDeviceToDevice, st));
        continue;
      }
      mlp_loss_kernel<<<dim3((unsigned)pl.loss_tiles, Cb), 256, 0, st>>>(O, p->y, N, lik.ll_const, lik.half_prec, lik.prec, dz0, part_ll);
      VIHMC_LAUNCH_OK("mlp_loss_kernel");
      reduce_partials_kernel<<<(Cb + 3) / 4, 128, 0, st>>>(part_ll, tiles, Cb, loglik, 1);
      if (grad != nullptr)
        if (int rc = stack_backward(pl.a, p->x, N, Wf, dWf, Dp, acts_a, dz0, dz1, p->act, Cb, scratch, scratch_floats, st)) return rc;
    }
    const int slabs = (int)((d + kFinSlab - 1) / kFinSlab);
    finalize_kernel<<<dim3(slabs, Cb), 256, 0, st>>>(dWf, reinterpret_cast<const long long*>(p->sens_ind), qb, p->prior_mu,
                                                     p->prior_sigma, p->prior_sigma_scalar, 1.0f / p->prior_scale, Dp, d, sb.pad_map,
                                                     prior_part, grad ? grad + c0 * d : nullptr);
    VIHMC_LAUNCH_OK("finalize_kernel");
    logp_kernel<<<(Cb + 127) / 128, 128, 0, st>>>(prior_part, slabs, loglik, 1.0f / p->prior_scale, p->prior_log_norm, Cb, logp + c0);
    VIHMC_LAUNCH_OK("logp_kernel");
  }
  return VIHMC_OK;
}

// vihmc_gemm_batched (include/vihmc.h)
int dense_gemm(const float* A, long long a_bs, long long a_sm, long long a_sk, const float* B, long long b_bs, long long b_sk,
               long long b_sn, float* C, long long c_bs, long long ldc, int M, int N, int K, int batch, int use_tc, float* scratch,
               cudaStream_t st) {
  if (A == nullptr || B == nullptr || C == nullptr) return fail(VIHMC_ERR_INVALID, "gemm: null operand");
  if (use_tc && (M < 32 || K < 16)) return fail(VIHMC_ERR_UNSUPPORTED, "gemm: the tensor-core kernel needs M >= 32 and K >= 16");
  GemmArgs g{};
  g.A = A; g.a_bs = a_bs; g.a_sm = a_sm; g.a_sk = a_sk;
  g.B = B; g.b_bs = b_bs; g.b_sk = b_sk; g.b_sn = b_sn;
  g.C = C; g.c_bs = c_bs; g.ldc = ldc; g.M = M; g.N = N; g.K = K;
  // the splitk_scratch contract of vihmc_gemm_batched: ceil(K/256) * batch * M * N floats
  const long long scratch_floats = scratch != nullptr ? (long long)((K + kSplitKChunk - 1) / kSplitKChunk) * batch * M * N : 0;
  return launch_gemm<EPI_STORE>(g, batch, st, scratch, scratch_floats, use_tc ? 1 : 0);
}

// vihmc_debug_umma (include/vihmc.h): layout probe of one tcgen05.mma
int dense_umma_probe(const float* a_img, const float* b_img, unsigned a_lbo, unsigned a_sbo, unsigned b_lbo, unsigned b_sbo,
                     unsigned a_type, unsigned b_type, unsigned idesc_extra, float* out, cudaStream_t st) {
  if (a_img == nullptr || b_img == nullptr || out == nullptr) return fail(VIHMC_ERR_INVALID, "umma probe: null pointer");
  VIHMC_CUDA_OK(cudaFuncSetAttribute(tc::umma_probe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::kProbeSmem));
  tc::umma_probe_kernel<<<1, 128, tc::kProbeSmem, st>>>(a_img, b_img, a_lbo, a_sbo, b_lbo, b_sbo, a_type, b_type, tc::kIdesc | idesc_extra, out);
  VIHMC_LAUNCH_OK("umma_probe_kernel");
  return VIHMC_OK;
}

// vihmc_debug_tanh (include/vihmc.h): the tanh variants of the dense path, evaluated elementwise (bias measurements)
__global__ void debug_tanh_kernel(int kind, const float* __restrict__ x, float* __restrict__ y, long long n) {
  const long long i = 2 * ((long long)blockIdx.x * blockDim.x + threadIdx.x);
  if (i + 1 >= n) return;
  float a = x[i], b = x[i + 1], ya, yb;
  if (kind == 0) { ya = tanh_sel(a); yb = tanh_sel(b); }
  else if (kind == 1) { ya = tanhf(a); yb = tanhf(b); }
  else { xg::tanh_acc2(a, b, ya, yb); }
  y[i] = ya; y[i + 1] = yb;
}
int dense_debug_tanh(int kind, const float* x, float* y, long long n, cudaStream_t st) {
  debug_tanh_kernel<<<(unsigned)((n / 2 + 255) / 256), 256, 0, st>>>(kind, x, y, n);
  VIHMC_LAUNCH_OK("debug_tanh_kernel");
  return VIHMC_OK;
}

// vihmc_debug_xgemm (include/vihmc.h): C[b] = A[b] B[b]^T through the exact-accumulation operand images (xgemm.cuh)
size_t dense_xgemm_workspace(int M, int N, int batch) {
  const long long mt = (M + 127) / 128, nt = (N + 127) / 128;
  return (size_t)((mt + nt) * batch * (long long)xg::XTILE + ((long long)M + N) * batch * 4 + 1024);
}
int dense_xgemm_debug(const float* A, long long lda, const float* B, long long ldb, float* C, long long ldc, int M, int N, int K,
                      int batch, void* ws, size_t ws_bytes, cudaStream_t st) {
  if (A == nullptr || B == nullptr || C == nullptr || ws == nullptr) return fail(VIHMC_ERR_INVALID, "xgemm: null pointer");
  if (K < 1 || K > xg::XK) return fail(VIHMC_ERR_UNSUPPORTED, "xgemm: K must be in [1, %d]", xg::XK);
  if (ws_bytes < dense_xgemm_workspace(M, N, batch)) return fail(VIHMC_ERR_WORKSPACE, "xgemm: workspace too small");
  const int mt = (M + 127) / 128, nt = (N + 127) / 128;
  unsigned char* a_img = static_cast<unsigned char*>(ws);
  unsigned char* b_img = a_img + (size_t)mt * batch * xg::XTILE;
  float* a_sc = reinterpret_cast<float*>(b_img + (size_t)nt * batch * xg::XTILE);
  float* b_sc = a_sc + (size_t)M * batch;
  xg::image3_kernel<<<dim3(mt, batch), 256, 0, st>>>(A, (long long)M * lda, lda, M, K, a_img, a_sc, M);
  VIHMC_LAUNCH_OK("image3_kernel");
  xg::image3_kernel<<<dim3(nt, batch), 256, 0, st>>>(B, (long long)N * ldb, ldb, N, K, b_img, b_sc, N);
  VIHMC_LAUNCH_OK("image3_kernel");
  VIHMC_CUDA_OK(cudaFuncSetAttribute(xg::xgemm_test_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, xg::XT_SMEM));
  xg::xgemm_test_kernel<<<dim3(nt, mt, batch), 256, xg::XT_SMEM, st>>>(a_img, a_sc, b_img, b_sc, M, N, K, C, ldc);
  VIHMC_LAUNCH_OK("xgemm_test_kernel");
  return VIHMC_OK;
}

}  // namespace vihmc
