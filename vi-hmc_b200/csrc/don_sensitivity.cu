// DeepONet sensitivity scores -- the VI -> HMC split selector of the operator network.
//
// Reference (Operator_network/VI/sensitivity.py:61-126, eval_std_dydw / eval_jac): jacrev of the functional DeepONet
// (my_make_func.py:46-85) gives J[n, p, i] = d out[n, p] / d w_i for every parameter; the score is
//     s_i = sigma_i^2 * mean_{n, p} J[n, p, i]^2 .
// Materialising J costs N * P * D floats (1000 x 100 x 172 401 in the shipped config, hence the reference's batch size of 1).
// Here the mean of squares is computed EXACTLY without J.  out[n, p] = sum_k B[n, k] T[p, k] + b, so for a branch parameter
//     sum_p J[n, p, i]^2 = (dB[n, :]/dw_i)^T  G_T  (dB[n, :]/dw_i),   G_T = T^T T  (K x K Gram matrix of the trunk features),
// and with G_T = R^T R (Cholesky) this is  sum_r ( R[r, :] . dB[n, :]/dw_i )^2 :  K back-propagations through the branch per
// function n, seeded with the rows of R, instead of P.  For a weight W_l[a, b] the r-th back-propagation contributes
// delta_l[r, a] * h_{l-1}[b], so
//     s(W_l[a, b]) = sigma^2 / (N P) * sum_n E_l[n, a] * h_{l-1}[n, b]^2,      E_l[n, a] = sum_r delta_l[n, r, a]^2,
//     s(b_l[a])    = sigma^2 / (N P) * sum_n E_l[n, a],                         s(b) = sigma_b^2,
// and symmetrically for the trunk with G_B = B^T B.  Kernels (all FP32 SIMT, Gram / Cholesky / final sums in FP64):
//   don_sens_forward_kernel   one CTA per row: activations of every layer at the VI means
//   don_sens_gram_kernel      G = F^T F over the rows of the last layer's output
//   don_sens_chol_kernel      positive-semidefinite-safe Cholesky in one CTA (zero pivot -> zero row)
//   don_sens_backward_kernel  one CTA per row: the K seeded back-propagations as [K x w] x [w x w] products in shared memory
//   don_sens_score_kernel     the E^T H^2 contractions, scaled by sigma^2 / (N P)
#include "common.cuh"

namespace vihmc {

namespace {

constexpr int kMaxDim = 128;   // widths, output neurons <= 128 (backward tile buffers live in shared memory)
// the forward kernel keeps two rows of max(input, widths) floats in shared memory: 227 KB, the most a block may opt in to,
// bounds the inputs at 29 056
constexpr size_t kMaxForwardSmem = 232448;

struct StackDesc {
  int n_layers, in_dim, maxdim;
  int dims[VIHMC_MAX_LAYERS];
  long long w_off[VIHMC_MAX_LAYERS], b_off[VIHMC_MAX_LAYERS];   // into the flat weight vector
  long long act_off[VIHMC_MAX_LAYERS];                          // into the activation / E buffers (floats): [rows, dims[l]] each
  long long rows;
};

__global__ void don_sens_features_kernel(const float* __restrict__ x2, long long P, float* __restrict__ F) {
  const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  const float t = x2[2 * p], x = x2[2 * p + 1];
  const float two_pi = 6.283185307179586f, four_pi = 12.566370614359172f;   // my_make_func.py:33-36 in fp32
  F[5 * p + 0] = t;
  F[5 * p + 1] = sinf(two_pi * x);
  F[5 * p + 2] = sinf(four_pi * x);
  F[5 * p + 3] = cosf(two_pi * x);
  F[5 * p + 4] = cosf(four_pi * x);
}

template <int ACT>
__device__ __forceinline__ float act_fwd(float z) { return ACT == VIHMC_ACT_TANH ? tanhf(z) : fmaxf(z, 0.f); }
template <int ACT>
__device__ __forceinline__ float act_deriv_from_output(float h) { return ACT == VIHMC_ACT_TANH ? 1.f - h * h : (h > 0.f ? 1.f : 0.f); }

// one CTA (4 warps) per row; a warp owns output units j = warp, warp + 4, ...: coalesced weight-row reads, shuffle reduction
template <int ACT>
__global__ void __launch_bounds__(128) don_sens_forward_kernel(StackDesc s, const float* __restrict__ w, const float* __restrict__ input,
                                                               int in_ld, float* __restrict__ acts) {
  extern __shared__ float sm[];
  float* cur = sm;
  float* nxt = sm + s.maxdim;
  const long long row = blockIdx.x;
  for (int i = threadIdx.x; i < s.in_dim; i += 128) cur[i] = input[row * in_ld + i];
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int in = s.in_dim;
  for (int l = 0; l < s.n_layers; ++l) {
    const int out = s.dims[l];
    const float* W = w + s.w_off[l];
    const float* B = w + s.b_off[l];
    for (int j = warp; j < out; j += 4) {
      float acc = 0.f;
      for (int k = lane; k < in; k += 32) acc = fmaf(W[(long long)j * in + k], cur[k], acc);
      for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
      if (lane == 0) {
        float z = acc + B[j];
        if (l < s.n_layers - 1) z = act_fwd<ACT>(z);
        nxt[j] = z;
        acts[s.act_off[l] + row * out + j] = z;
      }
    }
    __syncthreads();
    float* t = cur; cur = nxt; nxt = t;
    in = out;
  }
}

// G[i][j] = sum_rows F[row][i] F[row][j] in FP64; grid K, block 128 (j)
__global__ void __launch_bounds__(128) don_sens_gram_kernel(const float* __restrict__ F, long long rows, int K, double* __restrict__ G) {
  const int i = blockIdx.x, j = threadIdx.x;
  if (j >= K) return;
  double acc = 0.0;
  for (long long r = 0; r < rows; ++r) acc = fma((double)F[r * K + i], (double)F[r * K + j], acc);
  G[i * K + j] = acc;
}

// Upper Cholesky factor R (R^T R = G) of a positive SEMI-definite matrix, one CTA: a pivot that is not positive (relative to
// the largest diagonal entry) means the whole remaining row is zero in exact arithmetic, so R's row is set to zero.
__global__ void __launch_bounds__(256) don_sens_chol_kernel(const double* __restrict__ G, int K, float* __restrict__ R) {
  extern __shared__ double A[];   // [K][K]
  __shared__ double piv;
  for (int i = threadIdx.x; i < K * K; i += 256) A[i] = G[i];
  __syncthreads();
  double dmax = 0.0;
  for (int i = 0; i < K; ++i) dmax = fmax(dmax, A[i * K + i]);
  const double tol = 1e-12 * dmax;
  for (int k = 0; k < K; ++k) {
    if (threadIdx.x == 0) piv = A[k * K + k] > tol ? sqrt(A[k * K + k]) : 0.0;
    __syncthreads();
    const double p = piv;
    for (int j = threadIdx.x; j < K; j += 256) A[k * K + j] = (j < k || p == 0.0) ? 0.0 : (j == k ? p : A[k * K + j] / p);
    __syncthreads();
    if (p != 0.0) {
      const int m = K - k - 1;
      for (int t = threadIdx.x; t < m * m; t += 256) {
        const int i = k + 1 + t / m, j = k + 1 + t % m;
        if (j >= i) A[i * K + j] -= A[k * K + i] * A[k * K + j];
      }
    }
    __syncthreads();
  }
  for (int i = threadIdx.x; i < K * K; i += 256) R[i] = (float)A[i];
}

// One CTA per row n.  delta [K seeds x width] starts as R and is pulled back layer by layer:
//   E_l[n, a] = sum_r delta[r, a]^2 ;   delta <- (delta W_l) * act'(h_{l-1}[n, :])
// NB = padded dimension / 16 (both the seed count and the widths are padded to 16 NB with zeros); thread (tx, ty) of the 16 x 16
// block owns the NB x NB register tile rows ty + 16 i, columns tx + 16 j.
template <int ACT, int NB>
__global__ void __launch_bounds__(256) don_sens_backward_kernel(StackDesc s, const float* __restrict__ w, const float* __restrict__ R, int K,
                                                                const float* __restrict__ acts, float* __restrict__ E) {
  constexpr int Dp = 16 * NB;
  extern __shared__ float smf[];
  float* cur = smf;
  float* nxt = cur + Dp * Dp;
  float* Wl = nxt + Dp * Dp;
  float* hp = Wl + Dp * Dp;
  const long long row = blockIdx.x;
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  for (int i = tid; i < Dp * Dp; i += 256) {
    const int r = i / Dp, a = i % Dp;
    cur[i] = (r < K && a < K) ? R[r * K + a] : 0.f;
  }
  __syncthreads();
  for (int l = s.n_layers - 1; l >= 0; --l) {
    const int out = s.dims[l];
    if (tid < out) {
      float e = 0.f;
      for (int r = 0; r < Dp; ++r) {
        const float v = cur[r * Dp + tid];
        e = fmaf(v, v, e);
      }
      E[s.act_off[l] + row * out + tid] = e;
    }
    if (l == 0) break;
    const int in = s.dims[l - 1];
    const float* W = w + s.w_off[l];
    for (int i = tid; i < Dp * Dp; i += 256) {
      const int a = i / Dp, b = i % Dp;
      Wl[i] = (a < out && b < in) ? W[(long long)a * in + b] : 0.f;
    }
    if (tid < Dp) hp[tid] = tid < in ? act_deriv_from_output<ACT>(acts[s.act_off[l - 1] + row * in + tid]) : 0.f;
    __syncthreads();
    float acc[NB][NB];
#pragma unroll
    for (int i = 0; i < NB; ++i)
#pragma unroll
      for (int j = 0; j < NB; ++j) acc[i][j] = 0.f;
    const int a_end = (out + 3) & ~3;
    for (int a = 0; a < a_end; ++a) {
      float dv[NB], wv[NB];
#pragma unroll
      for (int i = 0; i < NB; ++i) dv[i] = cur[(ty + 16 * i) * Dp + a];
#pragma unroll
      for (int j = 0; j < NB; ++j) wv[j] = Wl[a * Dp + tx + 16 * j];
#pragma unroll
      for (int i = 0; i < NB; ++i)
#pragma unroll
        for (int j = 0; j < NB; ++j) acc[i][j] = fmaf(dv[i], wv[j], acc[i][j]);
    }
#pragma unroll
    for (int i = 0; i < NB; ++i)
#pragma unroll
      for (int j = 0; j < NB; ++j) nxt[(ty + 16 * i) * Dp + tx + 16 * j] = acc[i][j] * hp[tx + 16 * j];
    __syncthreads();
    float* t = cur; cur = nxt; nxt = t;
  }
}

// scores of W_l[a, b] and b_l[a]: grid (ceil(out / 4), ceil(in / 128)), block 128 over b; FP64 accumulation over the rows
__global__ void __launch_bounds__(128) don_sens_score_kernel(const float* __restrict__ El, const float* __restrict__ inl, int in_ld,
                                                             long long rows, int out, int in, const float* __restrict__ sigma_W,
                                                             const float* __restrict__ sigma_b, float* __restrict__ score_W,
                                                             float* __restrict__ score_b, double scale) {
  const int a0 = blockIdx.x * 4, b = blockIdx.y * 128 + threadIdx.x;
  const bool bias_lane = (blockIdx.y == 0 && threadIdx.x == 0);
  double acc[4] = {0.0, 0.0, 0.0, 0.0}, accb[4] = {0.0, 0.0, 0.0, 0.0};
  for (long long r = 0; r < rows; ++r) {
    const float x = b < in ? inl[r * in_ld + b] : 0.f;
    const double v = (double)x * (double)x;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const double e = (a0 + i < out) ? (double)El[r * out + a0 + i] : 0.0;
      acc[i] = fma(e, v, acc[i]);
      if (bias_lane) accb[i] += e;
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int a = a0 + i;
    if (a >= out) continue;
    if (b < in) {
      const float sg = sigma_W[(long long)a * in + b];
      score_W[(long long)a * in + b] = (float)(acc[i] * scale * (double)sg * (double)sg);
    }
    if (bias_lane) {
      const float sg = sigma_b[a];
      score_b[a] = (float)(accb[i] * scale * (double)sg * (double)sg);
    }
  }
}

__global__ void don_sens_outbias_kernel(const float* __restrict__ sigma, float* __restrict__ scores) {
  scores[0] = sigma[0] * sigma[0];   // d out / d b = 1 for every (n, p)
}

inline size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

struct Plan {
  StackDesc br, tr;
  int K, NB;
  size_t fwd_smem;
  size_t off_feat, off_acts_br, off_acts_tr, off_E_br, off_E_tr, off_G, off_R, total;
};

int make_plan(const vihmc_problem* p, Plan& pl) {
  if (p->model_kind != VIHMC_MODEL_DEEPONET) return fail(VIHMC_ERR_INVALID, "deeponet sensitivity: not a DeepONet problem");
  if (p->act != VIHMC_ACT_TANH && p->act != VIHMC_ACT_RELU)
    return fail(VIHMC_ERR_UNSUPPORTED, "deeponet sensitivity: activation should be relu or tanh");
  if (p->n_layers_a < 1 || p->n_layers_b < 1 || p->n_layers_a > VIHMC_MAX_LAYERS || p->n_layers_b > VIHMC_MAX_LAYERS)
    return fail(VIHMC_ERR_INVALID, "deeponet sensitivity: bad depth");
  if (p->N < 1 || p->P < 1) return fail(VIHMC_ERR_INVALID, "deeponet sensitivity: empty validation set");
  long long off = 1;   // w[0] is the output bias (model.py:26)
  auto fill = [&](StackDesc& s, int n_layers, int in_dim, const int32_t* dims, long long rows) {
    s.n_layers = n_layers; s.in_dim = in_dim; s.rows = rows; s.maxdim = in_dim;
    long long aoff = 0;
    int prev = in_dim;
    for (int l = 0; l < n_layers; ++l) {
      s.dims[l] = dims[l];
      s.w_off[l] = off; off += (long long)dims[l] * prev;
      s.b_off[l] = off; off += dims[l];
      s.act_off[l] = aoff; aoff += rows * dims[l];
      if (dims[l] > s.maxdim) s.maxdim = dims[l];
      prev = dims[l];
    }
    return aoff;
  };
  const long long acts_br = fill(pl.br, p->n_layers_a, p->in_a, p->dims_a, p->N);
  const long long acts_tr = fill(pl.tr, p->n_layers_b, p->in_b, p->dims_b, p->P);
  if (off != p->D) return fail(VIHMC_ERR_INVALID, "deeponet sensitivity: layer table has %lld parameters, D = %lld", off, (long long)p->D);
  pl.K = p->dims_a[p->n_layers_a - 1];
  if (pl.K != p->dims_b[p->n_layers_b - 1]) return fail(VIHMC_ERR_INVALID, "deeponet sensitivity: branch / trunk output widths differ");
  int maxw = pl.K;
  for (int l = 0; l < p->n_layers_a; ++l) maxw = p->dims_a[l] > maxw ? p->dims_a[l] : maxw;
  for (int l = 0; l < p->n_layers_b; ++l) maxw = p->dims_b[l] > maxw ? p->dims_b[l] : maxw;
  if (maxw > kMaxDim) return fail(VIHMC_ERR_UNSUPPORTED, "deeponet sensitivity: widths up to %d are implemented (got %d)", kMaxDim, maxw);
  pl.NB = (maxw + 15) / 16;
  pl.fwd_smem = (size_t)2 * (pl.br.maxdim > pl.tr.maxdim ? pl.br.maxdim : pl.tr.maxdim) * sizeof(float);
  if (pl.fwd_smem > kMaxForwardSmem)
    return fail(VIHMC_ERR_UNSUPPORTED, "deeponet sensitivity: branch / trunk inputs up to %d are implemented (got %d / %d)",
                (int)(kMaxForwardSmem / (2 * sizeof(float))), p->in_a, p->in_b);
  size_t o = 0;
  pl.off_feat = o;    o += align256((size_t)p->P * 5 * sizeof(float));
  pl.off_acts_br = o; o += align256((size_t)acts_br * sizeof(float));
  pl.off_acts_tr = o; o += align256((size_t)acts_tr * sizeof(float));
  pl.off_E_br = o;    o += align256((size_t)acts_br * sizeof(float));
  pl.off_E_tr = o;    o += align256((size_t)acts_tr * sizeof(float));
  pl.off_G = o;       o += align256((size_t)2 * pl.K * pl.K * sizeof(double));
  pl.off_R = o;       o += align256((size_t)2 * pl.K * pl.K * sizeof(float));
  pl.total = o;
  return VIHMC_OK;
}

template <int ACT, int NB>
int launch_backward(const StackDesc& s, const float* w, const float* R, int K, const float* acts, float* E, cudaStream_t st) {
  constexpr int Dp = 16 * NB;
  const size_t smem = (size_t)(3 * Dp * Dp + Dp) * sizeof(float);
  auto kern = don_sens_backward_kernel<ACT, NB>;
  VIHMC_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<(unsigned)s.rows, 256, smem, st>>>(s, w, R, K, acts, E);
  VIHMC_LAUNCH_OK("don_sens_backward_kernel");
  return VIHMC_OK;
}

template <int ACT>
int dispatch_backward(int NB, const StackDesc& s, const float* w, const float* R, int K, const float* acts, float* E, cudaStream_t st) {
  switch (NB) {
    case 1: return launch_backward<ACT, 1>(s, w, R, K, acts, E, st);
    case 2: return launch_backward<ACT, 2>(s, w, R, K, acts, E, st);
    case 3: return launch_backward<ACT, 3>(s, w, R, K, acts, E, st);
    case 4: return launch_backward<ACT, 4>(s, w, R, K, acts, E, st);
    case 5: return launch_backward<ACT, 5>(s, w, R, K, acts, E, st);
    case 6: return launch_backward<ACT, 6>(s, w, R, K, acts, E, st);
    case 7: return launch_backward<ACT, 7>(s, w, R, K, acts, E, st);
    default: return launch_backward<ACT, 8>(s, w, R, K, acts, E, st);
  }
}

template <int ACT>
int run(const vihmc_problem* p, const Plan& pl, const float* w, const float* sigma, float* scores, char* ws, cudaStream_t st) {
  float* feat = reinterpret_cast<float*>(ws + pl.off_feat);
  float* acts_br = reinterpret_cast<float*>(ws + pl.off_acts_br);
  float* acts_tr = reinterpret_cast<float*>(ws + pl.off_acts_tr);
  float* E_br = reinterpret_cast<float*>(ws + pl.off_E_br);
  float* E_tr = reinterpret_cast<float*>(ws + pl.off_E_tr);
  double* G_T = reinterpret_cast<double*>(ws + pl.off_G);
  double* G_B = G_T + (size_t)pl.K * pl.K;
  float* R_T = reinterpret_cast<float*>(ws + pl.off_R);
  float* R_B = R_T + (size_t)pl.K * pl.K;
  const int K = pl.K;
  const float* trunk_in = p->x2;
  if (p->impose_bc) {
    if (p->in_b != 5) return fail(VIHMC_ERR_INVALID, "deeponet sensitivity: the feature layer produces 5 trunk inputs, in_b = %d", p->in_b);
    don_sens_features_kernel<<<(unsigned)((p->P + 255) / 256), 256, 0, st>>>(p->x2, p->P, feat);
    VIHMC_LAUNCH_OK("don_sens_features_kernel");
    trunk_in = feat;
  }
  // 1. activations at the VI means (inputs past 6 144 floats need more than the 48 KB of shared memory a launch gets by default)
  VIHMC_CUDA_OK(cudaFuncSetAttribute(don_sens_forward_kernel<ACT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.fwd_smem));
  don_sens_forward_kernel<ACT><<<(unsigned)p->N, 128, 2 * pl.br.maxdim * sizeof(float), st>>>(pl.br, w, p->x, p->in_a, acts_br);
  VIHMC_LAUNCH_OK("don_sens_forward_kernel(branch)");
  don_sens_forward_kernel<ACT><<<(unsigned)p->P, 128, 2 * pl.tr.maxdim * sizeof(float), st>>>(pl.tr, w, trunk_in, p->in_b, acts_tr);
  VIHMC_LAUNCH_OK("don_sens_forward_kernel(trunk)");
  // 2. Gram matrices of the two feature sets and their Cholesky factors
  const float* Bout = acts_br + pl.br.act_off[pl.br.n_layers - 1];
  const float* Tout = acts_tr + pl.tr.act_off[pl.tr.n_layers - 1];
  don_sens_gram_kernel<<<K, 128, 0, st>>>(Tout, p->P, K, G_T);
  don_sens_gram_kernel<<<K, 128, 0, st>>>(Bout, p->N, K, G_B);
  VIHMC_LAUNCH_OK("don_sens_gram_kernel");
  const size_t chol_smem = (size_t)K * K * sizeof(double);
  VIHMC_CUDA_OK(cudaFuncSetAttribute(don_sens_chol_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)chol_smem));
  don_sens_chol_kernel<<<1, 256, chol_smem, st>>>(G_T, K, R_T);
  don_sens_chol_kernel<<<1, 256, chol_smem, st>>>(G_B, K, R_B);
  VIHMC_LAUNCH_OK("don_sens_chol_kernel");
  // 3. seeded back-propagations: the branch is seeded with the trunk's factor and vice versa
  if (int rc = dispatch_backward<ACT>(pl.NB, pl.br, w, R_T, K, acts_br, E_br, st)) return rc;
  if (int rc = dispatch_backward<ACT>(pl.NB, pl.tr, w, R_B, K, acts_tr, E_tr, st)) return rc;
  // 4. scores
  const double scale = 1.0 / ((double)p->N * (double)p->P);
  auto score_stack = [&](const StackDesc& s, const float* input, int in_ld, const float* acts, const float* E) {
    for (int l = 0; l < s.n_layers; ++l) {
      const int out = s.dims[l], in = l == 0 ? s.in_dim : s.dims[l - 1];
      const float* inl = l == 0 ? input : acts + s.act_off[l - 1];
      const int ld = l == 0 ? in_ld : in;
      dim3 grid((unsigned)((out + 3) / 4), (unsigned)((in + 127) / 128));
      don_sens_score_kernel<<<grid, 128, 0, st>>>(E + s.act_off[l], inl, ld, s.rows, out, in, sigma + s.w_off[l], sigma + s.b_off[l],
                                                  scores + s.w_off[l], scores + s.b_off[l], scale);
    }
  };
  score_stack(pl.br, p->x, p->in_a, acts_br, E_br);
  score_stack(pl.tr, trunk_in, p->in_b, acts_tr, E_tr);
  don_sens_outbias_kernel<<<1, 1, 0, st>>>(sigma, scores);
  VIHMC_LAUNCH_OK("don_sens_score_kernel");
  return VIHMC_OK;
}

}  // namespace

size_t deeponet_sensitivity_workspace(const vihmc_problem* prob) {
  Plan pl{};
  if (make_plan(prob, pl) != VIHMC_OK) return 0;
  return pl.total;
}

int deeponet_sensitivity(const vihmc_problem* prob, const float* weights, const float* sigma, float* scores, void* ws, size_t ws_bytes,
                         cudaStream_t st) {
  if (prob->d != prob->D || prob->sens_ind != nullptr || prob->frozen != nullptr)
    return fail(VIHMC_ERR_INVALID, "deeponet sensitivity: pass the full weight vector (d == D, no frozen / sens_ind)");
  // the plan first: an unsupported architecture is reported with its reason even when called with NULL buffers
  Plan pl{};
  if (int rc = make_plan(prob, pl)) return rc;
  if (weights == nullptr || sigma == nullptr || scores == nullptr || prob->x == nullptr || prob->x2 == nullptr)
    return fail(VIHMC_ERR_INVALID, "deeponet sensitivity: null pointer");
  if (ws == nullptr || ws_bytes < pl.total)
    return fail(VIHMC_ERR_WORKSPACE, "deeponet sensitivity: workspace too small, need %zu bytes", pl.total);
  char* base = static_cast<char*>(ws);
  return prob->act == VIHMC_ACT_TANH ? run<VIHMC_ACT_TANH>(prob, pl, weights, sigma, scores, base, st)
                                     : run<VIHMC_ACT_RELU>(prob, pl, weights, sigma, scores, base, st);
}

}  // namespace vihmc
