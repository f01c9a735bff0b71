// Small-MLP path: host-side validation, kernel selection and launch geometry (kernels: mlp_small.cuh).
#include <stdlib.h>

#include "mlp_small.cuh"

namespace vihmc {

// ------------------------------------------------------------------------------------------------
// host side: validation, dispatch on (padded width, hidden layers), launch geometry
// ------------------------------------------------------------------------------------------------
static int pick_width(int maxw) {
  if (maxw <= 10) return 10;
  if (maxw <= 16) return 16;
  if (maxw <= 32) return 32;
  return 0;
}

bool mlp_small_supported(const vihmc_problem* p) {
  if (p->model_kind != VIHMC_MODEL_MLP) return false;
  const int nh = p->n_layers_a - 1;
  if (nh < 1 || nh > kMaxHidden) return false;
  if (p->dims_a[nh] != 1) return false;
  int maxw = 0;
  for (int l = 0; l < nh; ++l) maxw = p->dims_a[l] > maxw ? p->dims_a[l] : maxw;
  if (pick_width(maxw) == 0) return false;
  if (p->in_a < 1 || p->in_a > 64) return false;
  const SmallLayout L = make_layout(pick_width(maxw), nh, p->in_a, p->d);
  if (L.act_total >= 65536) return false;                   // phase-B offsets are packed in 16 bits
  return (size_t)L.total * sizeof(float) <= 200u * 1024u;  // one chain must fit in one CTA's smem
}

static bool fast_path_enabled();
static int fast_version();

// allow_fast: the caller's kernel has a specialised variant (log-posterior/gradient and the sampler; not predict)
static int fill_params(const vihmc_problem* p, SmallParams& P, int& W, bool allow_fast, int& fast) {
  if (!mlp_small_supported(p))
    return fail(VIHMC_ERR_UNSUPPORTED, "MLP outside the small-net kernel's range (<=4 hidden layers of width <=32, out_dim 1)");
  if (p->x == nullptr || p->y == nullptr) return fail(VIHMC_ERR_INVALID, "x and y must be device pointers");
  if ((p->frozen == nullptr) != (p->sens_ind == nullptr))
    return fail(VIHMC_ERR_INVALID, "frozen and sens_ind must be given together");
  if (p->sens_ind == nullptr && p->d != p->D) return fail(VIHMC_ERR_INVALID, "d != D requires sens_ind");
  if (p->d < 1 || p->d > p->D || p->N < 1) return fail(VIHMC_ERR_INVALID, "bad d/D/N");
  const int nh = p->n_layers_a - 1;
  long long D = 0;
  int prev = p->in_a, maxw = 0;
  for (int l = 0; l <= nh; ++l) {
    const int o = p->dims_a[l];
    if (o < 1) return fail(VIHMC_ERR_INVALID, "layer width must be positive");
    D += (long long)o * prev + ((l < nh || p->last_bias) ? o : 0);
    if (l < nh && o > maxw) maxw = o;
    prev = o;
  }
  if (D != p->D) return fail(VIHMC_ERR_INVALID, "D=%lld does not match the architecture (%lld)", (long long)p->D, D);
  if (p->prior_scale == 0.0f) return fail(VIHMC_ERR_INVALID, "prior_scale must be non-zero");
  W = pick_width(maxw);
  P.act = p->act; P.loss = p->loss; P.last_bias = p->last_bias; P.n_hidden = nh; P.in_dim = p->in_a;
  for (int l = 0; l < kMaxHidden; ++l) P.widths[l] = l < nh ? p->dims_a[l] : 0;
  P.D = p->D; P.d = p->d; P.N = p->N;
  P.tau_out = p->tau_out; P.inv_prior_scale = 1.0f / p->prior_scale;
  P.prior_sigma_scalar = p->prior_sigma_scalar; P.prior_log_norm = p->prior_log_norm;
  P.x = p->x; P.y = p->y; P.frozen = p->frozen; P.frozen_cs = p->frozen_chain_stride; P.prior_mu = p->prior_mu; P.prior_sigma = p->prior_sigma;
  P.sens_ind = reinterpret_cast<const long long*>(p->sens_ind);
  fast = allow_fast && fast_path_enabled() && nh == 2 && p->in_a == 1 && p->act == VIHMC_ACT_TANH && p->N <= (32 / W) * 8;
  if (fast && W <= 16 && p->last_bias) fast = fast_version();
  P.lay = make_layout(W, nh, p->in_a, p->d, fast);
  return VIHMC_OK;
}

int mlp_small_launch_w10(SmallOp, const SmallParams&, const SmallLaunch&, cudaStream_t);
int mlp_small_launch_w16(SmallOp, const SmallParams&, const SmallLaunch&, cudaStream_t);
int mlp_small_launch_w32(SmallOp, const SmallParams&, const SmallLaunch&, cudaStream_t);

// VIHMC_SMALL_GENERIC=1 keeps every problem on the generic evaluation (the A/B baseline of the bit-exactness test)
static bool fast_path_enabled() {
  static const bool on = []() {
    const char* e = getenv("VIHMC_SMALL_GENERIC");
    return !(e != nullptr && e[0] == '1');
  }();
  return on;
}

// VIHMC_SMALL_FAST=1 keeps the round-1 specialised evaluation (eval_fast); default: version 2 (eval_fast2) for widths <= 16
static int fast_version() {
  static const int v = []() {
    const char* e = getenv("VIHMC_SMALL_FAST");
    return (e != nullptr && e[0] == '1') ? 1 : 2;
  }();
  return v;
}

// Geometry: one warp per chain; 1 chain per CTA for few chains so the 148 SMs fill evenly, up to 4 for many chains so
// the 32-CTA/SM limit does not cap residency.
static void pick_geometry(const SmallParams& P, long long C, SmallLaunch& a) {
  const SmallLayout& L = P.lay;
  const size_t per_chain = (size_t)L.total * sizeof(float);
  int cpb = 1;
  while (cpb < 4 && C > (long long)148 * 24 * cpb && per_chain * (cpb * 2) <= 200u * 1024u) cpb *= 2;
  a.chains_per_block = cpb;
  a.blocks = (int)((C + cpb - 1) / cpb);
  a.smem = per_chain * cpb;
  a.C = C;
}

static int dispatch(int W, SmallOp op, const SmallParams& P, const SmallLaunch& a, cudaStream_t st) {
  if (W == 10) return mlp_small_launch_w10(op, P, a, st);
  if (W == 16) return mlp_small_launch_w16(op, P, a, st);
  if (W == 32) return mlp_small_launch_w32(op, P, a, st);
  return fail(VIHMC_ERR_UNSUPPORTED, "no small-MLP instantiation for width %d", W);
}

int mlp_small_logp_grad(const vihmc_problem* prob, long long C, const float* q, float* logp, float* grad, cudaStream_t st) {
  SmallParams P{};
  int W = 0;
  SmallLaunch a{};
  if (int rc = fill_params(prob, P, W, true, a.fast)) return rc;
  pick_geometry(P, C, a);
  a.q = q; a.logp = logp; a.grad = grad;
  return dispatch(W, kOpLogpGrad, P, a, st);
}

int mlp_small_predict(const vihmc_problem* prob, long long C, const float* q, float* out, cudaStream_t st) {
  SmallParams P{};
  int W = 0;
  SmallLaunch a{};
  if (int rc = fill_params(prob, P, W, false, a.fast)) return rc;
  pick_geometry(P, C, a);
  a.q = q; a.out = out;
  return dispatch(W, kOpPredict, P, a, st);
}

// out[i] = sigma_i^2 * (sum_chunks partial[chunk, i]) / N
static __global__ void sensitivity_finish_kernel(const float* __restrict__ partial, int chunks, long long d, long long N,
                                          const float* __restrict__ sigma, float* __restrict__ out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= d) return;
  float s = 0.0f;
  for (int c = 0; c < chunks; ++c) s += partial[(long long)c * d + i];
  const float sg = sigma[i];
  out[i] = s / (float)N * (sg * sg);
}

// vihmc_mlp_sensitivity: prob->x = validation inputs [N, in], d == D (no VI split); workspace = chunks * D floats
size_t mlp_small_sensitivity_workspace(const vihmc_problem* prob) {
  if (!mlp_small_supported(prob)) return 0;
  int maxw = 0;
  for (int l = 0; l < prob->n_layers_a - 1; ++l) maxw = prob->dims_a[l] > maxw ? prob->dims_a[l] : maxw;
  const int NC = (32 / pick_width(maxw)) * 8;
  return (size_t)((prob->N + NC - 1) / NC) * (size_t)prob->D * sizeof(float);
}

int mlp_small_sensitivity(const vihmc_problem* prob, const float* weights, const float* sigma, float* out, void* ws, size_t ws_bytes,
                          cudaStream_t st) {
  if (prob->d != prob->D || prob->sens_ind != nullptr || prob->frozen != nullptr)
    return fail(VIHMC_ERR_INVALID, "sensitivity: pass the full weight vector (d == D, no frozen / sens_ind)");
  if (weights == nullptr || sigma == nullptr || out == nullptr) return fail(VIHMC_ERR_INVALID, "sensitivity: null pointer");
  vihmc_problem p = *prob;
  if (p.y == nullptr) p.y = p.x;   // targets are not used; the staging code reads one float per data point
  SmallParams P{};
  int W = 0;
  SmallLaunch a{};
  if (int rc = fill_params(&p, P, W, false, a.fast)) return rc;
  const size_t need = mlp_small_sensitivity_workspace(&p);
  if (ws == nullptr || ws_bytes < need) return fail(VIHMC_ERR_WORKSPACE, "sensitivity: workspace too small, need %zu bytes", need);
  const int chunks = (int)((P.N + P.lay.NC - 1) / P.lay.NC);
  a.chains_per_block = 1; a.blocks = chunks; a.smem = (size_t)P.lay.total * sizeof(float); a.C = 1;
  a.q = weights; a.out = static_cast<float*>(ws);
  if (int rc = dispatch(W, kOpSensitivity, P, a, st)) return rc;
  sensitivity_finish_kernel<<<(unsigned)((P.d + 127) / 128), 128, 0, st>>>(a.out, chunks, P.d, P.N, sigma, out);
  VIHMC_LAUNCH_OK("sensitivity_finish_kernel");
  return VIHMC_OK;
}

int mlp_small_sample(const vihmc_problem* prob, const vihmc_sampler_cfg* cfg, long long C, const float* q0, float* samples,
                     const vihmc_sampler_io* io, cudaStream_t st) {
  SmallParams P{};
  int W = 0;
  SmallLaunch a{};
  if (int rc = fill_params(prob, P, W, true, a.fast)) return rc;
  if (io != nullptr && io->inv_mass != nullptr) {
    // diagonal mass: the same variant with the per-coordinate m_i, s_i region appended to each chain's shared memory
    P.lay = make_layout(W, P.n_hidden, P.in_dim, P.d, a.fast, true);
    if ((size_t)P.lay.total * sizeof(float) > 227u * 1024u)
      return fail(VIHMC_ERR_UNSUPPORTED, "mlp_sample: d = %lld with a diagonal mass does not fit one CTA's shared memory", (long long)P.d);
    a.A.inv_mass = io->inv_mass;
  }
  pick_geometry(P, C, a);
  a.A.cfg = *cfg; a.A.C = C; a.A.q0 = q0; a.A.samples = samples;
  if (io != nullptr) {
    a.A.accepted = io->accepted; a.A.hamiltonians = io->hamiltonians; a.A.logp_out = io->logp; a.A.step_sizes = io->step_sizes;
    a.A.inj_p = io->inject_momenta; a.A.inj_u = io->inject_uniforms;
    a.A.vi_sigma = io->vi_sigma; a.A.vi_params = io->vi_params; a.A.inj_vi = io->inject_vi_normals;
    if (io->vi_sigma != nullptr && prob->frozen == nullptr)
      return fail(VIHMC_ERR_INVALID, "the VI redraw needs the variational means (prob->frozen) and sens_ind");
  }
  return dispatch(W, kOpSample, P, a, st);
}

}  // namespace vihmc
