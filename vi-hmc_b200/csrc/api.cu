// C ABI of libvihmc.so (declared in include/vihmc.h): argument validation, dispatch, the general
// host-orchestrated sampler and the host-buffer convenience entry.
//
// The general sampler restates hamiltorch.samplers.sample / leapfrog / hamiltonian (third-party,
// absent -- see oracle/hamiltorch_restated.py for the CPU restatement this is tested against) as a
// stream-ordered sequence of kernel launches with NO host synchronisation inside the loop: accept /
// reject, the fallback bookkeeping and the per-chain step-size adaptation are all device-side.
#include <stdarg.h>

#include <vector>

#include "common.cuh"

namespace vihmc {

// ---- implemented in the other translation units ----
bool mlp_small_supported(const vihmc_problem* p);
int mlp_small_logp_grad(const vihmc_problem*, long long C, const float* q, float* logp, float* grad, cudaStream_t);
int mlp_small_predict(const vihmc_problem*, long long C, const float* q, float* out, cudaStream_t);
size_t mlp_small_sensitivity_workspace(const vihmc_problem*);
int mlp_small_sensitivity(const vihmc_problem*, const float* weights, const float* sigma, float* out, void* ws, size_t ws_bytes,
                          cudaStream_t);
int mlp_small_sample(const vihmc_problem*, const vihmc_sampler_cfg*, long long C, const float* q0, float* samples,
                     const vihmc_sampler_io*, cudaStream_t);
size_t deeponet_sensitivity_workspace(const vihmc_problem*);
int deeponet_sensitivity(const vihmc_problem*, const float* weights, const float* sigma, float* scores, void* ws, size_t ws_bytes,
                         cudaStream_t);
size_t vi_workspace_bytes(long long D, int E);
void* vi_buffer(void* ws, long long D, int E, int which);
int vi_init(const vihmc_vi_cfg*, long long D, void* ws, size_t ws_bytes, cudaStream_t);
int vi_draw(const vihmc_vi_cfg*, long long D, const float* mu, const float* rho, const float* inject_eps, void* ws, size_t ws_bytes,
            cudaStream_t);
int vi_step(const vihmc_vi_cfg*, long long D, float nll_scale, float* mu, float* rho, void* ws, size_t ws_bytes, cudaStream_t);
int vi_epoch_end(const vihmc_vi_cfg*, long long D, const float* valid_logp, int n_valid, float valid_nll_scale, const float* mu,
                 const float* rho, float* history, void* ws, size_t ws_bytes, cudaStream_t);
bool dense_supported(const vihmc_problem* p);
size_t dense_workspace_bytes(const vihmc_problem*, long long C);
int dense_logp_grad(const vihmc_problem*, long long C, const float* q, float* logp, float* grad, void* ws, size_t ws_bytes,
                    cudaStream_t);
int dense_predict(const vihmc_problem*, long long C, const float* q, float* out, void* ws, size_t ws_bytes, cudaStream_t);
int dense_umma_probe(const float* a_img, const float* b_img, unsigned a_lbo, unsigned a_sbo, unsigned b_lbo, unsigned b_sbo,
                     unsigned a_type, unsigned b_type, unsigned idesc_extra, float* out, cudaStream_t);
int dense_debug_tanh(int kind, const float* x, float* y, long long n, cudaStream_t st);
size_t dense_xgemm_workspace(int M, int N, int batch);
int dense_xgemm_debug(const float* A, long long lda, const float* B, long long ldb, float* C, long long ldc, int M, int N, int K,
                      int batch, void* ws, size_t ws_bytes, cudaStream_t st);
int dense_gemm(const float* A, long long a_bs, long long a_sm, long long a_sk, const float* B, long long b_bs, long long b_sk,
               long long b_sn, float* C, long long c_bs, long long ldc, int M, int N, int K, int batch, int use_tc, float* scratch,
               cudaStream_t);
int row_partials(long long d);
int launch_momentum(unsigned long long, long long, long long, long long, long long, const float*, float*, cudaStream_t);
int launch_uniform(unsigned long long, long long, long long, long long, float*, cudaStream_t);
int launch_vi_redraw(unsigned long long, long long, long long, long long, long long, const float*, const float*, float*, cudaStream_t);
int launch_scatter(const float*, const long long*, const float*, float*, long long, long long, long long, cudaStream_t);
int launch_gather(const long long*, const float*, float*, long long, long long, long long, cudaStream_t);
int launch_update(float*, float*, const float*, float, const float*, float, float, long long, long long, const float*, float*,
                  cudaStream_t);
int launch_kinetic(const float*, long long, long long, const float*, float*, cudaStream_t);
int launch_sum_partials(const float*, int, long long, float*, cudaStream_t);
int launch_mh_accept(const float*, const float*, const float*, const float*, float*, float*, float*, int, unsigned char*,
                     const float*, float*, float*, long long, long long, cudaStream_t);

// ---------------------------------------------------------------------------------------------
static thread_local char g_error[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_error, sizeof(g_error), fmt, ap);
  va_end(ap);
}

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_error, sizeof(g_error), fmt, ap);
  va_end(ap);
  return code;
}

static int device_check() {
  int dev = 0;
  VIHMC_CUDA_OK(cudaGetDevice(&dev));
  int major = 0;
  VIHMC_CUDA_OK(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
  if (major != 10) return fail(VIHMC_ERR_DEVICE, "libvihmc is built for sm_100a only; device %d is sm_%d0", dev, major);
  return VIHMC_OK;
}

static int check_problem(const vihmc_problem* p) {
  if (p == nullptr) return fail(VIHMC_ERR_INVALID, "problem is NULL");
  if (p->model_kind != VIHMC_MODEL_MLP && p->model_kind != VIHMC_MODEL_DEEPONET)
    return fail(VIHMC_ERR_INVALID, "unknown model_kind %d", p->model_kind);
  if (p->act < 0 || p->act > VIHMC_ACT_SINE) return fail(VIHMC_ERR_INVALID, "Activation should be relu, sine or tanh");
  if (p->loss != VIHMC_LOSS_NLL && p->loss != VIHMC_LOSS_REGRESSION) return fail(VIHMC_ERR_INVALID, "unknown loss %d", p->loss);
  if (p->n_layers_a < 1 || p->n_layers_a > VIHMC_MAX_LAYERS || p->n_layers_b < 0 || p->n_layers_b > VIHMC_MAX_LAYERS)
    return fail(VIHMC_ERR_INVALID, "layer count out of range");
  if (p->d < 1 || p->D < p->d) return fail(VIHMC_ERR_INVALID, "need 1 <= d <= D");
  return VIHMC_OK;
}

// ---------------------------------------------------------------------------------------------
// small device-side scalar kernels of the general sampler
// ---------------------------------------------------------------------------------------------
__global__ void hamiltonian_kernel(const float* __restrict__ logp, const float* __restrict__ ke, long long C, float* __restrict__ H) {
  const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (c < C) H[c] = -logp[c] + ke[c];
}
__global__ void add_rows_kernel(float* __restrict__ acc, const float* __restrict__ v, long long C, int first) {
  const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (c < C) acc[c] = first ? v[c] : acc[c] + v[c];
}
// W[c, f] = mu[f] + sigma[f] z[c, f] with injected normals (the Philox form is vi_redraw_kernel in elementwise.cu)
__global__ void vi_apply_kernel(const float* __restrict__ mu, const float* __restrict__ sigma, const float* __restrict__ z, long long C,
                                long long D, float* __restrict__ W) {
  const long long total = C * D;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x)
    W[t] = fmaf(__ldg(sigma + t % D), z[t], __ldg(mu + t % D));
}
__global__ void fill_kernel(float* __restrict__ dst, float v, long long n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = v;
}
__global__ void record_h_kernel(const float* __restrict__ H0, const float* __restrict__ H1, long long C, float* __restrict__ out) {
  const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (c < C) {
    out[2 * c] = H0[c];
    out[2 * c + 1] = H1[c];
  }
}
// hamiltorch adaptation() per chain; state = (eps, eps_bar, H_t); n is the 0-based iteration
__global__ void adapt_kernel(const float* __restrict__ H0, const float* __restrict__ H1, long long C, int n, int burn,
                             float eps_init, float desired, float* __restrict__ eps, float* __restrict__ eps_bar,
                             float* __restrict__ Ht) {
  const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  if (n < burn) {
    const float h0 = H0[c], h1 = H1[c];
    const bool finite = isfinite(h0) && isfinite(h1);
    const float rho = fminf(0.0f, h0 - h1);
    const float t = (float)(n + 1);
    const float alpha = finite ? fminf(1.0f, expf(rho)) : 0.0f;
    const float mu = logf(10.0f * eps_init);
    const float ht = (1.0f - 1.0f / (t + 10.0f)) * Ht[c] + (1.0f / (t + 10.0f)) * (desired - alpha);
    const float x_new = mu - sqrtf(t) / 0.05f * ht;
    const float tk = powf(t, -0.75f);
    Ht[c] = ht;
    eps[c] = expf(x_new);
    eps_bar[c] = expf(tk * x_new + (1.0f - tk) * logf(eps_bar[c]));
  }
  if (n == burn) eps[c] = eps_bar[c];
}

static inline int blocks_for(long long n) { return (int)((n + 127) / 128); }

// ---------------------------------------------------------------------------------------------
// workspace carving
// ---------------------------------------------------------------------------------------------
struct Carver {
  char* base;
  size_t off = 0, cap;
  Carver(void* p, size_t c) : base(static_cast<char*>(p)), cap(c) {}
  template <typename T>
  T* take(size_t n) {
    off = (off + 255) / 256 * 256;
    T* r = reinterpret_cast<T*>(base + off);
    off += n * sizeof(T);
    return r;
  }
};

static size_t model_workspace(const vihmc_problem* p, long long C) {
  if (mlp_small_supported(p)) return 0;
  return dense_workspace_bytes(p, C);
}

static size_t sampler_state_bytes(long long C, long long d, long long D_redraw = 0) {
  size_t rows = 5;  // p, g, q_prop, q_cur, q_fb
  size_t bytes = rows * ((size_t)C * d * sizeof(float) + 256);
  bytes += (size_t)C * D_redraw * sizeof(float) + 256;                     // per-chain frozen weights of the VI redraw
  bytes += 16 * ((size_t)C * sizeof(float) + 256);                         // per-chain scalars
  bytes += (size_t)C * row_partials(d) * sizeof(float) + 256;              // ke partials
  return bytes;
}

static int model_logp_grad(const vihmc_problem* p, long long C, const float* q, float* logp, float* grad, void* ws, size_t ws_bytes,
                           cudaStream_t st) {
  if (mlp_small_supported(p)) return mlp_small_logp_grad(p, C, q, logp, grad, st);
  if (dense_supported(p)) return dense_logp_grad(p, C, q, logp, grad, ws, ws_bytes, st);
  return fail(VIHMC_ERR_UNSUPPORTED, "no kernel for this architecture");
}

}  // namespace vihmc

namespace {
struct DeviceArena {
  std::vector<void*> ptrs;
  ~DeviceArena() {
    for (void* p : ptrs) cudaFree(p);
  }
  template <typename T>
  int upload(const T* host, size_t n, const T** out) {
    *out = nullptr;
    if (host == nullptr || n == 0) return VIHMC_OK;
    void* dptr = nullptr;
    VIHMC_CUDA_OK(cudaMalloc(&dptr, n * sizeof(T)));
    ptrs.push_back(dptr);
    VIHMC_CUDA_OK(cudaMemcpy(dptr, host, n * sizeof(T), cudaMemcpyHostToDevice));
    *out = static_cast<const T*>(dptr);
    return VIHMC_OK;
  }
  template <typename T>
  int alloc(size_t n, T** out) {
    void* dptr = nullptr;
    VIHMC_CUDA_OK(cudaMalloc(&dptr, (n ? n : 1) * sizeof(T)));
    ptrs.push_back(dptr);
    *out = static_cast<T*>(dptr);
    return VIHMC_OK;
  }
};
}  // namespace

using namespace vihmc;

// =============================================================================================
// extern "C"
// =============================================================================================
extern "C" {

const char* vihmc_version(void) { return "vihmc 0.2.0 (sm_100a)"; }
const char* vihmc_last_error(void) { return g_error; }
int vihmc_device_check(void) { return device_check(); }

double vihmc_prior_log_norm(const float* sigma_host, int64_t d, float sigma_scalar) {
  const double half_log_2pi = 0.91893853320467274178;
  double s = 0.0;
  for (int64_t i = 0; i < d; ++i) {
    const double sg = sigma_host ? (double)sigma_host[i] : (double)sigma_scalar;
    if (!std::isinf(sg)) s += -log(sg) - half_log_2pi;
  }
  return s;
}

size_t vihmc_workspace_bytes(const vihmc_problem* prob, int64_t C) {
  if (check_problem(prob) != VIHMC_OK || C < 1) return 0;
  return model_workspace(prob, C) + sampler_state_bytes(C, prob->d, prob->frozen != nullptr ? prob->D : 0) + 4096;
}

int vihmc_logp_grad(const vihmc_problem* prob, int64_t C, const float* q, float* logp, float* grad, void* workspace,
                    size_t workspace_bytes, void* stream) {
  if (int rc = check_problem(prob)) return rc;
  if (C < 1 || q == nullptr || logp == nullptr) return fail(VIHMC_ERR_INVALID, "logp_grad: need C >= 1, q and logp");
  if (int rc = device_check()) return rc;
  return model_logp_grad(prob, C, q, logp, grad, workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
}

int vihmc_predict(const vihmc_problem* prob, int64_t C, const float* q, float* out, void* workspace, size_t workspace_bytes,
                  void* stream) {
  if (int rc = check_problem(prob)) return rc;
  if (C < 1 || q == nullptr || out == nullptr) return fail(VIHMC_ERR_INVALID, "predict: need C >= 1, q and out");
  if (int rc = device_check()) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (mlp_small_supported(prob)) return mlp_small_predict(prob, C, q, out, st);
  if (dense_supported(prob)) return dense_predict(prob, C, q, out, workspace, workspace_bytes, st);
  return fail(VIHMC_ERR_UNSUPPORTED, "no kernel for this architecture");
}

static int check_cfg(const vihmc_sampler_cfg* cfg) {
  if (cfg == nullptr) return fail(VIHMC_ERR_INVALID, "sampler cfg is NULL");
  if (cfg->num_samples < 1 || cfg->num_steps < 0) return fail(VIHMC_ERR_INVALID, "num_samples >= 1 and num_steps >= 0 required");
  if (cfg->burn < 0 || cfg->burn >= cfg->num_samples) return fail(VIHMC_ERR_INVALID, "burn must be less than num_samples.");
  if (cfg->adapt_step_size && cfg->burn == 0) return fail(VIHMC_ERR_INVALID, "burn must be greater than 0 for NUTS.");
  if (!(cfg->step_size > 0.0f)) return fail(VIHMC_ERR_INVALID, "step_size must be positive");
  return VIHMC_OK;
}

int vihmc_mlp_sample(const vihmc_problem* prob, const vihmc_sampler_cfg* cfg, int64_t C, const float* q0, float* samples,
                     const vihmc_sampler_io* io, void* stream) {
  if (int rc = check_problem(prob)) return rc;
  if (int rc = check_cfg(cfg)) return rc;
  if (C < 1 || q0 == nullptr || samples == nullptr) return fail(VIHMC_ERR_INVALID, "mlp_sample: need C >= 1, q0 and samples");
  if (cfg->integrator != VIHMC_INTEGRATOR_LEAPFROG)
    return fail(VIHMC_ERR_UNSUPPORTED, "mlp_sample runs the leapfrog integrator only; use vihmc_sample for splitting");
  if (int rc = device_check()) return rc;
  return mlp_small_sample(prob, cfg, C, q0, samples, io, static_cast<cudaStream_t>(stream));
}

int vihmc_sample(const vihmc_problem* probs, int32_t n_problems, const vihmc_sampler_cfg* cfg, int64_t C, const float* q0,
                 float* samples, const vihmc_sampler_io* io, void* workspace, size_t workspace_bytes, void* stream) {
  if (probs == nullptr || n_problems < 1) return fail(VIHMC_ERR_INVALID, "need at least one problem");
  for (int m = 0; m < n_problems; ++m) {
    if (int rc = check_problem(&probs[m])) return rc;
    if (probs[m].d != probs[0].d || probs[m].D != probs[0].D) return fail(VIHMC_ERR_INVALID, "split problems must share d and D");
  }
  if (int rc = check_cfg(cfg)) return rc;
  if (C < 1 || q0 == nullptr || samples == nullptr) return fail(VIHMC_ERR_INVALID, "sample: need C >= 1, q0 and samples");
  if (C > 65535) return fail(VIHMC_ERR_UNSUPPORTED, "sample: more than 65535 chains per call (shard the chains over calls / GPUs)");
  const bool split = cfg->integrator == VIHMC_INTEGRATOR_SPLITTING;
  if (split && n_problems < 2) return fail(VIHMC_ERR_UNSUPPORTED, "splitting needs at least two closures");
  if (!split && n_problems != 1) return fail(VIHMC_ERR_INVALID, "a list of closures requires Integrator.SPLITTING");
  if (int rc = device_check()) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const long long d = probs[0].d;
  const int M = n_problems, S = cfg->num_samples, L = cfg->num_steps, burn = cfg->burn;

  size_t model_ws = 0;
  for (int m = 0; m < M; ++m) {
    const size_t b = model_workspace(&probs[m], C);
    model_ws = b > model_ws ? b : model_ws;
  }
  const bool redraw = io != nullptr && io->vi_sigma != nullptr;
  const float* minv = io != nullptr ? io->inv_mass : nullptr;   // diagonal inverse mass [d], or identity
  const long long Dfull = probs[0].D;
  if (redraw)
    for (int m = 0; m < M; ++m)
      if (probs[m].frozen == nullptr || probs[m].frozen_chain_stride != 0)
        return fail(VIHMC_ERR_INVALID, "the VI redraw needs the shared variational means (prob->frozen[D]) and sens_ind");
  if (workspace_bytes < model_ws + sampler_state_bytes(C, d, redraw ? Dfull : 0) + 4096 || (workspace == nullptr))
    return fail(VIHMC_ERR_WORKSPACE, "workspace too small: have %zu bytes, need %zu", workspace_bytes,
                model_ws + sampler_state_bytes(C, d, redraw ? Dfull : 0) + 4096);
  Carver cv(workspace, workspace_bytes);
  const size_t cd = (size_t)C * d;
  float* p = cv.take<float>(cd);
  float* g = cv.take<float>(cd);
  float* q_prop = cv.take<float>(cd);
  float* q_cur = cv.take<float>(cd);
  float* q_fb = cv.take<float>(cd);
  float* logp = cv.take<float>(C);
  float* logp_part = cv.take<float>(C);
  float* logp_fb = cv.take<float>(C);
  float* logp_init = cv.take<float>(C);
  float* ke = cv.take<float>(C);
  float* H0 = cv.take<float>(C);
  float* H1 = cv.take<float>(C);
  float* u = cv.take<float>(C);
  float* eps = cv.take<float>(C);
  float* eps_bar = cv.take<float>(C);
  float* Ht = cv.take<float>(C);
  const int np = row_partials(d);
  float* ke_part = cv.take<float>((size_t)C * np);
  float* Wred = redraw ? cv.take<float>((size_t)C * Dfull) : nullptr;
  void* mws = cv.take<char>(model_ws);
  // with the redraw every chain evaluates the closures on its own draw of the frozen weights
  vihmc_problem local[16];
  if (M > 16) return fail(VIHMC_ERR_UNSUPPORTED, "more than 16 split closures");
  for (int m = 0; m < M; ++m) {
    local[m] = probs[m];
    if (redraw) { local[m].frozen = Wred; local[m].frozen_chain_stride = Dfull; }
  }
  const float* redraw_mu = probs[0].frozen;   // the variational means (shared by the closures)
  probs = local;
  const int cb = blocks_for(C);

  VIHMC_CUDA_OK(cudaMemcpyAsync(q_cur, q0, cd * sizeof(float), cudaMemcpyDeviceToDevice, st));
  VIHMC_CUDA_OK(cudaMemcpyAsync(q_fb, q0, cd * sizeof(float), cudaMemcpyDeviceToDevice, st));
  VIHMC_CUDA_OK(cudaMemcpyAsync(samples, q0, cd * sizeof(float), cudaMemcpyDeviceToDevice, st));
  fill_kernel<<<cb, 128, 0, st>>>(eps, cfg->step_size, C);
  fill_kernel<<<cb, 128, 0, st>>>(eps_bar, 1.0f, C);
  fill_kernel<<<cb, 128, 0, st>>>(Ht, 0.0f, C);
  VIHMC_LAUNCH_OK("fill_kernel");

  // total log-posterior (sum over the M closures) into `logp`; gradient of closure m into g
  auto total_logp = [&](const float* q) -> int {
    for (int m = 0; m < M; ++m) {
      if (int rc = model_logp_grad(&probs[m], C, q, M == 1 ? logp : logp_part, nullptr, mws, model_ws, st)) return rc;
      if (M > 1) add_rows_kernel<<<cb, 128, 0, st>>>(logp, logp_part, C, m == 0);
    }
    return VIHMC_OK;
  };

  for (int n = 0; n < S; ++n) {
    if (cfg->hamiltorch_fallback_rule && n == burn + 1) {
      VIHMC_CUDA_OK(cudaMemcpyAsync(q_fb, q0, cd * sizeof(float), cudaMemcpyDeviceToDevice, st));
      VIHMC_CUDA_OK(cudaMemcpyAsync(logp_fb, logp_init, C * sizeof(float), cudaMemcpyDeviceToDevice, st));
    }
    if (redraw) {   // my_make_func.py:45-50: all D frozen weights of every chain = mu + sigma z
      if (io->inject_vi_normals != nullptr) {
        vi_apply_kernel<<<blocks_for(C * Dfull), 128, 0, st>>>(redraw_mu, io->vi_sigma, io->inject_vi_normals + (size_t)n * C * Dfull, C, Dfull, Wred);
        VIHMC_LAUNCH_OK("vi_apply_kernel");
      } else if (int rc = launch_vi_redraw(cfg->seed, n, cfg->chain_offset, C, Dfull, redraw_mu, io->vi_sigma, Wred, st)) return rc;
      if (io->vi_params != nullptr)
        VIHMC_CUDA_OK(cudaMemcpyAsync(io->vi_params + (size_t)n * C * Dfull, Wred, (size_t)C * Dfull * sizeof(float), cudaMemcpyDeviceToDevice, st));
    }
    // momentum + its kinetic energy
    if (io != nullptr && io->inject_momenta != nullptr)
      VIHMC_CUDA_OK(cudaMemcpyAsync(p, io->inject_momenta + (size_t)n * cd, cd * sizeof(float), cudaMemcpyDeviceToDevice, st));
    else if (int rc = launch_momentum(cfg->seed, n, cfg->chain_offset, C, d, minv, p, st)) return rc;
    if (int rc = launch_kinetic(p, C, d, minv, ke_part, st)) return rc;
    if (int rc = launch_sum_partials(ke_part, np, C, ke, st)) return rc;
    VIHMC_CUDA_OK(cudaMemcpyAsync(q_prop, q_cur, cd * sizeof(float), cudaMemcpyDeviceToDevice, st));

    if (!split) {
      // leapfrog(): the first gradient evaluation also yields logp(q) for H0 (hamiltorch evaluates it twice)
      if (int rc = model_logp_grad(&probs[0], C, q_prop, logp, g, mws, model_ws, st)) return rc;
      hamiltonian_kernel<<<cb, 128, 0, st>>>(logp, ke, C, H0);
      if (n == 0) {
        VIHMC_CUDA_OK(cudaMemcpyAsync(logp_init, logp, C * sizeof(float), cudaMemcpyDeviceToDevice, st));
        VIHMC_CUDA_OK(cudaMemcpyAsync(logp_fb, logp, C * sizeof(float), cudaMemcpyDeviceToDevice, st));
      }
      if (L == 0) {
        VIHMC_CUDA_OK(cudaMemcpyAsync(H1, H0, C * sizeof(float), cudaMemcpyDeviceToDevice, st));
      } else {
        if (int rc = launch_update(q_prop, p, g, cfg->step_size, eps, 0.5f, 1.0f, C, d, minv, nullptr, st)) return rc;
        for (int s = 1; s <= L; ++s) {
          if (int rc = model_logp_grad(&probs[0], C, q_prop, logp, g, mws, model_ws, st)) return rc;
          if (int rc = launch_update(q_prop, p, g, cfg->step_size, eps, 1.0f, s < L ? 1.0f : 0.0f, C, d, minv, nullptr, st)) return rc;
        }
        // hamiltorch: ret_momenta[-1] - 0.5 * step_size * p_grad  (separate rounding, kept)
        if (int rc = launch_update(q_prop, p, g, cfg->step_size, eps, -0.5f, 0.0f, C, d, minv, ke_part, st)) return rc;
        if (int rc = launch_sum_partials(ke_part, np, C, ke, st)) return rc;
        hamiltonian_kernel<<<cb, 128, 0, st>>>(logp, ke, C, H1);
      }
    } else {
      if (int rc = total_logp(q_prop)) return rc;
      hamiltonian_kernel<<<cb, 128, 0, st>>>(logp, ke, C, H0);
      if (n == 0) {
        VIHMC_CUDA_OK(cudaMemcpyAsync(logp_init, logp, C * sizeof(float), cudaMemcpyDeviceToDevice, st));
        VIHMC_CUDA_OK(cudaMemcpyAsync(logp_fb, logp, C * sizeof(float), cudaMemcpyDeviceToDevice, st));
      }
      const float frac = 1.0f / (float)((M - 1) * 2);
      for (int s = 0; s < L; ++s) {
        for (int m = 0; m < M; ++m) {
          if (int rc = model_logp_grad(&probs[m], C, q_prop, logp_part, g, mws, model_ws, st)) return rc;
          if (int rc = launch_update(q_prop, p, g, cfg->step_size, eps, 0.5f, m < M - 1 ? frac : 0.0f, C, d, minv, nullptr, st)) return rc;
        }
        for (int m = M - 1; m >= 0; --m) {
          if (int rc = model_logp_grad(&probs[m], C, q_prop, logp_part, g, mws, model_ws, st)) return rc;
          if (int rc = launch_update(q_prop, p, g, cfg->step_size, eps, 0.5f, m > 0 ? frac : 0.0f, C, d, minv, nullptr, st)) return rc;
        }
      }
      if (int rc = total_logp(q_prop)) return rc;
      if (int rc = launch_kinetic(p, C, d, minv, ke_part, st)) return rc;
      if (int rc = launch_sum_partials(ke_part, np, C, ke, st)) return rc;
      hamiltonian_kernel<<<cb, 128, 0, st>>>(logp, ke, C, H1);
    }
    VIHMC_LAUNCH_OK("hamiltonian_kernel");

    if (io != nullptr && io->inject_uniforms != nullptr)
      VIHMC_CUDA_OK(cudaMemcpyAsync(u, io->inject_uniforms + (size_t)n * C, C * sizeof(float), cudaMemcpyDeviceToDevice, st));
    else if (int rc = launch_uniform(cfg->seed, n, cfg->chain_offset, C, u, st)) return rc;

    const int store = n > burn;
    float* row = store ? samples + (size_t)(n - burn) * cd : nullptr;
    float* logp_row = (store && io != nullptr && io->logp != nullptr) ? io->logp + (size_t)(n - burn) * C : nullptr;
    if (n == 0 && io != nullptr && io->logp != nullptr)
      VIHMC_CUDA_OK(cudaMemcpyAsync(io->logp, logp_init, C * sizeof(float), cudaMemcpyDeviceToDevice, st));
    if (int rc = launch_mh_accept(H0, H1, u, q_prop, q_cur, q_fb, row, store, io ? (io->accepted ? io->accepted + (size_t)n * C : nullptr) : nullptr,
                                  logp, logp_fb, logp_row, C, d, st))
      return rc;
    if (io != nullptr && io->hamiltonians != nullptr) record_h_kernel<<<cb, 128, 0, st>>>(H0, H1, C, io->hamiltonians + (size_t)n * C * 2);
    if (cfg->adapt_step_size && n <= burn)
      adapt_kernel<<<cb, 128, 0, st>>>(H0, H1, C, n, burn, cfg->step_size, cfg->desired_accept_rate, eps, eps_bar, Ht);
    VIHMC_LAUNCH_OK("sampler scalar kernels");
  }
  if (io != nullptr && io->step_sizes != nullptr)
    VIHMC_CUDA_OK(cudaMemcpyAsync(io->step_sizes, eps, C * sizeof(float), cudaMemcpyDeviceToDevice, st));
  return VIHMC_OK;
}

// ---- building blocks -------------------------------------------------------------------------
int vihmc_momentum_philox(uint64_t seed, int64_t iteration, int64_t chain0, int64_t C, int64_t d, float* p, void* stream) {
  return launch_momentum(seed, iteration, chain0, C, d, nullptr, p, static_cast<cudaStream_t>(stream));
}
int vihmc_momentum_philox_mass(uint64_t seed, int64_t iteration, int64_t chain0, int64_t C, int64_t d, const float* inv_mass, float* p,
                               void* stream) {
  if (inv_mass == nullptr) return fail(VIHMC_ERR_INVALID, "momentum_philox_mass: inv_mass is NULL");
  return launch_momentum(seed, iteration, chain0, C, d, inv_mass, p, static_cast<cudaStream_t>(stream));
}
static int kinetic_energy(const float* p, const float* inv_mass, int64_t C, int64_t d, float* ke, float* ke_scratch, void* stream) {
  if (ke == nullptr) return fail(VIHMC_ERR_INVALID, "kinetic_energy: ke is NULL");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (int rc = launch_kinetic(p, C, d, inv_mass, ke_scratch, st)) return rc;
  return launch_sum_partials(ke_scratch, row_partials(d), C, ke, st);
}
int vihmc_kinetic_energy(const float* p, int64_t C, int64_t d, float* ke, float* ke_scratch, void* stream) {
  return kinetic_energy(p, nullptr, C, d, ke, ke_scratch, stream);
}
int vihmc_kinetic_energy_mass(const float* p, const float* inv_mass, int64_t C, int64_t d, float* ke, float* ke_scratch, void* stream) {
  if (inv_mass == nullptr) return fail(VIHMC_ERR_INVALID, "kinetic_energy_mass: inv_mass is NULL");
  return kinetic_energy(p, inv_mass, C, d, ke, ke_scratch, stream);
}
int vihmc_uniform_philox(uint64_t seed, int64_t iteration, int64_t chain0, int64_t C, float* u, void* stream) {
  return launch_uniform(seed, iteration, chain0, C, u, static_cast<cudaStream_t>(stream));
}
int vihmc_vi_redraw_philox(uint64_t seed, int64_t iteration, int64_t chain0, int64_t C, int64_t D, const float* mu,
                           const float* sigma, float* W, void* stream) {
  return launch_vi_redraw(seed, iteration, chain0, C, D, mu, sigma, W, static_cast<cudaStream_t>(stream));
}
int vihmc_scatter_vi(const float* frozen, const int64_t* sens_ind, const float* q, float* W, int64_t C, int64_t D, int64_t d,
                     void* stream) {
  return launch_scatter(frozen, reinterpret_cast<const long long*>(sens_ind), q, W, C, D, d, static_cast<cudaStream_t>(stream));
}
int vihmc_gather_vi(const int64_t* sens_ind, const float* grad_W, float* grad_q, int64_t C, int64_t D, int64_t d, void* stream) {
  if (!sens_ind || !grad_W || !grad_q || C < 1 || d < 1 || D < d) return fail(VIHMC_ERR_INVALID, "gather_vi: bad arguments");
  return launch_gather(reinterpret_cast<const long long*>(sens_ind), grad_W, grad_q, C, D, d, static_cast<cudaStream_t>(stream));
}
int64_t vihmc_ke_partials(int64_t d) { return row_partials(d); }
static int leapfrog_update(float* q, float* p, const float* g, const float* inv_mass, float eps, const float* eps_per_chain, float kick,
                           float drift, int64_t C, int64_t d, float* ke, float* ke_scratch, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (ke != nullptr && ke_scratch == nullptr) return fail(VIHMC_ERR_INVALID, "leapfrog_update: ke needs ke_scratch");
  if (int rc = launch_update(q, p, g, eps, eps_per_chain, kick, drift, C, d, inv_mass, ke ? ke_scratch : nullptr, st)) return rc;
  if (ke != nullptr) return launch_sum_partials(ke_scratch, row_partials(d), C, ke, st);
  return VIHMC_OK;
}
int vihmc_leapfrog_update(float* q, float* p, const float* g, float eps, const float* eps_per_chain, float kick, float drift,
                          int64_t C, int64_t d, float* ke, float* ke_scratch, void* stream) {
  return leapfrog_update(q, p, g, nullptr, eps, eps_per_chain, kick, drift, C, d, ke, ke_scratch, stream);
}
int vihmc_leapfrog_update_mass(float* q, float* p, const float* g, const float* inv_mass, float eps, const float* eps_per_chain,
                               float kick, float drift, int64_t C, int64_t d, float* ke, float* ke_scratch, void* stream) {
  if (inv_mass == nullptr) return fail(VIHMC_ERR_INVALID, "leapfrog_update_mass: inv_mass is NULL");
  return leapfrog_update(q, p, g, inv_mass, eps, eps_per_chain, kick, drift, C, d, ke, ke_scratch, stream);
}
int vihmc_mh_accept(const float* H0, const float* H1, const float* u, const float* q_prop, float* q_cur, float* q_fallback,
                    float* stored_row, int32_t store, uint8_t* accepted, const float* logp_prop, float* logp_fallback,
                    float* logp_row, int64_t C, int64_t d, void* stream) {
  return launch_mh_accept(H0, H1, u, q_prop, q_cur, q_fallback, stored_row, store, accepted, logp_prop, logp_fallback, logp_row, C,
                          d, static_cast<cudaStream_t>(stream));
}

// ---- host-buffer convenience entry -------------------------------------------------------------

int vihmc_sample_host(const vihmc_problem* probs_host, int32_t n_problems, const vihmc_sampler_cfg* cfg, int64_t C,
                      const float* q0_host, float* samples_host, const vihmc_sampler_io* io_host) {
  if (probs_host == nullptr || n_problems < 1) return fail(VIHMC_ERR_INVALID, "need at least one problem");
  if (int rc = check_cfg(cfg)) return rc;
  if (C < 1 || q0_host == nullptr || samples_host == nullptr) return fail(VIHMC_ERR_INVALID, "sample_host: need C, q0, samples");
  if (int rc = device_check()) return rc;
  DeviceArena arena;
  std::vector<vihmc_problem> dev(probs_host, probs_host + n_problems);
  for (int m = 0; m < n_problems; ++m) {
    const vihmc_problem& h = probs_host[m];
    if (int rc = check_problem(&h)) return rc;
    const bool don = h.model_kind == VIHMC_MODEL_DEEPONET;
    const size_t x2_cols = h.impose_bc ? 2 : (size_t)h.in_b;
    if (int rc = arena.upload(h.x, (size_t)h.N * h.in_a, &dev[m].x)) return rc;
    if (int rc = arena.upload(h.x2, don ? (size_t)h.P * x2_cols : 0, &dev[m].x2)) return rc;
    if (int rc = arena.upload(h.y, (size_t)h.N * (don ? h.P : 1), &dev[m].y)) return rc;
    if (int rc = arena.upload(h.frozen, (size_t)h.D, &dev[m].frozen)) return rc;
    if (int rc = arena.upload(h.sens_ind, h.sens_ind ? (size_t)h.d : 0, &dev[m].sens_ind)) return rc;
    if (int rc = arena.upload(h.prior_mu, (size_t)h.d, &dev[m].prior_mu)) return rc;
    if (int rc = arena.upload(h.prior_sigma, (size_t)h.d, &dev[m].prior_sigma)) return rc;
  }
  const long long d = dev[0].d;
  const size_t cd = (size_t)C * d, rows = (size_t)(cfg->num_samples - cfg->burn), S = (size_t)cfg->num_samples;
  const float* q0 = nullptr;
  if (int rc = arena.upload(q0_host, cd, &q0)) return rc;
  float* samples = nullptr;
  if (int rc = arena.alloc(rows * cd, &samples)) return rc;
  vihmc_sampler_io io{};
  if (io_host != nullptr) {
    if (io_host->accepted && arena.alloc(S * C, &io.accepted)) return VIHMC_ERR_CUDA;
    if (io_host->hamiltonians && arena.alloc(S * C * 2, &io.hamiltonians)) return VIHMC_ERR_CUDA;
    if (io_host->logp && arena.alloc(rows * C, &io.logp)) return VIHMC_ERR_CUDA;
    if (io_host->step_sizes && arena.alloc((size_t)C, &io.step_sizes)) return VIHMC_ERR_CUDA;
    if (int rc = arena.upload(io_host->inject_momenta, io_host->inject_momenta ? S * cd : 0, &io.inject_momenta)) return rc;
    if (int rc = arena.upload(io_host->inject_uniforms, io_host->inject_uniforms ? S * C : 0, &io.inject_uniforms)) return rc;
    if (int rc = arena.upload(io_host->inv_mass, io_host->inv_mass ? (size_t)d : 0, &io.inv_mass)) return rc;
  }
  int rc;
  if (n_problems == 1 && cfg->integrator == VIHMC_INTEGRATOR_LEAPFROG && mlp_small_supported(&dev[0])) {
    rc = vihmc_mlp_sample(&dev[0], cfg, C, q0, samples, &io, nullptr);
  } else {
    size_t ws_bytes = 0;
    for (int m = 0; m < n_problems; ++m) {
      const size_t b = vihmc_workspace_bytes(&dev[m], C);
      ws_bytes = b > ws_bytes ? b : ws_bytes;
    }
    char* ws = nullptr;
    if (int rc2 = arena.alloc(ws_bytes, &ws)) return rc2;
    rc = vihmc_sample(dev.data(), n_problems, cfg, C, q0, samples, &io, ws, ws_bytes, nullptr);
  }
  if (rc != VIHMC_OK) return rc;
  VIHMC_CUDA_OK(cudaStreamSynchronize(nullptr));
  VIHMC_CUDA_OK(cudaMemcpy(samples_host, samples, rows * cd * sizeof(float), cudaMemcpyDeviceToHost));
  if (io_host != nullptr) {
    if (io_host->accepted) VIHMC_CUDA_OK(cudaMemcpy(io_host->accepted, io.accepted, S * C, cudaMemcpyDeviceToHost));
    if (io_host->hamiltonians)
      VIHMC_CUDA_OK(cudaMemcpy(io_host->hamiltonians, io.hamiltonians, S * C * 2 * sizeof(float), cudaMemcpyDeviceToHost));
    if (io_host->logp) VIHMC_CUDA_OK(cudaMemcpy(io_host->logp, io.logp, rows * C * sizeof(float), cudaMemcpyDeviceToHost));
    if (io_host->step_sizes) VIHMC_CUDA_OK(cudaMemcpy(io_host->step_sizes, io.step_sizes, C * sizeof(float), cudaMemcpyDeviceToHost));
  }
  return VIHMC_OK;
}

int vihmc_gemm_batched(const float* A, int64_t a_bs, int64_t a_sm, int64_t a_sk, const float* B, int64_t b_bs, int64_t b_sk,
                       int64_t b_sn, float* C, int64_t c_bs, int64_t ldc, int32_t M, int32_t N, int32_t K, int32_t batch,
                       int32_t use_tensor_cores, float* splitk_scratch, void* stream) {
  if (int rc = device_check()) return rc;
  return dense_gemm(A, a_bs, a_sm, a_sk, B, b_bs, b_sk, b_sn, C, c_bs, ldc, M, N, K, batch, use_tensor_cores, splitk_scratch,
                    static_cast<cudaStream_t>(stream));
}

int vihmc_debug_umma(const float* a_img, const float* b_img, uint32_t a_lbo, uint32_t a_sbo, uint32_t b_lbo, uint32_t b_sbo,
                     uint32_t a_layout_type, uint32_t b_layout_type, uint32_t idesc_extra, float* out, void* stream) {
  if (int rc = device_check()) return rc;
  return dense_umma_probe(a_img, b_img, a_lbo, a_sbo, b_lbo, b_sbo, a_layout_type, b_layout_type, idesc_extra, out,
                          static_cast<cudaStream_t>(stream));
}

int vihmc_debug_tanh(int32_t kind, const float* x, float* y, int64_t n, void* stream) {
  if (int rc = device_check()) return rc;
  return dense_debug_tanh(kind, x, y, n, static_cast<cudaStream_t>(stream));
}

size_t vihmc_debug_xgemm_workspace_bytes(int32_t M, int32_t N, int32_t batch) { return dense_xgemm_workspace(M, N, batch); }

int vihmc_debug_xgemm(const float* A, int64_t lda, const float* B, int64_t ldb, float* C, int64_t ldc, int32_t M, int32_t N, int32_t K,
                      int32_t batch, void* workspace, size_t workspace_bytes, void* stream) {
  if (int rc = device_check()) return rc;
  return dense_xgemm_debug(A, lda, B, ldb, C, ldc, M, N, K, batch, workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
}

size_t vihmc_mlp_sensitivity_workspace_bytes(const vihmc_problem* prob) {
  if (prob == nullptr) return 0;
  return mlp_small_sensitivity_workspace(prob);
}

int vihmc_mlp_sensitivity(const vihmc_problem* prob, const float* weights, const float* sigma, float* scores, void* workspace,
                          size_t workspace_bytes, void* stream) {
  if (int rc = device_check()) return rc;
  if (prob == nullptr) return fail(VIHMC_ERR_INVALID, "sensitivity: null problem");
  if (!mlp_small_supported(prob)) return fail(VIHMC_ERR_UNSUPPORTED, "sensitivity: only the small-MLP family is implemented");
  return mlp_small_sensitivity(prob, weights, sigma, scores, workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
}

size_t vihmc_deeponet_sensitivity_workspace_bytes(const vihmc_problem* prob) {
  if (prob == nullptr) return 0;
  return deeponet_sensitivity_workspace(prob);
}

int vihmc_deeponet_sensitivity(const vihmc_problem* prob, const float* weights, const float* sigma, float* scores, void* workspace,
                               size_t workspace_bytes, void* stream) {
  if (int rc = device_check()) return rc;
  if (prob == nullptr) return fail(VIHMC_ERR_INVALID, "deeponet sensitivity: null problem");
  return deeponet_sensitivity(prob, weights, sigma, scores, workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
}

size_t vihmc_vi_workspace_bytes(int64_t D, int32_t num_ens) { return vi_workspace_bytes(D, num_ens); }

void* vihmc_vi_buffer(void* workspace, int64_t D, int32_t num_ens, int32_t which) {
  if (workspace == nullptr || D < 1 || num_ens < 1) return nullptr;
  return vi_buffer(workspace, D, num_ens, which);
}

int vihmc_vi_init(const vihmc_vi_cfg* cfg, int64_t D, void* workspace, size_t workspace_bytes, void* stream) {
  if (int rc = device_check()) return rc;
  return vi_init(cfg, D, workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
}

int vihmc_vi_draw(const vihmc_vi_cfg* cfg, int64_t D, const float* mu, const float* rho, const float* inject_eps, void* workspace,
                  size_t workspace_bytes, void* stream) {
  return vi_draw(cfg, D, mu, rho, inject_eps, workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
}

int vihmc_vi_step(const vihmc_vi_cfg* cfg, int64_t D, float nll_scale, float* mu, float* rho, void* workspace, size_t workspace_bytes,
                  void* stream) {
  return vi_step(cfg, D, nll_scale, mu, rho, workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
}

int vihmc_vi_epoch_end(const vihmc_vi_cfg* cfg, int64_t D, const float* valid_logp, int32_t n_valid, float valid_nll_scale,
                       const float* mu, const float* rho, float* history, void* workspace, size_t workspace_bytes, void* stream) {
  return vi_epoch_end(cfg, D, valid_logp, n_valid, valid_nll_scale, mu, rho, history, workspace, workspace_bytes,
                      static_cast<cudaStream_t>(stream));
}

}  // extern "C"
