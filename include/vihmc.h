/*
 * vihmc.h -- C ABI of libvihmc.so, the B200 (sm_100a) engine for the VI-HMC hot path.
 *
 * The reference (ponkrshnan/VI-HMC) is pure Python; the interface this library replaces is the
 * Python call boundary between the reference's entry scripts and hamiltorch:
 *
 *   hamiltorch.samplers.sample(log_prob_func, params_init, num_samples, num_steps_per_sample,
 *                              step_size, burn, sampler, integrator, debug)
 *       call sites: Neural_network/VI_HMC/main_VI_HMC.py:379-380
 *                   Operator_network/VI_HMC/main_VI_HMC_burgers.py:286-287
 *                   Operator_network/HMC/main_HMC_splitting.py:362-369
 *                   Operator_network/HMC/NUTS_DeepOnets.py:289-290
 *   hamiltorch.sample_model(...)           Neural_network/HMC/main_regression_hmc.py:124-127
 *   log_prob_func(params) (+ autograd.grad) built by define_model_log_prob:
 *                   Neural_network/VI_HMC/main_VI_HMC.py:28-153
 *                   Operator_network/VI_HMC/main_VI_HMC_burgers.py:27-180
 *                   Operator_network/HMC/main_HMC_splitting.py:79-258
 *
 * Because a CUDA engine cannot call a Python closure once per leapfrog step, the closure is passed
 * as data: a `vihmc_problem` (architecture, training data, prior, likelihood, VI-HMC split).
 *
 * Conventions
 *   - every pointer inside vihmc_problem and every q/p/grad/sample buffer is a DEVICE pointer into
 *     caller-owned memory (fp32 unless stated; indices int64), except in the *_host entry points;
 *   - the library never allocates or frees device memory except inside the *_host entry points;
 *   - all work is enqueued on `stream` (a cudaStream_t passed as void*); no implicit synchronisation;
 *   - return 0 on success, a VIHMC_ERR_* code otherwise; vihmc_last_error() gives the message
 *     (thread-local);
 *   - there is no CPU fallback and no other backend: a device that is not sm_100 is an error.
 *   - chains are rows: q[C,d] row-major; C independent chains are advanced together.
 */
#ifndef VIHMC_H
#define VIHMC_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VIHMC_MAX_LAYERS 16

#if defined(__GNUC__)
#define VIHMC_API __attribute__((visibility("default")))
#else
#define VIHMC_API
#endif

enum vihmc_status {
  VIHMC_OK = 0,
  VIHMC_ERR_INVALID = 1,     /* bad argument / inconsistent descriptor */
  VIHMC_ERR_UNSUPPORTED = 2, /* valid request this build has no kernel for */
  VIHMC_ERR_WORKSPACE = 3,   /* workspace too small */
  VIHMC_ERR_CUDA = 4,        /* a CUDA runtime call failed */
  VIHMC_ERR_DEVICE = 5       /* current device is not sm_100 */
};

enum { VIHMC_MODEL_MLP = 0, VIHMC_MODEL_DEEPONET = 1 };
enum { VIHMC_ACT_TANH = 0, VIHMC_ACT_RELU = 1, VIHMC_ACT_SINE = 2 }; /* my_make_func.py:36-43 */
enum { VIHMC_LOSS_NLL = 0, VIHMC_LOSS_REGRESSION = 1 };              /* main_VI_HMC.py:132-136 */
enum { VIHMC_INTEGRATOR_LEAPFROG = 0, VIHMC_INTEGRATOR_SPLITTING = 1 };

/*
 * The log-posterior "closure" as data.
 *
 * Full weight vector W[D] in torch `model.parameters()` order (util.py:121-136):
 *   MLP      : W0[w0,in] b0[w0] W1[w1,w0] b1[w1] ... Wout[out,w_last] (bout[out] iff last_bias)
 *   DeepONet : b[1] | branch W,b x n_layers_a | trunk W,b x n_layers_b      (model.py:26,33-34)
 * VI-HMC split (my_make_func.py:56-57): W = frozen; W[sens_ind[i]] = q[i], i < d.
 *   frozen == NULL and sens_ind == NULL  <=>  d == D, W = q (plain HMC).
 * logp(q) = loglik(model(W), y) + [ sum_i -0.5 (q_i - mu_i)^2 / sigma_i^2 + prior_log_norm ] / prior_scale
 *   NLL        : loglik = -sum 0.5 (log v + (o-y)^2 / v), v = max(tau_out, 1e-6)  (GaussianNLLLoss)
 *   regression : loglik = -0.5 tau_out sum (o-y)^2
 *   prior_log_norm = sum_i ( -log sigma_i - 0.5 log 2 pi ) over coordinates with finite sigma;
 *   sigma_i = +inf means "no prior on coordinate i" (main_VI_HMC.py:107-112 slice quirk).
 */
typedef struct vihmc_problem {
  int32_t model_kind;                 /* VIHMC_MODEL_* */
  int32_t act;                        /* VIHMC_ACT_* */
  int32_t loss;                       /* VIHMC_LOSS_* */
  int32_t last_bias;                  /* MLP: bias on the output layer (cfg.bias) */
  int32_t impose_bc;                  /* DeepONet: trunk features [t,sin2pix,sin4pix,cos2pix,cos4pix] */
  int32_t n_layers_a;                 /* MLP: number of Linear layers; DeepONet: branch depth */
  int32_t n_layers_b;                 /* DeepONet: trunk depth; MLP: 0 */
  int32_t in_a;                       /* MLP input dim; DeepONet branch input dim (sensors) */
  int32_t in_b;                       /* DeepONet trunk input dim after the feature layer (5) */
  int32_t dims_a[VIHMC_MAX_LAYERS];   /* output width of each Linear of stack a */
  int32_t dims_b[VIHMC_MAX_LAYERS];   /* output width of each Linear of stack b */
  int64_t D;                          /* full parameter count */
  int64_t d;                          /* sampled parameter count */
  int64_t N;                          /* training rows (branch inputs) */
  int64_t P;                          /* DeepONet trunk points; MLP: 1 */
  float tau_out;
  float prior_scale;
  float prior_sigma_scalar;           /* used when prior_sigma == NULL */
  float prior_log_norm;               /* see above; vihmc_prior_log_norm() computes it */
  const float* x;                     /* MLP [N,in_a]; DeepONet branch inputs [N,in_a] */
  const float* x2;                    /* DeepONet trunk coordinates [P,2] (t,x) ([P,in_b] if !impose_bc) */
  const float* y;                     /* MLP [N]; DeepONet [N,P] */
  const float* frozen;                /* [D] or NULL */
  const int64_t* sens_ind;            /* [d] or NULL */
  const float* prior_mu;              /* [d] or NULL (zero) */
  const float* prior_sigma;           /* [d] or NULL (scalar) */
  int64_t frozen_chain_stride;        /* 0: frozen[D] is shared by every chain; D: frozen[C, D], one row per chain (the per-sample
                                         VI redraw, my_make_func.py:45-50: every chain then holds its own draw of the frozen weights) */
} vihmc_problem;

/*
 * Sampler controls == the keyword arguments the reference passes to hamiltorch.samplers.sample.
 * Storage rule restated from hamiltorch: output row 0 is params_init; iteration n (0-based) writes a
 * row only when n > burn, so the output holds num_samples - burn rows.
 */
typedef struct vihmc_sampler_cfg {
  int32_t num_samples;        /* num_samples */
  int32_t num_steps;          /* num_steps_per_sample (cfg.L) */
  int32_t burn;               /* burn */
  int32_t integrator;         /* VIHMC_INTEGRATOR_* (Integrator.SPLITTING needs >= 2 problems) */
  int32_t adapt_step_size;    /* 1 == Sampler.HMC_NUTS: dual averaging while n < burn */
  int32_t hamiltorch_fallback_rule; /* 1: first post-burn reject falls back to params_init (as hamiltorch) */
  float step_size;            /* step_size */
  float desired_accept_rate;  /* 0.8 in hamiltorch */
  uint64_t seed;              /* Philox key */
  int64_t chain_offset;       /* global id of local chain 0: draws are invariant to sharding */
} vihmc_sampler_cfg;

/* Optional per-iteration outputs / injected random streams (any member may be NULL). */
typedef struct vihmc_sampler_io {
  uint8_t* accepted;          /* [num_samples, C] 1 = accepted */
  float* hamiltonians;        /* [num_samples, C, 2] (H0, H1) */
  float* logp;                /* [num_samples - burn, C] log-posterior of each stored row */
  float* step_sizes;          /* [C] in: ignored; out: final (adapted) step size per chain */
  const float* inject_momenta;  /* [num_samples, C, d] replaces the Philox N(0,1) draws */
  const float* inject_uniforms; /* [num_samples, C] replaces the Philox U(0,1) draws */
  /* Per-sample VI redraw -- the reference's `sample_weights` hook (Neural_network/VI_HMC/my_make_func.py:45-50,
   * Operator_network/VI_HMC/my_make_func.py:38-42; trigger main_VI_HMC.py:96-99): at the start of every iteration ALL D frozen
   * weights of every chain are redrawn, W = mu + sigma z with mu = prob->frozen, z ~ N(0,1) from Philox stream 2 (the same draws
   * as vihmc_vi_redraw_philox), and the sampled coordinates are scattered on top.  Enabled by vi_sigma != NULL (needs frozen). */
  const float* vi_sigma;          /* [D] variational standard deviations */
  float* vi_params;               /* [num_samples, C, D] out (optional): the redrawn weight vectors, what the hook appends to vi_params */
  const float* inject_vi_normals; /* [num_samples, C, D] replaces the Philox N(0,1) draws of the redraw */
  /* Diagonal mass matrix (hamiltorch's 1-D inv_mass), shared by all chains.  With m = inv_mass, every product separately
   * rounded: momentum p_i = z_i * sqrt(1 / m_i), kinetic energy 0.5 sum_i p_i (m_i p_i), drift q_i += ((eps m_i) p_i); the
   * kick is unchanged.  Injected momenta are used as p verbatim (inject already-scaled draws).  Entries must be finite and
   * > 0: the library cannot check device data without a synchronisation, so this is the caller's contract.  Dense and
   * per-chain mass matrices are not supported.  m = 1 reproduces the identity run bit for bit. */
  const float* inv_mass;          /* [d] diagonal inverse mass (hamiltorch inv_mass); NULL = identity */
} vihmc_sampler_io;

VIHMC_API const char* vihmc_version(void);
VIHMC_API const char* vihmc_last_error(void);

/* 0 iff the current CUDA device is compute capability 10.x. */
VIHMC_API int vihmc_device_check(void);

/* Host helper: sum_i (-log sigma_i - 0.5 log 2pi) over finite sigma (sigma HOST pointer or NULL). */
VIHMC_API double vihmc_prior_log_norm(const float* sigma_host, int64_t d, float sigma_scalar);

/* Bytes of device workspace vihmc_logp_grad / vihmc_sample need for C chains of this problem. */
VIHMC_API size_t vihmc_workspace_bytes(const vihmc_problem* prob, int64_t C);

/*
 * log-posterior and its gradient for C chains: replaces `log_prob_func(q)` + `autograd.grad`
 * (hamiltorch params_grad; closures at main_VI_HMC.py:96-151, main_VI_HMC_burgers.py:86-178).
 * grad may be NULL (value only, as in hamiltorch's hamiltonian()).  outputs: logp[C], grad[C,d].
 */
VIHMC_API int vihmc_logp_grad(const vihmc_problem* prob, int64_t C, const float* q, float* logp, float* grad,
                    void* workspace, size_t workspace_bytes, void* stream);

/*
 * Model forward only (predict_model, main_VI_HMC.py:156-259): out[C,N] (MLP) or out[C,N,P] (DeepONet)
 * for C parameter vectors q[C,d] on the problem's x/x2.
 */
VIHMC_API int vihmc_predict(const vihmc_problem* prob, int64_t C, const float* q, float* out, void* workspace,
                  size_t workspace_bytes, void* stream);

/*
 * Whole sampling run for a small MLP in ONE persistent kernel launch (one warp per chain; weights,
 * momenta and activations live in shared memory; Philox momenta, both Hamiltonians, the L-step
 * leapfrog trajectory and the Metropolis test are fused).  Replaces hamiltorch.samplers.sample for
 * the BNN configs.  q0[C,d] -> samples[num_samples-burn, C, d].
 */
VIHMC_API int vihmc_mlp_sample(const vihmc_problem* prob, const vihmc_sampler_cfg* cfg, int64_t C, const float* q0,
                     float* samples, const vihmc_sampler_io* io, void* stream);

/*
 * General sampler (any model kind; n_problems >= 2 with VIHMC_INTEGRATOR_SPLITTING sums the
 * closures, main_HMC_splitting.py:209-258): host loop over the building blocks below.
 */
VIHMC_API int vihmc_sample(const vihmc_problem* probs, int32_t n_problems, const vihmc_sampler_cfg* cfg, int64_t C,
                 const float* q0, float* samples, const vihmc_sampler_io* io, void* workspace,
                 size_t workspace_bytes, void* stream);

/* ---- building blocks of the large-d path (all HBM-bound, float4-coalesced) ---- */

/* p[C,d] ~ N(0,1): Philox4x32-10, key = seed, counter = (global chain, iteration, d/4 block, stream 0). */
VIHMC_API int vihmc_momentum_philox(uint64_t seed, int64_t iteration, int64_t chain0, int64_t C, int64_t d, float* p,
                          void* stream);
/* The same draws scaled for a diagonal mass: p[c,i] = z[c,i] * sqrt(1 / inv_mass[i]) (inv_mass: device [d], finite, > 0). */
VIHMC_API int vihmc_momentum_philox_mass(uint64_t seed, int64_t iteration, int64_t chain0, int64_t C, int64_t d,
                               const float* inv_mass, float* p, void* stream);
/* u[C] ~ U(0,1): counter stream 1. */
VIHMC_API int vihmc_uniform_philox(uint64_t seed, int64_t iteration, int64_t chain0, int64_t C, float* u, void* stream);
/* W[C,D] = mu + sigma * N(0,1) (my_make_func.py:45-46 sample_weights), counter stream 2. */
VIHMC_API int vihmc_vi_redraw_philox(uint64_t seed, int64_t iteration, int64_t chain0, int64_t C, int64_t D,
                           const float* mu, const float* sigma, float* W, void* stream);
/* W[C,D] = frozen; W[c, sens_ind[i]] = q[c,i]  (my_make_func.py:56-57). */
VIHMC_API int vihmc_scatter_vi(const float* frozen, const int64_t* sens_ind, const float* q, float* W, int64_t C,
                     int64_t D, int64_t d, void* stream);
/*
 * Fused leapfrog update over [C,d]: p += kick*eps_c*g ; q += drift*eps_c*p ; ke[c] = 0.5 sum p^2.
 * kick/drift are the step fractions (0.5/1/-0.5 and 0/1/...); eps may be per chain (eps_per_chain[C])
 * or a scalar (eps_per_chain == NULL).  ke may be NULL; otherwise ke_scratch must hold
 * C * vihmc_ke_partials(d) floats (per-CTA partial sums, reduced in fixed order: no float atomics, so
 * H and therefore accept/reject are reproducible).
 */
VIHMC_API int64_t vihmc_ke_partials(int64_t d);
/* ke[c] = 0.5 sum_i p[c,i]^2 (hamiltorch hamiltonian(): the kinetic term of the freshly drawn momentum); ke_scratch as above. */
VIHMC_API int vihmc_kinetic_energy(const float* p, int64_t C, int64_t d, float* ke, float* ke_scratch, void* stream);
VIHMC_API int vihmc_leapfrog_update(float* q, float* p, const float* g, float eps, const float* eps_per_chain, float kick,
                          float drift, int64_t C, int64_t d, float* ke, float* ke_scratch, void* stream);
/* Diagonal-mass forms (inv_mass: device [d], finite, > 0, shared by all chains):
 *   ke[c] = 0.5 sum_i p[c,i] (inv_mass[i] p[c,i]);
 *   p += kick*eps_c*g ; q += ((drift*eps_c) inv_mass) p ; ke as above. */
VIHMC_API int vihmc_kinetic_energy_mass(const float* p, const float* inv_mass, int64_t C, int64_t d, float* ke, float* ke_scratch,
                              void* stream);
VIHMC_API int vihmc_leapfrog_update_mass(float* q, float* p, const float* g, const float* inv_mass, float eps,
                               const float* eps_per_chain, float kick, float drift, int64_t C, int64_t d, float* ke,
                               float* ke_scratch, void* stream);
/*
 * Metropolis test + state select: accept_c = isfinite(H0_c,H1_c) && min(0, H0_c - H1_c) >= log(u_c);
 * q_cur[c] = accept ? q_prop[c] : q_fallback[c]; on accept q_fallback[c] = q_prop[c]; when `store`
 * the resulting state is also written to stored_row[c] (hamiltorch's n > burn rule).  The optional
 * logp triple carries the log-posterior of the proposal / fallback / stored row the same way.
 */
VIHMC_API int vihmc_mh_accept(const float* H0, const float* H1, const float* u, const float* q_prop, float* q_cur,
                    float* q_fallback, float* stored_row, int32_t store, uint8_t* accepted, const float* logp_prop,
                    float* logp_fallback, float* logp_row, int64_t C, int64_t d, void* stream);
/* grad_q[c,i] = grad_W[c, sens_ind[i]] (autograd through the index_put at my_make_func.py:57). */
VIHMC_API int vihmc_gather_vi(const int64_t* sens_ind, const float* grad_W, float* grad_q, int64_t C, int64_t D, int64_t d,
                    void* stream);

/*
 * Sensitivity scores of the VI -> HMC split selector (Neural_network/VI/sensitivity.py:71-126, eval_std_dydw / eval_jac):
 *   scores[i] = sigma[i]^2 * mean_n (d o(x_n; w) / d w_i)^2,   n over the prob->N validation inputs prob->x,
 * for the small-MLP family (out_dim 1), evaluated at the full weight vector `weights` (the VI means): prob->d must equal
 * prob->D and prob->frozen / sens_ind must be NULL; prob->y and the prior / likelihood fields are not used.  weights, sigma,
 * scores: device [D].  Workspace: vihmc_mlp_sensitivity_workspace_bytes(prob).
 */
VIHMC_API size_t vihmc_mlp_sensitivity_workspace_bytes(const vihmc_problem* prob);
VIHMC_API int vihmc_mlp_sensitivity(const vihmc_problem* prob, const float* weights, const float* sigma, float* scores,
                          void* workspace, size_t workspace_bytes, void* stream);

/*
 * The same scores for a DeepONet (Operator_network/VI/sensitivity.py:61-126, eval_std_dydw / eval_jac over the functional
 * model my_make_func.py:46-85):
 *   scores[i] = sigma[i]^2 * mean_{n < N, p < P} (d out[n, p] / d w_i)^2
 * over the prob->N validation functions prob->x [N, in_a] and the prob->P trunk points prob->x2 they share.  The Jacobian
 * (N * P * D floats in the reference) is never formed: the sum over p (over n for trunk parameters) is folded into a K x K
 * Gram matrix whose Cholesky rows seed K back-propagations per row (csrc/don_sensitivity.cu).  d == D, frozen / sens_ind
 * NULL, tanh or relu, widths and output neurons <= 128; y, prior and likelihood fields are not used.
 */
VIHMC_API size_t vihmc_deeponet_sensitivity_workspace_bytes(const vihmc_problem* prob);
VIHMC_API int vihmc_deeponet_sensitivity(const vihmc_problem* prob, const float* weights, const float* sigma, float* scores,
                               void* workspace, size_t workspace_bytes, void* stream);

/*
 * Bayes-by-Backprop trainer -- the producer of the VI artefacts (means / stds) the VI-HMC path consumes.
 * Replaces train_model / validate_model / the epoch loop of Neural_network/VI/main_regression_VI.py:75-170,:279-346 and
 * Operator_network/VI/main_VI_deeponet.py:24-118,:130-203 (BBBLinear: W = mu + softplus(rho) * eps, ELBO = Gaussian NLL + beta KL,
 * torch.optim.Adam, ReduceLROnPlateau on the validation loss, best-validation checkpoint).  One optimiser step =
 *   vihmc_vi_draw   W[E, D] = mu + softplus(rho) * eps (Philox, or eps = inject_eps[step] for parity tests)
 *   vihmc_logp_grad on a prior-free problem with C = E and q = the W buffer -> the grad / logp buffers   (the hot-path kernel)
 *   vihmc_vi_step   ELBO gradient w.r.t. (mu, rho), Adam update in place, loss bookkeeping
 * and one epoch ends with vihmc_vi_epoch_end (validation loss from valid_logp[b] = log-likelihood at W = mu on validation batch b,
 * plateau scheduler, history row (train loss, validation loss, learning rate), snapshot of the best (mu, rho)).  Step count, learning
 * rate and scheduler state live in the device workspace: no call synchronises, the sequence can be captured in a CUDA graph.
 * kl_form 0 = the KL the reference actually evaluates (BBBLinear.kl_loss passes (prior, posterior) into calculate_kl(mu_q, sig_q,
 * mu_p, sig_p), i.e. KL(prior || q)); 1 = KL(q || prior).
 */
typedef struct vihmc_vi_cfg {
  int32_t num_ens;            /* E: Monte-Carlo draws per optimiser step (cfg.num_ens) */
  int32_t patience;           /* ReduceLROnPlateau patience (cfg.lr_patience) */
  int32_t kl_form;            /* see above */
  int32_t reserved;
  float lr_start;             /* cfg.lr_start */
  float min_lr;               /* 1e-5 in the reference */
  float lr_factor;            /* 0.1 (torch default) */
  float plateau_threshold;    /* 1e-4, relative (torch default) */
  float beta;                 /* KL weight (cfg.beta_type as a float) */
  float prior_mu, prior_sigma;/* cfg.priors */
  float adam_b1, adam_b2, adam_eps; /* 0.9, 0.999, 1e-8 */
  uint64_t seed;              /* Philox key of the eps draws */
} vihmc_vi_cfg;

VIHMC_API size_t vihmc_vi_workspace_bytes(int64_t D, int32_t num_ens);
/* Device pointers into the workspace: 0 = W[E,D], 1 = grad[E,D], 2 = logp[E], 3 = eps[E,D], 4 = best mu[D], 5 = best rho[D]. */
VIHMC_API void* vihmc_vi_buffer(void* workspace, int64_t D, int32_t num_ens, int32_t which);
VIHMC_API int vihmc_vi_init(const vihmc_vi_cfg* cfg, int64_t D, void* workspace, size_t workspace_bytes, void* stream);
VIHMC_API int vihmc_vi_draw(const vihmc_vi_cfg* cfg, int64_t D, const float* mu, const float* rho, const float* inject_eps,
                  void* workspace, size_t workspace_bytes, void* stream);
VIHMC_API int vihmc_vi_step(const vihmc_vi_cfg* cfg, int64_t D, float nll_scale, float* mu, float* rho, void* workspace,
                  size_t workspace_bytes, void* stream);
VIHMC_API int vihmc_vi_epoch_end(const vihmc_vi_cfg* cfg, int64_t D, const float* valid_logp, int32_t n_valid, float valid_nll_scale,
                       const float* mu, const float* rho, float* history, void* workspace, size_t workspace_bytes, void* stream);

/*
 * The dense path's batched-GEMM building block, exported so that every operand staging mode of the tensor-core
 * kernel can be parity-tested on its own (it replaces the torch.nn.functional.linear / einsum calls of
 * Operator_network/VI_HMC/my_make_func.py:53-79 and the matmuls autograd derives from them):
 *   C[b][m, n] = sum_k opA[b][m, k] * opB[b][k, n],   b < batch
 * with opA[b][m,k] at A + b*a_bs + m*a_sm + k*a_sk, opB[b][k,n] at B + b*b_bs + k*b_sk + n*b_sn and C[b][m,n] at
 * C + b*c_bs + m*ldc + n (element strides, a batch stride of 0 shares the operand).  use_tensor_cores = 1 runs the
 * tcgen05 3xTF32 kernel (needs M >= 32, K >= 16), 0 the FP32 SIMT kernel.  K > 2048 with a non-NULL
 * splitk_scratch (ceil(K/1024) * batch * M * N floats) is split into 1024-deep slices summed in fixed order.
 */
VIHMC_API int vihmc_gemm_batched(const float* A, int64_t a_bs, int64_t a_sm, int64_t a_sk, const float* B, int64_t b_bs,
                       int64_t b_sk, int64_t b_sn, float* C, int64_t c_bs, int64_t ldc, int32_t M, int32_t N, int32_t K,
                       int32_t batch, int32_t use_tensor_cores, float* splitk_scratch, void* stream);

/*
 * Test hook: ONE tcgen05.mma kind::tf32 (M = N = 128, K = 8, FP32 accumulate from zero) whose A / B shared-memory
 * tiles are copied verbatim from two 8 KB device images, with the given descriptor byte strides (leading / stride
 * byte offset), descriptor layout types (0 = no swizzle, 1 = 128B base 32B, 2 = 128B, 4 = 64B, 6 = 32B) and extra
 * instruction-descriptor bits (1<<15: A is MN-major, 1<<16: B is MN-major).  out = D[128,128].
 * Used by the tests to pin the operand layouts the staging code writes against what the tensor core reads.
 */
VIHMC_API int vihmc_debug_umma(const float* a_img, const float* b_img, uint32_t a_lbo, uint32_t a_sbo, uint32_t b_lbo,
                     uint32_t b_sbo, uint32_t a_layout_type, uint32_t b_layout_type, uint32_t idesc_extra, float* out,
                     void* stream);

/*
 * Test hook for the exact-accumulation forward products (csrc/xgemm.cuh): C[b][M,N] = A[b][M,K] B[b][N,K]^T, K <= 112,
 * row-major fp32 operands with row strides lda / ldb.  Builds the three-piece bf16 operand images + row scales in
 * `workspace` (vihmc_debug_xgemm_workspace_bytes) and multiplies them with tcgen05.mma.kind::f16; every accumulation inside
 * the tensor core is exact by construction, so C differs from the exactly-rounded product only by the 2^-24 rounding of the
 * operands and one fp32 rounding of the sum.  The tests pin that property against fp64.
 */
/* Test hook: y[i] = tanh(x[i]) by one of the dense path's implementations (0: MUFU ex2/rcp form of the 3xTF32 kernels, 1: CUDA
 * tanhf, 2: the unbiased Cody-Waite / Taylor form of the exact forward pass); n even. */
VIHMC_API int vihmc_debug_tanh(int32_t kind, const float* x, float* y, int64_t n, void* stream);
VIHMC_API size_t vihmc_debug_xgemm_workspace_bytes(int32_t M, int32_t N, int32_t batch);
VIHMC_API int vihmc_debug_xgemm(const float* A, int64_t lda, const float* B, int64_t ldb, float* C, int64_t ldc, int32_t M,
                      int32_t N, int32_t K, int32_t batch, void* workspace, size_t workspace_bytes, void* stream);

/*
 * Host-buffer convenience entry (everything is a HOST pointer, including those inside prob and io, e.g. io->inv_mass[d]):
 * allocates device memory, copies in, runs vihmc_mlp_sample or vihmc_sample, copies samples/diagnostics out.
 */
VIHMC_API int vihmc_sample_host(const vihmc_problem* probs_host, int32_t n_problems, const vihmc_sampler_cfg* cfg,
                      int64_t C, const float* q0_host, float* samples_host, const vihmc_sampler_io* io_host);

#ifdef __cplusplus
}
#endif
#endif /* VIHMC_H */
