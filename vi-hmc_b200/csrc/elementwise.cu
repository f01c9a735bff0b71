// HBM-bound building blocks of the large-d path: Philox momenta / uniforms / VI redraws, the VI-HMC
// scatter, the fused leapfrog update (+ kinetic energy) and the Metropolis accept / state select.
//
// Restated hamiltorch pieces (third-party, absent; see oracle/hamiltorch_restated.py): gibbs()
// (p ~ N(0,I)), leapfrog()'s `momentum += c*eps*grad; params = params + eps*momentum`, hamiltonian()'s
// 0.5*dot(p,p), and the accept test `min(0, H0-H1) >= log(rand)`.  Reference-owned pieces:
// my_make_func.py:45-46 (sample_weights) and :56-57 (scatter into the VI means).
//
// All kernels stream [C,d] row-major fp32 once: algorithmic traffic is 20 B/coordinate for the
// update (read q,p,g; write q,p), 4 B for a momentum draw, 12 B for a VI redraw.
//
// Diagonal mass (hamiltorch's 1-D inv_mass m[d], shared by all chains): the MASS instantiations of the
// momentum, kinetic and update kernels draw p = z * sqrt(1/m), weight the kinetic energy 0.5 sum p (m p)
// and drift q += ((drift eps) m) p, each product separately rounded.  m is one [d] vector read by scalar
// __ldg: every chain reads the same entries, so it is served from L1/L2 and adds no HBM traffic per chain.
// The identity instantiations (MASS = false) are the unchanged kernels.
#include "common.cuh"

namespace vihmc {

constexpr int kThreads = 256;

static inline int grid_for(long long work_items, int per_block) {
  long long b = (work_items + per_block - 1) / per_block;
  const long long cap = 148LL * 16;  // 16 resident 256-thread CTAs per SM is plenty for a streaming kernel
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (int)b;
}

// ---------------------------------------------------------------------------------------------
// sqrt(fl(1 / m)), both correctly rounded: the momentum scale of hamiltorch's Normal(0, (1 / inv_mass) ** 0.5)
__device__ __forceinline__ float mass_scale(float m) { return __fsqrt_rn(__fdiv_rn(1.0f, m)); }

template <bool MASS>
__global__ void __launch_bounds__(kThreads) momentum_philox_kernel(unsigned long long seed, unsigned int iteration,
                                                                   long long chain0, long long C, long long d,
                                                                   const float* __restrict__ inv_mass, float* __restrict__ p) {
  const long long blocks_per_row = (d + 3) / 4;
  const long long total = C * blocks_per_row;
  const bool vec_ok = (d % 4) == 0;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    const long long c = t / blocks_per_row, j = t % blocks_per_row;
    float4 z = philox_normal4(seed, (unsigned long long)(chain0 + c), iteration, (uint32_t)j, STREAM_MOMENTUM);
    if constexpr (MASS) {
      const long long i = 4 * j;
      z.x = __fmul_rn(z.x, mass_scale(__ldg(inv_mass + i)));
      if (i + 1 < d) z.y = __fmul_rn(z.y, mass_scale(__ldg(inv_mass + i + 1)));
      if (i + 2 < d) z.z = __fmul_rn(z.z, mass_scale(__ldg(inv_mass + i + 2)));
      if (i + 3 < d) z.w = __fmul_rn(z.w, mass_scale(__ldg(inv_mass + i + 3)));
    }
    float* dst = p + c * d + 4 * j;
    if (vec_ok) {
      *reinterpret_cast<float4*>(dst) = z;
    } else {
      const float zz[4] = {z.x, z.y, z.z, z.w};
      for (int k = 0; k < 4; ++k)
        if (4 * j + k < d) dst[k] = zz[k];
    }
  }
}

__global__ void uniform_philox_kernel(unsigned long long seed, unsigned int iteration, long long chain0, long long C,
                                      float* __restrict__ u) {
  const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (c < C) u[c] = philox_uniform(seed, (unsigned long long)(chain0 + c), iteration);
}

__global__ void __launch_bounds__(kThreads) vi_redraw_kernel(unsigned long long seed, unsigned int iteration, long long chain0,
                                                             long long C, long long D, const float* __restrict__ mu,
                                                             const float* __restrict__ sigma, float* __restrict__ W) {
  const long long blocks_per_row = (D + 3) / 4;
  const long long total = C * blocks_per_row;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    const long long c = t / blocks_per_row, j = t % blocks_per_row;
    const float4 z = philox_normal4(seed, (unsigned long long)(chain0 + c), iteration, (uint32_t)j, STREAM_VI_REDRAW);
    const float zz[4] = {z.x, z.y, z.z, z.w};
    for (int k = 0; k < 4; ++k) {
      const long long i = 4 * j + k;
      if (i < D) W[c * D + i] = fmaf(__ldg(sigma + i), zz[k], __ldg(mu + i));
    }
  }
}

// W[c,:] = frozen; W[c, ind[i]] = q[c,i].  Two passes inside one kernel would race, so: every thread
// copies its slice of frozen, then (after a grid-stride pass over d) overwrites the sampled entries.
// ind is sorted ascending (sensitivity.py:231) so the overwrite pass is near-coalesced.
__global__ void __launch_bounds__(kThreads) scatter_fill_kernel(const float* __restrict__ frozen, float* __restrict__ W,
                                                                long long C, long long D) {
  const long long total = C * D;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x)
    W[t] = __ldg(frozen + t % D);
}
__global__ void __launch_bounds__(kThreads) scatter_put_kernel(const long long* __restrict__ ind, const float* __restrict__ q,
                                                               float* __restrict__ W, long long C, long long D, long long d) {
  const long long total = C * d;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    const long long c = t / d, i = t % d;
    W[c * D + __ldg(ind + i)] = q[t];
  }
}
// grad_q[c,i] = grad_W[c, ind[i]]  (autograd through index_put: my_make_func.py:57)
__global__ void __launch_bounds__(kThreads) gather_kernel(const long long* __restrict__ ind, const float* __restrict__ gW,
                                                          float* __restrict__ gq, long long C, long long D, long long d) {
  const long long total = C * d;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    const long long c = t / d, i = t % d;
    gq[t] = gW[c * D + __ldg(ind + i)];
  }
}

// ---------------------------------------------------------------------------------------------
// fused leapfrog update.  grid = (row_blocks, C): each CTA streams a slab of one chain's row, so the
// kinetic energy is a per-CTA tree reduction followed by one atomicAdd per CTA... atomics would make
// H1 (and therefore accept/reject) depend on arrival order, so instead each CTA writes its partial to
// ke_part[c, blockIdx.x] and the accept kernel sums the few partials in fixed order.
// ---------------------------------------------------------------------------------------------
// position of a float pointer inside its 16-byte group (0 = aligned)
__device__ __forceinline__ int align_phase(const float* p) { return (int)((reinterpret_cast<uintptr_t>(p) >> 2) & 3u); }

constexpr int kUpdVec = 4;                 // float4 per thread per iteration
constexpr int kUpdSlab = kThreads * kUpdVec * 4;  // coordinates per CTA

// MASS: q += fl(fl(drift eps) m_i) p and ke += p fl(m_i p).  m is indexed by the coordinate, so its 16-byte phase differs from
// that of q[c*d + i] for odd d; it is therefore NOT part of the phase test below (most chains would fall to the scalar path) and
// is read by four scalar __ldg inside the float4 loop instead.
template <bool MASS>
__global__ void __launch_bounds__(kThreads) leapfrog_update_kernel(float* __restrict__ q, float* __restrict__ p,
                                                                   const float* __restrict__ g, float eps,
                                                                   const float* __restrict__ eps_pc, float kick, float drift,
                                                                   long long d, const float* __restrict__ inv_mass,
                                                                   float* __restrict__ ke_part, int n_part) {
  const long long c = blockIdx.y;
  const float e = eps_pc != nullptr ? __ldg(eps_pc + c) : eps;
  const float ck = kick * e, cd = drift * e;
  const long long row = c * d;
  const long long lo = (long long)blockIdx.x * kUpdSlab;
  const long long hi = lo + kUpdSlab < d ? lo + kUpdSlab : d;
  float ke = 0.0f;
  auto scalar = [&](long long i) {
    const float pv = axpy_unfused(ck, g[row + i], p[row + i]);
    if constexpr (MASS) {
      const float m = __ldg(inv_mass + i);
      if (drift != 0.0f) q[row + i] = axpy_unfused(__fmul_rn(cd, m), pv, q[row + i]);
      ke = fmaf(pv, __fmul_rn(m, pv), ke);
    } else {
      if (drift != 0.0f) q[row + i] = axpy_unfused(cd, pv, q[row + i]);
      ke = fmaf(pv, pv, ke);
    }
    p[row + i] = pv;
  };
  // d is odd for the reference's nets (172 401), so rows start at any alignment: peel to the first 16-byte boundary of
  // this slab, stream float4, finish the tail.  Needs q, p, g to share their alignment phase (else: all scalar).
  const int ph = align_phase(q + row + lo);
  long long a0 = (ph == align_phase(p + row + lo) && ph == align_phase(g + row + lo)) ? lo + ((4 - ph) & 3) : hi;
  if (a0 > hi) a0 = hi;
  const long long hi4 = a0 + ((hi - a0) / 4) * 4;
  for (long long i = lo + threadIdx.x; i < a0; i += kThreads) scalar(i);
  for (long long i = a0 + 4LL * threadIdx.x; i < hi4; i += 4LL * kThreads) {
    float4 qv = *reinterpret_cast<const float4*>(q + row + i);
    float4 pv = *reinterpret_cast<const float4*>(p + row + i);
    const float4 gv = *reinterpret_cast<const float4*>(g + row + i);
    pv.x = axpy_unfused(ck, gv.x, pv.x); pv.y = axpy_unfused(ck, gv.y, pv.y);
    pv.z = axpy_unfused(ck, gv.z, pv.z); pv.w = axpy_unfused(ck, gv.w, pv.w);
    if constexpr (MASS) {
      const float mx = __ldg(inv_mass + i), my = __ldg(inv_mass + i + 1), mz = __ldg(inv_mass + i + 2), mw = __ldg(inv_mass + i + 3);
      if (drift != 0.0f) {
        qv.x = axpy_unfused(__fmul_rn(cd, mx), pv.x, qv.x); qv.y = axpy_unfused(__fmul_rn(cd, my), pv.y, qv.y);
        qv.z = axpy_unfused(__fmul_rn(cd, mz), pv.z, qv.z); qv.w = axpy_unfused(__fmul_rn(cd, mw), pv.w, qv.w);
        *reinterpret_cast<float4*>(q + row + i) = qv;
      }
      *reinterpret_cast<float4*>(p + row + i) = pv;
      ke = fmaf(pv.x, __fmul_rn(mx, pv.x), ke); ke = fmaf(pv.y, __fmul_rn(my, pv.y), ke);
      ke = fmaf(pv.z, __fmul_rn(mz, pv.z), ke); ke = fmaf(pv.w, __fmul_rn(mw, pv.w), ke);
      continue;
    }
    if (drift != 0.0f) {
      qv.x = axpy_unfused(cd, pv.x, qv.x); qv.y = axpy_unfused(cd, pv.y, qv.y);
      qv.z = axpy_unfused(cd, pv.z, qv.z); qv.w = axpy_unfused(cd, pv.w, qv.w);
      *reinterpret_cast<float4*>(q + row + i) = qv;
    }
    *reinterpret_cast<float4*>(p + row + i) = pv;
    ke = fmaf(pv.x, pv.x, ke); ke = fmaf(pv.y, pv.y, ke); ke = fmaf(pv.z, pv.z, ke); ke = fmaf(pv.w, pv.w, ke);
  }
  for (long long i = hi4 + threadIdx.x; i < hi; i += kThreads) scalar(i);
  if (ke_part != nullptr) {
    __shared__ float red[kThreads / 32];
    ke = warp_sum(ke);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = ke;
    __syncthreads();
    if (threadIdx.x == 0) {
      float s = 0.0f;
      for (int w = 0; w < kThreads / 32; ++w) s += red[w];
      ke_part[c * n_part + blockIdx.x] = 0.5f * s;
    }
  }
}

__global__ void sum_partials_kernel(const float* __restrict__ part, int n_part, long long C, float* __restrict__ out) {
  const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  float s = 0.0f;
  for (int i = 0; i < n_part; ++i) s += part[c * n_part + i];
  out[c] = s;
}

// kinetic energy of a fresh momentum (no update): same partial layout; MASS: 0.5 sum_i p_i fl(m_i p_i)
template <bool MASS>
__global__ void __launch_bounds__(kThreads) kinetic_kernel(const float* __restrict__ p, long long d,
                                                           const float* __restrict__ inv_mass, float* __restrict__ ke_part,
                                                           int n_part) {
  const long long c = blockIdx.y, row = c * d;
  const long long lo = (long long)blockIdx.x * kUpdSlab;
  const long long hi = lo + kUpdSlab < d ? lo + kUpdSlab : d;
  float ke = 0.0f;
  for (long long i = lo + threadIdx.x; i < hi; i += kThreads) {
    if constexpr (MASS) ke = fmaf(p[row + i], __fmul_rn(__ldg(inv_mass + i), p[row + i]), ke);
    else ke = fmaf(p[row + i], p[row + i], ke);
  }
  __shared__ float red[kThreads / 32];
  ke = warp_sum(ke);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = ke;
  __syncthreads();
  if (threadIdx.x == 0) {
    float s = 0.0f;
    for (int w = 0; w < kThreads / 32; ++w) s += red[w];
    ke_part[c * n_part + blockIdx.x] = 0.5f * s;
  }
}

// ---------------------------------------------------------------------------------------------
// Metropolis accept + state select.  grid = (row_blocks, C).
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) mh_accept_kernel(const float* __restrict__ H0, const float* __restrict__ H1,
                                                             const float* __restrict__ u, const float* __restrict__ q_prop,
                                                             float* __restrict__ q_cur, float* __restrict__ q_fb,
                                                             float* __restrict__ stored, int store,
                                                             unsigned char* __restrict__ accepted,
                                                             const float* __restrict__ logp_prop, float* __restrict__ logp_fb,
                                                             float* __restrict__ logp_row, long long d) {
  const long long c = blockIdx.y, row = c * d;
  const float h0 = __ldg(H0 + c), h1 = __ldg(H1 + c);
  const bool acc = isfinite(h0) && isfinite(h1) && (fminf(0.0f, h0 - h1) >= logf(__ldg(u + c)));
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    if (accepted != nullptr) accepted[c] = acc ? 1 : 0;
    if (logp_fb != nullptr) {
      const float lp = acc ? logp_prop[c] : logp_fb[c];
      logp_fb[c] = lp;
      if (store && logp_row != nullptr) logp_row[c] = lp;
    }
  }
  const long long lo = (long long)blockIdx.x * kUpdSlab;
  const long long hi = lo + kUpdSlab < d ? lo + kUpdSlab : d;
  const float* __restrict__ src = acc ? q_prop : q_fb;   // accepted: proposal -> current, fallback, stored; rejected: fallback -> ...
  auto scalar = [&](long long i) {
    const float v = src[row + i];
    q_cur[row + i] = v;
    if (acc) q_fb[row + i] = v;
    if (store) stored[row + i] = v;
  };
  const int ph = align_phase(src + row + lo);
  const bool same = ph == align_phase(q_cur + row + lo) && (!acc || ph == align_phase(q_fb + row + lo)) &&
                    (!store || ph == align_phase(stored + row + lo));
  long long a0 = same ? lo + ((4 - ph) & 3) : hi;
  if (a0 > hi) a0 = hi;
  const long long hi4 = a0 + ((hi - a0) / 4) * 4;
  for (long long i = lo + threadIdx.x; i < a0; i += kThreads) scalar(i);
  for (long long i = a0 + 4LL * threadIdx.x; i < hi4; i += 4LL * kThreads) {
    const float4 v = *reinterpret_cast<const float4*>(src + row + i);
    *reinterpret_cast<float4*>(q_cur + row + i) = v;
    if (acc) *reinterpret_cast<float4*>(q_fb + row + i) = v;
    if (store) *reinterpret_cast<float4*>(stored + row + i) = v;
  }
  for (long long i = hi4 + threadIdx.x; i < hi; i += kThreads) scalar(i);
}

// ---------------------------------------------------------------------------------------------
// host wrappers (C ABI bodies live in api.cu)
// ---------------------------------------------------------------------------------------------
int row_partials(long long d) { return (int)((d + kUpdSlab - 1) / kUpdSlab); }

// inv_mass: [d] diagonal inverse mass, or nullptr (identity)
int launch_momentum(unsigned long long seed, long long iteration, long long chain0, long long C, long long d, const float* inv_mass,
                    float* p, cudaStream_t st) {
  if (C < 1 || d < 1 || p == nullptr) return fail(VIHMC_ERR_INVALID, "momentum_philox: bad arguments");
  const long long items = C * ((d + 3) / 4);
  if (inv_mass != nullptr)
    momentum_philox_kernel<true><<<grid_for(items, kThreads), kThreads, 0, st>>>(seed, (unsigned int)iteration, chain0, C, d, inv_mass, p);
  else
    momentum_philox_kernel<false><<<grid_for(items, kThreads), kThreads, 0, st>>>(seed, (unsigned int)iteration, chain0, C, d, nullptr, p);
  VIHMC_LAUNCH_OK("momentum_philox_kernel");
  return VIHMC_OK;
}

int launch_uniform(unsigned long long seed, long long iteration, long long chain0, long long C, float* u, cudaStream_t st) {
  if (C < 1 || u == nullptr) return fail(VIHMC_ERR_INVALID, "uniform_philox: bad arguments");
  uniform_philox_kernel<<<(int)((C + 127) / 128), 128, 0, st>>>(seed, (unsigned int)iteration, chain0, C, u);
  VIHMC_LAUNCH_OK("uniform_philox_kernel");
  return VIHMC_OK;
}

int launch_vi_redraw(unsigned long long seed, long long iteration, long long chain0, long long C, long long D, const float* mu,
                     const float* sigma, float* W, cudaStream_t st) {
  if (C < 1 || D < 1 || !mu || !sigma || !W) return fail(VIHMC_ERR_INVALID, "vi_redraw_philox: bad arguments");
  vi_redraw_kernel<<<grid_for(C * ((D + 3) / 4), kThreads), kThreads, 0, st>>>(seed, (unsigned int)iteration, chain0, C, D, mu,
                                                                               sigma, W);
  VIHMC_LAUNCH_OK("vi_redraw_kernel");
  return VIHMC_OK;
}

int launch_scatter(const float* frozen, const long long* ind, const float* q, float* W, long long C, long long D, long long d,
                   cudaStream_t st) {
  if (C < 1 || D < 1 || d < 1 || !q || !W) return fail(VIHMC_ERR_INVALID, "scatter_vi: bad arguments");
  if (frozen == nullptr || ind == nullptr) {
    if (d != D) return fail(VIHMC_ERR_INVALID, "scatter_vi: d != D needs frozen and sens_ind");
    VIHMC_CUDA_OK(cudaMemcpyAsync(W, q, sizeof(float) * C * D, cudaMemcpyDeviceToDevice, st));
    return VIHMC_OK;
  }
  scatter_fill_kernel<<<grid_for(C * D, kThreads), kThreads, 0, st>>>(frozen, W, C, D);
  VIHMC_LAUNCH_OK("scatter_fill_kernel");
  scatter_put_kernel<<<grid_for(C * d, kThreads), kThreads, 0, st>>>(ind, q, W, C, D, d);
  VIHMC_LAUNCH_OK("scatter_put_kernel");
  return VIHMC_OK;
}

int launch_gather(const long long* ind, const float* gW, float* gq, long long C, long long D, long long d, cudaStream_t st) {
  gather_kernel<<<grid_for(C * d, kThreads), kThreads, 0, st>>>(ind, gW, gq, C, D, d);
  VIHMC_LAUNCH_OK("gather_kernel");
  return VIHMC_OK;
}

// ke_part may be NULL; otherwise [C, row_partials(d)]
int launch_update(float* q, float* p, const float* g, float eps, const float* eps_pc, float kick, float drift, long long C,
                  long long d, const float* inv_mass, float* ke_part, cudaStream_t st) {
  if (C < 1 || d < 1 || !q || !p || !g) return fail(VIHMC_ERR_INVALID, "leapfrog_update: bad arguments");
  if (C > 65535) return fail(VIHMC_ERR_UNSUPPORTED, "leapfrog_update: more than 65535 chains per call");
  const int np = row_partials(d);
  const dim3 grid(np, (unsigned)C);
  if (inv_mass != nullptr)
    leapfrog_update_kernel<true><<<grid, kThreads, 0, st>>>(q, p, g, eps, eps_pc, kick, drift, d, inv_mass, ke_part, np);
  else
    leapfrog_update_kernel<false><<<grid, kThreads, 0, st>>>(q, p, g, eps, eps_pc, kick, drift, d, nullptr, ke_part, np);
  VIHMC_LAUNCH_OK("leapfrog_update_kernel");
  return VIHMC_OK;
}

int launch_kinetic(const float* p, long long C, long long d, const float* inv_mass, float* ke_part, cudaStream_t st) {
  if (C < 1 || d < 1 || !p || !ke_part) return fail(VIHMC_ERR_INVALID, "kinetic_energy: bad arguments");
  if (C > 65535) return fail(VIHMC_ERR_UNSUPPORTED, "kinetic_energy: more than 65535 chains per call");
  const int np = row_partials(d);
  if (inv_mass != nullptr)
    kinetic_kernel<true><<<dim3(np, (unsigned)C), kThreads, 0, st>>>(p, d, inv_mass, ke_part, np);
  else
    kinetic_kernel<false><<<dim3(np, (unsigned)C), kThreads, 0, st>>>(p, d, nullptr, ke_part, np);
  VIHMC_LAUNCH_OK("kinetic_kernel");
  return VIHMC_OK;
}

int launch_sum_partials(const float* part, int n_part, long long C, float* out, cudaStream_t st) {
  sum_partials_kernel<<<(int)((C + 127) / 128), 128, 0, st>>>(part, n_part, C, out);
  VIHMC_LAUNCH_OK("sum_partials_kernel");
  return VIHMC_OK;
}

int launch_mh_accept(const float* H0, const float* H1, const float* u, const float* q_prop, float* q_cur, float* q_fb,
                     float* stored, int store, unsigned char* accepted, const float* logp_prop, float* logp_fb, float* logp_row,
                     long long C, long long d, cudaStream_t st) {
  if (C < 1 || d < 1 || !H0 || !H1 || !u || !q_prop || !q_cur || !q_fb) return fail(VIHMC_ERR_INVALID, "mh_accept: bad arguments");
  if (store && stored == nullptr) return fail(VIHMC_ERR_INVALID, "mh_accept: store requested without a row");
  if (logp_fb != nullptr && logp_prop == nullptr) return fail(VIHMC_ERR_INVALID, "mh_accept: logp_fallback needs logp_prop");
  if (C > 65535) return fail(VIHMC_ERR_UNSUPPORTED, "mh_accept: more than 65535 chains per call");
  mh_accept_kernel<<<dim3(row_partials(d), (unsigned)C), kThreads, 0, st>>>(H0, H1, u, q_prop, q_cur, q_fb, stored, store, accepted,
                                                                            logp_prop, logp_fb, logp_row, d);
  VIHMC_LAUNCH_OK("mh_accept_kernel");
  return VIHMC_OK;
}

}  // namespace vihmc
