// Small-MLP path (BNN configs): one warp per chain, everything for a chain resident in shared memory.
//
// Replaces, for the BNN configs, hamiltorch's sample()/leapfrog()/hamiltonian() loop around the
// reference closure (Neural_network/VI_HMC/main_VI_HMC.py:96-151 + my_make_func.py:52-73; call sites
// main_VI_HMC.py:379-380 and Neural_network/HMC/main_regression_hmc.py:124-127).
//
// One gradient evaluation for one chain is 14 kFLOP + 400 tanh (1-10-10-1, N=20): far below any UMMA
// tile and with per-chain weights, so this kernel runs on the FP32 pipes and is latency / issue bound,
// not HBM or tensor bound.  v2 mapping (v1 = lane per data point measured 6.9 cycles per instruction,
// dominated by dependent-FMA waits and instruction-cache misses of fully unrolled code):
//   unit mode   lane = (hidden unit j, point group g), G = 32 / W groups, 8 data points per lane.
//               A lane keeps its weight row in registers and accumulates 8 independent dot products
//               (ILP 8 hides FMA / MUFU / shared-memory latency inside one warp); inputs are float4
//               reads of [unit][point] rows that all lanes of a group share (broadcast).  The layer
//               loop is a runtime loop, so the whole evaluation is a few hundred instructions of
//               re-used code.  The backward data pass is the same routine on a transposed weight table.
//   point mode  lane = data point: output layer, residual, likelihood.
//   phase B     lane = sampled coordinate: g_i = sum_n dz[row_i][n] * h[col_i][n] over float4 rows --
//               only the d sampled coordinates are reduced (VI-HMC subset); prior gradient, kick, drift
//               and the scatter of the new q_i into both weight tables are fused into the same pass.
//   The whole num_samples x (L+1) loop, Philox momenta, both Hamiltonians, the Metropolis test,
//   hamiltorch's storage rule and dual averaging run inside ONE launch; HBM sees only the samples.
#pragma once
#include "common.cuh"

namespace vihmc {

constexpr int kMaxHidden = 4;

#ifndef VIHMC_SMALL_MINBLOCKS
#define VIHMC_SMALL_MINBLOCKS 4   // register budget of the small-MLP kernels: 65536 / (128 * minblocks) = 128
#endif
constexpr int kRegRounds = 2;   // FAST == 3: sampled coordinates per lane held in registers (d <= 64)
#ifndef VIHMC_SMALL_MINBLOCKS2
#define VIHMC_SMALL_MINBLOCKS2 2  // eval_fast2 keeps 2 W activation quads in registers: 255 registers per thread
#endif

struct SmallLayout {
  // Per-chain shared memory, in floats from the chain base: [weight tables | activation rows | per-coordinate state].
  // The first two regions depend on (W, n_hidden, in_dim) only, so the specialised kernel gets their offsets as
  // compile-time constants; the per-coordinate arrays (dp = d rounded up to 4 entries each) come last.
  // weight region: row-major [unit][row stride] tables, and for the hidden->hidden layers a transposed copy
  // [input unit][WSW] used by the backward data pass
  int wbase[kMaxHidden + 1], ws[kMaxHidden + 1], bbase[kMaxHidden + 1], tbase[kMaxHidden + 1];
  int w_total;
  // activation region: rows of NCS floats, offsets relative to act_base
  int act_base, xs, h, da, dz, dO, ones, act_total;
  int NC, NCS;
  // per-coordinate state, each dp entries
  int coord_base, dp, q, p, g, qf, pmu, piv, meta, wpos, wposT;
  int part, pmeta;   // specialised path v2: per-lane partial gradient sums [2W+9 slots][33] and each coordinate's offset into them
  int perm;          // v2, register-resident coordinates: coordinate index of (lane, round), 64 entries (-1: none)
  int rot;           // v2: hidden->hidden tables in schedule order (column 2m + h of row j holds unit fast2_unit_at(JP, j % JP, m) + JP h)
  int minv, msq;     // sampler with a diagonal mass only (empty otherwise): inv_mass m_i and sqrt(1 / m_i), dp entries each
  int total;
};

struct SmallParams {
  int act, loss, last_bias, n_hidden, in_dim;
  int widths[kMaxHidden];
  long long D, d, N;
  float tau_out, inv_prior_scale, prior_sigma_scalar, prior_log_norm;
  const float *x, *y, *frozen, *prior_mu, *prior_sigma;
  long long frozen_cs;   // chain stride of `frozen` (0: shared by every chain)
  const long long* sens_ind;
  SmallLayout lay;
};

__host__ __device__ constexpr int round_up(int v, int m) { return (v + m - 1) / m * m; }

// Activation row stride of the specialised path (eval_fast): rows of s = NCS/4 float4 with s odd (phase B reads whole rows of
// different units: 8 rows then sit in 8 different bank groups) and s*jp + nq distinct mod 8 over every quarter warp of the
// lane = (unit pair jp, point quad nq) mapping, so the float4 row stores are conflict-free (found by enumeration).
__host__ __device__ constexpr int fast_ncs(int W) { return W == 10 ? 52 : W == 16 ? 20 : W == 32 ? 12 : ((32 / W) * 8 + 4); }

// Version 2 of the specialised path (eval_fast2): activation rows 64 floats apart, row r shifted by fast2_rowshift floats.
// Its contractions skip the lane's own two rows and read the others on a "spare row" schedule -- step m reads row m - 1,
// except the lane that owns row m - 1, which reads row JP - 1 -- so a quarter warp touches two rows per load.  The shifts
// (16-byte chunks mod 8) make those LDS.128 conflict-free for lane = jp + JP nq; found by enumeration for JP = 5 (the row
// stores then cost 6 wavefronts per 4 quarter warps instead of 4), trivial for JP = 8 (a quarter warp is one point quad).
__host__ __device__ constexpr int fast2_rowshift(int W, int r) {
  const int jp = r % (W / 2);
  return W == 10 ? 4 * (jp == 0 ? 0 : jp == 1 ? 2 : jp == 2 ? 3 : jp == 3 ? 7 : 5) : 4 * (jp % 8);
}
__host__ __device__ constexpr int fast2_rowoff(int W, int r) { return r * 64 + fast2_rowshift(W, r); }
// unit read at step m (m = 0: the lane's own) by the lane owning units jp, jp + JP; and the inverse (column of unit kk)
__host__ __device__ constexpr int fast2_unit_at(int JP, int jp, int m) { return m == 0 ? jp : (m - 1 != jp ? m - 1 : JP - 1); }
__host__ __device__ constexpr int fast2_step_of(int JP, int jp, int kk) { return kk == jp ? 0 : (kk == JP - 1 ? jp + 1 : kk + 1); }

// compile-time proofs of the two properties the version-2 contraction relies on
constexpr bool fast2_schedule_is_a_permutation(int JP) {   // every lane visits every unit once, and step_of inverts unit_at
  for (int jp = 0; jp < JP; ++jp) {
    int seen = 0;
    for (int m = 0; m < JP; ++m) {
      const int u = fast2_unit_at(JP, jp, m);
      if (u < 0 || u >= JP || (seen >> u & 1) || fast2_step_of(JP, jp, u) != m) return false;
      seen |= 1 << u;
    }
  }
  return true;
}
constexpr bool fast2_row_loads_conflict_free(int W) {   // per step and quarter warp: distinct 16-byte chunks hit distinct bank groups
  const int JP = W / 2, NQ = ((32 / W) * 8) / 4;
  for (int m = 1; m < JP; ++m)
    for (int qw = 0; qw < 4; ++qw) {
      int chunk_of_group[8] = {-1, -1, -1, -1, -1, -1, -1, -1};
      for (int ct = 8 * qw; ct < 8 * qw + 8; ++ct) {
        const int jp = ct < JP * NQ ? ct % JP : JP - 1, nq = ct < JP * NQ ? ct / JP : NQ - 1;   // spare lanes mimic the last unit lane
        const int chunk = (fast2_rowoff(W, fast2_unit_at(JP, jp, m)) + 4 * nq) / 4;
        if (chunk_of_group[chunk % 8] >= 0 && chunk_of_group[chunk % 8] != chunk) return false;
        chunk_of_group[chunk % 8] = chunk;
      }
    }
  return true;
}
static_assert(fast2_schedule_is_a_permutation(5) && fast2_schedule_is_a_permutation(8), "spare-row schedule must visit every unit once");
static_assert(fast2_row_loads_conflict_free(10) && fast2_row_loads_conflict_free(16), "row shifts must keep the activation-quad loads conflict-free");

// W = padded hidden width the kernel is compiled for; fast = layout of the specialised 1-W-W-1 tanh path; mass = the sampler's
// diagonal-mass region (appended last, so no other offset moves)
__host__ __device__ constexpr SmallLayout make_layout(int W, int n_hidden, int in_dim, long long d, int fast = 0, bool mass = false) {
  SmallLayout L{};
  const int WSW = round_up(W, 4);
  int off = 0;
  for (int l = 0; l <= n_hidden; ++l) {
    const int rows = l < n_hidden ? W : 1;
    L.ws[l] = l == 0 ? round_up(in_dim, 4) : WSW;
    L.wbase[l] = off;
    off += rows * L.ws[l];
    L.bbase[l] = off;
    off += l < n_hidden ? WSW : 4;
    L.tbase[l] = off;
    if (l >= 1 && l < n_hidden) off += W * WSW;
  }
  L.w_total = off;
  L.NC = (32 / W) * 8;
  L.NCS = fast >= 2 ? 64 : fast ? fast_ncs(W) : L.NC + 4;   // +4: eight different rows land in eight different bank groups
  L.act_base = off;
  int a = 0;
  L.xs = a; a += in_dim * L.NCS;
  L.h = a; a += n_hidden * W * L.NCS;
  L.da = a; a += fast ? 0 : n_hidden * W * L.NCS;   // act'(z) rows: only the sine activation stores them
  L.dz = a; a += n_hidden * W * L.NCS;
  L.dO = a; a += L.NCS;
  L.ones = a; a += L.NCS;
  L.act_total = a;
  off += a;
  L.coord_base = off;
  L.dp = round_up((int)d, 4);
  L.q = off; off += L.dp;
  L.p = off; off += L.dp;
  L.g = off; off += L.dp;
  L.qf = off; off += L.dp;
  L.pmu = off; off += L.dp;
  L.piv = off; off += L.dp;
  L.meta = off; off += L.dp;
  L.wpos = off; off += L.dp;
  L.wposT = off; off += L.dp;
  L.pmeta = off; off += fast ? L.dp : 0;
  L.part = off; off += fast ? (2 * W + 9) * 33 + 3 : 0;
  L.perm = off; off += fast ? 64 : 0;
  L.rot = fast >= 2 ? 1 : 0;
  L.minv = off; off += mass ? L.dp : 0;
  L.msq = off; off += mass ? L.dp : 0;
  L.total = off;
  return L;
}

// full flat index f -> positions in the weight tables and the phase-B row offsets
__device__ __forceinline__ void decode_coord(const SmallParams& P, int W, long long f, int& wpos, int& wposT, int& a_off,
                                             int& b_off) {
  const SmallLayout& L = P.lay;
  const int WSW = (W + 3) / 4 * 4;
  long long base = 0;
  wpos = 0; wposT = -1; a_off = L.dO; b_off = L.ones;
  for (int l = 0; l <= P.n_hidden; ++l) {
    const int out_l = l < P.n_hidden ? P.widths[l] : 1;
    const int in_l = l == 0 ? P.in_dim : P.widths[l - 1];
    const int arow = l < P.n_hidden ? L.dz + l * W * L.NCS : L.dO;
    const long long numel = (long long)out_l * in_l;
    if (f < base + numel) {
      const int j = (int)((f - base) / in_l), k = (int)((f - base) % in_l);
      wpos = L.wbase[l] + j * L.ws[l] + k;
      if (l >= 1 && l < P.n_hidden) wposT = L.tbase[l] + k * WSW + j;
      if (L.rot && l >= 1 && l < P.n_hidden) {
        const int JP = W / 2;
        wpos = L.wbase[l] + j * L.ws[l] + 2 * fast2_step_of(JP, j % JP, k % JP) + k / JP;
        wposT = L.tbase[l] + k * WSW + 2 * fast2_step_of(JP, k % JP, j % JP) + j / JP;
      }
      a_off = arow + (l < P.n_hidden ? j * L.NCS : 0);
      b_off = l == 0 ? L.xs + k * L.NCS : L.h + ((l - 1) * W + k) * L.NCS;
      return;
    }
    base += numel;
    if (l < P.n_hidden || P.last_bias) {
      if (f < base + out_l) {
        const int j = (int)(f - base);
        wpos = L.bbase[l] + j;
        a_off = arow + (l < P.n_hidden ? j * L.NCS : 0);
        b_off = L.ones;
        return;
      }
      base += out_l;
    }
  }
}

// in: z[P] pre-activations; out: z[P] = act(z), da[P] = act'(z)
template <int P>
__device__ __forceinline__ void activate8(int act, float (&z)[P], float (&da)[P]) {
  if (act == VIHMC_ACT_TANH) {
#pragma unroll
    for (int t = 0; t < P; ++t) {
      z[t] = tanh_sel(z[t]);
      da[t] = fmaf(-z[t], z[t], 1.0f);
    }
  } else if (act == VIHMC_ACT_RELU) {
#pragma unroll
    for (int t = 0; t < P; ++t) {
      da[t] = z[t] > 0.0f ? 1.0f : 0.0f;
      z[t] = z[t] > 0.0f ? z[t] : 0.0f;
    }
  } else {
#pragma unroll
    for (int t = 0; t < P; ++t) {
      float s, c;
      sincosf(z[t], &s, &c);
      z[t] = s;
      da[t] = c;
    }
  }
}

// act'(z) of a stored row: tanh and relu recompute it from the activation, sine reads the stored cos(z)
template <int P>
__device__ __forceinline__ void load8(const float* p, float (&v)[P]) {
#pragma unroll
  for (int c = 0; c < P / 4; ++c) {
    const float4 a = *reinterpret_cast<const float4*>(p + 4 * c);
    v[4 * c] = a.x; v[4 * c + 1] = a.y; v[4 * c + 2] = a.z; v[4 * c + 3] = a.w;
  }
}
template <int P>
__device__ __forceinline__ void store8(float* p, const float (&v)[P]) {
#pragma unroll
  for (int c = 0; c < P / 4; ++c) *reinterpret_cast<float4*>(p + 4 * c) = make_float4(v[4 * c], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]);
}

// act'(z) of a stored row: tanh and relu recompute it from the activation, sine reads the stored cos(z)
template <int P>
__device__ __forceinline__ void load_dact8(int act, const float* h_row, const float* da_row, float (&da)[P]) {
  if (act == VIHMC_ACT_SINE) {
    load8(da_row, da);
  } else {
    float h[P];
    load8(h_row, h);
    if (act == VIHMC_ACT_TANH) {
#pragma unroll
      for (int t = 0; t < P; ++t) da[t] = fmaf(-h[t], h[t], 1.0f);
    } else {
#pragma unroll
      for (int t = 0; t < P; ++t) da[t] = h[t] > 0.0f ? 1.0f : 0.0f;
    }
  }
}

// acc[t] += sum_k wrow[k] * rows[k][t], t < 8: the weight row sits in registers, 8 independent chains
template <int W, int NCS, int P>
__device__ __forceinline__ void dot_rows(const float* wrow, const float* rows, float (&acc)[P]) {
  constexpr int WSW = (W + 3) / 4 * 4;
  float w[WSW];
#pragma unroll
  for (int k4 = 0; k4 < WSW / 4; ++k4) {
    const float4 v = reinterpret_cast<const float4*>(wrow)[k4];
    w[4 * k4] = v.x; w[4 * k4 + 1] = v.y; w[4 * k4 + 2] = v.z; w[4 * k4 + 3] = v.w;
  }
#pragma unroll
  for (int k = 0; k < W; ++k) {
    float r[P];
    load8(rows + k * NCS, r);
#pragma unroll
    for (int t = 0; t < P; ++t) acc[t] = fmaf(w[k], r[t], acc[t]);
  }
}

// packed FP32 pairs (Blackwell FFMA2: one instruction, two IEEE fma.rn results -- bit-identical to two fmaf)
__device__ __forceinline__ unsigned long long pack2(float lo, float hi) {
  unsigned long long r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void unpack2(unsigned long long v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ unsigned long long ffma2(unsigned long long a, unsigned long long b, unsigned long long c) {
  unsigned long long d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}

// dot_rows on packed pairs: acc[t] += sum_k wrow[k] * rows[k][t], t < 8 (same order of operations as dot_rows)
template <int W, int NCS>
__device__ __forceinline__ void dot_rows2(const float* wrow, const float* rows, float (&acc)[8]) {
  constexpr int WSW = (W + 3) / 4 * 4;
  float w[WSW];
#pragma unroll
  for (int k4 = 0; k4 < WSW / 4; ++k4) {
    const float4 v = reinterpret_cast<const float4*>(wrow)[k4];
    w[4 * k4] = v.x; w[4 * k4 + 1] = v.y; w[4 * k4 + 2] = v.z; w[4 * k4 + 3] = v.w;
  }
  unsigned long long a[4];
#pragma unroll
  for (int m = 0; m < 4; ++m) a[m] = pack2(acc[2 * m], acc[2 * m + 1]);
#pragma unroll
  for (int k = 0; k < W; ++k) {
    const ulonglong2 r0 = *reinterpret_cast<const ulonglong2*>(rows + k * NCS);
    const ulonglong2 r1 = *reinterpret_cast<const ulonglong2*>(rows + k * NCS + 4);
    const unsigned long long ww = pack2(w[k], w[k]);
    a[0] = ffma2(ww, r0.x, a[0]);
    a[1] = ffma2(ww, r0.y, a[1]);
    a[2] = ffma2(ww, r1.x, a[2]);
    a[3] = ffma2(ww, r1.y, a[3]);
  }
#pragma unroll
  for (int m = 0; m < 4; ++m) unpack2(a[m], acc[2 * m], acc[2 * m + 1]);
}

// ------------------------------------------------------------------------------------------------
// chain-level geometry: one warp per chain, so every phase is warp-synchronous (__syncwarp between phases)
// ------------------------------------------------------------------------------------------------
template <int W>
struct Cfg {
  static constexpr int T = 32;               // threads per chain
  static constexpr int NC = (32 / W) * 8;    // data points per chunk
  static constexpr int NCS = NC + 4;         // activation row stride
  static constexpr int PPL = 8;              // data points per lane in unit mode
  static constexpr int G = NC / PPL;         // point groups
  static constexpr int WSW = (W + 3) / 4 * 4;
  static_assert(G * W <= T, "unit-mode lanes exceed the chain's threads");
};

// point-mode staging of one data chunk: x columns, validity row; returns this thread's target
template <int W>
__device__ __forceinline__ float stage_chunk(float* sm, const SmallParams& P, int ct, int chunk) {
  using C = Cfg<W>;
  const SmallLayout& L = P.lay;
  float* act = sm + L.act_base;
  float yv = 0.0f;
  if (ct < C::NC) {
    const long long n = (long long)chunk * C::NC + ct;
    const bool valid = n < P.N;
    for (int k = 0; k < P.in_dim; ++k) act[L.xs + k * C::NCS + ct] = valid ? __ldg(P.x + n * P.in_dim + k) : 0.0f;
    act[L.ones + ct] = valid ? 1.0f : 0.0f;
    yv = valid ? __ldg(P.y + n) : 0.0f;
  }
  return yv;
}

// One-time per-chain setup: zero the weight tables, load frozen weights, decode coordinates, load
// the prior and q (scattered into the tables).  Returns this thread's target when N fits one chunk.
// MASS (sampler with a diagonal mass): also m_i = inv_mass[i] and s_i = sqrt(fl(1 / m_i)), both correctly rounded.
template <int W, bool MASS = false>
__device__ float chain_init(float* sm, const SmallParams& P, const float* q_row, int ct, long long chain = 0,
                            const float* inv_mass = nullptr) {
  using C = Cfg<W>;
  const SmallLayout& L = P.lay;
  for (int i = ct; i < L.w_total; i += C::T) sm[i] = 0.0f;                 // padded units and weight-row padding stay zero
  for (int i = L.coord_base + ct; i < L.total; i += C::T) sm[i] = 0.0f;
  __syncwarp();
  if (P.frozen != nullptr) {
    for (long long f = ct; f < P.D; f += C::T) {
      int wpos, wposT, a, b;
      decode_coord(P, W, f, wpos, wposT, a, b);
      const float v = __ldg(P.frozen + chain * P.frozen_cs + f);
      sm[wpos] = v;
      if (wposT >= 0) sm[wposT] = v;
    }
  }
  __syncwarp();
  int* meta = reinterpret_cast<int*>(sm + L.meta);
  int* wposv = reinterpret_cast<int*>(sm + L.wpos);
  int* wposTv = reinterpret_cast<int*>(sm + L.wposT);
  for (int i = ct; i < (int)P.d; i += C::T) {
    const long long f = P.sens_ind ? __ldg(P.sens_ind + i) : (long long)i;
    int wpos, wposT, a, b;
    decode_coord(P, W, f, wpos, wposT, a, b);
    meta[i] = (a << 16) | b;
    wposv[i] = wpos;
    wposTv[i] = wposT;
    const float sig = P.prior_sigma ? __ldg(P.prior_sigma + i) : P.prior_sigma_scalar;
    sm[L.piv + i] = isinf(sig) ? 0.0f : 1.0f / (sig * sig);
    sm[L.pmu + i] = P.prior_mu ? __ldg(P.prior_mu + i) : 0.0f;
    if constexpr (MASS) {
      const float m = __ldg(inv_mass + i);
      sm[L.minv + i] = m;
      sm[L.msq + i] = __fsqrt_rn(__fdiv_rn(1.0f, m));
    }
    const float qv = q_row[i];
    sm[L.q + i] = qv;
    sm[L.qf + i] = qv;
    sm[wpos] = qv;
    if (wposT >= 0) sm[wposT] = qv;
  }
  const float yv = stage_chunk<W>(sm, P, ct, 0);
  __syncwarp();
  return yv;
}

// forward pass of the staged chunk; returns the network output of this thread's data point (point mode)
template <int W>
__device__ __forceinline__ float forward_chunk(float* sm, const SmallParams& P, int ct) {
  using C = Cfg<W>;
  constexpr int PPL = C::PPL, NCS = C::NCS, WSW = C::WSW;
  const SmallLayout& L = P.lay;
  float* act = sm + L.act_base;
  const int j = ct % W, c0 = (ct / W) * PPL;
  const bool unit = ct < C::G * W;
  if (unit) {  // layer 0: runtime input width
    float z[PPL], da[PPL];
    const float b = sm[L.bbase[0] + j];
#pragma unroll
    for (int t = 0; t < PPL; ++t) z[t] = b;
    if (P.in_dim == 1) {  // the reference's nets: Linear(1, w0)
      const float w = sm[L.wbase[0] + j * L.ws[0]];
      float r[PPL];
      load8(act + L.xs + c0, r);
#pragma unroll
      for (int t = 0; t < PPL; ++t) z[t] = fmaf(w, r[t], z[t]);
    } else {
#pragma unroll 1
      for (int k = 0; k < P.in_dim; ++k) {
        const float w = sm[L.wbase[0] + j * L.ws[0] + k];
        float r[PPL];
        load8(act + L.xs + k * NCS + c0, r);
#pragma unroll
        for (int t = 0; t < PPL; ++t) z[t] = fmaf(w, r[t], z[t]);
      }
    }
    activate8(P.act, z, da);
    store8(act + L.h + j * NCS + c0, z);
    if (P.act == VIHMC_ACT_SINE) store8(act + L.da + j * NCS + c0, da);
  }
  __syncwarp();
  for (int l = 1; l < P.n_hidden; ++l) {
    if (unit) {
      float z[PPL], da[PPL];
      const float b = sm[L.bbase[l] + j];
#pragma unroll
      for (int t = 0; t < PPL; ++t) z[t] = b;
      dot_rows<W, NCS>(sm + L.wbase[l] + j * WSW, act + L.h + (l - 1) * W * NCS + c0, z);
      activate8(P.act, z, da);
      store8(act + L.h + (l * W + j) * NCS + c0, z);
      if (P.act == VIHMC_ACT_SINE) store8(act + L.da + (l * W + j) * NCS + c0, da);
    }
    __syncwarp();
  }
  float o = 0.0f;
  if (ct < C::NC) {  // output layer, out_dim = 1
    const float* wo = sm + L.wbase[P.n_hidden];
    const float* hl = act + L.h + (P.n_hidden - 1) * W * NCS + ct;
    o = sm[L.bbase[P.n_hidden]];
#pragma unroll
    for (int k = 0; k < W; ++k) o = fmaf(wo[k], hl[k * NCS], o);
  }
  return o;
}

// backward pass: writes the pre-activation gradients dz of every hidden layer (dO is already in smem)
template <int W>
__device__ __forceinline__ void backward_chunk(float* sm, const SmallParams& P, int ct) {
  using C = Cfg<W>;
  constexpr int PPL = C::PPL, NCS = C::NCS, WSW = C::WSW;
  const SmallLayout& L = P.lay;
  float* act = sm + L.act_base;
  const int j = ct % W, c0 = (ct / W) * PPL;
  const bool unit = ct < C::G * W;
  const int top = P.n_hidden - 1;
  if (unit) {
    float dO[PPL], da[PPL], dz[PPL];
    const float wo = sm[L.wbase[P.n_hidden] + j];
    load8(act + L.dO + c0, dO);
    load_dact8(P.act, act + L.h + (top * W + j) * NCS + c0, act + L.da + (top * W + j) * NCS + c0, da);
#pragma unroll
    for (int t = 0; t < PPL; ++t) dz[t] = wo * dO[t] * da[t];
    store8(act + L.dz + (top * W + j) * NCS + c0, dz);
  }
  __syncwarp();
  for (int l = top; l >= 1; --l) {
    if (unit) {
      float acc[PPL], da[PPL];
#pragma unroll
      for (int t = 0; t < PPL; ++t) acc[t] = 0.0f;
      dot_rows<W, NCS>(sm + L.tbase[l] + j * WSW, act + L.dz + l * W * NCS + c0, acc);
      load_dact8(P.act, act + L.h + ((l - 1) * W + j) * NCS + c0, act + L.da + ((l - 1) * W + j) * NCS + c0, da);
#pragma unroll
      for (int t = 0; t < PPL; ++t) acc[t] *= da[t];
      store8(act + L.dz + ((l - 1) * W + j) * NCS + c0, acc);
    }
    __syncwarp();
  }
}

// phase B: thread = sampled coordinate; accumulates d loglik / d q_i of the staged chunk.  On the last
// chunk the finished likelihood gradient of coordinate i goes straight to `consume(i, g_i)` (prior, kick,
// drift, weight-table scatter: one pass, no round trip through sm[g]); earlier chunks park it in sm[g].
template <int W, typename Consume>
__device__ __forceinline__ void phase_b(float* sm, const SmallParams& P, int ct, bool first_chunk, bool last_chunk,
                                        Consume&& consume) {
  using C = Cfg<W>;
  const SmallLayout& L = P.lay;
  const float* act = sm + L.act_base;
  const int* meta = reinterpret_cast<const int*>(sm + L.meta);
  for (int i = ct; i < (int)P.d; i += C::T) {
    const int m = meta[i];
    const float4* A = reinterpret_cast<const float4*>(act + (m >> 16));
    const float4* B = reinterpret_cast<const float4*>(act + (m & 0xffff));
    // two packed accumulators = four independent sums (x, y | z, w lanes of the float4 rows), FFMA2
    unsigned long long acc01 = 0ull, acc23 = 0ull;
#pragma unroll
    for (int c = 0; c < C::NC / 4; ++c) {
      const ulonglong2 a = reinterpret_cast<const ulonglong2*>(A)[c], b = reinterpret_cast<const ulonglong2*>(B)[c];
      acc01 = ffma2(a.x, b.x, acc01);
      acc23 = ffma2(a.y, b.y, acc23);
    }
    float acc0, acc1, acc2, acc3;
    unpack2(acc01, acc0, acc1);
    unpack2(acc23, acc2, acc3);
    float gsum = (acc0 + acc1) + (acc2 + acc3);
    if (!first_chunk) gsum += sm[L.g + i];
    if (last_chunk) consume(i, gsum);
    else sm[L.g + i] = gsum;
  }
}

// One gradient evaluation: consume(i, d loglik / d q_i) is called once per sampled coordinate (no prior
// yet); returns this thread's share of the log-likelihood.  yv0 = the thread's target when N fits one chunk.
template <int W, typename Consume>
__device__ __forceinline__ float eval_likelihood_grad(float* sm, const SmallParams& P, const Likelihood lik, int ct, float yv0,
                                                      Consume&& consume) {
  using C = Cfg<W>;
  const SmallLayout& L = P.lay;
  float* act = sm + L.act_base;
  const int n_chunks = (int)((P.N + C::NC - 1) / C::NC);
  float ll_lane = 0.0f;
  for (int chunk = 0; chunk < n_chunks; ++chunk) {
    float yv = yv0;
    if (n_chunks > 1) {
      yv = stage_chunk<W>(sm, P, ct, chunk);
      __syncwarp();
    }
    const float o = forward_chunk<W>(sm, P, ct);
    if (ct < C::NC) {
      const bool valid = (long long)chunk * C::NC + ct < P.N;
      const float r = o - yv;
      act[L.dO + ct] = valid ? -lik.prec * r : 0.0f;
      if (valid) ll_lane += lik.ll_const - lik.half_prec * r * r;
    }
    __syncwarp();
    backward_chunk<W>(sm, P, ct);
    phase_b<W>(sm, P, ct, chunk == 0, chunk == n_chunks - 1, consume);
    __syncwarp();
  }
  return ll_lane;
}

// ------------------------------------------------------------------------------------------------
// Specialised evaluation for the reference's BNN family (Neural_network/*/config.py: Linear(1,w) - tanh -
// Linear(w,w) - tanh - Linear(w,1), all N data points in one chunk, one warp per chain).  Same arithmetic in the same
// order as eval_likelihood_grad -- results are bit-identical (tested) -- but: weight / activation offsets are
// compile-time constants (the layout of those regions depends on W only), the lane's inputs x and target y never
// change and live in registers, the lane's own activations h0 / h1 stay in registers for the backward pass instead of
// being re-read, and the dot products run on packed FFMA2.
// ------------------------------------------------------------------------------------------------
struct FastRegs {
  float x[4];   // the lane's 4 inputs (unit mode)
  float yv;     // the lane's target (point mode)
  float y4[4];  // the targets of the lane's 4 points (version 2: every lane of a point quad forms the residual)
  int roff[7];  // version 2: activation-row offsets (floats) of the units read at steps m = 1 .. JP - 1 (W <= 16: JP <= 8)
  int own_off;  // version 2: offset of the lane's own first row
};

// Unit-mode lane geometry of the specialised path: lane = (unit pair jp, point quad nq), i.e. a 2 x 4 register tile.
// Per reduction step a lane reads ONE float4 of activations for 8 FMAs (the 1 x 8 tile of the generic path reads two):
// the kernel is bound by shared-memory wavefronts, and an LDS.128 costs four of them however many lanes share its data.
template <int W>
struct FastLane {
  static constexpr int JP = W / 2, NQ = ((32 / W) * 8) / 4;
  static_assert(W % 2 == 0 && JP * NQ <= 32, "unit-mode lanes exceed the warp");
  bool unit;
  int j0, n0;   // the lane's units are j0 and j0 + JP (weight rows 12 floats apart stay conflict-free over consecutive j0)
  // spare lanes mimic the last unit lane: their (ignored) loads then hit the addresses of that lane and add no bank conflicts
  __device__ __forceinline__ explicit FastLane(int ct) : unit(ct < JP * NQ), j0(unit ? ct % JP : JP - 1), n0(unit ? 4 * (ct / JP) : 4 * (NQ - 1)) {}
};

template <int W>
__device__ __forceinline__ void fast_setup(const float* sm, int ct, float yv0, FastRegs& F) {
  constexpr SmallLayout L = make_layout(W, 2, 1, 0, true);
  const FastLane<W> ln(ct);
  load8(sm + L.act_base + L.xs + ln.n0, F.x);
  F.yv = yv0;
#pragma unroll
  for (int t = 0; t < 4; ++t) F.y4[t] = __shfl_sync(0xffffffffu, yv0, (ln.n0 + t) & 31);   // lane n holds the target of point n
#pragma unroll
  for (int m = 1; m < 8; ++m) F.roff[m - 1] = m < W / 2 ? fast2_rowoff(W, fast2_unit_at(W / 2, ln.j0, m)) : 0;
  F.own_off = fast2_rowoff(W, ln.j0);
}

// acc[u][t] += sum_k wrow_u[k] * rows[k][t], u < 2, t < 4, on packed pairs; k ascending as in dot_rows.
// wrows = row of the lane's first unit; the second unit's row is W/2 rows further
template <int W, int NCS>
__device__ __forceinline__ void dot_rows_2x4(const float* wrows, const float* rows, float (&acc)[2][4]) {
  constexpr int WSW = (W + 3) / 4 * 4;
  float w[2][WSW];
#pragma unroll
  for (int u = 0; u < 2; ++u)
#pragma unroll
    for (int k4 = 0; k4 < WSW / 4; ++k4) {
      const float4 v = reinterpret_cast<const float4*>(wrows + u * (W / 2) * WSW)[k4];
      w[u][4 * k4] = v.x; w[u][4 * k4 + 1] = v.y; w[u][4 * k4 + 2] = v.z; w[u][4 * k4 + 3] = v.w;
    }
  unsigned long long a[2][2];
#pragma unroll
  for (int u = 0; u < 2; ++u) {
    a[u][0] = pack2(acc[u][0], acc[u][1]);
    a[u][1] = pack2(acc[u][2], acc[u][3]);
  }
#pragma unroll
  for (int k = 0; k < W; ++k) {
    const ulonglong2 r = *reinterpret_cast<const ulonglong2*>(rows + k * NCS);
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const unsigned long long ww = pack2(w[u][k], w[u][k]);
      a[u][0] = ffma2(ww, r.x, a[u][0]);
      a[u][1] = ffma2(ww, r.y, a[u][1]);
    }
  }
#pragma unroll
  for (int u = 0; u < 2; ++u) {
    unpack2(a[u][0], acc[u][0], acc[u][1]);
    unpack2(a[u][1], acc[u][2], acc[u][3]);
  }
}

template <int W, typename Consume>
__device__ __forceinline__ float eval_fast(float* sm, const SmallParams& P, const Likelihood lik, int ct, const FastRegs& F,
                                           Consume&& consume) {
  constexpr SmallLayout L = make_layout(W, 2, 1, 0, true);
  constexpr int NC = L.NC, NCS = L.NCS, WSW = round_up(W, 4), JP = W / 2;
  float* act = sm + L.act_base;
  const FastLane<W> ln(ct);
  const int j0 = ln.j0, n0 = ln.n0;
  float h0[2][4], h1[2][4];
  {  // layer 0: Linear(1, W)
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const float w = sm[L.wbase[0] + (j0 + u * JP) * L.ws[0]], b = sm[L.bbase[0] + j0 + u * JP];
      // fmaf(w, x, b) and the tanh on packed pairs: the same IEEE operations as the scalar forms, two per instruction
      {
        const unsigned long long w2 = pack_f2(w, w), b2 = pack_f2(b, b);
        unpack_f2(tanh_sel2(fma_f2(w2, pack_f2(F.x[0], F.x[1]), b2)), h0[u][0], h0[u][1]);
        unpack_f2(tanh_sel2(fma_f2(w2, pack_f2(F.x[2], F.x[3]), b2)), h0[u][2], h0[u][3]);
      }
      if (ln.unit) store8(act + L.h + (j0 + u * JP) * NCS + n0, h0[u]);
    }
  }
  __syncwarp();
  {  // layer 1: Linear(W, W)
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const float b = sm[L.bbase[1] + j0 + u * JP];
#pragma unroll
      for (int t = 0; t < 4; ++t) h1[u][t] = b;
    }
    dot_rows_2x4<W, NCS>(sm + L.wbase[1] + j0 * WSW, act + L.h + n0, h1);
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      unpack_f2(tanh_sel2(pack_f2(h1[u][0], h1[u][1])), h1[u][0], h1[u][1]);
      unpack_f2(tanh_sel2(pack_f2(h1[u][2], h1[u][3])), h1[u][2], h1[u][3]);
      if (ln.unit) store8(act + L.h + (W + j0 + u * JP) * NCS + n0, h1[u]);
    }
  }
  __syncwarp();
  float ll_lane = 0.0f;
  if (ct < NC) {  // output layer + Gaussian residual, lane = data point
    const float4* wo4 = reinterpret_cast<const float4*>(sm + L.wbase[2]);   // the output row, padded to WSW floats: three broadcast
    const float* hl = act + L.h + W * NCS + ct;                            // LDS.128 instead of W scalar ones
    float wo[WSW];
#pragma unroll
    for (int k4 = 0; k4 < WSW / 4; ++k4) {
      const float4 v = wo4[k4];
      wo[4 * k4] = v.x; wo[4 * k4 + 1] = v.y; wo[4 * k4 + 2] = v.z; wo[4 * k4 + 3] = v.w;
    }
    float o = sm[L.bbase[2]];
#pragma unroll
    for (int k = 0; k < W; ++k) o = fmaf(wo[k], hl[k * NCS], o);
    const bool valid = ct < P.N;
    const float r = o - F.yv;
    act[L.dO + ct] = valid ? -lik.prec * r : 0.0f;
    if (valid) ll_lane = lik.ll_const - lik.half_prec * r * r;
  }
  __syncwarp();
  {  // backward through the output layer and the second tanh
    float dO[4];
    load8(act + L.dO + n0, dO);
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const float wo = sm[L.wbase[2] + j0 + u * JP];
      float dz[4];
      {  // dz = (wo * dO) * (1 - h1^2), packed: mul = fma(., ., 0) would turn -0 into +0, so the products use mul.rn.f32x2
        const unsigned long long one = pack_f2(1.0f, 1.0f), wo2 = pack_f2(wo, wo);
#pragma unroll
        for (int t = 0; t < 4; t += 2) {
          const unsigned long long h = pack_f2(h1[u][t], h1[u][t + 1]), nh = pack_f2(-h1[u][t], -h1[u][t + 1]);
          unsigned long long p, q;
          asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(p) : "l"(wo2), "l"(pack_f2(dO[t], dO[t + 1])));
          asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(q) : "l"(p), "l"(fma_f2(nh, h, one)));
          unpack_f2(q, dz[t], dz[t + 1]);
        }
      }
      if (ln.unit) store8(act + L.dz + (W + j0 + u * JP) * NCS + n0, dz);
    }
  }
  __syncwarp();
  {  // backward through Linear(W, W) (transposed table) and the first tanh
    float acc[2][4];
#pragma unroll
    for (int u = 0; u < 2; ++u)
#pragma unroll
      for (int t = 0; t < 4; ++t) acc[u][t] = 0.0f;
    dot_rows_2x4<W, NCS>(sm + L.tbase[1] + j0 * WSW, act + L.dz + W * NCS + n0, acc);
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      {
        const unsigned long long one = pack_f2(1.0f, 1.0f);
#pragma unroll
        for (int t = 0; t < 4; t += 2) {
          const unsigned long long h = pack_f2(h0[u][t], h0[u][t + 1]), nh = pack_f2(-h0[u][t], -h0[u][t + 1]);
          unsigned long long q;
          asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(q) : "l"(pack_f2(acc[u][t], acc[u][t + 1])), "l"(fma_f2(nh, h, one)));
          unpack_f2(q, acc[u][t], acc[u][t + 1]);
        }
      }
      if (ln.unit) store8(act + L.dz + (j0 + u * JP) * NCS + n0, acc[u]);
    }
  }
  __syncwarp();
  phase_b<W>(sm, P, ct, true, true, consume);
  __syncwarp();
  return ll_lane;
}


// ------------------------------------------------------------------------------------------------
// Specialised evaluation, version 2 (round 2).  ncu of version 1: shared-memory wavefronts 78 % of the pipe's peak, 303 per
// evaluation -- 128 in the two contractions, ~100 in phase B (lane = coordinate re-reading two 20-point rows per coordinate) and the
// row stores that only phase B needs, ~35 in the output layer (lane = data point).  Version 2 keeps the lane geometry of the
// contractions (2 units x 4 points per lane) and removes the other two:
//   * the activation / gradient quads a lane loads for a contraction STAY in registers, so the lane forms the partial sums of every
//     weight gradient of its two units over its four points in registers (dW1[j][k] += dz1[j][t] h0[k][t], ...): 2W + 9 values;
//   * those go to shared memory once (slot-major, stride 33: conflict-free scalar stores), and the owner lane of a sampled coordinate
//     adds the NQ partials of its coordinate in fixed order (NQ scalar loads instead of two rows);
//   * the output layer is a sum over the JP lanes of a point quad, done with shuffles in fixed order (every lane of the quad gets
//     the same value), so h1 and dz0 are never stored.
// Same operations per element, different summation order than the generic path: equal to rounding, not bit-identical.
// ------------------------------------------------------------------------------------------------
template <int W>
__device__ __forceinline__ int fast2_slot_count() { return 2 * W + 9; }

// offset of coordinate f's partial sums: slot * 33 + jp (the partials of lanes jp + JP nq, nq < NQ, are JP floats apart)
__device__ __forceinline__ int fast2_poff(const SmallParams& P, int W, long long f) {
  const int JP = W / 2, w0 = P.widths[0], w1 = P.widths[1];
  int slot, j;
  if (f < w0) { j = (int)f; slot = 2 * W + 2; }                                   // W0[j][0]
  else if (f < 2 * w0) { j = (int)f - w0; slot = 2 * W + 4; }                     // b0[j]
  else if (f < 2 * w0 + (long long)w1 * w0) {                                     // W1[j][k]
    const int r = (int)f - 2 * w0;
    j = r / w0;
    const int k = r % w0;
    return ((j / JP) * W + 2 * fast2_step_of(JP, j % JP, k % JP) + k / JP) * 33 + j % JP;   // schedule order of the columns (dot_rows_rot)
  }
  else if (f < 2 * w0 + (long long)w1 * w0 + w1) { j = (int)f - 2 * w0 - w1 * w0; slot = 2 * W; }        // b1[j]
  else if (f < 2 * w0 + (long long)w1 * w0 + 2 * w1) { j = (int)f - 2 * w0 - w1 * w0 - w1; slot = 2 * W + 6; }   // W2[0][j]
  else return (2 * W + 8) * 33;                                                   // b2
  return (slot + j / JP) * 33 + j % JP;
}

template <int W>
__device__ __forceinline__ void fast2_setup(float* sm, const SmallParams& P, int ct) {
  const SmallLayout& L = P.lay;
  int* pm = reinterpret_cast<int*>(sm + L.pmeta);
  for (int i = ct; i < (int)P.d; i += 32) pm[i] = fast2_poff(P, W, P.sens_ind ? __ldg(P.sens_ind + i) : (long long)i);
  __syncwarp();
  // Register-resident coordinates (d <= 64): which coordinates share a ROUND decides the bank conflicts of the partial-sum
  // loads (all lanes of a round read part[pm + nq JP] together; bank = pm mod 32).  Greedy split into two rounds: a coordinate
  // goes to the round that holds fewer coordinates of its bank (then the emptier round).  ncu before: 3.5 wavefronts per load.
  int* perm = reinterpret_cast<int*>(sm + L.perm);
  for (int i = ct; i < 64; i += 32) perm[i] = -1;
  __syncwarp();
  if (ct == 0 && P.d <= 64) {
    int* cnt = reinterpret_cast<int*>(sm + L.part);   // scratch: [2][32] coordinates of bank b in round r (part[] is free until the first evaluation)
    for (int i = 0; i < 64; ++i) cnt[i] = 0;
    int n0 = 0, n1 = 0;
    for (int i = 0; i < (int)P.d; ++i) {
      const int b = pm[i] & 31, c0 = cnt[b], c1 = cnt[32 + b];
      const bool to1 = n0 >= 32 || (n1 < 32 && (c1 < c0 || (c1 == c0 && n1 < n0)));
      if (to1) { perm[32 + n1++] = i; cnt[32 + b] = c1 + 1; }
      else { perm[n0++] = i; cnt[b] = c0 + 1; }
    }
  }
  __syncwarp();
}

// acc[u][t] += sum_k' wrow_u[k'] * quad(k')[t] with the schedule order of the v2 tables: column k' = 2m + h of the lane's
// weight rows belongs to unit fast2_unit_at(JP, jp, m) + JP h.  m = 0 are the lane's own two units, whose quads it already holds
// in registers (own[0], own[1]): only the 2 (JP - 1) quads of the other lanes of the point quad are read from shared memory.
// keep[k'] hands all quads back (the operands of the weight-gradient partial sums).
template <int W, int NCS>
__device__ __forceinline__ void dot_rows_rot(const float* wrows, const float* rows, const int (&roff)[7], const ulonglong2 (&own)[2],
                                             float (&acc)[2][4], ulonglong2 (&keep)[W]) {
  constexpr int WSW = (W + 3) / 4 * 4, JP = W / 2;
  float w[2][WSW];
#pragma unroll
  for (int u = 0; u < 2; ++u)
#pragma unroll
    for (int k4 = 0; k4 < WSW / 4; ++k4) {
      const float4 v = reinterpret_cast<const float4*>(wrows + u * JP * WSW)[k4];
      w[u][4 * k4] = v.x; w[u][4 * k4 + 1] = v.y; w[u][4 * k4 + 2] = v.z; w[u][4 * k4 + 3] = v.w;
    }
  keep[0] = own[0];
  keep[1] = own[1];
#pragma unroll
  for (int m = 1; m < JP; ++m)
#pragma unroll
    for (int h = 0; h < 2; ++h) keep[2 * m + h] = *reinterpret_cast<const ulonglong2*>(rows + roff[m - 1] + h * JP * 64);
  // eight independent chains (first / second half of the units x 2 units x 2 point pairs): with ~1.7 warps per scheduler the
  // dependent-issue distance inside one warp decides the FFMA2 rate (ncu: "wait" was the largest stall reason)
  unsigned long long a[2][2], b[2][2];
#pragma unroll
  for (int u = 0; u < 2; ++u) {
    a[u][0] = pack2(acc[u][0], acc[u][1]);
    a[u][1] = pack2(acc[u][2], acc[u][3]);
    b[u][0] = b[u][1] = 0ull;
  }
#pragma unroll
  for (int k = 0; k < W; k += 2) {
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const unsigned long long w0 = pack2(w[u][k], w[u][k]), w1 = pack2(w[u][k + 1], w[u][k + 1]);
      a[u][0] = ffma2(w0, keep[k].x, a[u][0]);
      a[u][1] = ffma2(w0, keep[k].y, a[u][1]);
      b[u][0] = ffma2(w1, keep[k + 1].x, b[u][0]);
      b[u][1] = ffma2(w1, keep[k + 1].y, b[u][1]);
    }
  }
  const unsigned long long one = pack2(1.0f, 1.0f);
#pragma unroll
  for (int u = 0; u < 2; ++u) {
    unpack2(ffma2(one, b[u][0], a[u][0]), acc[u][0], acc[u][1]);
    unpack2(ffma2(one, b[u][1], a[u][1]), acc[u][2], acc[u][3]);
  }
}

// p[i & 3] without branches (the compiler turns a chain of ?: on floats into divergent branches)
__device__ __forceinline__ float select4(int i, const float (&p)[4]) {
  float r;
  asm("{\n\t.reg .pred q0, q1;\n\t.reg .f32 a, b;\n\t"
      "setp.ne.s32 q0, %5, 0;\n\tsetp.ne.s32 q1, %6, 0;\n\t"
      "selp.f32 a, %2, %1, q0;\n\tselp.f32 b, %4, %3, q0;\n\tselp.f32 %0, b, a, q1;\n\t}"
      : "=f"(r)
      : "f"(p[0]), "f"(p[1]), "f"(p[2]), "f"(p[3]), "r"(i & 1), "r"(i & 2));
  return r;
}

// sum over the 4 points of a quad: a . b with a, b packed as (01, 23)
__device__ __forceinline__ float quad_dot(unsigned long long a01, unsigned long long a23, unsigned long long b01, unsigned long long b23) {
  unsigned long long p;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(p) : "l"(a01), "l"(b01));
  p = ffma2(a23, b23, p);
  float lo, hi;
  unpack2(p, lo, hi);
  return lo + hi;
}

// forward, backward and the partial sums; on return (after a warp barrier) part[] holds the partial gradient sums of every lane
template <int W>
__device__ __forceinline__ float eval_fast2_partials(float* sm, const SmallParams& P, const Likelihood lik, int ct, const FastRegs& F) {
  constexpr SmallLayout L0c = make_layout(W, 2, 1, 0, 2);   // weight / activation offsets do not depend on d
  constexpr int NCS = L0c.NCS, WSW = round_up(W, 4), JP = W / 2;
  const SmallLayout& L = P.lay;
  float* act = sm + L0c.act_base;
  const FastLane<W> ln(ct);
  const int j0 = ln.j0, n0 = ln.n0;
  float h0[2][4], h1[2][4];
  {  // layer 0: Linear(1, W)
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const float w = sm[L0c.wbase[0] + (j0 + u * JP) * L0c.ws[0]], b = sm[L0c.bbase[0] + j0 + u * JP];
      const unsigned long long w2 = pack_f2(w, w), b2 = pack_f2(b, b);
      unpack_f2(tanh_sel2(fma_f2(w2, pack_f2(F.x[0], F.x[1]), b2)), h0[u][0], h0[u][1]);
      unpack_f2(tanh_sel2(fma_f2(w2, pack_f2(F.x[2], F.x[3]), b2)), h0[u][2], h0[u][3]);
      if (ln.unit) store8(act + L0c.h + F.own_off + u * JP * 64 + n0, h0[u]);
    }
  }
  __syncwarp();
  ulonglong2 hk[W];   // h0[k][n0 .. n0+3] for every k: the operand of the weight-gradient partial sums
  {  // layer 1: Linear(W, W)
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const float b = sm[L0c.bbase[1] + j0 + u * JP];
#pragma unroll
      for (int t = 0; t < 4; ++t) h1[u][t] = b;
    }
    const ulonglong2 own[2] = {make_ulonglong2(pack_f2(h0[0][0], h0[0][1]), pack_f2(h0[0][2], h0[0][3])),
                               make_ulonglong2(pack_f2(h0[1][0], h0[1][1]), pack_f2(h0[1][2], h0[1][3]))};
    dot_rows_rot<W, NCS>(sm + L0c.wbase[1] + j0 * WSW, act + L0c.h + n0, F.roff, own, h1, hk);
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      unpack_f2(tanh_sel2(pack_f2(h1[u][0], h1[u][1])), h1[u][0], h1[u][1]);
      unpack_f2(tanh_sel2(pack_f2(h1[u][2], h1[u][3])), h1[u][2], h1[u][3]);
    }
  }
  // output layer: o[t] = b2 + sum over the JP lanes of this point quad (lanes nq*JP .. nq*JP + JP-1) of w2[j] h1[j][t], fixed order
  float wo[2], dO[4];
  float ll_lane = 0.0f;
  {
#pragma unroll
    for (int u = 0; u < 2; ++u) wo[u] = sm[L0c.wbase[2] + j0 + u * JP];
    float part[4];
#pragma unroll
    for (int t = 0; t < 4; ++t) part[t] = ln.unit ? fmaf(wo[1], h1[1][t], wo[0] * h1[0][t]) : 0.0f;
    // a shuffle costs a wavefront of the shared-memory pipe like an LDS (tools/probe_shfl_lds.cu), so instead of all-gathering
    // the JP x 4 partials (4 JP shuffles) the quad's lanes reduce-scatter them -- lane jp < 4 collects point jp: JP - 1 shuffles,
    // the sender picks the partial its receiver wants -- and then gather the four totals (4 shuffles).  Fixed order per point.
    const int base = (ct / JP) * JP;
    float tot = select4(j0, part);
#pragma unroll
    for (int r = 1; r < JP; ++r) {
      int si = j0 - r;                       // the lane r places below (cyclically) collects point si
      si += si < 0 ? JP : 0;
      const float send = select4(si, part);
      int src = j0 + r;
      src -= src >= JP ? JP : 0;
      tot += __shfl_sync(0xffffffffu, send, (base + src) & 31);
    }
    float o[4];
    const float b2 = sm[L0c.bbase[2]];
#pragma unroll
    for (int t = 0; t < 4; ++t) o[t] = b2 + __shfl_sync(0xffffffffu, tot, (base + t) & 31);
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const bool valid = ln.unit && n0 + t < (int)P.N;
      const float r = o[t] - F.y4[t];
      dO[t] = valid ? -lik.prec * r : 0.0f;
      if (valid && j0 == 0) ll_lane += lik.ll_const - lik.half_prec * r * r;
    }
  }
  float dz1[2][4], dz0[2][4];
  {  // backward through the output layer and the second tanh; dz1 rows are the operand of the backward contraction
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const unsigned long long one = pack_f2(1.0f, 1.0f), wo2 = pack_f2(wo[u], wo[u]);
#pragma unroll
      for (int t = 0; t < 4; t += 2) {
        const unsigned long long h = pack_f2(h1[u][t], h1[u][t + 1]), nh = pack_f2(-h1[u][t], -h1[u][t + 1]);
        unsigned long long p, q;
        asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(p) : "l"(wo2), "l"(pack_f2(dO[t], dO[t + 1])));
        asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(q) : "l"(p), "l"(fma_f2(nh, h, one)));
        unpack_f2(q, dz1[u][t], dz1[u][t + 1]);
      }
      if (ln.unit) store8(act + L0c.dz + W * NCS + F.own_off + u * JP * 64 + n0, dz1[u]);
    }
  }
  __syncwarp();
  {  // backward through Linear(W, W) (transposed table) and the first tanh
#pragma unroll
    for (int u = 0; u < 2; ++u)
#pragma unroll
      for (int t = 0; t < 4; ++t) dz0[u][t] = 0.0f;
    ulonglong2 zk[W];   // not needed afterwards; the compiler drops it
    const ulonglong2 own[2] = {make_ulonglong2(pack_f2(dz1[0][0], dz1[0][1]), pack_f2(dz1[0][2], dz1[0][3])),
                               make_ulonglong2(pack_f2(dz1[1][0], dz1[1][1]), pack_f2(dz1[1][2], dz1[1][3]))};
    dot_rows_rot<W, NCS>(sm + L0c.tbase[1] + j0 * WSW, act + L0c.dz + W * NCS + n0, F.roff, own, dz0, zk);
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const unsigned long long one = pack_f2(1.0f, 1.0f);
#pragma unroll
      for (int t = 0; t < 4; t += 2) {
        const unsigned long long h = pack_f2(h0[u][t], h0[u][t + 1]), nh = pack_f2(-h0[u][t], -h0[u][t + 1]);
        unsigned long long q;
        asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(q) : "l"(pack_f2(dz0[u][t], dz0[u][t + 1])), "l"(fma_f2(nh, h, one)));
        unpack_f2(q, dz0[u][t], dz0[u][t + 1]);
      }
    }
  }
  {  // partial sums of the weight gradients over this lane's four points -> part[slot][lane]
    float* pt = sm + L.part + ct;
    const unsigned long long x01 = pack_f2(F.x[0], F.x[1]), x23 = pack_f2(F.x[2], F.x[3]);
    const unsigned long long d01 = pack_f2(dO[0], dO[1]), d23 = pack_f2(dO[2], dO[3]);
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const unsigned long long z01 = pack_f2(dz1[u][0], dz1[u][1]), z23 = pack_f2(dz1[u][2], dz1[u][3]);
      const unsigned long long y01 = pack_f2(dz0[u][0], dz0[u][1]), y23 = pack_f2(dz0[u][2], dz0[u][3]);
#pragma unroll
      for (int k = 0; k < W; ++k) pt[(u * W + k) * 33] = quad_dot(z01, z23, hk[k].x, hk[k].y);
      pt[(2 * W + u) * 33] = (dz1[u][0] + dz1[u][1]) + (dz1[u][2] + dz1[u][3]);
      pt[(2 * W + 2 + u) * 33] = quad_dot(y01, y23, x01, x23);
      pt[(2 * W + 4 + u) * 33] = (dz0[u][0] + dz0[u][1]) + (dz0[u][2] + dz0[u][3]);
      pt[(2 * W + 6 + u) * 33] = quad_dot(d01, d23, pack_f2(h1[u][0], h1[u][1]), pack_f2(h1[u][2], h1[u][3]));
    }
    pt[(2 * W + 8) * 33] = (dO[0] + dO[1]) + (dO[2] + dO[3]);
  }
  __syncwarp();
  return ll_lane;
}

// likelihood gradient of the coordinate whose partial sums start at part[poff]: the NQ partials in fixed order
// (quads beyond the data, nq >= nq_used = ceil(N / 4), hold zeros and are not read)
template <int W>
__device__ __forceinline__ float fast2_reduce(const float* sm, const SmallParams& P, int poff, int nq_used) {
  constexpr int JP = W / 2, NQ = ((32 / W) * 8) / 4;
  const float* pp = sm + P.lay.part + poff;
  float v[NQ];
#pragma unroll
  for (int nq = 0; nq < NQ; ++nq) v[nq] = nq < nq_used ? pp[nq * JP] : 0.0f;
  float gsum = v[0];
#pragma unroll
  for (int nq = 1; nq < NQ; ++nq) gsum += v[nq];
  return gsum;
}

template <int W, typename Consume>
__device__ __forceinline__ float eval_fast2(float* sm, const SmallParams& P, const Likelihood lik, int ct, const FastRegs& F,
                                            Consume&& consume) {
  const float ll_lane = eval_fast2_partials<W>(sm, P, lik, ct, F);
  const int* pm = reinterpret_cast<const int*>(sm + P.lay.pmeta);
  const int nq_used = ((int)P.N + 3) / 4;
  for (int i = ct; i < (int)P.d; i += 32) consume(i, fast2_reduce<W>(sm, P, pm[i], nq_used));
  __syncwarp();
  return ll_lane;
}

// ------------------------------------------------------------------------------------------------
// kernel 1: log-posterior value + gradient for C chains (vihmc_logp_grad, MLP small path)
// ------------------------------------------------------------------------------------------------
template <int W, int FAST>
__global__ void __launch_bounds__(128, FAST >= 2 ? VIHMC_SMALL_MINBLOCKS2 : VIHMC_SMALL_MINBLOCKS) mlp_small_logp_grad_kernel(SmallParams P, long long C,
                                                                                         const float* __restrict__ q,
                                                                                         float* __restrict__ logp,
                                                                                         float* __restrict__ grad) {
  extern __shared__ __align__(16) float smem[];
  constexpr int T = Cfg<W>::T;
  const int ct = threadIdx.x % T, slot = threadIdx.x / T;
  const long long chain = (long long)blockIdx.x * (blockDim.x / T) + slot;
  if (chain >= C) return;
  const SmallLayout& L = P.lay;
  float* sm = smem + (size_t)slot * L.total;
  const float yv0 = chain_init<W>(sm, P, q + chain * P.d, ct, chain);
  const Likelihood lik = make_likelihood(P.loss, P.tau_out);
  float lp_lane = 0.0f;
  auto consume = [&](int i, float gl) {
    const float dq = sm[L.q + i] - sm[L.pmu + i], iv = sm[L.piv + i];
    lp_lane = fmaf(-0.5f * dq * dq, iv, lp_lane);
    if (grad != nullptr) grad[chain * P.d + i] = fmaf(-dq * iv, P.inv_prior_scale, gl);
  };
  float ll_lane;
  if constexpr (FAST >= 2) {
    FastRegs F;
    fast_setup<W>(sm, ct, yv0, F);
    fast2_setup<W>(sm, P, ct);
    ll_lane = eval_fast2<W>(sm, P, lik, ct, F, consume);
  } else if constexpr (FAST == 1) {
    FastRegs F;
    fast_setup<W>(sm, ct, yv0, F);
    ll_lane = eval_fast<W>(sm, P, lik, ct, F, consume);
  } else {
    ll_lane = eval_likelihood_grad<W>(sm, P, lik, ct, yv0, consume);
  }
  const float total = warp_sum(fmaf(lp_lane, P.inv_prior_scale, ll_lane)) + P.prior_log_norm * P.inv_prior_scale;
  if (ct == 0) logp[chain] = total;
}

// ------------------------------------------------------------------------------------------------
// kernel 1b: forward only (vihmc_predict, MLP small path): out[C, N]
// ------------------------------------------------------------------------------------------------
template <int W>
__global__ void __launch_bounds__(128) mlp_small_predict_kernel(SmallParams P, long long C, const float* __restrict__ q,
                                                                float* __restrict__ out) {
  extern __shared__ __align__(16) float smem[];
  using Cf = Cfg<W>;
  constexpr int T = Cf::T;
  const int ct = threadIdx.x % T, slot = threadIdx.x / T;
  const long long chain = (long long)blockIdx.x * (blockDim.x / T) + slot;
  if (chain >= C) return;
  float* sm = smem + (size_t)slot * P.lay.total;
  chain_init<W>(sm, P, q + chain * P.d, ct, chain);
  const int n_chunks = (int)((P.N + Cf::NC - 1) / Cf::NC);
  for (int chunk = 0; chunk < n_chunks; ++chunk) {
    if (chunk > 0) {
      stage_chunk<W>(sm, P, ct, chunk);
      __syncwarp();
    }
    const float o = forward_chunk<W>(sm, P, ct);
    const long long n = (long long)chunk * Cf::NC + ct;
    if (ct < Cf::NC && n < P.N) out[chain * P.N + n] = o;
    __syncwarp();
  }
}

// ------------------------------------------------------------------------------------------------
// kernel 1c: sensitivity scores of the VI -> HMC split selector (vihmc_mlp_sensitivity)
// Neural_network/VI/sensitivity.py:71-126: S_i = sigma_i^2 * mean_n (d o(x_n) / d w_i)^2 at w = the VI means.
// One CTA (one warp) per chunk of data points: forward, backward with d loss / d o = 1, then phase B with the
// SQUARED per-point products; partial[chunk, i] = sum over the chunk's points, summed in fixed order by the finish kernel.
// ------------------------------------------------------------------------------------------------
template <int W>
__global__ void __launch_bounds__(128) mlp_small_sensitivity_kernel(SmallParams P, const float* __restrict__ w,
                                                                    float* __restrict__ partial) {
  extern __shared__ __align__(16) float sm[];
  using Cf = Cfg<W>;
  const int ct = threadIdx.x;
  const int chunk = blockIdx.x;
  const SmallLayout& L = P.lay;
  chain_init<W>(sm, P, w, ct);
  if (chunk > 0) {
    stage_chunk<W>(sm, P, ct, chunk);
    __syncwarp();
  }
  forward_chunk<W>(sm, P, ct);
  float* act = sm + L.act_base;
  if (ct < Cf::NC) act[L.dO + ct] = ((long long)chunk * Cf::NC + ct < P.N) ? 1.0f : 0.0f;   // d o / d o
  __syncwarp();
  backward_chunk<W>(sm, P, ct);
  const int* meta = reinterpret_cast<const int*>(sm + L.meta);
  for (int i = ct; i < (int)P.d; i += Cf::T) {
    const int m = meta[i];
    const float4* A = reinterpret_cast<const float4*>(act + (m >> 16));
    const float4* B = reinterpret_cast<const float4*>(act + (m & 0xffff));
    float acc0 = 0.0f, acc1 = 0.0f, acc2 = 0.0f, acc3 = 0.0f;
#pragma unroll
    for (int c = 0; c < Cf::NC / 4; ++c) {
      const float4 a = A[c], b = B[c];
      const float t0 = a.x * b.x, t1 = a.y * b.y, t2 = a.z * b.z, t3 = a.w * b.w;
      acc0 = fmaf(t0, t0, acc0); acc1 = fmaf(t1, t1, acc1); acc2 = fmaf(t2, t2, acc2); acc3 = fmaf(t3, t3, acc3);
    }
    partial[(long long)chunk * P.d + i] = (acc0 + acc1) + (acc2 + acc3);
  }
}

// ------------------------------------------------------------------------------------------------
// kernel 2: the whole HMC run for C chains in one launch (vihmc_mlp_sample)
// ------------------------------------------------------------------------------------------------
struct SampleArgs {
  vihmc_sampler_cfg cfg;
  long long C;
  const float* q0;
  float* samples;
  unsigned char* accepted;
  float* hamiltonians;
  float* logp_out;
  float* step_sizes;
  const float* inj_p;
  const float* inj_u;
  const float* vi_sigma;   // per-sample VI redraw (vihmc_sampler_io): [D] standard deviations, or null
  float* vi_params;        // [num_samples, C, D] out, or null
  const float* inj_vi;     // [num_samples, C, D] injected normals, or null
  const float* inv_mass;   // [d] diagonal inverse mass (the MASS instantiation), or null
};

// MASS: diagonal mass m = A.inv_mass (hamiltorch's 1-D inv_mass).  p = fl(z s_i), ke = 0.5 sum p fl(m_i p), drift
// q += fl(fl(eps m_i) p); with MASS = false the code is exactly the identity-mass kernel.
template <int W, int FAST, bool MASS>
__global__ void __launch_bounds__(128, FAST >= 2 ? VIHMC_SMALL_MINBLOCKS2 : VIHMC_SMALL_MINBLOCKS) mlp_small_sample_kernel(SmallParams P, SampleArgs A) {
  extern __shared__ __align__(16) float smem[];
  constexpr int T = Cfg<W>::T;
  const int ct = threadIdx.x % T, slot = threadIdx.x / T;
  const long long chain = (long long)blockIdx.x * (blockDim.x / T) + slot;
  if (chain >= A.C) return;
  const SmallLayout& L = P.lay;
  float* sm = smem + (size_t)slot * L.total;
  const int d = (int)P.d;
  const long long C = A.C;
  const float* q0 = A.q0 + chain * d;
  const float yv0 = chain_init<W, MASS>(sm, P, q0, ct, chain, A.inv_mass);
  FastRegs F;
  if constexpr (FAST != 0) fast_setup<W>(sm, ct, yv0, F);
  if constexpr (FAST >= 2) fast2_setup<W>(sm, P, ct);
  // FAST == 3 (d <= 32 kRegRounds): the lane owns coordinates ct, ct + 32, ...; their constants live in registers for the whole run
  // and q, p for the length of a trajectory (ncu of FAST == 2: the dependent shared-memory round trips of the coordinate loop --
  // q, prior, p, table positions, then the stores -- were 29 % of all stall samples)
  constexpr int NR = FAST == 3 ? kRegRounds : 1;
  int r_pm[NR], r_wpos[NR], r_wposT[NR], r_idx[NR];
  const int nq_used = ((int)P.N + 3) / 4;
  float r_pmu[NR], r_piv[NR], r_q[NR], r_p[NR];
  float r_m[NR];   // MASS: the lane's inverse masses (s_i is read from shared memory by the once-per-iteration momentum draw)
  bool r_ok[NR];
  if constexpr (FAST == 3) {
    const int* pmv = reinterpret_cast<const int*>(sm + L.pmeta);
    const int* wpv = reinterpret_cast<const int*>(sm + L.wpos);
    const int* wtv = reinterpret_cast<const int*>(sm + L.wposT);
    const int* permv = reinterpret_cast<const int*>(sm + L.perm);
#pragma unroll
    for (int r = 0; r < NR; ++r) {
      const int i = permv[ct + 32 * r];
      r_idx[r] = i;
      r_ok[r] = i >= 0;
      r_pm[r] = r_ok[r] ? pmv[i] : 0;
      r_wpos[r] = r_ok[r] ? wpv[i] : 0;
      r_wposT[r] = r_ok[r] ? wtv[i] : -1;
      r_pmu[r] = r_ok[r] ? sm[L.pmu + i] : 0.0f;
      r_piv[r] = r_ok[r] ? sm[L.piv + i] : 0.0f;
      if constexpr (MASS) r_m[r] = r_ok[r] ? sm[L.minv + i] : 0.0f;
      r_q[r] = r_p[r] = 0.0f;
    }
  }
  const int* wposv = reinterpret_cast<const int*>(sm + L.wpos);
  const int* wposTv = reinterpret_cast<const int*>(sm + L.wposT);
  const Likelihood lik = make_likelihood(P.loss, P.tau_out);
  const unsigned long long gchain = (unsigned long long)(A.cfg.chain_offset + chain);
  const int S = A.cfg.num_samples, nsteps = A.cfg.num_steps, burn = A.cfg.burn;
  const float log_norm = P.prior_log_norm * P.inv_prior_scale;

  // dual-averaging state (Sampler.HMC_NUTS): every thread of the chain carries the same scalars
  float eps = A.cfg.step_size;
  const float eps_init = A.cfg.step_size;
  float eps_bar = 1.0f, H_t = 0.0f;

  for (int i = ct; i < d; i += T) A.samples[chain * d + i] = sm[L.q + i];  // stored row 0 = params_init
  float logp_init = 0.0f, logp_f = 0.0f;  // log-posterior of params_init / of the fallback state

  for (int n = 0; n < S; ++n) {
    if (A.cfg.hamiltorch_fallback_rule && n == burn + 1) {
      for (int i = ct; i < d; i += T) sm[L.qf + i] = q0[i];
      logp_f = logp_init;
    }
    // ---- per-sample VI redraw (my_make_func.py:45-50): all D frozen weights = mu + sigma z, then the sampled ones on top ----
    if (A.vi_sigma != nullptr) {
      const long long D = P.D;
      for (long long jb = ct; 4 * jb < D; jb += T) {
        float zz[4];
        if (A.inj_vi != nullptr) {
#pragma unroll
          for (int t = 0; t < 4; ++t) zz[t] = 4 * jb + t < D ? A.inj_vi[((long long)n * C + chain) * D + 4 * jb + t] : 0.0f;
        } else {
          const float4 z = philox_normal4(A.cfg.seed, gchain, (uint32_t)n, (uint32_t)jb, STREAM_VI_REDRAW);
          zz[0] = z.x; zz[1] = z.y; zz[2] = z.z; zz[3] = z.w;
        }
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          const long long f = 4 * jb + t;
          if (f < D) {
            int wpos, wposT, ao, bo;
            decode_coord(P, W, f, wpos, wposT, ao, bo);
            const float v = fmaf(__ldg(A.vi_sigma + f), zz[t], __ldg(P.frozen + chain * P.frozen_cs + f));
            sm[wpos] = v;
            if (wposT >= 0) sm[wposT] = v;
            if (A.vi_params != nullptr) A.vi_params[((long long)n * C + chain) * D + f] = v;
          }
        }
      }
      __syncwarp();
      for (int i = ct; i < d; i += T) {
        const float qv = sm[L.q + i];
        sm[wposv[i]] = qv;
        const int wt = wposTv[i];
        if (wt >= 0) sm[wt] = qv;
      }
      __syncwarp();
    }
    // ---- momentum ----
    float ke = 0.0f;
    if (A.inj_p != nullptr) {
      const float* src = A.inj_p + ((long long)n * C + chain) * d;
      for (int i = ct; i < d; i += T) {
        const float pv = src[i];   // injected momenta are used as p verbatim (already scaled for the mass)
        sm[L.p + i] = pv;
        if constexpr (MASS) ke = fmaf(pv, __fmul_rn(sm[L.minv + i], pv), ke);
        else ke = fmaf(pv, pv, ke);
      }
    } else {
      for (int jb = ct; 4 * jb < d; jb += T) {
        const float4 z = philox_normal4(A.cfg.seed, gchain, (uint32_t)n, (uint32_t)jb, STREAM_MOMENTUM);
        const float zz[4] = {z.x, z.y, z.z, z.w};
#pragma unroll
        for (int t = 0; t < 4; ++t)
          if (4 * jb + t < d) {
            if constexpr (MASS) {
              const int i = 4 * jb + t;
              const float pv = __fmul_rn(zz[t], sm[L.msq + i]);
              sm[L.p + i] = pv;
              ke = fmaf(pv, __fmul_rn(sm[L.minv + i], pv), ke);
            } else {
              sm[L.p + 4 * jb + t] = zz[t];
              ke = fmaf(zz[t], zz[t], ke);
            }
          }
      }
    }
    const float ke0 = 0.5f * warp_sum(ke);
    __syncwarp();

    // ---- trajectory: evaluation s = 0 yields H0 and the first half kick; s = nsteps yields H1 ----
    const float half_eps = 0.5f * eps;
    float logp0 = 0.0f, logp1 = 0.0f, ke1 = 0.0f;
    if constexpr (FAST == 3) {
#pragma unroll
      for (int r = 0; r < NR; ++r)
        if (r_ok[r]) { r_q[r] = sm[L.q + r_idx[r]]; r_p[r] = sm[L.p + r_idx[r]]; }
    }
    for (int s = 0; s <= nsteps; ++s) {
      const bool first = s == 0, last = s == nsteps;
      const float kick = first ? half_eps : eps;
      float lp_lane = 0.0f, ke_lane = 0.0f;
      if constexpr (FAST == 3) {   // the operations of consume() below on the register copies, all rounds in flight together
        const float ll3 = eval_fast2_partials<W>(sm, P, lik, ct, F);
        float gl[NR];
#pragma unroll
        for (int r = 0; r < NR; ++r) gl[r] = fast2_reduce<W>(sm, P, r_pm[r], nq_used);
        // branch-free (selects and predicated stores; empty slots carry q = p = 0, zero prior weights and wposT = -1)
#pragma unroll
        for (int r = 0; r < NR; ++r) {
          const float dq = r_q[r] - r_pmu[r], iv = r_piv[r];
          lp_lane = fmaf(-0.5f * dq * dq, iv, lp_lane);
          const float gi = r_ok[r] ? fmaf(-dq * iv, P.inv_prior_scale, gl[r]) : 0.0f;
          const float pk = axpy_unfused(kick, gi, r_p[r]);
          const float pv = last ? __fsub_rn(pk, __fmul_rn(half_eps, gi)) : pk;
          float qv;
          if constexpr (MASS) {
            ke_lane = fmaf(pv, __fmul_rn(r_m[r], pv), ke_lane);   // read only after the last evaluation
            qv = axpy_unfused(__fmul_rn(eps, r_m[r]), pv, r_q[r]);
          } else {
            ke_lane = fmaf(pv, pv, ke_lane);            // read only after the last evaluation
            qv = axpy_unfused(eps, pv, r_q[r]);
          }
          r_q[r] = last ? r_q[r] : qv;
          r_p[r] = pv;
          if (!last && r_ok[r]) sm[r_wpos[r]] = qv;
          if (!last && r_wposT[r] >= 0) sm[r_wposT[r]] = qv;
        }
        __syncwarp();
        if (first || last) {
          const float lp = warp_sum(fmaf(lp_lane, P.inv_prior_scale, ll3)) + log_norm;
          if (first) logp0 = lp;
          if (last) { logp1 = lp; ke1 = 0.5f * warp_sum(ke_lane); }
        }
        continue;
      }
      auto consume = [&](int i, float gl) {
        const float qv0 = sm[L.q + i];
        const float dq = qv0 - sm[L.pmu + i], iv = sm[L.piv + i];
        lp_lane = fmaf(-0.5f * dq * dq, iv, lp_lane);
        const float gi = fmaf(-dq * iv, P.inv_prior_scale, gl);
        float pv = axpy_unfused(kick, gi, sm[L.p + i]);
        if (last) {
          // hamiltorch: p += eps*g inside the loop, then ret_momenta[-1] - 0.5*eps*g (separately rounded)
          pv = __fsub_rn(pv, __fmul_rn(half_eps, gi));
          if constexpr (MASS) ke_lane = fmaf(pv, __fmul_rn(sm[L.minv + i], pv), ke_lane);
          else ke_lane = fmaf(pv, pv, ke_lane);
        } else {
          const float qv = axpy_unfused(MASS ? __fmul_rn(eps, sm[L.minv + i]) : eps, pv, qv0);
          sm[L.q + i] = qv;
          sm[wposv[i]] = qv;
          const int wt = wposTv[i];
          if (wt >= 0) sm[wt] = qv;
        }
        sm[L.p + i] = pv;
      };
      float ll_lane;
      if constexpr (FAST == 2) ll_lane = eval_fast2<W>(sm, P, lik, ct, F, consume);
      else if constexpr (FAST == 1) ll_lane = eval_fast<W>(sm, P, lik, ct, F, consume);
      else ll_lane = eval_likelihood_grad<W>(sm, P, lik, ct, yv0, consume);
      if (first || last) {
        const float lp = warp_sum(fmaf(lp_lane, P.inv_prior_scale, ll_lane)) + log_norm;
        if (first) logp0 = lp;
        if (last) { logp1 = lp; ke1 = 0.5f * warp_sum(ke_lane); }
      }
      __syncwarp();
    }
    if constexpr (FAST == 3) {
#pragma unroll
      for (int r = 0; r < NR; ++r)
        if (r_ok[r]) sm[L.q + r_idx[r]] = r_q[r];
      __syncwarp();
    }
    const float H0 = -logp0 + ke0, H1 = -logp1 + ke1;
    if (n == 0) {
      logp_init = logp0;
      logp_f = logp0;
      if (A.logp_out != nullptr && ct == 0) A.logp_out[chain] = logp0;
    }
    // ---- Metropolis test (hamiltorch: rho = min(0, H0-H1); accept iff rho >= log u) ----
    const float u = A.inj_u != nullptr ? A.inj_u[(long long)n * C + chain] : philox_uniform(A.cfg.seed, gchain, (uint32_t)n);
    const float rho = fminf(0.0f, H0 - H1);
    const bool finite = isfinite(logp1) && isfinite(H1) && isfinite(H0);
    const bool accept = finite && (rho >= logf(u));
    const bool store = n > burn;
    float* row = store ? A.samples + ((long long)(n - burn) * C + chain) * d : nullptr;
    if (accept) {
      logp_f = logp1;
      for (int i = ct; i < d; i += T) {
        const float qv = sm[L.q + i];
        sm[L.qf + i] = qv;
        if (store) row[i] = qv;
      }
    } else {
      for (int i = ct; i < d; i += T) {
        const float qv = sm[L.qf + i];
        sm[L.q + i] = qv;
        sm[wposv[i]] = qv;
        const int wt = wposTv[i];
        if (wt >= 0) sm[wt] = qv;
        if (store) row[i] = qv;
      }
    }
    if (ct == 0) {
      if (A.accepted != nullptr) A.accepted[(long long)n * C + chain] = accept ? 1 : 0;
      if (A.hamiltonians != nullptr) {
        A.hamiltonians[((long long)n * C + chain) * 2 + 0] = H0;
        A.hamiltonians[((long long)n * C + chain) * 2 + 1] = H1;
      }
      if (A.logp_out != nullptr && store) A.logp_out[(long long)(n - burn) * C + chain] = logp_f;
    }
    // ---- dual averaging (hamiltorch adaptation(): gamma .05, t0 10, kappa .75, mu = log(10 eps0)) ----
    if (A.cfg.adapt_step_size && n <= burn) {
      if (n < burn) {
        const float t = (float)(n + 1);
        const float alpha = finite ? fminf(1.0f, expf(rho)) : 0.0f;
        const float mu = logf(10.0f * eps_init);
        H_t = (1.0f - 1.0f / (t + 10.0f)) * H_t + (1.0f / (t + 10.0f)) * (A.cfg.desired_accept_rate - alpha);
        const float x_new = mu - sqrtf(t) / 0.05f * H_t;
        eps = expf(x_new);
        const float tk = powf(t, -0.75f);
        eps_bar = expf(tk * x_new + (1.0f - tk) * logf(eps_bar));
      }
      if (n == burn) eps = eps_bar;
    }
    __syncwarp();
  }
  if (A.step_sizes != nullptr && ct == 0) A.step_sizes[chain] = eps;
}

// ------------------------------------------------------------------------------------------------
// launch helpers shared by the per-width translation units
// ------------------------------------------------------------------------------------------------
enum SmallOp { kOpLogpGrad = 0, kOpPredict = 1, kOpSample = 2, kOpSensitivity = 3 };

struct SmallLaunch {
  int chains_per_block, blocks;
  int fast;   // specialised 1-W-W-1 tanh single-chunk evaluation: 1 = eval_fast, 2 = eval_fast2 (register partial sums, W <= 16)
  size_t smem;
  long long C;
  const float* q;
  float* logp;
  float* grad;
  float* out;
  SampleArgs A;
};

template <typename K>
static int set_smem(K kernel, size_t bytes) {
  if (bytes > 48u * 1024u) VIHMC_CUDA_OK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
  return VIHMC_OK;
}

template <int W, int FAST, bool MASS = false>
static int launch_small_wn(SmallOp op, const SmallParams& P, const SmallLaunch& a, cudaStream_t st) {
  const int threads = a.chains_per_block * 32;
  if (op == kOpLogpGrad) {
    auto k = mlp_small_logp_grad_kernel<W, FAST>;
    if (int rc = set_smem(k, a.smem)) return rc;
    k<<<a.blocks, threads, a.smem, st>>>(P, a.C, a.q, a.logp, a.grad);
    VIHMC_LAUNCH_OK("mlp_small_logp_grad_kernel");
  } else if (op == kOpSensitivity) {   // q = weights, out = partial sums [blocks, d]
    auto k = mlp_small_sensitivity_kernel<W>;
    if (int rc = set_smem(k, a.smem)) return rc;
    k<<<a.blocks, 32, a.smem, st>>>(P, a.q, a.out);
    VIHMC_LAUNCH_OK("mlp_small_sensitivity_kernel");
  } else if (op == kOpPredict) {
    auto k = mlp_small_predict_kernel<W>;
    if (int rc = set_smem(k, a.smem)) return rc;
    k<<<a.blocks, threads, a.smem, st>>>(P, a.C, a.q, a.out);
    VIHMC_LAUNCH_OK("mlp_small_predict_kernel");
  } else {
    auto k = mlp_small_sample_kernel<W, FAST, MASS>;
    if (int rc = set_smem(k, a.smem)) return rc;
    k<<<a.blocks, threads, a.smem, st>>>(P, a.A);
    VIHMC_LAUNCH_OK("mlp_small_sample_kernel");
  }
  return VIHMC_OK;
}

// the sampler with a diagonal mass takes the MASS instantiation of the same variant (only the sample kernel has one)
template <int W, int FAST>
static int launch_small_wm(SmallOp op, const SmallParams& P, const SmallLaunch& a, cudaStream_t st) {
  if (op == kOpSample && a.A.inv_mass != nullptr) return launch_small_wn<W, FAST, true>(op, P, a, st);
  return launch_small_wn<W, FAST, false>(op, P, a, st);
}

template <int W>
static int launch_small_w(SmallOp op, const SmallParams& P, const SmallLaunch& a, cudaStream_t st) {
  if constexpr (W <= 16) {   // version 2 keeps 2 W quads in registers: widths above 16 stay on version 1
    if (a.fast == 2 && op == kOpSample && P.d <= 32 * kRegRounds) return launch_small_wm<W, 3>(op, P, a, st);
    if (a.fast == 2) return launch_small_wm<W, 2>(op, P, a, st);
  }
  if (a.fast) return launch_small_wm<W, 1>(op, P, a, st);
  return launch_small_wm<W, 0>(op, P, a, st);
}

}  // namespace vihmc
