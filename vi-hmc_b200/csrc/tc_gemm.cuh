// Tensor-core batched GEMM for the dense path: tcgen05.mma kind::tf32 with FP32 accumulators in TMEM,
// 3xTF32 operand splitting for fp32-grade accuracy, and the dense path's fused epilogues.
//
//   C[b] = opA(A[b]) (MxK) * opB(B[b]) (KxN)          (same GemmArgs as the FP32-SIMT kernel in dense.cu)
//
// Why 3xTF32: the parity bar is rtol 1e-5 against the reference's fp32 closure; one TF32 product carries
// ~1e-3.  Every fp32 operand v is split into hi = rna_tf32(v) and lo = rna_tf32(v - hi) (both written to
// shared memory as exact tf32 values, low 13 mantissa bits zero, so the result does not depend on how the
// tensor core converts fp32 bits to tf32) and the product is hi*hi + lo*hi + hi*lo, accumulated in fp32.
//
// Structure of one CTA (256 threads, one 128 x 128 output tile, 3 x 32 KB smem stages, 256 TMEM columns => exactly
// 2 CTAs / SM, so no third CTA sits spinning in tcgen05.alloc so one CTA's
// epilogue overlaps another's main loop):
//   * all 8 warps stream the A / B k-tiles (16 floats deep) from global memory through registers, split
//     them, and store hi/lo tiles as 8x16B core matrices (no swizzle).  Three staging modes per operand:
//       KVEC   K is the contiguous dimension (activations, W[n,k]): float4 loads along K, K-major tile;
//       MNVEC  M/N is the contiguous dimension (dZ^T, X in dW = dZ^T X; W in dX = dZ W; G^T): float4 loads
//              along M/N stored as an MN-major tile -- the tensor core transposes (instruction-descriptor
//              a_major / b_major bits), so no operand is ever transposed through registers or copied;
//       SCALAR any element strides / alignment (101-wide branch input): predicated scalar loads, K-major.
//     The split needs the values in registers anyway, which is why the operands are not staged with TMA.
//   * three smem stages; thread 0 issues 3 MMAs per 8-deep k-step and commits to the stage's mbarrier;
//     the next tile's global loads are in flight while the tensor core works.
//   * epilogue: 8 warps read the accumulators with tcgen05.ld (warp w -> TMEM lanes 32*(w%4).., column
//     half w/4) into a shared-memory tile, then apply bias+act / act' / Gaussian residual and write C
//     row-wise so every warp instruction touches contiguous memory.
#pragma once
#include <stdlib.h>

#include "common.cuh"

namespace vihmc {

enum Epilogue {
  EPI_STORE = 0,      // C = acc
  EPI_BIAS_ACT = 1,   // C = act(acc + bias[n])           (act = identity when act < 0)
  EPI_DACT = 2,       // C = acc * act'(aux[m,n])         (aux = the layer's stored activation)
  EPI_HEAD = 3        // r = acc + bias0 - Y[m,n]; C = -prec r; partial sums of loglik and of C per CTA
};

struct GemmArgs {
  const float* A; long long a_bs, a_sm, a_sk;
  const float* B; long long b_bs, b_sk, b_sn;
  float* C; long long c_bs, ldc;
  int M, N, K;
  // epilogue operands
  const float* bias; long long bias_bs;   // [N] per batch (EPI_BIAS_ACT) or scalar per batch (EPI_HEAD)
  const float* aux; long long aux_bs, ld_aux;  // activation (EPI_DACT) or Y (EPI_HEAD; aux_bs = 0: shared)
  int act;
  int row_pad_ok;   // rows of C and aux are allocated up to round_up(N, 4) floats: float4 access may straddle N
  float ll_const, half_prec, prec;
  float* part_ll; float* part_g;          // [batch, tiles] (EPI_HEAD)
  // split-K (EPI_STORE only): blockIdx.z = b * splits + s handles k in [s*kc, min(K,(s+1)*kc)) and writes its
  // partial product to split_buf[(s*batch + b), M, N]; splits <= 1 means a plain GEMM
  int splits, kc, batch;
  int kc_hint;   // host side: preferred split-K slice length for this product (0: the default, kSplitKChunk)
  int slice_tiles;   // TMEM-A kernels: k-tiles per accumulation chain; the CTA sums its slices itself (0: one chain per CTA)
  float* split_buf;
  // row sums of opA over this CTA's K range (EPI_STORE, A staged MN-major, N <= 128): rowsum_part[(s*batch + b), M].
  // With opA = dZ^T these are the bias gradients sum_r dz[r, o], read off the operand stream the GEMM loads anyway.
  float* rowsum_part;
};

namespace tc {

constexpr int BM = 128, BN = 128, BK = 16, THREADS = 256, STAGES = 3;
constexpr int CHUNKS = BK / 4;                 // 16-byte chunks along K per row
constexpr int LBO = 128;                       // bytes between the K-chunks of a core-matrix row group
constexpr int SBO = CHUNKS * 128;              // bytes between 8-row groups
constexpr int TILE_BYTES = (BM / 8) * SBO;     // 8 KB: one 128 x 16 fp32 operand tile
constexpr int STAGE_BYTES = 4 * TILE_BYTES;    // A_hi, A_lo, B_hi, B_lo
constexpr int TILE_LD = BN + 4;                 // epilogue staging tile row stride (floats): conflict-free float4 rows
constexpr int EPI_BYTES = BM * TILE_LD * 4;     // 67,584 B >= the two operand stages
constexpr int SMEM_BYTES = (EPI_BYTES > STAGES * STAGE_BYTES ? EPI_BYTES : STAGES * STAGE_BYTES) + 128;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// Shared-memory matrix descriptor (cute::UMMA::SmemDescriptor bit layout, version 1 = Blackwell; bits 61-63 = layout type).
// K-major tile, no swizzle (type 0): core matrix = 8 rows x 16 B of K; LBO = bytes between the K chunks, SBO = bytes
//   between 8-row groups.
// MN-major tile: for 32-bit operands the tensor core only transposes the SWIZZLE_128B_BASE32B layout (type 1) -- every
//   other layout type returns zeros for an MN-major tf32 operand (measured with vihmc_debug_umma,
//   tools/probe_umma_layout.py, which also pinned the word map below).  An atom is 4 k-rows x 32 M/N elements (512 B):
//     byte(k, n) = (n/32)*LBO + (k/4)*SBO + (k%4)*128 + ((((n%32)/8) ^ (k%4))*32) + (n%8)*4
//   i.e. each k-row is 128 B of 32 consecutive M/N elements whose four 32-byte chunks are XOR-ed with the row index.
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo, uint32_t layout_type = 0) {
  return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)(lbo >> 4) << 16) | ((uint64_t)(sbo >> 4) << 32) | (1ull << 46) |
         ((uint64_t)layout_type << 61);
}
constexpr int MN_LBO = 512;                    // MN-major tile: the four 32-element M/N atoms of a k-atom are contiguous
constexpr int MN_SBO = (BM / 32) * MN_LBO;     // 2 KB: one 4-deep K atom of 128 rows
constexpr uint32_t MN_LAYOUT = 1;              // SWIZZLE_128B_BASE32B

// kind::tf32, FP32 accumulate, M = 128, N = BN (cute::UMMA::InstrDescriptor bit layout); bit 15 / 16 = A / B is MN-major
constexpr uint32_t kIdesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);

__device__ __forceinline__ void mma_tf32(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc),
      "r"(accumulate)
      : "memory");
}

// the same MMA with the A operand read from tensor memory ([taddr]: lane = row m, one 32-bit column per k) instead of through a
// shared-memory descriptor: A_hi / A_lo then never cross the shared-memory port, which is what bounds this kernel (DESIGN.md 3.2b')
__device__ __forceinline__ void mma_tf32_ta(uint32_t tmem_d, uint32_t tmem_a, uint64_t db, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}\n" ::"r"(tmem_d), "r"(tmem_a), "l"(db), "r"(idesc),
      "r"(accumulate)
      : "memory");
}

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// bounded spin: a wedged barrier traps (kernel error) instead of hanging the GPU
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = smem_u32(bar);
  for (uint32_t spin = 0; spin < (1u << 26); ++spin) {
    uint32_t done;
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
        : "=r"(done)
        : "r"(addr), "r"(parity)
        : "memory");
    if (done) return;
  }
  __trap();
}

// 3xTF32 split with ROUND-TO-NEAREST: hi = rna_tf32(v), lo = rna_tf32(v - hi) (v - hi is exact in fp32).
// Truncating instead (v & 0xFFFFE000) shrinks every operand toward zero, i.e. a coherent ~1e-6 relative
// bias on every output; sums with heavy cancellation (d/d b0 = sum of G over N*P outputs) then miss the
// 1e-5 parity bar.  With rounding the per-product error is zero-mean.
// rna = round to nearest, ties away from zero, on the sign-magnitude bit pattern: add half a tf32 ulp and clear
// the 13 low mantissa bits.  Two integer instructions; `cvt.rna.tf32.f32` compiles to the same pair plus an
// Inf/NaN guard (FSETP + predicate), which finite network values do not need (a non-finite value stays non-finite
// or becomes NaN, and the sampler rejects either).
__device__ __forceinline__ float rna_tf32(float v) { return __uint_as_float((__float_as_uint(v) + 0x1000u) & 0xFFFFE000u); }
// The split in the staging loops: TWO packed instructions per element instead of five.  These kernels are bound by instruction
// issue (ncu source view of a long-K product: 242 warp instructions per warp per k-tile, half of them indexing, an eighth the split;
// profiles/r01_summary.md E1), so every instruction per staged element counts.
//   hi: Veltkamp's splitter with 2^13 + 1 -- g = fl(8193 v), hi = fl(g + fl(v - g)) is v rounded to nearest at 11 significant bits,
//       i.e. a tf32 value -- as three fma.rn.f32x2 (Blackwell's packed FP32 pipe: two IEEE results per instruction);
//   lo: v - hi, exact in fp32, NOT rounded to tf32: the tensor core drops the 13 low mantissa bits of a tf32 operand, a truncation
//       toward zero OF LO.  lo's sign is unrelated to v's, so unlike truncating hi (the coherent bias described above) this is a
//       zero-mean error of at most 2^-22 |v| per operand, below the fp32 rounding of the products themselves.
// Non-finite or |v| > 4e34 inputs give NaN (8193 v overflows), which the sampler rejects like any non-finite log-posterior.
__device__ __forceinline__ unsigned long long pk2(float a, float b) {
  unsigned long long r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b));
  return r;
}
__device__ __forceinline__ unsigned long long fma2(unsigned long long a, unsigned long long b, unsigned long long c) {
  unsigned long long d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
__device__ __forceinline__ void split2(float a, float b, float& ha, float& hb, float& la, float& lb) {
  const unsigned long long v = pk2(a, b), c = pk2(8193.0f, 8193.0f), one = pk2(1.0f, 1.0f), mone = pk2(-1.0f, -1.0f);
  const unsigned long long g = fma2(v, c, 0ull);
  const unsigned long long d = fma2(g, mone, v);
  const unsigned long long h = fma2(d, one, g);
  const unsigned long long l = fma2(h, mone, v);
  asm("mov.b64 {%0, %1}, %2;" : "=f"(ha), "=f"(hb) : "l"(h));
  asm("mov.b64 {%0, %1}, %2;" : "=f"(la), "=f"(lb) : "l"(l));
}
__device__ __forceinline__ void split4(const float4 v, float4& hi, float4& lo) {
  split2(v.x, v.y, hi.x, hi.y, lo.x, lo.y);
  split2(v.z, v.w, hi.z, hi.w, lo.z, lo.w);
}

enum LoadMode { LOAD_SCALAR = 0, LOAD_KVEC = 1, LOAD_MNVEC = 2 };

// One operand tile: rows [r0, r0+128) x k [kt*16, kt*16+16).  Element (r, k) lives at base + r*s_r + k*s_k.
//   K-major modes: a warp instruction covers one 8-row group x 4 chunks: lane -> (row r8 = lane%8, chunk = lane/8).
//   MNVEC: a thread's float4 is 4 consecutive rows at one k; (warp, i) -> atom, lane -> (k row, 4-row block).
struct TileLoader {
  // Everything that does not depend on the k-tile is computed once per thread: the pointer of the thread's two float4
  // at k-tile 0 (null when its rows are outside the matrix), how many of a float4's rows are inside (MNVEC), and the k
  // offset inside a tile.  fetch(kt) then costs one pointer add and one k-bound test per float4.
  const float* p[2];
  long long s_k, step;   // element stride along K; pointer advance per k-tile
  int koff[2], nrow[2], soff[2];   // soff: byte offset of the float4 inside the staged tile
  int K, mode;
  __device__ __forceinline__ void init(const float* base, long long s_r, long long sk, int R, int K_, int r0, int mode_, int tid) {
    const int lane = tid & 31, warp = tid >> 5;
    s_k = sk; step = (long long)BK * sk; K = K_; mode = mode_;
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      int r;
      if (mode == LOAD_MNVEC) {
        // (warp, i) -> one atom: 4 k-rows x 32 rows; lane -> (k row lane%4, 4-row block lane/4): a k-row is 128 contiguous bytes
        const int atom = warp * 2 + i;   // mn atom = atom % 4, k atom = atom / 4
        koff[i] = (atom >> 2) * 4 + (lane & 3);
        r = r0 + (atom & 3) * 32 + (lane >> 2) * 4;
        nrow[i] = R - r < 4 ? (R - r > 0 ? R - r : 0) : 4;
        p[i] = base + r + (long long)koff[i] * sk;
        // a quarter warp (4 k-rows x 2 half chunks) covers 8 distinct 16-byte bank groups: conflict-free
        const int k4 = lane & 3;
        soff[i] = (atom & 3) * MN_LBO + (atom >> 2) * MN_SBO + k4 * 128 + (((lane >> 3) ^ k4) * 32) + ((lane >> 2) & 1) * 16;
      } else {
        // lane -> (row r8 = lane%8, chunk = lane/8): 16-byte stores of a quarter warp are conflict-free, 64 contiguous bytes per row
        koff[i] = (lane >> 3) * 4;
        r = r0 + (i * 8 + warp) * 8 + (lane & 7);
        nrow[i] = r < R ? 1 : 0;
        p[i] = base + (long long)r * s_r + (long long)koff[i] * sk;
        soff[i] = (i * 8 + warp) * SBO + (lane >> 3) * LBO + (lane & 7) * 16;
      }
    }
  }
  // MODE >= 0: the staging mode is a compile-time constant (TMEM-A kernels): no mode branches in the k loop, and k-tiles that lie
  // entirely below K -- all but the last -- skip the per-element bound tests.  MODE = -1: runtime mode.
  template <int MODE>
  __device__ __forceinline__ void fetch_t(int kt, float4 (&v)[2]) const {
    if (MODE >= 0 && (kt + 1) * BK <= K) {
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
        const float* q = p[i] + (long long)kt * step;
        if (MODE == LOAD_MNVEC) {
          if (nrow[i] == 4) x = __ldg(reinterpret_cast<const float4*>(q));
          else if (nrow[i] > 0) {
            x.x = __ldg(q);
            if (nrow[i] > 1) x.y = __ldg(q + 1);
            if (nrow[i] > 2) x.z = __ldg(q + 2);
          }
        } else if (MODE == LOAD_KVEC) {
          if (nrow[i] > 0) x = __ldg(reinterpret_cast<const float4*>(q));
        } else if (nrow[i] > 0) {
          x.x = __ldg(q); x.y = __ldg(q + s_k); x.z = __ldg(q + 2 * s_k); x.w = __ldg(q + 3 * s_k);
        }
        v[i] = x;
      }
    } else {
      fetch(kt, v);
    }
  }
  __device__ __forceinline__ void fetch(int kt, float4 (&v)[2]) const {
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
      const int k = kt * BK + koff[i];
      const float* q = p[i] + (long long)kt * step;
      if (nrow[i] > 0 && k < K) {
        if (mode == LOAD_MNVEC) {
          if (nrow[i] == 4) {
            x = __ldg(reinterpret_cast<const float4*>(q));
          } else {
            x.x = __ldg(q);
            if (nrow[i] > 1) x.y = __ldg(q + 1);
            if (nrow[i] > 2) x.z = __ldg(q + 2);
          }
        } else if (mode == LOAD_KVEC && k + 3 < K) {
          x = __ldg(reinterpret_cast<const float4*>(q));
        } else {
          x.x = __ldg(q);
          if (k + 1 < K) x.y = __ldg(q + s_k);
          if (k + 2 < K) x.z = __ldg(q + 2 * s_k);
          if (k + 3 < K) x.w = __ldg(q + 3 * s_k);
        }
      }
      v[i] = x;
    }
  }
};

// TMEM-A mode: a thread owns one row m of the A tile (its TMEM lane) and the 8 k of one half of a 16-deep k-tile
// (warps 0-3: k 0..7, warps 4-7: k 8..15).  MN-major A (m contiguous): 8 loads, each coalesced over the warp's 32 rows;
// K-major A: two float4 of the thread's own row.
constexpr int ATM_ACCN = 112;                 // accumulator columns / instruction N in TMEM-A mode (N <= 112)
constexpr int ATM_ACOL = 2 * ATM_ACCN;        // A stage: hi in columns [224, 240), lo in [240, 256) of the 256 allocated
struct RowLoader {
  const float* p;
  long long s_k;
  int K, kh, ok, vec;
  __device__ __forceinline__ void init(const float* base, long long s_m, long long sk, int M, int K_, int m0, int mode, int tid) {
    const int lane = tid & 31, warp = tid >> 5;
    const int row = m0 + 32 * (warp & 3) + lane;
    kh = (warp >> 2) * 8; s_k = sk; K = K_; ok = row < M; vec = mode == LOAD_KVEC;
    p = base + (long long)row * s_m + (long long)kh * sk;
  }
  template <int MODE>
  __device__ __forceinline__ void fetch(int kt, float (&v)[8]) const {
    const int k0 = kt * BK + kh;
    const float* q = p + (long long)kt * BK * s_k;
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = 0.0f;
    if (!ok) return;
    if (k0 + 8 <= K) {   // every k-tile but the last: no per-element bound tests
      if (MODE == LOAD_KVEC) {
        const float4 x = __ldg(reinterpret_cast<const float4*>(q)), y = __ldg(reinterpret_cast<const float4*>(q + 4));
        v[0] = x.x; v[1] = x.y; v[2] = x.z; v[3] = x.w; v[4] = y.x; v[5] = y.y; v[6] = y.z; v[7] = y.w;
      } else {
        // element j is j * s_k floats further: byte offsets fit 32 bits (leading dimensions are < 2^26 floats)
        const char* qb = reinterpret_cast<const char*>(q);
        const unsigned skb = (unsigned)s_k * 4u;
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = __ldg(reinterpret_cast<const float*>(qb + (size_t)((unsigned)j * skb)));
      }
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j)
        if (k0 + j < K) v[j] = __ldg(q + (long long)j * s_k);
    }
  }
};

// split the thread's 8 values (registers only) ...
__device__ __forceinline__ void split8(const float (&v)[8], uint32_t (&hi)[8], uint32_t (&lo)[8]) {
#pragma unroll
  for (int j = 0; j < 8; j += 2) {
    float h0, h1, l0, l1;
    split2(v[j], v[j + 1], h0, h1, l0, l1);
    hi[j] = __float_as_uint(h0); hi[j + 1] = __float_as_uint(h1);
    lo[j] = __float_as_uint(l0); lo[j + 1] = __float_as_uint(l1);
  }
}
// ... and write them to its TMEM lane: hi at column col, lo 16 columns further
__device__ __forceinline__ void store_tmem(uint32_t taddr, const uint32_t (&hi)[8], const uint32_t (&lo)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(hi[0]), "r"(hi[1]),
               "r"(hi[2]), "r"(hi[3]), "r"(hi[4]), "r"(hi[5]), "r"(hi[6]), "r"(hi[7])
               : "memory");
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr + 16u), "r"(lo[0]), "r"(lo[1]),
               "r"(lo[2]), "r"(lo[3]), "r"(lo[4]), "r"(lo[5]), "r"(lo[6]), "r"(lo[7])
               : "memory");
  asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}

__device__ __forceinline__ void stash(unsigned char* hi_tile, unsigned char* lo_tile, const TileLoader& ld, const float4 (&v)[2]) {
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    float4 hi, lo;
    split4(v[i], hi, lo);
    *reinterpret_cast<float4*>(hi_tile + ld.soff[i]) = hi;
    *reinterpret_cast<float4*>(lo_tile + ld.soff[i]) = lo;
  }
}

// operand descriptor of the ks-th K = 8 step inside a staged 16-deep tile
__device__ __forceinline__ uint64_t step_desc(uint32_t tile_saddr, int mode, int ks) {
  return mode == LOAD_MNVEC ? make_desc(tile_saddr + (uint32_t)ks * 2u * MN_SBO, MN_LBO, MN_SBO, MN_LAYOUT)
                            : make_desc(tile_saddr + (uint32_t)ks * 2u * LBO, LBO, SBO);
}


// Phase-2 epilogue of the staged tile: warp w owns rows w, w+8, ...; applies the fused epilogue and writes C.  With
// `vec` (C rows 16-byte aligned, N % 4 == 0 or padded rows) every lane handles 4 consecutive columns with one
// LDS.128 / STG.128 (one warp instruction = one 512-byte row); otherwise lane + 32*j columns (128 contiguous bytes
// each).  ACT is a template parameter so the activation is chosen once per kernel, not per element; the bias of a
// lane's columns is loaded once, row pointers advance by constant strides.
enum { ACT_NONE = -1 };

struct EpiCtx {
  const float* tile;       // staged accumulators [BM][ld]
  int ld;
  float* crow;             // C + (m0 + warp) * ldc + n0
  const float* arow;       // aux + (m0 + warp) * ld_aux + n0 (or null)
  const float* biasb;      // bias of this batch (EPI_BIAS_ACT)
  long long c_step, a_step;   // 8 rows of C / aux
  int rows, n0, N, lane, warp;
  bool vec, vec_aux;
  float bias0, ll_const, half_prec, prec;
};

template <int EPI, int ACT>
__device__ __forceinline__ void epilogue_rows(const EpiCtx& e, float& ll_acc, float& g_acc) {
  auto apply = [&](float v, float bias_v, float aux_v) -> float {
    if (EPI == EPI_BIAS_ACT) {
      v += bias_v;
      if (ACT == VIHMC_ACT_TANH) v = tanh_sel(v);   // 6 instructions, abs. error ~1.2e-7 (see common.cuh)
      else if (ACT == VIHMC_ACT_RELU) v = v > 0.0f ? v : 0.0f;
    } else if (EPI == EPI_DACT) {
      v *= (ACT == VIHMC_ACT_TANH) ? (1.0f - aux_v * aux_v) : (aux_v > 0.0f ? 1.0f : 0.0f);
    } else if (EPI == EPI_HEAD) {
      const float res = v + e.bias0 - aux_v;
      ll_acc += e.ll_const - e.half_prec * res * res;
      v = -e.prec * res;
      g_acc += v;
    }
    return v;
  };
  const float* trow = e.tile + e.warp * e.ld;
  float* crow = e.crow;
  const float* arow = e.arow;
  if (e.vec) {
    const int c = e.lane * 4;
    const int nv = e.N - (e.n0 + c);   // valid columns of this lane's float4 (N % 4 != 0 only with padded rows)
    if (nv <= 0) return;
    float4 bv = make_float4(0.f, 0.f, 0.f, 0.f);
    if (EPI == EPI_BIAS_ACT) {
      bv.x = __ldg(e.biasb + e.n0 + c);
      if (nv > 1) bv.y = __ldg(e.biasb + e.n0 + c + 1);
      if (nv > 2) bv.z = __ldg(e.biasb + e.n0 + c + 2);
      if (nv > 3) bv.w = __ldg(e.biasb + e.n0 + c + 3);
    }
    // Rows in batches of U: all aux loads (Y for the head product, the stored activation for DACT) of a batch are issued before
    // the first is used.  With two rows in flight the head product spent 35 % of its stall samples on the one FADD that
    // consumes the Y load (ncu source view): the epilogue, half of that kernel's instructions, was a chain of L2 latencies.
    constexpr int U = (EPI == EPI_DACT || EPI == EPI_HEAD) ? 8 : 2;
    constexpr int RS = THREADS / 32;
    for (int r0 = e.warp; r0 < e.rows; r0 += RS * U) {
      float4 av[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        av[u] = make_float4(0.f, 0.f, 0.f, 0.f);
        if ((EPI == EPI_DACT || EPI == EPI_HEAD) && r0 + RS * u < e.rows) {
          const float* ar = arow + u * e.a_step;
          if (e.vec_aux) av[u] = __ldg(reinterpret_cast<const float4*>(ar + c));
          else { av[u].x = __ldg(ar + c); av[u].y = __ldg(ar + c + 1); av[u].z = __ldg(ar + c + 2); av[u].w = __ldg(ar + c + 3); }
        }
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        if (r0 + RS * u < e.rows) {
          const float4 v = *reinterpret_cast<const float4*>(trow + u * RS * e.ld + c);
          float4 o;
          o.x = apply(v.x, bv.x, av[u].x);
          o.y = nv > 1 ? apply(v.y, bv.y, av[u].y) : 0.0f;
          o.z = nv > 2 ? apply(v.z, bv.z, av[u].z) : 0.0f;
          o.w = nv > 3 ? apply(v.w, bv.w, av[u].w) : 0.0f;
          *reinterpret_cast<float4*>(crow + u * e.c_step + c) = o;
        }
      }
      trow += U * RS * e.ld;
      crow += U * e.c_step;
      arow += U * e.a_step;
    }
  } else {
    float bias_v[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (EPI == EPI_BIAS_ACT && e.n0 + e.lane + 32 * j < e.N) bias_v[j] = __ldg(e.biasb + e.n0 + e.lane + 32 * j);
    for (int r = e.warp; r < e.rows; r += THREADS / 32) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int c = e.lane + 32 * j;
        if (e.n0 + c >= e.N) continue;
        const float aux_v = (EPI == EPI_DACT || EPI == EPI_HEAD) ? __ldg(arow + c) : 0.0f;
        crow[c] = apply(trow[c], bias_v[j], aux_v);
      }
      trow += (THREADS / 32) * e.ld;
      crow += e.c_step;
      arow += e.a_step;
    }
  }
}

__device__ __forceinline__ bool rows_vec_ok(const float* base, long long bs, long long ld, int N, int row_pad_ok) {
  return (reinterpret_cast<uintptr_t>(base) & 15u) == 0 && bs % 4 == 0 && ld % 4 == 0 && (N % 4 == 0 || row_pad_ok);
}

// ATM (EPI_STORE, N <= 112, one n-tile): the A operand lives in tensor memory (see RowLoader); accumulators are 112 columns wide and
// the single A stage takes the remaining 32 of the 256 allocated columns, so two CTAs per SM still hold TMEM at a time.
constexpr int ATM_PF = 3;   // k-tiles of register prefetch in TMEM-A mode (see the main loop)
// TMEM-A mode, round 2: the CTA sums its accumulation slices itself.  The tensor core's fp32 accumulate truncates, so a chain is
// bounded to slice_tiles k-tiles (256 deep by default); in round 2's first version every slice was its own CTA and wrote a
// partial tile (3 GB per DeepONet gradient batch, a fifth of the batch's time with the reduction kernel).  Now a CTA walks
// several slices: at a slice boundary the 8 warps read the two accumulators (tcgen05.ld), add main + correction and then the
// running sum -- a [128][116] fp32 tile in shared memory -- with round-to-nearest adds; the next slice starts a fresh chain.
// Shared memory: the A stages are not used in this mode, so the B stages are packed (3 x 16 KB) and the sum tile follows:
// 108.7 KB per CTA, still two CTAs per SM.  Cross-CTA splits remain only to fill the GPU.
// Two B stages are enough here: every k-tile waits for the previous k-tile's MMAs anyway (one A stage in tensor memory), so
// the stage of k-tile kt - 2 is free when k-tile kt is staged.  92 KB per CTA -- not more than before: with 2 x 109 KB the driver
// picks the 233 KB shared-memory carve-out, and the ~20 KB of L1 that leaves made the K-major A stream (row-strided 32-byte
// pieces, two k-tiles per 128-byte line) of the dxb product 1.7x slower.
constexpr int ATM_STAGES = 2;
constexpr int ATM_SUM_LD = ATM_ACCN + 4;
constexpr int ATM_SUM_OFF = ATM_STAGES * 2 * TILE_BYTES;
constexpr int SMEM_BYTES_ATM = ATM_SUM_OFF + BM * ATM_SUM_LD * 4 + 128;
template <int EPI, bool ATM = false, int AM = -1, int BMD = -1>
__global__ void __launch_bounds__(THREADS, AM >= 0 ? 2 : 3) tc_gemm_kernel(GemmArgs g, int a_mode, int b_mode) {
  constexpr bool RING = AM >= 0;   // compile-time staging modes + ATM_PF k-tiles of register prefetch (two CTAs per SM)
  if (AM >= 0) { a_mode = AM; b_mode = BMD; }   // compile-time staging modes (all TMEM-A kernels, and the K-major / K-major fast variant)
  constexpr int ACCN = ATM ? ATM_ACCN : BN;
  constexpr int NST = ATM ? ATM_STAGES : STAGES;   // shared-memory stages
  extern __shared__ __align__(1024) unsigned char smem_raw[];   // swizzled MN-major tiles need 1 KB-aligned bases
  unsigned char* smem = smem_raw;
  constexpr int SB = ATM ? SMEM_BYTES_ATM : SMEM_BYTES;
  uint64_t* mbar = reinterpret_cast<uint64_t*>(smem + SB - 128);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + SB - 64);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const bool split = (EPI == EPI_STORE) && g.splits > 1;
  const int b = split ? (int)blockIdx.z / g.splits : (int)blockIdx.z;
  const int ksplit = split ? (int)blockIdx.z % g.splits : 0;
  const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
  if (split) {   // restrict this CTA to its K slice and redirect the output to the partial buffer
    const int k_lo = ksplit * g.kc;
    g.A += (long long)k_lo * g.a_sk;
    g.B += (long long)k_lo * g.b_sk;
    g.K = (g.K - k_lo) < g.kc ? (g.K - k_lo) : g.kc;
    g.C = g.split_buf + ((long long)ksplit * g.batch) * (long long)g.M * g.N;
    g.c_bs = (long long)g.M * g.N;
    g.ldc = g.N;
  }

  if (tid == 0) {
    for (int s = 0; s < NST; ++s) mbar_init(&mbar[s], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"((uint32_t)(2 * BN)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_d = *tmem_slot;

  TileLoader la, lb;
  RowLoader lr;
  if (ATM) lr.init(g.A + (long long)b * g.a_bs, g.a_sm, g.a_sk, g.M, g.K, m0, a_mode, tid);
  else la.init(g.A + (long long)b * g.a_bs, g.a_sm, g.a_sk, g.M, g.K, m0, a_mode, tid);
  lb.init(g.B + (long long)b * g.b_bs, g.b_sn, g.b_sk, g.N, g.K, n0, b_mode, tid);
  const uint32_t idesc = ATM ? ((1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(ACCN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24) |
                                (b_mode == LOAD_MNVEC ? 1u << 16 : 0u))
                             : (kIdesc | (a_mode == LOAD_MNVEC ? 1u << 15 : 0u) | (b_mode == LOAD_MNVEC ? 1u << 16 : 0u));
  const uint32_t a_taddr = tmem_d + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)ATM_ACOL + (uint32_t)((warp >> 2) * 8);

  // One k-tile of register prefetch.  (Two tiles ahead was measured slower: 120+ registers leave room for only two
  // resident CTAs, and a third CTA parked in tcgen05.alloc is what hides the launch latency of the next tile.)
  const int nk = (g.K + BK - 1) / BK;
  const int SL = (ATM && g.slice_tiles > 0) ? g.slice_tiles : nk;   // k-tiles per accumulation chain
  float* sum_tile = reinterpret_cast<float*>(smem + ATM_SUM_OFF);
  // slice boundary (TMEM-A mode): sum_tile (+)= main + correction accumulators; every MMA of the slice has completed
  auto flush = [&](bool first_slice) {
    const int q = warp & 3, half = warp >> 2;
    float* srow = sum_tile + (q * 32 + lane) * ATM_SUM_LD + half * (ATM_ACCN / 2);
#pragma unroll 1
    for (int cc = 0; cc < ATM_ACCN / 2; cc += 8) {
      if (half * (ATM_ACCN / 2) + cc >= g.N) break;
      uint32_t r[8], rc[8];
      const uint32_t taddr = tmem_d + ((uint32_t)(q * 32) << 16) + (uint32_t)(half * (ATM_ACCN / 2) + cc);
      asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                   : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                   : "r"(taddr));
      asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                   : "=r"(rc[0]), "=r"(rc[1]), "=r"(rc[2]), "=r"(rc[3]), "=r"(rc[4]), "=r"(rc[5]), "=r"(rc[6]), "=r"(rc[7])
                   : "r"(taddr + (uint32_t)ATM_ACCN));
      asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
      float v[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = __uint_as_float(r[j]) + __uint_as_float(rc[j]);   // main + corrections (RN)
      if (!first_slice) {
        const float4 s0 = *reinterpret_cast<const float4*>(srow + cc), s1 = *reinterpret_cast<const float4*>(srow + cc + 4);
        v[0] += s0.x; v[1] += s0.y; v[2] += s0.z; v[3] += s0.w;
        v[4] += s1.x; v[5] += s1.y; v[6] += s1.z; v[7] += s1.w;
      }
      *reinterpret_cast<float4*>(srow + cc) = make_float4(v[0], v[1], v[2], v[3]);
      *reinterpret_cast<float4*>(srow + cc + 4) = make_float4(v[4], v[5], v[6], v[7]);
    }
  };
  float4 ra[2], rb[2];
  const bool want_rowsum = (EPI == EPI_STORE) && g.rowsum_part != nullptr;   // host guarantees a_mode == LOAD_MNVEC
  float4 rs[2] = {make_float4(0.f, 0.f, 0.f, 0.f), make_float4(0.f, 0.f, 0.f, 0.f)};
  float rsum = 0.0f;
  // TMEM-A mode keeps ATM_PF k-tiles of global loads in flight per thread.  These long-K products are bound by bytes in flight
  // (Little's law): with ONE 16 KB k-tile per CTA and two TMEM-holding CTAs per SM, 32 KB per SM against a loaded memory latency of
  // ~2 500 clk is 13 B/clk per SM = 3.6 TB/s for the whole GPU -- exactly the ~1 275 clk per k-tile both operand paths measured.
  // Dropping A from shared memory is what makes room for it: 72 registers -> ~110 still fits the two CTAs that can hold TMEM.
  float rva[ATM_PF][8];
  float4 raa[ATM_PF][2], rbb[ATM_PF][2];
  if (RING) {
#pragma unroll
    for (int i = 0; i < ATM_PF; ++i)
      if (i < nk) {
        if (ATM) lr.template fetch<AM>(i, rva[i]);
        else la.template fetch_t<AM>(i, raa[i]);
        lb.template fetch_t<BMD>(i, rbb[i]);
      }
  } else {
    la.template fetch_t<AM>(0, ra);
    lb.template fetch_t<BMD>(0, rb);
  }
  int sl_pos = 0;   // k-tile index inside the current accumulation slice (kept incrementally: no division in the loop)
  auto issue_mma = [&](int kt, unsigned char* st, int s) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t sa = smem_u32(st);
    const int k_left = g.K - kt * BK;
    const int steps = k_left > 8 ? 2 : 1;
    for (int ks = 0; ks < steps; ++ks) {
      const uint64_t b_hi = step_desc(sa + 2 * TILE_BYTES, b_mode, ks), b_lo = step_desc(sa + 3 * TILE_BYTES, b_mode, ks);
      const uint32_t acc = ((ATM ? sl_pos : kt) > 0 || ks > 0) ? 1u : 0u;
      if (ATM) {
        const uint32_t ta = tmem_d + (uint32_t)ATM_ACOL + (uint32_t)ks * 8u;
        mma_tf32_ta(tmem_d, ta, b_hi, idesc, acc);
        mma_tf32_ta(tmem_d + ACCN, ta + 16u, b_hi, idesc, acc);
        mma_tf32_ta(tmem_d + ACCN, ta, b_lo, idesc, 1u);
      } else {
        const uint64_t a_hi = step_desc(sa, a_mode, ks), a_lo = step_desc(sa + TILE_BYTES, a_mode, ks);
        mma_tf32(tmem_d, a_hi, b_hi, idesc, acc);
        mma_tf32(tmem_d + ACCN, a_lo, b_hi, idesc, acc);
        mma_tf32(tmem_d + ACCN, a_hi, b_lo, idesc, 1u);
      }
    }
    mma_commit(&mbar[s]);
  };
  if (RING) {
    for (int kt0 = 0; kt0 < nk; kt0 += ATM_PF) {
#pragma unroll
      for (int i = 0; i < ATM_PF; ++i) {
        const int kt = kt0 + i;
        if (kt < nk) {
          const int s = kt % NST;
          // (TMEM-A mode: packed B stages; the pointer is biased so that st + 2 TILE_BYTES is the stage's B_hi tile)
          unsigned char* st = ATM ? smem + s * 2 * TILE_BYTES - 2 * TILE_BYTES : smem + s * STAGE_BYTES;
          if (ATM) { sl_pos = (kt == 0 || sl_pos + 1 == SL) ? 0 : sl_pos + 1; }
          // one A stage in tensor memory: the MMAs of the previous k-tile must have read it (commits complete in order, so
          // this also frees the shared-memory stage of k-tile kt - STAGES)
          if (ATM) {
            // Everything that does not touch the single A stage runs BEFORE the wait for the previous k-tile's MMAs, i.e. while the
            // tensor core is still working on them: the split (registers), the B tile (its shared-memory stage was last read by
            // k-tile kt - STAGES, complete since the wait of the previous iteration) and the next global loads.
            uint32_t hi[8], lo[8];
            if (want_rowsum)
              rsum += ((rva[i][0] + rva[i][1]) + (rva[i][2] + rva[i][3])) + ((rva[i][4] + rva[i][5]) + (rva[i][6] + rva[i][7]));
            split8(rva[i], hi, lo);
            stash(st + 2 * TILE_BYTES, st + 3 * TILE_BYTES, lb, rbb[i]);
            if (kt + ATM_PF < nk) {
              lr.template fetch<AM>(kt + ATM_PF, rva[i]);
              lb.template fetch_t<BMD>(kt + ATM_PF, rbb[i]);
            }
            if (kt >= 1) mbar_wait(&mbar[(kt - 1) % NST], (uint32_t)((kt - 1) / NST) & 1u);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            if (kt > 0 && sl_pos == 0) flush(kt == SL);   // slice boundary: bank the finished chain before the next one starts
            store_tmem(a_taddr, hi, lo);
          } else {
            if (kt >= NST) mbar_wait(&mbar[s], (uint32_t)(kt / NST - 1) & 1u);   // shared-memory A: only the stage must be free
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            if (want_rowsum) {
#pragma unroll
              for (int j = 0; j < 2; ++j) { rs[j].x += raa[i][j].x; rs[j].y += raa[i][j].y; rs[j].z += raa[i][j].z; rs[j].w += raa[i][j].w; }
            }
            stash(st, st + TILE_BYTES, la, raa[i]);
            stash(st + 2 * TILE_BYTES, st + 3 * TILE_BYTES, lb, rbb[i]);
            if (kt + ATM_PF < nk) {
              la.template fetch_t<AM>(kt + ATM_PF, raa[i]);
              lb.template fetch_t<BMD>(kt + ATM_PF, rbb[i]);
            }
          }
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
          asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
          __syncthreads();
          if (tid == 0) issue_mma(kt, st, s);
        }
      }
    }
  }
  for (int kt = 0; !RING && kt < nk; ++kt) {
    const int s = kt % NST;
    unsigned char* st = smem + s * STAGE_BYTES;
    {
      if (kt >= NST) mbar_wait(&mbar[s], (uint32_t)(kt / NST - 1) & 1u);   // the MMAs that read this stage are done
      if (want_rowsum) {
#pragma unroll
        for (int i = 0; i < 2; ++i) { rs[i].x += ra[i].x; rs[i].y += ra[i].y; rs[i].z += ra[i].z; rs[i].w += ra[i].w; }
      }
      stash(st, st + TILE_BYTES, la, ra);
      stash(st + 2 * TILE_BYTES, st + 3 * TILE_BYTES, lb, rb);
      if (kt + 1 < nk) {   // next tile's global loads are in flight while the tensor core works on this one
        la.template fetch_t<AM>(kt + 1, ra);
        lb.template fetch_t<BMD>(kt + 1, rb);
      }
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy stores -> visible to the tensor core
    __syncthreads();
    if (tid == 0) {
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const uint32_t sa = smem_u32(st);
      const int k_left = g.K - kt * BK;
      const int steps = k_left > 8 ? 2 : 1;
      for (int ks = 0; ks < steps; ++ks) {
        const uint64_t a_hi = step_desc(sa, a_mode, ks), a_lo = step_desc(sa + TILE_BYTES, a_mode, ks);
        const uint64_t b_hi = step_desc(sa + 2 * TILE_BYTES, b_mode, ks), b_lo = step_desc(sa + 3 * TILE_BYTES, b_mode, ks);
        // The tensor core's fp32 accumulate rounds toward zero: every accumulate step shrinks the running sum
        // by up to one ulp, a COHERENT bias that grows with the number of chained MMAs.  The two correction
        // products therefore get their own accumulator (columns BN..2BN): the main chain sees one accumulate
        // per k-step instead of three, and the correction chain's truncation is 2^-11 smaller.
        const uint32_t acc = (kt > 0 || ks > 0) ? 1u : 0u;
        mma_tf32(tmem_d, a_hi, b_hi, idesc, acc);
        mma_tf32(tmem_d + BN, a_lo, b_hi, idesc, acc);
        mma_tf32(tmem_d + BN, a_hi, b_lo, idesc, 1u);
      }
      mma_commit(&mbar[s]);
    }
  }
  mbar_wait(&mbar[(nk - 1) % NST], (uint32_t)((nk - 1) / NST) & 1u);   // commits complete in order: everything is done
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");

  if (ATM && want_rowsum && blockIdx.x == 0) {
    // a thread summed its row over its half of every k-tile: add the two halves (fixed order)
    float* red = reinterpret_cast<float*>(smem);
    __syncthreads();
    red[(warp >> 2) * BM + (warp & 3) * 32 + lane] = rsum;
    __syncthreads();
    if (tid < BM && m0 + tid < g.M) g.rowsum_part[((long long)ksplit * g.batch + b) * g.M + m0 + tid] = red[tid] + red[BM + tid];
    __syncthreads();
  }
  if (!ATM && want_rowsum && blockIdx.x == 0) {
    // A thread's float4 i holds rows 32*(atom&3) + 4*(lane>>2) .. +3 at k rows (atom>>2)*4 + (lane&3) of every k-tile
    // (atom = 2*warp + i): sum over the 4 k rows by shuffle, over the 4 k atoms (= warp pairs) through shared memory.
    // Fixed order throughout: reproducible.
    float* red = reinterpret_cast<float*>(smem);   // [4 k atoms][128 rows]; the operand stages are dead
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      float v[4] = {rs[i].x, rs[i].y, rs[i].z, rs[i].w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        v[j] += __shfl_xor_sync(0xffffffffu, v[j], 1);
        v[j] += __shfl_xor_sync(0xffffffffu, v[j], 2);
      }
      const int atom = warp * 2 + i;
      if ((lane & 3) == 0)
        *reinterpret_cast<float4*>(red + (atom >> 2) * BM + (atom & 3) * 32 + (lane >> 2) * 4) = make_float4(v[0], v[1], v[2], v[3]);
    }
    __syncthreads();
    if (tid < BM && m0 + tid < g.M) {
      const float t = (red[tid] + red[BM + tid]) + (red[2 * BM + tid] + red[3 * BM + tid]);
      g.rowsum_part[((long long)ksplit * g.batch + b) * g.M + m0 + tid] = t;
    }
    __syncthreads();
  }

  // ---------------- epilogue ----------------
  // phase 1: TMEM -> registers -> shared tile [128][TILE_LD] (thread = one accumulator row, 8 columns per ld).
  // phase 2: coalesced pass: warp w owns rows w, w+8, ...; a warp instruction touches 512 contiguous bytes of
  // C / aux (each lane 4 columns), instead of 32 different rows as a row-per-thread epilogue would.
  float* tile = ATM ? sum_tile : reinterpret_cast<float*>(smem);   // operand stages are dead: every MMA has completed
  if (ATM) {
    flush(nk <= SL);   // the last slice; the sum tile is the staged tile of phase 2
  } else {
    const int q = warp & 3, half = warp >> 2;
    float* trow = tile + (q * 32 + lane) * TILE_LD + half * (BN / 2);
#pragma unroll 2
    for (int cc = 0; cc < BN / 2; cc += 8) {
      if (n0 + half * (BN / 2) + cc >= g.N) break;   // columns past N (100-wide layers in a 128-wide tile) are never read
      uint32_t r[8], rc[8];
      const uint32_t taddr = tmem_d + ((uint32_t)(q * 32) << 16) + (uint32_t)(half * (BN / 2) + cc);
      asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                   : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                   : "r"(taddr));
      asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                   : "=r"(rc[0]), "=r"(rc[1]), "=r"(rc[2]), "=r"(rc[3]), "=r"(rc[4]), "=r"(rc[5]), "=r"(rc[6]), "=r"(rc[7])
                   : "r"(taddr + (uint32_t)ACCN));
      asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
      float v[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = __uint_as_float(r[j]) + __uint_as_float(rc[j]);   // main + corrections (RN)
      *reinterpret_cast<float4*>(trow + cc) = make_float4(v[0], v[1], v[2], v[3]);
      *reinterpret_cast<float4*>(trow + cc + 4) = make_float4(v[4], v[5], v[6], v[7]);
    }
  }
  __syncthreads();
  EpiCtx e;
  e.tile = tile;
  e.ld = ATM ? ATM_SUM_LD : TILE_LD;
  e.crow = g.C + (long long)b * g.c_bs + (long long)(m0 + warp) * g.ldc + n0;
  e.arow = (EPI == EPI_DACT || EPI == EPI_HEAD) ? g.aux + (long long)b * g.aux_bs + (long long)(m0 + warp) * g.ld_aux + n0 : nullptr;
  e.biasb = (EPI == EPI_BIAS_ACT) ? g.bias + (long long)b * g.bias_bs : nullptr;
  e.c_step = (long long)(THREADS / 32) * g.ldc;
  e.a_step = (long long)(THREADS / 32) * g.ld_aux;
  e.rows = g.M - m0 < BM ? g.M - m0 : BM;
  e.n0 = n0; e.N = g.N; e.lane = lane; e.warp = warp;
  e.vec = rows_vec_ok(g.C, g.c_bs, g.ldc, g.N, g.row_pad_ok);
  e.vec_aux = e.arow != nullptr && rows_vec_ok(g.aux, g.aux_bs, g.ld_aux, g.N, g.row_pad_ok);
  e.bias0 = (EPI == EPI_HEAD) ? __ldg(g.bias + (long long)b * g.bias_bs) : 0.0f;
  e.ll_const = g.ll_const; e.half_prec = g.half_prec; e.prec = g.prec;
  float ll_acc = 0.0f, g_acc = 0.0f;
  if (EPI == EPI_BIAS_ACT || EPI == EPI_DACT) {
    if (g.act == VIHMC_ACT_TANH) epilogue_rows<EPI, VIHMC_ACT_TANH>(e, ll_acc, g_acc);
    else if (g.act == VIHMC_ACT_RELU) epilogue_rows<EPI, VIHMC_ACT_RELU>(e, ll_acc, g_acc);
    else epilogue_rows<EPI, ACT_NONE>(e, ll_acc, g_acc);
  } else {
    epilogue_rows<EPI, ACT_NONE>(e, ll_acc, g_acc);
  }
  if (EPI == EPI_HEAD) {
    float* red = reinterpret_cast<float*>(smem);
    ll_acc = warp_sum(ll_acc);
    g_acc = warp_sum(g_acc);
    __syncthreads();   // every warp is done reading the staged tile
    if (lane == 0) { red[warp] = ll_acc; red[8 + warp] = g_acc; }
    __syncthreads();
    if (tid == 0) {
      float s0 = 0.0f, s1 = 0.0f;
      for (int w = 0; w < THREADS / 32; ++w) { s0 += red[w]; s1 += red[8 + w]; }
      const long long tiles = (long long)gridDim.x * gridDim.y;
      const long long t = (long long)blockIdx.y * gridDim.x + blockIdx.x;
      g.part_ll[(long long)b * tiles + t] = s0;
      g.part_g[(long long)b * tiles + t] = s1;
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_d), "r"((uint32_t)(2 * BN)) : "memory");
}

}  // namespace tc

// ---------------------------------------------------------------------------------------------
// Layout probe (test hook, vihmc_debug_umma): ONE tcgen05.mma kind::tf32 (M = 128, N = 128, K = 8) on operand tiles
// taken verbatim from two 8 KB images, with caller-chosen descriptor strides and instruction descriptor.  Feeding an
// identity-like A and B[i] = i makes D spell out which shared-memory word the tensor core reads for every (k, n):
// this is how the MN-major staging layout above was pinned on hardware (tests/test_gpu_deeponet.py).
// ---------------------------------------------------------------------------------------------
namespace tc {
constexpr int kProbeSmem = 96 * 1024;
__global__ void __launch_bounds__(128) umma_probe_kernel(const float* __restrict__ a_img, const float* __restrict__ b_img,
                                                         uint32_t a_lbo, uint32_t a_sbo, uint32_t b_lbo, uint32_t b_sbo,
                                                         uint32_t a_type, uint32_t b_type, uint32_t idesc, float* __restrict__ out) {
  extern __shared__ __align__(1024) unsigned char tiles[];   // A image, B image, then zero-filled guard space
  __shared__ __align__(8) uint64_t bar;
  __shared__ uint32_t tmem_slot;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  for (int i = tid; i < kProbeSmem / 4; i += 128) reinterpret_cast<float*>(tiles)[i] = 0.0f;
  __syncthreads();
  for (int i = tid; i < TILE_BYTES / 4; i += 128) {
    reinterpret_cast<float*>(tiles)[i] = a_img[i];
    reinterpret_cast<float*>(tiles + TILE_BYTES)[i] = b_img[i];
  }
  if (tid == 0) {
    mbar_init(&bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_slot)), "r"(128u) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_d = tmem_slot;
  if (tid == 0) {
    mma_tf32(tmem_d, make_desc(smem_u32(tiles), a_lbo, a_sbo, a_type), make_desc(smem_u32(tiles + TILE_BYTES), b_lbo, b_sbo, b_type),
             idesc, 0u);
    mma_commit(&bar);
  }
  mbar_wait(&bar, 0u);
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  for (int cc = 0; cc < 128; cc += 8) {
    uint32_t r[8];
    const uint32_t taddr = tmem_d + ((uint32_t)(warp * 32) << 16) + (uint32_t)cc;
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
    for (int j = 0; j < 8; ++j) out[(warp * 32 + lane) * 128 + cc + j] = __uint_as_float(r[j]);
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_d), "r"(128u) : "memory");
}
}  // namespace tc

// C[b, m, n] = sum_s split_buf[s, b, m, n] in fixed order (fp32 round-to-nearest adds)
__global__ void __launch_bounds__(256) splitk_reduce_kernel(const float* __restrict__ buf, int splits, int batch, int M, int N,
                                                            float* __restrict__ C, long long c_bs, long long ldc) {
  const long long per = (long long)M * N, total = (long long)batch * per;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    float s = 0.0f;
    for (int k = 0; k < splits; ++k) s += buf[(long long)k * total + t];
    const long long b = t / per, r = t % per;
    C[b * c_bs + (r / N) * ldc + (r % N)] = s;
  }
}

// out[b*out_bs + m] = sum_s part[(s*batch + b), m]  (bias gradients from the row sums of the weight-gradient GEMM)
__global__ void rowsum_finish_kernel(const float* __restrict__ part, int splits, int batch, int M, float* __restrict__ out,
                                     long long out_bs) {
  // one thread per (batch, row), splits summed in ascending order (the loads are independent of the adds and pipeline); with one
  // block per batch entry the wide BNN's 391 slices x 512 rows took 243 us per layer on 8 blocks
  const int b = blockIdx.x, m = blockIdx.y * blockDim.x + threadIdx.x;
  if (m >= M) return;
  float s = 0.0f;
#pragma unroll 8
  for (int k = 0; k < splits; ++k) s += part[((long long)k * batch + b) * M + m];
  out[(long long)b * out_bs + m] = s;
}

// The fp32 accumulate of tcgen05.mma truncates toward zero: a chain of k accumulations shrinks the sum by ~k/2 ulp.  At BASELINE
// size (K = 10201) 1152-deep slices left 1.3e-5 relative error on the trunk's weight gradients (tests/diag_fullsize.py); with
// 256-deep slices (32 chained accumulations) summed by round-to-nearest adds it is below 4e-6.
constexpr int kSplitKChunk = 256;       // K slice per CTA once K exceeds 1.5 slices (K = 500, the M = 2 split closures -> two slices)
constexpr int kFillSplitMinK = 512;     // medium reductions are split only to put more CTAs on the GPU (few chains)
constexpr int kFillSplitMax = 8;

// The most K slices splitk_plan can choose for a reduction of K with this slice hint, at any batch: a split product needs
// slices * batch * M * N floats of scratch.
inline int splitk_max_slices(int K, int kc_hint) {
  const int chunk = kc_hint > 0 ? kc_hint : kSplitKChunk;
  if (K > chunk + chunk / 2) return (K + chunk - 1) / chunk;
  if (K >= kFillSplitMinK) return K / 128 < kFillSplitMax ? K / 128 : kFillSplitMax;
  return 1;
}

// shapes the tensor-core kernel is used for; everything else stays on the FP32-SIMT kernel
inline bool tc_gemm_eligible(const GemmArgs& g) { return g.M >= 32 && g.K >= 16 && (g.N >= 16 || g.K >= 512); }

inline int tc_num_sms() {
  static const int n = []() {
    int dev = 0, v = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev);
    return v;
  }();
  return n;
}

// staging mode of one operand: element (r, k) at base + b*bs + r*s_r + k*s_k
inline int operand_mode(const float* base, long long bs, long long s_r, long long s_k) {
  const bool aligned = (reinterpret_cast<uintptr_t>(base) & 15u) == 0 && bs % 4 == 0;
  if (aligned && s_k == 1 && s_r % 4 == 0) return tc::LOAD_KVEC;
  if (aligned && s_r == 1 && s_k % 4 == 0) return tc::LOAD_MNVEC;
  return tc::LOAD_SCALAR;
}

// Sets g.splits, g.kc and g.slice_tiles for `batch` products.  Only EPI_STORE products split, and only when scratch for the
// partial products is available (can_split); use_atm selects the TMEM-A kernel.  g.splits never exceeds
// splitk_max_slices(g.K, g.kc_hint).
inline void splitk_plan(GemmArgs& g, int batch, bool use_atm, bool can_split) {
  g.splits = 1;
  g.batch = batch;
  const int chunk = g.kc_hint > 0 ? g.kc_hint : kSplitKChunk, thresh = chunk + chunk / 2;
  const int max_splits = splitk_max_slices(g.K, g.kc_hint);
  g.slice_tiles = use_atm ? chunk / tc::BK : 0;
  if (!can_split) return;
  const long long slots = 2LL * tc_num_sms();
  if (use_atm && g.K > thresh) {
    // TMEM-A kernels sum their slices in shared memory: cross-CTA splits only fill the GPU.  Cost of a choice in k-units per
    // CTA slot: rounds x (slice-aligned K range + the partial tile's write and read, ~106 k-units of operand traffic)
    const long long tiles = (long long)((g.M + tc::BM - 1) / tc::BM) * batch;
    long long best_cost = -1;
    for (int sp = 1; sp <= max_splits; ++sp) {
      const int kc = ((g.K + sp - 1) / sp + chunk - 1) / chunk * chunk;
      if ((long long)kc * (sp - 1) >= g.K) continue;   // the last split would be empty
      const long long rounds = (tiles * sp + slots - 1) / slots;
      const long long cost = rounds * (kc + (sp > 1 ? 106 : 0));
      if (best_cost < 0 || cost < best_cost) { best_cost = cost; g.kc = kc; }
    }
    g.splits = (g.K + g.kc - 1) / g.kc;
  } else if (g.K > thresh) {
    // long reductions (dW = dZ^T X over thousands of rows): bound the length of one TMEM accumulation chain
    // (its fp32 accumulate truncates) and sum the slices with round-to-nearest adds
    // Slice length between one chunk (what the scratch is sized for) and 1.5 chunks, chosen so that the CTAs
    // fill whole rounds of the GPU: 2 CTAs per SM hold TMEM at a time, and e.g. 64 chains x 10 slices = 640 CTAs would
    // run 3 rounds for 2.16 rounds of work where 9 slices of 1152 run 2.
    const long long tiles = (long long)((g.N + tc::BN - 1) / tc::BN) * ((g.M + tc::BM - 1) / tc::BM) * batch;
    const int min_splits = (g.K + thresh - 1) / thresh;
    long long best_cost = -1;
    for (int sp = max_splits; sp >= min_splits && sp >= 1; --sp) {
      const int kc = ((g.K + sp - 1) / sp + tc::BK - 1) / tc::BK * tc::BK;
      const long long rounds = (tiles * sp + slots - 1) / slots;
      const long long cost = rounds * kc;
      if (best_cost < 0 || cost < best_cost) { best_cost = cost; g.kc = kc; }
    }
    g.splits = (g.K + g.kc - 1) / g.kc;
  } else if (g.K >= kFillSplitMinK) {
    // medium reduction, few output tiles (the branch's weight gradients: 64 chains = 64 CTAs): split to fill the GPU
    const long long tiles = (long long)((g.N + tc::BN - 1) / tc::BN) * ((g.M + tc::BM - 1) / tc::BM) * batch;
    long long sp = slots / tiles;
    if (sp > max_splits) sp = max_splits;
    if (sp >= 2 && (long long)batch * sp <= 65535) {
      g.kc = (int)(((g.K + sp - 1) / sp + tc::BK - 1) / tc::BK * tc::BK);
      g.splits = (g.K + g.kc - 1) / g.kc;
    }
  }
}

// scratch: room for scratch_floats floats of split-K partial products (splitk_max_slices(K, kc_hint) * batch * M * N are
// always enough); VIHMC_ERR_WORKSPACE if the plan needs more.
// rowsum_out (EPI_STORE, optional): receives sum_k opA[b][m, k] at rowsum_out[b*rowsum_bs + m]; rowsum_part is scratch of
// splits * batch * M floats (at most splitk_max_slices(K, kc_hint) * batch * M).  When the fused row sums cannot be used
// (*rowsum_done stays 0) the caller computes them itself.
template <int EPI>
static int launch_tc_gemm(GemmArgs g, int batch, cudaStream_t st, float* scratch = nullptr, long long scratch_floats = 0,
                          float* rowsum_part = nullptr, float* rowsum_out = nullptr, long long rowsum_bs = 0, int* rowsum_done = nullptr) {
  const int a_mode = operand_mode(g.A, g.a_bs, g.a_sm, g.a_sk);
  const int b_mode = operand_mode(g.B, g.b_bs, g.b_sn, g.b_sk);
  auto k = tc::tc_gemm_kernel<EPI>;
  static bool configured = false;
  if (!configured) {
    VIHMC_CUDA_OK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::SMEM_BYTES));
    configured = true;
  }
  // TMEM-A variant: plain-store products with one n-tile of at most 112 columns (the weight-gradient GEMMs and the two
  // head-backward products)
  const bool use_atm = EPI == EPI_STORE && g.N <= tc::ATM_ACCN;
  splitk_plan(g, batch, use_atm, EPI == EPI_STORE && scratch != nullptr);
  if (g.splits > 1) {
    if ((long long)batch * g.splits > 65535) return fail(VIHMC_ERR_UNSUPPORTED, "gemm: batch * splits > 65535");
    if ((long long)g.splits * batch * g.M * g.N > scratch_floats)
      return fail(VIHMC_ERR_WORKSPACE, "gemm: %d K slices need %lld floats of scratch, %lld given", g.splits,
                  (long long)g.splits * batch * g.M * g.N, scratch_floats);
    g.split_buf = scratch;
  }
  const int tiles_n = (g.N + tc::BN - 1) / tc::BN, tiles_m = (g.M + tc::BM - 1) / tc::BM;
  const bool fuse_rowsum = EPI == EPI_STORE && rowsum_part != nullptr && rowsum_out != nullptr && (a_mode == tc::LOAD_MNVEC || use_atm);
  g.rowsum_part = fuse_rowsum ? rowsum_part : nullptr;
  dim3 grid(tiles_n, tiles_m, batch * g.splits);
  if (EPI == EPI_STORE && use_atm) {
    using KernelT = void (*)(GemmArgs, int, int);
    static const KernelT table[3][3] = {
        {tc::tc_gemm_kernel<EPI_STORE, true, tc::LOAD_SCALAR, tc::LOAD_SCALAR>, tc::tc_gemm_kernel<EPI_STORE, true, tc::LOAD_SCALAR, tc::LOAD_KVEC>,
         tc::tc_gemm_kernel<EPI_STORE, true, tc::LOAD_SCALAR, tc::LOAD_MNVEC>},
        {tc::tc_gemm_kernel<EPI_STORE, true, tc::LOAD_KVEC, tc::LOAD_SCALAR>, tc::tc_gemm_kernel<EPI_STORE, true, tc::LOAD_KVEC, tc::LOAD_KVEC>,
         tc::tc_gemm_kernel<EPI_STORE, true, tc::LOAD_KVEC, tc::LOAD_MNVEC>},
        {tc::tc_gemm_kernel<EPI_STORE, true, tc::LOAD_MNVEC, tc::LOAD_SCALAR>, tc::tc_gemm_kernel<EPI_STORE, true, tc::LOAD_MNVEC, tc::LOAD_KVEC>,
         tc::tc_gemm_kernel<EPI_STORE, true, tc::LOAD_MNVEC, tc::LOAD_MNVEC>}};
    static bool configured_atm = false;
    if (!configured_atm) {
      for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j)
          VIHMC_CUDA_OK(cudaFuncSetAttribute(table[i][j], cudaFuncAttributeMaxDynamicSharedMemorySize, tc::SMEM_BYTES_ATM));
      configured_atm = true;
    }
    table[a_mode][b_mode]<<<grid, tc::THREADS, tc::SMEM_BYTES_ATM, st>>>(g, a_mode, b_mode);
  } else if (a_mode == tc::LOAD_KVEC && b_mode == tc::LOAD_KVEC) {
    // both operands K-contiguous and aligned (the head product, the wide-MLP layers): staging modes fixed at compile time
    auto kk = tc::tc_gemm_kernel<EPI, false, tc::LOAD_KVEC, tc::LOAD_KVEC>;
    static bool configured_kk = false;
    if (!configured_kk) {
      VIHMC_CUDA_OK(cudaFuncSetAttribute(kk, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::SMEM_BYTES));
      configured_kk = true;
    }
    kk<<<grid, tc::THREADS, tc::SMEM_BYTES, st>>>(g, a_mode, b_mode);
  } else {
    k<<<grid, tc::THREADS, tc::SMEM_BYTES, st>>>(g, a_mode, b_mode);
  }
  VIHMC_LAUNCH_OK("tc_gemm_kernel");
  if (g.splits > 1) {
    const long long total = (long long)batch * g.M * g.N;
    long long blocks = (total + 255) / 256;
    if (blocks > 148 * 8) blocks = 148 * 8;
    splitk_reduce_kernel<<<(unsigned)blocks, 256, 0, st>>>(scratch, g.splits, batch, g.M, g.N, g.C, g.c_bs, g.ldc);
    VIHMC_LAUNCH_OK("splitk_reduce_kernel");
  }
  if (fuse_rowsum) {
    rowsum_finish_kernel<<<dim3(batch, (g.M + 127) / 128), 128, 0, st>>>(rowsum_part, g.splits, batch, g.M, rowsum_out, rowsum_bs);
    VIHMC_LAUNCH_OK("rowsum_finish_kernel");
    if (rowsum_done != nullptr) *rowsum_done = 1;
  }
  return VIHMC_OK;
}

}  // namespace vihmc
