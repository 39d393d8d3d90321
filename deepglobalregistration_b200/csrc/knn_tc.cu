// Exact feature nearest neighbour with a tensor-core pre-filter (C % 32 == 0).
//
// The fp32 brute-force kernel (knn.cu) spends 2 instructions per (i, j, c) term on the fp32
// pipe.  Here the same answer - bit-identical indices - is produced in two tcgen05 sweeps:
//
//   pass 1  D = F0_tile . F1_tile^T on the tensor cores (TF32, accumulator in TMEM);
//           the epilogue (thread = F0 row = TMEM lane) forms d~2 = |a|^2 + |b|^2 - 2 D and
//           keeps the row minimum m~_i.  (Round 2 measured a pass 1 over every 8th column tile - any
//           upper bound of the minimum keeps the candidate set a superset: pass 1 fell from 0.55 to
//           0.09 ms but pass 2 grew from 0.91 to 1.68 ms on the looser bound; and 3xTF32 products
//           (kFine, a ~150x narrower band) cost more in operand staging than they save: 2.0 ms.
//           The full single-product sweep stays.  A SINGLE sweep with a running bound and a candidate buffer
//           (PASS 3 below, DGR_KNN_SWEEPS=1) is bit-identical too but measured 6.6 ms against 1.5 ms on the
//           benchmark's tightly clustered random-init features: profiles/r02_experiments.txt.)
//   pass 2  the same products again; every column with d~2 <= m~_i + 2 E_i is a CANDIDATE and
//           only candidates are evaluated with the reference arithmetic
//           (fp32 sum_c (a - b)^2 in ascending c, sqrt(d2 + 1e-7), lowest index on ties) - the
//           very code of the fp32 kernel.
//
// E_i bounds the error of d~2: operands are rounded to TF32 (relative 2^-11 each), so a dot
// product is off by at most 2^-10 |a||b| (+ accumulation slack), and d~2 by twice that.  The
// true nearest neighbour j* satisfies d~2(j*) <= d2(j*) + E <= d2(j) + E <= d~2(j) + 2E for
// every j, hence it is always among the candidates and the result equals the fp32 kernel's.
//
// FP16 operands (the default; DGR_KNN_TF32=1 selects the TF32 kernel): row i of F0 is multiplied by a power of
// two s_i, all of F1 by one power of two t, each mapping the absolute maximum into [2^14, 2^15) (exact, and below
// FP16's 65504), then rounded to FP16.  The epilogue multiplies the product by 1 / (s_i t) (exact), so estimates
// stay in the original units.  In scaled units x' = s_i a, y' = t b, rounding gives |dx'_c| <= 2^-11 |x'_c| + 2^-25
// (2^-11: FP16's unit roundoff for normal values, as TF32's; 2^-25: half the subnormal spacing 2^-24, which also
// covers values that flush to zero).  Summing over c with Cauchy-Schwarz (sum |y'_c| <= sqrt(C) |y'|):
//   |x'.y' - h(x').h(y')| <= (2^-10 + 2^-22) |x'||y'| + (2^-25 + 2^-36) sqrt(C) (|x'| + |y'|) + C 2^-50,
// and divided by s_i t:  (2^-10 + 2^-22) |a||b| + 1.001 * 2^-25 sqrt(C) (|a| / t + |b| / s_i) + C 2^-50 / (s_i t).
// The first term is the TF32 term; knn_error_bound_f16 adds the other two with |b| <= max_j |b_j|.
#include <cuda_fp16.h>
#include <stdlib.h>

#include "common.cuh"
#include "tc_common.cuh"

namespace {

using namespace tc;

constexpr int kLoadWarps = 4;
constexpr int kLoadThreads = kLoadWarps * 32;
constexpr int kMmaWarpK = kLoadWarps;
constexpr int kEpiWarps = 8;                          // two per TMEM lane group: column halves
constexpr int kThreadsK = (kLoadWarps + 1 + kEpiWarps) * 32;   // 416
constexpr int kRowsA = 128;
constexpr int kColsB = 256;
constexpr int kATile = kRowsA * 128;    // bytes per 32-float chunk
constexpr int kBTile = kColsB * 128;
constexpr int kCandCap = 16;           // single-sweep mode: buffered candidates per (row, column half)
constexpr int kEpiThreads = kEpiWarps * 32;
constexpr size_t kCandBytes = (size_t)2 * kCandCap * kEpiThreads * 4;   // column index + estimate
constexpr int kPass1Stride = 1;        // pass 1 column-tile stride (a sampled pass 1 was measured: see header)

__global__ void row_norms_kernel(const float* __restrict__ f, int64_t n, int c, float* __restrict__ n2,
                                 unsigned* __restrict__ max_bits) {
  int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 3;   // 8 lanes per row
  int sub = threadIdx.x & 7;
  float s = 0.f, amax = 0.f;
  if (row < n)
    for (int k = sub; k < c; k += 8) {
      float v = f[row * c + k];
      s = fmaf(v, v, s);
      amax = fmaxf(amax, fabsf(v));
    }
  s += __shfl_xor_sync(0xffffffffu, s, 1);
  s += __shfl_xor_sync(0xffffffffu, s, 2);
  s += __shfl_xor_sync(0xffffffffu, s, 4);
  amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, 1));
  amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, 2));
  amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, 4));
  if (row < n && sub == 0) {
    n2[row] = s;
    if (max_bits != nullptr) {
      atomicMax(max_bits, __float_as_uint(s));              // max |b|^2
      atomicMax(max_bits + 1, __float_as_uint(amax));       // max |b_c|: the FP16 pre-filter's F1 scale
    }
  }
}

__global__ void knn_tc_init_kernel(unsigned* __restrict__ rowmin_bits, unsigned long long* __restrict__ packed,
                                   int64_t n0, unsigned* max_bits) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n0) {
    rowmin_bits[i] = 0x7f800000u;
    packed[i] = ~0ull;
  }
  if (i == 0) max_bits[0] = max_bits[1] = 0u;
}

// thr_i = m~_i + 2 E_i with E_i = 2 * (dot-product error bound).
// coarse (one TF32 product): operands rounded to TF32, |a.b error| <= 2^-10 * 1.25 |a||b| (+ accumulation slack);
// fine (3xTF32, hi*hi + lo*hi + hi*lo): the dropped lo*lo term and the truncation of the lo parts are each
// <= 2^-22 |a||b|, fp32 accumulation of 32 products <= 32 * 2^-24 |a||b|: 4e-6 |a||b| covers them with margin.
// Both add the slack of the fp32 norms.
__device__ __forceinline__ float knn_error_bound(float na, float nb, bool fine) {
  const float rel = fine ? 4e-6f : (0.0009765625f * 1.25f + 4e-5f);
  return rel * na * nb + 1e-6f * (na + nb) * (na + nb) + 1e-7f;
}
// FP16 pre-filter (see the header): the same relative term, plus the absolute error of values that land in the
// FP16 subnormal range after scaling.  inv_sa, inv_sb: the (power-of-two) inverse scales of the row and of F1.
__device__ __forceinline__ float knn_error_bound_f16(float na, float nb, float inv_sa, float inv_sb, int c) {
  const float rc = sqrtf((float)c);
  return knn_error_bound(na, nb, false) + 3.1e-8f * rc * (na * inv_sb + nb * inv_sa) +
         (float)c * 1e-15f * inv_sa * inv_sb;
}
// inv_s0 != nullptr: FP16 pre-filter, per-row F0 scales inv_s0[i], F1 scale in nb2_max_bits[2]
__global__ void knn_tc_threshold_kernel(const unsigned* __restrict__ rowmin_bits, const float* __restrict__ na2,
                                        const unsigned* __restrict__ nb2_max_bits, int64_t n0, int fine,
                                        const float* __restrict__ inv_s0, int c, float* __restrict__ thr) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n0) return;
  const float na = sqrtf(na2[i]), nb = sqrtf(__uint_as_float(*nb2_max_bits));
  const float e = inv_s0 != nullptr ? knn_error_bound_f16(na, nb, inv_s0[i], __uint_as_float(nb2_max_bits[2]), c)
                                    : knn_error_bound(na, nb, fine != 0);
  // stored in the epilogue's units: candidates satisfy (0.5 |b|^2 - a.b) <= thr'
  thr[i] = 0.5f * (__uint_as_float(rowmin_bits[i]) + 4.f * e - na2[i]);
}

struct KnnShared {
  unsigned long long full[2];
  unsigned long long acc_full[2];
  unsigned long long acc_empty[2];
  uint32_t tmem_base;
  float nb[2][kColsB];
};

__device__ __forceinline__ void round_store(float4 v, unsigned char* tile, int row, int piece) {
  float4 h;
  h.x = tf32_round(v.x); h.y = tf32_round(v.y); h.z = tf32_round(v.z); h.w = tf32_round(v.w);
  *reinterpret_cast<float4*>(tile + row * 128 + ((piece ^ (row & 7)) << 4)) = h;
}

__device__ __forceinline__ void split_store2(float4 v, unsigned char* hi_tile, unsigned char* lo_tile, int row, int piece) {
  float4 h, l;
  h.x = tf32_round(v.x); h.y = tf32_round(v.y); h.z = tf32_round(v.z); h.w = tf32_round(v.w);
  l.x = v.x - h.x; l.y = v.y - h.y; l.z = v.z - h.z; l.w = v.w - h.w;
  const int off = row * 128 + ((piece ^ (row & 7)) << 4);
  *reinterpret_cast<float4*>(hi_tile + off) = h;
  *reinterpret_cast<float4*>(lo_tile + off) = l;
}

// exact reference arithmetic for one candidate column, as in knn.cu
template <int C>
__device__ __noinline__ void knn_exact_candidate(const float* __restrict__ f0, const float* __restrict__ f1,
                                                 int gi, int j, float& best_s, float& best_d2, int& best_j) {
  const float4* a = reinterpret_cast<const float4*>(f0 + (size_t)gi * C);
  const float4* b = reinterpret_cast<const float4*>(f1 + (size_t)j * C);
  float d2 = 0.f;
#pragma unroll
  for (int k = 0; k < C / 4; ++k) {
    const float4 x = __ldg(a + k), y = __ldg(b + k);
    float df = x.x - y.x; d2 = fmaf(df, df, d2);
    df = x.y - y.y; d2 = fmaf(df, df, d2);
    df = x.z - y.z; d2 = fmaf(df, df, d2);
    df = x.w - y.w; d2 = fmaf(df, df, d2);
  }
  if (d2 < best_d2) {
    const float sq = sqrtf(d2 + 1e-7f);
    if (sq < best_s) {
      best_s = sq;
      best_d2 = d2;
      best_j = j;
    }
  }
}

// the same arithmetic for candidates met in ANY order (single-sweep mode evaluates its buffered candidates after
// the sweep, overflowed ones during it): smallest sqrt distance, lowest index among equal ones - what the ascending
// walk above yields.  best_d2 is the smallest exact d2 seen; it only tightens the candidate bound.
template <int C>
__device__ __noinline__ void knn_exact_candidate_unordered(const float* __restrict__ f0, const float* __restrict__ f1,
                                                           int gi, int j, float& best_s, float& best_d2, int& best_j) {
  const float4* a = reinterpret_cast<const float4*>(f0 + (size_t)gi * C);
  const float4* b = reinterpret_cast<const float4*>(f1 + (size_t)j * C);
  float d2 = 0.f;
#pragma unroll
  for (int k = 0; k < C / 4; ++k) {
    const float4 x = __ldg(a + k), y = __ldg(b + k);
    float df = x.x - y.x; d2 = fmaf(df, df, d2);
    df = x.y - y.y; d2 = fmaf(df, df, d2);
    df = x.z - y.z; d2 = fmaf(df, df, d2);
    df = x.w - y.w; d2 = fmaf(df, df, d2);
  }
  const float sq = sqrtf(d2 + 1e-7f);
  if (sq < best_s || (sq == best_s && j < best_j)) {
    best_s = sq;
    best_j = j;
  }
  best_d2 = fminf(best_d2, d2);
}

__device__ __forceinline__ void tc_ld32_issue(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]),
        "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]),
        "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]),
        "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tc_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

template <int C, int PASS, bool kFine>
__global__ void __launch_bounds__(kThreadsK, 1)
knn_tc_kernel(const float* __restrict__ f0, int n0, const float* __restrict__ f1, int n1,
              const float* __restrict__ na2, const float* __restrict__ nb2, int cols_per_split,
              unsigned* __restrict__ rowmin_bits, const float* __restrict__ thr,
              unsigned long long* __restrict__ packed, const unsigned* __restrict__ nb2_max_bits) {
  constexpr int kChunks = C / 32;
  constexpr int kParts = kFine ? 2 : 1;            // operand tiles per chunk: TF32 hi (+ residual lo)
  extern __shared__ __align__(16) unsigned char smem_dyn[];
  KnnShared& sh = *reinterpret_cast<KnnShared*>(smem_dyn);
  unsigned char* a_tile = reinterpret_cast<unsigned char*>(
      (reinterpret_cast<uintptr_t>(smem_dyn) + sizeof(KnnShared) + 1023) & ~(uintptr_t)1023);
  unsigned char* b_stage0 = a_tile + kParts * kChunks * kATile;
  constexpr int kStageBytes = kParts * kChunks * kBTile;
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  const int row0 = blockIdx.x * kRowsA;
  const int col_begin = blockIdx.y * cols_per_split;
  const int col_end = min(n1, col_begin + cols_per_split);
  constexpr int kTS = PASS == 1 ? kPass1Stride : 1;               // tile stride of this pass
  const int n_tiles_all = (col_end - col_begin + kColsB - 1) / kColsB;
  const int n_tiles = (n_tiles_all + kTS - 1) / kTS;

  if (t == 0) {
    for (int s = 0; s < 2; ++s) {
      mbar_init(smem_u32(&sh.full[s]), kLoadThreads);
      mbar_init(smem_u32(&sh.acc_full[s]), 1);
      mbar_init(smem_u32(&sh.acc_empty[s]), kEpiWarps * 32);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == kMmaWarpK) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                     smem_u32(&sh.tmem_base)),
                 "r"(512u)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = sh.tmem_base;

  if (warp < kLoadWarps) {
    // ================================ loaders ============================================
    const int piece = t & 7, rgrp = t >> 3;   // 16 row groups
    // the F0 tile, once
#pragma unroll
    for (int ch = 0; ch < kChunks; ++ch)
#pragma unroll
      for (int i = 0; i < kRowsA / 16; ++i) {
        const int r = i * 16 + rgrp;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (row0 + r < n0) v = __ldg(reinterpret_cast<const float4*>(f0 + (size_t)(row0 + r) * C + ch * 32 + piece * 4));
        if (kFine) split_store2(v, a_tile + (2 * ch) * kATile, a_tile + (2 * ch + 1) * kATile, r, piece);
        else round_store(v, a_tile + ch * kATile, r, piece);
      }
    for (int it = 0; it < n_tiles; ++it) {
      const int s = it & 1;
      const uint32_t ph = (it >> 1) & 1;
      const int j0 = col_begin + it * kTS * kColsB;
      float4 bv[kChunks][kColsB / 16];
#pragma unroll
      for (int ch = 0; ch < kChunks; ++ch)
#pragma unroll
        for (int i = 0; i < kColsB / 16; ++i) {
          const int r = i * 16 + rgrp;
          bv[ch][i] = (j0 + r < col_end)
                          ? __ldg(reinterpret_cast<const float4*>(f1 + (size_t)(j0 + r) * C + ch * 32 + piece * 4))
                          : make_float4(0.f, 0.f, 0.f, 0.f);
        }
      const float nb_a = (j0 + t < col_end) ? nb2[j0 + t] : 0.f;
      const float nb_b = (j0 + 128 + t < col_end) ? nb2[j0 + 128 + t] : 0.f;
      // stage s (B tile + norms) and accumulator s travel together: both are free once the
      // epilogue has drained accumulator s of tile it - 2
      mbar_wait(smem_u32(&sh.acc_empty[s]), ph ^ 1);
      unsigned char* b_tile = b_stage0 + (size_t)s * kStageBytes;
#pragma unroll
      for (int ch = 0; ch < kChunks; ++ch)
#pragma unroll
        for (int i = 0; i < kColsB / 16; ++i) {
          if (kFine) split_store2(bv[ch][i], b_tile + (2 * ch) * kBTile, b_tile + (2 * ch + 1) * kBTile, i * 16 + rgrp, piece);
          else round_store(bv[ch][i], b_tile + ch * kBTile, i * 16 + rgrp, piece);
        }
      sh.nb[s][t] = 0.5f * nb_a;          // the epilogue works with 0.5 |b|^2 - a.b
      sh.nb[s][128 + t] = 0.5f * nb_b;
      fence_proxy_async();
      mbar_arrive(smem_u32(&sh.full[s]));
    }
  } else if (warp == kMmaWarpK) {
    // ================================ MMA issuer =========================================
    const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(kColsB >> 3) << 17) |
                           ((uint32_t)(kRowsA >> 4) << 24);
    for (int it = 0; it < n_tiles; ++it) {
      const int s = it & 1;
      const uint32_t ph = (it >> 1) & 1;
      mbar_wait(smem_u32(&sh.acc_empty[s]), ph ^ 1);
      mbar_wait(smem_u32(&sh.full[s]), ph);
      tc_fence_after();
      if (lane == 0) {
        const uint32_t a0 = smem_u32(a_tile);
        const uint32_t b0 = smem_u32(b_stage0 + (size_t)s * kStageBytes);
#pragma unroll
        for (int ch = 0; ch < kChunks; ++ch)
#pragma unroll
          for (int ks = 0; ks < 4; ++ks) {
            const uint32_t td = tmem_base + (uint32_t)s * kColsB;
            if (kFine) {
              const uint64_t ah = umma_desc(a0 + (2 * ch) * kATile + ks * 32), al = umma_desc(a0 + (2 * ch + 1) * kATile + ks * 32);
              const uint64_t bh = umma_desc(b0 + (2 * ch) * kBTile + ks * 32), bl = umma_desc(b0 + (2 * ch + 1) * kBTile + ks * 32);
              tc_mma_tf32(td, ah, bh, idesc, (ch | ks) != 0);
              tc_mma_tf32(td, al, bh, idesc, 1);
              tc_mma_tf32(td, ah, bl, idesc, 1);
            } else {
              tc_mma_tf32(td, umma_desc(a0 + ch * kATile + ks * 32), umma_desc(b0 + ch * kBTile + ks * 32), idesc,
                          (ch | ks) != 0);
            }
          }
        tc_commit(smem_u32(&sh.acc_full[s]));
      }
      __syncwarp();
    }
  } else if (PASS == 3) {
    // ================================ single sweep: thread = (F0 row, column half) ========
    // One pass over the products.  The candidate bound follows the RUNNING row minimum of this thread's columns
    // (any upper bound of the final minimum keeps the candidate set a superset, see the header): columns within the
    // bound are buffered in shared memory (column, estimate) and evaluated exactly after the sweep against the
    // final - tightest - bound; a full buffer evaluates the newcomer on the spot.
    const int lane_grp = warp & 3;
    const int half = (warp - kLoadWarps - 1) >> 2;
    const int gi = row0 + lane_grp * 32 + lane;
    const bool valid = gi < n0;
    const int etid = (warp - kLoadWarps - 1) * 32 + lane;                  // 0 .. kEpiThreads-1
    int* cand_j = reinterpret_cast<int*>(b_stage0 + 2 * (size_t)kStageBytes) + etid;       // [slot][thread]
    float* cand_g = reinterpret_cast<float*>(cand_j - etid + kCandCap * kEpiThreads) + etid;
    const float ninf = -__int_as_float(0x7f800000), pinf = __int_as_float(0x7f800000);
    const float na2_i = valid ? na2[gi] : 0.f;
    const float e4 = valid ? 4.f * knn_error_bound(sqrtf(na2_i), sqrtf(__uint_as_float(*nb2_max_bits)), kFine) : 0.f;
    float rmin = pinf, th_exact = pinf;
    float best_s = pinf, best_d2 = pinf;
    int best_j = 0x7fffffff, cnt = 0;
    // bound in the epilogue's units (0.5 |b|^2 - a.b), from the running minimum: thr kernel's formula
    auto bound = [&](float m) { return 0.5f * (fmaxf(fmaf(2.f, m, na2_i), 0.f) + e4 - na2_i); };
    auto take = [&](int j, float g) {
      if (cnt < kCandCap) {
        cand_j[cnt * kEpiThreads] = j;
        cand_g[cnt * kEpiThreads] = g;
        ++cnt;
      } else {
        knn_exact_candidate_unordered<C>(f0, f1, gi, j, best_s, best_d2, best_j);
        th_exact = fminf(th_exact, 0.5f * (best_d2 + e4 - na2_i));
      }
    };
    for (int it = 0; it < n_tiles; ++it) {
      const int s = it & 1;
      const uint32_t ph = (it >> 1) & 1;
      const int j0 = col_begin + it * kColsB + half * 128;
      mbar_wait(smem_u32(&sh.acc_full[s]), ph);
      tc_fence_after();
      const uint32_t taddr = tmem_base + (uint32_t)s * kColsB + half * 128 + ((uint32_t)(lane_grp * 32) << 16);
      const float* hb = sh.nb[s] + half * 128;
      uint32_t va[32], vb[32];
      tc_ld32_issue(taddr, va);
#pragma unroll
      for (int cc = 0; cc < 4; ++cc) {
        tc_ld_wait();
        uint32_t(&cur)[32] = (cc & 1) ? vb : va;
        uint32_t(&nxt)[32] = (cc & 1) ? va : vb;
        if (cc < 3) tc_ld32_issue(taddr + (cc + 1) * 32, nxt);
        const int jc = j0 + cc * 32;
        if (jc < col_end) {
          const int nq = min(32, col_end - jc);
          float cmin = pinf;
#pragma unroll
          for (int q = 0; q < 32; ++q)
            cmin = fminf(cmin, q < nq ? hb[cc * 32 + q] - __uint_as_float(cur[q]) : pinf);
          rmin = fminf(rmin, cmin);
          float th = valid ? fminf(th_exact, bound(rmin)) : ninf;
          if (cmin <= th) {
#pragma unroll
            for (int q = 0; q < 32; ++q) {
              const float g = hb[cc * 32 + q] - __uint_as_float(cur[q]);
              if (q < nq && g <= th) {
                take(jc + q, g);
                th = fminf(th, th_exact);
              }
            }
          }
        }
      }
      tc_fence_before();
      mbar_arrive(smem_u32(&sh.acc_empty[s]));
    }
    if (valid) {
      float th = fminf(th_exact, bound(rmin));
      for (int k = 0; k < cnt; ++k) {
        if (cand_g[k * kEpiThreads] <= th) {
          knn_exact_candidate_unordered<C>(f0, f1, gi, cand_j[k * kEpiThreads], best_s, best_d2, best_j);
          th = fminf(th, 0.5f * (best_d2 + e4 - na2_i));
        }
      }
      if (best_j != 0x7fffffff)
        atomicMin(packed + gi, ((unsigned long long)__float_as_uint(best_s) << 32) | (unsigned)best_j);
    }
  } else {
    // ================================ epilogue: thread = (F0 row, column half) ============
    const int lane_grp = warp & 3;
    const int half = (warp - kLoadWarps - 1) >> 2;      // 0: columns 0..127, 1: columns 128..255
    const int r = lane_grp * 32 + lane;
    const int gi = row0 + r;
    const bool valid = gi < n0;
    float th = (PASS == 2 && valid) ? thr[gi] : -__int_as_float(0x7f800000);
    // pass 2 tightens its bound with every exact distance it learns: a later column can only win if its true
    // d2 is below the best exact d2 so far, i.e. if its estimate is below best_d2 + (estimate error)
    const float na2_i = (PASS == 2 && valid) ? na2[gi] : 0.f;
    const float e4 = (PASS == 2 && valid)
                         ? 4.f * knn_error_bound(sqrtf(na2_i), sqrtf(__uint_as_float(*nb2_max_bits)), kFine)
                         : 0.f;
    float rmin = __int_as_float(0x7f800000);     // min over columns of 0.5 |b|^2 - a.b
    float best_s = __int_as_float(0x7f800000), best_d2 = best_s;
    int best_j = 0x7fffffff;
    for (int it = 0; it < n_tiles; ++it) {
      const int s = it & 1;
      const uint32_t ph = (it >> 1) & 1;
      const int j0 = col_begin + it * kTS * kColsB + half * 128;
      mbar_wait(smem_u32(&sh.acc_full[s]), ph);
      tc_fence_after();
      const uint32_t taddr = tmem_base + (uint32_t)s * kColsB + half * 128 + ((uint32_t)(lane_grp * 32) << 16);
      const float* hb = sh.nb[s] + half * 128;
      uint32_t va[32], vb[32];
      tc_ld32_issue(taddr, va);
#pragma unroll
      for (int cc = 0; cc < 4; ++cc) {
        tc_ld_wait();
        uint32_t(&cur)[32] = (cc & 1) ? vb : va;
        uint32_t(&nxt)[32] = (cc & 1) ? va : vb;
        if (cc < 3) tc_ld32_issue(taddr + (cc + 1) * 32, nxt);
        const int jc = j0 + cc * 32;
        if (jc < col_end) {
          if (jc + 32 <= col_end) {
            // both passes reduce the chunk to its minimum first (branch-free); pass 2 walks the
            // chunk element by element only when that minimum is within the candidate bound
            float cmin = __int_as_float(0x7f800000);
#pragma unroll
            for (int q = 0; q < 32; ++q) cmin = fminf(cmin, hb[cc * 32 + q] - __uint_as_float(cur[q]));
            if (PASS == 1) {
              rmin = fminf(rmin, cmin);
            } else if (cmin <= th) {
#pragma unroll
              for (int q = 0; q < 32; ++q) {
                const float g = hb[cc * 32 + q] - __uint_as_float(cur[q]);
                if (g <= th) {
                  knn_exact_candidate<C>(f0, f1, gi, jc + q, best_s, best_d2, best_j);
                  th = fminf(th, 0.5f * (best_d2 + e4 - na2_i));
                }
              }
            }
          } else {
#pragma unroll
            for (int q = 0; q < 32; ++q) {
              const float g = hb[cc * 32 + q] - __uint_as_float(cur[q]);
              if (jc + q < col_end) {
                if (PASS == 1) rmin = fminf(rmin, g);
                else if (g <= th) {
                  knn_exact_candidate<C>(f0, f1, gi, jc + q, best_s, best_d2, best_j);
                  th = fminf(th, 0.5f * (best_d2 + e4 - na2_i));
                }
              }
            }
          }
        }
      }
      tc_fence_before();
      mbar_arrive(smem_u32(&sh.acc_empty[s]));
    }
    if (valid) {
      if (PASS == 1) {
        atomicMin(rowmin_bits + gi, __float_as_uint(fmaxf(fmaf(2.f, rmin, na2[gi]), 0.f)));
      } else if (best_j != 0x7fffffff) {
        atomicMin(packed + gi, ((unsigned long long)__float_as_uint(best_s) << 32) | (unsigned)best_j);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kMmaWarpK) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
  }
}

// ================================ FP16 pre-filter (default) ==========================================
// Operands are packed once per call into FP16 SWIZZLE_128B images (knn_pack_f16_kernel) and bulk-copied into a
// ring of shared-memory stages by one thread; the grid is persistent: CTA b walks a contiguous range of
// (row tile, column tile) work items, so every SM is busy to the end and TMEM is allocated once per CTA.
// A CTA tile is 256 F0 rows (two M = 128 products sharing each B tile) x 128 F1 columns.
constexpr int kRowsH = 256;
constexpr int kColsH = 128;
constexpr int kStagesH = 6;
constexpr int kAImgH = kRowsH * 128;     // bytes: 128-byte rows, 64 halves (C = 32: halves 32..63 are zero)
constexpr int kBImgH = kColsH * 128;
constexpr int kThreadsH = (2 + kEpiWarps) * 32;     // producer warp, MMA warp, 8 epilogue warps

struct KnnSharedH {
  float nb[kStagesH][kColsH];            // 0.5 |b|^2 of the stage's columns (bulk-copied, first: 16-byte aligned)
  unsigned long long full[kStagesH];     // B stage landed (tx bytes)
  unsigned long long empty[kStagesH];    // B stage drained by the epilogue (its MMAs completed before that)
  unsigned long long a_full[2], a_empty[2];
  unsigned long long acc_full[2], acc_empty[2];
  uint32_t tmem_base;
};

// One row per 8 threads, one 16-byte piece (8 halves) per thread, written at its swizzled position:
// row r at r * 128 bytes, piece p at (p ^ (r & 7)) * 16 - the K-major SWIZZLE_128B image of umma_desc.
// amax_bits == nullptr: per-row scale (F0), inv_scale[row] = 1 / scale; otherwise one scale for all rows
// (F1), stored in inv_scale[0], and nbh[row] = 0.5 |b|^2 (+inf for padding rows: never a minimum).
template <int C>
__global__ void knn_pack_f16_kernel(const float* __restrict__ f, int64_t n, int64_t n_pad,
                                    const unsigned* __restrict__ amax_bits, float* __restrict__ inv_scale,
                                    const float* __restrict__ n2, float* __restrict__ nbh, uint4* __restrict__ img) {
  const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 3;
  const int p = threadIdx.x & 7;
  if (row >= n_pad) return;                 // n_pad % 4 == 0: whole warps leave
  float x[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (row < n && p * 8 < C) {
    const float4 u = __ldg(reinterpret_cast<const float4*>(f + row * C + p * 8));
    const float4 v = __ldg(reinterpret_cast<const float4*>(f + row * C + p * 8 + 4));
    x[0] = u.x; x[1] = u.y; x[2] = u.z; x[3] = u.w; x[4] = v.x; x[5] = v.y; x[6] = v.z; x[7] = v.w;
  }
  float am;
  if (amax_bits == nullptr) {
    am = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) am = fmaxf(am, fabsf(x[k]));
    am = fmaxf(am, __shfl_xor_sync(0xffffffffu, am, 1));
    am = fmaxf(am, __shfl_xor_sync(0xffffffffu, am, 2));
    am = fmaxf(am, __shfl_xor_sync(0xffffffffu, am, 4));
  } else {
    am = __uint_as_float(*amax_bits);
  }
  const float sc = f16_scale_for(am);       // a power of two: x * sc is exact
  uint32_t h[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const __half2 hh = __floats2half2_rn(x[2 * k] * sc, x[2 * k + 1] * sc);
    h[k] = *reinterpret_cast<const uint32_t*>(&hh);
  }
  img[row * 8 + (p ^ (int)(row & 7))] = make_uint4(h[0], h[1], h[2], h[3]);
  if (p == 0) {
    if (amax_bits == nullptr) {
      inv_scale[row] = 1.f / sc;
    } else {
      if (row == 0) inv_scale[0] = 1.f / sc;
      nbh[row] = row < n ? 0.5f * n2[row] : __int_as_float(0x7f800000);
    }
  }
}

template <int C, int PASS>
__global__ void __launch_bounds__(kThreadsH, 1)
knn_f16_kernel(const unsigned char* __restrict__ a_img, const unsigned char* __restrict__ b_img,
               const float* __restrict__ nbh, int n0, int n1, int n_ct, int64_t n_units,
               const float* __restrict__ f0, const float* __restrict__ f1, const float* __restrict__ na2,
               const float* __restrict__ inv_s0, const unsigned* __restrict__ max_bits,
               unsigned* __restrict__ rowmin_bits, const float* __restrict__ thr,
               unsigned long long* __restrict__ packed) {
  extern __shared__ __align__(16) unsigned char smem_dyn[];
  KnnSharedH& sh = *reinterpret_cast<KnnSharedH*>(smem_dyn);
  unsigned char* a_buf = reinterpret_cast<unsigned char*>(
      (reinterpret_cast<uintptr_t>(smem_dyn) + sizeof(KnnSharedH) + 1023) & ~(uintptr_t)1023);
  unsigned char* b_buf = a_buf + 2 * kAImgH;
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  const int64_t u_begin = (int64_t)blockIdx.x * n_units / gridDim.x;
  const int64_t u_end = (int64_t)(blockIdx.x + 1) * n_units / gridDim.x;

  if (t == 0) {
    for (int s = 0; s < kStagesH; ++s) {
      mbar_init(smem_u32(&sh.full[s]), 1);
      mbar_init(smem_u32(&sh.empty[s]), kEpiWarps * 32);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(smem_u32(&sh.a_full[b]), 1);
      mbar_init(smem_u32(&sh.a_empty[b]), 1);
      mbar_init(smem_u32(&sh.acc_full[b]), 1);
      mbar_init(smem_u32(&sh.acc_empty[b]), kEpiWarps * 32);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                     smem_u32(&sh.tmem_base)),
                 "r"(512u)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = sh.tmem_base;

  if (warp == 0) {
    // ================================ producer: one thread, bulk copies ===================
    if (lane == 0) {
      int it = 0, seg = 0;
      for (int64_t u = u_begin; u < u_end; ++u, ++it) {
        const int rt = (int)(u / n_ct), ct = (int)(u % n_ct);
        if (u == u_begin || ct == 0) {       // a new row tile: the other A buffer, once its products are done
          const int a = seg & 1;
          mbar_wait(smem_u32(&sh.a_empty[a]), ((seg >> 1) & 1) ^ 1);
          mbar_arrive_expect_tx(smem_u32(&sh.a_full[a]), kAImgH);
          bulk_g2s(smem_u32(a_buf + a * kAImgH), a_img + (size_t)rt * kAImgH, kAImgH, smem_u32(&sh.a_full[a]));
          ++seg;
        }
        const int s = it % kStagesH;
        mbar_wait(smem_u32(&sh.empty[s]), ((it / kStagesH) & 1) ^ 1);
        mbar_arrive_expect_tx(smem_u32(&sh.full[s]), kBImgH + kColsH * 4);
        bulk_g2s(smem_u32(b_buf + s * kBImgH), b_img + (size_t)ct * kBImgH, kBImgH, smem_u32(&sh.full[s]));
        bulk_g2s(smem_u32(sh.nb[s]), nbh + (size_t)ct * kColsH, kColsH * 4, smem_u32(&sh.full[s]));
      }
    }
  } else if (warp == 1) {
    // ================================ MMA issuer ==========================================
    // D = F32, A = B = F16, both K-major, N = 128, M = 128; K = 16 halves (32 bytes) per instruction
    const uint32_t idesc = (1u << 4) | ((uint32_t)(kColsH >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
    int it = 0, seg = 0, a = 0;
    for (int64_t u = u_begin; u < u_end; ++u, ++it) {
      const int ct = (int)(u % n_ct);
      if (u == u_begin || ct == 0) {
        a = seg & 1;
        mbar_wait(smem_u32(&sh.a_full[a]), (seg >> 1) & 1);
        ++seg;
      }
      const int b = it & 1, s = it % kStagesH;
      mbar_wait(smem_u32(&sh.acc_empty[b]), ((it >> 1) & 1) ^ 1);
      mbar_wait(smem_u32(&sh.full[s]), (it / kStagesH) & 1);
      tc_fence_after();
      if (lane == 0) {
        const uint32_t a0 = smem_u32(a_buf + a * kAImgH), b0 = smem_u32(b_buf + s * kBImgH);
        const uint32_t td = tmem_base + (uint32_t)b * 256;
#pragma unroll
        for (int ks = 0; ks < C / 16; ++ks) {
          const uint64_t bd = umma_desc(b0 + ks * 32);
          tc_mma_f16(td, umma_desc(a0 + ks * 32), bd, idesc, ks != 0);                      // rows 0..127
          tc_mma_f16(td + 128, umma_desc(a0 + kAImgH / 2 + ks * 32), bd, idesc, ks != 0);   // rows 128..255
        }
        tc_commit(smem_u32(&sh.acc_full[b]));
        if (u + 1 == u_end || ct == n_ct - 1) tc_commit(smem_u32(&sh.a_empty[a]));   // last tile of this A
      }
      __syncwarp();
    }
  } else {
    // ================================ epilogue: thread = F0 row ===========================
    const int lane_grp = warp & 3;                // TMEM lanes this warp may read
    const int mh = (warp - 2) >> 2;               // 0: rows 0..127 of the tile, 1: rows 128..255
    const int r = mh * 128 + lane_grp * 32 + lane;
    const float pinf = __int_as_float(0x7f800000);
    const float inv_s1 = __uint_as_float(max_bits[2]);
    const float nb_max = sqrtf(__uint_as_float(max_bits[0]));
    int gi = 0;
    bool valid = false;
    float inv = 0.f, th = -pinf, na2_i = 0.f, e4 = 0.f, rmin = pinf, best_s = pinf, best_d2 = pinf;
    int best_j = 0x7fffffff;
    int it = 0;
    for (int64_t u = u_begin; u < u_end; ++u, ++it) {
      const int rt = (int)(u / n_ct), ct = (int)(u % n_ct);
      if (u == u_begin || ct == 0) {
        gi = rt * kRowsH + r;
        valid = gi < n0;
        // D * inv is the product in the original units (inv: a power of two, the multiplication is exact)
        inv = valid ? inv_s0[gi] * inv_s1 : 0.f;
        rmin = pinf; best_s = pinf; best_d2 = pinf; best_j = 0x7fffffff;
        if (PASS == 2) {
          th = valid ? thr[gi] : -pinf;
          // pass 2 tightens its bound with every exact distance it learns (see the TF32 kernel)
          na2_i = valid ? na2[gi] : 0.f;
          e4 = valid ? 4.f * knn_error_bound_f16(sqrtf(na2_i), nb_max, inv_s0[gi], inv_s1, C) : 0.f;
        }
      }
      const int b = it & 1, s = it % kStagesH;
      mbar_wait(smem_u32(&sh.acc_full[b]), (it >> 1) & 1);
      mbar_wait(smem_u32(&sh.full[s]), (it / kStagesH) & 1);     // the norms' bulk copy
      tc_fence_after();
      const uint32_t taddr = tmem_base + (uint32_t)b * 256 + mh * 128 + ((uint32_t)(lane_grp * 32) << 16);
      const float4* hb = reinterpret_cast<const float4*>(sh.nb[s]);
      const int j0 = ct * kColsH;
      uint32_t va[32], vb[32];
      tc_ld32_issue(taddr, va);
#pragma unroll
      for (int cc = 0; cc < 4; ++cc) {
        tc_ld_wait();
        uint32_t(&cur)[32] = (cc & 1) ? vb : va;
        uint32_t(&nxt)[32] = (cc & 1) ? va : vb;
        if (cc < 3) tc_ld32_issue(taddr + (cc + 1) * 32, nxt);
        const int jc = j0 + cc * 32;
        if (jc < n1) {
          float g[32];
#pragma unroll
          for (int q4 = 0; q4 < 8; ++q4) {
            const float4 h4 = hb[cc * 8 + q4];
            g[4 * q4 + 0] = fmaf(-__uint_as_float(cur[4 * q4 + 0]), inv, h4.x);
            g[4 * q4 + 1] = fmaf(-__uint_as_float(cur[4 * q4 + 1]), inv, h4.y);
            g[4 * q4 + 2] = fmaf(-__uint_as_float(cur[4 * q4 + 2]), inv, h4.z);
            g[4 * q4 + 3] = fmaf(-__uint_as_float(cur[4 * q4 + 3]), inv, h4.w);
          }
          float cmin = pinf;
#pragma unroll
          for (int q = 0; q < 32; ++q) cmin = fminf(cmin, g[q]);
          if (PASS == 1) {
            rmin = fminf(rmin, cmin);
          } else if (cmin <= th) {
            const int nq = min(32, n1 - jc);
#pragma unroll
            for (int q = 0; q < 32; ++q) {
              if (q < nq && g[q] <= th) {
                knn_exact_candidate<C>(f0, f1, gi, jc + q, best_s, best_d2, best_j);
                th = fminf(th, 0.5f * (best_d2 + e4 - na2_i));
              }
            }
          }
        }
      }
      tc_fence_before();
      mbar_arrive(smem_u32(&sh.acc_empty[b]));
      mbar_arrive(smem_u32(&sh.empty[s]));
      if (valid && (u + 1 == u_end || ct == n_ct - 1)) {     // last column tile of this row tile in this CTA
        if (PASS == 1) atomicMin(rowmin_bits + gi, __float_as_uint(fmaxf(fmaf(2.f, rmin, na2[gi]), 0.f)));
        else if (best_j != 0x7fffffff)
          atomicMin(packed + gi, ((unsigned long long)__float_as_uint(best_s) << 32) | (unsigned)best_j);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
  }
}

__global__ void knn_tc_unpack_kernel(const unsigned long long* __restrict__ packed, int64_t n,
                                     int32_t* __restrict__ idx, float* __restrict__ dist) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  unsigned long long p = packed[i];
  idx[i] = (int32_t)(p & 0xffffffffu);
  if (dist != nullptr) dist[i] = __uint_as_float((unsigned)(p >> 32));
}

// Workspace of dgr_knn_top1_tc, in floats.  The first 3 n0 + n1 + 8 are used by both pre-filters; the FP16 one
// adds the operand images and per-row scales, each at a 256-byte boundary (bulk-copy sources need 16).
struct KnnWs {
  int64_t n0p, n1p, base, inv_s0, nbh, a_img, b_img, total;
  KnnWs(int64_t n0, int64_t n1) {
    n0p = (n0 + kRowsH - 1) / kRowsH * kRowsH;
    n1p = (n1 + kColsH - 1) / kColsH * kColsH;
    base = (3 * n0 + n1 + 8 + 63) / 64 * 64;
    inv_s0 = base;
    nbh = inv_s0 + n0p;
    a_img = nbh + n1p;
    b_img = a_img + n0p * 32;        // 128 bytes per row
    total = b_img + n1p * 32;
  }
};

int sm_count() {
  int dev = 0, n = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess)
    return 148;
  return n;
}

template <int C>
int32_t launch_knn_f16(const float* f0, int64_t n0, const float* f1, int64_t n1, float* ws, unsigned* rowmin,
                       float* thr, unsigned* max_bits, unsigned long long* packed, cudaStream_t st) {
  const KnnWs w(n0, n1);
  float* na2 = ws;
  float* nb2 = ws + 3 * n0;
  float* inv_s0 = ws + w.inv_s0;
  float* nbh = ws + w.nbh;
  unsigned char* a_img = reinterpret_cast<unsigned char*>(ws + w.a_img);
  unsigned char* b_img = reinterpret_cast<unsigned char*>(ws + w.b_img);
  knn_pack_f16_kernel<C><<<dgr_blocks(w.n0p * 8, 256), 256, 0, st>>>(f0, n0, w.n0p, nullptr, inv_s0, nullptr, nullptr,
                                                                       reinterpret_cast<uint4*>(a_img));
  knn_pack_f16_kernel<C><<<dgr_blocks(w.n1p * 8, 256), 256, 0, st>>>(
      f1, n1, w.n1p, max_bits + 1, reinterpret_cast<float*>(max_bits + 2), nb2, nbh, reinterpret_cast<uint4*>(b_img));
  const size_t smem = sizeof(KnnSharedH) + 1024 + 2 * (size_t)kAImgH + (size_t)kStagesH * kBImgH;
  DGR_ENSURE_SMEM((knn_f16_kernel<C, 1>), smem);
  DGR_ENSURE_SMEM((knn_f16_kernel<C, 2>), smem);
  const int n_ct = (int)(w.n1p / kColsH);
  const int64_t n_units = (w.n0p / kRowsH) * n_ct;
  static const int n_sm = sm_count();
  const int grid = (int)(n_units < n_sm ? n_units : n_sm);
  knn_f16_kernel<C, 1><<<grid, kThreadsH, smem, st>>>(a_img, b_img, nbh, (int)n0, (int)n1, n_ct, n_units, f0, f1, na2,
                                                      inv_s0, max_bits, rowmin, thr, packed);
  knn_tc_threshold_kernel<<<dgr_blocks(n0, 256), 256, 0, st>>>(rowmin, na2, max_bits, n0, 0, inv_s0, C, thr);
  knn_f16_kernel<C, 2><<<grid, kThreadsH, smem, st>>>(a_img, b_img, nbh, (int)n0, (int)n1, n_ct, n_units, f0, f1, na2,
                                                      inv_s0, max_bits, rowmin, thr, packed);
  return DGR_OK;
}

// single sweep (DGR_KNN_SWEEPS=1): no row-minimum pass, no threshold kernel
template <int C>
int32_t launch_knn_tc_single(const float* f0, int64_t n0, const float* f1, int64_t n1, float* na2, float* nb2,
                             unsigned* max_bits, unsigned long long* packed, cudaStream_t st) {
  constexpr int kChunks = C / 32;
  const size_t smem = sizeof(KnnShared) + 1024 + (size_t)kChunks * kATile + 2 * (size_t)kChunks * kBTile + kCandBytes;
  DGR_ENSURE_SMEM((knn_tc_kernel<C, 3, false>), smem);
  const int row_tiles = (int)((n0 + kRowsA - 1) / kRowsA);
  const int col_tiles = (int)((n1 + kColsB - 1) / kColsB);
  int splits = (148 * 4 + row_tiles - 1) / row_tiles;
  if (splits > col_tiles) splits = col_tiles;
  if (splits < 1) splits = 1;
  const int cols_per_split = ((col_tiles + splits - 1) / splits) * kColsB;
  splits = (int)((n1 + cols_per_split - 1) / cols_per_split);
  dim3 grid(row_tiles, splits);
  knn_tc_kernel<C, 3, false><<<grid, kThreadsK, smem, st>>>(f0, (int)n0, f1, (int)n1, na2, nb2, cols_per_split,
                                                            nullptr, nullptr, packed, max_bits);
  return DGR_OK;
}

template <int C, bool kFine>
int32_t launch_knn_tc(const float* f0, int64_t n0, const float* f1, int64_t n1, float* na2, float* nb2,
                      unsigned* rowmin, float* thr, unsigned* max_bits, unsigned long long* packed,
                      cudaStream_t st) {
  constexpr int kChunks = C / 32;
  constexpr int kParts = kFine ? 2 : 1;
  const size_t smem = sizeof(KnnShared) + 1024 + (size_t)kParts * kChunks * kATile + 2 * (size_t)kParts * kChunks * kBTile;
  DGR_ENSURE_SMEM((knn_tc_kernel<C, 1, kFine>), smem);
  DGR_ENSURE_SMEM((knn_tc_kernel<C, 2, kFine>), smem);
  const int row_tiles = (int)((n0 + kRowsA - 1) / kRowsA);
  const int col_tiles = (int)((n1 + kColsB - 1) / kColsB);
  int splits = (148 * 4 + row_tiles - 1) / row_tiles;
  if (splits > col_tiles) splits = col_tiles;
  if (splits < 1) splits = 1;
  const int cols_per_split = ((col_tiles + splits - 1) / splits) * kColsB;
  splits = (int)((n1 + cols_per_split - 1) / cols_per_split);
  dim3 grid(row_tiles, splits);
  knn_tc_kernel<C, 1, kFine><<<grid, kThreadsK, smem, st>>>(f0, (int)n0, f1, (int)n1, na2, nb2, cols_per_split,
                                                            rowmin, thr, packed, max_bits);
  knn_tc_threshold_kernel<<<dgr_blocks(n0, 256), 256, 0, st>>>(rowmin, na2, max_bits, n0, kFine ? 1 : 0, nullptr,
                                                               C, thr);
  knn_tc_kernel<C, 2, kFine><<<grid, kThreadsK, smem, st>>>(f0, (int)n0, f1, (int)n1, na2, nb2, cols_per_split,
                                                            rowmin, thr, packed, max_bits);
  return DGR_OK;
}

}  // namespace

extern "C" {

// floats of workspace dgr_knn_top1_tc needs
int64_t dgr_knn_tc_ws_elems(int64_t n0, int64_t n1) { return KnnWs(n0, n1).total; }

// 1 if the tensor-core pre-filter supports the channel count
int32_t dgr_knn_tc_supported(int32_t c) { return (c == 32 || c == 64) ? 1 : 0; }

// Same result as dgr_knn_top1 (bit-identical indices and distances), two tcgen05 sweeps
// plus exact fp32 evaluation of the few candidates per row.  ws: dgr_knn_tc_ws_elems floats.
int32_t dgr_knn_top1_tc(const float* f0, int64_t n0, const float* f1, int64_t n1, int32_t c,
                        uint64_t* packed_ws, float* ws, int32_t* idx, float* dist, void* stream) {
  DGR_ARG_CHECK(dgr_knn_tc_supported(c), "channel count not supported by the tensor-core kNN");
  DGR_ARG_CHECK(n1 >= 1 || n0 == 0, "F1 must not be empty");
  DGR_ARG_CHECK(n0 < (1ll << 31) && n1 < (1ll << 31), "too many rows");
  if (n0 == 0) return DGR_OK;
  cudaStream_t st = (cudaStream_t)stream;
  float* na2 = ws;
  float* thr = ws + n0;
  unsigned* rowmin = reinterpret_cast<unsigned*>(ws + 2 * n0);
  float* nb2 = ws + 3 * n0;
  unsigned* max_bits = reinterpret_cast<unsigned*>(ws + 3 * n0 + n1);
  unsigned long long* packed = reinterpret_cast<unsigned long long*>(packed_ws);
  knn_tc_init_kernel<<<dgr_blocks(n0, 256), 256, 0, st>>>(rowmin, packed, n0, max_bits);
  row_norms_kernel<<<dgr_blocks(n0 * 8, 256), 256, 0, st>>>(f0, n0, c, na2, nullptr);
  row_norms_kernel<<<dgr_blocks(n1 * 8, 256), 256, 0, st>>>(f1, n1, c, nb2, max_bits);
  // default: the FP16 pre-filter.  DGR_KNN_TF32=1: the TF32 kernel it replaced, read on every call so that
  // both can be timed in one process
  const char* tf32_env = getenv("DGR_KNN_TF32");
  const bool tf32 = tf32_env != nullptr && atoi(tf32_env) == 1;
  if (!tf32) {
    int32_t rc = (c == 32) ? launch_knn_f16<32>(f0, n0, f1, n1, ws, rowmin, thr, max_bits, packed, st)
                           : launch_knn_f16<64>(f0, n0, f1, n1, ws, rowmin, thr, max_bits, packed, st);
    if (rc != DGR_OK) return rc;
    knn_tc_unpack_kernel<<<dgr_blocks(n0, 256), 256, 0, st>>>(packed, n0, idx, dist);
    dgr_note_launches(9);
    DGR_LAUNCH_CHECK();
    return DGR_OK;
  }
  // DGR_KNN_TF32=1 only: DGR_KNN_FINE=1 (c = 32 only): 3xTF32 products, a ~150x narrower
  // candidate band, measured slower (the hi + lo tiles double the operand staging)
  static const bool coarse = getenv("DGR_KNN_FINE") == nullptr;        // A/B switch: 3xTF32 pre-filter (slower)
  // DGR_KNN_SWEEPS=1: the single-sweep variant (running bound + candidate buffer)
  static const bool single = getenv("DGR_KNN_SWEEPS") != nullptr && atoi(getenv("DGR_KNN_SWEEPS")) == 1;
  if (single) {
    int32_t rc1 = (c == 32) ? launch_knn_tc_single<32>(f0, n0, f1, n1, na2, nb2, max_bits, packed, st)
                            : launch_knn_tc_single<64>(f0, n0, f1, n1, na2, nb2, max_bits, packed, st);
    if (rc1 != DGR_OK) return rc1;
    knn_tc_unpack_kernel<<<dgr_blocks(n0, 256), 256, 0, st>>>(packed, n0, idx, dist);
    dgr_note_launches(5);
    DGR_LAUNCH_CHECK();
    return DGR_OK;
  }
  int32_t rc = (c == 32) ? (coarse ? launch_knn_tc<32, false>(f0, n0, f1, n1, na2, nb2, rowmin, thr, max_bits, packed, st)
                                   : launch_knn_tc<32, true>(f0, n0, f1, n1, na2, nb2, rowmin, thr, max_bits, packed, st))
                         : launch_knn_tc<64, false>(f0, n0, f1, n1, na2, nb2, rowmin, thr, max_bits, packed, st);
  if (rc != DGR_OK) return rc;
  knn_tc_unpack_kernel<<<dgr_blocks(n0, 256), 256, 0, st>>>(packed, n0, idx, dist);
  dgr_note_launches(7);
  DGR_LAUNCH_CHECK();
  return DGR_OK;
}

}  // extern "C"
