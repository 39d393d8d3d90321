// Sparse convolution forward on the 5th-generation tensor cores (tcgen05, sm_100a).
//
// Same contract as dgr_spconv_fwd (gather -> per-offset sub-GEMM -> scatter-add over the
// (kappa, j)-sorted pair lists) with the sub-GEMM issued as tcgen05.mma kind::tf32 and the
// accumulator in tensor memory:
//
//   * one work item = one 128-pair tile of one kernel offset, M = 128 rows (pairs),
//     N = cout (16..256), K = cin in chunks of 32 floats (one 128-byte swizzle row);
//   * 8 loader warps gather the 128 input rows (coalesced 16-byte pieces, 8 lanes per row,
//     prefetched one chunk ahead), split every fp32 value into a TF32 "hi" part and an fp32
//     "lo" residual in registers, and store both into shared memory in the canonical K-major
//     SWIZZLE_128B layout; one elected thread bulk-copies the weight slab of the stage;
//   * one elected thread of the MMA warp issues, per 8-wide k-step, the three products
//     hi*hi + lo*hi + hi*lo (3xTF32: fp32-accurate to ~2^-21 relative) into TMEM;
//     tcgen05.commit on an mbarrier frees the shared-memory stage / publishes the tile;
//   * 4 epilogue warps read the accumulator with tcgen05.ld (warp w owns TMEM lanes
//     32(w%4).. = pairs 32(w%4)..) and scatter-add rows with red.global.add.v4.f32; two
//     accumulators in TMEM let the epilogue of tile t overlap the MMAs of tile t+1.
//
// CTAs are persistent (one per SM); stages are mbarrier-pipelined so the gather of chunk c+1
// overlaps the MMAs of chunk c.  Weights come PRE-SPLIT and PRE-SWIZZLED (dgr_pack_weight_tf32,
// cached per layer by the host): per (offset, 32-channel chunk) one contiguous slab holding the
// TF32 hi tile and the lo tile in shared-memory image order, streamed by a single
// cp.async.bulk (TMA engine) per stage - the loader threads only touch the gathered rows.
#include <cuda_fp16.h>
#include <stdlib.h>

#include "common.cuh"
#include "tc_common.cuh"

namespace {

using namespace tc;

// gathered feature rows: ld.global.nc (default) or, with -DDGR_GATHER_CG, ld.global.cg (L2 only, no L1 allocation) -
// an A/B build switch kept for the record in profiles/r02_experiments.txt
#ifdef DGR_GATHER_CG
#define DGR_GATHER_LOAD(p) __ldcg(p)
#else
#define DGR_GATHER_LOAD(p) __ldg(p)
#endif

#define DGR_TRY_RC(expr)             \
  do {                              \
    int32_t rc__ = (expr);          \
    if (rc__ != DGR_OK) return rc__; \
  } while (0)

constexpr int kLoaderWarps = 8;
constexpr int kLoaderThreads = kLoaderWarps * 32;   // warps 0..7: gather + TF32 split
constexpr int kMmaWarp = kLoaderWarps;               // warp 8: tcgen05.mma issuer
// warps 9..12 (kLoaderWarps + 1 ..): epilogue, TMEM -> red.global
constexpr int kThreadsTC = (kLoaderWarps + 5) * 32;  // 416
constexpr int kTileM = 128;
constexpr int kChunk = 32;               // floats of K per stage (128 bytes)
constexpr int kATileBytes = kTileM * 128;

// split one float4 into a TF32 "hi" part (round to nearest) and the exact fp32 residual "lo"
// (the tensor core truncates lo to TF32: 2^-21 relative overall) and store both 16-byte pieces
__device__ __forceinline__ void split_store(float4 v, unsigned char* hi_tile, unsigned char* lo_tile,
                                            uint32_t off) {
  float4 h, l;
  h.x = tf32_round(v.x); h.y = tf32_round(v.y); h.z = tf32_round(v.z); h.w = tf32_round(v.w);
  l.x = v.x - h.x; l.y = v.y - h.y; l.z = v.z - h.z; l.w = v.w - h.w;
  *reinterpret_cast<float4*>(hi_tile + off) = h;
  *reinterpret_cast<float4*>(lo_tile + off) = l;
}

// 3xFP16 split (cta_group::2 kernel, kF16): fp16 carries the same 11 significant bits as TF32 at half the
// bytes and twice the tensor rate.  x is first scaled by a power of two `sx` (exact) that maps the tensor's
// absolute maximum into [2^14, 2^15) - below fp16's 65504, far above its 2^-14 normal floor - then split into
// hi = fp16(x'), lo = fp16(x' - hi): the same hi*hi + lo*hi + hi*lo products as 3xTF32, 2^-21 relative
// (an element more than 2^17 below the tensor's maximum loses bits of its lo part: <= 2^-39 of the maximum).
__device__ __forceinline__ void split_store_f16(float4 a, float4 b, float sx, unsigned char* hi_tile,
                                                unsigned char* lo_tile, uint32_t off) {
  const float x[8] = {a.x * sx, a.y * sx, a.z * sx, a.w * sx, b.x * sx, b.y * sx, b.z * sx, b.w * sx};
  uint32_t h[4], l[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const __half2 hh = __floats2half2_rn(x[2 * i], x[2 * i + 1]);
    const float2 hf = __half22float2(hh);
    const __half2 ll = __floats2half2_rn(x[2 * i] - hf.x, x[2 * i + 1] - hf.y);
    h[i] = *reinterpret_cast<const uint32_t*>(&hh);
    l[i] = *reinterpret_cast<const uint32_t*>(&ll);
  }
  *reinterpret_cast<uint4*>(hi_tile + off) = make_uint4(h[0], h[1], h[2], h[3]);
  *reinterpret_cast<uint4*>(lo_tile + off) = make_uint4(l[0], l[1], l[2], l[3]);
}

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// bulk copy delivered to the same CTA-relative offsets of every CTA in `mask`; each destination's
// mbarrier (same offset) receives the complete_tx of the bytes written into that CTA
__device__ __forceinline__ void bulk_g2s_multicast(uint32_t dst_smem, const void* src, uint32_t bytes,
                                                   uint32_t bar, uint16_t mask) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1], %2, [%3], %4;"
      ::"r"(dst_smem), "l"(src), "r"(bytes), "r"(bar), "h"(mask)
      : "memory");
}
__device__ __forceinline__ void tc_commit_multicast(uint32_t bar, uint16_t mask) {
  asm volatile(
      "tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
      "h"(mask)
      : "memory");
}


// Epilogue scatter of 32 accumulator columns [col, col + 32) of a warp's 32 rows.
// tcgen05.ld hands every thread ONE row (lane = row): scattering from that layout makes each warp
// instruction touch 32 different output rows with 16 bytes each - 32 memory requests per
// instruction, 8192 per tile at cout = 256, which is what bounded the wide layers (every other
// knob - atomics vs stores, weight multicast, A in tensor memory, cta_group::2, gather lookahead -
// left their time unchanged).  Transposing through a 4 KB shared-memory tile (XOR-swizzled, no
// bank conflicts) lets 8 lanes cover one row's 128-byte line: 4 full lines per instruction.
__device__ __forceinline__ void scatter32_lines(unsigned char* stg, int lane, float* __restrict__ out, int cout,
                                                int col, int j, const uint32_t (&v)[32]) {
#pragma unroll
  for (int q = 0; q < 8; ++q)
    *reinterpret_cast<uint4*>(stg + lane * 128 + ((q ^ (lane & 7)) << 4)) =
        make_uint4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
  __syncwarp();
  const int p = lane & 7, rsub = lane >> 3;
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const int R = rsub + 4 * k;
    const int jr = __shfl_sync(0xffffffffu, j, R);
    const float4 x = *reinterpret_cast<const float4*>(stg + R * 128 + ((p ^ (R & 7)) << 4));
    if (jr >= 0) red_add_v4(out + (size_t)jr * cout + col + p * 4, x.x, x.y, x.z, x.w);
  }
  __syncwarp();      // the tile is rewritten by the next column group
}
__device__ __forceinline__ void scatter32_rows(float* __restrict__ out, int cout, int col, int j,
                                               const uint32_t (&v)[32]) {
  if (j >= 0) {
    float* dst = out + (size_t)j * cout + col;
#pragma unroll
    for (int q = 0; q < 8; ++q)
      red_add_v4(dst + 4 * q, __uint_as_float(v[4 * q]), __uint_as_float(v[4 * q + 1]),
                 __uint_as_float(v[4 * q + 2]), __uint_as_float(v[4 * q + 3]));
  }
}
constexpr int kEpiStageBytes = 4 * 4096;     // one 32 x 32 fp32 transpose tile per epilogue warp

struct TcShared {
  unsigned long long full[4];      // gathered A tiles (256 arrivals) + B hi tile (bulk-copy bytes)
  unsigned long long full_lo[4];   // B lo tile (bulk-copy bytes): needed only by the third product
  unsigned long long empty[4];
  unsigned long long acc_full[2];
  unsigned long long acc_empty[2];
  uint32_t tmem_base;
};

// Warp-specialised persistent kernel.  Roles iterate the same tile sequence
// (tile = blockIdx.x + i * gridDim.x) and meet only through mbarriers:
//   loaders  --full[s]-->  MMA issuer  --empty[s]-->  loaders        (shared-memory stages)
//   MMA issuer  --acc_full[b]-->  epilogue  --acc_empty[b]-->  MMA   (two TMEM accumulators)
template <int kCluster, int kPD>
__global__ void __launch_bounds__(kThreadsTC, 1)
spconv_tc_kernel(const float* __restrict__ in_feat, int cin, const float* __restrict__ wt, int cout,
                 const int32_t* __restrict__ in_idx, const int32_t* __restrict__ out_idx,
                 const int32_t* __restrict__ kofs, const int32_t* __restrict__ tile_k,
                 const int32_t* __restrict__ tile_start, int n_tiles, int n_stages, int tmem_cols,
                 int passes, int epi, float* __restrict__ out) {
  extern __shared__ __align__(16) unsigned char smem_dyn[];
  TcShared& sh = *reinterpret_cast<TcShared*>(smem_dyn);
  // stage buffers start at the next 1024-byte boundary (SWIZZLE_128B atom alignment)
  unsigned char* stage0 = reinterpret_cast<unsigned char*>(
      (reinterpret_cast<uintptr_t>(smem_dyn) + sizeof(TcShared) + 1023) & ~(uintptr_t)1023);
  const int b_tile_bytes = cout * 128;
  const int stage_bytes = 2 * kATileBytes + 2 * b_tile_bytes;
  const int t = threadIdx.x;
  const int warp = t >> 5, lane = t & 31;
  const int n_chunks = cin / kChunk;
  const uint32_t acc_stride = (uint32_t)tmem_cols >> 1;   // columns between the two accumulators

  if (t == 0) {
    for (int s = 0; s < n_stages; ++s) {
      mbar_init(smem_u32(&sh.full[s]), kLoaderThreads);
      mbar_init(smem_u32(&sh.full_lo[s]), 1);
      mbar_init(smem_u32(&sh.empty[s]), kCluster);   // one tcgen05.commit per CTA that reads the stage's B
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(smem_u32(&sh.acc_full[b]), 1);
      mbar_init(smem_u32(&sh.acc_empty[b]), 128);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == kMmaWarp) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                     smem_u32(&sh.tmem_base)),
                 "r"((uint32_t)tmem_cols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  if (kCluster > 1) cluster_sync_all();     // peers' barriers are initialised before anyone multicasts
  tc_fence_after();
  const uint32_t tmem_base = sh.tmem_base;
  const uint32_t cta_rank = kCluster > 1 ? cluster_ctarank() : 0;

  if (warp < kLoaderWarps) {
    // ================================ loaders ============================================
    // B (weights): one elected thread streams the pre-split, pre-swizzled [hi | lo] slab of
    // (kappa, chunk) with a single bulk copy that lands on full[s] (complete_tx).
    // A (features): every thread gathers 4 x 16 B, software-pipelined one chunk ahead.
    const int piece = t & 7, rgrp = t >> 3;   // 8 lanes cover one 128-byte row; 32 row groups
    const uint32_t a_off = (uint32_t)(rgrp * 128 + ((piece ^ (rgrp & 7)) << 4));   // + i * 4096
    const uint32_t slab_bytes = 2u * (uint32_t)b_tile_bytes;
    auto load_rows = [&](int tile_id, int (&src)[4]) {
      const int kap = tile_k[tile_id];
      const int q0 = tile_start[tile_id];
      const int nrows = min(kTileM, kofs[kap + 1] - q0);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int r = i * 32 + rgrp;
        src[i] = (r < nrows) ? __ldg(in_idx + q0 + r) : -1;
      }
    };
    auto load_a = [&](const int (&src)[4], int c, float4 (&v)[4]) {
#pragma unroll
      for (int i = 0; i < 4; ++i)
        v[i] = src[i] >= 0 ? DGR_GATHER_LOAD(reinterpret_cast<const float4*>(in_feat + (size_t)src[i] * cin + c * kChunk +
                                                                    piece * 4))
                           : make_float4(0.f, 0.f, 0.f, 0.f);
    };
    // The gather runs kPD chunks ahead of the chunk being stored (register queue q[0..kPD]): a
    // stage can only be published when the SLOWEST of its 1024 row loads has landed, and with ~1/5
    // of the rows missing L2 that is a loaded-DRAM latency (~3k cycles) every chunk - more than one
    // chunk's worth of MMAs, so one chunk of lookahead left the tensor pipe waiting.
    uint32_t it = 0;
    float4 q[kPD + 1][4];
    int pf_tile = blockIdx.x, pf_c = 0;          // prefetch cursor (tile, chunk) and the rows of its tile
    int pf_src[4], pf_nsrc[4];                   // ... and of the tile after it (indices one tile ahead)
    load_rows(pf_tile, pf_src);
    if (pf_tile + (int)gridDim.x < n_tiles) load_rows(pf_tile + gridDim.x, pf_nsrc);
    auto pf_issue = [&](float4 (&v)[4]) {
      if (pf_tile < n_tiles) load_a(pf_src, pf_c, v);
      if (++pf_c == n_chunks) {
        pf_c = 0;
        pf_tile += gridDim.x;
#pragma unroll
        for (int i = 0; i < 4; ++i) pf_src[i] = pf_nsrc[i];
        if (pf_tile + (int)gridDim.x < n_tiles) load_rows(pf_tile + gridDim.x, pf_nsrc);
      }
    };
#pragma unroll
    for (int d = 0; d < kPD; ++d) pf_issue(q[d]);
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
      const int kappa = tile_k[tile];
      const float* slab = wt + (size_t)kappa * n_chunks * (slab_bytes / 4);
      for (int c = 0; c < n_chunks; ++c, ++it) {
        const int s = it % n_stages;
        const uint32_t ph = (it / n_stages) & 1;
        pf_issue(q[kPD]);
        mbar_wait(smem_u32(&sh.empty[s]), ph ^ 1);
        unsigned char* a_hi = stage0 + (size_t)s * stage_bytes;
        unsigned char* a_lo = a_hi + kATileBytes;
        if (t == 0) {
          // hi tile first, on the barrier the first two products wait for; the lo tile lands on its
          // own barrier while those products already run
          const float* src = slab + (size_t)c * (slab_bytes / 4);
          mbar_expect_tx(smem_u32(&sh.full[s]), (uint32_t)b_tile_bytes);
          mbar_arrive_expect_tx(smem_u32(&sh.full_lo[s]), (uint32_t)b_tile_bytes);
          if (kCluster == 1) {
            bulk_g2s(smem_u32(a_lo + kATileBytes), src, (uint32_t)b_tile_bytes, smem_u32(&sh.full[s]));
            bulk_g2s(smem_u32(a_lo + kATileBytes + b_tile_bytes), src + b_tile_bytes / 4, (uint32_t)b_tile_bytes,
                     smem_u32(&sh.full_lo[s]));
          } else if (cta_rank == 0) {
            // the CTA pair works on two tiles of the SAME offset: one L2 read of each B tile feeds both
            // SMs - rank 0 multicasts the hi tile, rank 1 the lo tile (empty[s] counts both CTAs' MMAs)
            bulk_g2s_multicast(smem_u32(a_lo + kATileBytes), src, (uint32_t)b_tile_bytes, smem_u32(&sh.full[s]),
                               (uint16_t)0x3);
          } else {
            bulk_g2s_multicast(smem_u32(a_lo + kATileBytes + b_tile_bytes), src + b_tile_bytes / 4,
                               (uint32_t)b_tile_bytes, smem_u32(&sh.full_lo[s]), (uint16_t)0x3);
          }
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) split_store(q[0][i], a_hi, a_lo, a_off + i * 4096);
        fence_proxy_async();
        mbar_arrive(smem_u32(&sh.full[s]));
#pragma unroll
        for (int d = 0; d < kPD; ++d)
#pragma unroll
          for (int i = 0; i < 4; ++i) q[d][i] = q[d + 1][i];
      }
    }
  } else if (warp == kMmaWarp) {
    // ================================ MMA issuer =========================================
    // instruction descriptor: D = F32, A = B = TF32, both K-major, N = cout, M = 128
    const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(cout >> 3) << 17) |
                           ((uint32_t)(kTileM >> 4) << 24);
    uint32_t it = 0, tile_iter = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++tile_iter) {
      const uint32_t buf = tile_iter & 1;
      const uint32_t tmem_d = tmem_base + buf * acc_stride;
      mbar_wait(smem_u32(&sh.acc_empty[buf]), ((tile_iter >> 1) & 1) ^ 1);   // epilogue drained it
      tc_fence_after();
      for (int c = 0; c < n_chunks; ++c, ++it) {
        const int s = it % n_stages;
        const uint32_t ph = (it / n_stages) & 1;
        mbar_wait(smem_u32(&sh.full[s]), ph);
        tc_fence_after();
        if (lane == 0) {
          const uint32_t a_hi = smem_u32(stage0 + (size_t)s * stage_bytes);
          const uint32_t a_lo = a_hi + kATileBytes;
          const uint32_t b_hi = a_lo + kATileBytes;
#pragma unroll
          for (int ks = 0; ks < kChunk / 8; ++ks) {   // hi*hi and lo*hi need only the B hi tile
            const uint32_t ko = ks * 32;   // 8 tf32 = 32 bytes along K inside the swizzle row
            const uint64_t dbh = umma_desc(b_hi + ko);
            tc_mma_tf32(tmem_d, umma_desc(a_hi + ko), dbh, idesc, (c | ks) != 0);
            if (passes == 3) tc_mma_tf32(tmem_d, umma_desc(a_lo + ko), dbh, idesc, 1);
          }
        }
        mbar_wait(smem_u32(&sh.full_lo[s]), ph);       // the B lo tile has landed meanwhile
        tc_fence_after();
        if (lane == 0) {
          const uint32_t a_hi = smem_u32(stage0 + (size_t)s * stage_bytes);
          const uint32_t b_lo = a_hi + 2 * kATileBytes + b_tile_bytes;
          if (passes == 3) {
#pragma unroll
            for (int ks = 0; ks < kChunk / 8; ++ks)
              tc_mma_tf32(tmem_d, umma_desc(a_hi + ks * 32), umma_desc(b_lo + ks * 32), idesc, 1);
          }
          if (kCluster == 1) tc_commit(smem_u32(&sh.empty[s]));
          else tc_commit_multicast(smem_u32(&sh.empty[s]), (uint16_t)0x3);   // frees the stage in both CTAs
          if (c == n_chunks - 1) tc_commit(smem_u32(&sh.acc_full[buf]));
        }
        __syncwarp();
      }
    }
  } else {
    // ================================ epilogue ===========================================
    const int lane_grp = warp & 3;            // TMEM lanes 32 * (warp % 4) .. + 31
    unsigned char* epi_stage = stage0 + (size_t)n_stages * stage_bytes + (warp - kLoaderWarps - 1) * 4096;
    uint32_t tile_iter = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++tile_iter) {
      const uint32_t buf = tile_iter & 1;
      const int kappa = tile_k[tile];
      const int p0 = tile_start[tile];
      const int rows = min(kTileM, kofs[kappa + 1] - p0);
      const int r = lane_grp * 32 + lane;
      const int j = r < rows ? out_idx[p0 + r] : -1;
      mbar_wait(smem_u32(&sh.acc_full[buf]), (tile_iter >> 1) & 1);
      tc_fence_after();
      const uint32_t taddr = tmem_base + buf * acc_stride + ((uint32_t)(lane_grp * 32) << 16);
      int col = 0;
      for (; col + 32 <= cout; col += 32) {
        uint32_t v[32];
        tc_ld32(taddr + col, v);
        if (epi) scatter32_lines(epi_stage, lane, out, cout, col, j, v);
        else scatter32_rows(out, cout, col, j, v);
      }
      if (col < cout) {   // cout % 32 == 16
        uint32_t v[16];
        tc_ld16(taddr + col, v);
        if (j >= 0) {
          float* dst = out + (size_t)j * cout + col;
#pragma unroll
          for (int q = 0; q < 4; ++q)
            red_add_v4(dst + 4 * q, __uint_as_float(v[4 * q]), __uint_as_float(v[4 * q + 1]),
                       __uint_as_float(v[4 * q + 2]), __uint_as_float(v[4 * q + 3]));
        }
      }
      tc_fence_before();
      mbar_arrive(smem_u32(&sh.acc_empty[buf]));
    }
  }
  tc_fence_before();
  __syncthreads();
  if (kCluster > 1) cluster_sync_all();     // nobody exits while a peer may still signal its barriers
  if (warp == kMmaWarp) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base),
                 "r"((uint32_t)tmem_cols)
                 : "memory");
  }
}


// ---------------------------------------------------------------------------------------
// Variant with the A operand in TENSOR MEMORY.
// With both operands in shared memory every one of the three TF32 products re-reads A and B
// from shared memory: 12 MMAs x 12 KB + 96 KB of stores per 32-channel chunk = 240 KB against a
// 128 B/clk port - the SS kernel above is shared-memory-bandwidth bound (ncu: tensor pipe 55 %).
// Here the loaders put the split A tiles straight into TMEM (tcgen05.st; thread = row = lane),
// the MMAs read only B from shared memory (96 KB per chunk) and shared memory holds nothing but
// the bulk-copied weight slabs, which also makes room for deeper pipelines.
// TMEM columns: [accumulator(s)] [stage 0: A hi (32) | A lo (32)] [stage 1 ...].
// Loader warps 0-3 fill even chunks, warps 4-7 odd chunks (warp w owns TMEM lanes 32 (w % 4) ..).
// ---------------------------------------------------------------------------------------
struct TcAtShared {
  unsigned long long full[4];      // 128 loader arrivals (A in TMEM) + B hi bytes
  unsigned long long full_lo[4];   // B lo bytes
  unsigned long long empty[4];
  unsigned long long acc_full[2];
  unsigned long long acc_empty[2];
  uint32_t tmem_base;
};

__global__ void __launch_bounds__(kThreadsTC, 1)
spconv_tc_at_kernel(const float* __restrict__ in_feat, int cin, const float* __restrict__ wt, int cout,
                    const int32_t* __restrict__ in_idx, const int32_t* __restrict__ out_idx,
                    const int32_t* __restrict__ kofs, const int32_t* __restrict__ tile_k,
                    const int32_t* __restrict__ tile_start, int n_tiles, int n_stages, int tmem_cols,
                    int n_acc, int acc_cols, int passes, float* __restrict__ out) {
  extern __shared__ __align__(16) unsigned char smem_dyn[];
  TcAtShared& sh = *reinterpret_cast<TcAtShared*>(smem_dyn);
  unsigned char* stage0 = reinterpret_cast<unsigned char*>(
      (reinterpret_cast<uintptr_t>(smem_dyn) + sizeof(TcAtShared) + 1023) & ~(uintptr_t)1023);
  const int b_tile_bytes = cout * 128;
  const int stage_bytes = 2 * b_tile_bytes;          // shared memory holds only [B hi | B lo]
  const int t = threadIdx.x;
  const int warp = t >> 5, lane = t & 31;
  const int n_chunks = cin / kChunk;
  const uint32_t a_col0 = (uint32_t)(n_acc * acc_cols);   // first column of the A stages

  if (t == 0) {
    for (int s = 0; s < n_stages; ++s) {
      mbar_init(smem_u32(&sh.full[s]), 128);
      mbar_init(smem_u32(&sh.full_lo[s]), 1);
      mbar_init(smem_u32(&sh.empty[s]), 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(smem_u32(&sh.acc_full[b]), 1);
      mbar_init(smem_u32(&sh.acc_empty[b]), 128);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == kMmaWarp) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                     smem_u32(&sh.tmem_base)),
                 "r"((uint32_t)tmem_cols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = sh.tmem_base;

  if (warp < kLoaderWarps) {
    // ================================ loaders ============================================
    const int group = warp >> 2;                       // 0: even chunks, 1: odd chunks
    const int row = (warp & 3) * 32 + lane;            // tile row == TMEM lane of this thread
    const uint32_t lane_addr = tmem_base + ((uint32_t)((warp & 3) * 32) << 16);
    const bool issuer = (t == group * 128);            // one bulk-copy issuer per group
    const uint32_t slab_bytes = 2u * (uint32_t)b_tile_bytes;
    uint32_t it = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
      const int kappa = tile_k[tile];
      const int p0 = tile_start[tile];
      const int rows = min(kTileM, kofs[kappa + 1] - p0);
      const int src = row < rows ? __ldg(in_idx + p0 + row) : -1;
      const float4* src_row = reinterpret_cast<const float4*>(in_feat + (size_t)(src < 0 ? 0 : src) * cin);
      const float* slab = wt + (size_t)kappa * n_chunks * (slab_bytes / 4);
      for (int c = 0; c < n_chunks; ++c, ++it) {
        if ((int)(it & 1) != group) continue;
        const int s = it % n_stages;
        const uint32_t ph = (it / n_stages) & 1;
        float4 v[8];
#pragma unroll
        for (int q = 0; q < 8; ++q)
          v[q] = src >= 0 ? __ldg(src_row + c * 8 + q) : make_float4(0.f, 0.f, 0.f, 0.f);
        mbar_wait(smem_u32(&sh.empty[s]), ph ^ 1);
        tc_fence_after();
        if (issuer) {
          const float* bsrc = slab + (size_t)c * (slab_bytes / 4);
          unsigned char* b_hi = stage0 + (size_t)s * stage_bytes;
          mbar_expect_tx(smem_u32(&sh.full[s]), (uint32_t)b_tile_bytes);
          bulk_g2s(smem_u32(b_hi), bsrc, (uint32_t)b_tile_bytes, smem_u32(&sh.full[s]));
          mbar_arrive_expect_tx(smem_u32(&sh.full_lo[s]), (uint32_t)b_tile_bytes);
          bulk_g2s(smem_u32(b_hi + b_tile_bytes), bsrc + b_tile_bytes / 4, (uint32_t)b_tile_bytes,
                   smem_u32(&sh.full_lo[s]));
        }
        uint32_t hi[32], lo[32];
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          const float f[4] = {v[q].x, v[q].y, v[q].z, v[q].w};
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float h = tf32_round(f[e]);
            hi[4 * q + e] = __float_as_uint(h);
            lo[4 * q + e] = __float_as_uint(f[e] - h);
          }
        }
        const uint32_t a_addr = lane_addr + a_col0 + (uint32_t)s * 64;
        tc_st32(a_addr, hi);
        tc_st32(a_addr + 32, lo);
        tc_st_wait();
        tc_fence_before();
        mbar_arrive(smem_u32(&sh.full[s]));
      }
    }
  } else if (warp == kMmaWarp) {
    // ================================ MMA issuer =========================================
    const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(cout >> 3) << 17) |
                           ((uint32_t)(kTileM >> 4) << 24);
    uint32_t it = 0, tile_iter = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++tile_iter) {
      const uint32_t buf = n_acc == 2 ? (tile_iter & 1) : 0;
      const uint32_t use = n_acc == 2 ? (tile_iter >> 1) : tile_iter;     // uses of this accumulator so far
      const uint32_t tmem_d = tmem_base + buf * (uint32_t)acc_cols;
      mbar_wait(smem_u32(&sh.acc_empty[buf]), (use & 1) ^ 1);
      tc_fence_after();
      for (int c = 0; c < n_chunks; ++c, ++it) {
        const int s = it % n_stages;
        const uint32_t ph = (it / n_stages) & 1;
        const uint32_t a_hi = tmem_base + a_col0 + (uint32_t)s * 64, a_lo = a_hi + 32;
        const uint32_t b_hi = smem_u32(stage0 + (size_t)s * stage_bytes), b_lo = b_hi + b_tile_bytes;
        mbar_wait(smem_u32(&sh.full[s]), ph);
        tc_fence_after();
        if (lane == 0) {
#pragma unroll
          for (int ks = 0; ks < kChunk / 8; ++ks) {
            const uint64_t dbh = umma_desc(b_hi + ks * 32);
            tc_mma_tf32_ts(tmem_d, a_hi + ks * 8, dbh, idesc, (c | ks) != 0);
            if (passes == 3) tc_mma_tf32_ts(tmem_d, a_lo + ks * 8, dbh, idesc, 1);
          }
        }
        mbar_wait(smem_u32(&sh.full_lo[s]), ph);
        tc_fence_after();
        if (lane == 0) {
          if (passes == 3) {
#pragma unroll
            for (int ks = 0; ks < kChunk / 8; ++ks)
              tc_mma_tf32_ts(tmem_d, a_hi + ks * 8, umma_desc(b_lo + ks * 32), idesc, 1);
          }
          tc_commit(smem_u32(&sh.empty[s]));
          if (c == n_chunks - 1) tc_commit(smem_u32(&sh.acc_full[buf]));
        }
        __syncwarp();
      }
    }
  } else {
    // ================================ epilogue ===========================================
    const int lane_grp = warp & 3;
    uint32_t tile_iter = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++tile_iter) {
      const uint32_t buf = n_acc == 2 ? (tile_iter & 1) : 0;
      const uint32_t use = n_acc == 2 ? (tile_iter >> 1) : tile_iter;
      const int kappa = tile_k[tile];
      const int p0 = tile_start[tile];
      const int rows = min(kTileM, kofs[kappa + 1] - p0);
      const int r = lane_grp * 32 + lane;
      const int j = r < rows ? out_idx[p0 + r] : -1;
      mbar_wait(smem_u32(&sh.acc_full[buf]), use & 1);
      tc_fence_after();
      const uint32_t taddr = tmem_base + buf * (uint32_t)acc_cols + ((uint32_t)(lane_grp * 32) << 16);
      int col = 0;
      for (; col + 32 <= cout; col += 32) {
        uint32_t v[32];
        tc_ld32(taddr + col, v);
        if (j >= 0) {
          float* dst = out + (size_t)j * cout + col;
#pragma unroll
          for (int q = 0; q < 8; ++q)
            red_add_v4(dst + 4 * q, __uint_as_float(v[4 * q]), __uint_as_float(v[4 * q + 1]),
                       __uint_as_float(v[4 * q + 2]), __uint_as_float(v[4 * q + 3]));
        }
      }
      if (col < cout) {
        uint32_t v[16];
        tc_ld16(taddr + col, v);
        if (j >= 0) {
          float* dst = out + (size_t)j * cout + col;
#pragma unroll
          for (int q = 0; q < 4; ++q)
            red_add_v4(dst + 4 * q, __uint_as_float(v[4 * q]), __uint_as_float(v[4 * q + 1]),
                       __uint_as_float(v[4 * q + 2]), __uint_as_float(v[4 * q + 3]));
        }
      }
      tc_fence_before();
      mbar_arrive(smem_u32(&sh.acc_empty[buf]));
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kMmaWarp) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base),
                 "r"((uint32_t)tmem_cols)
                 : "memory");
  }
}

// ---------------------------------------------------------------------------------------
// CTA-PAIR variant (tcgen05 cta_group::2): two CTAs of a cluster (the two SMs of a TPC) work on
// two 128-pair tiles of the SAME kernel offset as ONE M = 256 MMA.  Each CTA gathers its own
// 128 rows of A and holds only HALF of every weight tile (B rows = output channels
// [rank * cout/2, (rank + 1) * cout/2)); the tensor core reads the peer's half over the pair's
// on-chip path.  What every SM must RECEIVE per 32-channel chunk drops from 64 KB + 16 KB to
// 32 KB + 16 KB - the wide layers are bound by exactly that ingress (DESIGN.md section 3).
//
// Protocol (rank 0 = leader issues all MMAs):
//   full[s]       local: 256 loader arrivals + this CTA's two B halves (bulk-copy bytes)
//   peer_full[s]  leader's: the peer's relay thread arrives once ITS full[s] has completed
//   empty[s]      both:  tcgen05.commit.cta_group::2 multicast - the stage may be refilled
//   acc_full[b]   both:  multicast commit - the accumulator (128 lanes x cout in each CTA) is final
//   acc_empty[b]  leader's: 128 local + 128 remote epilogue threads have drained accumulator b
// ---------------------------------------------------------------------------------------
struct Tc2Shared {
  unsigned long long full[4];
  unsigned long long peer_full[4];
  unsigned long long empty[4];
  unsigned long long acc_full[2];
  unsigned long long acc_empty[2];
  uint32_t tmem_base;
};

__device__ __forceinline__ uint32_t mapa_u32(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void mbar_wait_cluster(uint32_t bar, uint32_t parity) {
  uint32_t ok = 0;
  while (!ok) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
  }
}
__device__ __forceinline__ void tc_mma_tf32_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                                 uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tc_mma_f16_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                                uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tc_commit_pair(uint32_t bar) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
      "h"((uint16_t)0x3)
      : "memory");
}

// kF16: 3xFP16 instead of 3xTF32 (64 channels per 128-byte stage row; `wt` then holds the fp16 slabs of
// dgr_pack_weight_f16, amax_in the input tensor's absolute maximum, w_inv_scale the inverse of the weight scale)
template <int kPD, bool kF16>
__global__ void __launch_bounds__(kThreadsTC, 1)
spconv_tc_pair_kernel(const float* __restrict__ in_feat, int cin, const float* __restrict__ wt, int cout,
                      const int32_t* __restrict__ in_idx, const int32_t* __restrict__ out_idx,
                      const int32_t* __restrict__ kofs, const int32_t* __restrict__ tile_k,
                      const int32_t* __restrict__ tile_start, int n_tiles, int n_stages, int tmem_cols,
                      int passes, int epi, const float* __restrict__ amax_in,
                      const float* __restrict__ w_inv_scale, float* __restrict__ out) {
  constexpr int kCh = kF16 ? 64 : kChunk;        // channels per stage (one 128-byte swizzle row)
  constexpr int kV = kF16 ? 2 : 1;               // float4 loads per (thread, row, chunk)
  extern __shared__ __align__(16) unsigned char smem_dyn[];
  Tc2Shared& sh = *reinterpret_cast<Tc2Shared*>(smem_dyn);
  unsigned char* stage0 = reinterpret_cast<unsigned char*>(
      (reinterpret_cast<uintptr_t>(smem_dyn) + sizeof(Tc2Shared) + 1023) & ~(uintptr_t)1023);
  const int b_tile_bytes = cout * 128;             // a whole B tile (hi or lo) in the packed slab
  const int b_half_bytes = b_tile_bytes >> 1;      // what this CTA holds of it
  const int stage_bytes = 2 * kATileBytes + 2 * b_half_bytes;
  const int t = threadIdx.x;
  const int warp = t >> 5, lane = t & 31;
  const int n_chunks = cin / kCh;
  const uint32_t acc_stride = (uint32_t)tmem_cols >> 1;
  const uint32_t rank = cluster_ctarank();
  const int n_pairs = n_tiles >> 1;
  const int pair0 = blockIdx.x >> 1, pair_step = gridDim.x >> 1;

  if (t == 0) {
    for (int s = 0; s < n_stages; ++s) {
      mbar_init(smem_u32(&sh.full[s]), kLoaderThreads);
      mbar_init(smem_u32(&sh.peer_full[s]), 1);
      mbar_init(smem_u32(&sh.empty[s]), 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(smem_u32(&sh.acc_full[b]), 1);
      mbar_init(smem_u32(&sh.acc_empty[b]), 256);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == kMmaWarp) {      // pair-wide allocation: the same warp of BOTH CTAs issues it
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                     smem_u32(&sh.tmem_base)),
                 "r"((uint32_t)tmem_cols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();          // both CTAs' barriers are initialised before anyone signals across
  tc_fence_after();
  const uint32_t tmem_base = sh.tmem_base;

  if (warp < kLoaderWarps) {
    // ================================ loaders (both CTAs) ================================
    const int piece = t & 7, rgrp = t >> 3;
    const uint32_t a_off = (uint32_t)(rgrp * 128 + ((piece ^ (rgrp & 7)) << 4));
    const uint32_t slab_floats = 2u * (uint32_t)b_tile_bytes / 4;
    auto load_rows = [&](int tile_id, int (&src)[4]) {
      const int kap = tile_k[tile_id];
      const int q0 = tile_start[tile_id];
      const int nrows = min(kTileM, kofs[kap + 1] - q0);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int r = i * 32 + rgrp;
        src[i] = (r < nrows) ? __ldg(in_idx + q0 + r) : -1;
      }
    };
    auto load_a = [&](const int (&src)[4], int c, float4 (&v)[4][kV]) {
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int u = 0; u < kV; ++u)
          v[i][u] = src[i] >= 0 ? DGR_GATHER_LOAD(reinterpret_cast<const float4*>(in_feat + (size_t)src[i] * cin + c * kCh +
                                                                         piece * (4 * kV) + 4 * u))
                                : make_float4(0.f, 0.f, 0.f, 0.f);
    };
    const float sx = kF16 ? f16_scale_for(__ldg(amax_in)) : 1.f;
    uint32_t it = 0;
    const int tstep = 2 * pair_step;             // this CTA's tiles: 2 * pair + rank
    float4 q[kPD + 1][4][kV];                    // gather queue, kPD chunks ahead (see spconv_tc_kernel)
    int pf_tile = 2 * pair0 + (int)rank, pf_c = 0;
    int pf_src[4], pf_nsrc[4];
    if (pf_tile < n_tiles) load_rows(pf_tile, pf_src);
    if (pf_tile + tstep < n_tiles) load_rows(pf_tile + tstep, pf_nsrc);
    auto pf_issue = [&](float4 (&v)[4][kV]) {
      if (pf_tile < n_tiles) load_a(pf_src, pf_c, v);
      if (++pf_c == n_chunks) {
        pf_c = 0;
        pf_tile += tstep;
#pragma unroll
        for (int i = 0; i < 4; ++i) pf_src[i] = pf_nsrc[i];
        if (pf_tile + tstep < n_tiles) load_rows(pf_tile + tstep, pf_nsrc);
      }
    };
#pragma unroll
    for (int d = 0; d < kPD; ++d) pf_issue(q[d]);
    for (int pair = pair0; pair < n_pairs; pair += pair_step) {
      const int tile = 2 * pair + (int)rank;
      const int kappa = tile_k[tile];
      const float* slab = wt + (size_t)kappa * n_chunks * slab_floats;
      for (int c = 0; c < n_chunks; ++c, ++it) {
        const int s = it % n_stages;
        const uint32_t ph = (it / n_stages) & 1;
        pf_issue(q[kPD]);
        mbar_wait(smem_u32(&sh.empty[s]), ph ^ 1);
        unsigned char* a_hi = stage0 + (size_t)s * stage_bytes;
        unsigned char* a_lo = a_hi + kATileBytes;
        if (t == 0) {
          // this CTA's half (rows rank * cout/2 ..) of the hi tile and of the lo tile
          const float* bsrc = slab + (size_t)c * slab_floats + (size_t)rank * (b_half_bytes / 4);
          mbar_expect_tx(smem_u32(&sh.full[s]), 2u * (uint32_t)b_half_bytes);
          bulk_g2s(smem_u32(a_lo + kATileBytes), bsrc, (uint32_t)b_half_bytes, smem_u32(&sh.full[s]));
          bulk_g2s(smem_u32(a_lo + kATileBytes + b_half_bytes), bsrc + b_tile_bytes / 4, (uint32_t)b_half_bytes,
                   smem_u32(&sh.full[s]));
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          if (kF16) split_store_f16(q[0][i][0], q[0][i][kV - 1], sx, a_hi, a_lo, a_off + i * 4096);
          else split_store(q[0][i][0], a_hi, a_lo, a_off + i * 4096);
        }
        fence_proxy_async();
        mbar_arrive(smem_u32(&sh.full[s]));
#pragma unroll
        for (int d = 0; d < kPD; ++d)
#pragma unroll
          for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int u = 0; u < kV; ++u) q[d][i][u] = q[d + 1][i][u];
      }
    }
  } else if (warp == kMmaWarp) {
    if (rank != 0) {
      // ============================ peer: relay "my stage is full" to the leader ==========
      uint32_t it = 0;
      for (int pair = pair0; pair < n_pairs; pair += pair_step) {
        for (int c = 0; c < n_chunks; ++c, ++it) {
          const int s = it % n_stages;
          const uint32_t ph = (it / n_stages) & 1;
          mbar_wait(smem_u32(&sh.full[s]), ph);
          if (lane == 0) mbar_arrive_cluster(mapa_u32(smem_u32(&sh.peer_full[s]), 0));
          __syncwarp();
        }
      }
    } else {
      // ============================ leader: MMA issuer for the pair =======================
      // instruction descriptor: D = F32, A = B = TF32, both K-major, N = cout, M = 256 (128 per CTA)
      // (kF16: A = B = F16, format code 0; K per instruction 16 halves = the same 32 bytes)
      const uint32_t fmt = kF16 ? 0u : 2u;
      const uint32_t idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(cout >> 3) << 17) |
                             ((uint32_t)((2 * kTileM) >> 4) << 24);
      uint32_t it = 0, tile_iter = 0;
      for (int pair = pair0; pair < n_pairs; pair += pair_step, ++tile_iter) {
        const uint32_t buf = tile_iter & 1;
        const uint32_t tmem_d = tmem_base + buf * acc_stride;
        mbar_wait_cluster(smem_u32(&sh.acc_empty[buf]), ((tile_iter >> 1) & 1) ^ 1);
        tc_fence_after();
        for (int c = 0; c < n_chunks; ++c, ++it) {
          const int s = it % n_stages;
          const uint32_t ph = (it / n_stages) & 1;
          mbar_wait(smem_u32(&sh.full[s]), ph);
          mbar_wait_cluster(smem_u32(&sh.peer_full[s]), ph);
          tc_fence_after();
          if (lane == 0) {
            const uint32_t a_hi = smem_u32(stage0 + (size_t)s * stage_bytes);
            const uint32_t a_lo = a_hi + kATileBytes;
            const uint32_t b_hi = a_lo + kATileBytes;
            const uint32_t b_lo = b_hi + b_half_bytes;
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) {       // 4 k-steps of 32 bytes per 128-byte row
              const uint32_t ko = ks * 32;
              const uint64_t dbh = umma_desc(b_hi + ko);
              if (kF16) {
                tc_mma_f16_pair(tmem_d, umma_desc(a_hi + ko), dbh, idesc, (c | ks) != 0);
                if (passes == 3) {
                  tc_mma_f16_pair(tmem_d, umma_desc(a_lo + ko), dbh, idesc, 1);
                  tc_mma_f16_pair(tmem_d, umma_desc(a_hi + ko), umma_desc(b_lo + ko), idesc, 1);
                }
              } else {
                tc_mma_tf32_pair(tmem_d, umma_desc(a_hi + ko), dbh, idesc, (c | ks) != 0);
                if (passes == 3) {
                  tc_mma_tf32_pair(tmem_d, umma_desc(a_lo + ko), dbh, idesc, 1);
                  tc_mma_tf32_pair(tmem_d, umma_desc(a_hi + ko), umma_desc(b_lo + ko), idesc, 1);
                }
              }
            }
            tc_commit_pair(smem_u32(&sh.empty[s]));                       // frees the stage in both CTAs
            if (c == n_chunks - 1) tc_commit_pair(smem_u32(&sh.acc_full[buf]));
          }
          __syncwarp();
        }
      }
    }
  } else {
    // ================================ epilogue (both CTAs, own 128 rows) ==================
    const int lane_grp = warp & 3;
    unsigned char* epi_stage = stage0 + (size_t)n_stages * stage_bytes + (warp - kLoaderWarps - 1) * 4096;
    // kF16: the accumulator holds (sx * x) . (sw * w); both scales are powers of two, undone exactly here
    const float inv = kF16 ? __ldg(w_inv_scale) / f16_scale_for(__ldg(amax_in)) : 1.f;
    uint32_t tile_iter = 0;
    for (int pair = pair0; pair < n_pairs; pair += pair_step, ++tile_iter) {
      const int tile = 2 * pair + (int)rank;
      const uint32_t buf = tile_iter & 1;
      const int kappa = tile_k[tile];
      const int p0 = tile_start[tile];
      const int rows = min(kTileM, kofs[kappa + 1] - p0);
      const int r = lane_grp * 32 + lane;
      const int j = r < rows ? out_idx[p0 + r] : -1;
      mbar_wait(smem_u32(&sh.acc_full[buf]), (tile_iter >> 1) & 1);
      tc_fence_after();
      const uint32_t taddr = tmem_base + buf * acc_stride + ((uint32_t)(lane_grp * 32) << 16);
      int col = 0;
      for (; col + 32 <= cout; col += 32) {
        uint32_t v[32];
        tc_ld32(taddr + col, v);
        if (kF16) {
#pragma unroll
          for (int e = 0; e < 32; ++e) v[e] = __float_as_uint(__uint_as_float(v[e]) * inv);
        }
        if (epi) scatter32_lines(epi_stage, lane, out, cout, col, j, v);
        else scatter32_rows(out, cout, col, j, v);
      }
      if (col < cout) {   // cout % 32 == 16
        uint32_t v[16];
        tc_ld16(taddr + col, v);
        if (kF16) {
#pragma unroll
          for (int e = 0; e < 16; ++e) v[e] = __float_as_uint(__uint_as_float(v[e]) * inv);
        }
        if (j >= 0) {
          float* dst = out + (size_t)j * cout + col;
#pragma unroll
          for (int q = 0; q < 4; ++q)
            red_add_v4(dst + 4 * q, __uint_as_float(v[4 * q]), __uint_as_float(v[4 * q + 1]),
                       __uint_as_float(v[4 * q + 2]), __uint_as_float(v[4 * q + 3]));
        }
      }
      tc_fence_before();
      if (rank == 0) mbar_arrive(smem_u32(&sh.acc_empty[buf]));
      else mbar_arrive_cluster(mapa_u32(smem_u32(&sh.acc_empty[buf]), 0));
    }
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();          // nobody exits (or frees TMEM) while the peer may still use or signal it
  if (warp == kMmaWarp) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base),
                 "r"((uint32_t)tmem_cols)
                 : "memory");
  }
}

// W[K, cin, cout] fp32  ->  packed[K][cin/32][2][cout][32]: for every (kappa, 32-channel chunk) the
// K-major SWIZZLE_128B shared-memory image of the B operand, TF32 "hi" tile followed by the "lo"
// residual tile - exactly what one bulk copy drops into a pipeline stage.
__global__ void pack_weight_kernel(const float* __restrict__ w, int cin, int cout, float* __restrict__ packed) {
  const int n_chunks = cin / kChunk;
  const int64_t total = (int64_t)n_chunks * cout * 8;          // 16-byte pieces per kappa
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= total) return;
  const int kappa = blockIdx.y;
  const int n = (int)(e % cout);                                 // output channel = B row (fastest: coalesced)
  const int q = (int)((e / cout) % 8);                           // 16-byte piece inside the 128-byte row
  const int ch = (int)(e / ((int64_t)cout * 8));
  const float* src = w + ((size_t)kappa * cin + ch * kChunk + q * 4) * cout + n;
  float4 v = make_float4(src[0], src[cout], src[2 * (size_t)cout], src[3 * (size_t)cout]);
  float4 h, l;
  h.x = tf32_round(v.x); h.y = tf32_round(v.y); h.z = tf32_round(v.z); h.w = tf32_round(v.w);
  l.x = v.x - h.x; l.y = v.y - h.y; l.z = v.z - h.z; l.w = v.w - h.w;
  float* slab = packed + ((size_t)kappa * n_chunks + ch) * 2 * cout * 32;
  const int off = n * 32 + ((q ^ (n & 7)) << 2);                 // floats
  *reinterpret_cast<float4*>(slab + off) = h;
  *reinterpret_cast<float4*>(slab + (size_t)cout * 32 + off) = l;
}

// |x| maximum of a tensor as float bits (non-negative floats order like unsigned ints)
__global__ void absmax_kernel(const float* __restrict__ x, int64_t n, unsigned* __restrict__ out) {
  float m = 0.f;
  const int64_t n4 = n >> 2;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(x) + i);
    m = fmaxf(fmaxf(m, fmaxf(fabsf(v.x), fabsf(v.y))), fmaxf(fabsf(v.z), fabsf(v.w)));
  }
  if (blockIdx.x == 0 && threadIdx.x < (n & 3)) m = fmaxf(m, fabsf(x[(n4 << 2) + threadIdx.x]));
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, d));
  if ((threadIdx.x & 31) == 0 && m > 0.f) atomicMax(out, __float_as_uint(m));
}

// W[K, cin, cout] fp32 -> packed[K][cin/64][2][cout][64 halves]: per (kappa, 64-channel chunk) the K-major
// SWIZZLE_128B image of the B operand, fp16 hi tile then fp16 lo tile of (sw * W); scale[0] = 1 / sw.
__global__ void pack_weight_f16_kernel(const float* __restrict__ w, int cin, int cout, const float* __restrict__ amax,
                                       unsigned char* __restrict__ packed, float* __restrict__ scale) {
  const int n_chunks = cin / 64;
  const int64_t total = (int64_t)n_chunks * cout * 8;          // 16-byte pieces (8 halves) per kappa
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const float sw = f16_scale_for(*amax);
  if (e == 0 && blockIdx.y == 0) scale[0] = 1.f / sw;
  if (e >= total) return;
  const int kappa = blockIdx.y;
  const int n = (int)(e % cout);
  const int q = (int)((e / cout) % 8);
  const int ch = (int)(e / ((int64_t)cout * 8));
  const float* src = w + ((size_t)kappa * cin + ch * 64 + q * 8) * cout + n;
  uint32_t h[4], l[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float x0 = src[(size_t)(2 * i) * cout] * sw, x1 = src[(size_t)(2 * i + 1) * cout] * sw;
    const __half2 hh = __floats2half2_rn(x0, x1);
    const float2 hf = __half22float2(hh);
    const __half2 ll = __floats2half2_rn(x0 - hf.x, x1 - hf.y);
    h[i] = *reinterpret_cast<const uint32_t*>(&hh);
    l[i] = *reinterpret_cast<const uint32_t*>(&ll);
  }
  unsigned char* slab = packed + ((size_t)kappa * n_chunks + ch) * 2 * cout * 128;
  const int off = n * 128 + ((q ^ (n & 7)) << 4);
  *reinterpret_cast<uint4*>(slab + off) = make_uint4(h[0], h[1], h[2], h[3]);
  *reinterpret_cast<uint4*>(slab + (size_t)cout * 128 + off) = make_uint4(l[0], l[1], l[2], l[3]);
}

}  // namespace

extern "C" {

// Layout transform the tensor-core path needs once per layer: W[K, cin, cout] ->
// packed[K][cin/32][2][cout][32] (TF32 hi / lo tiles in shared-memory image order), 2x the size.
int32_t dgr_pack_weight_tf32(const float* w, int32_t K, int32_t cin, int32_t cout, float* packed, void* stream) {
  DGR_ARG_CHECK(K >= 1 && cin >= 32 && cin % 32 == 0 && cout >= 8 && cout % 8 == 0, "bad weight shape");
  DGR_ARG_CHECK(K <= 65535, "K too large");
  const int64_t per_k = (int64_t)(cin / kChunk) * cout * 8;
  dim3 grid(dgr_blocks(per_k, 256), K);
  pack_weight_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(w, cin, cout, packed);
  dgr_note_launches(1);
  DGR_LAUNCH_CHECK();
  return DGR_OK;
}

// 1 if dgr_spconv_tc_fwd supports the shape (cin % 32 == 0, cout % 16 == 0, 16 <= cout <= 256).
int32_t dgr_spconv_tc_supported(int32_t cin, int32_t cout) {
  return (cin >= 32 && cin % 32 == 0 && cout >= 16 && cout <= 256 && cout % 16 == 0) ? 1 : 0;
}

// Tensor-core variant of dgr_spconv_fwd.  weight_t is the packed layout of dgr_pack_weight_tf32.
// passes = 3: 3xTF32 (fp32-accurate, default); passes = 1: single TF32 product (~1e-3 rel.).
int32_t dgr_spconv_tc_fwd(const float* in_feat, int32_t cin, const float* weight_t, int32_t cout,
                          const int32_t* in_idx, const int32_t* out_idx, const int32_t* kofs,
                          const int32_t* tile_k, const int32_t* tile_start, int32_t n_tiles,
                          int32_t tile_rows, int32_t passes, int32_t cluster, float* out, void* stream) {
  DGR_ARG_CHECK(tile_rows == kTileM, "tile_rows must be 128");
  DGR_ARG_CHECK(dgr_spconv_tc_supported(cin, cout), "shape not supported by the tensor-core path");
  DGR_ARG_CHECK(passes == 1 || passes == 3, "passes must be 1 or 3");
  DGR_ARG_CHECK(cluster >= 0 && cluster <= 3,
                "variant must be 0 (A in TMEM), 1 (A in smem), 2 (CTA pairs, multicast B) or 3 (cta_group::2)");
  if (n_tiles == 0) return DGR_OK;
  cudaStream_t st = (cudaStream_t)stream;
  // gather lookahead in chunks (1..3); DGR_TC_PREFETCH overrides the default for experiments
  static const int pd = [] {
    const char* e = getenv("DGR_TC_PREFETCH");
    int v = e ? atoi(e) : 1;
    return v < 1 ? 1 : (v > 3 ? 3 : v);
  }();
  const int stage_bytes = 2 * kATileBytes + 2 * cout * 128;
  const int n_chunks = cin / kChunk;
  int n_stages = (200 * 1024) / stage_bytes;
  if (n_stages > 4) n_stages = 4;
  if (n_stages < 2) n_stages = 2;
  const size_t smem = sizeof(TcShared) + 1024 + (size_t)n_stages * stage_bytes + kEpiStageBytes;
  // epilogue scatter: 1 = line-coalesced through shared memory (default), 0 = one row per lane
  static const int epi = [] {
    const char* e = getenv("DGR_TC_EPILOGUE");
    return e ? (atoi(e) != 0) : 1;
  }();
  int acc_cols = 32;                       // one accumulator: power of two >= cout
  while (acc_cols < cout) acc_cols <<= 1;
  const int tmem_cols = 2 * acc_cols;      // two accumulators: epilogue overlaps the next tile
  int dev = 0, sms = 148;
  DGR_CUDA_CHECK(cudaGetDevice(&dev));
  DGR_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  (void)n_chunks;
  int grid = sms;                          // persistent: one warp-specialised CTA per SM
  if (grid > n_tiles) grid = n_tiles;
  if (cluster == 0) {
    // A operand in tensor memory: shared memory holds only the weight slabs
    const int sb = 2 * cout * 128;
    int ns = (200 * 1024) / sb;
    if (ns > 4) ns = 4;
    int n_acc = 2;
    if (2 * acc_cols + 64 * 2 > 512) n_acc = 1;            // cout > 128: one accumulator
    while (ns > 2 && n_acc * acc_cols + 64 * ns > 512) --ns;
    int cols = 32;
    while (cols < n_acc * acc_cols + 64 * ns) cols <<= 1;
    const size_t smem_at = sizeof(TcAtShared) + 1024 + (size_t)ns * sb;
    DGR_ENSURE_SMEM(spconv_tc_at_kernel, smem_at);
    spconv_tc_at_kernel<<<grid, kThreadsTC, smem_at, st>>>(in_feat, cin, weight_t, cout, in_idx, out_idx, kofs,
                                                           tile_k, tile_start, n_tiles, ns, cols, n_acc, acc_cols,
                                                           passes, out);
  } else if (cluster == 3) {
    // cta_group::2: one M = 256 MMA per tile pair, each CTA holds half of every weight tile
    DGR_ARG_CHECK(n_tiles % 2 == 0, "a paired tile list has an even number of tiles");
    const int sb2 = 2 * kATileBytes + cout * 128;
    int ns2 = (200 * 1024) / sb2;
    if (ns2 > 4) ns2 = 4;
    const size_t smem2 = sizeof(Tc2Shared) + 1024 + (size_t)ns2 * sb2 + kEpiStageBytes;
    grid = sms & ~1;
    if (grid > n_tiles) grid = n_tiles;
    auto pair_kernel = pd == 1 ? spconv_tc_pair_kernel<1, false> : pd == 2 ? spconv_tc_pair_kernel<2, false> : spconv_tc_pair_kernel<3, false>;
    DGR_ENSURE_SMEM(pair_kernel, smem2);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(kThreadsTC);
    cfg.dynamicSmemBytes = smem2;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    DGR_CUDA_CHECK(cudaLaunchKernelEx(&cfg, pair_kernel, in_feat, (int)cin, weight_t, (int)cout, in_idx,
                                      out_idx, kofs, tile_k, tile_start, (int)n_tiles, ns2, tmem_cols,
                                      (int)passes, epi, (const float*)nullptr, (const float*)nullptr, out));
  } else if (cluster == 2) {
    // CTA pairs on two tiles of the same offset, B tiles multicast to both (paired tile list)
    DGR_ARG_CHECK(n_tiles % 2 == 0, "a paired tile list has an even number of tiles");
    grid &= ~1;
    auto k2 = pd == 1 ? spconv_tc_kernel<2, 1> : pd == 2 ? spconv_tc_kernel<2, 2> : spconv_tc_kernel<2, 3>;
    DGR_ENSURE_SMEM(k2, smem);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(kThreadsTC);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    DGR_CUDA_CHECK(cudaLaunchKernelEx(&cfg, k2, in_feat, (int)cin, weight_t, (int)cout, in_idx,
                                      out_idx, kofs, tile_k, tile_start, (int)n_tiles, n_stages, tmem_cols,
                                      (int)passes, epi, out));
  } else {
    auto k1 = pd == 1 ? spconv_tc_kernel<1, 1> : pd == 2 ? spconv_tc_kernel<1, 2> : spconv_tc_kernel<1, 3>;
    DGR_ENSURE_SMEM(k1, smem);
    k1<<<grid, kThreadsTC, smem, st>>>(in_feat, cin, weight_t, cout, in_idx, out_idx, kofs,
                                                        tile_k, tile_start, n_tiles, n_stages, tmem_cols, passes,
                                                        epi, out);
  }
  dgr_note_launches(1);
  DGR_LAUNCH_CHECK();
  return DGR_OK;
}

// amax[0] (device float) = max |x| over n floats; the slot is zeroed by the call.
int32_t dgr_absmax_f32(const float* x, int64_t n, float* amax, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  DGR_CUDA_CHECK(cudaMemsetAsync(amax, 0, sizeof(float), st));
  if (n <= 0) return DGR_OK;
  unsigned blocks = dgr_blocks(n / 4 + 1, 256);
  if (blocks > 592) blocks = 592;
  absmax_kernel<<<blocks, 256, 0, st>>>(x, n, reinterpret_cast<unsigned*>(amax));
  dgr_note_launches(1);
  DGR_LAUNCH_CHECK();
  return DGR_OK;
}

// 1 if dgr_spconv_tc_f16_fwd supports the shape: the cta_group::2 kernel in 3xFP16 mode
int32_t dgr_spconv_tc_f16_supported(int32_t cin, int32_t cout) {
  return (cin >= 64 && cin % 64 == 0 && cout >= 32 && cout <= 256 && cout % 32 == 0) ? 1 : 0;
}

// W[K, cin, cout] -> fp16 hi|lo slabs [K][cin/64][2][cout][64] (4 * K * cin * cout BYTES, half of the TF32
// slabs) of sw * W with sw the power of two that maps max|W| into [2^14, 2^15); scale_ws (device float[2]):
// [0] = 1 / sw (read by the kernel's epilogue), [1] = max |W| (workspace).
int32_t dgr_pack_weight_f16(const float* w, int32_t K, int32_t cin, int32_t cout, void* packed, float* scale_ws,
                            void* stream) {
  DGR_ARG_CHECK(K >= 1 && K <= 65535 && dgr_spconv_tc_f16_supported(cin, cout), "bad weight shape");
  DGR_TRY_RC(dgr_absmax_f32(w, (int64_t)K * cin * cout, scale_ws + 1, stream));
  const int64_t per_k = (int64_t)(cin / 64) * cout * 8;
  dim3 grid(dgr_blocks(per_k, 256), K);
  pack_weight_f16_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(w, cin, cout, scale_ws + 1, (unsigned char*)packed,
                                                               scale_ws);
  dgr_note_launches(1);
  DGR_LAUNCH_CHECK();
  return DGR_OK;
}

// dgr_spconv_tc_fwd's cta_group::2 kernel with every product evaluated as hi*hi + lo*hi + hi*lo on FP16 splits
// of power-of-two-scaled operands (same 2^-21 accuracy as 3xTF32, half the weight bytes, twice the tensor rate).
// amax_in: device float = max |in_feat| (dgr_absmax_f32, or an upper bound); w_scale: scale_ws of
// dgr_pack_weight_f16.  Needs the PAIRED tile list (dgr_kernel_map_tiles(pair = 1)).
int32_t dgr_spconv_tc_f16_fwd(const float* in_feat, int32_t cin, const void* weight_h, int32_t cout,
                              const int32_t* in_idx, const int32_t* out_idx, const int32_t* kofs,
                              const int32_t* tile_k, const int32_t* tile_start, int32_t n_tiles, int32_t tile_rows,
                              const float* amax_in, const float* w_scale, float* out, void* stream) {
  DGR_ARG_CHECK(tile_rows == kTileM, "tile_rows must be 128");
  DGR_ARG_CHECK(dgr_spconv_tc_f16_supported(cin, cout), "shape not supported by the 3xFP16 path");
  DGR_ARG_CHECK(n_tiles % 2 == 0, "a paired tile list has an even number of tiles");
  DGR_ARG_CHECK(amax_in != nullptr && w_scale != nullptr, "scales missing");
  if (n_tiles == 0) return DGR_OK;
  cudaStream_t st = (cudaStream_t)stream;
  static const int pd = [] {
    const char* e = getenv("DGR_TC_PREFETCH");
    int v = e ? atoi(e) : 1;
    return v < 1 ? 1 : (v > 2 ? 2 : v);
  }();
  int acc_cols = 32;
  while (acc_cols < cout) acc_cols <<= 1;
  const int tmem_cols = 2 * acc_cols;
  int dev = 0, sms = 148;
  DGR_CUDA_CHECK(cudaGetDevice(&dev));
  DGR_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const int sb2 = 2 * kATileBytes + cout * 128;
  int ns2 = (200 * 1024) / sb2;
  if (ns2 > 4) ns2 = 4;
  const size_t smem2 = sizeof(Tc2Shared) + 1024 + (size_t)ns2 * sb2 + kEpiStageBytes;
  int grid = sms & ~1;
  if (grid > n_tiles) grid = n_tiles;
  auto kern = pd == 1 ? spconv_tc_pair_kernel<1, true> : spconv_tc_pair_kernel<2, true>;
  DGR_ENSURE_SMEM(kern, smem2);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(kThreadsTC);
  cfg.dynamicSmemBytes = smem2;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  DGR_CUDA_CHECK(cudaLaunchKernelEx(&cfg, kern, in_feat, (int)cin, (const float*)weight_h, (int)cout, in_idx, out_idx,
                                    kofs, tile_k, tile_start, (int)n_tiles, ns2, tmem_cols, 3, 1, amax_in, w_scale,
                                    out));
  dgr_note_launches(1);
  DGR_LAUNCH_CHECK();
  return DGR_OK;
}

}  // extern "C"
