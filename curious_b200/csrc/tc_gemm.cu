// Large-batch layer GEMMs of the DDPG actor/critic MLPs on the 5th-generation tensor cores (sm_100a).
//
// Replaces, for batches where the tensor pipe pays off (BASELINE config 5, per-GPU batch sweep 256-16384), the dense
// layers of reference baselines/her/util.py:56-107 (forward), and the tf.gradients of ddpg.py:443-449 through them
// (dX = dY W^T, dW = X^T dY) - the same problems the FFMA grouped kernel (mlp_kernels.cuh) executes at batch 256.
//
// Precision: the parity target is an fp32 restatement of the TF graph (rel 1e-5, SURVEY 8c), which a single TF32 pass
// (10-bit mantissa) misses by two orders of magnitude.  Every operand is therefore split in shared memory into
//   x = hi + lo,  hi = x rounded to TF32,  lo = x - hi (exact in fp32, then cut to TF32)      ("3xTF32")
// and each k-step issues three tcgen05.mma.kind::tf32: hi*hi into TMEM accumulator 0, lo*hi + hi*lo into TMEM
// accumulator 1.  Two accumulators because the tensor core's fp32 accumulation does not round to nearest: keeping the
// small cross terms out of the large sum cuts the number of lossy additions into it by 3x; the epilogue adds the two.
//
// One CTA = one 128 x 256 output tile (one K split of it), 14 warps, warp specialised:
//   warp 0      TMA producer: raw fp32 operand tiles, cp.async.bulk.tensor.2d with 128-byte swizzle, 2-stage ring,
//               mbarrier complete_tx; out-of-bounds rows / columns are zero-filled by the TMA unit, which is how
//               K = 44..60 first layers and M = 12..48 first-layer weight gradients ride the same 128 x 256 x 32 tiles
//   warps 2-5   splitters: rewrite the landed tile in place as `hi` and write `lo` next to it (element-wise integer /
//               FADD work, so the swizzled image is preserved), fence.proxy.async, arrive on the "split" barrier
//   warp 1      MMA issuer: one lane issues 4 k-steps x 3 tcgen05.mma (M=128, N=256, K=8) per stage from shared-memory
//               descriptors, tcgen05.commit frees the stage / publishes the accumulators; owns the TMEM allocation
//   warps 6-13  epilogue: tcgen05.ld (32 lanes x 32 columns per warp and instruction), transposed through a padded
//               shared-memory slab so that bias / ReLU / ReLU-mask and the stores are 128-byte coalesced
// Operands are read in their NATIVE row-major orientation; whether an operand is K-major or MN-major for the MMA is
// expressed in the shared-memory / instruction descriptors only:
//   K-major  (fwd A = X[n][K]; dX B = W[k_in][n_out]): one box {32 k, 128|256 rows}, SWIZZLE_128B; k-step = +32 B
//   MN-major (fwd B = W[K][N]; dW A = X[n][M], B = dY[n][N]): boxes {32 mn, 32 k rows}, one per 32-wide MN block
//             (LBO = 4 KB), SWIZZLE_128B_BASE32B (the only MN-major layout 32-bit operands have); k-step = +1 KB
// A problem may have a second K segment (first layer: [o|td|u] W0 + g W0g, util.py:92-99) - the producer switches
// tensor maps, the accumulators keep going.  The weight gradients have K = batch: K is split over CTAs into partial
// tiles that a second small kernel sums in fixed order (deterministic, no atomics).
#include <cuda.h>
#include <stdlib.h>
#include <string.h>

#include "net_layout.cuh"
#include "tc_gemm.cuh"
#include "tc_ptx.cuh"

namespace cur {

constexpr int TC_BM = 128;
constexpr int TC_BN = 256;
// floats per stage and k-block / ring depth.  32 x 2 (128-byte K-major rows, SWIZZLE_128B) and 16 x 4 (64-byte rows,
// SWIZZLE_64B) both work; measured the same speed within 5 % (accumulator ready after 22.1 k vs 23.4 k cycles at
// K = 256): the main loop is bound by shared-memory bandwidth (TMA writes + split + three operand passes), not by the
// depth of the ring.
constexpr int TC_BK = 32;
constexpr int TC_STAGES = 2;
constexpr int TC_MNBLK = TC_BK * 128;           // bytes of one 32-wide MN block of an MN-major operand tile
static_assert(TC_BK == 16 || TC_BK == 32, "K-major rows are one 64- or 128-byte swizzle row");
constexpr int TC_A_BYTES = TC_BM * TC_BK * 4;   // 16 KB
constexpr int TC_B_BYTES = TC_BN * TC_BK * 4;   // 32 KB
constexpr int TC_STAGE_BYTES = 2 * TC_A_BYTES + 2 * TC_B_BYTES;   // A_hi | A_lo | B_hi | B_lo = 96 KB
constexpr int TC_SPLIT_GROUPS = 1;                             // split groups take alternate k-blocks; 2 groups x (16 x 4)
constexpr int TC_SPLIT_GROUP_WARPS = 4;                        // measured no faster than 1 group x (32 x 2), see profiles/
constexpr int TC_SPLIT_WARPS = TC_SPLIT_GROUPS * TC_SPLIT_GROUP_WARPS;
constexpr int TC_SPLIT_WARP0 = 2, TC_EPI_WARP0 = TC_SPLIT_WARP0 + TC_SPLIT_WARPS;
constexpr int TC_EPI_WARPS = 8;                                // two per TMEM lane quarter, 4 column chunks each
constexpr int TC_THREADS = (TC_EPI_WARP0 + TC_EPI_WARPS) * 32;   // 576
constexpr int TC_EPI_LD = 36;                                  // padded row of the epilogue slab (floats)
constexpr int TC_EPI_BYTES = TC_EPI_WARPS * 32 * TC_EPI_LD * 4;   // one 32 x 32 slab per epilogue warp
static_assert(TC_EPI_BYTES <= TC_STAGE_BYTES, "the epilogue slabs reuse stage 0 once the accumulators are complete");
constexpr size_t TC_SMEM_BYTES = (size_t)TC_STAGES * TC_STAGE_BYTES + 1024 /* alignment slack */ + 256 /* barriers */;
constexpr int TC_TMEM_COLS = 512;                              // accumulator 0: columns 0..255, accumulator 1: 256..511

struct TcProb {
  int M, N, K;
  int a_mn, b_mn;                 // 1: operand is MN-major in memory
  int splits, k_per_split;        // K split over CTAs (weight gradients)
  int nkb1, nkb2;                 // k-blocks of 32 per CTA: first segment (of this split), second segment
  float* C; int64_t ldc; int64_t split_stride;   // split s writes C + s * split_stride
  const float* bias; const float* aux; int64_t ldaux; int epi;
  int tile_begin, tiles_m;
};

struct __align__(64) TcBatch {
  CUtensorMap mapA[TC_MAX_PROBS];
  CUtensorMap mapB[TC_MAX_PROBS];
  CUtensorMap mapA2[TC_MAX_PROBS];   // second K segment (nkb2 > 0)
  CUtensorMap mapB2[TC_MAX_PROBS];
  TcProb p[TC_MAX_PROBS];
  int n, total_tiles;
  long long* tl;                     // debug timeline of CTA 0 (cur_tc_gemm_timeline), normally NULL
};

// Epilogue of one warp: 4 column chunks of 32 for its 32 accumulator rows.  Per chunk: both accumulators TMEM ->
// registers (lane = row), summed, transposed through the warp's padded shared-memory slab so that 8 lanes cover one
// 128-byte row segment, then bias / ReLU / ReLU-mask and 16-byte coalesced stores.  Bias and the mask of the first
// chunk are fetched before the accumulators are waited for; the next chunk's mask streams in behind the stores.
template <int EPI, bool FULL>
__device__ __forceinline__ void tc_epilogue(const TcProb& P, uint32_t taddr, float* slab, float* cbase, int row0, int c_begin,
                                            int lane, uint32_t accb, long long* tl) {
  const int rr = lane >> 3, ch = lane & 7;            // phase 2: this lane owns rows rr + 4 i, columns 4 ch .. 4 ch + 3
  const int M = P.M;
  const int64_t ldc = P.ldc, ldaux = P.ldaux;
  const float* aux = P.aux + (int64_t)(row0 + rr) * ldaux + 4 * ch;
  float* crow = cbase + (int64_t)(row0 + rr) * ldc + 4 * ch;
  float4 bias4[4];
#pragma unroll
  for (int cc = 0; cc < 4; ++cc)
    bias4[cc] = P.bias ? *reinterpret_cast<const float4*>(P.bias + (c_begin + cc) * 32 + 4 * ch) : make_float4(0.f, 0.f, 0.f, 0.f);
  float4 mk[8];
  if (EPI == EPI_RELU_MASK) {
#pragma unroll
    for (int i = 0; i < 8; ++i)
      if (FULL || row0 + rr + 4 * i < M) mk[i] = *reinterpret_cast<const float4*>(aux + (int64_t)(4 * i) * ldaux + c_begin * 32);
  }
  tc_bar_wait(accb, 0);
  tc_fence_after();
  if (tl) tl[88] = clock64();
#pragma unroll 1
  for (int cc = 0; cc < 4; ++cc) {
    const int c = c_begin + cc;
    uint32_t r0[32], r1[32];
    tc_ld32(taddr + (uint32_t)(c * 32), r0);
    tc_ld32(taddr + (uint32_t)(TC_BN + c * 32), r1);
    tc_ld_wait();
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float4 v;
      v.x = __uint_as_float(r0[4 * j]) + __uint_as_float(r1[4 * j]);
      v.y = __uint_as_float(r0[4 * j + 1]) + __uint_as_float(r1[4 * j + 1]);
      v.z = __uint_as_float(r0[4 * j + 2]) + __uint_as_float(r1[4 * j + 2]);
      v.w = __uint_as_float(r0[4 * j + 3]) + __uint_as_float(r1[4 * j + 3]);
      *reinterpret_cast<float4*>(slab + lane * TC_EPI_LD + 4 * j) = v;      // conflict-free: row pitch 36 floats
    }
    __syncwarp();
    const float4 b = cc == 0 ? bias4[0] : cc == 1 ? bias4[1] : cc == 2 ? bias4[2] : bias4[3];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      float4 v = *reinterpret_cast<const float4*>(slab + (rr + 4 * i) * TC_EPI_LD + 4 * ch);
      v.x += b.x; v.y += b.y; v.z += b.z; v.w += b.w;
      if (EPI == EPI_RELU) {
        v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f);
      } else if (EPI == EPI_RELU_MASK) {
        const float4 a = mk[i];
        v.x = a.x > 0.f ? v.x : 0.f; v.y = a.y > 0.f ? v.y : 0.f; v.z = a.z > 0.f ? v.z : 0.f; v.w = a.w > 0.f ? v.w : 0.f;
        // the next chunk's mask streams in behind this chunk's stores
        if (cc + 1 < 4 && (FULL || row0 + rr + 4 * i < M))
          mk[i] = *reinterpret_cast<const float4*>(aux + (int64_t)(4 * i) * ldaux + (c + 1) * 32);
      }
      if (FULL || row0 + rr + 4 * i < M) *reinterpret_cast<float4*>(crow + (int64_t)(4 * i) * ldc + c * 32) = v;
    }
    __syncwarp();
    if (tl) tl[89 + cc] = clock64();
  }
}

// PAIR: two CTAs of a cluster (one TPC) compute a 256 x 256 tile with tcgen05.mma.cta_group::2: each CTA stages its own 128
// rows of A and only HALF of the B tile (128 of the 256 N columns) - a third less operand traffic through each SM's L2 port
// and shared memory.  Rank 0 issues the MMAs for both; every CTA splits / drains its own half.
template <bool PAIR>
__device__ __forceinline__ void tc_gemm_body(const TcBatch& G) {
  extern __shared__ uint8_t tc_smem_raw[];
  __shared__ uint32_t s_tmem;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (G.tl != nullptr && blockIdx.x == 0 && threadIdx.x == 0) G.tl[0] = clock64();

  // ---- which tile
  int pi = 0;
#pragma unroll 1
  while (pi + 1 < G.n && (PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x) >= G.p[pi + 1].tile_begin) ++pi;
  const TcProb& P = G.p[pi];
  const uint32_t rank = PAIR ? tc_cta_rank() : 0u;
  const int tile = (PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x) - P.tile_begin;
  const int tm = tile % P.tiles_m, split = tile / P.tiles_m;
  const int m0 = PAIR ? tm * 2 * TC_BM + (int)rank * TC_BM : tm * TC_BM;
  constexpr int B_BYTES_OWN = PAIR ? TC_B_BYTES / 2 : TC_B_BYTES;      // bytes of B this CTA stages per k-block
  constexpr int BN_OWN = PAIR ? TC_BN / 2 : TC_BN;
  // stage = A_hi | A_lo | B_hi | B_lo; a CTA of a pair holds half of B, which makes room for a third stage in the same 192 KB
  constexpr int STAGE_BYTES = 2 * TC_A_BYTES + 2 * B_BYTES_OWN;
  constexpr int STAGES = PAIR ? (TC_STAGES * TC_STAGE_BYTES) / STAGE_BYTES : TC_STAGES;
  static_assert(TC_EPI_BYTES <= STAGE_BYTES, "the epilogue slabs reuse stage 0");
  const int k_begin = split * P.k_per_split;
  const int nkb = P.nkb1 + P.nkb2;

  const uint32_t base = (tc_smem(tc_smem_raw) + 1023u) & ~1023u;
  const uint32_t bars = base + STAGES * STAGE_BYTES;
  const uint32_t full = bars, splitb = bars + 8 * STAGES, empty = bars + 16 * STAGES, accb = bars + 24 * STAGES;
  uint8_t* gen_base = tc_smem_raw + (base - tc_smem(tc_smem_raw));

  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) {
      tc_bar_init(full + 8 * s, 1);
      tc_bar_init(splitb + 8 * s, PAIR ? 2 * TC_SPLIT_GROUP_WARPS : TC_SPLIT_GROUP_WARPS);
      tc_bar_init(empty + 8 * s, 1);
    }
    tc_bar_init(accb, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (PAIR) tc_cluster_sync();        // both CTAs' barriers exist before anything in the pair signals or allocates
  if (warp == 1) {
    if (PAIR) {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tc_smem(&s_tmem)), "n"(TC_TMEM_COLS)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tc_smem(&s_tmem)), "n"(TC_TMEM_COLS)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
  }
  tc_fence_before();
  if (PAIR) tc_cluster_sync(); else __syncthreads();
  tc_fence_after();
  const uint32_t tmem = s_tmem;
  long long* tl = (G.tl != nullptr && blockIdx.x == 0 && lane == 0) ? G.tl : nullptr;
  if (tl && warp == 0) tl[1] = clock64();

  if (warp == 0) {
    // ===== TMA producer
    if (lane == 0) {
      for (int kb = 0; kb < nkb; ++kb) {
        const int s = kb % STAGES, round = kb / STAGES;
        if (round > 0) tc_bar_wait(empty + 8 * s, (round - 1) & 1);
        const uint32_t st = base + s * STAGE_BYTES;
        const uint32_t a_hi = st, b_hi = st + 2 * TC_A_BYTES;
        const bool seg2 = kb >= P.nkb1;
        const CUtensorMap* mA = seg2 ? &G.mapA2[pi] : &G.mapA[pi];
        const CUtensorMap* mB = seg2 ? &G.mapB2[pi] : &G.mapB[pi];
        const int k0 = seg2 ? (kb - P.nkb1) * TC_BK : k_begin + kb * TC_BK;
        if (tl && kb < 16) tl[8 + kb] = clock64();
        tc_bar_expect_tx(full + 8 * s, TC_A_BYTES + B_BYTES_OWN);     // zero-filled out-of-bounds bytes count too
        if (!P.a_mn) {
          tc_tma_2d(a_hi, mA, k0, m0, full + 8 * s);                           // [128 m][32 k]
        } else {
          for (int j = 0; j < TC_BM / 32; ++j) tc_tma_2d(a_hi + j * TC_MNBLK, mA, m0 + 32 * j, k0, full + 8 * s);   // [BK k][32 m]
        }
        if (!P.b_mn) {
          tc_tma_2d(b_hi, mB, k0, (int)rank * BN_OWN, full + 8 * s);           // [256 | 128 n][BK k]
        } else {
          for (int j = 0; j < BN_OWN / 32; ++j)
            tc_tma_2d(b_hi + j * TC_MNBLK, mB, (int)rank * BN_OWN + 32 * j, k0, full + 8 * s);                    // [BK k][32 n]
        }
      }
    }
  } else if (warp == 1 && rank == 0) {
    // ===== MMA issuer (the pair's leader issues for both CTAs)
    // instruction descriptor (cute::UMMA::InstrDescriptor): D = F32 (1 << 4), A = B = TF32 (2 << 7, 2 << 10),
    // a_major at 15, b_major at 16, N >> 3 at [17,23), M >> 4 at [24,29)
    const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)P.a_mn << 15) | ((uint32_t)P.b_mn << 16) |
                           ((uint32_t)(TC_BN >> 3) << 17) | ((uint32_t)((PAIR ? 2 * TC_BM : TC_BM) >> 4) << 24);
    const uint32_t a_step = P.a_mn ? 1024u : 32u, b_step = P.b_mn ? 1024u : 32u;   // bytes per k-step of 8
    // K-major: rows of TC_BK floats (64 B: SWIZZLE_64B, layout type 4; 128 B: SWIZZLE_128B, type 2), 8-row groups
    // 8 rows apart (SBO), LBO unused.  MN-major: SWIZZLE_128B_BASE32B (type 1), 32-wide MN blocks TC_MNBLK apart (LBO),
    // 4-row k atoms 512 B apart (SBO)
    constexpr uint32_t kmaj_sbo = 8u * TC_BK * 4u, kmaj_lt = (TC_BK == 32) ? 2u : 4u;
    const uint32_t a_lbo = P.a_mn ? (uint32_t)TC_MNBLK : 16u, b_lbo = P.b_mn ? (uint32_t)TC_MNBLK : 16u;
    const uint32_t a_sbo = P.a_mn ? 512u : kmaj_sbo, b_sbo = P.b_mn ? 512u : kmaj_sbo;
    const uint32_t a_lt = P.a_mn ? 1u : kmaj_lt, b_lt = P.b_mn ? 1u : kmaj_lt;
    for (int kb = 0; kb < nkb; ++kb) {
      const int s = kb % STAGES, round = kb / STAGES;
      if (PAIR) tc_bar_wait_cluster(splitb + 8 * s, round & 1); else tc_bar_wait(splitb + 8 * s, round & 1);
      tc_fence_after();
      if (tl && kb < 16) tl[56 + 2 * kb] = clock64();
      if (lane == 0) {
        const uint32_t st = base + s * STAGE_BYTES;
        const uint32_t a_hi = st, a_lo = st + TC_A_BYTES, b_hi = st + 2 * TC_A_BYTES, b_lo = b_hi + B_BYTES_OWN;
#pragma unroll
        for (int ks = 0; ks < TC_BK / 8; ++ks) {
          const uint64_t dah = tc_desc(a_hi + ks * a_step, a_lbo, a_sbo, a_lt), dal = tc_desc(a_lo + ks * a_step, a_lbo, a_sbo, a_lt);
          const uint64_t dbh = tc_desc(b_hi + ks * b_step, b_lbo, b_sbo, b_lt), dbl = tc_desc(b_lo + ks * b_step, b_lbo, b_sbo, b_lt);
          if (PAIR) {
            tc_mma_tf32_pair(tmem + TC_BN, dal, dbh, idesc, (kb | ks) != 0);
            tc_mma_tf32_pair(tmem + TC_BN, dah, dbl, idesc, 1u);
            tc_mma_tf32_pair(tmem, dah, dbh, idesc, (kb | ks) != 0);
          } else {
            tc_mma_tf32(tmem + TC_BN, dal, dbh, idesc, (kb | ks) != 0);      // cross terms -> accumulator 1
            tc_mma_tf32(tmem + TC_BN, dah, dbl, idesc, 1u);
            tc_mma_tf32(tmem, dah, dbh, idesc, (kb | ks) != 0);              // main term   -> accumulator 0
          }
        }
        if (PAIR) {
          tc_commit_pair(empty + 8 * s);
          if (kb == nkb - 1) tc_commit_pair(accb);
        } else {
          tc_commit(empty + 8 * s);                 // stage reusable once these MMAs have read it
          if (kb == nkb - 1) tc_commit(accb);       // accumulators complete
        }
        if (tl && kb < 16) tl[57 + 2 * kb] = clock64();
      }
      __syncwarp();
    }
  } else if (warp >= TC_SPLIT_WARP0 && warp < TC_EPI_WARP0) {
    // ===== splitters
    const int group = (warp - TC_SPLIT_WARP0) / TC_SPLIT_GROUP_WARPS;
    const int t = threadIdx.x - (TC_SPLIT_WARP0 + group * TC_SPLIT_GROUP_WARPS) * 32;
    for (int kb = group; kb < nkb; kb += TC_SPLIT_GROUPS) {
      const int s = kb % STAGES, round = kb / STAGES;
      tc_bar_wait(full + 8 * s, round & 1);
      if (tl && warp == TC_SPLIT_WARP0 && kb < 16) tl[24 + 2 * kb] = clock64();
      float* st = reinterpret_cast<float*>(gen_base + s * STAGE_BYTES);
      tc_split_tile(st, TC_A_BYTES / 4, TC_A_BYTES / 16, t, TC_SPLIT_GROUP_WARPS * 32);
      tc_split_tile(st + 2 * TC_A_BYTES / 4, B_BYTES_OWN / 4, B_BYTES_OWN / 16, t, TC_SPLIT_GROUP_WARPS * 32);
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      __syncwarp();
      if (tl && warp == TC_SPLIT_WARP0 && kb < 16) tl[25 + 2 * kb] = clock64();
      if (lane == 0) {
        if (PAIR) tc_bar_arrive_leader(splitb + 8 * s); else tc_bar_arrive(splitb + 8 * s);
      }
    }
  } else if (warp >= TC_EPI_WARP0) {
    // ===== epilogue (8 warps; warp w may only touch TMEM lanes 32 (w % 4) .. + 31; the two warps of a lane quarter
    // take 4 of the 8 column chunks each)
    const int q = warp & 3, ew = warp - TC_EPI_WARP0;
    const int row0 = m0 + 32 * q;
    float* slab = reinterpret_cast<float*>(gen_base) + ew * 32 * TC_EPI_LD;   // stage 0 is free once `accb` fires
    float* cbase = P.C + (int64_t)split * P.split_stride;
    const bool full_rows = row0 + 32 <= P.M;
    const uint32_t taddr = tmem + ((uint32_t)(32 * q) << 16);
    const int c_begin = (ew >> 2) * 4;
    long long* etl = (tl && warp == TC_EPI_WARP0) ? tl : nullptr;
    // the epilogue kind and the row-tail handling are resolved once, outside the chunk loop
    if (P.epi == EPI_RELU_MASK) {
      if (full_rows) tc_epilogue<EPI_RELU_MASK, true>(P, taddr, slab, cbase, row0, c_begin, lane, accb, etl);
      else tc_epilogue<EPI_RELU_MASK, false>(P, taddr, slab, cbase, row0, c_begin, lane, accb, etl);
    } else if (P.epi == EPI_RELU) {
      if (full_rows) tc_epilogue<EPI_RELU, true>(P, taddr, slab, cbase, row0, c_begin, lane, accb, etl);
      else tc_epilogue<EPI_RELU, false>(P, taddr, slab, cbase, row0, c_begin, lane, accb, etl);
    } else {
      if (full_rows) tc_epilogue<EPI_NONE, true>(P, taddr, slab, cbase, row0, c_begin, lane, accb, etl);
      else tc_epilogue<EPI_NONE, false>(P, taddr, slab, cbase, row0, c_begin, lane, accb, etl);
    }
    tc_fence_before();
  }
  if (PAIR) tc_cluster_sync(); else __syncthreads();
  if (tl && warp == 0) tl[2] = clock64();
  if (warp == 1) {
    tc_fence_after();
    if (PAIR) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(TC_TMEM_COLS) : "memory");
    else asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(TC_TMEM_COLS) : "memory");
  }
}

__global__ void __launch_bounds__(TC_THREADS, 1) tc_gemm_kernel(const __grid_constant__ TcBatch G) { tc_gemm_body<false>(G); }
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(TC_THREADS, 1)
tc_gemm_pair_kernel(const __grid_constant__ TcBatch G) { tc_gemm_body<true>(G); }

// out[i] = sum_s part[s][i], fixed order (split-K weight gradients)
__global__ void __launch_bounds__(256) tc_reduce_kernel(const __grid_constant__ TcReduceBatch R) {
  int pi = 0;
#pragma unroll 1
  while (pi + 1 < R.n && (int)blockIdx.x >= R.p[pi + 1].block_begin) ++pi;
  const TcReduce& P = R.p[pi];
  const int64_t i4 = (int64_t)(blockIdx.x - P.block_begin) * 256 + threadIdx.x;
  if (i4 * 4 >= P.count) return;
  if (P.vec) {
    // fixed order s = 0, 1, 2, ...; the loads of 8 slices are issued together (the loop is latency-bound otherwise)
    float4 acc = *reinterpret_cast<const float4*>(P.part + i4 * 4);
    int s = 1;
    for (; s + 7 < P.splits; s += 8) {
      float4 x[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) x[u] = *reinterpret_cast<const float4*>(P.part + (int64_t)(s + u) * P.stride + i4 * 4);
#pragma unroll
      for (int u = 0; u < 8; ++u) { acc.x += x[u].x; acc.y += x[u].y; acc.z += x[u].z; acc.w += x[u].w; }
    }
    for (; s < P.splits; ++s) {
      const float4 x = *reinterpret_cast<const float4*>(P.part + (int64_t)s * P.stride + i4 * 4);
      acc.x += x.x; acc.y += x.y; acc.z += x.z; acc.w += x.w;
    }
    *reinterpret_cast<float4*>(P.out + i4 * 4) = acc;
  } else {
    for (int64_t i = i4 * 4; i < i4 * 4 + 4 && i < P.count; ++i) {
      float acc = P.part[i];
      for (int s = 1; s < P.splits; ++s) acc += P.part[(int64_t)s * P.stride + i];
      P.out[i] = acc;
    }
  }
}

// Row reductions at large batch, partial over chunks of TC_COLSUM_ROWS rows (summed by tc_reduce_kernel):
//   Y == NULL:  part[chunk][m]    = sum_r X[r][m]                      bias gradients  db = 1^T dY
//   Y != NULL:  part[chunk][m][j] = sum_r X[r][m] * Y[r][j], j < NJ    output-layer weight gradients (N = 1 or dimu)
// Block = 16 column quads x 16 row lanes: every thread owns 4 columns and every 16th row of the chunk; the 16 row
// lanes are folded through shared memory in fixed order.
struct RowRed {
  const float* X; int64_t ldx; const float* Y; int64_t ldy;
  int64_t rows; int M, NJ; float* part;
  int col_blocks, block_begin;
};
struct RowRedBatch {
  RowRed p[TC_MAX_PROBS];
  int n;
};
__global__ void __launch_bounds__(256) tc_rowred_kernel(const __grid_constant__ RowRedBatch R) {
  __shared__ float red[16][16][4 * 4 + 1];
  int pi = 0;
#pragma unroll 1
  while (pi + 1 < R.n && (int)blockIdx.x >= R.p[pi + 1].block_begin) ++pi;
  const RowRed& P = R.p[pi];
  const int lb = blockIdx.x - P.block_begin;
  const int cb = lb % P.col_blocks;
  const int cq = threadIdx.x & 15, rl = threadIdx.x >> 4;
  const int m = cb * 64 + 4 * cq;
  const int chunk = lb / P.col_blocks;
  const int64_t r0 = (int64_t)chunk * TC_COLSUM_ROWS;
  const int64_t r1 = r0 + TC_COLSUM_ROWS < P.rows ? r0 + TC_COLSUM_ROWS : P.rows;
  const int NJ = P.Y ? P.NJ : 1;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  const bool vec = (m + 3 < P.M) && ((P.ldx & 3) == 0) && ((reinterpret_cast<uintptr_t>(P.X) & 15) == 0);
  for (int64_t r = r0 + rl; r < r1; r += 16) {
    float x[4];
    if (vec) {
      const float4 v = *reinterpret_cast<const float4*>(P.X + r * P.ldx + m);
      x[0] = v.x; x[1] = v.y; x[2] = v.z; x[3] = v.w;
    } else {
#pragma unroll
      for (int i = 0; i < 4; ++i) x[i] = (m + i < P.M) ? P.X[r * P.ldx + m + i] : 0.f;
    }
    if (P.Y) {
      float y[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) y[j] = j < NJ ? P.Y[r * P.ldy + j] : 0.f;
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(x[i], y[j], acc[i][j]);
    } else {
#pragma unroll
      for (int i = 0; i < 4; ++i) acc[i][0] += x[i];
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) red[rl][cq][4 * i + j] = acc[i][j];
  __syncthreads();
  // 256 threads -> 16 column quads x 16 (i, j) slots
  const int slot = threadIdx.x >> 4;       // 4 i + j
  const int i = slot >> 2, j = slot & 3;
  float sum = 0.f;
#pragma unroll
  for (int l = 0; l < 16; ++l) sum += red[l][cq][slot];
  const int mm = cb * 64 + 4 * cq + i;
  if (mm < P.M && j < NJ) P.part[((int64_t)chunk * P.M + mm) * NJ + j] = sum;
}

// Skinny problems of the large-batch schedule (M = batch rows, one of N / K is <= 4): bandwidth-bound streams that the
// 32x32-tile FFMA kernel runs at a few percent of HBM speed (scalar generic path).  One grouped launch per level.
//   SK_ROWDOT  out[r][j] = epi( sum_k X[r][k] W(k, j) + b[j] ), N <= 4, K <= 1024: output layers (util.py:65-71,
//              N = 1 critic / dimu actor, tanh) and the action gradient d pi_loss / d(pre-tanh) (ddpg.py:440-447)
//   SK_OUTER   dX[r][c] = mask(aux[r][c]) * sum_{j<K} dY[r][j] W[c][j], K <= 4: backward through the output layers
enum { SK_ROWDOT = 0, SK_OUTER = 1 };
struct Skinny {
  int kind;
  const float* X; int64_t ldx;       // ROWDOT: X [M][K];          OUTER: dY [M][K]
  const float* W; int64_t ldw; int w_nk;   // ROWDOT: W [K][N] (w_nk = 0) or [N][K] (w_nk = 1);  OUTER: W [N][K]
  const float* bias;
  const float* aux; int64_t ldaux;
  float* C; int64_t ldc;
  int M, N, K, epi;
  float coef;
  int block_begin, blocks;
};
struct SkinnyBatch {
  Skinny p[TC_MAX_PROBS];
  int n;
};
constexpr int SK_ROWS_PER_BLOCK = 64;   // ROWDOT: 8 warps x 8 rows; OUTER: 64 rows x N columns per block

__global__ void __launch_bounds__(256) tc_skinny_kernel(const __grid_constant__ SkinnyBatch S) {
  __shared__ __align__(16) float wsm[4 * 1024];
  int pi = 0;
#pragma unroll 1
  while (pi + 1 < S.n && (int)blockIdx.x >= S.p[pi + 1].block_begin) ++pi;
  const Skinny& P = S.p[pi];
  const int lb = blockIdx.x - P.block_begin;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (P.kind == SK_ROWDOT) {
    // weights as [j][k] in shared memory
    for (int i = threadIdx.x; i < P.N * P.K; i += 256) {
      const int j = i / P.K, k = i - j * P.K;
      wsm[j * P.K + k] = P.w_nk ? P.W[(int64_t)j * P.ldw + k] : P.W[(int64_t)k * P.ldw + j];
    }
    __syncthreads();
    const int64_t r0 = (int64_t)lb * SK_ROWS_PER_BLOCK + warp * 8;
    const int k4 = P.K >> 2;
#pragma unroll 1
    for (int rr = 0; rr < 8; rr += 4) {
      float acc[4][4];
#pragma unroll
      for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[a][j] = 0.f;
      for (int q = lane; q < k4; q += 32) {
        float4 x[4];
#pragma unroll
        for (int a = 0; a < 4; ++a) {
          const int64_t r = r0 + rr + a;
          x[a] = r < P.M ? *reinterpret_cast<const float4*>(P.X + r * P.ldx + 4 * q) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          if (j < P.N) {
            const float4 w = *reinterpret_cast<const float4*>(wsm + j * P.K + 4 * q);
#pragma unroll
            for (int a = 0; a < 4; ++a)
              acc[a][j] = fmaf(x[a].w, w.w, fmaf(x[a].z, w.z, fmaf(x[a].y, w.y, fmaf(x[a].x, w.x, acc[a][j]))));
          }
        }
      }
#pragma unroll
      for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) acc[a][j] += __shfl_xor_sync(0xffffffffu, acc[a][j], o);
      // lane 4 a + j writes output (row a, column j)
      const int a = lane >> 2, j = lane & 3;
      if (lane < 16 && j < P.N) {
        const int64_t r = r0 + rr + a;
        if (r < P.M) {
          float v = 0.f;
#pragma unroll
          for (int aa = 0; aa < 4; ++aa)
#pragma unroll
            for (int jj = 0; jj < 4; ++jj)
              if (aa == a && jj == j) v = acc[aa][jj];
          if (P.bias) v += P.bias[j];
          if (P.epi == EPI_TANH) v = tanhf(v);
          else if (P.epi == EPI_ACTOR_DY) {
            const float th = P.aux[r * P.ldaux + j];
            v = (v + P.coef * th) * (1.f - th * th);
          }
          P.C[r * P.ldc + j] = v;
        }
      }
    }
  } else {
    // OUTER: weights [c][j] (j < K <= 4) in shared memory, padded to 4 per column
    for (int i = threadIdx.x; i < P.N * 4; i += 256) {
      const int c = i >> 2, j = i & 3;
      wsm[i] = j < P.K ? P.W[(int64_t)c * P.ldw + j] : 0.f;
    }
    __syncthreads();
    const int n4 = P.N >> 2;
    const int64_t r0 = (int64_t)lb * SK_ROWS_PER_BLOCK;
    for (int i = threadIdx.x; i < SK_ROWS_PER_BLOCK * n4; i += 256) {
      const int64_t r = r0 + i / n4;
      const int c4 = i % n4;
      if (r >= P.M) break;
      float y[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) y[j] = j < P.K ? P.X[r * P.ldx + j] : 0.f;
      float o[4];
#pragma unroll
      for (int cc = 0; cc < 4; ++cc) {
        const float4 w = *reinterpret_cast<const float4*>(wsm + (4 * c4 + cc) * 4);
        // same association as a K-loop: ((y0 w0 + y1 w1) + y2 w2) + y3 w3
        o[cc] = fmaf(y[3], w.w, fmaf(y[2], w.z, fmaf(y[1], w.y, y[0] * w.x)));
      }
      float4 v = make_float4(o[0], o[1], o[2], o[3]);
      if (P.epi == EPI_RELU_MASK) {
        const float4 a = *reinterpret_cast<const float4*>(P.aux + r * P.ldaux + 4 * c4);
        v.x = a.x > 0.f ? v.x : 0.f; v.y = a.y > 0.f ? v.y : 0.f; v.z = a.z > 0.f ? v.z : 0.f; v.w = a.w > 0.f ? v.w : 0.f;
      }
      *reinterpret_cast<float4*>(P.C + r * P.ldc + 4 * c4) = v;
    }
  }
}

// ------------------------------------------------------------------------------------------------ host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// row-major [rows][cols] fp32 with leading dimension ld; K-major operands: box = {TC_BK floats, box_rows}, 16-byte chunks
// swizzled within the 64- / 128-byte row; MN-major operands: box = {32 floats, TC_BK rows}, 32-byte chunks swizzled
// within the 128-byte row
static int make_map(CUtensorMap* m, const float* ptr, int64_t rows, int64_t cols, int64_t ld, int box_rows, bool mn_major) {
  EncodeTiledFn fn = encode_fn();
  CUR_REQUIRE(fn != nullptr, "cuTensorMapEncodeTiled is not available");
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld * 4};
  cuuint32_t box[2] = {mn_major ? 32u : (cuuint32_t)TC_BK, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1u, 1u};
  CUresult rc = fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(ptr), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE,
                   mn_major ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : (TC_BK == 32 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B),
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (rc != CUDA_SUCCESS) {
    snprintf(g_last_error, sizeof(g_last_error), "cuTensorMapEncodeTiled failed (%d): rows %lld cols %lld ld %lld", (int)rc,
             (long long)rows, (long long)cols, (long long)ld);
    return CUR_ERR_CUDA;
  }
  return CUR_OK;
}

int tc_make_map(void* map, const float* ptr, int64_t rows, int64_t cols, int64_t ld, int box_rows, bool mn_major) {
  return make_map(reinterpret_cast<CUtensorMap*>(map), ptr, rows, cols, ld, box_rows, mn_major);
}

static long long* g_tc_timeline = nullptr;
void tc_set_timeline(long long* dev) { g_tc_timeline = dev; }

bool tc_supported(const GemmProb& p) {
  if (p.ones_a || p.C2 != nullptr) return false;
  if (p.N != TC_BN || p.M <= 0 || p.K <= 0) return false;
  if (p.K2 != 0 && (p.a_trans || p.b_trans || p.A2 == nullptr || p.B2 == nullptr)) return false;
  if (!(p.epi == EPI_NONE || p.epi == EPI_RELU || p.epi == EPI_RELU_MASK)) return false;
  auto al = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15) == 0; };
  if (!al(p.A) || !al(p.B) || !al(p.C) || (p.bias && !al(p.bias)) || (p.aux && !al(p.aux))) return false;
  if ((p.lda % 4) || (p.ldb % 4) || (p.ldc % 4) || (p.aux && (p.ldaux % 4))) return false;
  if (p.K2 != 0 && (!al(p.A2) || !al(p.B2) || (p.lda2 % 4) || (p.ldb2 % 4))) return false;
  if (tc_pick_splits(p) > 1 && (p.bias != nullptr || p.epi != EPI_NONE || p.ldc != p.N || p.K2 != 0)) return false;
  return true;
}

// rows of K one CTA of a split weight gradient covers: 256 (8 k-blocks, like every other tile of a dependency level), or -
// split_k == 2, the weight-gradient launch behind the chain kernel, where nothing else shares the launch - 512 above
// batch 2048: a CTA pays ~8 k cycles of prologue / epilogue around ~2.6 k per k-block, and at batch 4864 the 19 x 12 tiles of
// the 256-row split need two waves (41 us) where 10 x 12 tiles of 16 k-blocks fit one (25 us)
static int tc_k_per_split(const GemmProb& p) { return (p.split_k == 2 && p.K > 2048) ? 512 : 256; }

int tc_pick_splits(const GemmProb& p) {
  // forward / dX problems have M = batch: plenty of tiles.  Weight gradients (M <= 256, K = batch) split K over CTAs;
  // the last split may be shorter (the TMA unit zero-fills the rows beyond K)
  if (p.M >= 1024 || !(p.a_trans || p.split_k)) return 1;
  const int kps = tc_k_per_split(p);
  const int s = (p.K + kps - 1) / kps;
  return s < 1 ? 1 : s;
}

int64_t tc_partial_floats(const GemmProb& p) {
  const int s = tc_pick_splits(p);
  return s > 1 ? (int64_t)s * p.M * p.N : 0;
}

// Adds `p` to the batch.  `partial` (tc_partial_floats(p) floats, 16-byte aligned) is needed when K is split.
int TcLauncher::add(const GemmProb& p, float* partial) {
  CUR_REQUIRE(tc_supported(p), "problem does not fit the tensor-core GEMM");
  CUR_REQUIRE(G.n < TC_MAX_PROBS, "too many problems in one tensor-core batch");
  TcBatch& B = *reinterpret_cast<TcBatch*>(storage);
  const int i = G.n;
  TcProb& q = B.p[i];
  memset(&q, 0, sizeof(q));
  q.M = p.M; q.N = p.N; q.K = p.K;
  q.a_mn = p.a_trans ? 1 : 0;          // A stored [K][M]
  q.b_mn = p.b_trans ? 0 : 1;          // B stored [K][N] is N-major; stored [N][K] is K-major
  q.splits = tc_pick_splits(p);
  q.k_per_split = (q.splits > 1) ? tc_k_per_split(p) : p.K;
  q.nkb1 = (q.k_per_split + TC_BK - 1) / TC_BK;       // a K tail is zero-filled by the TMA unit
  q.nkb2 = (p.K2 + TC_BK - 1) / TC_BK;
  q.bias = p.bias; q.aux = p.aux; q.ldaux = p.ldaux; q.epi = p.epi;
  if (q.splits > 1) {
    CUR_REQUIRE(partial != nullptr, "split-K needs a partial buffer");
    q.C = partial; q.ldc = p.N; q.split_stride = (int64_t)p.M * p.N;
    CUR_REQUIRE(R.n < 2 * TC_MAX_PROBS, "too many reductions");
    TcReduce& r = R.p[R.n++];
    r.part = partial; r.out = p.C; r.count = (int64_t)p.M * p.N; r.stride = q.split_stride; r.splits = q.splits;
    r.vec = 1;
  } else {
    q.C = p.C; q.ldc = p.ldc; q.split_stride = 0;
  }
  q.tiles_m = (p.M + TC_BM - 1) / TC_BM;              // rows beyond M: zero-filled operands, stores suppressed
  if (pair) {                                         // CTA pairs: 256-row tiles, each CTA stages half of B
    CUR_REQUIRE(p.M % (2 * TC_BM) == 0, "the CTA-pair kernel needs M to be a multiple of 256");
    q.tiles_m = p.M / (2 * TC_BM);
  }
  q.tile_begin = G.total_tiles;
  G.total_tiles += q.tiles_m * q.splits;
  if (!q.a_mn) CUR_TRY(make_map(&B.mapA[i], p.A, p.M, p.K, p.lda, TC_BM, false));
  else CUR_TRY(make_map(&B.mapA[i], p.A, p.K, p.M, p.lda, TC_BK, true));
  if (!q.b_mn) CUR_TRY(make_map(&B.mapB[i], p.B, p.N, p.K, p.ldb, pair ? TC_BN / 2 : TC_BN, false));
  else CUR_TRY(make_map(&B.mapB[i], p.B, p.K, p.N, p.ldb, TC_BK, true));
  if (q.nkb2 > 0) {                                   // plain NN second segment: A2 [M][K2], B2 [K2][N]
    CUR_TRY(make_map(&B.mapA2[i], p.A2, p.M, p.K2, p.lda2, TC_BM, false));
    CUR_TRY(make_map(&B.mapB2[i], p.B2, p.K2, p.N, p.ldb2, TC_BK, true));
  }
  G.n = i + 1;
  return CUR_OK;
}

int TcLauncher::add_rowred(const float* X, int64_t ldx, int M, const float* Y, int64_t ldy, int NJ, int64_t rows, float* out,
                           float* partial) {
  CUR_REQUIRE(n_rowred < TC_MAX_PROBS && R.n < 2 * TC_MAX_PROBS, "too many row reductions");
  CUR_REQUIRE(X && M > 0 && rows > 0 && partial != nullptr && (Y == nullptr || (NJ >= 1 && NJ <= 4)), "bad row reduction");
  RowRedDesc& c = rowred[n_rowred++];
  c.X = X; c.ldx = ldx; c.Y = Y; c.ldy = ldy; c.rows = rows; c.M = M; c.NJ = Y ? NJ : 1; c.part = partial;
  c.chunks = (int)((rows + TC_COLSUM_ROWS - 1) / TC_COLSUM_ROWS);
  const int64_t count = (int64_t)M * c.NJ;
  TcReduce& r = R.p[R.n++];
  r.part = partial; r.out = out; r.count = count; r.stride = count; r.splits = c.chunks;
  r.vec = ((count % 4) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0 && (reinterpret_cast<uintptr_t>(partial) & 15) == 0) ? 1 : 0;
  return CUR_OK;
}

bool tc_skinny_supported(const GemmProb& p) {
  if (p.ones_a || p.a_trans || p.K2 != 0 || p.C2 != nullptr || p.M <= 0) return false;
  auto al = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15) == 0; };
  if (p.N <= 4 && p.N >= 1 && p.K >= 4 && p.K <= 1024 && (p.K % 4) == 0 && (p.lda % 4) == 0 && al(p.A) &&
      (p.epi == EPI_NONE || p.epi == EPI_TANH || p.epi == EPI_ACTOR_DY))
    return true;                                                        // SK_ROWDOT
  if (p.b_trans && p.K >= 1 && p.K <= 4 && p.N >= 4 && p.N <= 1024 && (p.N % 4) == 0 && (p.ldc % 4) == 0 && al(p.C) &&
      p.bias == nullptr && (p.epi == EPI_NONE || (p.epi == EPI_RELU_MASK && al(p.aux) && (p.ldaux % 4) == 0)))
    return true;                                                        // SK_OUTER
  return false;
}

int TcLauncher::add_skinny(const GemmProb& p) {
  CUR_REQUIRE(tc_skinny_supported(p), "problem does not fit the skinny kernels");
  CUR_REQUIRE(n_skinny < TC_MAX_PROBS, "too many skinny problems");
  SkinnyDesc& q = skinny[n_skinny++];
  q.p = p;
  return CUR_OK;
}

int64_t tc_rowred_partial_floats(int64_t rows, int M, int NJ) {
  return ((rows + TC_COLSUM_ROWS - 1) / TC_COLSUM_ROWS) * (int64_t)M * (NJ < 1 ? 1 : NJ);
}

// The bandwidth-bound helpers of a level (skinny problems, row reductions) are independent of its tensor-core launch:
// they run on a side stream forked from / joined to the caller's stream with events (capturable: inside a CUDA graph
// the two become parallel branches), filling the SMs' idle issue slots and the L2 while the tcgen05 tiles run.
struct SideStream {
  cudaStream_t stream = nullptr;
  cudaEvent_t fork = nullptr, join = nullptr, gemm = nullptr;
  cudaEvent_t red[2] = {nullptr, nullptr};      // "the reductions of the last level that used partial set 0 / 1 are done"
  int device = -1;
};
static int side_stream(SideStream** out) {
  static thread_local SideStream ss;
  int dev = 0;
  CUR_CUDA_TRY(cudaGetDevice(&dev));
  if (ss.stream == nullptr || ss.device != dev) {
    CUR_CUDA_TRY(cudaStreamCreateWithFlags(&ss.stream, cudaStreamNonBlocking));
    CUR_CUDA_TRY(cudaEventCreateWithFlags(&ss.fork, cudaEventDisableTiming));
    CUR_CUDA_TRY(cudaEventCreateWithFlags(&ss.join, cudaEventDisableTiming));
    CUR_CUDA_TRY(cudaEventCreateWithFlags(&ss.gemm, cudaEventDisableTiming));
    CUR_CUDA_TRY(cudaEventCreateWithFlags(&ss.red[0], cudaEventDisableTiming));
    CUR_CUDA_TRY(cudaEventCreateWithFlags(&ss.red[1], cudaEventDisableTiming));
    ss.device = dev;
  }
  *out = &ss;
  return CUR_OK;
}

int TcLauncher::flush(cudaStream_t s_main) {
  TcBatch& B = *reinterpret_cast<TcBatch*>(storage);
  static bool configured = false;
  if (!configured) {
    CUR_CUDA_TRY(cudaFuncSetAttribute(tc_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TC_SMEM_BYTES));
    CUR_CUDA_TRY(cudaFuncSetAttribute(tc_gemm_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TC_SMEM_BYTES));
    configured = true;
  }
  cudaStream_t s = s_main;
  SideStream* ss = nullptr;
  const bool forked = G.n > 0 && (n_skinny > 0 || n_rowred > 0 || R.n > 0);
  const int set = level & 1;
  if (forked) {
    CUR_TRY(side_stream(&ss));
    CUR_CUDA_TRY(cudaEventRecord(ss->fork, s_main));
    CUR_CUDA_TRY(cudaStreamWaitEvent(ss->stream, ss->fork, 0));
    s = ss->stream;                       // helpers below go to the side stream
  }
  // the split-K / row-reduction partials of this level live in workspace set `set`: the deferred reductions of the
  // level that used the set before (two levels ago) must have read them
  if (red_pending[set]) {
    if (!ss) CUR_TRY(side_stream(&ss));
    CUR_CUDA_TRY(cudaStreamWaitEvent(s_main, ss->red[set], 0));
    if (forked) CUR_CUDA_TRY(cudaStreamWaitEvent(ss->stream, ss->red[set], 0));
    red_pending[set] = false;
  }
  if (G.n > 0) {
    B.n = G.n; B.total_tiles = G.total_tiles; B.tl = g_tc_timeline;
    if (pair) tc_gemm_pair_kernel<<<2 * G.total_tiles, TC_THREADS, TC_SMEM_BYTES, s_main>>>(B);
    else tc_gemm_kernel<<<G.total_tiles, TC_THREADS, TC_SMEM_BYTES, s_main>>>(B);
    CUR_CHECK_LAUNCH();
    if (forked) CUR_CUDA_TRY(cudaEventRecord(ss->gemm, s_main));
  }
  if (n_skinny > 0) {
    SkinnyBatch S;
    int blocks = 0;
    for (int i = 0; i < n_skinny; ++i) {
      const GemmProb& p = skinny[i].p;
      Skinny& q = S.p[i];
      memset(&q, 0, sizeof(q));
      q.M = p.M; q.N = p.N; q.K = p.K; q.epi = p.epi; q.coef = p.coef;
      q.X = p.A; q.ldx = p.lda; q.W = p.B; q.ldw = p.ldb; q.bias = p.bias; q.aux = p.aux; q.ldaux = p.ldaux;
      q.C = p.C; q.ldc = p.ldc;
      if (p.N <= 4) { q.kind = SK_ROWDOT; q.w_nk = p.b_trans ? 1 : 0; }
      else { q.kind = SK_OUTER; q.w_nk = 1; }
      q.block_begin = blocks;
      q.blocks = (p.M + SK_ROWS_PER_BLOCK - 1) / SK_ROWS_PER_BLOCK;
      blocks += q.blocks;
    }
    S.n = n_skinny;
    tc_skinny_kernel<<<blocks, 256, 0, s>>>(S);
    CUR_CHECK_LAUNCH();
  }
  if (n_rowred > 0) {
    RowRedBatch RB;
    int blocks = 0;
    for (int i = 0; i < n_rowred; ++i) {
      const RowRedDesc& c = rowred[i];
      RowRed& P = RB.p[i];
      P.X = c.X; P.ldx = c.ldx; P.Y = c.Y; P.ldy = c.ldy; P.rows = c.rows; P.M = c.M; P.NJ = c.NJ; P.part = c.part;
      P.col_blocks = (c.M + 63) / 64;
      P.block_begin = blocks;
      blocks += P.col_blocks * c.chunks;
    }
    RB.n = n_rowred;
    tc_rowred_kernel<<<blocks, 256, 0, s>>>(RB);
    CUR_CHECK_LAUNCH();
  }
  if (forked) {
    // the caller's stream only waits for the skinny kernels / row reductions (their outputs may feed the next level);
    // the fixed-order sums of the partials produce weight / bias gradients that nothing reads before the optimiser,
    // so they stay on the side stream behind the tensor-core launch and are joined in finish()
    CUR_CUDA_TRY(cudaEventRecord(ss->join, ss->stream));
    CUR_CUDA_TRY(cudaStreamWaitEvent(s_main, ss->join, 0));
    CUR_CUDA_TRY(cudaStreamWaitEvent(ss->stream, ss->gemm, 0));
  }
  if (R.n > 0) {
    CUR_REQUIRE(R.n <= 2 * TC_MAX_PROBS, "too many reductions");
    int blocks = 0;
    for (int i = 0; i < R.n; ++i) {
      R.p[i].block_begin = blocks;
      blocks += (int)(((R.p[i].count + 3) / 4 + 255) / 256);
    }
    tc_reduce_kernel<<<blocks, 256, 0, s>>>(R);
    CUR_CHECK_LAUNCH();
    if (forked) {
      CUR_CUDA_TRY(cudaEventRecord(ss->red[set], ss->stream));
      red_pending[set] = true;
    }
  }
  ++level;
  G.n = 0; G.total_tiles = 0; R.n = 0; n_rowred = 0; n_skinny = 0;
  return CUR_OK;
}

// Join the deferred reductions into the caller's stream (end of cur_ddpg_grads, before the optimiser reads the gradients).
int TcLauncher::finish(cudaStream_t s_main) {
  SideStream* ss = nullptr;
  for (int set = 0; set < 2; ++set) {
    if (!red_pending[set]) continue;
    if (!ss) CUR_TRY(side_stream(&ss));
    CUR_CUDA_TRY(cudaStreamWaitEvent(s_main, ss->red[set], 0));
    red_pending[set] = false;
  }
  return CUR_OK;
}

TcLauncher::TcLauncher() : n_rowred(0), n_skinny(0), level(0) {
  static const bool pair_env = getenv("CUR_TC_PAIR") != nullptr && getenv("CUR_TC_PAIR")[0] == '1';
  pair = pair_env;
  red_pending[0] = red_pending[1] = false;
  static_assert(sizeof(TcBatch) <= sizeof(storage), "TcLauncher storage too small");
  G.n = 0; G.total_tiles = 0; R.n = 0;
}

}  // namespace cur

using namespace cur;

extern "C" int cur_tc_gemm_timeline(long long* device_buffer_128) {
  tc_set_timeline(device_buffer_128);
  return CUR_OK;
}

extern "C" int cur_tc_gemm_supported(int64_t M, int64_t N, int64_t K) {
  return (N == TC_BN && M > 0 && K > 0 && M < (1 << 30) && K < (1 << 30)) ? 1 : 0;
}

extern "C" int64_t cur_tc_gemm_workspace_floats(int64_t M, int64_t N, int64_t K, int a_trans) {
  GemmProb p = zero_prob();
  p.M = (int)M; p.N = (int)N; p.K = (int)K; p.a_trans = a_trans;
  return tc_partial_floats(p);
}

extern "C" int cur_tc_gemm(void* stream, const float* A, int64_t lda, int a_trans, const float* B, int64_t ldb, int b_trans,
                           float* C, int64_t ldc, int64_t M, int64_t N, int64_t K, const float* bias, const float* aux,
                           int64_t ldaux, int epilogue, float* workspace) {
  CUR_REQUIRE(A && B && C, "NULL argument");
  CUR_REQUIRE(cur_tc_gemm_supported(M, N, K), "shape: N must be 256");
  GemmProb p = zero_prob();
  p.A = A; p.lda = (int)lda; p.a_trans = a_trans; p.B = B; p.ldb = (int)ldb; p.b_trans = b_trans;
  p.C = C; p.ldc = (int)ldc; p.M = (int)M; p.N = (int)N; p.K = (int)K;
  p.bias = bias; p.aux = aux; p.ldaux = (int)ldaux;
  p.epi = epilogue == 1 ? EPI_RELU : epilogue == 2 ? EPI_RELU_MASK : EPI_NONE;
  CUR_REQUIRE(tc_supported(p), "alignment: pointers 16-byte aligned, leading dimensions multiples of 4");
  TcLauncher L;
  CUR_TRY(L.add(p, workspace));
  CUR_TRY(L.flush((cudaStream_t)stream));
  return L.finish((cudaStream_t)stream);          // the split-K sum runs on the side stream: join it
}
