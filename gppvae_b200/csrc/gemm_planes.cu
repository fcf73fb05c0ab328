// Pass 1 and pass 2 on PRE-SPLIT fp16 operand planes: every fp32 operand x is stored once as two fp16 matrices
//   hi = x rounded to 11 significant bits,  lo = fp16(x - hi),  both scaled by one power of two per operand
// (pass1_common.cuh), and  a.b ~= hi(a).hi(b) + hi(a).lo(b) + lo(a).hi(b)  is three kind::f16 tcgen05 MMAs whose
// operands the TMA writes straight into shared memory, MMA-ready: no converter warps, nothing between the copy engine
// and the tensor core.  The planes cost the same 4 bytes per element as the fp32 matrix they replace.
//
// Why (round-2 measurements on B200, experiments/tc/exp3_f16_planes.cu): a TMA stream is bounded by BOXES per second
// (3.0 G boxes/s chip-wide whatever the box size: 6.2 TB/s with the 2 KB boxes of the round-1 kernel, 24.6 TB/s with
// 8 KB boxes), and three SS-form fp16 MMAs per 16 k-rows run at 2.2 PFLOP/s from shared memory alone; with 64-row
// boxes the stream + MMA pipeline sustains that same rate.  Multicast inside larger clusters bought nothing.
//
// Tile = 256 x 256 per CTA pair (cta_group::2), K block = 64 rows = ONE accumulation window (the TMEM accumulator
// rounds toward zero after every MMA: windows stay 64 k-rows long, inside a window the correction terms are issued
// first, and finished windows are added in fp32 registers, round-to-nearest, by the drain warps -- as in gemm_tc.cu).
// TMEM holds TWO accumulators (columns [0,256) and [256,512)): the issuer fills one while the drain warps empty the
// other.  Shared memory: 3 stages x 64 KB, a stage = 8 boxes {64 halfs, 64 rows} (SWIZZLE_128B):
//   pass 1:  [Ah g0][Ah g1][Al g0][Al g1][Bh g0][Bh g1][Bl g0][Bl g1]   both operands MN-major (contraction over ROWS)
//   rows  :  [Ah 128 rows][Al 128 rows][Bh g0][Bh g1][Bl g0][Bl g1]     A K-major boxes {64 halfs, 128 rows}
// Both CTAs' loads signal the full barrier of the pair LEADER (cta_group::2 form of cp.async.bulk.tensor).
// Warps: 0 TMA producer, 1 MMA issuer (leader) + TMEM owner, 4-11 drain / epilogue (setmaxnreg 64 / 216).
#include <cuda_fp16.h>
#include <stdlib.h>

#include <mutex>

#include "common.cuh"
#include "kernels.h"
#include "pass1_common.cuh"
#include "tc_common.cuh"

namespace gpp {

using namespace tc;

namespace {

constexpr int PBK = 64;                     // k-rows per stage
#ifndef GPP_PL_WIN
#define GPP_PL_WIN 64
#endif
constexpr int kWin = GPP_PL_WIN;            // k-rows per accumulation window in TMEM (16, 32 or 64)
constexpr int kSub = PBK / kWin;            // windows per stage
static_assert(kWin == 16 || kWin == 32 || kWin == 64, "window length");
constexpr int kPlStages = 3;
constexpr int kBoxBytes = 64 * 128;         // {64 halfs, 64 rows}
constexpr int kPlStageBytes = 8 * kBoxBytes;
constexpr int kPlThreads = 384;
constexpr int kPlSmemBytes = kPlStages * kPlStageBytes + 1024 /*align*/ + 256 /*barriers*/;
static_assert(kPlSmemBytes <= 232448, "shared memory budget");

struct PlShared {
  uint64_t full[kPlStages], empty[kPlStages], tfull[2], tempty[2];
  uint32_t tmem_base;
};

// ---- PTX pieces this file adds to tc_common.cuh ---------------------------------------------------------------
// TMA load whose completion is signalled on the barrier at the same offset in the pair LEADER (address with the peer
// bit cleared, as CUTLASS' SM100_TMA_2SM_LOAD does).
__device__ __forceinline__ void tma_load_2d_pair(uint32_t dst, const CUtensorMap* m, int x, int y, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::
          "r"(dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(x), "r"(y)
      : "memory");
}
__device__ __forceinline__ void umma_f16_pair_ss(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                                 uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}

__device__ __forceinline__ PlShared* pl_prologue(uint8_t* base, uint32_t& tmem) {
  PlShared* sm = reinterpret_cast<PlShared*>(base + kPlStages * kPlStageBytes);
  if (threadIdx.x == 0) {
    for (int s = 0; s < kPlStages; ++s) {
      mbar_init(&sm->full[s], 1);     // the leader's arrive.expect_tx (both CTAs' bytes)
      mbar_init(&sm->empty[s], 1);    // MMA commit, multicast to both CTAs
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&sm->tfull[b], 1);    // MMA commit, multicast to both CTAs
      mbar_init(&sm->tempty[b], 16);  // 8 drain warps x 2 CTAs (used in the leader)
    }
    fence_mbar_init();
  }
  if ((threadIdx.x >> 5) == 1) tmem_alloc_pair(&sm->tmem_base, 512);
  tcgen05_fence_before();
  cluster_sync_all();
  tcgen05_fence_after();
  tmem = sm->tmem_base;
  return sm;
}

__device__ __forceinline__ void pl_epilogue(uint32_t tmem) {
  tcgen05_fence_before();
  cluster_sync_all();
  if ((threadIdx.x >> 5) == 1) tmem_dealloc_pair(tmem, 512);
}

// One stage (64 k-rows) of a 256 x 256 tile, as kSub accumulation windows of kWin rows: inside a window the correction
// terms of its K = 16 steps first (into the still-small accumulator), the hi.hi terms last; every window goes to the
// drain warps through the next of the two TMEM accumulators, and after the last one the stage goes back to the producers.
// A_KMAJOR: A boxes are {64 halfs of k, 128 rows} (row GEMM), else MN-major like B (pass 1).  w: windows issued so far.
template <bool A_KMAJOR>
__device__ __forceinline__ void issue_stage(uint8_t* base, PlShared* sm, uint32_t tmem, uint32_t it, uint32_t& w) {
  constexpr uint32_t idesc = umma_idesc_f16(kTileM, kTileN, !A_KMAJOR, true);
  const int s = it % kPlStages;
  const uint32_t sb = smem_u32(base + s * kPlStageBytes);
  const uint32_t ah = sb, al = sb + 2 * kBoxBytes, bh = sb + 4 * kBoxBytes, bl = sb + 6 * kBoxBytes;
  // MN-major SWIZZLE_128B: 64-column groups kBoxBytes apart (LBO), 8-row k-groups 1 KB apart (SBO), K = 16 -> +2 KB;
  // K-major SWIZZLE_128B: 8-row groups 1 KB apart (SBO), K = 16 -> +32 B inside the 128-byte row
  auto adesc = [&](uint32_t a0, int kk) {
    return A_KMAJOR ? umma_desc(a0 + kk * 32, 16, 1024, kLayoutSw128) : umma_desc(a0 + kk * 2048, kBoxBytes, 1024, kLayoutSw128);
  };
  auto bdesc = [&](uint32_t b0, int kk) { return umma_desc(b0 + kk * 2048, kBoxBytes, 1024, kLayoutSw128); };
#pragma unroll
  for (int sw = 0; sw < kSub; ++sw, ++w) {
    const int buf = w & 1;
    mbar_wait_cluster(&sm->tempty[buf], ((w >> 1) & 1) ^ 1);   // drain warps of both CTAs are done with this accumulator
    if (sw == 0) mbar_wait(&sm->full[s], (it / kPlStages) & 1);  // both CTAs' boxes have landed
    tcgen05_fence_after();
    const uint32_t d = tmem + buf * 256;
    constexpr int kSteps = kWin / 16;
#pragma unroll
    for (int k = 0; k < kSteps; ++k) {
      const int kk = sw * kSteps + k;
      umma_f16_pair_ss(d, adesc(ah, kk), bdesc(bl, kk), idesc, k > 0);
      umma_f16_pair_ss(d, adesc(al, kk), bdesc(bh, kk), idesc, 1);
    }
#pragma unroll
    for (int k = 0; k < kSteps; ++k) {
      const int kk = sw * kSteps + k;
      umma_f16_pair_ss(d, adesc(ah, kk), bdesc(bh, kk), idesc, 1);
    }
    if (sw == kSub - 1) umma_commit_pair(&sm->empty[s], 3);
    umma_commit_pair(&sm->tfull[buf], 3);
  }
}

// 32 lanes x 32 consecutive fp32 columns -> 32 registers per thread, no wait (pair with tmem_ld_wait)
__device__ __forceinline__ void tmem_ld_32x32_nowait(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// acc (two packed fp32) += {lo, hi}, round-to-nearest: one FADD2 for two accumulator columns
__device__ __forceinline__ void add2(unsigned long long& acc, uint32_t lo, uint32_t hi) {
  unsigned long long v;
  asm("mov.b64 %0, {%1, %2};" : "=l"(v) : "r"(lo), "r"(hi));
  asm("add.rn.f32x2 %0, %0, %1;" : "+l"(acc) : "l"(v));
}
__device__ __forceinline__ float2 unpack2(unsigned long long v) {
  uint32_t lo, hi;
  asm("mov.b64 {%0, %1}, %2;" : "=r"(lo), "=r"(hi) : "l"(v));
  return make_float2(__uint_as_float(lo), __uint_as_float(hi));
}

// Drain warps (4-11): add window w (this CTA's 128 rows x this warp's 128 columns) into registers (packed pairs).
__device__ __forceinline__ void drain_window(PlShared* sm, uint32_t tmem, uint32_t tempty0_leader, uint32_t w,
                                             unsigned long long (&acc)[64]) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int buf = w & 1;
  const uint32_t lane_addr = (uint32_t)((warp & 3) * 32) << 16;
  const int cb = (warp - 4) >> 2;
  mbar_wait(&sm->tfull[buf], (w >> 1) & 1);
  tcgen05_fence_after();
  const uint32_t t0 = tmem + lane_addr + buf * 256 + cb * 128;
#pragma unroll
  for (int c = 0; c < 4; c += 2) {
    uint32_t v0[32], v1[32];
    tmem_ld_32x32_nowait(t0 + c * 32, v0);
    tmem_ld_32x32_nowait(t0 + c * 32 + 32, v1);
    tmem_ld_wait();
#pragma unroll
    for (int j = 0; j < 16; ++j) add2(acc[c * 16 + j], v0[2 * j], v0[2 * j + 1]);
#pragma unroll
    for (int j = 0; j < 16; ++j) add2(acc[c * 16 + 16 + j], v1[2 * j], v1[2 * j + 1]);
  }
  tcgen05_fence_before();
  __syncwarp();
  if (lane == 0) mbar_arrive_cluster(tempty0_leader + 8u * buf);
}

// =====================================================================================================
// Pass 1:  GC = V^T [V | X] from the planes of V and X.
// =====================================================================================================
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kPlThreads, 1)
pl_pass1_kernel(const __grid_constant__ CUtensorMap tmVh, const __grid_constant__ CUtensorMap tmVl,
                const __grid_constant__ CUtensorMap tmXh, const __grid_constant__ CUtensorMap tmXl, Pass1Params p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;
  uint32_t tmem;
  PlShared* sm = pl_prologue(base, tmem);
  const int nunits = p.tiles * p.splits;

  if (warp < 4) {
    setmaxnreg_dec<64>();
    if (warp == 0 && lane == 0) {
      // ===================================================== TMA producer (this CTA's halves of A and B)
      tma_prefetch_desc(&tmVh); tma_prefetch_desc(&tmVl); tma_prefetch_desc(&tmXh); tma_prefetch_desc(&tmXl);
      const uint32_t full0 = smem_u32(&sm->full[0]) & 0xFEFFFFFFu;   // the leader's barrier
      uint32_t it = 0;
      bool wave_sync = p.wave_ctr != nullptr;
      for (int u = pair; u < nunits; u += npairs) {
        // Wave alignment (a hint, not a dependency; see gemm_tc.cu): no producer starts the loads of wave w before every
        // producer has issued all loads of wave w - 1, so the pairs of a wave read the same rows of V while L2 holds them.
        if (wave_sync && u >= npairs) {
          const unsigned int target = 2u * (unsigned int)min((u / npairs) * npairs, nunits);
          const long long t0 = clock64();
          while (*reinterpret_cast<volatile unsigned int*>(p.wave_ctr) < target) {
            if (clock64() - t0 > 4000000ll) {
              wave_sync = false;
              break;
            }
          }
        }
        const int split = u / p.tiles, tile = u - split * p.tiles;   // consecutive pairs share a k-range (L2 reuse)
        int tm, tn;
        bool is_c;
        decode_tile(p, tile, tm, tn, is_c);
        const int64_t r0 = (int64_t)split * p.rows_per_split;
        const int64_t r1 = min(p.n, r0 + p.rows_per_split);
        const int nst = (int)((r1 - r0 + PBK - 1) / PBK);
        const CUtensorMap* mbh = is_c ? &tmXh : &tmVh;
        const CUtensorMap* mbl = is_c ? &tmXl : &tmVl;
        const int acol = tm * kTileM + (int)rank * 128, bcol = tn * kTileN + (int)rank * 128;
        for (int st = 0; st < nst; ++st, ++it) {
          const int s = it % kPlStages;
          mbar_wait(&sm->empty[s], ((it / kPlStages) & 1) ^ 1);
          if (rank == 0) mbar_arrive_expect_tx(&sm->full[s], 2 * kPlStageBytes);
          const uint32_t dst = smem_u32(base + s * kPlStageBytes), bar = full0 + 8u * s;
          const int row = (int)(r0 + (int64_t)st * PBK);
          tma_load_2d_pair(dst + 0 * kBoxBytes, &tmVh, acol, row, bar);
          tma_load_2d_pair(dst + 1 * kBoxBytes, &tmVh, acol + 64, row, bar);
          tma_load_2d_pair(dst + 2 * kBoxBytes, &tmVl, acol, row, bar);
          tma_load_2d_pair(dst + 3 * kBoxBytes, &tmVl, acol + 64, row, bar);
          tma_load_2d_pair(dst + 4 * kBoxBytes, mbh, bcol, row, bar);
          tma_load_2d_pair(dst + 5 * kBoxBytes, mbh, bcol + 64, row, bar);
          tma_load_2d_pair(dst + 6 * kBoxBytes, mbl, bcol, row, bar);
          tma_load_2d_pair(dst + 7 * kBoxBytes, mbl, bcol + 64, row, bar);
        }
        if (p.wave_ctr) atomicAdd(p.wave_ctr, 1u);
      }
    } else if (warp == 1 && lane == 0 && rank == 0) {
      // ===================================================== MMA issuer (leader CTA)
      uint32_t it = 0, w = 0;
      for (int u = pair; u < nunits; u += npairs) {
        const int split = u / p.tiles;
        const int64_t r0 = (int64_t)split * p.rows_per_split;
        const int64_t r1 = min(p.n, r0 + p.rows_per_split);
        const int nst = (int)((r1 - r0 + PBK - 1) / PBK);
        for (int st = 0; st < nst; ++st, ++it) issue_stage<false>(base, sm, tmem, it, w);
      }
    }
  } else {
    // ======================================================= drain warps: TMEM windows -> fp32 registers -> partial tile
    setmaxnreg_inc<216>();
    const uint32_t tempty0 = mapa_u32(&sm->tempty[0], 0);
    const int q = warp & 3, cb = (warp - 4) >> 2;
    const int eV = exp_of_bits(p.amax), eX = exp_of_bits(p.amax_x);
    const float out_g = exp2f((float)(2 * eV - 2 * kF16Top)), out_c = exp2f((float)(eV + eX - 2 * kF16Top));
    uint32_t w = 0;
    for (int u = pair; u < nunits; u += npairs) {
      const int split = u / p.tiles, tile = u - split * p.tiles;
      const int64_t r0 = (int64_t)split * p.rows_per_split;
      const int64_t r1 = min(p.n, r0 + p.rows_per_split);
      const int nst = (int)((r1 - r0 + PBK - 1) / PBK);
      unsigned long long acc[64];
#pragma unroll
      for (int i = 0; i < 64; ++i) acc[i] = 0ull;
      for (int st = 0; st < nst * kSub; ++st, ++w) drain_window(sm, tmem, tempty0, w, acc);
      const float os = tile < p.tiles_g ? out_g : out_c;   // undo the common power-of-two scale of the split (exact)
      float* out = p.partial + ((size_t)tile * p.splits + split) * (size_t)(kTileM * kTileN) +
                   (size_t)(rank * 128 + q * 32 + lane) * kTileN + cb * 128;
#pragma unroll
      for (int i = 0; i < 64; i += 2) {
        const float2 a = unpack2(acc[i]), b = unpack2(acc[i + 1]);
        *reinterpret_cast<float4*>(out + 2 * i) = make_float4(os * a.x, os * a.y, os * b.x, os * b.y);
      }
    }
  }
  pl_epilogue(tmem);
}

// =====================================================================================================
// Row GEMM:  D(256 rows x 256 cols per pair) = sum_k [A1 | A2][row, k] * B[k, col]   (all operands as planes)
//   mode 0 (pass 2): out = alpha (X - D), per-row quad partials and sum out^2 partials;  mode 1 (Vb): out = alpha D
// =====================================================================================================
struct PlRowsParams {
  int64_t n;
  int K1, K2;          // contraction lengths of A1 and A2 (K2 may be 0); B has K1 + K2 rows
  int ncols;
  int col_tiles;
  int64_t row_tiles;
  int mode;
  const uint32_t* amax_a1; const uint32_t* amax_a2; const uint32_t* amax_b;
  const float* X; int64_t ldx;
  float* out; int64_t ldo;
  const double* scal;  // mode 0: alpha = 1 / scal[VN] when set, else alpha_host
  float alpha_host;
  float* quad_part;    // [col_tiles * 2][n]
  double* xb2_part;    // [units * 16]
  unsigned int* wave_ctr;  // device, zeroed before the launch: producer-units issued so far (wave alignment); may be null
};

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kPlThreads, 1)
pl_rows_kernel(const __grid_constant__ CUtensorMap tmA1h, const __grid_constant__ CUtensorMap tmA1l,
               const __grid_constant__ CUtensorMap tmA2h, const __grid_constant__ CUtensorMap tmA2l,
               const __grid_constant__ CUtensorMap tmBh, const __grid_constant__ CUtensorMap tmBl, PlRowsParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;
  uint32_t tmem;
  PlShared* sm = pl_prologue(base, tmem);
  const int64_t nunits = p.row_tiles * p.col_tiles;
  const int nst1 = (p.K1 + PBK - 1) / PBK, nst2 = (p.K2 + PBK - 1) / PBK;
  const int nst = nst1 + nst2;

  if (warp < 4) {
    setmaxnreg_dec<64>();
    if (warp == 0 && lane == 0) {
      tma_prefetch_desc(&tmA1h); tma_prefetch_desc(&tmA1l); tma_prefetch_desc(&tmBh); tma_prefetch_desc(&tmBl);
      const uint32_t full0 = smem_u32(&sm->full[0]) & 0xFEFFFFFFu;
      uint32_t it = 0;
      // Wave alignment, as in pass 1 (a hint, not a dependency): the col_tiles pairs that work on one row tile read the
      // same 4.4 MB of A; left alone they drift apart by more than L2 holds and every one of them fetches its A tile from
      // DRAM again (ncu, c3 `Vb` product: 268 GB read per launch against 17.5 GB of operands).
      bool wave_sync = p.wave_ctr != nullptr && p.col_tiles > 1;
      for (int64_t u = pair; u < nunits; u += npairs) {
        if (wave_sync && u >= npairs) {
          const unsigned int target = 2u * (unsigned int)min((u / npairs) * npairs, nunits);
          const long long t0 = clock64();
          while (*reinterpret_cast<volatile unsigned int*>(p.wave_ctr) < target) {
            if (clock64() - t0 > 4000000ll) {
              wave_sync = false;
              break;
            }
          }
        }
        const int64_t rt = u / p.col_tiles;
        const int ct = (int)(u - rt * p.col_tiles);
        const int row = (int)(rt * kTileM) + (int)rank * 128;
        const int bcol = ct * kTileN + (int)rank * 128;
        for (int st = 0; st < nst; ++st, ++it) {
          const int s = it % kPlStages;
          mbar_wait(&sm->empty[s], ((it / kPlStages) & 1) ^ 1);
          if (rank == 0) mbar_arrive_expect_tx(&sm->full[s], 2 * kPlStageBytes);
          const uint32_t dst = smem_u32(base + s * kPlStageBytes), bar = full0 + 8u * s;
          int kb;   // row of B where this k-block starts
          if (st < nst1) {
            tma_load_2d_pair(dst, &tmA1h, st * PBK, row, bar);
            tma_load_2d_pair(dst + 2 * kBoxBytes, &tmA1l, st * PBK, row, bar);
            kb = st * PBK;
          } else {
            tma_load_2d_pair(dst, &tmA2h, (st - nst1) * PBK, row, bar);
            tma_load_2d_pair(dst + 2 * kBoxBytes, &tmA2l, (st - nst1) * PBK, row, bar);
            kb = p.K1 + (st - nst1) * PBK;
          }
          tma_load_2d_pair(dst + 4 * kBoxBytes, &tmBh, bcol, kb, bar);
          tma_load_2d_pair(dst + 5 * kBoxBytes, &tmBh, bcol + 64, kb, bar);
          tma_load_2d_pair(dst + 6 * kBoxBytes, &tmBl, bcol, kb, bar);
          tma_load_2d_pair(dst + 7 * kBoxBytes, &tmBl, bcol + 64, kb, bar);
        }
        if (p.wave_ctr) atomicAdd(p.wave_ctr, 1u);
      }
    } else if (warp == 1 && lane == 0 && rank == 0) {
      uint32_t it = 0, w = 0;
      for (int64_t u = pair; u < nunits; u += npairs)
        for (int st = 0; st < nst; ++st, ++it) issue_stage<true>(base, sm, tmem, it, w);
    }
  } else {
    setmaxnreg_inc<216>();
    const uint32_t tempty0 = mapa_u32(&sm->tempty[0], 0);
    const int q = warp & 3, cb = (warp - 4) >> 2;
    float alpha = p.alpha_host;
    if (p.mode == 0 && p.scal) alpha = (float)(1.0 / p.scal[GPP_S_VN]);
    // [A1 | A2] share the accumulator: their planes carry the SAME scale (the caller splits A2 with A1's exponent)
    const int eA = exp_of_bits(p.amax_a1), eB = exp_of_bits(p.amax_b);
    const float os = exp2f((float)(eA + eB - 2 * kF16Top));
    uint32_t w = 0;
    for (int64_t u = pair; u < nunits; u += npairs) {
      const int64_t rt = u / p.col_tiles;
      const int ct = (int)(u - rt * p.col_tiles);
      unsigned long long acc2[64];
#pragma unroll
      for (int i = 0; i < 64; ++i) acc2[i] = 0ull;
      if (p.mode == 0) {   // this thread's row of X for the epilogue: ask L2 for it now, behind the unit's MMAs
        const int64_t prow = rt * kTileM + rank * 128 + q * 32 + lane;
        if (prow < p.n) {
          const float* xr = p.X + prow * p.ldx + ct * kTileN + cb * 128;
#pragma unroll
          for (int i = 0; i < 128; i += 32)
            if (ct * kTileN + cb * 128 + i < p.ncols) asm volatile("prefetch.global.L2 [%0];" ::"l"(xr + i));
        }
      }
      for (int st = 0; st < nst * kSub; ++st, ++w) drain_window(sm, tmem, tempty0, w, acc2);
      float acc[128];
#pragma unroll
      for (int i = 0; i < 64; ++i) {
        const float2 a = unpack2(acc2[i]);
        acc[2 * i] = a.x;
        acc[2 * i + 1] = a.y;
      }
      const int64_t row = rt * kTileM + rank * 128 + q * 32 + lane;
      const int col0 = ct * kTileN + cb * 128;
      float xb2 = 0.f;
      if (row < p.n) {
        if (p.mode == 0) {
          float quad = 0.f;
          const float* xr = p.X + row * p.ldx + col0;
          float* orow = p.out + row * p.ldo + col0;
          // X and out may be the same matrix (in-place updates), so the compiler keeps every load behind the previous
          // store: read X in batches of 8 x 128 bit, all loads of a batch before its first store (4 exposed round trips
          // per unit instead of 32 -- the drain warps are what the issuer waits for at the end of a unit)
#pragma unroll
          for (int b8 = 0; b8 < 128; b8 += 32) {
            float4 xv[8];
#pragma unroll
            for (int t = 0; t < 8; ++t) {
              xv[t] = make_float4(0.f, 0.f, 0.f, 0.f);
              if (col0 + b8 + 4 * t < p.ncols) xv[t] = *reinterpret_cast<const float4*>(xr + b8 + 4 * t);
            }
#pragma unroll
            for (int t = 0; t < 8; ++t) {
              const int i = b8 + 4 * t;
              if (col0 + i < p.ncols) {
                const float4 x = xv[t];
                float4 o;
                o.x = (x.x - os * acc[i + 0]) * alpha;
                o.y = (x.y - os * acc[i + 1]) * alpha;
                o.z = (x.z - os * acc[i + 2]) * alpha;
                o.w = (x.w - os * acc[i + 3]) * alpha;
                *reinterpret_cast<float4*>(orow + i) = o;
                quad = fmaf(x.x, o.x, quad); quad = fmaf(x.y, o.y, quad);
                quad = fmaf(x.z, o.z, quad); quad = fmaf(x.w, o.w, quad);
                xb2 = fmaf(o.x, o.x, xb2); xb2 = fmaf(o.y, o.y, xb2);
                xb2 = fmaf(o.z, o.z, xb2); xb2 = fmaf(o.w, o.w, xb2);
              }
            }
          }
          if (p.quad_part) p.quad_part[(int64_t)(ct * 2 + cb) * p.n + row] = quad;
        } else {
          float* orow = p.out + row * p.ldo + col0;
          const float a = alpha * os;
#pragma unroll
          for (int i = 0; i < 128; i += 4)
            if (col0 + i < p.ncols)
              *reinterpret_cast<float4*>(orow + i) = make_float4(a * acc[i], a * acc[i + 1], a * acc[i + 2], a * acc[i + 3]);
        }
      }
      if (p.mode == 0 && p.xb2_part) {
        const float s = warp_sum(xb2);
        if (lane == 0) p.xb2_part[u * 16 + rank * 8 + (warp - 4)] = (double)s;
      }
    }
  }
  pl_epilogue(tmem);
}

// =====================================================================================================
// Producers of planes
// =====================================================================================================
// planes buffer (caller-owned, opaque to the caller):
//   [meta: 64 x u32][colsq: cols doubles][hi: n x ldp halfs][lo: n x ldp halfs],  ldp = cols rounded up to 8
// meta[0] = bit pattern of max|x| (the exponent of the common scale), meta[1] = 1 when colsq holds the column sums of
// squares of the source matrix.
struct PlanesView {
  uint32_t* meta;
  double* colsq;
  __half* hi;
  __half* lo;
  int64_t ldp;
};
__host__ __device__ inline int64_t planes_ld(int cols) { return ((int64_t)cols + 7) / 8 * 8; }
inline size_t planes_off_colsq() { return 256; }
inline size_t planes_off_hi(int cols) { return 256 + align_up((size_t)cols * 8, 256); }
inline size_t planes_plane_bytes(int64_t n, int cols) { return align_up((size_t)(n > 0 ? n : 1) * planes_ld(cols) * 2, 256); }
inline PlanesView planes_view(void* buf, int64_t n, int cols) {
  char* b = static_cast<char*>(buf);
  PlanesView v;
  v.meta = reinterpret_cast<uint32_t*>(b);
  v.colsq = reinterpret_cast<double*>(b + planes_off_colsq());
  v.hi = reinterpret_cast<__half*>(b + planes_off_hi(cols));
  v.lo = reinterpret_cast<__half*>(b + planes_off_hi(cols) + planes_plane_bytes(n, cols));
  v.ldp = planes_ld(cols);
  return v;
}

__device__ __forceinline__ void split4(const float4 v, float sc, uint2& h, uint2& l) {
  const float hx = hi11_round(__float_as_uint(v.x)), hy = hi11_round(__float_as_uint(v.y));
  const float hz = hi11_round(__float_as_uint(v.z)), hw = hi11_round(__float_as_uint(v.w));
  h.x = pack_f16x2(hx * sc, hy * sc);
  h.y = pack_f16x2(hz * sc, hw * sc);
  l.x = pack_f16x2((v.x - hx) * sc, (v.y - hy) * sc);
  l.y = pack_f16x2((v.z - hz) * sc, (v.w - hw) * sc);
}

constexpr int kSplitRowBlocks = 8;   // upper bound of resident 256-thread CTAs per SM (2048 threads)

// fp32 matrix -> planes (+ optional per-row-block column sums of squares, fp64).  Thread = one float4 column group,
// walking the rows of its block: coalesced 16-byte loads, 8-byte stores into each plane.
__global__ void __launch_bounds__(256)
split_planes_kernel(const float* __restrict__ X, int64_t ldx, int64_t n, int cols, __half* __restrict__ H,
                    __half* __restrict__ Lo, int64_t ldp, const uint32_t* __restrict__ amax, int64_t rows_per_block,
                    double* __restrict__ colsq_part) {
  const int c = (blockIdx.x * 256 + threadIdx.x) * 4;
  if (c >= cols) return;
  const float sc = exp2f((float)(kF16Top - exp_of_bits(amax)));
  const int64_t r0 = (int64_t)blockIdx.y * rows_per_block, r1 = min(n, r0 + rows_per_block);
  double s0 = 0, s1 = 0, s2 = 0, s3 = 0;
#pragma unroll 4
  for (int64_t r = r0; r < r1; ++r) {
    const float4 v = *reinterpret_cast<const float4*>(X + r * ldx + c);
    uint2 h, l;
    split4(v, sc, h, l);
    *reinterpret_cast<uint2*>(H + r * ldp + c) = h;
    *reinterpret_cast<uint2*>(Lo + r * ldp + c) = l;
    if (colsq_part) {
      s0 = fma((double)v.x, (double)v.x, s0); s1 = fma((double)v.y, (double)v.y, s1);
      s2 = fma((double)v.z, (double)v.z, s2); s3 = fma((double)v.w, (double)v.w, s3);
    }
  }
  if (colsq_part) {
    double* o = colsq_part + (int64_t)blockIdx.y * cols + c;
    o[0] = s0; o[1] = s1; o[2] = s2; o[3] = s3;
  }
}

// Khatri-Rao map (vmod.py:28-35) writing V (fp32, what the API returns) AND its planes AND the exact column sums of
// squares in one sweep: same thread layout as split_planes_kernel, the thread's four (j, k) pairs are loop-invariant.
//
// Everything that depends on the ROW alone -- the two index loads, their range checks and the 64-bit table offsets -- is
// the same for all 256 threads of the CTA, so one thread per row does it once per chunk of kKrChunk rows and leaves
// {byte offset of the object row, byte offset of the view row, 1.0f or NaN} in shared memory; the row loop of a thread is
// then one 128-bit shared-memory read, two gathers, the arithmetic and three stores.  (First version: every thread
// loaded and checked the indices itself; ~120 instructions per row and thread, issue slots 56 % busy at 1.96 GHz, so
// behind pass 1 -- SM clock 1.1-1.3 GHz under the power cap -- the kernel turned issue-bound: 8.07 ms against 5.98 ms
// on a cool chip while a plain device copy of the same size only went from 4.9 to 5.5 ms; experiments/bench/kr_instep.py.)
constexpr int kKrChunk = 256;
struct __align__(16) KrRow {
  long long xoff;   // bytes from xn to the row's object features
  int woff;         // bytes from wn to the row's view features
  float ok;         // 1.0f, or NaN for a row whose index is outside its table (the whole row of V becomes NaN)
};
template <bool QUAD>
__global__ void __launch_bounds__(256)
kr_planes_kernel(const float* __restrict__ xn, int64_t P, int p, const float* __restrict__ wn, int64_t nviews, int q,
                 const int64_t* __restrict__ d, const int64_t* __restrict__ w, int64_t n, float* __restrict__ V,
                 int64_t ldv, __half* __restrict__ H, __half* __restrict__ Lo, int64_t ldp, int64_t rows_per_block,
                 double* __restrict__ colsq_part) {
  __shared__ KrRow rows[kKrChunk];
  const int cols = p * q;
  const int c = (blockIdx.x * 256 + threadIdx.x) * 4;
  const bool active = c < cols;
  int j[4], k[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const int ce = active ? c + e : 0;
    j[e] = ce / q;
    k[e] = ce - j[e] * q;
  }
  // QUAD (q % 4 == 0): the four columns share j and their k are one aligned float4 of the view row
  const char* xb[4];
  const char* wb[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    xb[e] = reinterpret_cast<const char*>(xn + j[e]);
    wb[e] = reinterpret_cast<const char*>(wn + k[e]);
  }
  const float sc = exp2f((float)(kF16Top - 1));   // |v| <= 1 (product of two unit-norm rows): max|v| < 2^1
  const int64_t r0 = (int64_t)blockIdx.y * rows_per_block, r1 = min(n, r0 + rows_per_block);
  double s0 = 0, s1 = 0, s2 = 0, s3 = 0;
  char* vp = reinterpret_cast<char*>(V + r0 * ldv + c);
  char* hp = reinterpret_cast<char*>(H + r0 * ldp + c);
  char* lp = reinterpret_cast<char*>(Lo + r0 * ldp + c);
  const int64_t vstep = ldv * 4, pstep = ldp * 2;

  // one row: gathers (issued by the caller in batches), products, split, stores, sums of squares
  auto finish_row = [&](const float (&x)[4], const float4 w4) {
    const float4 v = make_float4(x[0] * w4.x, x[1] * w4.y, x[2] * w4.z, x[3] * w4.w);
    *reinterpret_cast<float4*>(vp) = v;
    uint2 h, l;
    split4(v, sc, h, l);
    *reinterpret_cast<uint2*>(hp) = h;
    *reinterpret_cast<uint2*>(lp) = l;
    s0 = fma((double)v.x, (double)v.x, s0); s1 = fma((double)v.y, (double)v.y, s1);
    s2 = fma((double)v.z, (double)v.z, s2); s3 = fma((double)v.w, (double)v.w, s3);
    vp += vstep; hp += pstep; lp += pstep;
  };
  auto gather = [&](const KrRow rw, float (&x)[4], float4& w4) {
    if (QUAD) {
      const float xv = *reinterpret_cast<const float*>(xb[0] + rw.xoff) * rw.ok;
      x[0] = x[1] = x[2] = x[3] = xv;
      w4 = *reinterpret_cast<const float4*>(wb[0] + rw.woff);
    } else {
#pragma unroll
      for (int e = 0; e < 4; ++e) x[e] = *reinterpret_cast<const float*>(xb[e] + rw.xoff) * rw.ok;
      w4 = make_float4(*reinterpret_cast<const float*>(wb[0] + rw.woff), *reinterpret_cast<const float*>(wb[1] + rw.woff),
                       *reinterpret_cast<const float*>(wb[2] + rw.woff), *reinterpret_cast<const float*>(wb[3] + rw.woff));
    }
  };

  for (int64_t rc = r0; rc < r1; rc += kKrChunk) {
    const int nr = (int)min((int64_t)kKrChunk, r1 - rc);
    __syncthreads();                       // the previous chunk's entries have been read by everybody
    if ((int)threadIdx.x < nr) {
      const int64_t di = d[rc + threadIdx.x], wi = w[rc + threadIdx.x];
      const bool ok = (di >= 0) & (di < P) & (wi >= 0) & (wi < nviews);
      KrRow rw;
      rw.xoff = ok ? di * (int64_t)p * 4 : 0;
      rw.woff = ok ? (int)(wi * q * 4) : 0;
      rw.ok = ok ? 1.f : __int_as_float(0x7fc00000);
      rows[threadIdx.x] = rw;
    }
    __syncthreads();
    if (!active) continue;
    // rows in batches of kB: all gathers of a batch in flight before the first store
    constexpr int kB = 4;
    int r = 0;
    for (; r + kB <= nr; r += kB) {
      float x[kB][4];
      float4 w4[kB];
#pragma unroll
      for (int u = 0; u < kB; ++u) gather(rows[r + u], x[u], w4[u]);
#pragma unroll
      for (int u = 0; u < kB; ++u) finish_row(x[u], w4[u]);
    }
    for (; r < nr; ++r) {
      float x[4];
      float4 w4;
      gather(rows[r], x, w4);
      finish_row(x, w4);
    }
  }
  if (active) {
    double* o = colsq_part + (int64_t)blockIdx.y * cols + c;
    o[0] = s0; o[1] = s1; o[2] = s2; o[3] = s3;
  }
}

// colsq[c] = sum over the row blocks, in a fixed order; meta[1] = 1
__global__ void __launch_bounds__(256) colsq_reduce_kernel(const double* __restrict__ part, int nparts, int cols,
                                                           double* __restrict__ colsq, uint32_t* __restrict__ meta) {
  const int c = blockIdx.x * 256 + threadIdx.x;
  if (c < cols) {
    double s = 0;
    for (int i = 0; i < nparts; ++i) s += part[(int64_t)i * cols + c];
    colsq[c] = s;
  }
  if (c == 0) meta[1] = 1u;
}

__global__ void planes_meta_kernel(uint32_t* meta, uint32_t amax_bits, uint32_t has_colsq) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    if (amax_bits) meta[0] = amax_bits;
    meta[1] = has_colsq;
  }
}
__global__ void copy_u32_kernel(uint32_t* dst, const uint32_t* src) {
  if (threadIdx.x == 0 && blockIdx.x == 0) *dst = *src;
}

// Slot sums of the structured route (structured.cu, kr_slot_sum_kernel) written DIRECTLY as operand planes, so that the
// P-long product xn^T [cnt (x) xn | Xs] runs on the planes kernel without the 2 GB fp32 matrix, without a magnitude scan
// of it and without converter warps:  XZ[o, v p + j] = cnt[s] xn[o, j],  XZ[o, zcol0 + v L + l] = sum of X[i, l] over the
// rows of slot s = o nviews + v (added in the order of `order`: deterministic).  The scale comes from a BOUND instead of a
// scan of the result: |cnt xn| <= max_count (unit rows), |slot sum| <= max_count max|X| -- meta[0] is set by
// slot_scale_kernel from the exact max|X| (one read of X) and the largest slot count (known to the caller from the
// index).  One warp per slot.  mode (the entry's with_x): 0 the slot sums alone, bound max_count max|X|;  2 cnt (x) xn
// alone, bound max_count;  1 both ranges in one buffer under ONE scale, max_count max(1, max|X|) -- the range whose
// magnitude is far below that bound keeps fewer bits (DESIGN 5.4), so the route splits the two (modes 2 and 0).
__global__ void slot_scale_kernel(uint32_t* __restrict__ meta, int max_count, int mode) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    float xmax = mode == 2 ? 1.f : __uint_as_float(meta[2]);   // bits of max|X| (tc_absmax wrote them there)
    if (mode == 1) xmax = fmaxf(xmax, 1.f);
    meta[0] = __float_as_uint((float)max_count * xmax);
    meta[1] = 0u;
  }
}
__global__ void __launch_bounds__(256)
kr_slot_sum_planes_kernel(const float* __restrict__ X, int64_t ldx, const int64_t* __restrict__ order,
                          const int64_t* __restrict__ slot_start, const float* __restrict__ xn, int64_t P, int p,
                          int nviews, int L, int with_x, __half* __restrict__ H, __half* __restrict__ Lo, int64_t ldp,
                          const uint32_t* __restrict__ meta) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  const int zcol0 = with_x ? nviews * p : 0;
  const float sc = exp2f((float)(kF16Top - exp_of_bits(meta)));
  for (int64_t s = warp; s < P * nviews; s += nwarps) {
    const int64_t o = s / nviews;
    const int v = (int)(s - o * nviews);
    const int64_t b = slot_start[s], e = slot_start[s + 1];
    const int64_t zoff = o * ldp + zcol0 + (int64_t)v * L;
    for (int c = lane * 4; c < L; c += 128) {
      float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
      for (int64_t t = b; t < e; ++t) {
        const float4 x = *reinterpret_cast<const float4*>(X + order[t] * ldx + c);
        acc.x += x.x; acc.y += x.y; acc.z += x.z; acc.w += x.w;
      }
      uint2 h, l;
      split4(acc, sc, h, l);
      *reinterpret_cast<uint2*>(H + zoff + c) = h;
      *reinterpret_cast<uint2*>(Lo + zoff + c) = l;
    }
    if (!with_x) continue;
    const float cnt = (float)(e - b);
    const int64_t xoff = o * ldp + (int64_t)v * p;
    for (int c = lane * 4; c < p; c += 128) {
      const float4 x = *reinterpret_cast<const float4*>(xn + o * p + c);
      uint2 h, l;
      split4(make_float4(cnt * x.x, cnt * x.y, cnt * x.z, cnt * x.w), sc, h, l);
      *reinterpret_cast<uint2*>(H + xoff + c) = h;
      *reinterpret_cast<uint2*>(Lo + xoff + c) = l;
    }
  }
}

// ctas_per_sm > 0: one full wave of equal row blocks for a kernel that holds that many CTAs per SM; 0: 8 x SMs CTAs (the
// upper bound the workspace is sized for).
void split_grid(int64_t n, int cols, dim3& grid, int64_t& rows_per_block, int ctas_per_sm = 0) {
  const int gx = (int)ceil_div(cols, 1024);
  if (ctas_per_sm <= 0 || ctas_per_sm > kSplitRowBlocks) ctas_per_sm = kSplitRowBlocks;
  int64_t gy = (int64_t)ctas_per_sm * sm_count() / gx;
  if (gy < 1) gy = 1;
  if (gy > ceil_div(n, 16)) gy = ceil_div(n, 16);
  if (gy < 1) gy = 1;
  rows_per_block = ceil_div(n > 0 ? n : 1, gy);
  gy = ceil_div(n > 0 ? n : 1, rows_per_block);
  grid = dim3((unsigned)gx, (unsigned)gy);
}

// resident 256-thread CTAs per SM of a producer kernel (register-limited; static shared memory only)
template <typename K>
int resident_ctas_256(K kernel) {
  int nb = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kernel, 256, 0) != cudaSuccess || nb <= 0) {
    cudaGetLastError();
    nb = 4;
  }
  return nb;
}

template <typename K>
int pl_pair_count(K kernel) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(2 * (unsigned)sm_count());
  cfg.blockDim = dim3(kPlThreads);
  cfg.dynamicSmemBytes = kPlSmemBytes;
  cudaLaunchAttribute at{};
  at.id = cudaLaunchAttributeClusterDimension;
  at.val.clusterDim.x = 2; at.val.clusterDim.y = 1; at.val.clusterDim.z = 1;
  cfg.attrs = &at; cfg.numAttrs = 1;
  int n = 0;
  if (cudaOccupancyMaxActiveClusters(&n, kernel, &cfg) != cudaSuccess || n <= 0) {
    cudaGetLastError();
    n = sm_count() / 2;
  }
  return n;
}

constexpr int kMaxDevices = 64;
std::mutex g_pl_mutex;
int pl_pairs() {
  static int n[kMaxDevices] = {0};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= kMaxDevices) dev = 0;
  std::lock_guard<std::mutex> lock(g_pl_mutex);
  if (n[dev] == 0) {
    cudaFuncSetAttribute(pl_pass1_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kPlSmemBytes);
    cudaFuncSetAttribute(pl_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kPlSmemBytes);
    const int a = pl_pair_count(pl_pass1_kernel), b = pl_pair_count(pl_rows_kernel);
    n[dev] = a < b ? a : b;
  }
  return n[dev];
}

}  // namespace

// ---------------------------------------------------------------- planes: sizes and producers
size_t planes_bytes(int64_t n, int cols) { return planes_off_hi(cols) + 2 * planes_plane_bytes(n, cols); }

size_t split_workspace_bytes(int64_t n, int cols) {
  dim3 grid;
  int64_t rpb;
  split_grid(n, cols, grid, rpb);
  return align_up((size_t)grid.y * cols * sizeof(double), 256);
}

// X (n x cols fp32) -> planes.  exp_hint != 0: max|x| < 2^exp_hint is known (no scan);  share_scale_of: take the scale
// from another planes buffer (operands that share an accumulator).  want_colsq needs ws (split_workspace_bytes).
int launch_split_planes(const float* X, int64_t ldx, int64_t n, int cols, void* planes, const void* share_scale_of,
                        int exp_hint, bool want_colsq, void* ws, size_t ws_bytes, cudaStream_t st) {
  PlanesView pv = planes_view(planes, n, cols);
  if (share_scale_of) {
    copy_u32_kernel<<<1, 32, 0, st>>>(pv.meta, static_cast<const uint32_t*>(share_scale_of));
    GPP_LAUNCH_CHECK();
  } else if (exp_hint != 0) {
    // bit pattern of 2^(exp_hint - 1): exponent field exp_hint - 1 + 127
    planes_meta_kernel<<<1, 32, 0, st>>>(pv.meta, (uint32_t)(exp_hint - 1 + 127) << 23, 0u);
    GPP_LAUNCH_CHECK();
  } else {
    GPP_TRY(tc_absmax(X, ldx, n, cols, pv.meta, st));
  }
  if (n <= 0) return GPP_OK;
  dim3 grid;
  int64_t rpb;
  split_grid(n, cols, grid, rpb);   // (one wave measured here too: 5.29 -> 5.47 ms at c3 shape; the fixed grid stays)
  double* part = nullptr;
  if (want_colsq) {
    const size_t need = align_up((size_t)grid.y * cols * sizeof(double), 256);
    if (!ws || ws_bytes < need) {
      set_error("split_planes: workspace too small (%zu < %zu bytes)", ws_bytes, need);
      return GPP_ERR_WORKSPACE;
    }
    part = static_cast<double*>(ws);
  }
  split_planes_kernel<<<grid, 256, 0, st>>>(X, ldx, n, cols, pv.hi, pv.lo, pv.ldp, pv.meta, rpb, part);
  GPP_LAUNCH_CHECK();
  if (want_colsq) {
    colsq_reduce_kernel<<<(unsigned)ceil_div(cols, 256), 256, 0, st>>>(part, (int)grid.y, cols, pv.colsq, pv.meta);
    GPP_LAUNCH_CHECK();
  } else {
    planes_meta_kernel<<<1, 32, 0, st>>>(pv.meta, 0u, 0u);
    GPP_LAUNCH_CHECK();
  }
  return GPP_OK;
}

// Planes of the column concatenation [X_0 | ... | X_{k-1}] (every cols[i] a multiple of 4) written straight into one
// planes buffer of n x sum(cols): no fp32 concatenation.  One common scale: the exact scans of all sources fold into
// meta[0] before any source is split (or the bound |x| <= 1 when unit_bound).  Source i is split by the single-matrix
// kernels at its column offset, and its column sums of squares are reduced into its column range -- fixed order, so
// diag(G) is exact and reproducible.  The sources are processed one after the other on `st`, so the partial sums reuse
// one workspace of the largest source's size.
size_t split_stacked_workspace_bytes(int64_t n, int k, const int* cols) {
  size_t b = 0;
  for (int i = 0; i < k; ++i) {
    const size_t s = split_workspace_bytes(n, cols[i]);
    if (s > b) b = s;
  }
  return b;
}

int launch_split_planes_stacked(int k, const float* const* X, const int64_t* ldx, const int* cols, int64_t n, void* planes,
                                bool unit_bound, bool want_colsq, void* ws, size_t ws_bytes, cudaStream_t st) {
  int total = 0;
  for (int i = 0; i < k; ++i) total += cols[i];
  PlanesView pv = planes_view(planes, n, total);
  if (want_colsq && (!ws || ws_bytes < split_stacked_workspace_bytes(n, k, cols))) {
    set_error("split_planes_stacked: workspace too small (%zu < %zu bytes)", ws_bytes,
              split_stacked_workspace_bytes(n, k, cols));
    return GPP_ERR_WORKSPACE;
  }
  if (unit_bound) {
    planes_meta_kernel<<<1, 32, 0, st>>>(pv.meta, (uint32_t)(1 - 1 + 127) << 23, 0u);   // max|x| < 2^1
    GPP_LAUNCH_CHECK();
  } else {
    GPP_CUDA(cudaMemsetAsync(pv.meta, 0, 4, st));
    for (int i = 0; i < k; ++i) GPP_TRY(tc_absmax_fold(X[i], ldx[i], n, cols[i], pv.meta, st));
  }
  if (n <= 0) return GPP_OK;
  int off = 0;
  for (int i = 0; i < k; ++i) {
    dim3 grid;
    int64_t rpb;
    split_grid(n, cols[i], grid, rpb);
    double* part = want_colsq ? static_cast<double*>(ws) : nullptr;
    split_planes_kernel<<<grid, 256, 0, st>>>(X[i], ldx[i], n, cols[i], pv.hi + off, pv.lo + off, pv.ldp, pv.meta, rpb,
                                              part);
    GPP_LAUNCH_CHECK();
    if (want_colsq) {
      colsq_reduce_kernel<<<(unsigned)ceil_div(cols[i], 256), 256, 0, st>>>(part, (int)grid.y, cols[i], pv.colsq + off,
                                                                            pv.meta);
      GPP_LAUNCH_CHECK();
    }
    off += cols[i];
  }
  if (!want_colsq) {
    planes_meta_kernel<<<1, 32, 0, st>>>(pv.meta, 0u, 0u);
    GPP_LAUNCH_CHECK();
  }
  return GPP_OK;
}

int launch_kr_planes(const float* xn, int64_t P, int p, const float* wn, int64_t nviews, int q, const int64_t* d,
                     const int64_t* w, int64_t n, float* V, int64_t ldv, void* planes, void* ws, size_t ws_bytes,
                     cudaStream_t st) {
  const int cols = p * q;
  PlanesView pv = planes_view(planes, n, cols);
  planes_meta_kernel<<<1, 32, 0, st>>>(pv.meta, (uint32_t)(1 - 1 + 127) << 23, 0u);   // max|v| < 2^1
  GPP_LAUNCH_CHECK();
  if (n <= 0) return GPP_OK;
  // one full wave of equal row blocks (measured at c3, cool chip / behind pass 1: 5.89 / 7.11 ms; with the fixed
  // 8 x SMs grid 6.40 / 8.15 ms; the first version of the kernel 5.97 / 7.67 and 6.06 / 7.44 ms)
  dim3 grid;
  int64_t rpb;
  split_grid(n, cols, grid, rpb, (q & 3) == 0 ? resident_ctas_256(kr_planes_kernel<true>) : resident_ctas_256(kr_planes_kernel<false>));
  const size_t need = align_up((size_t)grid.y * cols * sizeof(double), 256);
  if (!ws || ws_bytes < need) {
    set_error("khatri_rao_fwd_planes: workspace too small (%zu < %zu bytes)", ws_bytes, need);
    return GPP_ERR_WORKSPACE;
  }
  double* part = static_cast<double*>(ws);
  if ((int64_t)nviews * q * 4 > 0x7fffffffLL) {
    set_error("khatri_rao_fwd_planes: view table larger than 2 GB");
    return GPP_ERR_UNSUPPORTED;
  }
  if ((q & 3) == 0)
    kr_planes_kernel<true><<<grid, 256, 0, st>>>(xn, P, p, wn, nviews, q, d, w, n, V, ldv, pv.hi, pv.lo, pv.ldp, rpb, part);
  else
    kr_planes_kernel<false><<<grid, 256, 0, st>>>(xn, P, p, wn, nviews, q, d, w, n, V, ldv, pv.hi, pv.lo, pv.ldp, rpb, part);
  GPP_LAUNCH_CHECK();
  colsq_reduce_kernel<<<(unsigned)ceil_div(cols, 256), 256, 0, st>>>(part, (int)grid.y, cols, pv.colsq, pv.meta);
  GPP_LAUNCH_CHECK();
  return GPP_OK;
}

// ---------------------------------------------------------------- pass 1 on planes
bool pl_pass1_supported(int64_t n, int Q, int L) { return Q >= 128 && n >= 512 && tc_available(); }

size_t pl_pass1_workspace_bytes(int64_t n, int Q, int L, bool skip_g) {
  Pass1Params p{};
  pass1_geometry(n, Q, L, skip_g, pl_pairs(), PBK, p);
  return (size_t)p.tiles * p.splits * kTileM * kTileN * sizeof(float) + 256 /* wave counter */;
}

// G (Q x Q, optional) = V^T V and C (Q x L) = V^T X from planes.  use_colsq: overwrite the diagonal of G with the exact
// column sums of squares stored with V's planes (they must have been produced with want_colsq).
int launch_pl_pass1(const void* planesV, const void* planesX, int64_t n, int Q, int L, float* G, int64_t ldg, float* C,
                    int64_t ldc, bool use_colsq, void* ws, size_t ws_bytes, cudaStream_t st) {
  Pass1Params p{};
  pass1_geometry(n, Q, L, G == nullptr, pl_pairs(), PBK, p);
  const size_t part_bytes = (size_t)p.tiles * p.splits * kTileM * kTileN * sizeof(float), need = part_bytes + 256;
  if (!ws || ws_bytes < need) {
    set_error("gram_vtz (planes): workspace too small (%zu < %zu bytes)", ws_bytes, need);
    return GPP_ERR_WORKSPACE;
  }
  if (p.tiles == 0) return GPP_OK;
  const PlanesView pv = planes_view(const_cast<void*>(planesV), n, Q);
  const PlanesView px = L > 0 ? planes_view(const_cast<void*>(planesX), n, L) : pv;
  p.partial = static_cast<float*>(ws);
  p.amax = pv.meta;
  p.amax_x = px.meta;
  p.wave_ctr = reinterpret_cast<unsigned int*>(static_cast<char*>(ws) + part_bytes);
  if (const char* e = getenv("GPP_TC_WAVE_SYNC")) {   // experiment knob: 0 switches the wave alignment off
    if (e[0] == '0') p.wave_ctr = nullptr;
  }
  if (p.wave_ctr) GPP_CUDA(cudaMemsetAsync(p.wave_ctr, 0, 4, st));
  p.G = G; p.ldg = ldg; p.C = C; p.ldc = ldc; p.scal_c = nullptr;
  p.diag = (use_colsq && G) ? pv.colsq : nullptr;
  CUtensorMap tmVh, tmVl, tmXh, tmXl;
  GPP_TRY(make_tensor_map_2d(&tmVh, pv.hi, 2, n, Q, pv.ldp, 64, PBK, CU_TENSOR_MAP_SWIZZLE_128B));
  GPP_TRY(make_tensor_map_2d(&tmVl, pv.lo, 2, n, Q, pv.ldp, 64, PBK, CU_TENSOR_MAP_SWIZZLE_128B));
  if (L > 0) {
    GPP_TRY(make_tensor_map_2d(&tmXh, px.hi, 2, n, L, px.ldp, 64, PBK, CU_TENSOR_MAP_SWIZZLE_128B));
    GPP_TRY(make_tensor_map_2d(&tmXl, px.lo, 2, n, L, px.ldp, 64, PBK, CU_TENSOR_MAP_SWIZZLE_128B));
  } else {
    tmXh = tmVh;
    tmXl = tmVl;
  }
  const int nunits = p.tiles * p.splits;
  const int pairs = nunits < pl_pairs() ? nunits : pl_pairs();
  pl_pass1_kernel<<<2 * pairs, kPlThreads, kPlSmemBytes, st>>>(tmVh, tmVl, tmXh, tmXl, p);
  GPP_LAUNCH_CHECK();
  return launch_pass1_reduce(p, st);
}

// ---------------------------------------------------------------- row GEMMs on planes
bool pl_rows_supported(int64_t n, int K, int ncols) { return n >= 512 && K >= 64 && ncols >= 64 && tc_available(); }

static int launch_pl_rows(const PlanesView& a1, int K1, const PlanesView* a2, int K2, const PlanesView& b, int64_t n,
                          int ncols, PlRowsParams& p, cudaStream_t st) {
  p.n = n; p.K1 = K1; p.K2 = K2; p.ncols = ncols;
  p.col_tiles = (int)ceil_div(ncols, kTileN);
  p.row_tiles = ceil_div(n, kTileM);
  p.amax_a1 = a1.meta; p.amax_a2 = a2 ? a2->meta : a1.meta; p.amax_b = b.meta;
  CUtensorMap tA1h, tA1l, tA2h, tA2l, tBh, tBl;
  GPP_TRY(make_tensor_map_2d(&tA1h, a1.hi, 2, n, K1, a1.ldp, 64, 128, CU_TENSOR_MAP_SWIZZLE_128B));
  GPP_TRY(make_tensor_map_2d(&tA1l, a1.lo, 2, n, K1, a1.ldp, 64, 128, CU_TENSOR_MAP_SWIZZLE_128B));
  if (a2 && K2 > 0) {
    GPP_TRY(make_tensor_map_2d(&tA2h, a2->hi, 2, n, K2, a2->ldp, 64, 128, CU_TENSOR_MAP_SWIZZLE_128B));
    GPP_TRY(make_tensor_map_2d(&tA2l, a2->lo, 2, n, K2, a2->ldp, 64, 128, CU_TENSOR_MAP_SWIZZLE_128B));
  } else {
    tA2h = tA1h;
    tA2l = tA1l;
  }
  GPP_TRY(make_tensor_map_2d(&tBh, b.hi, 2, (int64_t)K1 + K2, ncols, b.ldp, 64, PBK, CU_TENSOR_MAP_SWIZZLE_128B));
  GPP_TRY(make_tensor_map_2d(&tBl, b.lo, 2, (int64_t)K1 + K2, ncols, b.ldp, 64, PBK, CU_TENSOR_MAP_SWIZZLE_128B));
  const int64_t nunits = p.row_tiles * p.col_tiles;
  const int pairs = (int)(nunits < pl_pairs() ? nunits : pl_pairs());
  if (pairs <= 0) return GPP_OK;
  if (const char* e = getenv("GPP_TC_WAVE_SYNC")) {   // experiment knob: 0 switches the wave alignment off
    if (e[0] == '0') p.wave_ctr = nullptr;
  }
  if (p.wave_ctr) GPP_CUDA(cudaMemsetAsync(p.wave_ctr, 0, 4, st));
  pl_rows_kernel<<<2 * pairs, kPlThreads, kPlSmemBytes, st>>>(tA1h, tA1l, tA2h, tA2l, tBh, tBl, p);
  GPP_LAUNCH_CHECK();
  return GPP_OK;
}

// workspace of pass 2: planes of W, the quad / xb2 partials and the finalize scratch
size_t pl_xb_workspace_bytes(int64_t n, int Q, int L) {
  const int64_t col_tiles = ceil_div(L, kTileN), row_tiles = ceil_div(n, kTileM);
  return align_up(planes_bytes(Q, L), 256) + align_up((size_t)col_tiles * 2 * n * sizeof(float), 256) +
         align_up((size_t)row_tiles * col_tiles * 16 * sizeof(double), 256) + align_up(xb_finalize_bytes(), 256) +
         256 /* wave counter */;
}

// Xb = alpha (X - V W) from the planes of V (W is split here: Q x L, small); with nll != nullptr the NLL epilogue.
int launch_pl_xb(const void* planesV, const float* X, int64_t ldx, const float* W, int64_t ldw, int64_t n, int Q, int L,
                 double* scal, float alpha_host, float* Xb, int64_t ldxb, float* nll, void* ws, size_t ws_bytes,
                 cudaStream_t st) {
  const size_t need = pl_xb_workspace_bytes(n, Q, L);
  if (!ws || ws_bytes < need) {
    set_error("xb_nll (planes): workspace too small (%zu < %zu bytes)", ws_bytes, need);
    return GPP_ERR_WORKSPACE;
  }
  char* wsb = static_cast<char*>(ws);
  void* planesW = wsb;
  size_t off = align_up(planes_bytes(Q, L), 256);
  GPP_TRY(launch_split_planes(W, ldw, Q, L, planesW, nullptr, 0, false, nullptr, 0, st));
  const int64_t col_tiles = ceil_div(L, kTileN), row_tiles = ceil_div(n, kTileM);
  PlRowsParams p{};
  p.mode = 0; p.X = X; p.ldx = ldx; p.out = Xb; p.ldo = ldxb; p.scal = scal; p.alpha_host = alpha_host;
  if (nll) {
    p.quad_part = reinterpret_cast<float*>(wsb + off);
    off += align_up((size_t)col_tiles * 2 * n * sizeof(float), 256);
    p.xb2_part = reinterpret_cast<double*>(wsb + off);
    off += align_up((size_t)row_tiles * col_tiles * 16 * sizeof(double), 256);
  }
  const PlanesView pv = planes_view(const_cast<void*>(planesV), n, Q);
  const PlanesView pw = planes_view(planesW, Q, L);
  p.wave_ctr = reinterpret_cast<unsigned int*>(wsb + need - 256);
  GPP_TRY(launch_pl_rows(pv, Q, nullptr, 0, pw, n, L, p, st));
  if (nll) {
    double* fin = reinterpret_cast<double*>(wsb + off);
    GPP_TRY(launch_xb_finalize(p.quad_part, (int)(col_tiles * 2), n, p.xb2_part, row_tiles * col_tiles * 16, fin, scal,
                               nll, st));
  }
  return GPP_OK;
}

// ---------------------------------------------------------------- Vb on planes
// Vb = (v0/vn) L_true V B^-1 - Xb W^T = [V | Xb] . [ (v0/vn) L_true Binv ; -W^T ]   (gp.py:68-71)
// The two parts of A share one accumulator, hence one scale: V's planes carry 2^(7 - eV), Xb's their own 2^(7 - eXb);
// the difference 2^(eXb - eV) (exact) goes into the -W^T rows of the stacked right-hand side before IT is split.
__global__ void __launch_bounds__(256) build_bstk_scaled_kernel(const float* __restrict__ Binv, const float* __restrict__ W,
                                                                int64_t ldw, const double* __restrict__ scal, int Q, int L,
                                                                int L_true, const uint32_t* __restrict__ metaV,
                                                                const uint32_t* __restrict__ metaXb,
                                                                float* __restrict__ Bstk) {
  const float coef = (float)(scal[GPP_S_V0] / scal[GPP_S_VN] * (double)L_true);
  const float wsc = -exp2f((float)(exp_of_bits(metaXb) - exp_of_bits(metaV)));
  const int64_t total = (int64_t)(Q + L) * Q;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int r = (int)(e / Q), c = (int)(e - (int64_t)r * Q);
    Bstk[e] = r < Q ? coef * Binv[(int64_t)r * Q + c] : wsc * W[(int64_t)c * ldw + (r - Q)];
  }
}

size_t pl_vb_workspace_bytes(int64_t n, int Q, int L) {
  return align_up(planes_bytes(n, L), 256) + align_up((size_t)(Q + L) * Q * sizeof(float), 256) +
         align_up(planes_bytes(Q + L, Q), 256) + 256 /* wave counter */;
}

int launch_pl_vb(const void* planesV, const float* Xb, int64_t ldxb, const float* Binv, const float* W, int64_t ldw,
                 const double* scal, int64_t n, int Q, int L, int L_true, float* Vb, int64_t ldvb, void* ws,
                 size_t ws_bytes, cudaStream_t st) {
  const size_t need = pl_vb_workspace_bytes(n, Q, L);
  if (!ws || ws_bytes < need) {
    set_error("vb (planes): workspace too small (%zu < %zu bytes)", ws_bytes, need);
    return GPP_ERR_WORKSPACE;
  }
  char* wsb = static_cast<char*>(ws);
  void* planesXb = wsb;
  float* Bstk = reinterpret_cast<float*>(wsb + align_up(planes_bytes(n, L), 256));
  void* planesB = wsb + align_up(planes_bytes(n, L), 256) + align_up((size_t)(Q + L) * Q * sizeof(float), 256);
  GPP_TRY(launch_split_planes(Xb, ldxb, n, L, planesXb, nullptr, 0, false, nullptr, 0, st));
  const PlanesView pv = planes_view(const_cast<void*>(planesV), n, Q);
  const PlanesView px = planes_view(planesXb, n, L);
  build_bstk_scaled_kernel<<<1024, 256, 0, st>>>(Binv, W, ldw, scal, Q, L, L_true, pv.meta, px.meta, Bstk);
  GPP_LAUNCH_CHECK();
  GPP_TRY(launch_split_planes(Bstk, Q, (int64_t)Q + L, Q, planesB, nullptr, 0, false, nullptr, 0, st));
  const PlanesView pb = planes_view(planesB, (int64_t)Q + L, Q);
  PlRowsParams p{};
  p.mode = 1; p.out = Vb; p.ldo = ldvb; p.alpha_host = 1.f;
  p.wave_ctr = reinterpret_cast<unsigned int*>(wsb + need - 256);
  return launch_pl_rows(pv, Q, &px, L, pb, n, Q, p, st);
}

// ---------------------------------------------------------------- structured route on planes
// planes (P x nviews ((with_x ? p : 0) + L)) <- [cnt (x) xn | slot sums of X]; n = rows of X.  with_x = 2: the
// cnt (x) xn part alone (P x nviews p, X is not read).
int launch_kr_slot_sums_planes(const float* X, int64_t ldx, int64_t n, const int64_t* order, const int64_t* slot_start,
                               const float* xn, int64_t P, int p, int nviews, int L, int with_x, int max_count,
                               void* planes, cudaStream_t st) {
  const int Lz = with_x == 2 ? 0 : L;
  const int cols = nviews * ((with_x ? p : 0) + Lz);
  PlanesView pv = planes_view(planes, P, cols);
  if (Lz) GPP_TRY(tc_absmax(X, ldx, n, L, pv.meta + 2, st));
  slot_scale_kernel<<<1, 32, 0, st>>>(pv.meta, max_count > 0 ? max_count : 1, with_x);
  GPP_LAUNCH_CHECK();
  const int64_t slots = P * nviews;
  const int grid = (int)(ceil_div(slots, 8) < 8192 ? ceil_div(slots, 8) : 8192);
  kr_slot_sum_planes_kernel<<<grid, 256, 0, st>>>(X, ldx, order, slot_start, xn, P, p, nviews, Lz, with_x != 0, pv.hi,
                                                  pv.lo, pv.ldp, pv.meta);
  GPP_LAUNCH_CHECK();
  return GPP_OK;
}

// out (n x ncols) = alpha A B with A (n x K) and B (K x ncols) as planes; ws: 256 bytes (wave counter)
int launch_pl_am(const void* planesA, const void* planesB, int64_t n, int K, int ncols, float alpha, float* out,
                 int64_t ldo, void* ws, size_t ws_bytes, cudaStream_t st) {
  if (!ws || ws_bytes < 256) {
    set_error("am (planes): workspace too small (%zu < 256 bytes)", ws_bytes);
    return GPP_ERR_WORKSPACE;
  }
  const PlanesView pa = planes_view(const_cast<void*>(planesA), n, K);
  const PlanesView pb = planes_view(const_cast<void*>(planesB), K, ncols);
  PlRowsParams p{};
  p.mode = 1; p.out = out; p.ldo = ldo; p.alpha_host = alpha;
  p.wave_ctr = static_cast<unsigned int*>(ws);
  return launch_pl_rows(pa, K, nullptr, 0, pb, n, ncols, p, st);
}

}  // namespace gpp
