// Pass 1, pass 2, Vb and the Q-space block GEMMs on the 5th-generation tensor cores, fp32-accurate through a 3-term
// operand split  a.b ~= hi(a).hi(b) + hi(a).lo(b) + lo(a).hi(b),  on CTA PAIRS, with the M operand in TENSOR MEMORY.
//
// Every GEMM tile is 256 x 256 and belongs to a cluster of two CTAs (tcgen05 cta_group::2): each CTA stages ITS 128
// rows of the M operand (A) and ITS 128 columns of the N operand (B); the leader CTA issues M = 256, N = 256 MMAs whose
// A operand is read from both CTAs' TMEM and whose B operand is read from both CTAs' shared memory; each CTA's TMEM
// receives its 128 accumulator rows.
//
//   pass 1:  D = sum_k A[k, m]^T B[k, n]   A = V[:, 256 tm ..], B = V[:, 256 tn ..] or X[:, 256 j ..]
//            both operands are row-major with the contraction over ROWS.  The raw fp32 tiles are written by a TMA box
//            {32 floats, BK rows} with SWIZZLE_128B_ATOM_32B (atom = 32 floats x 4 k-rows, 32-byte chunks XORed with
//            row % 4) -- for tf32 the only MN-major UMMA layout (LBO = BK * 128 B between 32-float column groups,
//            SBO = 512 B between 4-row k-groups, 1 KB per K = 8), which the wide-range variant feeds to the tensor
//            core as it landed.  A is TRANSPOSED into TMEM by the converter warps (thread m reads column m of the
//            tile: conflict-free, one 128-byte row per warp and k).
//   rows  :  D = sum_k [A1 | A2][row, k] B[k, col]   (pass 2: A1 = V, B = W; Vb: A1 = V, A2 = Xb, B = [rL Binv; -W^T])
//            A lands K-major: TMA box {16 floats, 128 rows} with SWIZZLE_64B; thread m reads its row (4 x 128 bit).
//
// The three terms per 16-row stage come in two variants (template parameter F16; see the comment at F16Scales).
// Hardware facts measured on B200 (experiments/tc/exp1_gram.cu): kind::tf32 TRUNCATES fp32 operands, and the TMEM
// accumulator is rounded toward zero after every MMA.
//   F16 = true (data passes): hi(x) = x rounded to 11 significant bits, lo(x) = x - hi(x); all three terms are ONE
//            K = 16 kind::f16 MMA each, on fp16 operands that carry one common power-of-two scale per operand
//            (absmax_bits_kernel): A hi / lo from TMEM, B hi / lo from two fp16 planes in shared memory.
//   F16 = false (Q-space block GEMMs, wide dynamic range): hi.hi as two K = 8 kind::tf32 MMAs on the RAW fp32 data
//            (the hardware truncation is the split; B = the TMA tile as it landed), the correction terms a.lo(b) and
//            lo(a).b as one K = 16 kind::f16 MMA each with their own scale.
//   Accumulation in TMEM is limited to WINDOWS of 4 stages (64 k-rows); inside a window ALL correction terms are
//   issued first, into the still-small accumulator, the hi.hi terms last (a correction term added to a large
//   accumulator is truncated at the accumulator's ulp: measured 1.5e-6 with 2-stage groups in an 8-stage window).
//   Finished windows are added in fp32 registers (round-to-nearest) by the drain warps.
//
// Why A lives in TMEM.  With both operands in shared memory a 16-row stage cost, per CTA, 48 KB of MMA operand reads
// + 32 KB of converter traffic + 16 KB of TMA writes = 848 shared-memory wavefronts against 768 tensor-pipe cycles:
// the first pair kernel was shared-memory-bandwidth bound.  Now: 16 KB of B reads + 24 KB converter + 16 KB TMA.
// TMEM map (512 columns): [0, 256) the accumulator tile; [256, 512) ring of 8 A slots of 32 columns per stage: 8 columns
// of fp16 hi pairs + 8 of lo pairs (F16), or 16 columns a 2^g in fp32 + 8 + 8 columns of fp16 pairs (wide-range).
// (Measured and dropped: two staggered 128-column half accumulators -- an N = 128 MMA with A from TMEM takes ~117
//  cycles, not 64; separate rings for the raw A and B tiles; L2 prefetch of later stages -- 30 % SLOWER; k-splits from
//  2 k to 55 k rows -- no effect.  Kept: the per-wave alignment of the producers, see the producer loop of pass 1.)
//
// Warp roles per CTA (512 threads, setmaxnreg re-balanced): warp 0 TMA producer (own halves), warp 1 MMA issuer
// (leader CTA only) + TMEM owner, warps 4-7 converters (thread = A row = TMEM lane), warps 8-15 drain / epilogue.
// Rings: raw tiles (TMA -> converter -> MMA, 16 KB: A raw + B raw = B hi) and lo slots (the two fp16 planes of B in
// shared memory + the A slot in TMEM; converter -> MMA).  Barriers: full[s] (local TMA -> local converters), conv[s]
// (converters of BOTH CTAs -> leader), empty[s], lo_empty[s] and tfull (MMA commit, multicast to both CTAs), tempty
// (drain warps of both CTAs -> leader).  Remote arrives use the default .release.cta semantics on purpose
// (.release.cluster compiles to MEMBAR.ALL.GPU per arrive).
// Pass 1 is persistent over (tile, k-split) units with a deterministic split-K: every unit writes its own partial
// tile, tc_reduce_kernel sums them in a fixed order (fp64) and tc_mirror_kernel fills the upper triangle of G.
#include <stdlib.h>

#include <mutex>

#include "common.cuh"
#include "kernels.h"
#include "pass1_common.cuh"
#include "tc_common.cuh"

namespace gpp {

using namespace tc;

namespace {

#ifndef GPP_TC_RAW
#define GPP_TC_RAW 10    // raw tiles in flight: TMA -> converter -> MMA (wide-range variant: B hi is read from them)
#endif
#ifndef GPP_TC_LO
#define GPP_TC_LO 8      // converted slots in flight (fp16 planes of B in shared memory + A slot in TMEM): converter -> MMA
#endif
constexpr int TM = kTileM, TN = kTileN;   // tile of a CTA pair
constexpr int HM = 128, HN = 128;   // what one CTA stages of it
constexpr int TBK = 16, kRaw = GPP_TC_RAW, kLo = GPP_TC_LO;
#ifndef GPP_TC_GROUP
#define GPP_TC_GROUP 4
#endif
#ifndef GPP_TC_WINGROUPS
#define GPP_TC_WINGROUPS 1
#endif
constexpr int kGroup = GPP_TC_GROUP;           // stages per issue group (cross terms of the group first, then hi.hi)
constexpr int kWinGroups = GPP_TC_WINGROUPS;   // groups per accumulation window (window = 4 stages = 64 k-rows)
constexpr int kABytes = HM * TBK * 4, kBBytes = HN * TBK * 4, kRawBytes = kABytes + kBBytes;   // 8 K + 8 K
constexpr int kTcThreads = 512;
constexpr int kSmemBytes = kRaw * kRawBytes + kLo * kBBytes + 1024 /*align*/ + 512 /*barriers*/;
#ifndef GPP_TC_F16_LBO
#define GPP_TC_F16_LBO 2048
#endif
#ifndef GPP_TC_F16_SBO
#define GPP_TC_F16_SBO 1024
#endif
// Scales of the split (all exact powers of two), from eA, eB = the binary exponents of max|A|, max|B| (measured on the
// device by absmax_bits_kernel; 0 when unknown).
// Two splits live side by side, chosen per launch (template parameter F16):
//   F16 = true   all three terms on the fp16 pipe (three K = 16 fp16 MMAs per stage, 1.5 TF32-pass equivalents): the
//                large data passes (V^T [V | Z], Z - V W, Vb, the structured route's products);
//   F16 = false  hi.hi as 2 x kind::tf32 on the raw fp32 tile, the two correction terms in fp16 with their own scale (2.0
//                pass equivalents): the Q-space block GEMMs, whose operands (Cholesky factor, its inverse) span many
//                orders of magnitude -- the common scale of the fp16 split gives elements below 2^-10 of the largest
//                one absolute instead of relative precision, which cond(B) ~ 1e4 amplifies (c1 at lvs = (2, -4): W
//                error 1.7e-3 against 2.7e-4, dNLL/dZ 1.1e-4 against 1.5e-5; experiments/bench/c1_diag.py).
struct F16Scales {
  float a32, a_hi, a_lo, b_hi, b_lo, out;
};
// The 11 leading significant bits of an fp32 number (given as its bit pattern): the tf32 pipe truncates, so its split
// truncates too; the fp16 split rounds (half away from zero), which halves the remainder and makes its sign random --
// the dropped lo.lo term is then zero-mean instead of a coherent bias.
template <bool F16>
__device__ __forceinline__ float hi11(uint32_t bits) {
  return __uint_as_float(F16 ? ((bits + 0x1000u) & 0xFFFFE000u) : (bits & 0xFFFFE000u));
}
// (the fp16 split and its common scale kF16Top are described in pass1_common.cuh)
// tf32 split: each fp16 factor of the correction terms is normalised by its own operand's magnitude,
//   a.lo(b) -> (a 2^-eA) . (lo(b) 2^(11 - eB))      lo(a).b -> (lo(a) 2^(11 - eA)) . (b 2^-eB)
// both scaled by 2^g, g = 11 - eA - eB; hi.hi is brought to the same scale by writing a 2^g (exact) as its A operand.
template <bool F16>
__device__ __forceinline__ F16Scales make_scales(int eA, int eB) {
  F16Scales s;
  if (F16) {
    s.a32 = 1.f;
    s.a_hi = s.a_lo = exp2f((float)(kF16Top - eA));
    s.b_hi = s.b_lo = exp2f((float)(kF16Top - eB));
    s.out = exp2f((float)(eA + eB - 2 * kF16Top));
  } else {
    const int g = 11 - eA - eB;
    s.a32 = exp2f((float)g);          s.out = exp2f((float)-g);
    s.a_hi = exp2f((float)-eA);       s.a_lo = exp2f((float)(11 - eA));
    s.b_hi = exp2f((float)-eB);       s.b_lo = exp2f((float)(11 - eB));
  }
  return s;
}

// out[0] = max over the matrix of the bit pattern of |x| (monotonic in |x|); out must be zeroed before the launch.
// Flat walk over the float4 groups of the matrix, four loads in flight per thread.  (First version: one CTA per row with
// a thread per float4 of it -- for the 256-column latent matrix only 64 of 256 threads had work and each had one load
// outstanding: 0.50 ms for the 1 GB of Z at c3, 2 TB/s.)
__global__ void __launch_bounds__(256) absmax_bits_kernel(const float* __restrict__ X, int64_t ld, int64_t rows, int cols,
                                                          uint32_t* __restrict__ out) {
  const int c4n = cols >> 2;
  const int64_t total = rows * c4n, stride = (int64_t)gridDim.x * blockDim.x;
  const bool flat = ld == cols;
  uint32_t m = 0;
  auto fold = [&](const float4 v) {
    m = max(m, __float_as_uint(v.x) & 0x7FFFFFFFu); m = max(m, __float_as_uint(v.y) & 0x7FFFFFFFu);
    m = max(m, __float_as_uint(v.z) & 0x7FFFFFFFu); m = max(m, __float_as_uint(v.w) & 0x7FFFFFFFu);
  };
  auto at = [&](int64_t i) -> float4 {
    if (flat) return reinterpret_cast<const float4*>(X)[i];
    const int64_t r = i / c4n;
    return reinterpret_cast<const float4*>(X + r * ld)[i - r * c4n];
  };
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  for (; i + 3 * stride < total; i += 4 * stride) {
    const float4 v0 = at(i), v1 = at(i + stride), v2 = at(i + 2 * stride), v3 = at(i + 3 * stride);
    fold(v0); fold(v1); fold(v2); fold(v3);
  }
  for (; i < total; i += stride) fold(at(i));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0 && m) atomicMax(out, m);
}
constexpr int kAccCols = 256, kASlotCols = 32;   // TMEM: accumulator tile, then kLo A slots (16 hi + 16 lo columns)
static_assert(kGroup < kLo && kLo <= kRaw && kAccCols + kLo * kASlotCols <= 512, "ring sizes");
static_assert(kSmemBytes <= 232448, "shared memory budget");

// Optional role profiling (-DGPP_TC_PROF): cycles each role spends waiting on its barriers, per CTA.
#ifdef GPP_TC_PROF
__device__ unsigned long long g_prof[512][16];
#define PROF_DECL unsigned long long pw0 = 0, pw1 = 0; const unsigned long long pt0 = clock64()
#define PROF_WAIT(var, stmt) do { const unsigned long long c0__ = clock64(); stmt; var += clock64() - c0__; } while (0)
#define PROF_STORE(slot) do { g_prof[blockIdx.x][(slot) * 3 + 0] = pw0; g_prof[blockIdx.x][(slot) * 3 + 1] = pw1; \
                              g_prof[blockIdx.x][(slot) * 3 + 2] = clock64() - pt0; } while (0)
#else
#define PROF_DECL unsigned long long pw0 = 0, pw1 = 0
#define PROF_WAIT(var, stmt) stmt
#define PROF_STORE(slot) do { } while (0)
#endif

struct TcShared {
  uint64_t full[kRaw], empty[kRaw], conv[kLo], lo_empty[kLo], tfull[2], tempty[2];
  uint32_t tmem_base;
};

// ---- pieces shared by the two kernels ----------------------------------------------------------------------
// Raw slots are handed back to the TMA producer by the MMA commit in both splits.  (Releasing them from the converter
// warps as soon as the tile is in registers -- possible in the fp16 split, whose MMAs never read the raw tile -- was
// measured: no gain, the kernel is bound by the L2 -> shared-memory stream, and an intermittent 6e-4 error in the
// Gram tiles, i.e. the arrive does not order the converters' outstanding shared-memory loads before the next TMA write.)
template <bool F16>
__device__ __forceinline__ TcShared* tc_prologue(uint8_t* base, uint32_t& tmem) {
  TcShared* sm = reinterpret_cast<TcShared*>(base + kRaw * kRawBytes + kLo * kBBytes);
  if (threadIdx.x == 0) {
    for (int s = 0; s < kRaw; ++s) {
      mbar_init(&sm->full[s], 1);
      mbar_init(&sm->empty[s], 1);
    }
    for (int s = 0; s < kLo; ++s) {
      mbar_init(&sm->conv[s], 12);    // (4 A + 2 B converter warps) x 2 CTAs (used in the leader)
      mbar_init(&sm->lo_empty[s], 1);
    }
    for (int h = 0; h < 2; ++h) {
      mbar_init(&sm->tfull[h], 1);
      mbar_init(&sm->tempty[h], 16);  // 8 drain warps x 2 CTAs (used in the leader)
    }
    fence_mbar_init();
  }
  if ((threadIdx.x >> 5) == 1) tmem_alloc_pair(&sm->tmem_base, 512);
  tcgen05_fence_before();
  cluster_sync_all();   // barriers of both CTAs initialised, TMEM allocated
  tcgen05_fence_after();
  tmem = sm->tmem_base;
  return sm;
}

__device__ __forceinline__ void tc_epilogue(uint32_t tmem) {
  tcgen05_fence_before();
  cluster_sync_all();   // no CTA leaves (or frees TMEM) while its peer may still touch its shared memory / barriers
  if ((threadIdx.x >> 5) == 1) tmem_dealloc_pair(tmem, 512);
}

__device__ __forceinline__ float lds_f32(uint32_t addr) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
  return v;
}
__device__ __forceinline__ float4 lds_f32x4(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}

// The B half-tile of a stage (16 k-rows x 128 columns of fp32) is converted in 16 units of one float4 per lane: unit m
// covers 64-column group m & 1 and k-rows 2 (m >> 1) + {0, 1}.  float4 (k-row kb, 32-float group 2 jj + bb, 16-byte
// position qb) is chosen so that 16 lanes cover the 64 columns of one fp16 row: conflict-free 128-bit loads and
// conflict-free 64-bit stores into the fp16 planes (hi plane at +0, lo plane at +4 KB), each MN-major SWIZZLE_128B:
// 64-column group g at g * 2 KB, k-row k at (k / 8) * 1 KB + (k % 8) * 128 B, 16-byte chunk ((c % 64) / 8) ^ (k % 8),
// element (c % 8) * 2 B.
// Eight units per B-converter warp.  (Giving the four A-converter warps one unit each was measured: no gain -- the
// kernel is bound by the L2 -> shared-memory stream of the raw tiles, not by the converters.)
constexpr int kBUnitsB = 8;

__device__ __forceinline__ float4 b_unit_load(uint32_t braw, int m, int lane) {
  const int qb = lane & 7, bb = (lane >> 3) & 1, kpar = lane >> 4;
  const int jj = m & 1, kb = 2 * (m >> 1) + kpar;
  return lds_f32x4(braw + (2 * jj + bb) * (TBK * 128) + kb * 128 + qb * 16);
}
template <bool F16>
__device__ __forceinline__ void b_unit_store(uint32_t bplane, int m, int lane, const float4 v, const F16Scales& sc) {
  const int qb = lane & 7, bb = (lane >> 3) & 1, kpar = lane >> 4;
  const int jj = m & 1, kb = 2 * (m >> 1) + kpar;
  const int chunk = 4 * bb + ((qb >> 1) ^ (kb & 3));          // logical 8-column chunk within the 64-column group
  const uint32_t dst = bplane + jj * 2048 + (kb >> 3) * 1024 + (kb & 7) * 128 + ((chunk ^ (kb & 7)) << 4) + (qb & 1) * 8;
  const float hx = hi11<F16>(__float_as_uint(v.x)), hy = hi11<F16>(__float_as_uint(v.y));
  const float hz = hi11<F16>(__float_as_uint(v.z)), hw = hi11<F16>(__float_as_uint(v.w));
  const uint32_t h0 = F16 ? pack_f16x2(hx * sc.b_hi, hy * sc.b_hi) : pack_f16x2(v.x * sc.b_hi, v.y * sc.b_hi);
  const uint32_t h1 = F16 ? pack_f16x2(hz * sc.b_hi, hw * sc.b_hi) : pack_f16x2(v.z * sc.b_hi, v.w * sc.b_hi);
  const uint32_t l0 = pack_f16x2((v.x - hx) * sc.b_lo, (v.y - hy) * sc.b_lo);
  const uint32_t l1 = pack_f16x2((v.z - hz) * sc.b_lo, (v.w - hw) * sc.b_lo);
  asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(dst), "r"(h0), "r"(h1) : "memory");
  asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(dst + kBBytes / 2), "r"(l0), "r"(l1) : "memory");
}

// Converter warps.  Two independent chains per stage, so that neither is as long as a tensor-pipe stage:
//   A chain, warps 4-7 (thread t = A row t of this CTA = TMEM lane t): raw A tile -> TMEM slot: 16 columns a 2^g
//            (hi.hi term), 8 columns fp16 pairs of the normalised a, 8 columns fp16 pairs of the normalised lo(a);
//   B chain, warps 2-3: raw B tile -> the two fp16 planes (normalised b, normalised lo(b)) in the lo slot.
// Explicit shared-space accesses, all loads before the first store (through generic pointers the compiler kept every
// load behind the previous store).  A_MN: the raw A tile is MN-major (pass 1: [k-row][32-float group],
// SWIZZLE_128B_BASE32B) or K-major (row GEMM: [row][16 floats], SWIZZLE_64B).
template <bool A_MN, bool F16>
__device__ __forceinline__ void convert_a_stage(uint8_t* base, TcShared* sm, uint32_t tmem, uint32_t conv0_leader,
                                                uint32_t it, const F16Scales& sc, unsigned long long& pw0,
                                                unsigned long long& pw1) {
  const int t = threadIdx.x - 128, lane = threadIdx.x & 31, wq = t >> 5;
  const int s = it % kRaw, sl = it % kLo;
  PROF_WAIT(pw0, mbar_wait(&sm->full[s], (it / kRaw) & 1));
  const uint32_t raw = smem_u32(base + s * kRawBytes);
  uint32_t ahi[TBK];
  if (A_MN) {
    // element (k, m = t): group wq, k-row k, 32-byte chunk ((lane / 8) ^ (k % 4)), word lane % 8
    const uint32_t a0 = raw + wq * (TBK * 128) + (lane & 7) * 4;
#pragma unroll
    for (int k = 0; k < TBK; ++k)
      ahi[k] = __float_as_uint(lds_f32(a0 + k * 128 + (((lane >> 3) ^ (k & 3)) << 5)));
  } else {
    // row t: 64 bytes, 16-byte chunk c stored at c ^ ((t / 2) % 4)
    const uint32_t a0 = raw + t * 64;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const float4 v = lds_f32x4(a0 + ((c ^ ((t >> 1) & 3)) << 4));
      ahi[4 * c + 0] = __float_as_uint(v.x); ahi[4 * c + 1] = __float_as_uint(v.y);
      ahi[4 * c + 2] = __float_as_uint(v.z); ahi[4 * c + 3] = __float_as_uint(v.w);
    }
  }
  uint32_t a16[TBK];
#pragma unroll
  for (int c = 0; c < TBK / 2; ++c) {
    const float x0 = __uint_as_float(ahi[2 * c]), x1 = __uint_as_float(ahi[2 * c + 1]);
    const float l0 = x0 - hi11<F16>(ahi[2 * c]), l1 = x1 - hi11<F16>(ahi[2 * c + 1]);
    // even k in the low half of the TMEM column
    a16[c] = F16 ? pack_f16x2((x0 - l0) * sc.a_hi, (x1 - l1) * sc.a_hi) : pack_f16x2(x0 * sc.a_hi, x1 * sc.a_hi);
    a16[TBK / 2 + c] = pack_f16x2(l0 * sc.a_lo, l1 * sc.a_lo);
  }
  if (!F16) {
#pragma unroll
    for (int k = 0; k < TBK; ++k) ahi[k] = __float_as_uint(__uint_as_float(ahi[k]) * sc.a32);   // exact
  }
  PROF_WAIT(pw1, mbar_wait(&sm->lo_empty[sl], ((it / kLo) & 1) ^ 1));
  tcgen05_fence_after();
  const uint32_t ta = tmem + ((uint32_t)(wq * 32) << 16) + kAccCols + sl * kASlotCols;
  if (F16) {
    tmem_st_32x16(ta, a16);            // columns [0, 8): hi, [8, 16): lo
  } else {
    tmem_st_32x16(ta, ahi);            // columns [0, 16): a 2^g (fp32), [16, 24): a (fp16), [24, 32): lo(a)
    tmem_st_32x16(ta + TBK, a16);
  }
  tmem_wait_st();
  tcgen05_fence_before();
  __syncwarp();
  if (lane == 0) mbar_arrive_cluster(conv0_leader + 8u * sl);
}

template <bool F16>
__device__ __forceinline__ void convert_b_stage(uint8_t* base, TcShared* sm, uint32_t conv0_leader, uint32_t it,
                                                const F16Scales& sc, unsigned long long& pw0, unsigned long long& pw1) {
  const int lane = threadIdx.x & 31, w2 = (threadIdx.x >> 5) - 2;
  const int s = it % kRaw, sl = it % kLo;
  PROF_WAIT(pw0, mbar_wait(&sm->full[s], (it / kRaw) & 1));
  const uint32_t braw = smem_u32(base + s * kRawBytes) + kABytes;
  float4 bv[kBUnitsB];
#pragma unroll
  for (int i = 0; i < kBUnitsB; ++i) bv[i] = b_unit_load(braw, w2 * kBUnitsB + i, lane);
  PROF_WAIT(pw1, mbar_wait(&sm->lo_empty[sl], ((it / kLo) & 1) ^ 1));
  const uint32_t bplane = smem_u32(base + kRaw * kRawBytes + sl * kBBytes);
#pragma unroll
  for (int i = 0; i < kBUnitsB; ++i) b_unit_store<F16>(bplane, w2 * kBUnitsB + i, lane, bv[i], sc);
  fence_proxy_async_smem();   // generic-proxy writes -> visible to the tensor core (async proxy)
  __syncwarp();
  if (lane == 0) mbar_arrive_cluster(conv0_leader + 8u * sl);
}

// ---- window schedule ------------------------------------------------------------------------------------------
// A unit of `nst` stages is issued in groups of kGroup stages; the accumulator collects windows of kWinGroups groups.
// Both the issuer and the drain warps walk this schedule.
__device__ __forceinline__ bool win_begins(int g) { return (g % kWinGroups) == 0; }
__device__ __forceinline__ bool win_ends(int g, int ngroups) { return g == ngroups - 1 || (g % kWinGroups) == kWinGroups - 1; }

// MMA issuer (one thread of the leader): group g of a unit (stages [it, it + gst)).
// wc: windows issued so far (barrier phase).
template <bool F16>
__device__ __forceinline__ void issue_group(uint8_t* base, TcShared* sm, uint32_t tmem, uint32_t it, int gst, int g,
                                            int ngroups, uint32_t& wc, unsigned long long& pw0,
                                            unsigned long long& pw1) {
  constexpr uint32_t idesc = umma_idesc_tf32(TM, TN, false, true);
  const uint32_t d = tmem;
  uint32_t acc = 1;
  if (win_begins(g)) {
    PROF_WAIT(pw0, mbar_wait_cluster(&sm->tempty[0], (wc & 1) ^ 1));
    tcgen05_fence_after();
    acc = 0;
  }
  for (int j = 0; j < gst; ++j) {   // cross terms of the group first: they land in a still-small accumulator
    const int sl = (it + j) % kLo;
    PROF_WAIT(pw1, mbar_wait_cluster(&sm->conv[sl], ((it + j) / kLo) & 1));
    tcgen05_fence_after();
    // one K = 16 fp16 MMA per correction term: (a 2^-6) . (b_lo 2^6) and (a_lo 2^6) . (b 2^-6)
    constexpr uint32_t idesc16 = umma_idesc_f16(TM, TN, false, true);
    const uint32_t b16 = smem_u32(base + kRaw * kRawBytes + sl * kBBytes);
    const uint32_t a16 = tmem + kAccCols + sl * kASlotCols + (F16 ? 0 : TBK);
    umma_f16_pair_ts(d, a16, umma_desc(b16 + kBBytes / 2, GPP_TC_F16_LBO, GPP_TC_F16_SBO, kLayoutSw128), idesc16, acc);
    umma_f16_pair_ts(d, a16 + TBK / 2, umma_desc(b16, GPP_TC_F16_LBO, GPP_TC_F16_SBO, kLayoutSw128), idesc16, 1);
    acc = 1;
  }
  for (int j = 0; j < gst; ++j) {   // then the hi.hi terms
    const int s = (it + j) % kRaw, sl = (it + j) % kLo;
    if (F16) {
      constexpr uint32_t idesc16 = umma_idesc_f16(TM, TN, false, true);
      const uint32_t b16 = smem_u32(base + kRaw * kRawBytes + sl * kBBytes);
      umma_f16_pair_ts(d, tmem + kAccCols + sl * kASlotCols, umma_desc(b16, GPP_TC_F16_LBO, GPP_TC_F16_SBO, kLayoutSw128),
                       idesc16, 1);
    } else {
      const uint32_t b_hi = smem_u32(base + s * kRawBytes) + kABytes;
      const uint32_t a_hi = tmem + kAccCols + sl * kASlotCols;
#pragma unroll
      for (int kk = 0; kk < TBK / 8; ++kk)
        umma_tf32_pair_ts(d, a_hi + kk * 8, umma_desc(b_hi + kk * 1024, TBK * 128, 512, kLayoutSw128Base32), idesc, 1);
    }
    umma_commit_pair(&sm->empty[s], 3);       // raw tile, fp16 planes and A slot are free in both CTAs
    umma_commit_pair(&sm->lo_empty[sl], 3);
  }
  if (win_ends(g, ngroups)) {
    umma_commit_pair(&sm->tfull[0], 3);
    ++wc;
  }
}

// Drain warps: after a group that ends a window, add the window (this CTA's 128 rows x this warp's 128 columns) into
// registers.
__device__ __forceinline__ void drain_group(TcShared* sm, uint32_t tmem, uint32_t tempty0_leader, int g, int ngroups,
                                            uint32_t& wc, float (&acc)[128], unsigned long long& pw0) {
  if (!win_ends(g, ngroups)) return;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t lane_addr = (uint32_t)((warp & 3) * 32) << 16;
  const int cb = (warp - 8) >> 2;
  PROF_WAIT(pw0, mbar_wait(&sm->tfull[0], wc & 1));
  ++wc;
  tcgen05_fence_after();
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    float v[32];
    tmem_ld_32x32(tmem + lane_addr + cb * 128 + c * 32, v);
#pragma unroll
    for (int j = 0; j < 32; ++j) acc[c * 32 + j] += v[j];
  }
  tcgen05_fence_before();
  __syncwarp();
  if (lane == 0) mbar_arrive_cluster(tempty0_leader);
}

// =====================================================================================================
template <bool F16>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kTcThreads, 1)
tc_pass1_kernel(const __grid_constant__ CUtensorMap tmV, const __grid_constant__ CUtensorMap tmX, Pass1Params p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;
  uint32_t tmem;
  TcShared* sm = tc_prologue<F16>(base, tmem);
  const int nunits = p.tiles * p.splits;

  if (warp < 4) {
    setmaxnreg_dec<80>();
    if (warp >= 2) {
      // ===================================================== B converters
      const uint32_t conv0 = mapa_u32(&sm->conv[0], 0);
      const int eV = exp_of_bits(p.amax), eX = exp_of_bits(p.amax ? p.amax + 1 : nullptr);
      const F16Scales sc_g = make_scales<F16>(eV, eV), sc_c = make_scales<F16>(eV, eX);
      PROF_DECL;
      uint32_t it = 0;
      for (int u = pair; u < nunits; u += npairs) {
        const int split = u / p.tiles, tile = u - split * p.tiles;
        const int64_t r0 = (int64_t)split * p.rows_per_split;
        const int64_t r1 = min(p.n, r0 + p.rows_per_split);
        const int nst = (int)((r1 - r0 + TBK - 1) / TBK);
        const F16Scales sc = tile < p.tiles_g ? sc_g : sc_c;
        for (int st = 0; st < nst; ++st, ++it) convert_b_stage<F16>(base, sm, conv0, it, sc, pw0, pw1);
      }
      if (threadIdx.x == 64) PROF_STORE(4);
    } else if (warp == 0 && lane == 0) {
      // ===================================================== TMA producer (this CTA's halves of A and B)
      PROF_DECL;
      tma_prefetch_desc(&tmV);
      tma_prefetch_desc(&tmX);
      uint32_t it = 0;
      bool wave_sync = p.wave_ctr != nullptr;
      for (int u = pair; u < nunits; u += npairs) {
        // Wave alignment: the pairs of one wave read the same rows of V at the same time (consecutive pairs share a
        // k-range), which is what lets L2 serve most of their loads -- but only while they stay within the L2
        // residency window of each other, and persistent CTAs drift apart (measured at c3: L2 hit rate 47 %, 166 GB
        // of DRAM reads per launch; aligned: 79 %, 42 GB, and 8 % less time under the power cap).  So no producer
        // starts the loads of wave w before every producer has issued all loads of wave w - 1.  It is a hint, not a
        // dependency: a producer that has waited 2 ms (CTAs not co-resident, e.g. another stream holds SMs) stops
        // aligning for the rest of the launch; the rings keep the tensor cores busy while a producer waits.
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
        const int nst = (int)((r1 - r0 + TBK - 1) / TBK);
        const CUtensorMap* mb = is_c ? &tmX : &tmV;
        const int acol = tm * TM + (int)rank * HM, bcol = tn * TN + (int)rank * HN;
        for (int st = 0; st < nst; ++st, ++it) {
          const int s = it % kRaw;
          PROF_WAIT(pw0, mbar_wait(&sm->empty[s], ((it / kRaw) & 1) ^ 1));
          uint8_t* dst = base + s * kRawBytes;
          const int row = (int)(r0 + (int64_t)st * TBK);
          mbar_arrive_expect_tx(&sm->full[s], kRawBytes);
#pragma unroll
          for (int g = 0; g < HM / 32; ++g) tma_load_2d(dst + g * (TBK * 128), &tmV, acol + g * 32, row, &sm->full[s]);
#pragma unroll
          for (int g = 0; g < HN / 32; ++g)
            tma_load_2d(dst + kABytes + g * (TBK * 128), mb, bcol + g * 32, row, &sm->full[s]);
        }
        if (p.wave_ctr) atomicAdd(p.wave_ctr, 1u);
      }
      PROF_STORE(0);
    } else if (warp == 1 && lane == 0 && rank == 0) {
      // ===================================================== MMA issuer (leader CTA)
      PROF_DECL;
      uint32_t it = 0, wc = 0;
      for (int u = pair; u < nunits; u += npairs) {
        const int split = u / p.tiles;
        const int64_t r0 = (int64_t)split * p.rows_per_split;
        const int64_t r1 = min(p.n, r0 + p.rows_per_split);
        const int nst = (int)((r1 - r0 + TBK - 1) / TBK);
        const int ngroups = (nst + kGroup - 1) / kGroup;
        for (int g = 0; g < ngroups; ++g) {
          const int gst = min(kGroup, nst - g * kGroup);
          issue_group<F16>(base, sm, tmem, it, gst, g, ngroups, wc, pw0, pw1);
          it += gst;
        }
      }
      PROF_STORE(1);
    }
  } else if (warp < 8) {
    setmaxnreg_dec<80>();
    // ======================================================= A converters
    PROF_DECL;
    const uint32_t conv0 = mapa_u32(&sm->conv[0], 0);
    const int eV = exp_of_bits(p.amax), eX = exp_of_bits(p.amax ? p.amax + 1 : nullptr);
    const F16Scales sc_g = make_scales<F16>(eV, eV), sc_c = make_scales<F16>(eV, eX);
    uint32_t it = 0;
    for (int u = pair; u < nunits; u += npairs) {
      const int split = u / p.tiles, tile = u - split * p.tiles;
      const int64_t r0 = (int64_t)split * p.rows_per_split;
      const int64_t r1 = min(p.n, r0 + p.rows_per_split);
      const int nst = (int)((r1 - r0 + TBK - 1) / TBK);
      const F16Scales sc = tile < p.tiles_g ? sc_g : sc_c;
      for (int st = 0; st < nst; ++st, ++it) convert_a_stage<true, F16>(base, sm, tmem, conv0, it, sc, pw0, pw1);
    }
    if (threadIdx.x == 128) PROF_STORE(2);
  } else {
    // ======================================================= drain warps: TMEM windows -> fp32 registers -> partial tile
    setmaxnreg_inc<176>();
    PROF_DECL;
    const uint32_t tempty0 = mapa_u32(&sm->tempty[0], 0);
    const int q = warp & 3, cb = (warp - 8) >> 2;
    const int eV = exp_of_bits(p.amax), eX = exp_of_bits(p.amax ? p.amax + 1 : nullptr);
    const float out_g = make_scales<F16>(eV, eV).out, out_c = make_scales<F16>(eV, eX).out;
    uint32_t wc = 0;
    for (int u = pair; u < nunits; u += npairs) {
      const int split = u / p.tiles, tile = u - split * p.tiles;
      const int64_t r0 = (int64_t)split * p.rows_per_split;
      const int64_t r1 = min(p.n, r0 + p.rows_per_split);
      const int nst = (int)((r1 - r0 + TBK - 1) / TBK);
      const int ngroups = (nst + kGroup - 1) / kGroup;
      float acc[128];
#pragma unroll
      for (int i = 0; i < 128; ++i) acc[i] = 0.f;
      for (int g = 0; g < ngroups; ++g) drain_group(sm, tmem, tempty0, g, ngroups, wc, acc, pw0);
      const float os = tile < p.tiles_g ? out_g : out_c;   // undo the common power-of-two scale of the split (exact)
      float* out = p.partial + ((size_t)tile * p.splits + split) * (size_t)(TM * TN) +
                   (size_t)(rank * HM + q * 32 + lane) * TN + cb * 128;
#pragma unroll
      for (int i = 0; i < 128; i += 4) {
        *reinterpret_cast<float4*>(out + i) = make_float4(os * acc[i], os * acc[i + 1], os * acc[i + 2], os * acc[i + 3]);
      }
    }
    if (threadIdx.x == 256) PROF_STORE(3);
  }
  tc_epilogue(tmem);
}

// GC[r][c] = sum_s partial[tile][s][..] for every computed tile (fixed order, fp64 accumulation).
// grid = tiles * 8: CTA (tile, j) reduces rows [32 j, 32 j + 32) of the tile.
__global__ void __launch_bounds__(256) tc_reduce_kernel(Pass1Params p) {
  const int tile = blockIdx.x >> 3, rblk = blockIdx.x & 7;
  int tm, tn;
  bool is_c;
  decode_tile(p, tile, tm, tn, is_c);
  const int ncols = is_c ? p.L : p.Q;
  const int col0 = tn * TN, row0 = tm * TM + rblk * 32;
  const float* src = p.partial + (size_t)tile * p.splits * (size_t)(TM * TN) + (size_t)rblk * 32 * TN;
  const double scale = (is_c && p.scal_c) ? p.scal_c[GPP_S_V0] / p.scal_c[GPP_S_VN] : 1.0;
  for (int e = threadIdx.x; e < 32 * TN / 4; e += blockDim.x) {
    const int r = e / (TN / 4), c4 = (e - r * (TN / 4)) * 4;
    if (row0 + r >= p.Q || col0 + c4 >= ncols) continue;
    double s0 = 0, s1 = 0, s2 = 0, s3 = 0;
    for (int s = 0; s < p.splits; ++s) {
      const float4 v = *reinterpret_cast<const float4*>(src + (size_t)s * (TM * TN) + r * TN + c4);
      s0 += v.x; s1 += v.y; s2 += v.z; s3 += v.w;
    }
    if (!is_c && tm == tn && p.diag) {   // diagonal entries of G: the exactly accumulated column sums of squares
      const int dc = row0 + r - (col0 + c4);
      if (dc == 0) s0 = p.diag[row0 + r];
      else if (dc == 1) s1 = p.diag[row0 + r];
      else if (dc == 2) s2 = p.diag[row0 + r];
      else if (dc == 3) s3 = p.diag[row0 + r];
    }
    float* dst = (is_c ? p.C + (int64_t)(row0 + r) * p.ldc : p.G + (int64_t)(row0 + r) * p.ldg) + col0 + c4;
    *reinterpret_cast<float4*>(dst) =
        make_float4((float)(scale * s0), (float)(scale * s1), (float)(scale * s2), (float)(scale * s3));
  }
}

// G[r][c] = G[c][r] for c > r: the strict upper triangle is the transpose of the lower one (exact symmetry).
__global__ void __launch_bounds__(256) tc_mirror_kernel(float* __restrict__ G, int64_t ldg, int Q) {
  __shared__ float tile[32][33];
  const int bx = blockIdx.x, by = blockIdx.y;   // block (by, bx) of 32 x 32, processed only when bx >= by
  if (bx < by) return;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;   // 32 x 8
  for (int i = ty; i < 32; i += 8) {
    const int r = bx * 32 + i, c = by * 32 + tx;
    tile[i][tx] = (r < Q && c < Q) ? G[(int64_t)r * ldg + c] : 0.f;
  }
  __syncthreads();
  for (int i = ty; i < 32; i += 8) {
    const int r = by * 32 + i, c = bx * 32 + tx;   // upper block element (r, c) = lower (c, r)
    if (r < Q && c < Q && c > r) G[(int64_t)r * ldg + c] = tile[tx][i];
  }
}

// =====================================================================================================
// Row GEMM:  D(256 rows x 256 cols per pair) = sum_k [A1 | A2][row, k] * B[k, col]
//   pass 2  : A1 = V, B = W            epilogue  Xb = (X - D) * inv_vn, row quad partials, sum Xb^2
//   Vb      : A1 = V, A2 = Xb, B = [r L Binv ; -W^T]   epilogue  out = D
//   generic : out = alpha * (X - A M)
// =====================================================================================================
struct RowsParams {
  int64_t n;
  int K1, K2;          // contraction lengths of A1 and A2 (K2 may be 0)
  int ncols;           // columns of B / of the output
  int col_tiles;       // ceil(ncols / 256)
  int64_t row_tiles;   // ceil(n / 256)
  // epilogue
  int mode;            // 0: out = alpha * (X - D) (+ quad / xb2 partials when quad_part != nullptr); 1: out = alpha * D
  // batched blocks of larger matrices (Q-space solves): batch b reads A rows from a_row0 + b a_row_step and A columns
  // (= k) from a_k0 + b a_k_step, B rows (= k) from b_k0 + b b_k_step and B columns from b_col0 + b b_col_step, and
  // writes out + b out_step; the last batch has n_last (<= n) rows.  tri_a: A[row, k] = 0 for k > row (stop the
  // contraction at the row tile's end); tri_b: B[k, col] = 0 for k < col (start it at the column tile's start).
  int batches, a_row0, a_row_step, a_k0, a_k_step, b_k0, b_k_step, b_col0, b_col_step, tri_a, tri_b;
  int lower_only;      // square output: only the tiles on and below the block diagonal (symmetric rank-k updates)
  int64_t out_step, n_last;
  const uint32_t* amax;   // device: [0] bits of max|A1|, [1] bits of max|B|, [2] bits of max|A2| (fp16 scales); may be null
  const float* X; int64_t ldx;
  float* out; int64_t ldo;
  const double* scal;  // mode 0: alpha = 1 / scal[VN] when set, else alpha_host
  float alpha_host;
  float* quad_part;    // [col_tiles * 2][n]
  double* xb2_part;    // [units * 16]
};

struct RowsUnit {
  int batch, ct, k_begin, k_end;   // stage range [k_begin, k_end) of this unit
  int64_t rt;
};
__device__ __forceinline__ RowsUnit rows_unit(const RowsParams& p, int64_t u, int nst) {
  RowsUnit r;
  const int64_t per = p.lower_only ? p.row_tiles * (p.row_tiles + 1) / 2 : p.row_tiles * p.col_tiles;
  r.batch = (int)(u / per);
  const int64_t v = u - (int64_t)r.batch * per;
  if (p.lower_only) {
    int64_t t = (int64_t)((sqrtf(8.f * (float)v + 1.f) - 1.f) * 0.5f);
    while ((t + 1) * (t + 2) / 2 <= v) ++t;
    while (t * (t + 1) / 2 > v) --t;
    r.rt = t;
    r.ct = (int)(v - t * (t + 1) / 2);
  } else {
    r.rt = v / p.col_tiles;
    r.ct = (int)(v - r.rt * p.col_tiles);
  }
  r.k_begin = p.tri_b ? r.ct * (TN / TBK) : 0;
  r.k_end = p.tri_a ? min(nst, (int)(r.rt + 1) * (TM / TBK)) : nst;
  return r;
}

// one scale set per launch: the [A1 | A2] parts share the accumulator, hence the common scale (larger magnitude wins)
template <bool F16>
__device__ __forceinline__ F16Scales rows_scales(const RowsParams& p) {
  int eA = exp_of_bits(p.amax);
  if (p.K2 > 0 && p.amax) eA = max(eA, exp_of_bits(p.amax + 2));
  return make_scales<F16>(eA, exp_of_bits(p.amax ? p.amax + 1 : nullptr));
}

template <bool F16>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kTcThreads, 1)
tc_rows_kernel(const __grid_constant__ CUtensorMap tmA1, const __grid_constant__ CUtensorMap tmA2,
               const __grid_constant__ CUtensorMap tmB, RowsParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;
  uint32_t tmem;
  TcShared* sm = tc_prologue<F16>(base, tmem);
  const int64_t nunits = (p.lower_only ? p.row_tiles * (p.row_tiles + 1) / 2 : p.row_tiles * p.col_tiles) * p.batches;
  const int nst1 = (p.K1 + TBK - 1) / TBK, nst2 = (p.K2 + TBK - 1) / TBK;
  const int nst = nst1 + nst2;

  if (warp < 4) {
    setmaxnreg_dec<80>();
    if (warp >= 2) {
      const uint32_t conv0 = mapa_u32(&sm->conv[0], 0);
      const F16Scales sc = rows_scales<F16>(p);
      PROF_DECL;
      uint32_t it = 0;
      for (int64_t u = pair; u < nunits; u += npairs) {
        const RowsUnit un = rows_unit(p, u, nst);
        for (int st = un.k_begin; st < un.k_end; ++st, ++it) convert_b_stage<F16>(base, sm, conv0, it, sc, pw0, pw1);
      }
      if (threadIdx.x == 64) PROF_STORE(4);
    } else if (warp == 0 && lane == 0) {
      PROF_DECL;
      tma_prefetch_desc(&tmA1);
      tma_prefetch_desc(&tmA2);
      tma_prefetch_desc(&tmB);
      uint32_t it = 0;
      for (int64_t u = pair; u < nunits; u += npairs) {
        const RowsUnit un = rows_unit(p, u, nst);
        const int row = p.a_row0 + un.batch * p.a_row_step + (int)(un.rt * TM) + (int)rank * HM;
        const int bcol = p.b_col0 + un.batch * p.b_col_step + un.ct * TN + (int)rank * HN;
        const int ak0 = p.a_k0 + un.batch * p.a_k_step, bk0 = p.b_k0 + un.batch * p.b_k_step;
        for (int st = un.k_begin; st < un.k_end; ++st, ++it) {
          const int s = it % kRaw;
          PROF_WAIT(pw0, mbar_wait(&sm->empty[s], ((it / kRaw) & 1) ^ 1));
          uint8_t* dst = base + s * kRawBytes;
          mbar_arrive_expect_tx(&sm->full[s], kRawBytes);
          int kb;   // row of B where this k-block starts
          if (st < nst1) {
            tma_load_2d(dst, &tmA1, ak0 + st * TBK, row, &sm->full[s]);
            kb = bk0 + st * TBK;
          } else {
            tma_load_2d(dst, &tmA2, (st - nst1) * TBK, row, &sm->full[s]);
            kb = p.K1 + (st - nst1) * TBK;
          }
#pragma unroll
          for (int g = 0; g < HN / 32; ++g)
            tma_load_2d(dst + kABytes + g * (TBK * 128), &tmB, bcol + g * 32, kb, &sm->full[s]);
        }
      }
      PROF_STORE(0);
    } else if (warp == 1 && lane == 0 && rank == 0) {
      PROF_DECL;
      uint32_t it = 0, wc = 0;
      for (int64_t u = pair; u < nunits; u += npairs) {
        const RowsUnit un = rows_unit(p, u, nst);
        const int ust = un.k_end - un.k_begin;
        const int ngroups = (ust + kGroup - 1) / kGroup;
        for (int g = 0; g < ngroups; ++g) {
          const int gst = min(kGroup, ust - g * kGroup);
          issue_group<F16>(base, sm, tmem, it, gst, g, ngroups, wc, pw0, pw1);
          it += gst;
        }
      }
      PROF_STORE(1);
    }
  } else if (warp < 8) {
    setmaxnreg_dec<80>();
    PROF_DECL;
    const uint32_t conv0 = mapa_u32(&sm->conv[0], 0);
    uint32_t it = 0;
    const F16Scales sc = rows_scales<F16>(p);
    for (int64_t u = pair; u < nunits; u += npairs) {
      const RowsUnit un = rows_unit(p, u, nst);
      for (int st = un.k_begin; st < un.k_end; ++st, ++it) convert_a_stage<false, F16>(base, sm, tmem, conv0, it, sc, pw0, pw1);
    }
    if (threadIdx.x == 128) PROF_STORE(2);
  } else {
    setmaxnreg_inc<176>();
    PROF_DECL;
    const uint32_t tempty0 = mapa_u32(&sm->tempty[0], 0);
    const int q = warp & 3, cb = (warp - 8) >> 2;
    uint32_t wc = 0;
    float alpha = p.alpha_host;
    if (p.mode == 0 && p.scal) alpha = (float)(1.0 / p.scal[GPP_S_VN]);
    const float os = rows_scales<F16>(p).out;
    for (int64_t u = pair; u < nunits; u += npairs) {
      const RowsUnit un = rows_unit(p, u, nst);
      const int64_t rt = un.rt;
      const int ct = un.ct;
      const int ust = un.k_end - un.k_begin;
      const int ngroups = (ust + kGroup - 1) / kGroup;
      float acc[128];
#pragma unroll
      for (int i = 0; i < 128; ++i) acc[i] = 0.f;
      for (int g = 0; g < ngroups; ++g) drain_group(sm, tmem, tempty0, g, ngroups, wc, acc, pw0);
#pragma unroll
      for (int i = 0; i < 128; ++i) acc[i] *= os;   // undo the common power-of-two scale of the split (exact)
      // ---- epilogue for this unit: this CTA's 128 rows, this warp's 128 columns
      const int64_t row = rt * TM + rank * HM + q * 32 + lane;
      const int col0 = ct * TN + cb * 128;
      float xb2 = 0.f;
      if (row < (un.batch == p.batches - 1 ? p.n_last : p.n)) {
        if (p.mode == 0) {
          float quad = 0.f;
          const float* xr = p.X + row * p.ldx + col0;
          float* orow = p.out + row * p.ldo + col0;
          // X and out may be the same matrix (the Cholesky's in-place rank-k update), so the compiler keeps every load
          // behind the previous store: read X in batches of 8 x 128 bit, all loads of a batch before its first store
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
                o.x = (x.x - acc[i + 0]) * alpha;
                o.y = (x.y - acc[i + 1]) * alpha;
                o.z = (x.z - acc[i + 2]) * alpha;
                o.w = (x.w - acc[i + 3]) * alpha;
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
          float* orow = p.out + un.batch * p.out_step + row * p.ldo + col0;
#pragma unroll
          for (int i = 0; i < 128; i += 4)
            if (col0 + i < p.ncols)
              *reinterpret_cast<float4*>(orow + i) =
                  make_float4(alpha * acc[i], alpha * acc[i + 1], alpha * acc[i + 2], alpha * acc[i + 3]);
        }
      }
      if (p.mode == 0 && p.xb2_part) {
        const float s = warp_sum(xb2);
        if (lane == 0) p.xb2_part[u * 16 + rank * 8 + (warp - 8)] = (double)s;
      }
    }
    if (threadIdx.x == 256) PROF_STORE(3);
  }
  tc_epilogue(tmem);
}

// Bstk (Q + L rows, Q cols) = [ (v0/vn) L_true Binv ; -W^T ]
__global__ void __launch_bounds__(256) build_bstk_kernel(const float* __restrict__ Binv, const float* __restrict__ W,
                                                         int64_t ldw, const double* __restrict__ scal, int Q, int L,
                                                         int L_true, float* __restrict__ Bstk) {
  const float coef = (float)(scal[GPP_S_V0] / scal[GPP_S_VN] * (double)L_true);
  const int64_t total = (int64_t)(Q + L) * Q;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int r = (int)(e / Q), c = (int)(e - (int64_t)r * Q);
    Bstk[e] = r < Q ? coef * Binv[(int64_t)r * Q + c] : -W[(int64_t)c * ldw + (r - Q)];
  }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(ptr);
  }
  return fn;
}

// 2-D row-major matrix (rows x cols, leading dimension ld elements), box = {box_cols elements, box_rows rows}.
int make_map_2d_any(CUtensorMap* m, const void* ptr, int elem_bytes, int64_t rows, int64_t cols, int64_t ld, int box_cols,
                    int box_rows, CUtensorMapSwizzle swz) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) {
    set_error("cuTensorMapEncodeTiled is not available from this driver");
    return GPP_ERR_CUDA;
  }
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)(rows > 0 ? rows : 1)};
  cuuint64_t strides[1] = {(cuuint64_t)ld * (cuuint64_t)elem_bytes};
  cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
  cuuint32_t es[2] = {1, 1};
  CUresult r = fn(m, elem_bytes == 2 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2,
                  const_cast<void*>(ptr), dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE, swz,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed with CUresult %d (rows=%lld cols=%lld ld=%lld elem=%d)", (int)r,
              (long long)rows, (long long)cols, (long long)ld, elem_bytes);
    return GPP_ERR_CUDA;
  }
  return GPP_OK;
}
int make_map_2d(CUtensorMap* m, const float* ptr, int64_t rows, int64_t cols, int64_t ld, int box_cols, int box_rows,
                CUtensorMapSwizzle swz) {
  return make_map_2d_any(m, ptr, 4, rows, cols, ld, box_cols, box_rows, swz);
}

// Record the bit pattern of max|X| over ALL of X in *slot (zeroed here); the kernels derive the power-of-two scales of
// the fp16 operands from it.  The scan is exact (one streaming read, cheap next to the GEMM it feeds): an operand scaled
// from a sampled maximum would silently saturate on an outlier row the sample missed.
// zero_slot = false: fold X into what *slot already holds (one scale shared by several matrices).
int launch_absmax(const float* X, int64_t ld, int64_t rows, int cols, uint32_t* slot, cudaStream_t st,
                  bool zero_slot = true) {
  if (zero_slot) GPP_CUDA(cudaMemsetAsync(slot, 0, 4, st));
  if (rows <= 0 || cols < 4) return GPP_OK;
  const int64_t want = ceil_div(rows * (int64_t)cols, 256 * 4 * 8);   // >= 8 float4 per thread
  const int cap = 8 * sm_count();                                      // one wave of 256-thread CTAs
  const int grid = (int)(want < 1 ? 1 : (want < cap ? want : cap));
  absmax_bits_kernel<<<grid, 256, 0, st>>>(X, ld, rows, cols, slot);
  GPP_LAUNCH_CHECK();
  return GPP_OK;
}

// CTA pairs that can be co-resident (persistent grid = 2 x this); B200: 148 SMs -> up to 74 pairs.
template <typename K>
int pair_count(K kernel) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(2 * (unsigned)sm_count());
  cfg.blockDim = dim3(kTcThreads);
  cfg.dynamicSmemBytes = kSmemBytes;
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

// per-device caches (a second device in the process needs its own cudaFuncSetAttribute and occupancy query)
constexpr int kMaxDevices = 64;
int current_device() {
  int dev = 0;
  cudaGetDevice(&dev);
  return dev < 0 || dev >= kMaxDevices ? 0 : dev;
}
std::mutex g_attr_mutex;
int pass1_pairs() {
  static int n[kMaxDevices] = {0};
  const int dev = current_device();
  std::lock_guard<std::mutex> lock(g_attr_mutex);
  if (n[dev] == 0) {
    cudaFuncSetAttribute(tc_pass1_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes);
    cudaFuncSetAttribute(tc_pass1_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes);
    n[dev] = pair_count(tc_pass1_kernel<true>);
  }
  return n[dev];
}
int rows_pairs() {
  static int n[kMaxDevices] = {0};
  const int dev = current_device();
  std::lock_guard<std::mutex> lock(g_attr_mutex);
  if (n[dev] == 0) {
    cudaFuncSetAttribute(tc_rows_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes);
    cudaFuncSetAttribute(tc_rows_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes);
    n[dev] = pair_count(tc_rows_kernel<true>);
  }
  return n[dev];
}

}  // namespace

void pass1_geometry(int64_t n, int Q, int L, bool skip_g, int pairs, int kblock, Pass1Params& p) {
  p.n = n; p.Q = Q; p.L = L;
  p.tm_count = (int)ceil_div(Q, TM);
  p.tiles_g = skip_g ? 0 : p.tm_count * (p.tm_count + 1) / 2;
  p.tn_c = (int)ceil_div(L, TN);
  p.tiles = p.tiles_g + p.tm_count * p.tn_c;
  // choose the split count on the persistent grid of CTA pairs (>= 512 rows per split, <= 1 GB of partial tiles): the
  // smallest estimated time  units-per-pair x (rows per split + kUnitOverheadRows).  A unit ends with the drain of its
  // accumulator and a 256 KB partial tile (and the reduction reads it back): 10-23 us, the time of ~1000 rows, measured at
  // n = 125k, Q = 4096 (experiments/bench/shard_stages.py: V^T Z, 16 tiles, 0.80 ms as 37 splits of 3392 rows -- what pure
  // wave efficiency picks -- against 0.64 ms as 4 splits; the 136 Gram tiles 4.51 ms at 7 splits, 4.6-4.9 ms at 1, 2, 14, 28).
  constexpr int64_t kUnitOverheadRows = 1024;
  const int64_t max_by_rows = n / 512 > 1 ? n / 512 : 1;
  const int64_t max_by_ws = (int64_t)(1024ll << 20) / ((int64_t)(p.tiles > 0 ? p.tiles : 1) * TM * TN * 4);
  int64_t smax = max_by_rows < max_by_ws ? max_by_rows : max_by_ws;
  if (smax < 1) smax = 1;
  if (smax > 2 * pairs) smax = 2 * pairs;
  int best = 1;
  int64_t best_cost = -1;
  for (int s = 1; s <= smax; ++s) {
    const int64_t rps = ceil_div(ceil_div(n > 0 ? n : 1, s), kblock) * kblock;
    const int64_t units = (int64_t)p.tiles * ceil_div(n > 0 ? n : 1, rps);
    const int64_t cost = ceil_div(units, pairs) * (rps + kUnitOverheadRows);
    if (best_cost < 0 || cost < best_cost) {   // ties: fewer splits
      best_cost = cost;
      best = s;
    }
  }
  if (const char* e = getenv("GPP_TC_SPLIT_ROWS")) {   // experiment knob: target rows per split
    const long long r = atoll(e);
    if (r >= 512) best = (int)ceil_div(n > 0 ? n : 1, r);
  }
  p.rows_per_split = ceil_div(ceil_div(n > 0 ? n : 1, best), kblock) * kblock;
  p.splits = (int)ceil_div(n > 0 ? n : 1, p.rows_per_split);
}

int launch_pass1_reduce(const Pass1Params& p, cudaStream_t st) {
  if (p.tiles == 0) return GPP_OK;
  tc_reduce_kernel<<<p.tiles * 8, 256, 0, st>>>(p);
  GPP_LAUNCH_CHECK();
  if (p.tiles_g > 0 && p.G) {
    dim3 mg((unsigned)ceil_div(p.Q, 32), (unsigned)ceil_div(p.Q, 32));
    tc_mirror_kernel<<<mg, 256, 0, st>>>(p.G, p.ldg, p.Q);
    GPP_LAUNCH_CHECK();
  }
  return GPP_OK;
}

int make_tensor_map_2d(CUtensorMap* m, const void* ptr, int elem_bytes, int64_t rows, int64_t cols, int64_t ld_elems,
                       int box_cols, int box_rows, CUtensorMapSwizzle swz) {
  return make_map_2d_any(m, ptr, elem_bytes, rows, cols, ld_elems, box_cols, box_rows, swz);
}

bool tc_available() { return encode_fn() != nullptr; }

#ifdef GPP_TC_PROF
extern "C" int gpp_debug_prof(unsigned long long* out /* [512][16] */) {
  return cudaMemcpyFromSymbol(out, g_prof, sizeof(g_prof)) == cudaSuccess ? 0 : -1;
}
#endif

int tc_absmax(const float* X, int64_t ld, int64_t rows, int cols, uint32_t* slot, cudaStream_t st) {
  return launch_absmax(X, ld, rows, cols, slot, st);
}

int tc_absmax_fold(const float* X, int64_t ld, int64_t rows, int cols, uint32_t* slot, cudaStream_t st) {
  return launch_absmax(X, ld, rows, cols, slot, st, false);
}

bool tc_pass1_supported(int64_t n, int Q, int L) { return Q >= 128 && n >= 512 && encode_fn() != nullptr; }

size_t tc_pass1_workspace_bytes(int64_t n, int Q, int L, bool skip_g) {
  Pass1Params p;
  pass1_geometry(n, Q, L, skip_g, pass1_pairs(), TBK, p);
  return (size_t)p.tiles * p.splits * TM * TN * sizeof(float) + 256 /* absmax slots */;
}

// G (Q x Q, optional) = V^T V and C (Q x L) = V^T X [* v0/vn when scal_c is set]; G == nullptr skips the Gram tiles.
int launch_tc_pass1(const float* V, int64_t ldv, const float* X, int64_t ldx, int64_t n, int Q, int L, float* G,
                    int64_t ldg, float* C, int64_t ldc, const double* scal_c, void* ws, size_t ws_bytes,
                    bool wide_range, cudaStream_t st) {
  Pass1Params p{};
  pass1_geometry(n, Q, L, G == nullptr, pass1_pairs(), TBK, p);
  const size_t part_bytes = (size_t)p.tiles * p.splits * TM * TN * sizeof(float), need = part_bytes + 256;
  if (!ws || ws_bytes < need) {
    set_error("gram_vtz (tcgen05): workspace too small (%zu < %zu bytes)", ws_bytes, need);
    return GPP_ERR_WORKSPACE;
  }
  if (p.tiles == 0) return GPP_OK;
  p.partial = static_cast<float*>(ws);
  uint32_t* amax = reinterpret_cast<uint32_t*>(static_cast<char*>(ws) + part_bytes);
  GPP_TRY(launch_absmax(V, ldv, n, Q, amax, st));
  if (L > 0) GPP_TRY(launch_absmax(X, ldx, n, L, amax + 1, st));
  p.amax = amax;
  p.wave_ctr = reinterpret_cast<unsigned int*>(amax + 8);
  if (const char* e = getenv("GPP_TC_WAVE_SYNC")) {   // experiment knob: 0 switches the wave alignment off
    if (e[0] == '0') p.wave_ctr = nullptr;
  }
  if (p.wave_ctr) GPP_CUDA(cudaMemsetAsync(p.wave_ctr, 0, 4, st));
  p.G = G; p.ldg = ldg; p.C = C; p.ldc = ldc; p.scal_c = scal_c;
  CUtensorMap tmV, tmX;
  GPP_TRY(make_map_2d(&tmV, V, n, Q, ldv, 32, TBK, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B));
  if (L > 0) GPP_TRY(make_map_2d(&tmX, X, n, L, ldx, 32, TBK, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B));
  else tmX = tmV;
  const int nunits = p.tiles * p.splits;
  const int pairs = nunits < pass1_pairs() ? nunits : pass1_pairs();
  if (wide_range) tc_pass1_kernel<false><<<2 * pairs, kTcThreads, kSmemBytes, st>>>(tmV, tmX, p);
  else tc_pass1_kernel<true><<<2 * pairs, kTcThreads, kSmemBytes, st>>>(tmV, tmX, p);
  GPP_LAUNCH_CHECK();
  return launch_pass1_reduce(p, st);
}

bool tc_rows_supported(int64_t n, int K, int ncols) { return n >= 512 && K >= 64 && ncols >= 64 && encode_fn() != nullptr; }

size_t tc_xb_workspace_bytes(int64_t n, int L) {
  const int64_t col_tiles = ceil_div(L, TN), row_tiles = ceil_div(n, TM);
  return align_up((size_t)col_tiles * 2 * n * sizeof(float), 256) +
         align_up((size_t)row_tiles * col_tiles * 16 * sizeof(double), 256) + align_up(xb_finalize_bytes(), 256) +
         256 /* absmax slots */;
}

static int launch_rows_maps(const CUtensorMap& tmA1, const CUtensorMap& tmA2, const CUtensorMap& tmB, int64_t n,
                            int K1, int K2, int ncols, RowsParams& p, bool wide_range, cudaStream_t st) {
  p.n = n; p.K1 = K1; p.K2 = K2; p.ncols = ncols;
  if (p.batches <= 0) p.batches = 1;
  if (p.n_last <= 0) p.n_last = n;
  p.col_tiles = (int)ceil_div(ncols, TN);
  p.row_tiles = ceil_div(n, TM);
  const int64_t nunits = (p.lower_only ? p.row_tiles * (p.row_tiles + 1) / 2 : p.row_tiles * p.col_tiles) * p.batches;
  const int pairs = (int)(nunits < rows_pairs() ? nunits : rows_pairs());
  if (pairs <= 0) return GPP_OK;
  if (wide_range) tc_rows_kernel<false><<<2 * pairs, kTcThreads, kSmemBytes, st>>>(tmA1, tmA2, tmB, p);
  else tc_rows_kernel<true><<<2 * pairs, kTcThreads, kSmemBytes, st>>>(tmA1, tmA2, tmB, p);
  GPP_LAUNCH_CHECK();
  return GPP_OK;
}

static int launch_rows(const float* A1, int64_t lda1, int K1, const float* A2, int64_t lda2, int K2, const float* B,
                       int64_t ldb, int64_t n, int ncols, RowsParams& p, uint32_t* amax, cudaStream_t st) {
  if (amax) {
    GPP_TRY(launch_absmax(A1, lda1, n, K1, amax, st));
    GPP_TRY(launch_absmax(B, ldb, (int64_t)K1 + K2, ncols, amax + 1, st));
    if (K2 > 0) GPP_TRY(launch_absmax(A2, lda2, n, K2, amax + 2, st));
    p.amax = amax;
  }
  CUtensorMap tmA1, tmA2, tmB;
  GPP_TRY(make_map_2d(&tmA1, A1, n, K1, lda1, TBK, HM, CU_TENSOR_MAP_SWIZZLE_64B));
  if (K2 > 0) GPP_TRY(make_map_2d(&tmA2, A2, n, K2, lda2, TBK, HM, CU_TENSOR_MAP_SWIZZLE_64B));
  else tmA2 = tmA1;
  GPP_TRY(make_map_2d(&tmB, B, (int64_t)K1 + K2, ncols, ldb, 32, TBK, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B));
  return launch_rows_maps(tmA1, tmA2, tmB, n, K1, K2, ncols, p, false, st);
}

// Batched block GEMM inside larger row-major matrices (the Q-space solves):
//   out_b (n x ncols) = alpha * A_b (n x K) . B_b (K x ncols),  b < g.batches,
// A_b = Amat[a_row0 + b a_row_step .., a_k0 + b a_k_step ..], B_b = Bmat[b_k0 + b b_k_step .., b_col0 + b b_col_step ..],
// out_b = out + b out_step.  Reads outside a block but inside its matrix only feed outputs that are not stored; reads
// outside the matrix are zero (TMA), which is what the ragged last batch (n_last rows, at the matrix edge) relies on.
bool tc_blockgemm_supported(int n, int K, int ncols) { return n >= 512 && K >= 64 && ncols >= 64 && encode_fn() != nullptr; }

int launch_tc_blockgemm(const float* Amat, int64_t a_rows, int64_t a_cols, int64_t lda, const float* Bmat, int64_t b_rows,
                        int64_t b_cols, int64_t ldb, float* out, int64_t ldo, const TcBlockGemm& g,
                        const uint32_t* amax, cudaStream_t st) {
  CUtensorMap tmA, tmB;
  GPP_TRY(make_map_2d(&tmA, Amat, a_rows, a_cols, lda, TBK, HM, CU_TENSOR_MAP_SWIZZLE_64B));
  GPP_TRY(make_map_2d(&tmB, Bmat, b_rows, b_cols, ldb, 32, TBK, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B));
  RowsParams p{};
  p.mode = 1; p.out = out; p.ldo = ldo; p.alpha_host = g.alpha;
  p.batches = g.batches; p.n_last = g.n_last;
  p.a_row0 = g.a_row0; p.a_row_step = g.a_row_step; p.a_k0 = g.a_k0; p.a_k_step = g.a_k_step;
  p.b_k0 = g.b_k0; p.b_k_step = g.b_k_step; p.b_col0 = g.b_col0; p.b_col_step = g.b_col_step;
  p.tri_a = g.tri_a; p.tri_b = g.tri_b; p.out_step = g.out_step; p.amax = amax;
  return launch_rows_maps(tmA, tmA, tmB, g.n, g.K, 0, g.ncols, p, g.wide_range != 0, st);
}

// Symmetric rank-K update of the lower block triangle, in place:  C -= A A^T  with A (n x K, ld = lda) and its transpose
// At (K x n, ld = ldat) both given (the Cholesky's trailing update; only tiles with column tile <= row tile are touched).
int launch_tc_syrk_sub(float* C, int64_t ldc, const float* A, int64_t lda, const float* At, int64_t ldat, int n, int K,
                       const uint32_t* amax, cudaStream_t st) {
  CUtensorMap tmA, tmB;
  GPP_TRY(make_map_2d(&tmA, A, n, K, lda, TBK, HM, CU_TENSOR_MAP_SWIZZLE_64B));
  GPP_TRY(make_map_2d(&tmB, At, K, n, ldat, 32, TBK, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B));
  RowsParams p{};
  p.mode = 0; p.X = C; p.ldx = ldc; p.out = C; p.ldo = ldc; p.alpha_host = 1.f; p.lower_only = 1; p.amax = amax;
  return launch_rows_maps(tmA, tmA, tmB, n, K, 0, n, p, true, st);
}

// out = alpha (X - A M); with nll != nullptr also the NLL epilogue (quad partials -> xb_finalize).
int launch_tc_xb(const float* V, int64_t ldv, const float* X, int64_t ldx, const float* W, int64_t ldw, int64_t n,
                 int Q, int L, double* scal, float alpha_host, float* Xb, int64_t ldxb, float* nll, void* ws,
                 size_t ws_bytes, cudaStream_t st) {
  RowsParams p{};
  p.mode = 0; p.X = X; p.ldx = ldx; p.out = Xb; p.ldo = ldxb; p.scal = scal; p.alpha_host = alpha_host;
  const int64_t col_tiles = ceil_div(L, TN), row_tiles = ceil_div(n, TM);
  if (nll) {
    const size_t need = tc_xb_workspace_bytes(n, L);
    if (!ws || ws_bytes < need) {
      set_error("xb_nll (tcgen05): workspace too small (%zu < %zu bytes)", ws_bytes, need);
      return GPP_ERR_WORKSPACE;
    }
    p.quad_part = static_cast<float*>(ws);
    p.xb2_part = reinterpret_cast<double*>(static_cast<char*>(ws) + align_up((size_t)col_tiles * 2 * n * sizeof(float), 256));
  }
  // exact operand maxima (fp16 scales): the last 256 bytes of the NLL workspace, or the whole 256-byte workspace of the
  // generic X - A M form
  uint32_t* amax = nullptr;
  if (nll)
    amax = reinterpret_cast<uint32_t*>(static_cast<char*>(ws) + tc_xb_workspace_bytes(n, L) - 256);
  else if (ws && ws_bytes >= 256)
    amax = static_cast<uint32_t*>(ws);
  GPP_TRY(launch_rows(V, ldv, Q, nullptr, 0, 0, W, ldw, n, L, p, amax, st));
  if (nll) {
    double* fin = p.xb2_part + align_up((size_t)row_tiles * col_tiles * 16 * sizeof(double), 256) / sizeof(double);
    GPP_TRY(launch_xb_finalize(p.quad_part, (int)(col_tiles * 2), n, p.xb2_part, row_tiles * col_tiles * 16, fin, scal,
                               nll, st));
  }
  return GPP_OK;
}

size_t tc_vb_workspace_bytes(int Q, int L) { return align_up((size_t)(Q + L) * Q * sizeof(float), 256) + 256; }

int launch_tc_vb(const float* V, int64_t ldv, const float* Xb, int64_t ldxb, const float* Binv, const float* W,
                 int64_t ldw, const double* scal, int64_t n, int Q, int L, int L_true, float* Vb, int64_t ldvb, void* ws,
                 size_t ws_bytes, cudaStream_t st) {
  const size_t need = tc_vb_workspace_bytes(Q, L);
  if (!ws || ws_bytes < need) {
    set_error("vb (tcgen05): workspace too small (%zu < %zu bytes)", ws_bytes, need);
    return GPP_ERR_WORKSPACE;
  }
  float* Bstk = static_cast<float*>(ws);
  build_bstk_kernel<<<1024, 256, 0, st>>>(Binv, W, ldw, scal, Q, L, L_true, Bstk);
  GPP_LAUNCH_CHECK();
  RowsParams p{};
  p.mode = 1; p.out = Vb; p.ldo = ldvb; p.alpha_host = 1.f;
  uint32_t* amax = reinterpret_cast<uint32_t*>(static_cast<char*>(ws) + align_up((size_t)(Q + L) * Q * sizeof(float), 256));
  return launch_rows(V, ldv, Q, Xb, ldxb, L, Bstk, Q, n, Q, p, amax, st);
}

}  // namespace gpp
