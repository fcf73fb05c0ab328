// Q-space solve (replicated on every rank): from GC = V^T [V | X] and lvs
//   B = I + (v0/vn) G = Lc Lc^T      blocked right-looking Cholesky, 64-wide panels; the diagonal
//                                    block is factored AND inverted in shared memory / registers by
//                                    one 64-thread CTA, which turns the panel TRSM into a GEMM
//   log|B| = 2 sum log diag(Lc)      (replaces the svd of gp.py:33 through the determinant lemma)
//   Linv   = Lc^-1                   recursive-doubling triangular inverse (log2(Q/64) batched levels)
//   [Binv | W] = Linv^T [Linv | (v0/vn) Linv C]   (replaces torch.inverse of gp.py:35)
// Q is padded to Qp (multiple of 64) with an identity block, which changes neither log|B| nor W.
#include <math.h>

#include "common.cuh"
#include "gemm_simt.cuh"
#include <cstdlib>
#include <mutex>
#include "kernels.h"

namespace gpp {

constexpr int NB = 64;  // Cholesky panel width

// ------------------------------------------------------------------ scalars
__global__ void scal_init_kernel(const float* __restrict__ vs, double* __restrict__ scal) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    scal[GPP_S_V0] = (double)vs[0];
    scal[GPP_S_VN] = (double)vs[1];
  }
}

// Bm (Qp x Qp) = I + (v0/vn) G on the real Q x Q block, identity on the padding.
__global__ void __launch_bounds__(256) build_b_kernel(const float* __restrict__ G, int64_t ldg, int Q, int Qp,
                                                      const double* __restrict__ scal, float* __restrict__ Bm) {
  const float r = (float)(scal[GPP_S_V0] / scal[GPP_S_VN]);
  const int64_t total4 = (int64_t)Qp * (Qp / 4);
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total4; e += (int64_t)gridDim.x * blockDim.x) {
    const int i = (int)(e / (Qp / 4));
    const int j4 = (int)(e - (int64_t)i * (Qp / 4)) * 4;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (i < Q && j4 < Q) {  // Q % 4 == 0, so a float4 never straddles the edge
      const float4 g = *reinterpret_cast<const float4*>(G + (int64_t)i * ldg + j4);
      v = make_float4(r * g.x, r * g.y, r * g.z, r * g.w);
    }
    if (i == j4 + 0) v.x += 1.f;
    if (i == j4 + 1) v.y += 1.f;
    if (i == j4 + 2) v.z += 1.f;
    if (i == j4 + 3) v.w += 1.f;
    *reinterpret_cast<float4*>(Bm + (int64_t)i * Qp + j4) = v;
  }
}

// ------------------------------------------------------------------ diagonal block: factor / invert / panel solve
// 64 x 64 blocks live in shared memory (pitch 68) and are processed by one CTA of 256 threads:
//   panel_factor_solve : a panel CTA's [diagonal block; its own block of the panel] eliminated in one go (below)
//   invert64           : Xs <- L^-1 from the four 16 x 16 inverses and two recursive-doubling levels
//   diag_inv_kernel    : after the factorisation, all 64 x 64 diagonal inverses in one batched launch.
// (History of the panel step: v1 unrolled everything over registers -- 400 KB of straight-line code, ~50 us per panel;
//  v2 rank-1 updates in shared memory with a barrier per column -- 48 us; v3 factor + invert in one CTA -- 39 us; v4
//  (rounds 1-2) redundant 64 x 64 factor by warp 0 + blocked substitution against 16 x 16 inverses -- 23 us; v5 = this.)
constexpr int kPotfThreads = 256;
constexpr int SB = 16;
constexpr int kPitch = NB + 4;   // 68: conflict-free for "4 lanes per row" access patterns

struct Block64 {
  float a[NB][kPitch];
};

// Fused elimination of a panel CTA's stacked block [D; P] (D = the 64 x 64 diagonal block, P = this CTA's 64 x 64 block
// of the panel below it; P absent for CTA 0): on return D holds its Cholesky factor L11 (lower triangle; the strict upper
// triangle is NOT cleaned) and P holds P L11^-T.  Four 16-column sub-panels, each in two phases:
//   AB  warp-synchronous, no shared-memory traffic inside: every active warp holds the 16 x 16 diagonal sub-block in
//       lanes 0..15 (redundantly: that is what makes the phase barrier-free) and 16 further rows of the sub-panel in
//       lanes 16..31 (the rows of D below the sub-block first, then the rows of P), one row per lane in registers.  Column
//       jj: every lane fetches the pivot and the sub-block's column entries A[c][jj] with shuffles that do not depend on
//       the reciprocal square root computed meanwhile, scales its own entry and updates its row,
//       a[c] -= a[jj] A[c][jj] / piv.  ~80 cycles of dependent latency per column.
//   C   rank-16 update of everything right of the sub-panel with 4 x 4 register tiles whose rows / columns are strided
//       over the threads so that a quarter-warp reads consecutive shared-memory rows (pitch 68: conflict-free).
// (Round 2 before this: a 64 x 64 factorisation by warp 0 + substitution + rank-16 updates, 20.2 k cycles, then a blocked
// substitution for P against the four 16 x 16 inverses, 11.0 k cycles -- profiles/r02_chol_step_q4096_ncu_full.txt.)
__device__ __forceinline__ void panel_factor_solve(Block64& As, Block64& Xs, const bool has_p) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const unsigned full = 0xffffffffu;
  const int l = lane & 15;
#pragma unroll
  for (int kb = 0; kb < NB / SB; ++kb) {
    const int o = kb * SB;
    const int nd = NB / SB - 1 - kb;                 // 16-row groups of D below the diagonal sub-block
    const int ngroups = nd + (has_p ? NB / SB : 0);  // <= 7: one group per warp
    if (warp < ngroups || warp == 0) {
      float* rowp;
      if (lane < SB || warp >= ngroups) rowp = &As.a[o + l][o];             // (no group left: lanes 16.. mirror 0..15)
      else if (warp < nd)              rowp = &As.a[o + SB + SB * warp + l][o];
      else                             rowp = &Xs.a[SB * (warp - nd) + l][o];
      float d[SB];
#pragma unroll
      for (int c4 = 0; c4 < SB / 4; ++c4) {
        const float4 v = *reinterpret_cast<const float4*>(rowp + 4 * c4);
        d[4 * c4 + 0] = v.x; d[4 * c4 + 1] = v.y; d[4 * c4 + 2] = v.z; d[4 * c4 + 3] = v.w;
      }
#pragma unroll
      for (int jj = 0; jj < SB; ++jj) {
        const float piv = __shfl_sync(full, d[jj], jj);
        float colv[SB];
#pragma unroll
        for (int c = jj + 1; c < SB; ++c) colv[c] = __shfl_sync(full, d[jj], c);   // A[c][jj], before scaling
        float rinv = rsqrtf(piv);                               // MUFU estimate + one Newton step: ~1 ulp
        rinv = rinv * fmaf(-0.5f * piv * rinv, rinv, 1.5f);
        const float m = d[jj] * (rinv * rinv);                  // a[jj] / piv
        d[jj] = (lane == jj) ? piv * rinv : d[jj] * rinv;
#pragma unroll
        for (int c = jj + 1; c < SB; ++c) d[c] = fmaf(-m, colv[c], d[c]);
      }
      const bool store = lane < SB ? (warp == 0) : (warp < ngroups);
      if (store) {
#pragma unroll
        for (int c4 = 0; c4 < SB / 4; ++c4)
          *reinterpret_cast<float4*>(rowp + 4 * c4) = make_float4(d[4 * c4 + 0], d[4 * c4 + 1], d[4 * c4 + 2], d[4 * c4 + 3]);
      }
    }
    __syncthreads();
    if (kb == NB / SB - 1) break;
    // ---- phase C: rows = D rows [c0, 64) followed by the rows of P; columns [c0, 64)
    const int c0 = o + SB, ncols = NB - c0;
    const int ncx = ncols >> 2;                                 // column threads: 12, 8, 4
    const int nrows = ncols + (has_p ? NB : 0);
    const int nry = nrows >> 2;                                 // row threads
    for (int t = tid; t < ncx * nry; t += kPotfThreads) {
      const int cx = t % ncx, ry = t / ncx;
      float* rp[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int ci = ry + nry * i;
        rp[i] = ci < ncols ? &As.a[c0 + ci][0] : &Xs.a[ci - ncols][0];
      }
      float acc[4][4];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int jx = 0; jx < 4; ++jx) acc[i][jx] = 0.f;
#pragma unroll
      for (int k4 = 0; k4 < SB / 4; ++k4) {
        float4 av[4], bv[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) av[i] = *reinterpret_cast<const float4*>(rp[i] + o + 4 * k4);
#pragma unroll
        for (int jx = 0; jx < 4; ++jx) bv[jx] = *reinterpret_cast<const float4*>(&As.a[c0 + cx + ncx * jx][o + 4 * k4]);
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int jx = 0; jx < 4; ++jx) {
            acc[i][jx] = fmaf(av[i].x, bv[jx].x, acc[i][jx]);
            acc[i][jx] = fmaf(av[i].y, bv[jx].y, acc[i][jx]);
            acc[i][jx] = fmaf(av[i].z, bv[jx].z, acc[i][jx]);
            acc[i][jx] = fmaf(av[i].w, bv[jx].w, acc[i][jx]);
          }
      }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int jx = 0; jx < 4; ++jx) rp[i][c0 + cx + ncx * jx] -= acc[i][jx];
    }
    __syncthreads();
  }
}

// Xs <- As^-1 (As lower triangular, strict upper part zero).  Ts: scratch of at least 32 x 33 floats.
__device__ __forceinline__ void invert64(const Block64& As, Block64& Xs, float (*Ts)[NB / 2 + 1]) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const unsigned full = 0xffffffffu;
  for (int e = tid; e < NB * NB; e += kPotfThreads) Xs.a[e >> 6][e & 63] = 0.f;
  __syncthreads();
  if (warp < NB / SB) {   // warp w inverts diagonal sub-block w: lane l computes column l by forward substitution
    const int o = warp * SB, l = lane & 15;
    float d[SB], x[SB];
#pragma unroll
    for (int c = 0; c < SB; ++c) d[c] = As.a[o + l][o + c];   // row l of the 16 x 16 factor
#pragma unroll
    for (int i2 = 0; i2 < SB; ++i2) {
      float s = 0.f;
#pragma unroll
      for (int k = 0; k < i2; ++k) s = fmaf(__shfl_sync(full, d[k], i2), x[k], s);
      const float lii = __shfl_sync(full, d[i2], i2);
      x[i2] = ((i2 == l ? 1.f : 0.f) - s) / lii;
    }
    if (lane < SB) {
#pragma unroll
      for (int c = 0; c < SB; ++c) Xs.a[o + c][o + l] = x[c];
    }
  }
  __syncthreads();
  for (int b = SB; b < NB; b *= 2) {   // inv([[A,0],[C,D]]) = [[Ai,0],[-Di C Ai, Di]]
    const int npairs = NB / (2 * b), bb = b * b, sh = (b == SB) ? 4 : 5;
    for (int e = tid; e < npairs * bb; e += kPotfThreads) {
      const int pr = e / bb, rem = e - pr * bb, r = rem >> sh, c = rem & (b - 1), p0 = pr * 2 * b;
      float s = 0.f;
      for (int k = c; k < b; ++k) s = fmaf(As.a[p0 + b + r][p0 + k], Xs.a[p0 + k][p0 + c], s);
      Ts[pr * b + r][c] = s;
    }
    __syncthreads();
    for (int e = tid; e < npairs * bb; e += kPotfThreads) {
      const int pr = e / bb, rem = e - pr * bb, r = rem >> sh, c = rem & (b - 1), p0 = pr * 2 * b;
      float s = 0.f;
      for (int k = 0; k <= r; ++k) s = fmaf(Xs.a[p0 + b + r][p0 + b + k], Ts[pr * b + k][c], s);
      Xs.a[p0 + b + r][p0 + c] = -s;
    }
    __syncthreads();
  }
}

// One step of the blocked Cholesky with look-ahead, ONE kernel per 64-wide panel j:
//   panel CTAs (blockIdx < nb - j; CTA 0 = the diagonal block only, CTA b >= 1 = block row j + b):
//       apply the rank-64 update of panel j-1 to their own 64 x 64 blocks of column j (the diagonal block redundantly
//       in every CTA), eliminate [diagonal block; own block] (the diagonal block redundantly: it removes a launch and a
//       grid-wide dependency from the critical path), CTA 0 parks L11 in Ld, CTA b stores its rows of the panel;
//   wide CTAs (the rest) prepare LATER columns, off the critical path of this step, in one of three ways:
//     * left-looking (wide_mode 2, the default below the outer-block sizes): column block j+1 -- the one the NEXT step
//       factors -- receives ALL the panels finished so far in one product, A[i, j+1] -= L[i, 0:64j] L[j+1, 0:64j]^T, on
//       128 x 64 tiles with the contraction split into chunks; the chunks of a row tile wait for each other and each
//       sums the partial tiles, in chunk order, on its own slice of rows and applies it (deterministic).
//       Nothing right of column j+1 is touched before its turn.  Work per step (nb-j-1)*j block products: it peaks in
//       the MIDDLE of the factorisation at a quarter of the right-looking scheme's first step, and the grid is sized
//       to the SMs the panel CTAs leave free, so every CTA of the step has an SM of its own.
//     * right-looking (wide_mode 0): A[i, c] -= L[i, j-1] L[c, j-1]^T on 128 x 128 tiles of all columns >= j + 1
//       (rounds 1-2: 2.1 waves of read-modify-write tiles at step 1, 47 us against a 22 us panel chain);
//     * outer-block (wide_mode 1): right-looking inside the current 256-wide block only (see launch_factor).
// Both roles only read what earlier launches finished and write disjoint blocks.
// ---- 3xTF32 warp-MMA tile engine of the Cholesky's rank-k updates
// out(128 x 64) = A(128 x K) . B(64 x K)^T with both operands row-major, the contraction along their rows: eight warps
// as 4 x 2, a 32 x 32 tile per warp from mma.sync.m16n8k8 TF32 (measured on B200: 510 MAC / clk / SM against 125 for
// FFMA, profiles/r02_exp4_mma_sync_rate.txt).  fp32 accuracy from three MMAs per product: x = hi + lo with hi = the 19
// leading bits (what the tensor core reads), lo = x - hi (exact);  a b ~ a_lo b_hi + a_hi b_lo + a_hi b_hi.  The tensor
// core's accumulator rounds toward zero, so the large term never accumulates inside it: every hi.hi MMA starts from a
// zero accumulator and is added to the running sum in fp32 registers (round-to-nearest); only the two correction
// terms, 2^-11 of the product, chain through the MMA accumulator (Ootomo & Yokota's scheme).
// Operands sit in shared memory as [row][k] with a pitch that is 4 mod 32 floats: the fragment loads (lane = 4 g + t
// reads row g, column t) hit 32 different banks.
__device__ __forceinline__ void mma_tf32(float (&d)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}
__device__ __forceinline__ void split_tf32(float x, uint32_t& hi, uint32_t& lo) {
  hi = __float_as_uint(x) & 0xFFFFE000u;
  lo = __float_as_uint(x - __uint_as_float(hi));
}
struct MmaAcc {
  float h[2][4][4];   // sum of the hi.hi products (added in fp32 registers)
  float l[2][4][4];   // the two correction terms (chained through the MMA accumulator)
  float p[2][4][4];   // hi.hi products of the latest contraction step, not yet added to h (see mma_warp_tile)
  __device__ __forceinline__ void clear() {
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j)
#pragma unroll
        for (int e = 0; e < 4; ++e) h[i][j][e] = l[i][j][e] = p[i][j][e] = 0.f;
  }
  // fold everything into h (call once, after the last mma_warp_tile)
  __device__ __forceinline__ void finish() {
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j)
#pragma unroll
        for (int e = 0; e < 4; ++e) h[i][j][e] += p[i][j][e] + l[i][j][e];
  }
};
// One contraction step of 8 on a warp's 32 x 32 tile: 24 MMAs in three rounds of eight INDEPENDENT ones (a warp issues in
// order, and back-to-back dependent MMAs each wait out the tensor pipe's latency: the first version of this loop, which
// issued the three MMAs of a fragment one after the other and added each hi.hi product right away, ran at a third of
// the mma.sync rate).  The hi.hi products land in `c` and are added to the running sums one step LATER, by the caller.
template <int PITCH>
__device__ __forceinline__ void mma_step(const float* __restrict__ ap, const float* __restrict__ bp, int kk,
                                         float (&c)[2][4][4], float (&l)[2][4][4]) {
  uint32_t ah[2][4], al[2][4], bh[4][2], bl[4][2];
#pragma unroll
  for (int nt = 0; nt < 4; ++nt) {
    split_tf32(bp[nt * 8 * PITCH + kk], bh[nt][0], bl[nt][0]);
    split_tf32(bp[nt * 8 * PITCH + kk + 4], bh[nt][1], bl[nt][1]);
  }
#pragma unroll
  for (int mt = 0; mt < 2; ++mt) {
    split_tf32(ap[(mt * 16) * PITCH + kk], ah[mt][0], al[mt][0]);
    split_tf32(ap[(mt * 16 + 8) * PITCH + kk], ah[mt][1], al[mt][1]);
    split_tf32(ap[(mt * 16) * PITCH + kk + 4], ah[mt][2], al[mt][2]);
    split_tf32(ap[(mt * 16 + 8) * PITCH + kk + 4], ah[mt][3], al[mt][3]);
  }
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) {
#pragma unroll
      for (int e = 0; e < 4; ++e) c[mt][nt][e] = 0.f;
      mma_tf32(c[mt][nt], ah[mt], bh[nt]);
    }
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) mma_tf32(l[mt][nt], al[mt], bh[nt]);
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) mma_tf32(l[mt][nt], ah[mt], bl[nt]);
}
__device__ __forceinline__ void add_frag(float (&h)[2][4][4], const float (&c)[2][4][4]) {
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int nt = 0; nt < 4; ++nt)
#pragma unroll
      for (int e = 0; e < 4; ++e) h[mt][nt][e] += c[mt][nt][e];
}
// NK8 (even) contraction steps of 8 on a warp's 32 x 32 tile: a_rows = the warp's first A row, b_rows = its first B row
// (both at the first k of the slab), PITCH floats between rows.  (Not unrolled: unrolling all steps of a slab was measured,
// no faster and it spills.)
template <int PITCH, int NK8>
__device__ __forceinline__ void mma_warp_tile(const float* __restrict__ a_rows, const float* __restrict__ b_rows,
                                              MmaAcc& acc) {
  const int lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const float* ap = a_rows + g * PITCH + t;
  const float* bp = b_rows + g * PITCH + t;
  float c[2][4][4];
#pragma unroll 1
  for (int ks = 0; ks < NK8; ks += 2) {
    mma_step<PITCH>(ap, bp, ks * 8, c, acc.l);
    add_frag(acc.h, acc.p);          // the previous step's products: long finished
    mma_step<PITCH>(ap, bp, ks * 8 + 8, acc.p, acc.l);
    add_frag(acc.h, c);
  }
}
// element e of accumulator fragment (mt, nt) of warp (wm, wn): tile-local row / column
__device__ __forceinline__ int mma_row(int wm, int mt, int e) { return wm * 32 + mt * 16 + ((threadIdx.x & 31) >> 2) + (e >> 1) * 8; }
__device__ __forceinline__ int mma_col(int wn, int nt, int e) { return wn * 32 + nt * 8 + (threadIdx.x & 3) * 2 + (e & 1); }

constexpr int kMmaBK = 64;                 // k per shared-memory stage of the global-memory tile
constexpr int kMmaPitch = kMmaBK + 4;      // 68 = 4 mod 32
constexpr int kMmaStages = 3;
struct TileSmemMma {
  float a[kMmaStages][BM][kMmaPitch];
  float b[kMmaStages][NB][kMmaPitch];
};
__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
  const unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(s), "l"(gmem) : "memory");
}
// acc = A(128 x klen) . B(64 x klen)^T from global memory (leading dimension ld, klen a multiple of 64): cp.async ring of
// three 64-deep slabs, two in flight, ONE block barrier per slab (with 32-deep slabs and two barriers per slab a quarter
// of the kernel's stall samples sat on the barriers).  Rows of A at and beyond a_valid (64 or 128) are read from row 0
// instead: their results are garbage the caller never stores.
__device__ __forceinline__ void mma_tile_global(const float* __restrict__ A, int a_valid, const float* __restrict__ B,
                                                int64_t ld, int klen, TileSmemMma& sm, MmaAcc& acc) {
  const int tid = threadIdx.x, warp = tid >> 5, wm = warp >> 1, wn = warp & 1;
  const int nst = klen / kMmaBK;
  auto stage = [&](int buf, int k0) {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int idx = tid + i * kPotfThreads, r = idx >> 4, c4 = (idx & 15) << 2;
      cp_async16(&sm.a[buf][r][c4], A + (int64_t)(r < a_valid ? r : 0) * ld + k0 + c4);
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int idx = tid + i * kPotfThreads, r = idx >> 4, c4 = (idx & 15) << 2;
      cp_async16(&sm.b[buf][r][c4], B + (int64_t)r * ld + k0 + c4);
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
  if (nst > 0) stage(0, 0);
  if (nst > 1) stage(1, kMmaBK);
  for (int s = 0; s < nst; ++s) {
    if (s + 1 < nst)
      asm volatile("cp.async.wait_group 1;" ::: "memory");
    else
      asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncthreads();   // slab s has landed for everybody, and everybody is done with slab s - 1: its buffer is free
    if (s + 2 < nst) stage((s + 2) % kMmaStages, (s + 2) * kMmaBK);
    const int cur = s % kMmaStages;
#ifndef GPP_LL_NO_MMA   // (timing experiment: the load pipeline alone)
    mma_warp_tile<kMmaPitch, kMmaBK / 8>(&sm.a[cur][wm * 32][0], &sm.b[cur][wn * 32][0], acc);
#endif
  }
}

#ifdef GPP_CHOL_PROF
__device__ long long g_chol_prof[64][8];
#define CPROF(slot) do { if (threadIdx.x == 0 && blockIdx.x == (npanel > 1 ? 1 : 0)) { g_chol_prof[j][slot] = clock64(); \
  if ((slot) == 0) { unsigned long long gt__; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt__)); g_chol_prof[j][6] = (long long)gt__; } } } while (0)
extern "C" int gpp_debug_chol_prof(long long* out) {
  return cudaMemcpyFromSymbol(out, g_chol_prof, sizeof(g_chol_prof)) == cudaSuccess ? 0 : -1;
}
// wide role (left-looking): stamps of wide CTA 0 (slots 0..3: entry, main loop done, partial stored + counted, exit) and
// of whichever CTA reduces row tile 0 (slots 4, 5: reduction start, exit); globaltimer in ns
__device__ long long g_chol_prof_w[64][8];
#define WPROF(cond, slot) do { if (threadIdx.x == 0 && (cond)) { unsigned long long gt__; \
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt__)); g_chol_prof_w[j][slot] = (long long)gt__; \
  if ((slot) < 2) g_chol_prof_w[j][6 + (slot)] = clock64(); } } while (0)
extern "C" int gpp_debug_chol_prof_w(long long* out) {
  return cudaMemcpyFromSymbol(out, g_chol_prof_w, sizeof(g_chol_prof_w)) == cudaSuccess ? 0 : -1;
}
#else
#define CPROF(slot) do { } while (0)
#define WPROF(cond, slot) do { } while (0)
#endif

struct StepSmem {
  Block64 As, Xs, LsT, PsT;   // diagonal block, this CTA's block row, L[j, j-1]^T, L[j+b, j-1]^T
};
constexpr size_t kStepSmemBytes = sizeof(StepSmem) > sizeof(TileSmem) ? sizeof(StepSmem) : sizeof(TileSmem);
constexpr size_t kStepSmemBytesLL = sizeof(StepSmem) > sizeof(TileSmemMma) ? sizeof(StepSmem) : sizeof(TileSmemMma);
static_assert(kStepSmemBytesLL <= 227 * 1024, "left-looking tile does not fit the shared memory of an SM");

constexpr int kLLTileFloats = BM * NB;     // one partial tile of the left-looking update
constexpr int kLLMaxRowTiles = 64;         // counters per step (row tiles of 128 rows: padded Q up to 8192)
constexpr int kLLMaxParts = 256;           // wide CTAs of one left-looking step (one SM each; more than any device has)

constexpr int kOuterCholMinQ = 6144;   // padded Q from which the Cholesky uses 256-wide outer blocks + tensor-core updates

// apply_prev: panel j - 1 has not been applied to column j and beyond yet (false for the first panel of an outer block,
// whose columns received everything from the tensor-core update of the previous outer block).  wide_cols < 0: the wide
// role covers the whole trailing matrix; otherwise only its first wide_cols (<= 2) 64-column blocks, all rows -- the
// columns of the current 256-wide outer block; the rest of the matrix gets the whole outer block in one rank-256 update.
// LL selects the left-looking wide role: ll_S chunks of ll_chunk 64-wide panels per row tile, partial tiles in `part`
// (one per wide CTA), arrival counters in `counters` (one per row tile, zero on entry).  Two instantiations because the
// roles want different register budgets: the left-looking grid has one CTA per SM, the right-looking one two.
template <bool LL>
__global__ void __launch_bounds__(kPotfThreads, LL ? 1 : 2) chol_step_kernel(float* __restrict__ Bm, int Qp, int j,
                                                                 float* __restrict__ Ld, int apply_prev, int wide_cols,
                                                                 int ll_S, int ll_chunk, float* __restrict__ part,
                                                                 unsigned int* __restrict__ counters) {
  extern __shared__ __align__(16) uint8_t step_smem[];
  const int tid = threadIdx.x;
  const int nb = Qp / NB, k0 = j * NB;
  const int npanel = nb - j;
  if (LL) {
    // Programmatic dependent launch: the next step's grid may be scheduled while this one runs (its CTAs become resident
    // as SMs free up -- the register budget allows one CTA per SM, so they never share one with a running CTA -- and
    // block right here until this grid has completed and flushed): the launch latency between two steps disappears.
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");
  }
  if (LL && (int)blockIdx.x >= npanel) {
    // ------------------------------------------------------------ wide role, left-looking: column block j + 1
    TileSmemMma& sm = *reinterpret_cast<TileSmemMma*>(step_smem);
    const int widx = (int)blockIdx.x - npanel;
    const int rt = widx / ll_S, sp = widx - rt * ll_S;
    const int c0 = k0 + NB;                              // first row / column of block j + 1
    const int r0 = c0 + rt * BM;
    const int a_valid = min(BM, Qp - r0);                // 64 or 128
    const int kbeg = sp * ll_chunk * NB, kend = min(k0, (sp + 1) * ll_chunk * NB);
    const int warp = tid >> 5, wm = warp >> 1, wn = warp & 1;
    MmaAcc acc;
    acc.clear();
    WPROF(widx == 0, 0);
#ifdef GPP_LL_FAKE_A     // (timing experiment: every CTA reads the same, cache-resident rows)
    mma_tile_global(Bm + kbeg, a_valid, Bm + kbeg, Qp, kend - kbeg, sm, acc);
#else
    mma_tile_global(Bm + (int64_t)r0 * Qp + kbeg, a_valid, Bm + (int64_t)c0 * Qp + kbeg, Qp, kend - kbeg, sm, acc);
#endif
    acc.finish();
    WPROF(widx == 0, 1);
    float* Cc = Bm + (int64_t)r0 * Qp + c0;
    if (ll_S == 1) {   // the whole contraction in this CTA: apply it
#pragma unroll
      for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int r = mma_row(wm, mt, 2 * h);
          if (r >= a_valid) continue;
          float2 v[4];
#pragma unroll
          for (int nt = 0; nt < 4; ++nt) v[nt] = *reinterpret_cast<const float2*>(Cc + (int64_t)r * Qp + mma_col(wn, nt, 0));
#pragma unroll
          for (int nt = 0; nt < 4; ++nt) {
            v[nt].x -= acc.h[mt][nt][2 * h];
            v[nt].y -= acc.h[mt][nt][2 * h + 1];
            *reinterpret_cast<float2*>(Cc + (int64_t)r * Qp + mma_col(wn, nt, 0)) = v[nt];
          }
        }
      return;
    }
    // partial tile -> global; then the ll_S CTAs of the row tile wait for each other and each one sums and applies its own
    // slice of the tile's rows, the partials in chunk order (deterministic).  (First version: the last CTA to arrive
    // reduced the whole tile alone -- 2.8 us at 7 chunks, 6.6 us at 30, on the critical path of the step.)  Waiting is
    // safe: the grid has at most one CTA per SM and at most as many CTAs as SMs, and the next step's grid is only
    // scheduled once every CTA of this one is running, so every CTA waited for is resident or will be as soon as
    // unrelated kernels (which never wait for us) release their SMs; a bounded spin turns a broken assumption into a
    // trap instead of a hang.
    float* mine = part + (size_t)widx * kLLTileFloats;
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
      for (int nt = 0; nt < 4; ++nt)
#pragma unroll
        for (int h = 0; h < 2; ++h)
          __stcg(reinterpret_cast<float2*>(mine + mma_row(wm, mt, 2 * h) * NB + mma_col(wn, nt, 0)),
                 make_float2(acc.h[mt][nt][2 * h], acc.h[mt][nt][2 * h + 1]));
    __syncthreads();
    if (tid == 0) {   // one fence after the barrier covers the whole CTA's stores (fences are cumulative)
      __threadfence();
      atomicAdd(counters + rt, 1u);
      WPROF(widx == 0, 2);
      const volatile unsigned int* cnt = counters + rt;
      unsigned int spins = 0;
      while (*cnt < (unsigned int)ll_S) {
        __nanosleep(32);
        if (++spins > (1u << 20)) __trap();
      }
      __threadfence();
    }
    __syncthreads();
    WPROF(widx == 0, 4);
    {
      const int rows_per = (a_valid + ll_S - 1) / ll_S;
      const int rlo = sp * rows_per, rhi = min(a_valid, rlo + rows_per);
      const int tx = tid & 15, ty = tid >> 4;
      const float* p0 = part + (size_t)(rt * ll_S) * kLLTileFloats + tx * 4;
      for (int r = rlo + ty; r < rhi; r += 16) {
        float* dst = Cc + (int64_t)r * Qp + tx * 4;
        const float4 v = *reinterpret_cast<const float4*>(dst);
        float4 sum = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int q0 = 0; q0 < ll_S; q0 += 8) {   // eight partial rows in flight per round trip, summed in chunk order
          float4 t[8];
#pragma unroll
          for (int u = 0; u < 8; ++u)
            t[u] = q0 + u < ll_S ? __ldcg(reinterpret_cast<const float4*>(p0 + (size_t)(q0 + u) * kLLTileFloats + r * NB))
                                 : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            sum.x += t[u].x; sum.y += t[u].y; sum.z += t[u].z; sum.w += t[u].w;
          }
        }
        *reinterpret_cast<float4*>(dst) = make_float4(v.x - sum.x, v.y - sum.y, v.z - sum.z, v.w - sum.w);
      }
    }
    WPROF(widx == 0, 5);
    return;
  }
  if (!LL && (int)blockIdx.x >= npanel) {
    // ------------------------------------------------------------ wide role: trailing update of panel j - 1
    TileSmem& sm = *reinterpret_cast<TileSmem*>(step_smem);
    const int widx = (int)blockIdx.x - npanel;
    int ti, tc;
    if (wide_cols < 0) {
      ti = (int)((sqrtf(8.f * (float)widx + 1.f) - 1.f) * 0.5f);
      while ((ti + 1) * (ti + 2) / 2 <= widx) ++ti;
      while (ti * (ti + 1) / 2 > widx) --ti;
      tc = widx - ti * (ti + 1) / 2;
    } else {
      ti = widx;
      tc = 0;
    }
    const int t0 = k0 + NB;
    const int r0 = t0 + ti * BM, c0 = t0 + tc * BN;
    Operand A, B;
    A.base = Bm + (int64_t)r0 * Qp + (k0 - NB); A.ld = Qp; A.mn_valid = min(BM, Qp - r0);
    B.base = Bm + (int64_t)c0 * Qp + (k0 - NB); B.ld = Qp; B.mn_valid = min(BN, Qp - c0);
    if (wide_cols >= 0) B.mn_valid = min(B.mn_valid, wide_cols * NB);
    float acc[8][8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int jj = 0; jj < 8; ++jj) acc[i][jj] = 0.f;
    // the output tile comes from L2 / HBM: ask for it now, behind the main loop
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int r = acc_row(i);
      if (r >= A.mn_valid) continue;
#pragma unroll
      for (int jj = 0; jj < 2; ++jj) {
        const int c = acc_col(jj * 4);
        if (c < B.mn_valid)
          asm volatile("prefetch.global.L2 [%0];" ::"l"(Bm + (int64_t)(r0 + r) * Qp + c0 + c));
      }
    }
    tile_mainloop<false, false>(A, B, NB, sm, acc);
    // read-modify-write of the tile in two batches of 8 x 128 bit: all loads of a batch before its first store (one
    // exposed round trip per batch; load -> subtract -> store row by row was sixteen of them -- ncu: 34 % of the kernel's
    // stall samples sat on these subtractions, profiles/r02_chol_step_q4096_ncu_full.txt)
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      float4 v[4][2];
#pragma unroll
      for (int ii = 0; ii < 4; ++ii) {
        const int r = acc_row(4 * h + ii);
#pragma unroll
        for (int jj = 0; jj < 2; ++jj) {
          const int c = acc_col(jj * 4);
          v[ii][jj] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (r < A.mn_valid && c < B.mn_valid)   // mn_valid is a multiple of 64, so a float4 never straddles the edge
            v[ii][jj] = *reinterpret_cast<const float4*>(Bm + (int64_t)(r0 + r) * Qp + c0 + c);
        }
      }
#pragma unroll
      for (int ii = 0; ii < 4; ++ii) {
        const int i = 4 * h + ii, r = acc_row(i);
#pragma unroll
        for (int jj = 0; jj < 2; ++jj) {
          const int c = acc_col(jj * 4);
          if (r < A.mn_valid && c < B.mn_valid) {
            float4 o = v[ii][jj];
            o.x -= acc[i][jj * 4 + 0]; o.y -= acc[i][jj * 4 + 1]; o.z -= acc[i][jj * 4 + 2]; o.w -= acc[i][jj * 4 + 3];
            *reinterpret_cast<float4*>(Bm + (int64_t)(r0 + r) * Qp + c0 + c) = o;
          }
        }
      }
    }
    return;
  }
  // -------------------------------------------------------------- panel role
  CPROF(0);
  StepSmem& S = *reinterpret_cast<StepSmem*>(step_smem);
  const int b = (int)blockIdx.x;
  const float* D = Bm + (int64_t)k0 * (Qp + 1);
  float* P = Bm + (int64_t)(k0 + b * NB) * Qp + k0;   // block (j + b, j); unused for b == 0
  // all global loads of this CTA (up to four 64 x 64 blocks) are issued before the first shared-memory store, as
  // 128-bit loads: one L2 round trip instead of sixteen
  {
    const int lr = tid >> 4, lc = (tid & 15) * 4;   // 16 rows x 16 float4 per pass, 4 passes per block
    const float* Lj = D - NB;
    const float* Lp = P - NB;
    float4 vd[4], vp[4], vl[4], vq[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int64_t off = (int64_t)(lr + 16 * i) * Qp + lc;
      vd[i] = *reinterpret_cast<const float4*>(D + off);
      if (b > 0) vp[i] = *reinterpret_cast<const float4*>(P + off);
      if (apply_prev) {
        vl[i] = *reinterpret_cast<const float4*>(Lj + off);
        if (b > 0) vq[i] = *reinterpret_cast<const float4*>(Lp + off);
      }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int r = lr + 16 * i;
      *reinterpret_cast<float4*>(&S.As.a[r][lc]) = vd[i];
      if (b > 0) *reinterpret_cast<float4*>(&S.Xs.a[r][lc]) = vp[i];
      if (apply_prev) {   // rank-64 update operands, row-major like everything else (pitch 68 = 4 mod 32)
        *reinterpret_cast<float4*>(&S.LsT.a[r][lc]) = vl[i];
        if (b > 0) *reinterpret_cast<float4*>(&S.PsT.a[r][lc]) = vq[i];
      }
    }
  }
  if (apply_prev) {
    // rank-64 update from panel j - 1 on the tensor cores (3xTF32):  [D; P] -= [Lj; Lp] Lj^T, a 128 x 64 x 64 product;
    // warps 0..3 own D, warps 4..7 own P (idle in CTA 0)
    __syncthreads();
    CPROF(1);
    const int warp = tid >> 5, wm = warp >> 1, wn = warp & 1;
    if (b > 0 || wm < 2) {
      MmaAcc acc;
      acc.clear();
      const Block64& Asrc = wm < 2 ? S.LsT : S.PsT;
      Block64& Cdst = wm < 2 ? S.As : S.Xs;
      const int rb = (wm & 1) * 32;
      mma_warp_tile<kPitch, NB / 8>(&Asrc.a[rb][0], &S.LsT.a[wn * 32][0], acc);
      acc.finish();
#pragma unroll
      for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int nt = 0; nt < 4; ++nt)
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            float2* dst = reinterpret_cast<float2*>(&Cdst.a[mma_row(wm & 1, mt, 2 * h)][mma_col(wn, nt, 0)]);
            float2 v = *dst;
            v.x -= acc.h[mt][nt][2 * h];
            v.y -= acc.h[mt][nt][2 * h + 1];
            *dst = v;
          }
    }
  }
  __syncthreads();
  CPROF(2);
  panel_factor_solve(S.As, S.Xs, b > 0);   // ends with a block barrier
  CPROF(3);
  CPROF(4);
  if (b == 0) {   // the diagonal factor, as a dense lower-triangular block
    float* dst = Ld + (size_t)j * NB * NB;
    for (int e = tid; e < NB * NB; e += kPotfThreads) dst[e] = (e & 63) <= (e >> 6) ? S.As.a[e >> 6][e & 63] : 0.f;
    return;
  }
  for (int e = tid; e < NB * NB / 4; e += kPotfThreads) {
    const int r = e >> 4, c = (e & 15) << 2;
    *reinterpret_cast<float4*>(P + (int64_t)r * Qp + c) = *reinterpret_cast<const float4*>(&S.Xs.a[r][c]);
  }
  CPROF(5);
}

// Linv diagonal blocks: one CTA per 64 x 64 diagonal factor (Ld[j]) -> Linv[j*64.., j*64..] (ld = ldd).
__global__ void __launch_bounds__(kPotfThreads) diag_inv_kernel(const float* __restrict__ Ld, float* __restrict__ Linv,
                                                                int64_t ldd) {
  __shared__ Block64 As;
  __shared__ Block64 Xs;
  __shared__ float Ts[NB / 2][NB / 2 + 1];
  const int tid = threadIdx.x;
  const float* src = Ld + (size_t)blockIdx.x * NB * NB;
  for (int e = tid; e < NB * NB; e += kPotfThreads) As.a[e >> 6][e & 63] = src[e];
  __syncthreads();
  invert64(As, Xs, Ts);
  float* dst = Linv + (int64_t)blockIdx.x * NB * (ldd + 1);
  for (int e = tid; e < NB * NB; e += kPotfThreads) dst[(int64_t)(e >> 6) * ldd + (e & 63)] = Xs.a[e >> 6][e & 63];
}

// Copy the diagonal factors back into the big matrix (so Bm holds the complete Lc).
__global__ void __launch_bounds__(kPotfThreads) diag_store_kernel(const float* __restrict__ Ld, float* __restrict__ Bm,
                                                                  int64_t ld) {
  const float* src = Ld + (size_t)blockIdx.x * NB * NB;
  float* dst = Bm + (int64_t)blockIdx.x * NB * (ld + 1);
  for (int e = threadIdx.x; e < NB * NB; e += kPotfThreads) dst[(int64_t)(e >> 6) * ld + (e & 63)] = src[e];
}

// At (cols x rows, ld = ldt) = A^T for A (rows x cols, ld = lda)
__global__ void __launch_bounds__(256) transpose_kernel(const float* __restrict__ A, int64_t lda, int rows, int cols,
                                                        float* __restrict__ At, int64_t ldt) {
  __shared__ float tile[32][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int r0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  for (int i = ty; i < 32; i += 8)
    tile[i][tx] = (r0 + i < rows && c0 + tx < cols) ? A[(int64_t)(r0 + i) * lda + c0 + tx] : 0.f;
  __syncthreads();
  for (int i = ty; i < 32; i += 8)
    if (c0 + i < cols && r0 + tx < rows) At[(int64_t)(c0 + i) * ldt + r0 + tx] = tile[tx][i];
}

// magnitude slots for the tensor-core block GEMMs (bit patterns of floats; see launch_tc_blockgemm)
__global__ void amax_slots_kernel(uint32_t* __restrict__ a, int mode) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const uint32_t one = 0x3F800000u;
  if (mode == 0) {
    a[1] = one; a[2] = one; a[3] = a[0];
  } else if (mode == 1) {
    a[0] = one;
  } else {
    a[1] = a[0];
  }
}

// ------------------------------------------------------------------ reductions
// partials[blockIdx.x] = sum over this CTA's rows of sum_{c < cols} A[r][c]^2 (fixed order).  Squares are summed in
// fp32 over 16 elements at a time and those short sums in double (B200's fp64 pipe is slow; a 16-term fp32 sum of
// squares carries ~1e-7 relative error, far below what tr B^-1 / ||W||^2 need).  cols % 4 == 0, rows 16-byte aligned.
__global__ void __launch_bounds__(256) sumsq_partial_kernel(const float* __restrict__ A, int64_t ld, int rows, int cols,
                                                            double* __restrict__ partials) {
  __shared__ double red[8];
  double s = 0;
  const int c4n = cols >> 2;
  for (int r = blockIdx.x; r < rows; r += gridDim.x) {
    const float4* row = reinterpret_cast<const float4*>(A + (int64_t)r * ld);
    for (int c0 = threadIdx.x; c0 < c4n; c0 += 4 * blockDim.x) {
      float f = 0.f;
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int c = c0 + u * blockDim.x;
        if (c < c4n) {
          const float4 v = row[c];
          f = fmaf(v.x, v.x, f); f = fmaf(v.y, v.y, f); f = fmaf(v.z, v.z, f); f = fmaf(v.w, v.w, f);
        }
      }
      s += (double)f;
    }
  }
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0;
    for (int w = 0; w < 8; ++w) t += red[w];
    partials[blockIdx.x] = t;
  }
}

constexpr int kSumsqBlocks = 592;

// deterministic single-CTA sum of `nparts` doubles (+ optional 2 sum log diag(Lc))
__device__ __forceinline__ double block_sum_256(double v, double* red) {
  v = warp_sum(v);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  double t = 0;
  for (int w = 0; w < 8; ++w) t += red[w];
  __syncthreads();
  return t;
}

// after the factorisation: logdetB from diag(Lc), tr Binv from the partial sums of Linv^2
__global__ void __launch_bounds__(256) factor_scalars_kernel(const float* __restrict__ Lc, int Qp, int Q,
                                                             const double* __restrict__ part_linv, int nparts,
                                                             double* __restrict__ scal) {
  __shared__ double red[8];
  double ld = 0, tr = 0;
  for (int i = threadIdx.x; i < Q; i += blockDim.x) ld += 2.0 * log((double)Lc[(int64_t)i * Qp + i]);
  for (int i = threadIdx.x; i < nparts; i += blockDim.x) tr += part_linv[i];
  ld = block_sum_256(ld, red);
  tr = block_sum_256(tr, red);
  if (threadIdx.x == 0) {
    scal[GPP_S_LOGDETB] = ld;
    scal[GPP_S_TRBINV] = tr;
  }
}

// after W: ||W||_F^2 and the per-row constant of the NLL
__global__ void __launch_bounds__(256) solve_scalars_kernel(int L, int64_t n_total, const double* __restrict__ part_w,
                                                            int nparts, double* __restrict__ scal) {
  __shared__ double red[8];
  double w2 = 0;
  for (int i = threadIdx.x; i < nparts; i += blockDim.x) w2 += part_w[i];
  w2 = block_sum_256(w2, red);
  if (threadIdx.x == 0) {
    scal[GPP_S_WNORM2] = w2;
    scal[GPP_S_ROWCONST] = 0.5 * (double)L * (log(scal[GPP_S_VN]) + scal[GPP_S_LOGDETB] / (double)n_total);
  }
}

// vbs (gp.py:75-76, 79-81) in Q-space form (SURVEY.md section 7.2):
//   vbs[0] = -0.5 ||W||^2 / v0^2 + 0.5 L (Q - tr Binv) / (r vn),  r = v0/vn
//   vbs[1] = -0.5 ||Xb||^2      + 0.5 L (N - Q + tr Binv) / vn
__global__ void vbs_kernel(const double* __restrict__ scal, int64_t n_total, int Q, int L, float* __restrict__ vbs) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    const double v0 = scal[GPP_S_V0], vn = scal[GPP_S_VN];
    const double trb = scal[GPP_S_TRBINV];
    vbs[0] = (float)(-0.5 * scal[GPP_S_WNORM2] / (v0 * v0) + 0.5 * (double)L * ((double)Q - trb) / v0);
    vbs[1] = (float)(-0.5 * scal[GPP_S_XB2] + 0.5 * (double)L * ((double)n_total - (double)Q + trb) / vn);
  }
}

int launch_vbs(const double* scal, int64_t n_total, int Q, int L, float* vbs, cudaStream_t st) {
  vbs_kernel<<<1, 32, 0, st>>>(scal, n_total, Q, L, vbs);
  GPP_LAUNCH_CHECK();
  return GPP_OK;
}

// ------------------------------------------------------------------ k stacked designs (block form)
// V = [V_0 | ... | V_{k-1}], v_i = vs[i], vn = vs[k], D = diag(sqrt(v_i) on the columns of block i):
//   B = I + D G D / vn,  W = D B^-1 D C / vn,  Binv <- D B^-1 D.
// The factorisation is the single-design one on that B; afterwards Linv's columns are scaled by D (Linv' = Linv D, still
// lower triangular and |Linv'| <= |Linv| <= 1), so that the unchanged solve computes Linv'^T Linv' C / vn = W and the
// unchanged Binv product gives D B^-1 D.  With scal[V0] = 1 the N-long kernels (pass 2, Vb) then compute the k-design
// Xb and Vb as they stand.  Per block (caller-owned blk[2k]): blk[2i] = tr_i B^-1 (column block i of the UNSCALED Linv),
// blk[2i + 1] = ||W_i||^2 (row block i of W).

// scal[V0] = 1, scal[VN] = vn; dcol[a] = sqrt(v_i) for the columns a of block i, 1 on the padding up to Qp
__global__ void blocks_init_kernel(const float* __restrict__ vs, BlockSpec bs, int Qp, double* __restrict__ scal,
                                   float* __restrict__ dcol) {
  const int a = blockIdx.x * blockDim.x + threadIdx.x;
  if (a == 0) {
    scal[GPP_S_V0] = 1.0;
    scal[GPP_S_VN] = (double)vs[bs.k];
  }
  if (a >= Qp) return;
  float d = 1.f;
#pragma unroll
  for (int i = 0; i < kMaxBlocks; ++i)
    if (i < bs.k && a >= bs.start[i] && a < bs.start[i + 1]) d = sqrtf(vs[i]);
  dcol[a] = d;
}

// Bm (Qp x Qp) = I + D G D / vn on the real Q x Q block, identity on the padding.
__global__ void __launch_bounds__(256) build_b_blocks_kernel(const float* __restrict__ G, int64_t ldg, int Q, int Qp,
                                                             const float* __restrict__ dcol,
                                                             const double* __restrict__ scal, float* __restrict__ Bm) {
  const float rvn = (float)(1.0 / scal[GPP_S_VN]);
  const int64_t total4 = (int64_t)Qp * (Qp / 4);
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total4; e += (int64_t)gridDim.x * blockDim.x) {
    const int i = (int)(e / (Qp / 4));
    const int j4 = (int)(e - (int64_t)i * (Qp / 4)) * 4;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (i < Q && j4 < Q) {
      const float4 g = *reinterpret_cast<const float4*>(G + (int64_t)i * ldg + j4);
      const float4 dj = *reinterpret_cast<const float4*>(dcol + j4);
      const float ri = dcol[i] * rvn;
      v = make_float4(ri * dj.x * g.x, ri * dj.y * g.y, ri * dj.z * g.z, ri * dj.w * g.w);
    }
    if (i == j4 + 0) v.x += 1.f;
    if (i == j4 + 1) v.y += 1.f;
    if (i == j4 + 2) v.z += 1.f;
    if (i == j4 + 3) v.w += 1.f;
    *reinterpret_cast<float4*>(Bm + (int64_t)i * Qp + j4) = v;
  }
}

// A[r][c] *= dcol[c] over the Q x Q block (Linv -> Linv D)
__global__ void __launch_bounds__(256) scale_cols_kernel(float* __restrict__ A, int64_t ld, int Q,
                                                         const float* __restrict__ dcol) {
  const int64_t total4 = (int64_t)Q * (Q / 4);
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total4; e += (int64_t)gridDim.x * blockDim.x) {
    const int i = (int)(e / (Q / 4));
    const int j4 = (int)(e - (int64_t)i * (Q / 4)) * 4;
    float4* p = reinterpret_cast<float4*>(A + (int64_t)i * ld + j4);
    const float4 d = *reinterpret_cast<const float4*>(dcol + j4);
    float4 v = *p;
    v.x *= d.x; v.y *= d.y; v.z *= d.z; v.w *= d.w;
    *p = v;
  }
}

// partials[blockIdx.x * k + i] = sum of squares of block i of A (rows x cols): the column block [start[i], start[i+1])
// over all rows (by_cols), or the row block over all columns.  Same fixed-order arithmetic as sumsq_partial_kernel.
__global__ void __launch_bounds__(256) block_sumsq_partial_kernel(const float* __restrict__ A, int64_t ld, int rows,
                                                                  int cols, BlockSpec bs, int by_cols,
                                                                  double* __restrict__ partials) {
  __shared__ double red[8];
  for (int b = 0; b < bs.k; ++b) {
    const int r_lo = by_cols ? 0 : bs.start[b], r_hi = by_cols ? rows : bs.start[b + 1];
    const int c_lo = by_cols ? bs.start[b] : 0, c4n = ((by_cols ? bs.start[b + 1] : cols) - c_lo) >> 2;
    double s = 0;
    for (int r = r_lo + blockIdx.x; r < r_hi; r += gridDim.x) {
      const float4* row = reinterpret_cast<const float4*>(A + (int64_t)r * ld + c_lo);
      for (int c0 = threadIdx.x; c0 < c4n; c0 += 4 * blockDim.x) {
        float f = 0.f;
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int c = c0 + u * blockDim.x;
          if (c < c4n) {
            const float4 v = row[c];
            f = fmaf(v.x, v.x, f); f = fmaf(v.y, v.y, f); f = fmaf(v.z, v.z, f); f = fmaf(v.w, v.w, f);
          }
        }
        s += (double)f;
      }
    }
    s = warp_sum(s);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
      double t = 0;
      for (int w = 0; w < 8; ++w) t += red[w];
      partials[(int64_t)blockIdx.x * bs.k + b] = t;
    }
    __syncthreads();
  }
}

// blk[2i + slot] = sum over the CTAs of partials[c * k + i], in a fixed order
__global__ void __launch_bounds__(256) block_reduce_kernel(const double* __restrict__ partials, int nparts, int k,
                                                           int slot, double* __restrict__ blk) {
  __shared__ double red[8];
  for (int b = 0; b < k; ++b) {
    double s = 0;
    for (int c = threadIdx.x; c < nparts; c += blockDim.x) s += partials[(int64_t)c * k + b];
    s = block_sum_256(s, red);
    if (threadIdx.x == 0) blk[2 * b + slot] = s;
  }
}

// vbs (k + 1 entries) of the block form:
//   vbs[i] = -0.5 ||W_i||^2 / v_i^2 + 0.5 L (Q_i - tr_i B^-1) / v_i,   vbs[k] = -0.5 ||Xb||^2 + 0.5 L (N - Q + tr B^-1) / vn
__global__ void vbs_blocks_kernel(const double* __restrict__ scal, const double* __restrict__ blk,
                                  const float* __restrict__ vs, BlockSpec bs, int64_t n_total, int L,
                                  float* __restrict__ vbs) {
  const int i = threadIdx.x;
  const int Q = bs.start[bs.k];
  if (i < bs.k) {
    const double v = (double)vs[i];
    const double Qi = (double)(bs.start[i + 1] - bs.start[i]);
    vbs[i] = (float)(-0.5 * blk[2 * i + 1] / (v * v) + 0.5 * (double)L * (Qi - blk[2 * i]) / v);
  } else if (i == bs.k) {
    vbs[i] = (float)(-0.5 * scal[GPP_S_XB2] +
                     0.5 * (double)L * ((double)n_total - (double)Q + scal[GPP_S_TRBINV]) / scal[GPP_S_VN]);
  }
}

int launch_vbs_blocks(const double* scal, const double* blk, const float* vs, const BlockSpec& bs, int64_t n_total, int L,
                      float* vbs, cudaStream_t st) {
  vbs_blocks_kernel<<<1, 32, 0, st>>>(scal, blk, vs, bs, n_total, L, vbs);
  GPP_LAUNCH_CHECK();
  return GPP_OK;
}

// ------------------------------------------------------------------ driver
// The factor workspace doubles as the factorisation *state*: after launch_factor() it holds Lc and
// Linv, which launch_solve_w() reuses for any number of right-hand sides (train_gppvae.py builds the
// same factorisation twice per epoch, at :235 and inside :166; the caller caches this buffer).
struct FactorLayout {
  int Qp;
  size_t off_bm, off_linv, off_tm, off_ld, off_part, off_amax, off_cnt, cnt_bytes, off_llp, llp_bytes, off_tn, total;
  size_t tn_bytes;
};

static FactorLayout factor_layout(int Q) {
  FactorLayout f;
  f.Qp = (int)(ceil_div(Q, NB) * NB);
  const size_t qq = align_up((size_t)f.Qp * f.Qp * sizeof(float), 256);
  size_t o = 0;
  f.off_bm = o;   o += qq;
  f.off_linv = o; o += qq;
  f.off_tm = o;   o += qq;
  f.off_ld = o;   o += align_up((size_t)f.Qp * NB * sizeof(float), 256);   // the 64 x 64 diagonal factors
  f.off_part = o; o += align_up((size_t)kSumsqBlocks * sizeof(double), 256);
  f.off_amax = o; o += 256;
  f.off_cnt = o;                                                                   // arrival counters of the left-looking
  f.cnt_bytes = align_up((size_t)(f.Qp / NB) * kLLMaxRowTiles * sizeof(unsigned int), 256);   // updates, per step
  o += f.cnt_bytes;
  f.off_llp = o;                                                                   // partial tiles of the left-looking
  f.llp_bytes = align_up((size_t)kLLMaxParts * kLLTileFloats * sizeof(float), 256);   // updates (one per wide CTA)
  o += f.llp_bytes;
  f.off_tn = o;
  f.tn_bytes = tn_workspace_bytes(Q, Q, Q, 0, 1);
  if (tc_pass1_supported(Q, Q, 0)) {
    const size_t tcb = tc_pass1_workspace_bytes(Q, Q, 0, false);
    if (tcb > f.tn_bytes) f.tn_bytes = tcb;
  }
  o += align_up(f.tn_bytes, 256);
  f.total = o;
  return f;
}

struct SolveLayout {
  size_t off_t1, off_t1p, off_part, off_amax, off_tn, total;
  size_t tn_bytes;
  int ksplit;   // T1 = Linv C as `ksplit` products over slices of the contraction (partials in t1p), summed in order
};

// How many slices of the contraction T1 = Linv . C is cut into: as ONE product it is Q / 256 row tiles on the tensor-core
// row kernel, 16 CTA pairs at Q = 4096, each walking up to the whole contraction -- 145 us of a 0.29 ms solve (launch
// list of round 2).  Slices of >= 1024 multiply the units; the triangular structure of Linv is not exploited then (the
// zero blocks above the diagonal are multiplied like any other), which costs tensor time nobody was using.
static int solve_ksplit(int Q) {
  int ks = 1;
  while (ks < 8 && Q % (2 * ks * 256) == 0 && Q / (2 * ks) >= 1024) ks *= 2;
  return ks;
}

static SolveLayout solve_layout(int Q, int L) {
  SolveLayout f;
  size_t o = 0;
  f.off_t1 = o;   o += align_up((size_t)Q * L * sizeof(float), 256);
  f.ksplit = solve_ksplit(Q);
  f.off_t1p = o;  o += f.ksplit > 1 ? align_up((size_t)f.ksplit * Q * L * sizeof(float), 256) : 0;
  f.off_part = o; o += align_up((size_t)kSumsqBlocks * sizeof(double), 256);
  f.off_amax = o; o += 256;
  f.off_tn = o;
  f.tn_bytes = tn_workspace_bytes(Q, Q, 0, L, 0);
  if (tc_pass1_supported(Q, Q, L)) {
    const size_t tcb = tc_pass1_workspace_bytes(Q, Q, L, true);
    if (tcb > f.tn_bytes) f.tn_bytes = tcb;
  }
  o += align_up(f.tn_bytes, 256);
  f.total = o;
  return f;
}

// out = sum of `ns` consecutive slices of n4 float4 each, in slice order
__global__ void __launch_bounds__(256) sum_slices_kernel(const float* __restrict__ part, int ns, int64_t n4,
                                                         float* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n4) return;
  float4 s = reinterpret_cast<const float4*>(part)[i];
  for (int q = 1; q < ns; ++q) {
    const float4 v = reinterpret_cast<const float4*>(part)[(int64_t)q * n4 + i];
    s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
  }
  reinterpret_cast<float4*>(out)[i] = s;
}

size_t factor_workspace_bytes(int Q) { return factor_layout(Q).total; }
size_t solve_workspace_bytes(int Q, int L) { return solve_layout(Q, L).total; }

// ---- Linv by recursive doubling: inv([[A,0],[C,D]]) = [[Ai,0],[-Di C Ai, Di]]
// Levels b_lo <= b < b_hi (pair half-width b, doubling) restricted to the diagonal block [r0, r0 + size) of Lc / Linv;
// `do_t` launches T = C . Ai of each level, `do_x` launches X = -Di . T.  From 512 rows up the products run on the tensor
// cores (3xTF32 wide-range split); amax = {bound of max|Lc|, 1, 1, bound of max|Lc|}: the magnitudes the fp16 scales of
// their correction terms come from (B >= I, so ||Linv||_2 <= 1; T = C . Ai inherits Lc's magnitude).
static int inverse_levels(float* Bm0, float* Linv0, float* Tm0, int Qp, int r0, int size, int b_lo, int b_hi, bool do_t,
                          bool do_x, const uint32_t* amax, cudaStream_t st) {
  float* Bm = Bm0 + (int64_t)r0 * (Qp + 1);
  float* Linv = Linv0 + (int64_t)r0 * (Qp + 1);
  float* Tm = Tm0 + (int64_t)r0 * (Qp + 1);
  for (int b = b_lo; b < b_hi && b < size; b *= 2) {
    const int npairs = (int)ceil_div(size - b, 2 * b);
    int m_last = size - (2 * (npairs - 1) * b + b);  // rows of the last pair's D block
    if (m_last > b) m_last = b;                      // (a trailing unpaired block waits for the next level)
    const int64_t pair_stride = (int64_t)2 * b * (Qp + 1);
    if (tc_blockgemm_supported(b, b, b)) {
      if (do_t) {
        TcBlockGemm g{};
        g.wide_range = 1;
        g.n = b; g.n_last = m_last; g.K = b; g.ncols = b; g.batches = npairs; g.out_step = pair_stride;
        g.a_row0 = b; g.a_row_step = 2 * b; g.a_k0 = 0; g.a_k_step = 2 * b;       // C block of Lc: rows p0 + b, cols p0
        g.b_k0 = 0; g.b_k_step = 2 * b; g.b_col0 = 0; g.b_col_step = 2 * b;       // Ai: rows p0, cols p0
        g.tri_b = 1; g.alpha = 1.f;
        GPP_TRY(launch_tc_blockgemm(Bm, size, size, Qp, Linv, size, size, Qp, Tm + (int64_t)b * Qp, Qp, g, amax, st));
      }
      if (do_x) {
        TcBlockGemm x{};
        x.wide_range = 1;
        x.n = b; x.n_last = m_last; x.K = b; x.ncols = b; x.batches = npairs; x.out_step = pair_stride;
        x.a_row0 = b; x.a_row_step = 2 * b; x.a_k0 = b; x.a_k_step = 2 * b;       // Di: rows p0 + b, cols p0 + b
        x.b_k0 = b; x.b_k_step = 2 * b; x.b_col0 = 0; x.b_col_step = 2 * b;       // T: rows p0 + b, cols p0
        x.tri_a = 1; x.alpha = -1.f;
        GPP_TRY(launch_tc_blockgemm(Linv, size, size, Qp, Tm, size, size, Qp, Linv + (int64_t)b * Qp, Qp, x, amax + 2, st));
      }
      continue;
    }
    if (do_t) {
      GemmParams t{};
      t.A = Bm + (int64_t)b * Qp;  t.lda = Qp; t.strideA = pair_stride;      // C block of Lc
      t.B = Linv;                  t.ldb = Qp; t.strideB = pair_stride;      // Ai, read as B(n,k) = Ai[k][n]
      t.C = Tm + (int64_t)b * Qp;  t.ldc = Qp; t.strideC = pair_stride;
      t.M = b; t.N = b; t.K = b; t.M_last = m_last; t.alpha = 1.f; t.beta = 0.f; t.tri_b = 1;
      GPP_TRY(launch_gemm(t, false, true, npairs, st));                      // T = C . Ai
    }
    if (do_x) {
      GemmParams x{};
      x.A = Linv + (int64_t)b * (Qp + 1); x.lda = Qp; x.strideA = pair_stride;  // Di
      x.B = Tm + (int64_t)b * Qp;         x.ldb = Qp; x.strideB = pair_stride;  // T, read as B(n,k) = T[k][n]
      x.C = Linv + (int64_t)b * Qp;       x.ldc = Qp; x.strideC = pair_stride;
      x.M = b; x.N = b; x.K = b; x.K_is_M = 1; x.M_last = m_last; x.alpha = -1.f; x.beta = 0.f; x.tri_a = 1;
      GPP_TRY(launch_gemm(x, false, true, npairs, st));                      // X = -Di . T
    }
  }
  return GPP_OK;
}

// amax[0] = amax[3] = bit pattern of sqrt(max_i B_ii) (every |Lc_ij| <= sqrt(B_ii): row i of Lc has squared norm B_ii),
// amax[1] = amax[2] = 1.  Known BEFORE the factorisation, so the leading part of the triangular inverse can start on the
// side stream while the panel chain is still running.
__global__ void __launch_bounds__(256) lc_bound_kernel(const float* __restrict__ Bm, int Qp, uint32_t* __restrict__ amax) {
  __shared__ float red[8];
  float m = 0.f;
  for (int i = threadIdx.x; i < Qp; i += blockDim.x) m = fmaxf(m, Bm[(int64_t)i * Qp + i]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < 8; ++w) m = fmaxf(m, red[w]);
    const uint32_t bits = __float_as_uint(sqrtf(m));
    amax[0] = bits; amax[3] = bits;
    amax[1] = 0x3F800000u; amax[2] = 0x3F800000u;
  }
}

// Side stream + fork / join events of the factorisation, per device (created on first use, never destroyed).
struct SideStream {
  cudaStream_t s = nullptr;
  cudaEvent_t fork = nullptr, join = nullptr;
};
static int side_stream(SideStream** out) {
  static std::mutex mu;
  static SideStream per_dev[64];
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64) dev = 0;
  std::lock_guard<std::mutex> lock(mu);
  SideStream& ss = per_dev[dev];
  if (!ss.s) {
    GPP_CUDA(cudaStreamCreateWithFlags(&ss.s, cudaStreamNonBlocking));
    GPP_CUDA(cudaEventCreateWithFlags(&ss.fork, cudaEventDisableTiming));
    GPP_CUDA(cudaEventCreateWithFlags(&ss.join, cudaEventDisableTiming));
  }
  *out = &ss;
  return GPP_OK;
}


// Block form (k designs): the per-column scales and the per-block partial sums follow the single-design state.
static size_t blocks_off_dcol(int Q) { return align_up(factor_layout(Q).total, 256); }
static size_t blocks_off_part(int Q) {
  return blocks_off_dcol(Q) + align_up((size_t)factor_layout(Q).Qp * sizeof(float), 256);
}
size_t factor_blocks_workspace_bytes(int Q, int k) {
  return blocks_off_part(Q) + align_up((size_t)kSumsqBlocks * k * sizeof(double), 256);
}

// bs == nullptr: the single-design factorisation (scal[V0] = v0); otherwise the block form above, blk[2i] = tr_i B^-1.
static int factor_impl(const float* G, int64_t ldg, int Q, const float* vs, uint32_t flags, float* Binv, double* scal,
                       const BlockSpec* bs, double* blk, void* ws, size_t ws_bytes, cudaStream_t st) {
  const FactorLayout f = factor_layout(Q);
  const size_t need = bs ? factor_blocks_workspace_bytes(Q, bs->k) : f.total;
  if (!ws || ws_bytes < need) {
    set_error("factor: workspace too small (%zu < %zu bytes)", ws_bytes, need);
    return GPP_ERR_WORKSPACE;
  }
  char* base = static_cast<char*>(ws);
  float* Bm = reinterpret_cast<float*>(base + f.off_bm);
  float* Linv = reinterpret_cast<float*>(base + f.off_linv);
  float* Tm = reinterpret_cast<float*>(base + f.off_tm);
  double* part = reinterpret_cast<double*>(base + f.off_part);
  void* tnws = base + f.off_tn;
  uint32_t* amax = reinterpret_cast<uint32_t*>(base + f.off_amax);
  const int Qp = f.Qp;
  const int nb = Qp / NB;

  float* dcol = bs ? reinterpret_cast<float*>(base + blocks_off_dcol(Q)) : nullptr;
  double* bpart = bs ? reinterpret_cast<double*>(base + blocks_off_part(Q)) : nullptr;
  {
    const int64_t total4 = (int64_t)Qp * (Qp / 4);
    int blocks = (int)(ceil_div(total4, 256) < 4096 ? ceil_div(total4, 256) : 4096);
    if (bs) {
      blocks_init_kernel<<<(unsigned)ceil_div(Qp, 256), 256, 0, st>>>(vs, *bs, Qp, scal, dcol);
      GPP_LAUNCH_CHECK();
      build_b_blocks_kernel<<<blocks, 256, 0, st>>>(G, ldg, Q, Qp, dcol, scal, Bm);
    } else {
      scal_init_kernel<<<1, 32, 0, st>>>(vs, scal);
      GPP_LAUNCH_CHECK();
      build_b_kernel<<<blocks, 256, 0, st>>>(G, ldg, Q, Qp, scal, Bm);
    }
    GPP_LAUNCH_CHECK();
  }
  GPP_CUDA(cudaMemsetAsync(Linv, 0, (size_t)Qp * Qp * sizeof(float), st));
  GPP_CUDA(cudaMemsetAsync(Tm, 0, (size_t)Qp * Qp * sizeof(float), st));   // scratch of the triangular inverse: finite

  // ---- blocked Cholesky with look-ahead: ONE kernel per 64-wide panel (see chol_step_kernel); the diagonal factors
  //      are parked in Ld so that no CTA reads a block another one rewrites
  float* Ld = reinterpret_cast<float*>(base + f.off_ld);
  {   // per device: a second device in the process needs its own attribute (ADVICE r1)
    static std::mutex mu;
    static bool step_attr[64] = {false};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64) dev = 0;
    std::lock_guard<std::mutex> lock(mu);
    if (!step_attr[dev]) {
      GPP_CUDA(cudaFuncSetAttribute(chol_step_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kStepSmemBytes));
      GPP_CUDA(cudaFuncSetAttribute(chol_step_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kStepSmemBytesLL));
      step_attr[dev] = true;
    }
  }
  // Outer blocks of kOuter panels: inside a block the panels update each other (rank-64 updates in chol_step_kernel),
  // everything to the right of the block gets the block's kOuter panels at once, as ONE rank-256 update on the tensor
  // cores (C -= Lp Lp^T, lower tiles).  Measured (factor_only.py): Q = 8192 10.1 -> 8.1 ms, where the SIMT trailing
  // updates were the larger half of the stage; Q = 4096 2.40 -> 2.84 ms, where the look-ahead of the single-level scheme
  // hides them completely behind the panel chain (64 x 23 us) and the 16 serial rank-256 updates (37-70 us each, a
  // 256-deep contraction does not amortise the tensor-core kernel's pipeline fill and epilogue) do not.  Hence the switch.
  constexpr int kOuter = 4;
  const char* min_q_env = getenv("GPP_CHOL_OUTER_MIN_Q");             // tests force the outer scheme at small Q
  const bool outer = Qp >= (min_q_env ? atoi(min_q_env) : kOuterCholMinQ) && tc_blockgemm_supported(512, kOuter * NB, 512);
  // Below the outer-block sizes the trailing updates are left-looking (see chol_step_kernel); GPP_CHOL_WIDE=rl selects the
  // right-looking scheme of rounds 1-2 (kept for A/B timing).
  const char* wide_env = getenv("GPP_CHOL_WIDE");
  const bool left_looking = !outer && !(wide_env && wide_env[0] == 'r') && nb <= 2 * kLLMaxRowTiles;
  const char* pdl_env = getenv("GPP_CHOL_PDL");
  const bool use_pdl = !(pdl_env && pdl_env[0] == '0');
  unsigned int* counters = reinterpret_cast<unsigned int*>(base + f.off_cnt);
  if (left_looking) GPP_CUDA(cudaMemsetAsync(counters, 0, f.cnt_bytes, st));
  const int sms = sm_count();
  const int64_t part_cap = kLLMaxParts;
  float* ll_part = reinterpret_cast<float*>(base + f.off_llp);
  // The triangular inverse of the LEADING diagonal block [0, b_top), b_top = the largest power-of-two multiple of the
  // panel below Qp, only needs the panels < jsplit = b_top / 64: it runs on a side stream beside the TAIL of the panel
  // chain, followed by T = L21 . L11^-1 of the top level.  Where the side stream forks matters: the left-looking updates
  // keep every SM's tensor pipe busy through the middle of the chain, and forking at jsplit - 1 (the earliest possible
  // step) with SMs set aside for the side stream cost 0.05 ms at Q = 4096 instead of saving anything; forking at 3/4 of
  // the chain, where few wide CTAs are left, and setting no SMs aside saves 0.06 ms (1.623 -> 1.558-1.571 ms for forks at
  // steps 44..52; factor_only.py).  GPP_INV_OVERLAP=0 disables it, GPP_INV_FORK=<step> / GPP_INV_SIDE_SMS=<n> move it.
  int b_top = NB;
  while (b_top * 2 < Qp) b_top *= 2;
  const int jsplit = b_top / NB;
  const char* ov_env = getenv("GPP_INV_OVERLAP");
  const bool want_side = !outer && Qp >= 1024 && !(ov_env && ov_env[0] == '0');
  const char* fork_env = getenv("GPP_INV_FORK");
  int fork_step = jsplit - 1 > (3 * nb) / 4 ? jsplit - 1 : (3 * nb) / 4;
  if (fork_env && atoi(fork_env) >= jsplit - 1) fork_step = atoi(fork_env);
  if (fork_step > nb - 1) fork_step = nb - 1;
  const char* sms_env = getenv("GPP_INV_SIDE_SMS");
  const int side_sms = sms_env ? atoi(sms_env) : 0;
  SideStream* side = nullptr;
  bool side_started = false;
  if (want_side) GPP_TRY(side_stream(&side));
  lc_bound_kernel<<<1, 256, 0, st>>>(Bm, Qp, amax);
  GPP_LAUNCH_CHECK();
  for (int j = 0; j < nb; ++j) {
    const int npanel = nb - j;
    const int jj = outer ? j % kOuter : 0;
    const int blk_end = outer ? ((j / kOuter + 1) * kOuter < nb ? (j / kOuter + 1) * kOuter : nb) : nb;   // first block after the outer block
    const int apply_prev = outer ? (jj > 0) : (j > 0);
    int wide_cols, wide_ctas, ll_S = 0, ll_chunk = 0;
    if (left_looking) {
      wide_cols = -1;
      wide_ctas = 0;
      if (j >= 1 && j + 1 < nb) {
        // row tiles of column block j + 1, contraction over the j finished panels split so that the step's CTAs have
        // an SM each
        const int T = (int)ceil_div(Qp - (j + 1) * NB, BM);
        int free_sms = sms - npanel - ((want_side && j > fork_step) ? side_sms : 0);   // the side stream's kernels need room
        if (free_sms < T) free_sms = T;
        int S = free_sms / T;
        if (S > j) S = j;
        // a unit costs ~2 us per 64 k of its chunk plus ~0.1 us per partial tile its row tile's last arriver sums
        const int s_opt = (int)(sqrtf(20.f * (float)j) + 0.5f);
        if (S > s_opt) S = s_opt;
        if (S < 1) S = 1;
        while (S > 1 && (int64_t)T * S > part_cap) --S;
        ll_chunk = (int)ceil_div(j, S);
        ll_S = (int)ceil_div(j, ll_chunk);
        wide_ctas = T * ll_S;
      }
    } else if (!outer) {
      const int trail = Qp - (j + 1) * NB;
      const int T = j > 0 ? (trail + BM - 1) / BM : 0;
      wide_cols = -1;
      wide_ctas = T * (T + 1) / 2;
    } else {
      wide_cols = apply_prev ? blk_end - (j + 1) : 0;                 // column blocks j+1 .. blk_end-1 of this outer block
      wide_ctas = wide_cols > 0 ? (Qp - (j + 1) * NB + BM - 1) / BM : 0;
    }
    if (left_looking) {
      cudaLaunchConfig_t cfg = {};
      cfg.gridDim = dim3((unsigned)(npanel + wide_ctas));
      cfg.blockDim = dim3(kPotfThreads);
      cfg.dynamicSmemBytes = kStepSmemBytesLL;
      cfg.stream = st;
      cudaLaunchAttribute attr[1];
      attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
      attr[0].val.programmaticStreamSerializationAllowed = use_pdl ? 1 : 0;
      cfg.attrs = attr;
      cfg.numAttrs = 1;
      GPP_CUDA(cudaLaunchKernelEx(&cfg, chol_step_kernel<true>, Bm, Qp, j, Ld, apply_prev, wide_cols, ll_S, ll_chunk, ll_part,
                                  counters + (size_t)j * kLLMaxRowTiles));
    } else
      chol_step_kernel<false><<<npanel + wide_ctas, kPotfThreads, kStepSmemBytes, st>>>(
          Bm, Qp, j, Ld, apply_prev, wide_cols, ll_S, ll_chunk, ll_part, counters + (size_t)j * kLLMaxRowTiles);
    GPP_LAUNCH_CHECK();
    if (want_side && j == fork_step) {
      cudaStream_t s2 = side->s;
      GPP_CUDA(cudaEventRecord(side->fork, st));
      GPP_CUDA(cudaStreamWaitEvent(s2, side->fork, 0));
      diag_store_kernel<<<jsplit, kPotfThreads, 0, s2>>>(Ld, Bm, Qp);
      GPP_LAUNCH_CHECK();
      diag_inv_kernel<<<jsplit, kPotfThreads, 0, s2>>>(Ld, Linv, Qp);
      GPP_LAUNCH_CHECK();
      GPP_TRY(inverse_levels(Bm, Linv, Tm, Qp, 0, b_top, NB, b_top, true, true, amax, s2));
      GPP_TRY(inverse_levels(Bm, Linv, Tm, Qp, 0, Qp, b_top, Qp, true, false, amax, s2));
      GPP_CUDA(cudaEventRecord(side->join, s2));
      side_started = true;
    }
    if (outer && j + 1 == blk_end && blk_end < nb) {
      // rank-(kOuter * 64) update of everything right of the outer block
      const int c0 = (j / kOuter) * kOuter * NB;               // first column of the outer block
      const int K = (blk_end * NB) - c0;
      const int r0 = blk_end * NB, rem = Qp - r0;
      const float* Lp = Bm + (int64_t)r0 * Qp + c0;          // rem x K panel
      float* Cc = Bm + (int64_t)r0 * (Qp + 1);               // trailing matrix
      if (rem >= 512) {
        dim3 tg((unsigned)ceil_div(rem, 32), (unsigned)ceil_div(K, 32));
        transpose_kernel<<<tg, 256, 0, st>>>(Lp, Qp, rem, K, Tm, Qp);
        GPP_LAUNCH_CHECK();
        GPP_TRY(tc_absmax(Lp, Qp, rem, K, amax + 4, st));     // (slots 0..3 hold the bounds of the triangular inverse)
        amax_slots_kernel<<<1, 32, 0, st>>>(amax + 4, 2);
        GPP_LAUNCH_CHECK();
        GPP_TRY(launch_tc_syrk_sub(Cc, Qp, Lp, Qp, Tm, Qp, rem, K, amax + 4, st));
      } else {
        GemmParams g{};
        g.A = Lp; g.lda = Qp; g.B = Lp; g.ldb = Qp; g.C = Cc; g.ldc = Qp;
        g.M = rem; g.N = rem; g.K = K; g.M_last = -1; g.alpha = -1.f; g.beta = 1.f; g.lower_only = 1;
        GPP_TRY(launch_gemm(g, false, false, 1, st));
      }
    }
  }
  // ---- the rest of the triangular inverse: the trailing diagonal block [b_top, Qp) level by level, then (after the side
  //      stream has delivered the inverse of the leading block and T = L21 . L11^-1) the top level X = -L22^-1 . T
  {
    const int j0 = side_started ? jsplit : 0;          // diagonal blocks not handled on the side stream
    diag_store_kernel<<<nb - j0, kPotfThreads, 0, st>>>(Ld + (size_t)j0 * NB * NB, Bm + (int64_t)j0 * NB * (Qp + 1), Qp);
    GPP_LAUNCH_CHECK();
    diag_inv_kernel<<<nb - j0, kPotfThreads, 0, st>>>(Ld + (size_t)j0 * NB * NB, Linv + (int64_t)j0 * NB * (Qp + 1), Qp);
    GPP_LAUNCH_CHECK();
    if (side_started) {
      GPP_TRY(inverse_levels(Bm, Linv, Tm, Qp, b_top, Qp - b_top, NB, Qp, true, true, amax, st));
      GPP_CUDA(cudaStreamWaitEvent(st, side->join, 0));
      GPP_TRY(inverse_levels(Bm, Linv, Tm, Qp, 0, Qp, b_top, Qp, false, true, amax, st));
    } else {
      GPP_TRY(inverse_levels(Bm, Linv, Tm, Qp, 0, Qp, NB, Qp, true, true, amax, st));
    }
  }

  if (bs) {   // tr_i B^-1 from the unscaled Linv, then Linv <- Linv D
    block_sumsq_partial_kernel<<<kSumsqBlocks, 256, 0, st>>>(Linv, Qp, Q, Q, *bs, 1, bpart);
    GPP_LAUNCH_CHECK();
    block_reduce_kernel<<<1, 256, 0, st>>>(bpart, kSumsqBlocks, bs->k, 0, blk);
    GPP_LAUNCH_CHECK();
    const int64_t total4 = (int64_t)Q * (Q / 4);
    scale_cols_kernel<<<(unsigned)(ceil_div(total4, 256) < 4096 ? ceil_div(total4, 256) : 4096), 256, 0, st>>>(Linv, Qp, Q,
                                                                                                              dcol);
    GPP_LAUNCH_CHECK();
  }
  if (flags & GPP_WANT_BINV) {  // Binv = Linv^T Linv  (block form: D B^-1 D)
    if (!Binv) {
      set_error("factor: GPP_WANT_BINV set but Binv is null");
      return GPP_ERR_INVALID_ARGUMENT;
    }
    if (tc_pass1_supported(Q, Q, 0))
      GPP_TRY(launch_tc_pass1(Linv, Qp, nullptr, 0, Q, Q, 0, Binv, Q, nullptr, 0, nullptr, tnws, f.tn_bytes, true, st));
    else
      GPP_TRY(launch_tn(Linv, Qp, Q, Linv, Qp, Q, nullptr, 0, 0, Q, 1, Binv, Q, nullptr, 0, nullptr, tnws, f.tn_bytes, st));
  }
  if (bs) {   // tr B^-1 = the sum of the per-block partials
    factor_scalars_kernel<<<1, 256, 0, st>>>(Bm, Qp, Q, bpart, kSumsqBlocks * bs->k, scal);
    GPP_LAUNCH_CHECK();
    return GPP_OK;
  }
  sumsq_partial_kernel<<<kSumsqBlocks, 256, 0, st>>>(Linv, Qp, Q, Q, part);
  GPP_LAUNCH_CHECK();
  factor_scalars_kernel<<<1, 256, 0, st>>>(Bm, Qp, Q, part, kSumsqBlocks, scal);
  GPP_LAUNCH_CHECK();
  return GPP_OK;
}

int launch_factor(const float* G, int64_t ldg, int Q, const float* vs, uint32_t flags, float* Binv, double* scal,
                  void* ws, size_t ws_bytes, cudaStream_t st) {
  return factor_impl(G, ldg, Q, vs, flags, Binv, scal, nullptr, nullptr, ws, ws_bytes, st);
}

int launch_factor_blocks(const float* G, int64_t ldg, const BlockSpec& bs, const float* vs, uint32_t flags, float* Binv,
                         double* scal, double* blk, void* ws, size_t ws_bytes, cudaStream_t st) {
  return factor_impl(G, ldg, bs.start[bs.k], vs, flags, Binv, scal, &bs, blk, ws, ws_bytes, st);
}

// W = (v0/vn) Linv^T (Linv C) for C (Q x L); `state` is the workspace launch_factor filled for the same Q.
// L_true (<= L) is the number of real latent columns (the rest is zero padding) and enters ROWCONST.
int launch_solve_w(const float* C, int64_t ldc, int Q, int L, int L_true, int64_t n_total, float* W, int64_t ldw,
                   double* scal, const void* state, size_t state_bytes, void* ws, size_t ws_bytes, cudaStream_t st) {
  const FactorLayout f = factor_layout(Q);
  const SolveLayout sl = solve_layout(Q, L);
  if (!state || state_bytes < f.total) {
    set_error("solve_w: factorisation state too small (%zu < %zu bytes)", state_bytes, f.total);
    return GPP_ERR_WORKSPACE;
  }
  if (!ws || ws_bytes < sl.total) {
    set_error("solve_w: workspace too small (%zu < %zu bytes)", ws_bytes, sl.total);
    return GPP_ERR_WORKSPACE;
  }
  const float* Linv = reinterpret_cast<const float*>(static_cast<const char*>(state) + f.off_linv);
  char* base = static_cast<char*>(ws);
  float* T1 = reinterpret_cast<float*>(base + sl.off_t1);
  double* part = reinterpret_cast<double*>(base + sl.off_part);
  void* tnws = base + sl.off_tn;
  const int Qp = f.Qp;
  if (tc_blockgemm_supported(Q, Q, L) && tc_pass1_supported(Q, Q, L)) {
    // tensor cores (3xTF32): T1 = Linv . C as a row GEMM, W = (v0/vn) Linv^T T1 as a transposed-A GEMM
    TcBlockGemm g{};
    g.wide_range = 1;
    g.n = Q; g.n_last = Q; g.K = Q; g.ncols = L; g.batches = 1; g.tri_a = 1; g.alpha = 1.f;
    uint32_t* amax = reinterpret_cast<uint32_t*>(base + sl.off_amax);   // {1 (Linv), max|C|}
    GPP_TRY(tc_absmax(C, ldc, Q, L, amax + 1, st));
    amax_slots_kernel<<<1, 32, 0, st>>>(amax, 1);
    GPP_LAUNCH_CHECK();
    if (sl.ksplit > 1) {
      float* T1p = reinterpret_cast<float*>(base + sl.off_t1p);
      const int Kc = Q / sl.ksplit;
      g.K = Kc; g.batches = sl.ksplit; g.tri_a = 0;
      g.a_k_step = Kc; g.b_k_step = Kc; g.out_step = (int64_t)Q * L;      // same rows of Linv, next slice of its columns
      GPP_TRY(launch_tc_blockgemm(Linv, Q, Q, Qp, C, Q, L, ldc, T1p, L, g, amax, st));
      const int64_t n4 = (int64_t)Q * L / 4;
      sum_slices_kernel<<<(unsigned)((n4 + 255) / 256), 256, 0, st>>>(T1p, sl.ksplit, n4, T1);
      GPP_LAUNCH_CHECK();
    } else {
      GPP_TRY(launch_tc_blockgemm(Linv, Q, Q, Qp, C, Q, L, ldc, T1, L, g, amax, st));
    }
    GPP_TRY(launch_tc_pass1(Linv, Qp, T1, L, Q, Q, L, nullptr, 0, W, ldw, scal, tnws, sl.tn_bytes, true, st));
  } else {
    GemmParams g{};
    g.A = Linv; g.lda = Qp; g.B = C; g.ldb = ldc; g.C = T1; g.ldc = L;
    g.M = Q; g.N = L; g.K = Q; g.M_last = -1; g.alpha = 1.f; g.beta = 0.f; g.tri_a = 1;
    GPP_TRY(launch_gemm(g, false, true, 1, st));  // T1 = Linv . C
    GPP_TRY(launch_tn(Linv, Qp, Q, nullptr, 0, 0, T1, L, L, Q, 0, nullptr, 0, W, ldw, scal, tnws, sl.tn_bytes, st));
  }
  sumsq_partial_kernel<<<kSumsqBlocks, 256, 0, st>>>(W, ldw, Q, L, part);
  GPP_LAUNCH_CHECK();
  solve_scalars_kernel<<<1, 256, 0, st>>>(L_true, n_total, part, kSumsqBlocks, scal);
  GPP_LAUNCH_CHECK();
  return GPP_OK;
}

size_t solve_blocks_workspace_bytes(int Q, int L, int k) {
  return align_up(solve_layout(Q, L).total, 256) + align_up((size_t)kSumsqBlocks * k * sizeof(double), 256);
}

// The state of launch_factor_blocks holds Linv D, so the single-design solve yields W = D B^-1 D C / vn; then
// blk[2i + 1] = ||W_i||^2 over row block i.
int launch_solve_w_blocks(const float* C, int64_t ldc, const BlockSpec& bs, int L, int L_true, int64_t n_total, float* W,
                          int64_t ldw, double* scal, double* blk, const void* state, size_t state_bytes, void* ws,
                          size_t ws_bytes, cudaStream_t st) {
  const int Q = bs.start[bs.k];
  if (!state || state_bytes < factor_blocks_workspace_bytes(Q, bs.k)) {
    set_error("solve_w_blocks: factorisation state too small (%zu < %zu bytes)", state_bytes,
              factor_blocks_workspace_bytes(Q, bs.k));
    return GPP_ERR_WORKSPACE;
  }
  if (!ws || ws_bytes < solve_blocks_workspace_bytes(Q, L, bs.k)) {
    set_error("solve_w_blocks: workspace too small (%zu < %zu bytes)", ws_bytes, solve_blocks_workspace_bytes(Q, L, bs.k));
    return GPP_ERR_WORKSPACE;
  }
  const size_t off = align_up(solve_layout(Q, L).total, 256);
  GPP_TRY(launch_solve_w(C, ldc, Q, L, L_true, n_total, W, ldw, scal, state, state_bytes, ws, off, st));
  double* bpart = reinterpret_cast<double*>(static_cast<char*>(ws) + off);
  block_sumsq_partial_kernel<<<kSumsqBlocks, 256, 0, st>>>(W, ldw, Q, L, bs, 0, bpart);
  GPP_LAUNCH_CHECK();
  block_reduce_kernel<<<1, 256, 0, st>>>(bpart, kSumsqBlocks, bs.k, 1, blk);
  GPP_LAUNCH_CHECK();
  return GPP_OK;
}

}  // namespace gpp
