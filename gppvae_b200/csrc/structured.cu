// Structured (never-materialised) Khatri-Rao path -- SURVEY.md section 8(f) row 4.
//
// V[i, j q + k] = xn[d_i, j] wn[w_i, k] (vmod.py:28-35) has only P x p + nviews x q free numbers, and every sum over
// the rows of V factors through the (object, view) slots:
//
//   G = V^T V      G[(j,k),(j',k')] = sum_v wn[v,k] wn[v,k'] S_v[j,j'],   S_v = xn^T diag(cnt[:, v]) xn      (p x p)
//   C = V^T X      C[(j,k), l]      = sum_v wn[v,k] T_v[j,l],             T_v = xn^T Xs_v                      (p x L)
//   V W            (V W)[i, :]      = Y[d_i, w_i L ..],   Y = xn [M_0 | M_1 | ...],  M_v[j,l] = sum_k wn[v,k] W[(j,k),l]
//
// with cnt[o, v] = number of rows in slot (o, v) and Xs_v[o, :] = the sum of the rows of X in that slot.  S and T are
// ONE tall-skinny GEMM  xn^T [cnt (x) xn | Xs]  over the P objects, Y is one (P x p)(p x nviews L) GEMM -- both run on
// the tensor-core kernels of gemm_tc.cu -- so the GP term costs O(P p nviews (p + L)) instead of O(N Q (Q + L)) flops
// (c3: 1.3e11 instead of 1.9e13) and V (16 GB at c3) is never written.  What remains per row of X is streaming:
// the slot sums (read X once) and the epilogue Xb = (X - gather(Y)) / vn (read X, read Y, write Xb).
//
// The slot sums are deterministic: the Python layer sorts the rows by slot once per (d, w) (index preparation, the
// data set does not change between epochs, train_gppvae.py:123-126) and kr_slot_sum_kernel adds each slot's rows in
// that fixed order -- no atomics.
#include "common.cuh"
#include "kernels.h"

namespace gpp {

// XZ[o, zcol0 + v L + l] = sum over the rows i of slot s = o nviews + v (order[slot_start[s] .. slot_start[s+1]))
// of X[i, l];  XZ[o, v p + j] = cnt[s] xn[o, j].  One warp per slot.
__global__ void __launch_bounds__(256) kr_slot_sum_kernel(const float* __restrict__ X, int64_t ldx,
                                                          const int64_t* __restrict__ order,
                                                          const int64_t* __restrict__ slot_start,
                                                          const float* __restrict__ xn, int64_t P, int p, int nviews,
                                                          int L, int with_x, float* __restrict__ XZ, int64_t ldxz) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  const int zcol0 = with_x ? nviews * p : 0;
  for (int64_t s = warp; s < P * nviews; s += nwarps) {
    const int64_t o = s / nviews;
    const int v = (int)(s - o * nviews);
    const int64_t b = slot_start[s], e = slot_start[s + 1];
    float* zrow = XZ + o * ldxz + zcol0 + (int64_t)v * L;
    for (int c = lane * 4; c < L; c += 128) {
      float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
      for (int64_t t = b; t < e; ++t) {
        const float4 x = *reinterpret_cast<const float4*>(X + order[t] * ldx + c);
        acc.x += x.x; acc.y += x.y; acc.z += x.z; acc.w += x.w;
      }
      *reinterpret_cast<float4*>(zrow + c) = acc;
    }
    if (!with_x) continue;
    const float cnt = (float)(e - b);
    float* xrow = XZ + o * ldxz + (int64_t)v * p;
    for (int c = lane * 4; c < p; c += 128) {
      const float4 x = *reinterpret_cast<const float4*>(xn + o * p + c);
      *reinterpret_cast<float4*>(xrow + c) = make_float4(cnt * x.x, cnt * x.y, cnt * x.z, cnt * x.w);
    }
  }
}

// GC (Q x (Q + L), ld = ldgc) from ST (p x nviews (p + L), ld = ldst): see the header of this file.
// One thread per float4 of a GC row; the view weights of the row's k sit in registers.
__global__ void __launch_bounds__(256) kr_assemble_gc_kernel(const float* __restrict__ ST, int64_t ldst,
                                                             const float* __restrict__ wn, int p, int q, int nviews,
                                                             int L, int with_g, float* __restrict__ GC, int64_t ldgc) {
  extern __shared__ float wsm[];   // wn, nviews x q
  for (int e = threadIdx.x; e < nviews * q; e += blockDim.x) wsm[e] = wn[e];
  __syncthreads();
  const int Q = with_g ? p * q : 0;       // columns of the G part in GC (0: GC is C alone, ST holds only T)
  const int r = blockIdx.x;               // GC row (j, k)
  const int j = r / q, k = r - j * q;
  const int zcol0 = with_g ? nviews * p : 0;
  const int ncol4 = (Q + L) >> 2;
  for (int c4 = threadIdx.x; c4 < ncol4; c4 += blockDim.x) {
    const int c = c4 << 2;
    float o[4] = {0.f, 0.f, 0.f, 0.f};
    if (c < Q) {
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int cc = c + e, j2 = cc / q, k2 = cc - j2 * q;
        float s = 0.f;
        for (int v = 0; v < nviews; ++v) s = fmaf(wsm[v * q + k] * wsm[v * q + k2], ST[(int64_t)j * ldst + v * p + j2], s);
        o[e] = s;
      }
    } else {
      const int l = c - Q;
      for (int v = 0; v < nviews; ++v) {
        const float4 t = *reinterpret_cast<const float4*>(ST + (int64_t)j * ldst + zcol0 + (int64_t)v * L + l);
        const float wk = wsm[v * q + k];
        o[0] = fmaf(wk, t.x, o[0]); o[1] = fmaf(wk, t.y, o[1]); o[2] = fmaf(wk, t.z, o[2]); o[3] = fmaf(wk, t.w, o[3]);
      }
    }
    *reinterpret_cast<float4*>(GC + (int64_t)r * ldgc + c) = make_float4(o[0], o[1], o[2], o[3]);
  }
}

// M (p x nviews L, ld = ldm):  M[j, v L + l] = sum_k wn[v, k] W[(j, k), l]
__global__ void __launch_bounds__(256) kr_assemble_m_kernel(const float* __restrict__ W, int64_t ldw,
                                                            const float* __restrict__ wn, int p, int q, int nviews,
                                                            int L, float* __restrict__ M, int64_t ldm) {
  const int j = blockIdx.x;
  const int n4 = (nviews * L) >> 2;
  for (int c4 = threadIdx.x; c4 < n4; c4 += blockDim.x) {
    const int c = c4 << 2, v = c / L, l = c - v * L;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int k = 0; k < q; ++k) {
      const float wk = wn[v * q + k];
      const float4 x = *reinterpret_cast<const float4*>(W + (int64_t)(j * q + k) * ldw + l);
      acc.x = fmaf(wk, x.x, acc.x); acc.y = fmaf(wk, x.y, acc.y); acc.z = fmaf(wk, x.z, acc.z); acc.w = fmaf(wk, x.w, acc.w);
    }
    *reinterpret_cast<float4*>(M + (int64_t)j * ldm + c) = acc;
  }
}

// Epilogue of the structured pass 2: Xb_i = (X_i - Y[d_i, w_i L ..]) / vn, quad_i = X_i . Xb_i, per-block sum Xb^2.
// One warp per row.
__global__ void __launch_bounds__(256) kr_xb_kernel(const float* __restrict__ X, int64_t ldx, const float* __restrict__ Y,
                                                    int64_t ldy, const int64_t* __restrict__ d,
                                                    const int64_t* __restrict__ w, int64_t n, int64_t P, int nviews, int L,
                                                    const double* __restrict__ scal, float* __restrict__ Xb, int64_t ldxb,
                                                    float* __restrict__ quad, double* __restrict__ xb2_part) {
  __shared__ double red[8];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int64_t warp = (int64_t)blockIdx.x * 8 + wib, nwarps = (int64_t)gridDim.x * 8;
  const float inv_vn = (float)(1.0 / scal[GPP_S_VN]);
  const float qnan = __int_as_float(0x7fc00000);
  double xb2 = 0;
  for (int64_t i = warp; i < n; i += nwarps) {
    const int64_t di = d[i], wi = w[i];
    const bool ok = (di >= 0) & (di < P) & (wi >= 0) & (wi < nviews);
    const float* y = Y + (ok ? di * ldy + wi * L : 0);
    float qs = 0.f, x2 = 0.f;
    for (int c = lane * 4; c < L; c += 128) {
      const float4 x = *reinterpret_cast<const float4*>(X + i * ldx + c);
      const float4 yy = *reinterpret_cast<const float4*>(y + c);
      float4 o;
      o.x = ok ? (x.x - yy.x) * inv_vn : qnan; o.y = ok ? (x.y - yy.y) * inv_vn : qnan;
      o.z = ok ? (x.z - yy.z) * inv_vn : qnan; o.w = ok ? (x.w - yy.w) * inv_vn : qnan;
      *reinterpret_cast<float4*>(Xb + i * ldxb + c) = o;
      qs = fmaf(x.x, o.x, qs); qs = fmaf(x.y, o.y, qs); qs = fmaf(x.z, o.z, qs); qs = fmaf(x.w, o.w, qs);
      x2 = fmaf(o.x, o.x, x2); x2 = fmaf(o.y, o.y, x2); x2 = fmaf(o.z, o.z, x2); x2 = fmaf(o.w, o.w, x2);
    }
    qs = warp_sum(qs);
    x2 = warp_sum(x2);
    if (lane == 0) quad[i] = qs;
    xb2 += (double)x2;
  }
  if (lane == 0) red[wib] = xb2;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0;
    for (int k = 0; k < 8; ++k) t += red[k];
    xb2_part[blockIdx.x] = t;
  }
}

constexpr int kKrXbBlocks = 1184;   // 8 x 148

// ---------------------------------------------------------------- several factored designs (GP(n_rand_effs = k))
// Object-only x^[d] and view-only w^[w] designs are slot functions too.  Beside S_v and T_v they need the per-view
// first moments  z_v = sum_{i: w_i = v} X_i (L),  a_v = x^T cnt_v (p),  n_v = sum_o cnt[o, v]:
// every block of GC = V^T [V | X] for V = [V_K | V_O | V_W] (any order, each kind at most once) is then a sum over v
// of (row weight) (column weight) (S_v, a_v or n_v), the weight being wn[v, k] for a K or W index and 1 for an O index.
struct EffLayout {
  int k;
  int kind[3];   // GPP_EFFECT_*
  int off[4];    // first column of every block, off[k] = Q
};

// Row or column t of the stacked design: its kind, its object column j (-1 for a W index) and its view column k
// (-1 for an O index); a W index at or past q is padding (kind = -1: an exactly zero row / column).
__device__ __forceinline__ void eff_decode(const EffLayout& lay, int t, int q, int& kind, int& j, int& kk) {
  int b = 0;
  while (b + 1 < lay.k && t >= lay.off[b + 1]) ++b;
  const int u = t - lay.off[b];
  kind = lay.kind[b];
  if (kind == GPP_EFFECT_KR) { j = u / q; kk = u - j * q; }
  else if (kind == GPP_EFFECT_OBJECT) { j = u; kk = -1; }
  else { j = -1; kk = u; if (u >= q) kind = -1; }
}

// Partials of the per-view moments.  Block (c, v) walks the objects of chunk c in order and, for each, the rows of
// slot (o, v) in slot order; part[(c nviews + v) ldp + ...] = [z (L) | a (p) | n, 0, 0, 0].  Four rows are loaded
// before they are added (in row order), so the sums do not depend on the launch.
__global__ void __launch_bounds__(256) kr_view_sums_partial_kernel(const float* __restrict__ X, int64_t ldx,
                                                                    const int64_t* __restrict__ order,
                                                                    const int64_t* __restrict__ slot_start,
                                                                    const float* __restrict__ xn, int64_t P, int p,
                                                                    int nviews, int L, int with_x, int64_t chunk,
                                                                    float* __restrict__ part, int64_t ldp) {
  const int v = blockIdx.y;
  const int64_t o0 = (int64_t)blockIdx.x * chunk, o1 = (o0 + chunk < P) ? o0 + chunk : P;
  float* out = part + ((int64_t)blockIdx.x * nviews + v) * ldp;
  for (int c = threadIdx.x * 4; c < L; c += blockDim.x * 4) {
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int64_t o = o0; o < o1; ++o) {
      const int64_t s = o * nviews + v;
      int64_t t = slot_start[s];
      const int64_t e = slot_start[s + 1];
      for (; t + 4 <= e; t += 4) {
        float4 x[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) x[u] = *reinterpret_cast<const float4*>(X + order[t + u] * ldx + c);
#pragma unroll
        for (int u = 0; u < 4; ++u) { acc.x += x[u].x; acc.y += x[u].y; acc.z += x[u].z; acc.w += x[u].w; }
      }
      for (; t < e; ++t) {
        const float4 x = *reinterpret_cast<const float4*>(X + order[t] * ldx + c);
        acc.x += x.x; acc.y += x.y; acc.z += x.z; acc.w += x.w;
      }
    }
    *reinterpret_cast<float4*>(out + c) = acc;
  }
  if (!with_x) return;
  for (int c = threadIdx.x * 4; c < p; c += blockDim.x * 4) {
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int64_t o = o0; o < o1; ++o) {
      const int64_t s = o * nviews + v;
      const float cnt = (float)(slot_start[s + 1] - slot_start[s]);
      const float4 x = *reinterpret_cast<const float4*>(xn + o * p + c);
      acc.x = fmaf(cnt, x.x, acc.x); acc.y = fmaf(cnt, x.y, acc.y); acc.z = fmaf(cnt, x.z, acc.z); acc.w = fmaf(cnt, x.w, acc.w);
    }
    *reinterpret_cast<float4*>(out + L + c) = acc;
  }
  if (threadIdx.x == 0) {
    int64_t n = 0;
    for (int64_t o = o0; o < o1; ++o) n += slot_start[o * nviews + v + 1] - slot_start[o * nviews + v];
    *reinterpret_cast<float4*>(out + L + p) = make_float4((float)n, 0.f, 0.f, 0.f);
  }
}

// VM[v, c] = sum over the chunks, in chunk order, of the partials (n_v in double: an exact count).
__global__ void __launch_bounds__(256) kr_view_sums_reduce_kernel(const float* __restrict__ part, int64_t ldp,
                                                                   int nchunks, int nviews, int width, int ncnt,
                                                                   float* __restrict__ VM, int64_t ldvm) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= (int64_t)nviews * width) return;
  const int v = (int)(e / width), c = (int)(e - (int64_t)v * width);
  if (c == ncnt) {
    double n = 0;
    for (int ch = 0; ch < nchunks; ++ch) n += (double)part[((int64_t)ch * nviews + v) * ldp + c];
    VM[(int64_t)v * ldvm + c] = (float)n;
    return;
  }
  float s = 0.f;
  for (int ch = 0; ch < nchunks; ++ch) s += part[((int64_t)ch * nviews + v) * ldp + c];
  VM[(int64_t)v * ldvm + c] = s;
}

// The stacked GC (Q x ((with_g ? Q : 0) + L)) of the layout from ST (as kr_assemble_gc reads it) and VM
// (nviews rows [z_v | a_v | n_v]).  One block per GC row; wn in shared memory.
__global__ void __launch_bounds__(256) kr_assemble_gc_blocks_kernel(const float* __restrict__ ST, int64_t ldst,
                                                                    const float* __restrict__ VM, int64_t ldvm,
                                                                    const float* __restrict__ wn, int p, int q,
                                                                    int nviews, int L, int with_g, EffLayout lay,
                                                                    float* __restrict__ GC, int64_t ldgc) {
  extern __shared__ float wsm[];   // wn, nviews x q
  for (int e = threadIdx.x; e < nviews * q; e += blockDim.x) wsm[e] = wn[e];
  __syncthreads();
  const int Q = lay.off[lay.k];
  const int Qg = with_g ? Q : 0;
  const int zcol0 = with_g ? nviews * p : 0;
  const int r = blockIdx.x;
  int rkind, rj, rk;
  eff_decode(lay, r, q, rkind, rj, rk);
  const int ncol4 = (Qg + L) >> 2;
  for (int c4 = threadIdx.x; c4 < ncol4; c4 += blockDim.x) {
    const int c = c4 << 2;
    float o[4] = {0.f, 0.f, 0.f, 0.f};
    if (rkind < 0) {
      // padding row of the view block: exactly zero
    } else if (c < Qg) {
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        int ckind, cj, ck;
        eff_decode(lay, c + e, q, ckind, cj, ck);
        if (ckind < 0) continue;
        float s = 0.f;
        for (int v = 0; v < nviews; ++v) {
          const float wr = rk >= 0 ? wsm[v * q + rk] : 1.f;
          const float wc = ck >= 0 ? wsm[v * q + ck] : 1.f;
          float base;
          if (rj >= 0 && cj >= 0) base = ST[(int64_t)rj * ldst + v * p + cj];
          else if (rj >= 0) base = VM[(int64_t)v * ldvm + L + rj];
          else if (cj >= 0) base = VM[(int64_t)v * ldvm + L + cj];
          else base = VM[(int64_t)v * ldvm + L + p];
          s = fmaf(wr * wc, base, s);
        }
        o[e] = s;
      }
    } else {
      const int l = c - Qg;
      for (int v = 0; v < nviews; ++v) {
        const float4 t = rj >= 0 ? *reinterpret_cast<const float4*>(ST + (int64_t)rj * ldst + zcol0 + (int64_t)v * L + l)
                                 : *reinterpret_cast<const float4*>(VM + (int64_t)v * ldvm + l);
        const float wk = rk >= 0 ? wsm[v * q + rk] : 1.f;
        o[0] = fmaf(wk, t.x, o[0]); o[1] = fmaf(wk, t.y, o[1]); o[2] = fmaf(wk, t.z, o[2]); o[3] = fmaf(wk, t.w, o[3]);
      }
    }
    *reinterpret_cast<float4*>(GC + (int64_t)r * ldgc + c) = make_float4(o[0], o[1], o[2], o[3]);
  }
}

// Blocks 0 .. p-1: M[j, v L + l] = sum_k wn[v,k] W_K[(j,k), l] + W_O[j, l];  blocks p .. p + nviews - 1:
// R[v, l] = sum_k wn[v,k] W_W[k, l].  offK / offO / offW: the row of W where the block starts, -1 when absent.
__global__ void __launch_bounds__(256) kr_assemble_m_blocks_kernel(const float* __restrict__ W, int64_t ldw,
                                                                   const float* __restrict__ wn, int p, int q,
                                                                   int nviews, int L, int offK, int offO, int offW,
                                                                   float* __restrict__ M, int64_t ldm,
                                                                   float* __restrict__ R, int64_t ldr) {
  const int L4 = L >> 2;
  if ((int)blockIdx.x >= p) {
    const int v = blockIdx.x - p;
    for (int c4 = threadIdx.x; c4 < L4; c4 += blockDim.x) {
      const int l = c4 << 2;
      float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
      for (int k = 0; k < q; ++k) {
        const float wk = wn[v * q + k];
        const float4 x = *reinterpret_cast<const float4*>(W + (int64_t)(offW + k) * ldw + l);
        acc.x = fmaf(wk, x.x, acc.x); acc.y = fmaf(wk, x.y, acc.y); acc.z = fmaf(wk, x.z, acc.z); acc.w = fmaf(wk, x.w, acc.w);
      }
      *reinterpret_cast<float4*>(R + (int64_t)v * ldr + l) = acc;
    }
    return;
  }
  const int j = blockIdx.x;
  for (int c4 = threadIdx.x; c4 < nviews * L4; c4 += blockDim.x) {
    const int c = c4 << 2, v = c / L, l = c - v * L;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    if (offK >= 0) {
      for (int k = 0; k < q; ++k) {
        const float wk = wn[v * q + k];
        const float4 x = *reinterpret_cast<const float4*>(W + (int64_t)(offK + j * q + k) * ldw + l);
        acc.x = fmaf(wk, x.x, acc.x); acc.y = fmaf(wk, x.y, acc.y); acc.z = fmaf(wk, x.z, acc.z); acc.w = fmaf(wk, x.w, acc.w);
      }
    }
    if (offO >= 0) {
      const float4 x = *reinterpret_cast<const float4*>(W + (int64_t)(offO + j) * ldw + l);
      acc.x += x.x; acc.y += x.y; acc.z += x.z; acc.w += x.w;
    }
    *reinterpret_cast<float4*>(M + (int64_t)j * ldm + c) = acc;
  }
}

// kr_xb_kernel with the per-view row: Xb_i = (X_i - Y[d_i, w_i L ..] - R[w_i]) / vn.
__global__ void __launch_bounds__(256) kr_xb_views_kernel(const float* __restrict__ X, int64_t ldx,
                                                          const float* __restrict__ Y, int64_t ldy,
                                                          const float* __restrict__ R, int64_t ldr,
                                                          const int64_t* __restrict__ d, const int64_t* __restrict__ w,
                                                          int64_t n, int64_t P, int nviews, int L,
                                                          const double* __restrict__ scal, float* __restrict__ Xb,
                                                          int64_t ldxb, float* __restrict__ quad,
                                                          double* __restrict__ xb2_part) {
  __shared__ double red[8];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int64_t warp = (int64_t)blockIdx.x * 8 + wib, nwarps = (int64_t)gridDim.x * 8;
  const float inv_vn = (float)(1.0 / scal[GPP_S_VN]);
  const float qnan = __int_as_float(0x7fc00000);
  double xb2 = 0;
  for (int64_t i = warp; i < n; i += nwarps) {
    const int64_t di = d[i], wi = w[i];
    const bool ok = (di >= 0) & (di < P) & (wi >= 0) & (wi < nviews);
    const float* y = Y + (ok ? di * ldy + wi * L : 0);
    const float* rr = R + (ok ? wi * ldr : 0);
    float qs = 0.f, x2 = 0.f;
    for (int c = lane * 4; c < L; c += 128) {
      const float4 x = *reinterpret_cast<const float4*>(X + i * ldx + c);
      const float4 yy = *reinterpret_cast<const float4*>(y + c);
      const float4 r4 = *reinterpret_cast<const float4*>(rr + c);
      float4 o;
      o.x = ok ? (x.x - (yy.x + r4.x)) * inv_vn : qnan; o.y = ok ? (x.y - (yy.y + r4.y)) * inv_vn : qnan;
      o.z = ok ? (x.z - (yy.z + r4.z)) * inv_vn : qnan; o.w = ok ? (x.w - (yy.w + r4.w)) * inv_vn : qnan;
      *reinterpret_cast<float4*>(Xb + i * ldxb + c) = o;
      qs = fmaf(x.x, o.x, qs); qs = fmaf(x.y, o.y, qs); qs = fmaf(x.z, o.z, qs); qs = fmaf(x.w, o.w, qs);
      x2 = fmaf(o.x, o.x, x2); x2 = fmaf(o.y, o.y, x2); x2 = fmaf(o.z, o.z, x2); x2 = fmaf(o.w, o.w, x2);
    }
    qs = warp_sum(qs);
    x2 = warp_sum(x2);
    if (lane == 0) quad[i] = qs;
    xb2 += (double)x2;
  }
  if (lane == 0) red[wib] = xb2;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0;
    for (int k = 0; k < 8; ++k) t += red[k];
    xb2_part[blockIdx.x] = t;
  }
}

// ---------------------------------------------------------------- NLL gradient to the tables (DESIGN 5.8)
// Both entries walk B^-1 in tiles of q rows (j', .) by jc q columns (j0 .. j0 + jc, .): a tile is staged in shared memory
// once (row stride jc q + 1, so that lanes walking k' hit distinct banks) and every view is served from it.
inline int grad_tile_jc(int p, int q) {
  const int jc = 4096 / (q * q);
  return jc < 1 ? 1 : (jc > p ? p : jc);
}
inline size_t grad_smem_bytes(int p, int q, int nviews) {
  const int jc = grad_tile_jc(p, q);
  return ((size_t)nviews * q + (size_t)q * (jc * q + 1)) * sizeof(float);
}
constexpr size_t kGradSmemMax = 160 * 1024;

__device__ __forceinline__ void grad_stage_tile(const float* __restrict__ Binv, int64_t ldb, int jp, int j0, int nj, int q,
                                                float* tile, int ts) {
  const int tw = nj * q;
  for (int e = threadIdx.x; e < q * tw; e += blockDim.x) {
    const int kk = e / tw, c = e - kk * tw;
    tile[kk * ts + c] = Binv[(int64_t)(jp * q + kk) * ldb + (int64_t)j0 * q + c];
  }
}

// R[v p + j', j] = alpha sum_{k', k} wn[v,k'] Binv[(j',k'), (j,k)] wn[v,k]  (alpha H_v).  Block (j', chunk of jc j's);
// one warp per (view, j), lanes over the q x q entries of the tile, fixed-order warp sum.
__global__ void __launch_bounds__(256) kr_grad_rhs_h_kernel(const float* __restrict__ Binv, int64_t ldb,
                                                            const float* __restrict__ wn, int p, int q, int nviews,
                                                            int jc, double alpha, float* __restrict__ R, int64_t ldr) {
  extern __shared__ float gsm[];
  float* wsm = gsm;                     // wn, nviews x q
  float* tile = gsm + nviews * q;       // q x (jc q + 1)
  const int jp = blockIdx.x, j0 = blockIdx.y * jc, nj = (p - j0 < jc) ? p - j0 : jc;
  const int ts = jc * q + 1;
  for (int e = threadIdx.x; e < nviews * q; e += blockDim.x) wsm[e] = wn[e];
  grad_stage_tile(Binv, ldb, jp, j0, nj, q, tile, ts);
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  for (int pr = warp; pr < nviews * nj; pr += nw) {
    const int v = pr / nj, jj = pr - v * nj;
    const float* wv = wsm + v * q;
    float s = 0.f;
    for (int e = lane; e < q * q; e += 32) {
      const int kk = e / q, k = e - kk * q;
      s = fmaf(wv[kk] * wv[k], tile[kk * ts + jj * q + k], s);
    }
    s = warp_sum(s);
    if (lane == 0) R[(int64_t)(v * p + jp) * ldr + j0 + jj] = (float)(alpha * (double)s);
  }
}

// R[nviews p + v L + l, j] = -sum_k wn[v,k] W[(j,k), l]  (-M_v^T; the sum of kr_assemble_m_kernel, in its order).
__global__ void __launch_bounds__(256) kr_grad_rhs_m_kernel(const float* __restrict__ W, int64_t ldw,
                                                            const float* __restrict__ wn, int p, int q, int nviews, int L,
                                                            float* __restrict__ R, int64_t ldr) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= (int64_t)nviews * L * p) return;
  const int64_t row = e / p;
  const int j = (int)(e - row * p), v = (int)(row / L), l = (int)(row - (int64_t)v * L);
  float s = 0.f;
  for (int k = 0; k < q; ++k) s = fmaf(wn[v * q + k], W[(int64_t)(j * q + k) * ldw + l], s);
  R[((int64_t)nviews * p + row) * ldr + j] = -s;
}

// part[j' nviews q + v q + k] = alpha sum_{j, k'} S_v[j, j'] wn[v,k'] Binv[(j',k'), (j,k)] - sum_l T_v[j',l] W[(j',k), l]
// with S_v[j, j'] = ST[j, v p + j'] and T_v[j', l] = ST[j', nviews p + v L + l].  Block j' walks its q rows of B^-1 in
// tiles; one warp per (view, k), lanes over (j, k') of the tile; a pair's sums over the tiles add in tile order.
__global__ void __launch_bounds__(256) kr_grad_views_part_kernel(const float* __restrict__ ST, int64_t ldst,
                                                                 const float* __restrict__ Binv, int64_t ldb,
                                                                 const float* __restrict__ W, int64_t ldw,
                                                                 const float* __restrict__ wn, int p, int q, int nviews,
                                                                 int L, int jc, double alpha, float* __restrict__ part) {
  extern __shared__ float gsm[];
  float* wsm = gsm;                     // wn, nviews x q
  float* tile = gsm + nviews * q;       // q x (jc q + 1)
  const int jp = blockIdx.x, ts = jc * q + 1;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const int npairs = nviews * q;
  float* out = part + (int64_t)jp * npairs;
  for (int e = threadIdx.x; e < nviews * q; e += blockDim.x) wsm[e] = wn[e];
  for (int j0 = 0; j0 < p; j0 += jc) {
    const int nj = (p - j0 < jc) ? p - j0 : jc;
    __syncthreads();                    // the previous tile is consumed
    grad_stage_tile(Binv, ldb, jp, j0, nj, q, tile, ts);
    __syncthreads();
    for (int pr = warp; pr < npairs; pr += nw) {
      const int v = pr / q, k = pr - v * q;
      const float* wv = wsm + v * q;
      float s = 0.f;
      for (int e = lane; e < nj * q; e += 32) {
        const int jj = e / q, kk = e - jj * q;
        s = fmaf(ST[(int64_t)(j0 + jj) * ldst + v * p + jp] * wv[kk], tile[kk * ts + jj * q + k], s);
      }
      s = warp_sum(s);
      if (lane == 0) out[pr] = (j0 == 0 ? 0.f : out[pr]) + s;   // only this lane of this block touches out[pr]
    }
  }
  for (int pr = warp; pr < npairs; pr += nw) {
    const int v = pr / q, k = pr - v * q;
    const float* t = ST + (int64_t)jp * ldst + (int64_t)nviews * p + (int64_t)v * L;
    const float* wr = W + (int64_t)(jp * q + k) * ldw;
    float s = 0.f;
    for (int l = lane; l < L; l += 32) s = fmaf(t[l], wr[l], s);
    s = warp_sum(s);
    if (lane == 0) out[pr] = (float)(alpha * (double)out[pr]) - s;
  }
}

// gw[v, k] = sum over j' of part[j'][v, k]: one warp per (v, k), lanes over j', fixed-order warp sum.
__global__ void __launch_bounds__(256) kr_grad_views_reduce_kernel(const float* __restrict__ part, int p, int npairs,
                                                                   int q, float* __restrict__ gw, int64_t ldgw) {
  const int lane = threadIdx.x & 31;
  const int pr = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (pr >= npairs) return;
  float s = 0.f;
  for (int jp = lane; jp < p; jp += 32) s += part[(int64_t)jp * npairs + pr];
  s = warp_sum(s);
  if (lane == 0) {
    const int v = pr / q, k = pr - v * q;
    gw[(int64_t)v * ldgw + k] = s;
  }
}

// ---------------------------------------------------------------- posterior prediction at new rows (DESIGN 5.9)
// The stacked new row is u = A_v x + b_v (x = xn[o], v its view), so var* = scal[V0] (x^T H_v x + 2 x^T h_v + c_v) with
// H_v = A_v^T Binv A_v, h_v = A_v^T Binv b_v, c_v = b_v^T Binv b_v.  offK / offO / offW: first row of the K / O / W block
// in Binv, -1 when the kind is absent.  Only the q true columns of the view block are read (wn has q columns).

// H[j', v p + j] = sum_{k',k} wn[v,k'] wn[v,k] Binv[K(j',k'), K(j,k)] + sum_k' wn[v,k'] Binv[K(j',k'), O j]
//                + sum_k wn[v,k] Binv[O j', K(j,k)] + Binv[O j', O j].
// Block (j', chunk of jc j's): the KK tile is staged as in kr_grad_rhs_h_kernel and serves every view; one warp per
// (view, j), lanes over the tile and the q KO / OK terms, fixed-order warp sum, then the OO entry.
__global__ void __launch_bounds__(256) kr_predict_h_kernel(const float* __restrict__ Binv, int64_t ldb,
                                                           const float* __restrict__ wn, int p, int q, int nviews,
                                                           int jc, int offK, int offO, float* __restrict__ H,
                                                           int64_t ldh) {
  extern __shared__ float gsm[];
  float* wsm = gsm;                     // wn, nviews x q
  float* tile = gsm + nviews * q;       // q x (jc q + 1), with K only
  const int jp = blockIdx.x, j0 = blockIdx.y * jc, nj = (p - j0 < jc) ? p - j0 : jc;
  const int ts = jc * q + 1;
  for (int e = threadIdx.x; e < nviews * q; e += blockDim.x) wsm[e] = wn[e];
  if (offK >= 0) grad_stage_tile(Binv + (int64_t)offK * ldb + offK, ldb, jp, j0, nj, q, tile, ts);
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  for (int pr = warp; pr < nviews * nj; pr += nw) {
    const int v = pr / nj, jj = pr - v * nj, j = j0 + jj;
    const float* wv = wsm + v * q;
    float s = 0.f;
    if (offK >= 0) {
      for (int e = lane; e < q * q; e += 32) {
        const int kk = e / q, k = e - kk * q;
        s = fmaf(wv[kk] * wv[k], tile[kk * ts + jj * q + k], s);
      }
      if (offO >= 0) {
        for (int k = lane; k < q; k += 32) {
          s = fmaf(wv[k], Binv[(int64_t)(offK + jp * q + k) * ldb + offO + j], s);
          s = fmaf(wv[k], Binv[(int64_t)(offO + jp) * ldb + offK + j * q + k], s);
        }
      }
    }
    s = warp_sum(s);
    if (lane == 0) {
      if (offO >= 0) s += Binv[(int64_t)(offO + jp) * ldb + offO + j];
      H[(int64_t)jp * ldh + (int64_t)v * p + j] = s;
    }
  }
}

// Blocks j < p:  h[v p + j] = sum_{k,k'} wn[v,k] Binv[K(j,k), W k'] wn[v,k'] + sum_k' Binv[O j, W k'] wn[v,k'];
// block p:       c[v] = sum_{k,k'} wn[v,k] Binv[W k, W k'] wn[v,k'].
// The block stages its q x q tile of Binv (and the O row) once; one warp per view, fixed-order warp sum.
__global__ void __launch_bounds__(256) kr_predict_hc_kernel(const float* __restrict__ Binv, int64_t ldb,
                                                            const float* __restrict__ wn, int p, int q, int nviews,
                                                            int offK, int offO, int offW, float* __restrict__ h,
                                                            float* __restrict__ c) {
  extern __shared__ float gsm[];
  float* wsm = gsm;                     // wn, nviews x q
  float* tile = gsm + nviews * q;       // q x (q + 1)
  float* orow = tile + q * (q + 1);     // q
  const int j = blockIdx.x, ts = q + 1;
  const bool is_c = j == p;
  const bool with_tile = is_c || offK >= 0, with_o = !is_c && offO >= 0;
  for (int e = threadIdx.x; e < nviews * q; e += blockDim.x) wsm[e] = wn[e];
  if (is_c) grad_stage_tile(Binv + (int64_t)offW * ldb + offW, ldb, 0, 0, 1, q, tile, ts);
  else if (offK >= 0) grad_stage_tile(Binv + (int64_t)offK * ldb + offW, ldb, j, 0, 1, q, tile, ts);
  if (with_o)
    for (int e = threadIdx.x; e < q; e += blockDim.x) orow[e] = Binv[(int64_t)(offO + j) * ldb + offW + e];
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  for (int v = warp; v < nviews; v += nw) {
    const float* wv = wsm + v * q;
    float s = 0.f;
    if (with_tile) {
      for (int e = lane; e < q * q; e += 32) {
        const int kk = e / q, k = e - kk * q;
        s = fmaf(wv[kk] * wv[k], tile[kk * ts + k], s);
      }
    }
    if (with_o)
      for (int k = lane; k < q; k += 32) s = fmaf(orow[k], wv[k], s);
    s = warp_sum(s);
    if (lane == 0) {
      if (is_c) c[v] = s;
      else h[(int64_t)v * p + j] = s;
    }
  }
}

// One warp per new row i (o = d_i, v = w_i):  mean_i = Y[o, v L ..] (+ R[v]),
// var_i = scal[V0] (xn[o] . YH[o, v p ..] + 2 xn[o] . h[v] + c[v]).  Rows with an index outside the tables are NaN.
__global__ void __launch_bounds__(256) kr_predict_rows_kernel(const float* __restrict__ Y, int64_t ldy,
                                                              const float* __restrict__ R, int64_t ldr,
                                                              const float* __restrict__ YH, int64_t ldyh,
                                                              const float* __restrict__ xn,
                                                              const float* __restrict__ h, const float* __restrict__ c,
                                                              const int64_t* __restrict__ d,
                                                              const int64_t* __restrict__ w, int64_t m, int64_t P,
                                                              int p, int nviews, int L, const double* __restrict__ scal,
                                                              float* __restrict__ mean, int64_t ldmean,
                                                              float* __restrict__ var) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  const float qnan = __int_as_float(0x7fc00000);
  const double v0 = scal[GPP_S_V0];
  for (int64_t i = warp; i < m; i += nwarps) {
    const int64_t di = d[i], wi = w[i];
    const bool ok = (di >= 0) & (di < P) & (wi >= 0) & (wi < nviews);
    float* out = mean + i * ldmean;
    if (!ok) {
      for (int cc = lane * 4; cc < L; cc += 128) *reinterpret_cast<float4*>(out + cc) = make_float4(qnan, qnan, qnan, qnan);
      if (lane == 0) var[i] = qnan;
      continue;
    }
    for (int cc = lane * 4; cc < L; cc += 128) {
      float4 o;
      if (Y) {
        o = *reinterpret_cast<const float4*>(Y + di * ldy + wi * L + cc);
        if (R) {
          const float4 r4 = *reinterpret_cast<const float4*>(R + wi * ldr + cc);
          o.x += r4.x; o.y += r4.y; o.z += r4.z; o.w += r4.w;
        }
      } else {
        o = *reinterpret_cast<const float4*>(R + wi * ldr + cc);
      }
      *reinterpret_cast<float4*>(out + cc) = o;
    }
    float a = 0.f, b = 0.f;
    if (YH) {
      const float* x = xn + di * p;
      const float* yh = YH + di * ldyh + wi * p;
      for (int j = lane; j < p; j += 32) a = fmaf(x[j], yh[j], a);
      if (h)
        for (int j = lane; j < p; j += 32) b = fmaf(x[j], h[wi * p + j], b);
    }
    a = warp_sum(a);
    b = warp_sum(b);
    if (lane == 0) var[i] = (float)(v0 * (double)(a + 2.f * b + (c ? c[wi] : 0.f)));
  }
}

// out_i = scal[V0] sum_c A[i, c] B[i, c]: one warp per row, float4 lanes, fixed-order warp sum.
__global__ void __launch_bounds__(256) rows_dot_kernel(const float* __restrict__ A, int64_t lda,
                                                       const float* __restrict__ B, int64_t ldb, int64_t m, int cols,
                                                       const double* __restrict__ scal, float* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  const double v0 = scal[GPP_S_V0];
  for (int64_t i = warp; i < m; i += nwarps) {
    float s = 0.f;
    for (int cc = lane * 4; cc < cols; cc += 128) {
      const float4 a = *reinterpret_cast<const float4*>(A + i * lda + cc);
      const float4 b = *reinterpret_cast<const float4*>(B + i * ldb + cc);
      s = fmaf(a.x, b.x, s); s = fmaf(a.y, b.y, s); s = fmaf(a.z, b.z, s); s = fmaf(a.w, b.w, s);
    }
    s = warp_sum(s);
    if (lane == 0) out[i] = (float)(v0 * (double)s);
  }
}

inline size_t predict_hc_smem_bytes(int q, int nviews) {
  return ((size_t)nviews * q + (size_t)q * (q + 1) + q) * sizeof(float);
}

inline int grad_set_smem(const void* kernel, size_t smem) {
  if (smem > 48 * 1024) GPP_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  return GPP_OK;
}

// Chunks of objects per view for the moments: about 8 blocks per SM over all views, a function of the shape alone.
inline int64_t view_sums_chunks(int64_t P, int nviews) {
  const int64_t target = (1184 + nviews - 1) / nviews;
  return target < P ? target : P;
}

inline int view_sums_width(int p, int L, int with_x) { return L + (with_x ? p + 4 : 0); }

// Checks the kinds list and fills the layout (block widths p q, p, round4(q)).
inline int eff_layout(int32_t k, const int32_t* kinds_host, int p, int q, EffLayout& lay, int& has) {
  if (!(k >= 1 && k <= 3 && kinds_host)) return 0;
  lay.k = k;
  has = 0;
  int off = 0;
  for (int b = 0; b < k; ++b) {
    const int kd = kinds_host[b];
    if (kd < GPP_EFFECT_KR || kd > GPP_EFFECT_VIEW || (has & (1 << kd))) return 0;
    has |= 1 << kd;
    lay.kind[b] = kd;
    lay.off[b] = off;
    off += kd == GPP_EFFECT_KR ? p * q : kd == GPP_EFFECT_OBJECT ? p : (q + 3) / 4 * 4;
  }
  lay.off[k] = off;
  return 1;
}

}  // namespace gpp

using namespace gpp;

extern "C" int gpp_kr_slot_sums(const float* X, int64_t ldx, const int64_t* order, const int64_t* slot_start,
                                const float* xn, int64_t P, int32_t p, int32_t nviews, int32_t L, int32_t with_x,
                                float* XZ, int64_t ldxz, gpp_stream_t stream) {
  GPP_REQUIRE(X && order && slot_start && xn && XZ, "kr_slot_sums: null pointer");
  GPP_REQUIRE(P > 0 && p > 0 && nviews > 0 && L > 0 && p % 4 == 0 && L % 4 == 0, "kr_slot_sums: p and L must be multiples of 4");
  GPP_REQUIRE(ldx >= L && ldx % 4 == 0 && ldxz >= (int64_t)nviews * ((with_x ? p : 0) + L) && ldxz % 4 == 0 && aligned16(X) &&
                  aligned16(XZ) && aligned16(xn),
              "kr_slot_sums: bad leading dimension / alignment");
  const int64_t slots = P * nviews;
  const int grid = (int)(ceil_div(slots, 8) < 8192 ? ceil_div(slots, 8) : 8192);
  kr_slot_sum_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(X, ldx, order, slot_start, xn, P, p, nviews, L, with_x, XZ,
                                                             ldxz);
  GPP_LAUNCH_CHECK();
  return GPP_OK;
}

extern "C" int gpp_kr_assemble_gc(const float* ST, int64_t ldst, const float* wn, int32_t p, int32_t q, int32_t nviews,
                                  int32_t L, int32_t with_g, float* GC, int64_t ldgc, gpp_stream_t stream) {
  GPP_REQUIRE(ST && wn && GC, "kr_assemble_gc: null pointer");
  const int64_t Q = (int64_t)p * q;
  GPP_REQUIRE(p > 0 && q > 0 && nviews > 0 && L >= 0 && Q % 4 == 0 && L % 4 == 0 && p % 4 == 0,
              "kr_assemble_gc: p, p*q and L must be multiples of 4");
  GPP_REQUIRE(ldst >= (int64_t)nviews * ((with_g ? p : 0) + L) && ldst % 4 == 0 && ldgc >= (with_g ? Q : 0) + L &&
                  ldgc % 4 == 0 && aligned16(ST) &&
                  aligned16(GC),
              "kr_assemble_gc: bad leading dimension / alignment");
  const size_t smem = (size_t)nviews * q * sizeof(float);
  GPP_REQUIRE(smem <= 48 * 1024, "kr_assemble_gc: view table too large");
  kr_assemble_gc_kernel<<<(unsigned)Q, 256, smem, (cudaStream_t)stream>>>(ST, ldst, wn, p, q, nviews, L, with_g, GC, ldgc);
  GPP_LAUNCH_CHECK();
  return GPP_OK;
}

extern "C" int gpp_kr_assemble_m(const float* W, int64_t ldw, const float* wn, int32_t p, int32_t q, int32_t nviews,
                                 int32_t L, float* M, int64_t ldm, gpp_stream_t stream) {
  GPP_REQUIRE(W && wn && M, "kr_assemble_m: null pointer");
  GPP_REQUIRE(p > 0 && q > 0 && nviews > 0 && L > 0 && L % 4 == 0, "kr_assemble_m: L must be a multiple of 4");
  GPP_REQUIRE(ldw >= L && ldw % 4 == 0 && ldm >= (int64_t)nviews * L && ldm % 4 == 0 && aligned16(W) && aligned16(M),
              "kr_assemble_m: bad leading dimension / alignment");
  kr_assemble_m_kernel<<<(unsigned)p, 256, 0, (cudaStream_t)stream>>>(W, ldw, wn, p, q, nviews, L, M, ldm);
  GPP_LAUNCH_CHECK();
  return GPP_OK;
}

extern "C" size_t gpp_kr_xb_workspace_bytes(int64_t n) {
  return align_up((size_t)(n > 0 ? n : 1) * sizeof(float), 256) + align_up((size_t)kKrXbBlocks * sizeof(double), 256) +
         xb_finalize_bytes();
}

extern "C" int gpp_kr_xb_nll(const float* X, int64_t ldx, const float* Y, int64_t ldy, const int64_t* d,
                             const int64_t* w, int64_t n, int64_t P, int32_t nviews, int32_t L, double* scal, float* Xb,
                             int64_t ldxb, float* nll, void* workspace, size_t workspace_bytes, gpp_stream_t stream) {
  GPP_REQUIRE(X && Y && d && w && scal && Xb && nll, "kr_xb_nll: null pointer");
  GPP_REQUIRE(n >= 0 && P > 0 && nviews > 0 && L > 0 && L % 4 == 0, "kr_xb_nll: bad shape");
  GPP_REQUIRE(ldx >= L && ldx % 4 == 0 && ldxb >= L && ldxb % 4 == 0 && ldy >= (int64_t)nviews * L && ldy % 4 == 0 &&
                  aligned16(X) && aligned16(Y) && aligned16(Xb),
              "kr_xb_nll: bad leading dimension / alignment");
  const size_t need = gpp_kr_xb_workspace_bytes(n);
  if (!workspace || workspace_bytes < need) {
    set_error("kr_xb_nll: workspace too small (%zu < %zu bytes)", workspace_bytes, need);
    return GPP_ERR_WORKSPACE;
  }
  char* ws = static_cast<char*>(workspace);
  float* quad = reinterpret_cast<float*>(ws);
  double* part = reinterpret_cast<double*>(ws + align_up((size_t)(n > 0 ? n : 1) * sizeof(float), 256));
  double* fin = part + align_up((size_t)kKrXbBlocks * sizeof(double), 256) / sizeof(double);
  cudaStream_t st = (cudaStream_t)stream;
  kr_xb_kernel<<<kKrXbBlocks, 256, 0, st>>>(X, ldx, Y, ldy, d, w, n, P, nviews, L, scal, Xb, ldxb, quad, part);
  GPP_LAUNCH_CHECK();
  return launch_xb_finalize(quad, 1, n, part, kKrXbBlocks, fin, scal, nll, st);
}

extern "C" size_t gpp_kr_view_sums_workspace_bytes(int64_t P, int32_t p, int32_t nviews, int32_t L, int32_t with_x) {
  if (P <= 0 || p <= 0 || nviews <= 0 || L <= 0) return 0;
  return align_up((size_t)view_sums_chunks(P, nviews) * nviews * view_sums_width(p, L, with_x) * sizeof(float), 256);
}

extern "C" int gpp_kr_view_sums(const float* X, int64_t ldx, const int64_t* order, const int64_t* slot_start,
                                const float* xn, int64_t P, int32_t p, int32_t nviews, int32_t L, int32_t with_x,
                                float* VM, int64_t ldvm, void* workspace, size_t workspace_bytes, gpp_stream_t stream) {
  GPP_REQUIRE(X && order && slot_start && VM && (xn || !with_x), "kr_view_sums: null pointer");
  GPP_REQUIRE(P > 0 && p > 0 && nviews > 0 && L > 0 && p % 4 == 0 && L % 4 == 0,
              "kr_view_sums: p and L must be positive multiples of 4");
  const int width = view_sums_width(p, L, with_x);
  GPP_REQUIRE(ldx >= L && ldx % 4 == 0 && ldvm >= width && ldvm % 4 == 0 && aligned16(X) && aligned16(VM) &&
                  (!with_x || aligned16(xn)),
              "kr_view_sums: bad leading dimension / alignment");
  const size_t need = gpp_kr_view_sums_workspace_bytes(P, p, nviews, L, with_x);
  if (!workspace || workspace_bytes < need) {
    set_error("kr_view_sums: workspace too small (%zu < %zu bytes)", workspace_bytes, need);
    return GPP_ERR_WORKSPACE;
  }
  const int64_t nch = view_sums_chunks(P, nviews);
  const int64_t chunk = ceil_div(P, nch);
  const int cols = (with_x && p > L) ? p : L;
  int threads = (int)ceil_div((int64_t)cols / 4, 32) * 32;
  threads = threads > 256 ? 256 : threads;
  float* part = static_cast<float*>(workspace);
  cudaStream_t st = (cudaStream_t)stream;
  kr_view_sums_partial_kernel<<<dim3((unsigned)nch, (unsigned)nviews), threads, 0, st>>>(
      X, ldx, order, slot_start, xn, P, p, nviews, L, with_x, chunk, part, width);
  GPP_LAUNCH_CHECK();
  const int64_t total = (int64_t)nviews * width;
  kr_view_sums_reduce_kernel<<<(unsigned)ceil_div(total, 256), 256, 0, st>>>(part, width, (int)nch, nviews, width,
                                                                            with_x ? L + p : -1, VM, ldvm);
  GPP_LAUNCH_CHECK();
  return GPP_OK;
}

extern "C" int gpp_kr_assemble_gc_blocks(const float* ST, int64_t ldst, const float* VM, int64_t ldvm, const float* wn,
                                         int32_t p, int32_t q, int32_t nviews, int32_t L, int32_t k,
                                         const int32_t* kinds_host, int32_t with_g, float* GC, int64_t ldgc,
                                         gpp_stream_t stream) {
  EffLayout lay;
  int has = 0;
  GPP_REQUIRE(p > 0 && q > 0 && nviews > 0 && L >= 0 && p % 4 == 0 && L % 4 == 0 && (L > 0 || with_g),
              "kr_assemble_gc_blocks: p and L must be multiples of 4");
  GPP_REQUIRE(eff_layout(k, kinds_host, p, q, lay, has),
              "kr_assemble_gc_blocks: kinds must list 1..3 distinct GPP_EFFECT_* values");
  const bool need_st = has & ((1 << GPP_EFFECT_KR) | (1 << GPP_EFFECT_OBJECT));
  const bool need_vm = has & (1 << GPP_EFFECT_VIEW);
  GPP_REQUIRE(wn && GC && (ST || !need_st) && (VM || !need_vm), "kr_assemble_gc_blocks: null pointer");
  const int64_t Q = lay.off[k];
  GPP_REQUIRE((!need_st || (ldst >= (int64_t)nviews * ((with_g ? p : 0) + L) && ldst % 4 == 0 && aligned16(ST))) &&
                  (!need_vm || (ldvm >= L + (with_g ? p + 4 : 0) && ldvm % 4 == 0 && aligned16(VM))) &&
                  ldgc >= (with_g ? Q : 0) + L && ldgc % 4 == 0 && aligned16(GC),
              "kr_assemble_gc_blocks: bad leading dimension / alignment");
  const size_t smem = (size_t)nviews * q * sizeof(float);
  GPP_REQUIRE(smem <= 48 * 1024, "kr_assemble_gc_blocks: view table too large");
  kr_assemble_gc_blocks_kernel<<<(unsigned)Q, 256, smem, (cudaStream_t)stream>>>(ST, ldst, VM, ldvm, wn, p, q, nviews, L,
                                                                                 with_g, lay, GC, ldgc);
  GPP_LAUNCH_CHECK();
  return GPP_OK;
}

extern "C" int gpp_kr_assemble_m_blocks(const float* W, int64_t ldw, const float* wn, int32_t p, int32_t q,
                                        int32_t nviews, int32_t L, int32_t k, const int32_t* kinds_host, float* M,
                                        int64_t ldm, float* R, int64_t ldr, gpp_stream_t stream) {
  EffLayout lay;
  int has = 0;
  GPP_REQUIRE(p > 0 && q > 0 && nviews > 0 && L > 0 && p % 4 == 0 && L % 4 == 0,
              "kr_assemble_m_blocks: p and L must be positive multiples of 4");
  GPP_REQUIRE(eff_layout(k, kinds_host, p, q, lay, has),
              "kr_assemble_m_blocks: kinds must list 1..3 distinct GPP_EFFECT_* values");
  const bool need_m = has & ((1 << GPP_EFFECT_KR) | (1 << GPP_EFFECT_OBJECT));
  const bool need_r = has & (1 << GPP_EFFECT_VIEW);
  GPP_REQUIRE(W && wn && (M || !need_m) && (R || !need_r), "kr_assemble_m_blocks: null pointer");
  GPP_REQUIRE(ldw >= L && ldw % 4 == 0 && aligned16(W) &&
                  (!need_m || (ldm >= (int64_t)nviews * L && ldm % 4 == 0 && aligned16(M))) &&
                  (!need_r || (ldr >= L && ldr % 4 == 0 && aligned16(R))),
              "kr_assemble_m_blocks: bad leading dimension / alignment");
  int off[3] = {-1, -1, -1};
  for (int b = 0; b < k; ++b) off[lay.kind[b]] = lay.off[b];
  const unsigned grid = (unsigned)((need_m ? p : 0) + (need_r ? nviews : 0));
  // without M the R blocks start at 0: shift them by passing p = 0
  kr_assemble_m_blocks_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(W, ldw, wn, need_m ? p : 0, q, nviews, L,
                                                                      off[GPP_EFFECT_KR], off[GPP_EFFECT_OBJECT],
                                                                      off[GPP_EFFECT_VIEW], M, ldm, R, ldr);
  GPP_LAUNCH_CHECK();
  return GPP_OK;
}

extern "C" int gpp_kr_xb_nll_views(const float* X, int64_t ldx, const float* Y, int64_t ldy, const float* R, int64_t ldr,
                                   const int64_t* d, const int64_t* w, int64_t n, int64_t P, int32_t nviews, int32_t L,
                                   double* scal, float* Xb, int64_t ldxb, float* nll, void* workspace,
                                   size_t workspace_bytes, gpp_stream_t stream) {
  GPP_REQUIRE(X && Y && R && d && w && scal && Xb && nll, "kr_xb_nll_views: null pointer");
  GPP_REQUIRE(n >= 0 && P > 0 && nviews > 0 && L > 0 && L % 4 == 0, "kr_xb_nll_views: bad shape");
  GPP_REQUIRE(ldx >= L && ldx % 4 == 0 && ldxb >= L && ldxb % 4 == 0 && ldy >= (int64_t)nviews * L && ldy % 4 == 0 &&
                  ldr >= L && ldr % 4 == 0 && aligned16(X) && aligned16(Y) && aligned16(R) && aligned16(Xb),
              "kr_xb_nll_views: bad leading dimension / alignment");
  const size_t need = gpp_kr_xb_workspace_bytes(n);
  if (!workspace || workspace_bytes < need) {
    set_error("kr_xb_nll_views: workspace too small (%zu < %zu bytes)", workspace_bytes, need);
    return GPP_ERR_WORKSPACE;
  }
  char* ws = static_cast<char*>(workspace);
  float* quad = reinterpret_cast<float*>(ws);
  double* part = reinterpret_cast<double*>(ws + align_up((size_t)(n > 0 ? n : 1) * sizeof(float), 256));
  double* fin = part + align_up((size_t)kKrXbBlocks * sizeof(double), 256) / sizeof(double);
  cudaStream_t st = (cudaStream_t)stream;
  kr_xb_views_kernel<<<kKrXbBlocks, 256, 0, st>>>(X, ldx, Y, ldy, R, ldr, d, w, n, P, nviews, L, scal, Xb, ldxb, quad,
                                                  part);
  GPP_LAUNCH_CHECK();
  return launch_xb_finalize(quad, 1, n, part, kKrXbBlocks, fin, scal, nll, st);
}

extern "C" int gpp_kr_grad_rhs(const float* Binv, int64_t ldb, const float* W, int64_t ldw, const float* wn, int32_t p,
                               int32_t q, int32_t nviews, int32_t L, double alpha, float* R, int64_t ldr,
                               gpp_stream_t stream) {
  GPP_REQUIRE(Binv && W && wn && R, "kr_grad_rhs: null pointer");
  GPP_REQUIRE(p > 0 && q > 0 && nviews > 0 && L > 0 && p % 4 == 0 && L % 4 == 0,
              "kr_grad_rhs: p and L must be positive multiples of 4");
  GPP_REQUIRE(ldb >= (int64_t)p * q && ldw >= L && ldr >= p, "kr_grad_rhs: bad leading dimension");
  GPP_REQUIRE((size_t)nviews * q * sizeof(float) <= 48 * 1024 && grad_smem_bytes(p, q, nviews) <= kGradSmemMax,
              "kr_grad_rhs: view table or q too large for one tile of B^-1 in shared memory");
  const int jc = grad_tile_jc(p, q);
  const size_t smem = grad_smem_bytes(p, q, nviews);
  GPP_TRY(grad_set_smem((const void*)kr_grad_rhs_h_kernel, smem));
  cudaStream_t st = (cudaStream_t)stream;
  kr_grad_rhs_h_kernel<<<dim3((unsigned)p, (unsigned)ceil_div(p, jc)), 256, smem, st>>>(Binv, ldb, wn, p, q, nviews, jc,
                                                                                       alpha, R, ldr);
  GPP_LAUNCH_CHECK();
  const int64_t total = (int64_t)nviews * L * p;
  kr_grad_rhs_m_kernel<<<(unsigned)ceil_div(total, 256), 256, 0, st>>>(W, ldw, wn, p, q, nviews, L, R, ldr);
  GPP_LAUNCH_CHECK();
  return GPP_OK;
}

extern "C" size_t gpp_kr_grad_views_workspace_bytes(int32_t p, int32_t q, int32_t nviews) {
  if (p <= 0 || q <= 0 || nviews <= 0) return 0;
  return align_up((size_t)p * nviews * q * sizeof(float), 256);
}

extern "C" int gpp_kr_grad_views(const float* ST, int64_t ldst, const float* Binv, int64_t ldb, const float* W,
                                 int64_t ldw, const float* wn, int32_t p, int32_t q, int32_t nviews, int32_t L,
                                 double alpha, float* gw, int64_t ldgw, void* workspace, size_t workspace_bytes,
                                 gpp_stream_t stream) {
  GPP_REQUIRE(ST && Binv && W && wn && gw, "kr_grad_views: null pointer");
  GPP_REQUIRE(p > 0 && q > 0 && nviews > 0 && L > 0 && p % 4 == 0 && L % 4 == 0,
              "kr_grad_views: p and L must be positive multiples of 4");
  GPP_REQUIRE(ldst >= (int64_t)nviews * (p + L) && ldb >= (int64_t)p * q && ldw >= L && ldgw >= q,
              "kr_grad_views: bad leading dimension");
  GPP_REQUIRE((size_t)nviews * q * sizeof(float) <= 48 * 1024 && grad_smem_bytes(p, q, nviews) <= kGradSmemMax,
              "kr_grad_views: view table or q too large for one tile of B^-1 in shared memory");
  const size_t need = gpp_kr_grad_views_workspace_bytes(p, q, nviews);
  if (!workspace || workspace_bytes < need) {
    set_error("kr_grad_views: workspace too small (%zu < %zu bytes)", workspace_bytes, need);
    return GPP_ERR_WORKSPACE;
  }
  const int jc = grad_tile_jc(p, q);
  const size_t smem = grad_smem_bytes(p, q, nviews);
  GPP_TRY(grad_set_smem((const void*)kr_grad_views_part_kernel, smem));
  float* part = static_cast<float*>(workspace);
  cudaStream_t st = (cudaStream_t)stream;
  kr_grad_views_part_kernel<<<(unsigned)p, 256, smem, st>>>(ST, ldst, Binv, ldb, W, ldw, wn, p, q, nviews, L, jc, alpha,
                                                            part);
  GPP_LAUNCH_CHECK();
  const int npairs = nviews * q;
  kr_grad_views_reduce_kernel<<<(unsigned)ceil_div(npairs, 8), 256, 0, st>>>(part, p, npairs, q, gw, ldgw);
  GPP_LAUNCH_CHECK();
  return GPP_OK;
}

extern "C" int gpp_kr_predict_views(const float* Binv, int64_t ldb, const float* wn, int32_t p, int32_t q,
                                    int32_t nviews, int32_t k, const int32_t* kinds_host, float* H, int64_t ldh,
                                    float* h, float* c, gpp_stream_t stream) {
  EffLayout lay;
  int has = 0;
  GPP_REQUIRE(p > 0 && q > 0 && nviews > 0 && p % 4 == 0, "kr_predict_views: p must be a positive multiple of 4");
  GPP_REQUIRE(eff_layout(k, kinds_host, p, q, lay, has),
              "kr_predict_views: kinds must list 1..3 distinct GPP_EFFECT_* values");
  const bool with_k = has & (1 << GPP_EFFECT_KR), with_o = has & (1 << GPP_EFFECT_OBJECT);
  const bool need_h = with_k || with_o, need_hc = has & (1 << GPP_EFFECT_VIEW);
  GPP_REQUIRE(Binv && wn && (H || !need_h) && ((h && c) || !need_hc), "kr_predict_views: null pointer");
  GPP_REQUIRE(ldb >= lay.off[k] && (!need_h || ldh >= (int64_t)nviews * p), "kr_predict_views: bad leading dimension");
  GPP_REQUIRE((size_t)nviews * q * sizeof(float) <= 48 * 1024 && grad_smem_bytes(p, q, nviews) <= kGradSmemMax &&
                  predict_hc_smem_bytes(q, nviews) <= kGradSmemMax,
              "kr_predict_views: view table or q too large for one tile of B^-1 in shared memory");
  int off[3] = {-1, -1, -1};
  for (int b = 0; b < k; ++b) off[lay.kind[b]] = lay.off[b];
  cudaStream_t st = (cudaStream_t)stream;
  if (need_h) {
    const int jc = with_k ? grad_tile_jc(p, q) : p;
    const size_t smem = with_k ? grad_smem_bytes(p, q, nviews) : (size_t)nviews * q * sizeof(float);
    GPP_TRY(grad_set_smem((const void*)kr_predict_h_kernel, smem));
    kr_predict_h_kernel<<<dim3((unsigned)p, (unsigned)ceil_div(p, jc)), 256, smem, st>>>(
        Binv, ldb, wn, p, q, nviews, jc, off[GPP_EFFECT_KR], off[GPP_EFFECT_OBJECT], H, ldh);
    GPP_LAUNCH_CHECK();
  }
  if (need_hc) {
    const size_t smem = predict_hc_smem_bytes(q, nviews);
    GPP_TRY(grad_set_smem((const void*)kr_predict_hc_kernel, smem));
    kr_predict_hc_kernel<<<(unsigned)(p + 1), 256, smem, st>>>(Binv, ldb, wn, p, q, nviews, off[GPP_EFFECT_KR],
                                                                off[GPP_EFFECT_OBJECT], off[GPP_EFFECT_VIEW], h, c);
    GPP_LAUNCH_CHECK();
  }
  return GPP_OK;
}

extern "C" int gpp_kr_predict_rows(const float* Y, int64_t ldy, const float* R, int64_t ldr, const float* YH,
                                   int64_t ldyh, const float* xn, const float* h, const float* c, const int64_t* d,
                                   const int64_t* w, int64_t m, int64_t P, int32_t p, int32_t nviews, int32_t L,
                                   const double* scal, float* mean, int64_t ldmean, float* var, gpp_stream_t stream) {
  GPP_REQUIRE(d && w && scal && mean && var && (Y || R) && (!YH || xn) && (!R || c), "kr_predict_rows: null pointer");
  GPP_REQUIRE(m >= 0 && P > 0 && p > 0 && nviews > 0 && L > 0 && L % 4 == 0, "kr_predict_rows: bad shape");
  GPP_REQUIRE((!Y || (ldy >= (int64_t)nviews * L && ldy % 4 == 0 && aligned16(Y))) &&
                  (!R || (ldr >= L && ldr % 4 == 0 && aligned16(R))) && (!YH || ldyh >= (int64_t)nviews * p) &&
                  ldmean >= L && ldmean % 4 == 0 && aligned16(mean),
              "kr_predict_rows: bad leading dimension / alignment");
  if (m == 0) return GPP_OK;
  const int grid = (int)(ceil_div(m, 8) < 8192 ? ceil_div(m, 8) : 8192);
  kr_predict_rows_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(Y, ldy, R, ldr, YH, ldyh, xn, h, c, d, w, m, P, p,
                                                                 nviews, L, scal, mean, ldmean, var);
  GPP_LAUNCH_CHECK();
  return GPP_OK;
}

extern "C" int gpp_rows_dot(const float* A, int64_t lda, const float* B, int64_t ldb, int64_t m, int32_t cols,
                            const double* scal, float* out, gpp_stream_t stream) {
  GPP_REQUIRE(A && B && scal && out, "rows_dot: null pointer");
  GPP_REQUIRE(m >= 0 && cols > 0 && cols % 4 == 0, "rows_dot: cols must be a positive multiple of 4");
  GPP_REQUIRE(lda >= cols && lda % 4 == 0 && ldb >= cols && ldb % 4 == 0 && aligned16(A) && aligned16(B),
              "rows_dot: bad leading dimension / alignment");
  if (m == 0) return GPP_OK;
  const int grid = (int)(ceil_div(m, 8) < 8192 ? ceil_div(m, 8) : 8192);
  rows_dot_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(A, lda, B, ldb, m, cols, scal, out);
  GPP_LAUNCH_CHECK();
  return GPP_OK;
}
