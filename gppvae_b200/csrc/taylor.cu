// Taylor surrogate of gp.py:127-133 and its backward, fused into one launch each.
//   fwd: out_i = Xb_i . X_i + Vb_i . V_i + <vbs, softmax(lvs)> / n
//   bwd: gX_i = g_i Xb_i ; gV_i = g_i Vb_i ; glvs = J_softmax^T vbs * sum(g) / n
// n is the minibatch (64 rows in train_gppvae.py:293): launch-latency bound, hence the fusion.
#include "common.cuh"

namespace gpp {

constexpr int kTeWarps = 8;
constexpr int kMaxDesigns = GPP_MAX_DESIGNS;

__device__ __forceinline__ float row_dot(const float* __restrict__ a, const float* __restrict__ b, int len, int lane) {
  float s = 0.f;
  const int len4 = len >> 2;
  const float4* a4 = reinterpret_cast<const float4*>(a);
  const float4* b4 = reinterpret_cast<const float4*>(b);
  for (int c = lane; c < len4; c += 32) {
    const float4 x = a4[c], y = b4[c];
    s = fmaf(x.x, y.x, s); s = fmaf(x.y, y.y, s); s = fmaf(x.z, y.z, s); s = fmaf(x.w, y.w, s);
  }
  return s;
}

__global__ void __launch_bounds__(kTeWarps * 32)
taylor_fwd_kernel(const float* __restrict__ X, int64_t ldx, const float* __restrict__ Xb, int64_t ldxb,
                  const float* __restrict__ V, int64_t ldv, const float* __restrict__ Vb, int64_t ldvb, int64_t n, int L,
                  int Q, const float* __restrict__ vbs, const float* __restrict__ lvs, float* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (int64_t)blockIdx.x * kTeWarps + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * kTeWarps;
  double v0, vn;
  softmax2(lvs, v0, vn);
  const float cterm = (float)(((double)vbs[0] * v0 + (double)vbs[1] * vn) / (double)n);
  for (int64_t r = warp; r < n; r += nwarps) {
    float s = row_dot(Xb + r * ldxb, X + r * ldx, L, lane);
    if (Q > 0) s += row_dot(Vb + r * ldvb, V + r * ldv, Q, lane);
    s = warp_sum(s);
    if (lane == 0) out[r] = s + cterm;
  }
}

__global__ void __launch_bounds__(kTeWarps * 32)
taylor_bwd_rows_kernel(const float* __restrict__ gout, const float* __restrict__ Xb, int64_t ldxb,
                       const float* __restrict__ Vb, int64_t ldvb, int64_t n, int L, int Q, float* __restrict__ gX,
                       int64_t ldgx, float* __restrict__ gV, int64_t ldgv) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (int64_t)blockIdx.x * kTeWarps + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * kTeWarps;
  for (int64_t r = warp; r < n; r += nwarps) {
    const float g = gout[r];
    if (gX) {
      const float4* s4 = reinterpret_cast<const float4*>(Xb + r * ldxb);
      float4* d4 = reinterpret_cast<float4*>(gX + r * ldgx);
      for (int c = lane; c < (L >> 2); c += 32) {
        const float4 v = s4[c];
        d4[c] = make_float4(g * v.x, g * v.y, g * v.z, g * v.w);
      }
    }
    if (gV) {
      const float4* s4 = reinterpret_cast<const float4*>(Vb + r * ldvb);
      float4* d4 = reinterpret_cast<float4*>(gV + r * ldgv);
      for (int c = lane; c < (Q >> 2); c += 32) {
        const float4 v = s4[c];
        d4[c] = make_float4(g * v.x, g * v.y, g * v.z, g * v.w);
      }
    }
  }
}

// glvs_b = (sum g / n) * vs_b * (vbs_b - <vbs, vs>)   (softmax Jacobian of gp.py:50 applied to vbs)
__global__ void __launch_bounds__(256)
taylor_bwd_lvs_kernel(const float* __restrict__ gout, int64_t n, const float* __restrict__ vbs,
                      const float* __restrict__ lvs, float* __restrict__ glvs) {
  __shared__ double red[8];
  double s = 0;
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) s += (double)gout[i];
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0;
    for (int w = 0; w < 8; ++w) t += red[w];
    double v0, vn;
    softmax2(lvs, v0, vn);
    const double b0 = (double)vbs[0], b1 = (double)vbs[1];
    const double mean = b0 * v0 + b1 * vn;
    const double scale = t / (double)n;
    glvs[0] = (float)(scale * v0 * (b0 - mean));
    glvs[1] = (float)(scale * vn * (b1 - mean));
  }
}

// ---- k designs (gp.py:127-133 summed over the designs, gp.py:130-131), k + 1 variances: one launch each whatever k is
struct TeTable {
  int k;
  const float* V[kMaxDesigns];
  const float* Vb[kMaxDesigns];
  float* gV[kMaxDesigns];
  int64_t ldv[kMaxDesigns], ldvb[kMaxDesigns], ldgv[kMaxDesigns];
  int Q[kMaxDesigns];
};

// softmax(lvs[0..m)) (gp.py:48-50) in double, without a per-thread array: vs_b = exp(lvs_b - mx) / s.
// Returns <vbs, vs>.
__device__ __forceinline__ double softmax_dot(const float* __restrict__ lvs, const float* __restrict__ vbs, int m,
                                              double& mx, double& s) {
  mx = (double)lvs[0];
  for (int b = 1; b < m; ++b) mx = fmax(mx, (double)lvs[b]);
  s = 0;
  double d = 0;
  for (int b = 0; b < m; ++b) {
    const double e = exp((double)lvs[b] - mx);
    s += e;
    d += (double)vbs[b] * e;
  }
  return d / s;
}

__global__ void __launch_bounds__(kTeWarps * 32)
taylor_fwd_multi_kernel(const float* __restrict__ X, int64_t ldx, const float* __restrict__ Xb, int64_t ldxb, TeTable t,
                        int64_t n, int L, const float* __restrict__ vbs, const float* __restrict__ lvs,
                        float* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (int64_t)blockIdx.x * kTeWarps + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * kTeWarps;
  double mx, se;
  const float cterm = (float)(softmax_dot(lvs, vbs, t.k + 1, mx, se) / (double)n);
  for (int64_t r = warp; r < n; r += nwarps) {
    float s = row_dot(Xb + r * ldxb, X + r * ldx, L, lane);
    for (int j = 0; j < t.k; ++j) s += row_dot(t.Vb[j] + r * t.ldvb[j], t.V[j] + r * t.ldv[j], t.Q[j], lane);
    s = warp_sum(s);
    if (lane == 0) out[r] = s + cterm;
  }
}

__global__ void __launch_bounds__(kTeWarps * 32)
taylor_bwd_multi_rows_kernel(const float* __restrict__ gout, const float* __restrict__ Xb, int64_t ldxb, TeTable t,
                             int64_t n, int L, float* __restrict__ gX, int64_t ldgx) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (int64_t)blockIdx.x * kTeWarps + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * kTeWarps;
  auto scale_row = [&](const float* src, float* dst, int len, float g) {
    const float4* s4 = reinterpret_cast<const float4*>(src);
    float4* d4 = reinterpret_cast<float4*>(dst);
    for (int c = lane; c < (len >> 2); c += 32) {
      const float4 v = s4[c];
      d4[c] = make_float4(g * v.x, g * v.y, g * v.z, g * v.w);
    }
  };
  for (int64_t r = warp; r < n; r += nwarps) {
    const float g = gout[r];
    if (gX) scale_row(Xb + r * ldxb, gX + r * ldgx, L, g);
    for (int j = 0; j < t.k; ++j)
      if (t.gV[j]) scale_row(t.Vb[j] + r * t.ldvb[j], t.gV[j] + r * t.ldgv[j], t.Q[j], g);
  }
}

// glvs_b = (sum g / n) * vs_b * (vbs_b - <vbs, vs>),  b = 0..m-1
__global__ void __launch_bounds__(256)
taylor_bwd_multi_lvs_kernel(const float* __restrict__ gout, int64_t n, int m, const float* __restrict__ vbs,
                            const float* __restrict__ lvs, float* __restrict__ glvs) {
  __shared__ double red[8];
  double s = 0;
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) s += (double)gout[i];
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0;
    for (int w = 0; w < 8; ++w) t += red[w];
    double mx, se;
    const double mean = softmax_dot(lvs, vbs, m, mx, se);
    const double scale = t / (double)n;
    for (int b = 0; b < m; ++b)
      glvs[b] = (float)(scale * (exp((double)lvs[b] - mx) / se) * ((double)vbs[b] - mean));
  }
}

static int rows_grid(int64_t n) {
  const int64_t want = ceil_div(n, kTeWarps);
  const int64_t cap = (int64_t)sm_count() * 8;
  return (int)(want < cap ? (want > 0 ? want : 1) : cap);
}

}  // namespace gpp

using namespace gpp;

extern "C" int gpp_taylor_expansion_fwd(const float* X, int64_t ldx, const float* Xb, int64_t ldxb, const float* V,
                                        int64_t ldv, const float* Vb, int64_t ldvb, int64_t n, int32_t L, int32_t Q,
                                        const float* vbs, const float* lvs, float* out, gpp_stream_t stream) {
  GPP_REQUIRE(X && Xb && vbs && lvs && out, "taylor_expansion_fwd: null pointer");
  GPP_REQUIRE(Q == 0 || (V && Vb), "taylor_expansion_fwd: null V / Vb");
  GPP_REQUIRE(n > 0 && L > 0 && L % 4 == 0 && Q >= 0 && Q % 4 == 0, "taylor_expansion_fwd: bad shape");
  GPP_REQUIRE(ldx % 4 == 0 && ldxb % 4 == 0 && ldv % 4 == 0 && ldvb % 4 == 0, "taylor_expansion_fwd: ld %% 4 != 0");
  GPP_REQUIRE(aligned16(X) && aligned16(Xb) && aligned16(V) && aligned16(Vb), "taylor_expansion_fwd: misaligned");
  taylor_fwd_kernel<<<rows_grid(n), kTeWarps * 32, 0, (cudaStream_t)stream>>>(X, ldx, Xb, ldxb, V, ldv, Vb, ldvb, n, L,
                                                                              Q, vbs, lvs, out);
  GPP_LAUNCH_CHECK();
  return GPP_OK;
}

extern "C" int gpp_taylor_expansion_bwd(const float* gout, const float* Xb, int64_t ldxb, const float* Vb, int64_t ldvb,
                                        int64_t n, int32_t L, int32_t Q, const float* vbs, const float* lvs, float* gX,
                                        int64_t ldgx, float* gV, int64_t ldgv, float* glvs, gpp_stream_t stream) {
  GPP_REQUIRE(gout && vbs && lvs, "taylor_expansion_bwd: null pointer");
  GPP_REQUIRE(n > 0 && L > 0 && L % 4 == 0 && Q >= 0 && Q % 4 == 0, "taylor_expansion_bwd: bad shape");
  GPP_REQUIRE(!gX || (Xb && aligned16(Xb) && aligned16(gX) && ldxb % 4 == 0 && ldgx % 4 == 0),
              "taylor_expansion_bwd: bad gX / Xb");
  GPP_REQUIRE(!gV || (Vb && aligned16(Vb) && aligned16(gV) && ldvb % 4 == 0 && ldgv % 4 == 0),
              "taylor_expansion_bwd: bad gV / Vb");
  if (gX || gV) {
    taylor_bwd_rows_kernel<<<rows_grid(n), kTeWarps * 32, 0, (cudaStream_t)stream>>>(gout, Xb, ldxb, Vb, ldvb, n, L, Q,
                                                                                     gX, ldgx, gV, ldgv);
    GPP_LAUNCH_CHECK();
  }
  if (glvs) {
    taylor_bwd_lvs_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(gout, n, vbs, lvs, glvs);
    GPP_LAUNCH_CHECK();
  }
  return GPP_OK;
}

// Fill the pointer table of the k-design entries from the caller's host arrays.
static int te_table(const char* who, int32_t k, const float* const* V, const int64_t* ldv, const float* const* Vb,
                    const int64_t* ldvb, float* const* gV, const int64_t* ldgv, const int32_t* Q, TeTable& t) {
  GPP_REQUIRE(k >= 1 && k <= kMaxDesigns, "%s: k = %d designs (1..%d supported)", who, k, kMaxDesigns);
  GPP_REQUIRE(Vb && ldvb && Q, "%s: null host array", who);
  t = TeTable{};
  t.k = k;
  for (int j = 0; j < k; ++j) {
    GPP_REQUIRE(Q[j] > 0 && Q[j] % 4 == 0, "%s: design %d has %d columns (a positive multiple of 4 is required)", who, j,
                Q[j]);
    GPP_REQUIRE(Vb[j] && aligned16(Vb[j]) && ldvb[j] >= Q[j] && ldvb[j] % 4 == 0, "%s: bad Vb of design %d", who, j);
    t.Vb[j] = Vb[j];
    t.ldvb[j] = ldvb[j];
    t.Q[j] = Q[j];
    if (V) {
      GPP_REQUIRE(ldv && V[j] && aligned16(V[j]) && ldv[j] >= Q[j] && ldv[j] % 4 == 0, "%s: bad V of design %d", who, j);
      t.V[j] = V[j];
      t.ldv[j] = ldv[j];
    }
    if (gV && gV[j]) {
      GPP_REQUIRE(ldgv && aligned16(gV[j]) && ldgv[j] >= Q[j] && ldgv[j] % 4 == 0, "%s: bad gV of design %d", who, j);
      t.gV[j] = gV[j];
      t.ldgv[j] = ldgv[j];
    }
  }
  return GPP_OK;
}

extern "C" int gpp_taylor_expansion_fwd_multi(const float* X, int64_t ldx, const float* Xb, int64_t ldxb, int32_t k,
                                              const float* const* V_host, const int64_t* ldv_host,
                                              const float* const* Vb_host, const int64_t* ldvb_host, const int32_t* Q_host,
                                              int64_t n, int32_t L, const float* vbs, const float* lvs, float* out,
                                              gpp_stream_t stream) {
  GPP_REQUIRE(X && Xb && vbs && lvs && out && V_host, "taylor_expansion_fwd_multi: null pointer");
  GPP_REQUIRE(n > 0 && L > 0 && L % 4 == 0, "taylor_expansion_fwd_multi: bad shape");
  GPP_REQUIRE(ldx >= L && ldxb >= L && ldx % 4 == 0 && ldxb % 4 == 0 && aligned16(X) && aligned16(Xb),
              "taylor_expansion_fwd_multi: bad X / Xb");
  TeTable t;
  GPP_TRY(te_table("taylor_expansion_fwd_multi", k, V_host, ldv_host, Vb_host, ldvb_host, nullptr, nullptr, Q_host, t));
  taylor_fwd_multi_kernel<<<rows_grid(n), kTeWarps * 32, 0, (cudaStream_t)stream>>>(X, ldx, Xb, ldxb, t, n, L, vbs, lvs,
                                                                                    out);
  GPP_LAUNCH_CHECK();
  return GPP_OK;
}

extern "C" int gpp_taylor_expansion_bwd_multi(const float* gout, const float* Xb, int64_t ldxb, int32_t k,
                                              const float* const* Vb_host, const int64_t* ldvb_host, const int32_t* Q_host,
                                              int64_t n, int32_t L, const float* vbs, const float* lvs, float* gX,
                                              int64_t ldgx, float* const* gV_host, const int64_t* ldgv_host, float* glvs,
                                              gpp_stream_t stream) {
  GPP_REQUIRE(gout && vbs && lvs, "taylor_expansion_bwd_multi: null pointer");
  GPP_REQUIRE(n > 0 && L > 0 && L % 4 == 0, "taylor_expansion_bwd_multi: bad shape");
  GPP_REQUIRE(!gX || (Xb && aligned16(Xb) && aligned16(gX) && ldxb >= L && ldgx >= L && ldxb % 4 == 0 && ldgx % 4 == 0),
              "taylor_expansion_bwd_multi: bad gX / Xb");
  TeTable t;
  GPP_TRY(te_table("taylor_expansion_bwd_multi", k, nullptr, nullptr, Vb_host, ldvb_host, gV_host, ldgv_host, Q_host, t));
  bool any_gv = false;
  for (int j = 0; j < k; ++j) any_gv = any_gv || t.gV[j] != nullptr;
  if (gX || any_gv) {
    taylor_bwd_multi_rows_kernel<<<rows_grid(n), kTeWarps * 32, 0, (cudaStream_t)stream>>>(gout, Xb, ldxb, t, n, L, gX,
                                                                                           ldgx);
    GPP_LAUNCH_CHECK();
  }
  if (glvs) {
    taylor_bwd_multi_lvs_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(gout, n, k + 1, vbs, lvs, glvs);
    GPP_LAUNCH_CHECK();
  }
  return GPP_OK;
}
