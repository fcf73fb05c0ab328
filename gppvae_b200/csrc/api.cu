// C ABI of libgppvae_b200 (see include/gppvae_b200.h): argument validation and dispatch to the
// kernel launchers, plus the host-buffer end-to-end entry.
#include <stdarg.h>
#include <string.h>

#include <atomic>
#include <string>

#include "common.cuh"
#include "kernels.h"

namespace gpp {

static thread_local std::string g_last_error;
static std::atomic<unsigned long long> g_launches{0};

void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

void set_error(const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_last_error = buf;
}

int sm_count() {
  static thread_local int cached_dev = -1, cached = 148;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return cached;
  if (dev != cached_dev) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0) cached = n;
    cached_dev = dev;
  }
  return cached;
}

static bool mat_ok(const float* p, int64_t ld, int64_t cols) { return p && aligned16(p) && ld >= cols && ld % 4 == 0; }

}  // namespace gpp

using namespace gpp;

extern "C" int gpp_version(void) { return 100; }
extern "C" const char* gpp_last_error(void) { return g_last_error.c_str(); }
extern "C" const char* gpp_gemm_engine(void) { return "tcgen05-3xf16"; }
extern "C" uint64_t gpp_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

// ------------------------------------------------------------------ pass 1
extern "C" size_t gpp_gram_workspace_bytes(int64_t n, int32_t Q, int32_t L) {
  const size_t a = tn_workspace_bytes(n, Q, Q, L, 1);
  const size_t b = tc_pass1_supported(n, Q, L) ? tc_pass1_workspace_bytes(n, Q, L, false) : 0;
  return a > b ? a : b;
}

extern "C" int gpp_gram_vtz(const float* V, int64_t ldv, const float* X, int64_t ldx, int64_t n, int32_t Q, int32_t L,
                            float* GC, int64_t ldgc, void* workspace, size_t workspace_bytes, gpp_stream_t stream) {
  GPP_REQUIRE(n >= 0 && Q > 0 && L >= 0 && Q % 4 == 0 && L % 4 == 0, "gram_vtz: bad shape n=%lld Q=%d L=%d",
              (long long)n, Q, L);
  GPP_REQUIRE(mat_ok(V, ldv, Q), "gram_vtz: V must be 16-byte aligned with ldv >= Q and ldv %% 4 == 0");
  GPP_REQUIRE(L == 0 || mat_ok(X, ldx, L), "gram_vtz: X must be 16-byte aligned with ldx >= L and ldx %% 4 == 0");
  GPP_REQUIRE(mat_ok(GC, ldgc, (int64_t)Q + L), "gram_vtz: GC must be 16-byte aligned with ldgc >= Q + L");
  // large problems run on the tensor cores (3-term split); tiles that cannot fill a 256 x 256 pair UMMA use the fp32 tile engine
  if (tc_pass1_supported(n, Q, L))
    return launch_tc_pass1(V, ldv, X, ldx, n, Q, L, GC, ldgc, GC + Q, ldgc, nullptr, workspace, workspace_bytes, false,
                           (cudaStream_t)stream);
  return launch_tn(V, ldv, Q, V, ldv, Q, X, ldx, L, n, 1, GC, ldgc, GC + Q, ldgc, nullptr, workspace, workspace_bytes,
                   (cudaStream_t)stream);
}

// Debug / cross-check entry: pass 1 on the fp32 SIMT tile engine regardless of size (tests compare the two).
extern "C" int gpp_gram_vtz_simt(const float* V, int64_t ldv, const float* X, int64_t ldx, int64_t n, int32_t Q,
                                 int32_t L, float* GC, int64_t ldgc, void* workspace, size_t workspace_bytes,
                                 gpp_stream_t stream) {
  GPP_REQUIRE(n >= 0 && Q > 0 && L >= 0 && Q % 4 == 0 && L % 4 == 0, "gram_vtz_simt: bad shape");
  GPP_REQUIRE(mat_ok(V, ldv, Q) && (L == 0 || mat_ok(X, ldx, L)) && mat_ok(GC, ldgc, (int64_t)Q + L),
              "gram_vtz_simt: bad pointer / leading dimension");
  return launch_tn(V, ldv, Q, V, ldv, Q, X, ldx, L, n, 1, GC, ldgc, GC + Q, ldgc, nullptr, workspace, workspace_bytes,
                   (cudaStream_t)stream);
}

// ------------------------------------------------------------------ operand planes
static bool planes_ok(const void* p) { return p && (reinterpret_cast<uintptr_t>(p) & 255u) == 0; }

extern "C" size_t gpp_planes_bytes(int64_t n, int32_t cols) { return planes_bytes(n, cols); }
extern "C" size_t gpp_split_workspace_bytes(int64_t n, int32_t cols) { return split_workspace_bytes(n, cols); }
extern "C" int gpp_planes_supported(int64_t n, int32_t Q, int32_t L) {
  return pl_pass1_supported(n, Q, L) && pl_rows_supported(n, Q, L > 0 ? L : 64) ? 1 : 0;
}

extern "C" int gpp_split_planes(const float* X, int64_t ldx, int64_t n, int32_t cols, uint32_t flags, void* planes,
                                size_t planes_bytes_, void* workspace, size_t workspace_bytes, gpp_stream_t stream) {
  GPP_REQUIRE(n >= 0 && cols > 0 && cols % 4 == 0, "split_planes: bad shape n=%lld cols=%d", (long long)n, cols);
  GPP_REQUIRE(mat_ok(X, ldx, cols), "split_planes: X must be 16-byte aligned with ldx >= cols and ldx %% 4 == 0");
  GPP_REQUIRE(planes_ok(planes) && planes_bytes_ >= planes_bytes(n, cols),
              "split_planes: planes buffer must be 256-byte aligned and gpp_planes_bytes() long");
  return launch_split_planes(X, ldx, n, cols, planes, nullptr, (flags & GPP_PLANES_UNIT_BOUND) ? 1 : 0,
                             (flags & GPP_PLANES_COLSQ) != 0, workspace, workspace_bytes, (cudaStream_t)stream);
}

extern "C" int gpp_khatri_rao_fwd_planes(const float* xn, int64_t P, int32_t p, const float* wn, int64_t nviews,
                                         int32_t q, const int64_t* d, const int64_t* w, int64_t n, float* V,
                                         int64_t ldv, void* planes, size_t planes_bytes_, void* workspace,
                                         size_t workspace_bytes, gpp_stream_t stream) {
  GPP_REQUIRE(xn && wn && d && w && V, "khatri_rao_fwd_planes: null pointer");
  GPP_REQUIRE(P > 0 && p > 0 && nviews > 0 && q > 0 && n >= 0 && ((int64_t)p * q) % 4 == 0 && (int64_t)p * q < (1 << 30),
              "khatri_rao_fwd_planes: bad shape");
  GPP_REQUIRE(mat_ok(V, ldv, (int64_t)p * q), "khatri_rao_fwd_planes: V must be 16-byte aligned with ldv >= p*q");
  GPP_REQUIRE((q % 4 != 0) || (aligned16(wn)), "khatri_rao_fwd_planes: wn must be 16-byte aligned");
  GPP_REQUIRE(planes_ok(planes) && planes_bytes_ >= planes_bytes(n, p * q),
              "khatri_rao_fwd_planes: planes buffer must be 256-byte aligned and gpp_planes_bytes() long");
  return launch_kr_planes(xn, P, p, wn, nviews, q, d, w, n, V, ldv, planes, workspace, workspace_bytes,
                          (cudaStream_t)stream);
}

extern "C" size_t gpp_gram_planes_workspace_bytes(int64_t n, int32_t Q, int32_t L) {
  // serves gpp_gram_vtz_planes (Gram tiles + V^T X) and gpp_atb_planes (no Gram tiles): their split counts differ
  const size_t a = pl_pass1_workspace_bytes(n, Q, L, false), b = L > 0 ? pl_pass1_workspace_bytes(n, Q, L, true) : 0;
  return a > b ? a : b;
}

extern "C" int gpp_gram_vtz_planes(const void* planesV, const void* planesX, int64_t n, int32_t Q, int32_t L,
                                   int32_t use_colsq, float* GC, int64_t ldgc, void* workspace, size_t workspace_bytes,
                                   gpp_stream_t stream) {
  GPP_REQUIRE(Q > 0 && L >= 0 && Q % 4 == 0 && L % 4 == 0, "gram_vtz_planes: bad shape n=%lld Q=%d L=%d", (long long)n,
              Q, L);
  GPP_REQUIRE(pl_pass1_supported(n, Q, L), "gram_vtz_planes: shape below the tensor-core tile (n >= 512, Q >= 128)");
  GPP_REQUIRE(planes_ok(planesV) && (L == 0 || planes_ok(planesX)), "gram_vtz_planes: planes must be 256-byte aligned");
  GPP_REQUIRE(mat_ok(GC, ldgc, (int64_t)Q + L), "gram_vtz_planes: GC must be 16-byte aligned with ldgc >= Q + L");
  return launch_pl_pass1(planesV, planesX, n, Q, L, GC, ldgc, GC + Q, ldgc, use_colsq != 0, workspace, workspace_bytes,
                         (cudaStream_t)stream);
}

extern "C" int gpp_atb_planes(const void* planesA, const void* planesB, int64_t n, int32_t ka, int32_t kb, float* out,
                              int64_t ldo, void* workspace, size_t workspace_bytes, gpp_stream_t stream) {
  GPP_REQUIRE(ka > 0 && kb > 0 && ka % 4 == 0 && kb % 4 == 0, "atb_planes: bad shape");
  GPP_REQUIRE(pl_pass1_supported(n, ka, kb), "atb_planes: shape below the tensor-core tile (n >= 512, ka >= 128)");
  GPP_REQUIRE(planes_ok(planesA) && planes_ok(planesB) && mat_ok(out, ldo, kb), "atb_planes: bad pointer");
  return launch_pl_pass1(planesA, planesB, n, ka, kb, nullptr, 0, out, ldo, false, workspace, workspace_bytes,
                         (cudaStream_t)stream);
}

extern "C" size_t gpp_xb_planes_workspace_bytes(int64_t n, int32_t Q, int32_t L) { return pl_xb_workspace_bytes(n, Q, L); }

extern "C" int gpp_xb_nll_planes(const void* planesV, const float* X, int64_t ldx, const float* W, int64_t ldw,
                                 int64_t n, int32_t Q, int32_t L, double* scal, float* Xb, int64_t ldxb, float* nll,
                                 void* workspace, size_t workspace_bytes, gpp_stream_t stream) {
  GPP_REQUIRE(Q > 0 && L > 0 && Q % 4 == 0 && L % 4 == 0, "xb_nll_planes: bad shape");
  GPP_REQUIRE(pl_rows_supported(n, Q, L), "xb_nll_planes: shape below the tensor-core tile (n >= 512, Q, L >= 64)");
  GPP_REQUIRE(planes_ok(planesV) && mat_ok(X, ldx, L) && mat_ok(W, ldw, L) && mat_ok(Xb, ldxb, L),
              "xb_nll_planes: bad pointer / leading dimension");
  GPP_REQUIRE(scal && nll, "xb_nll_planes: null scal / nll");
  return launch_pl_xb(planesV, X, ldx, W, ldw, n, Q, L, scal, 0.f, Xb, ldxb, nll, workspace, workspace_bytes,
                      (cudaStream_t)stream);
}

extern "C" size_t gpp_atb_workspace_bytes(int64_t n, int32_t ka, int32_t kb) {
  const size_t a = tn_workspace_bytes(n, ka, 0, kb, 0);
  const size_t b = tc_pass1_supported(n, ka, kb) ? tc_pass1_workspace_bytes(n, ka, kb, true) : 0;
  return a > b ? a : b;
}

extern "C" int gpp_atb(const float* A, int64_t lda, const float* B, int64_t ldb, int64_t n, int32_t ka, int32_t kb,
                       float* out, int64_t ldo, void* workspace, size_t workspace_bytes, gpp_stream_t stream) {
  GPP_REQUIRE(n >= 0 && ka > 0 && kb > 0 && ka % 4 == 0 && kb % 4 == 0, "atb: bad shape");
  GPP_REQUIRE(mat_ok(A, lda, ka) && mat_ok(B, ldb, kb) && mat_ok(out, ldo, kb), "atb: bad pointer / leading dimension");
  if (tc_pass1_supported(n, ka, kb))   // pass 1 without the Gram tiles
    return launch_tc_pass1(A, lda, B, ldb, n, ka, kb, nullptr, 0, out, ldo, nullptr, workspace, workspace_bytes, false,
                           (cudaStream_t)stream);
  return launch_tn(A, lda, ka, nullptr, 0, 0, B, ldb, kb, n, 0, nullptr, 0, out, ldo, nullptr, workspace,
                   workspace_bytes, (cudaStream_t)stream);
}

// ------------------------------------------------------------------ Q-space solve
extern "C" size_t gpp_factor_state_bytes(int32_t Q) { return factor_workspace_bytes(Q); }
extern "C" size_t gpp_solve_workspace_bytes(int32_t Q, int32_t L) { return solve_workspace_bytes(Q, L); }

extern "C" int gpp_factor(const float* G, int64_t ldg, int32_t Q, const float* vs, uint32_t flags, float* Binv,
                          double* scal, void* state, size_t state_bytes, gpp_stream_t stream) {
  GPP_REQUIRE(Q > 0 && Q % 4 == 0, "factor: bad shape Q=%d", Q);
  GPP_REQUIRE(mat_ok(G, ldg, Q), "factor: bad G");
  GPP_REQUIRE(vs && scal, "factor: null vs / scal");
  GPP_REQUIRE(!(flags & GPP_WANT_BINV) || (Binv && aligned16(Binv)), "factor: Binv required with GPP_WANT_BINV");
  return launch_factor(G, ldg, Q, vs, flags, Binv, scal, state, state_bytes, (cudaStream_t)stream);
}

extern "C" int gpp_solve_w(const float* C, int64_t ldc, int32_t Q, int32_t L, int32_t L_true, int64_t n_total,
                           float* W, int64_t ldw, double* scal, const void* state, size_t state_bytes, void* workspace,
                           size_t workspace_bytes, gpp_stream_t stream) {
  GPP_REQUIRE(Q > 0 && L > 0 && Q % 4 == 0 && L % 4 == 0 && n_total > 0 && L_true > 0 && L_true <= L,
              "solve_w: bad shape Q=%d L=%d L_true=%d", Q, L, L_true);
  GPP_REQUIRE(mat_ok(C, ldc, L) && mat_ok(W, ldw, L) && scal, "solve_w: bad C / W / scal");
  return launch_solve_w(C, ldc, Q, L, L_true, n_total, W, ldw, scal, state, state_bytes, workspace, workspace_bytes,
                        (cudaStream_t)stream);
}

extern "C" int gpp_factor_solve(const float* GC, int64_t ldgc, int32_t Q, int32_t L, const float* vs, int64_t n_total,
                                uint32_t flags, float* W, int64_t ldw, float* Binv, double* scal, void* workspace,
                                size_t workspace_bytes, gpp_stream_t stream) {
  GPP_REQUIRE(Q > 0 && L > 0 && Q % 4 == 0 && L % 4 == 0 && n_total > 0, "factor_solve: bad shape Q=%d L=%d", Q, L);
  GPP_REQUIRE(mat_ok(GC, ldgc, (int64_t)Q + L), "factor_solve: bad GC");
  const size_t sb = align_up(factor_workspace_bytes(Q), 256);
  if (!workspace || workspace_bytes < sb + solve_workspace_bytes(Q, L)) {
    set_error("factor_solve: workspace too small (%zu < %zu bytes)", workspace_bytes, sb + solve_workspace_bytes(Q, L));
    return GPP_ERR_WORKSPACE;
  }
  GPP_TRY(gpp_factor(GC, ldgc, Q, vs, flags, Binv, scal, workspace, sb, stream));
  return gpp_solve_w(GC + Q, ldgc, Q, L, L, n_total, W, ldw, scal, workspace, sb, static_cast<char*>(workspace) + sb,
                     workspace_bytes - sb, stream);
}

// ------------------------------------------------------------------ pass 2
extern "C" size_t gpp_xb_workspace_bytes(int64_t n, int32_t Q, int32_t L) {
  const size_t a = xb_workspace_bytes(n, L);
  const size_t b = tc_rows_supported(n, Q, L) ? tc_xb_workspace_bytes(n, L) : 0;
  return a > b ? a : b;
}

extern "C" int gpp_xb_nll(const float* V, int64_t ldv, const float* X, int64_t ldx, const float* W, int64_t ldw,
                          int64_t n, int32_t Q, int32_t L, double* scal, float* Xb, int64_t ldxb, float* nll,
                          void* workspace, size_t workspace_bytes, gpp_stream_t stream) {
  GPP_REQUIRE(n >= 0 && Q > 0 && L > 0 && Q % 4 == 0 && L % 4 == 0, "xb_nll: bad shape");
  GPP_REQUIRE(mat_ok(V, ldv, Q) && mat_ok(X, ldx, L) && mat_ok(W, ldw, L) && mat_ok(Xb, ldxb, L),
              "xb_nll: bad pointer / leading dimension");
  GPP_REQUIRE(scal && nll, "xb_nll: null scal / nll");
  if (tc_rows_supported(n, Q, L))
    return launch_tc_xb(V, ldv, X, ldx, W, ldw, n, Q, L, scal, 0.f, Xb, ldxb, nll, workspace, workspace_bytes,
                        (cudaStream_t)stream);
  return launch_xb(V, ldv, X, ldx, W, ldw, n, Q, L, scal, 0.f, Xb, ldxb, nll, workspace, workspace_bytes,
                   (cudaStream_t)stream);
}

// 256 bytes: the device slots that receive the operands' exact maxima (scales of the fp16 operands)
extern "C" size_t gpp_rows_workspace_bytes(void) { return 256; }

extern "C" int gpp_x_minus_am(const float* X, int64_t ldx, const float* A, int64_t lda, const float* M, int64_t ldm,
                              int64_t n, int32_t k, int32_t m, float alpha, float* out, int64_t ldo, void* workspace,
                              size_t workspace_bytes, gpp_stream_t stream) {
  GPP_REQUIRE(n >= 0 && k > 0 && m > 0 && k % 4 == 0 && m % 4 == 0, "x_minus_am: bad shape");
  GPP_REQUIRE(mat_ok(X, ldx, m) && mat_ok(A, lda, k) && mat_ok(M, ldm, m) && mat_ok(out, ldo, m),
              "x_minus_am: bad pointer / leading dimension");
  if (tc_rows_supported(n, k, m)) {
    if (!workspace || workspace_bytes < 256 || !aligned16(workspace)) {
      set_error("x_minus_am: workspace of gpp_rows_workspace_bytes() required (%zu bytes given)", workspace_bytes);
      return GPP_ERR_WORKSPACE;
    }
    return launch_tc_xb(A, lda, X, ldx, M, ldm, n, k, m, nullptr, alpha, out, ldo, nullptr, workspace, workspace_bytes,
                        (cudaStream_t)stream);
  }
  return launch_xb(A, lda, X, ldx, M, ldm, n, k, m, nullptr, alpha, out, ldo, nullptr, nullptr, 0,
                   (cudaStream_t)stream);
}

extern "C" int gpp_am(const float* A, int64_t lda, const float* M, int64_t ldm, int64_t n, int32_t k, int32_t m,
                      float alpha, float* out, int64_t ldo, void* workspace, size_t workspace_bytes, gpp_stream_t stream) {
  GPP_REQUIRE(n >= 0 && k > 0 && m > 0 && k % 4 == 0 && m % 4 == 0 && n < (1ll << 31), "am: bad shape");
  GPP_REQUIRE(mat_ok(A, lda, k) && mat_ok(M, ldm, m) && mat_ok(out, ldo, m), "am: bad pointer / leading dimension");
  if (n == 0) return GPP_OK;
  if (tc_blockgemm_supported((int)n, k, m)) {
    if (!workspace || workspace_bytes < 256 || !aligned16(workspace)) {
      set_error("am: workspace of gpp_rows_workspace_bytes() required (%zu bytes given)", workspace_bytes);
      return GPP_ERR_WORKSPACE;
    }
    uint32_t* amax = static_cast<uint32_t*>(workspace);
    GPP_TRY(tc_absmax(A, lda, n, k, amax, (cudaStream_t)stream));
    GPP_TRY(tc_absmax(M, ldm, k, m, amax + 1, (cudaStream_t)stream));
    TcBlockGemm g{};
    g.n = (int)n; g.n_last = (int)n; g.K = k; g.ncols = m; g.batches = 1; g.alpha = alpha;
    return launch_tc_blockgemm(A, n, k, lda, M, k, m, ldm, out, ldo, g, amax, (cudaStream_t)stream);
  }
  GemmParams g{};
  g.A = A; g.lda = lda; g.B = M; g.ldb = ldm; g.C = out; g.ldc = ldo;
  g.M = (int)n; g.N = m; g.K = k; g.M_last = -1; g.alpha = alpha; g.beta = 0.f;
  return launch_gemm(g, false, true, 1, (cudaStream_t)stream);
}

extern "C" int gpp_vbs(const double* scal, int64_t n_total, int32_t Q, int32_t L, float* vbs, gpp_stream_t stream) {
  GPP_REQUIRE(scal && vbs && n_total > 0 && Q > 0 && L > 0, "vbs: bad argument");
  return launch_vbs(scal, n_total, Q, L, vbs, (cudaStream_t)stream);
}

// ------------------------------------------------------------------ k stacked designs
// BlockSpec from the caller's host array of block column counts (each a positive multiple of 4)
static int block_spec(const char* who, int32_t k, const int32_t* cols_host, BlockSpec& bs) {
  GPP_REQUIRE(k >= 1 && k <= GPP_MAX_DESIGNS, "%s: k = %d designs (1..%d supported)", who, k, GPP_MAX_DESIGNS);
  GPP_REQUIRE(cols_host, "%s: null column counts", who);
  bs = BlockSpec{};
  bs.k = k;
  int64_t q = 0;
  for (int i = 0; i < k; ++i) {
    GPP_REQUIRE(cols_host[i] > 0 && cols_host[i] % 4 == 0,
                "%s: design %d has %d columns (a positive multiple of 4 is required)", who, i, cols_host[i]);
    q += cols_host[i];
    GPP_REQUIRE(q < (1 << 20), "%s: too many stacked columns", who);
    bs.start[i + 1] = (int)q;
  }
  return GPP_OK;
}

extern "C" size_t gpp_split_stacked_workspace_bytes(int64_t n, int32_t k, const int32_t* cols_host) {
  if (!cols_host || k < 1 || k > GPP_MAX_DESIGNS) return 0;
  return split_stacked_workspace_bytes(n, k, cols_host);
}

extern "C" int gpp_split_planes_stacked(int32_t k, const float* const* X_host, const int64_t* ldx_host,
                                        const int32_t* cols_host, int64_t n, uint32_t flags, void* planes,
                                        size_t planes_bytes_, void* workspace, size_t workspace_bytes,
                                        gpp_stream_t stream) {
  BlockSpec bs;
  GPP_TRY(block_spec("split_planes_stacked", k, cols_host, bs));
  GPP_REQUIRE(n >= 0 && X_host && ldx_host, "split_planes_stacked: bad n / null host array");
  for (int i = 0; i < k; ++i)
    GPP_REQUIRE(mat_ok(X_host[i], ldx_host[i], cols_host[i]),
                "split_planes_stacked: source %d must be 16-byte aligned with ldx >= cols and ldx %% 4 == 0", i);
  GPP_REQUIRE(planes_ok(planes) && planes_bytes_ >= planes_bytes(n, bs.start[k]),
              "split_planes_stacked: planes buffer must be 256-byte aligned and gpp_planes_bytes(n, sum cols) long");
  return launch_split_planes_stacked(k, X_host, ldx_host, cols_host, n, planes, (flags & GPP_PLANES_UNIT_BOUND) != 0,
                                     (flags & GPP_PLANES_COLSQ) != 0, workspace, workspace_bytes, (cudaStream_t)stream);
}

extern "C" size_t gpp_factor_blocks_state_bytes(int32_t Q, int32_t k) {
  return Q > 0 && k >= 1 && k <= GPP_MAX_DESIGNS ? factor_blocks_workspace_bytes(Q, k) : 0;
}
extern "C" size_t gpp_solve_blocks_workspace_bytes(int32_t Q, int32_t L, int32_t k) {
  return Q > 0 && L > 0 && k >= 1 && k <= GPP_MAX_DESIGNS ? solve_blocks_workspace_bytes(Q, L, k) : 0;
}

extern "C" int gpp_factor_blocks(const float* G, int64_t ldg, int32_t k, const int32_t* cols_host, const float* vs,
                                 uint32_t flags, float* Binv, double* scal, double* blk, void* state, size_t state_bytes,
                                 gpp_stream_t stream) {
  BlockSpec bs;
  GPP_TRY(block_spec("factor_blocks", k, cols_host, bs));
  const int Q = bs.start[k];
  GPP_REQUIRE(mat_ok(G, ldg, Q), "factor_blocks: bad G");
  GPP_REQUIRE(vs && scal && blk, "factor_blocks: null vs / scal / blk");
  GPP_REQUIRE(!(flags & GPP_WANT_BINV) || (Binv && aligned16(Binv)), "factor_blocks: Binv required with GPP_WANT_BINV");
  return launch_factor_blocks(G, ldg, bs, vs, flags, Binv, scal, blk, state, state_bytes, (cudaStream_t)stream);
}

extern "C" int gpp_solve_w_blocks(const float* C, int64_t ldc, int32_t k, const int32_t* cols_host, int32_t L,
                                  int32_t L_true, int64_t n_total, float* W, int64_t ldw, double* scal, double* blk,
                                  const void* state, size_t state_bytes, void* workspace, size_t workspace_bytes,
                                  gpp_stream_t stream) {
  BlockSpec bs;
  GPP_TRY(block_spec("solve_w_blocks", k, cols_host, bs));
  GPP_REQUIRE(L > 0 && L % 4 == 0 && n_total > 0 && L_true > 0 && L_true <= L, "solve_w_blocks: bad shape L=%d L_true=%d",
              L, L_true);
  GPP_REQUIRE(mat_ok(C, ldc, L) && mat_ok(W, ldw, L) && scal && blk, "solve_w_blocks: bad C / W / scal / blk");
  return launch_solve_w_blocks(C, ldc, bs, L, L_true, n_total, W, ldw, scal, blk, state, state_bytes, workspace,
                               workspace_bytes, (cudaStream_t)stream);
}

extern "C" int gpp_vbs_blocks(const double* scal, const double* blk, const float* vs, int32_t k, const int32_t* cols_host,
                              int64_t n_total, int32_t L, float* vbs, gpp_stream_t stream) {
  BlockSpec bs;
  GPP_TRY(block_spec("vbs_blocks", k, cols_host, bs));
  GPP_REQUIRE(scal && blk && vs && vbs && n_total > 0 && L > 0, "vbs_blocks: bad argument");
  return launch_vbs_blocks(scal, blk, vs, bs, n_total, L, vbs, (cudaStream_t)stream);
}

// ------------------------------------------------------------------ Vb
extern "C" size_t gpp_vb_workspace_bytes(int64_t n, int32_t Q, int32_t L) {
  return tc_rows_supported(n, Q + L, Q) ? tc_vb_workspace_bytes(Q, L) : 0;
}

extern "C" int gpp_vb(const float* V, int64_t ldv, const float* Xb, int64_t ldxb, const float* Binv, const float* W,
                      int64_t ldw, const double* scal, int64_t n, int32_t Q, int32_t L, int32_t L_true, float* Vb,
                      int64_t ldvb, void* workspace, size_t workspace_bytes, gpp_stream_t stream) {
  GPP_REQUIRE(n >= 0 && Q > 0 && L > 0 && Q % 4 == 0 && L % 4 == 0 && L_true > 0 && L_true <= L, "vb: bad shape");
  GPP_REQUIRE(mat_ok(V, ldv, Q) && mat_ok(Xb, ldxb, L) && mat_ok(W, ldw, L) && mat_ok(Vb, ldvb, Q) && Binv &&
                  aligned16(Binv) && scal,
              "vb: bad pointer / leading dimension");
  if (tc_rows_supported(n, Q + L, Q))
    return launch_tc_vb(V, ldv, Xb, ldxb, Binv, W, ldw, scal, n, Q, L, L_true, Vb, ldvb, workspace, workspace_bytes,
                        (cudaStream_t)stream);
  return launch_vb(V, ldv, Xb, ldxb, Binv, Q, W, ldw, scal, n, Q, L, L_true, Vb, ldvb, (cudaStream_t)stream);
}

extern "C" int gpp_kr_slot_sums_planes(const float* X, int64_t ldx, int64_t n, const int64_t* order,
                                       const int64_t* slot_start, const float* xn, int64_t P, int32_t p, int32_t nviews,
                                       int32_t L, int32_t with_x, int32_t max_count, void* planes, size_t planes_bytes_,
                                       gpp_stream_t stream) {
  GPP_REQUIRE(with_x >= 0 && with_x <= 2, "kr_slot_sums_planes: with_x must be 0, 1 or 2");
  const bool reads_x = with_x != 2;
  GPP_REQUIRE((X || !reads_x) && order && slot_start && xn && planes, "kr_slot_sums_planes: null pointer");
  GPP_REQUIRE(n > 0 && P > 0 && p > 0 && nviews > 0 && p % 4 == 0 && (!reads_x || (L > 0 && L % 4 == 0)) && max_count >= 0,
              "kr_slot_sums_planes: p and L must be multiples of 4");
  GPP_REQUIRE((!reads_x || mat_ok(X, ldx, L)) && aligned16(xn) && planes_ok(planes),
              "kr_slot_sums_planes: bad leading dimension / alignment");
  const int64_t cols = (int64_t)nviews * (with_x == 2 ? p : (with_x ? p : 0) + L);
  GPP_REQUIRE(cols < (1ll << 31) && planes_bytes_ >= planes_bytes(P, (int)cols), "kr_slot_sums_planes: planes buffer too small");
  return launch_kr_slot_sums_planes(X, ldx, n, order, slot_start, xn, P, p, nviews, L, with_x, max_count, planes,
                                    (cudaStream_t)stream);
}

extern "C" int gpp_am_planes(const void* planesA, const void* planesB, int64_t n, int32_t k, int32_t m, float alpha,
                             float* out, int64_t ldo, void* workspace, size_t workspace_bytes, gpp_stream_t stream) {
  GPP_REQUIRE(k > 0 && m > 0 && k % 4 == 0 && m % 4 == 0, "am_planes: k and m must be positive multiples of 4");
  GPP_REQUIRE(pl_rows_supported(n, k, m), "am_planes: shape below the tensor-core tile");
  GPP_REQUIRE(planes_ok(planesA) && planes_ok(planesB) && mat_ok(out, ldo, m), "am_planes: bad pointer / leading dimension");
  return launch_pl_am(planesA, planesB, n, k, m, alpha, out, ldo, workspace, workspace_bytes, (cudaStream_t)stream);
}

extern "C" size_t gpp_vb_planes_workspace_bytes(int64_t n, int32_t Q, int32_t L) { return pl_vb_workspace_bytes(n, Q, L); }

extern "C" int gpp_vb_planes(const void* planesV, const float* Xb, int64_t ldxb, const float* Binv, const float* W,
                             int64_t ldw, const double* scal, int64_t n, int32_t Q, int32_t L, int32_t L_true, float* Vb,
                             int64_t ldvb, void* workspace, size_t workspace_bytes, gpp_stream_t stream) {
  GPP_REQUIRE(Q > 0 && L > 0 && Q % 4 == 0 && L % 4 == 0 && L_true > 0 && L_true <= L, "vb_planes: bad shape");
  GPP_REQUIRE(pl_rows_supported(n, Q + L, Q) && Q >= 128, "vb_planes: shape below the tensor-core tile");
  GPP_REQUIRE(planes_ok(planesV) && mat_ok(Xb, ldxb, L) && mat_ok(W, ldw, L) && mat_ok(Vb, ldvb, Q) && Binv &&
                  aligned16(Binv) && scal,
              "vb_planes: bad pointer / leading dimension");
  return launch_pl_vb(planesV, Xb, ldxb, Binv, W, ldw, scal, n, Q, L, L_true, Vb, ldvb, workspace, workspace_bytes,
                      (cudaStream_t)stream);
}

// ------------------------------------------------------------------ host-buffer entry
namespace gpp {
__global__ void softmax2_kernel(const float* __restrict__ lvs, float* __restrict__ vs) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    double v0, vn;
    softmax2(lvs, v0, vn);
    vs[0] = (float)v0;
    vs[1] = (float)vn;
  }
}
}  // namespace gpp

// The host-buffer entry overlaps the PCIe copies with the compute they do not feed:
//   copy-in stream : ALL inputs -> device, the small ones (tables, indices, lvs) first, then X (the N x L latent matrix),
//                    every one double-buffered (slot s), so that a submission's inputs can travel while the previous
//                    submission computes.  One stream because the order matters and nothing else guarantees it: there is
//                    one host -> device copy engine, and the 16 MB of d, w queued behind the 1 GB of X hold the first
//                    kernel back by the whole transfer (experiments/bench/e2e_trace.py, c_entry_trace.py)
//   compute stream : (after the small-inputs event) tables, Khatri-Rao map + planes, the Gram tiles of pass 1 and the
//                    Cholesky -- none of which needs X -- then (after the copy-in event) split X, V^T X, W, pass 2
//   copy-out stream: nll, Xb, vbs -> host, behind the compute of the NEXT submission (two host-facing buffer sets)
// gpp_gp_term_host_submit / _wait expose that pipeline; gpp_gp_term_host = submit + wait.
struct gpp_host_ctx {
  cudaStream_t compute = nullptr, copy_in = nullptr, copy_out = nullptr;
  cudaEvent_t in_done[2] = {nullptr, nullptr}, comp_done[2] = {nullptr, nullptr}, out_done[2] = {nullptr, nullptr};
  cudaEvent_t small_done[2] = {nullptr, nullptr};
  bool out_pending[2] = {false, false}, used[2] = {false, false};
  void* arena = nullptr;
  size_t arena_bytes = 0;
  unsigned next = 0;
};

extern "C" int gpp_host_ctx_create(gpp_host_ctx** ctx) {
  GPP_REQUIRE(ctx, "host_ctx_create: null");
  gpp_host_ctx* c = new gpp_host_ctx();
  cudaError_t e = cudaStreamCreateWithFlags(&c->compute, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&c->copy_in, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&c->copy_out, cudaStreamNonBlocking);
  for (int i = 0; i < 2 && e == cudaSuccess; ++i) {
    e = cudaEventCreateWithFlags(&c->in_done[i], cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->comp_done[i], cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->out_done[i], cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->small_done[i], cudaEventDisableTiming);
  }
  if (e != cudaSuccess) {
    gpp_host_ctx_destroy(c);
    set_error("host_ctx_create: %s", cudaGetErrorString(e));
    return GPP_ERR_CUDA;
  }
  *ctx = c;
  return GPP_OK;
}

extern "C" int gpp_host_ctx_destroy(gpp_host_ctx* ctx) {
  if (!ctx) return GPP_OK;
  if (ctx->compute) cudaStreamSynchronize(ctx->compute);
  if (ctx->copy_out) cudaStreamSynchronize(ctx->copy_out);
  if (ctx->arena) cudaFree(ctx->arena);
  for (int i = 0; i < 2; ++i) {
    if (ctx->in_done[i]) cudaEventDestroy(ctx->in_done[i]);
    if (ctx->comp_done[i]) cudaEventDestroy(ctx->comp_done[i]);
    if (ctx->out_done[i]) cudaEventDestroy(ctx->out_done[i]);
    if (ctx->small_done[i]) cudaEventDestroy(ctx->small_done[i]);
  }
  if (ctx->compute) cudaStreamDestroy(ctx->compute);
  if (ctx->copy_in) cudaStreamDestroy(ctx->copy_in);
  if (ctx->copy_out) cudaStreamDestroy(ctx->copy_out);
  delete ctx;
  return GPP_OK;
}

extern "C" int gpp_gp_term_host_wait(gpp_host_ctx* ctx, int32_t ticket) {
  GPP_REQUIRE(ctx && (ticket == 0 || ticket == 1), "gp_term_host_wait: bad ticket");
  if (ctx->out_pending[ticket]) {
    GPP_CUDA(cudaEventSynchronize(ctx->out_done[ticket]));
    ctx->out_pending[ticket] = false;
  }
  return GPP_OK;
}

extern "C" int gpp_gp_term_host_submit(gpp_host_ctx* ctx, const float* x0_host, int64_t P, int32_t p,
                                       const float* v0_host, int64_t nviews, int32_t q, const int64_t* d_host,
                                       const int64_t* w_host, const float* X_host, int64_t n, int32_t L,
                                       const float* lvs_host, float* nll_host, float* Xb_host, float* vbs_host,
                                       int32_t* ticket) {
  GPP_REQUIRE(ctx && x0_host && v0_host && d_host && w_host && X_host && lvs_host && nll_host && ticket,
              "gp_term_host: null pointer");
  GPP_REQUIRE(P > 0 && p > 0 && nviews > 0 && q > 0 && n > 0 && L > 0, "gp_term_host: bad shape");
  const int64_t Q64 = (int64_t)p * q;
  GPP_REQUIRE(Q64 % 4 == 0 && L % 4 == 0 && Q64 < (1 << 30), "gp_term_host: p*q and L must be multiples of 4");
  const int Q = (int)Q64;
  const bool planes = gpp_planes_supported(n, Q, L) != 0;
  const int s = (int)(ctx->next & 1u);
  // the results of the submission that used this slot must have been collected (its host buffers may be these again)
  GPP_TRY(gpp_gp_term_host_wait(ctx, s));

  // carve the device arena; X, Xb and nll are double-buffered (slot s), everything else is reused submission to submission
  size_t off = 0;
  auto take = [&](size_t bytes) {
    const size_t o = off;
    off += align_up(bytes, 256);
    return o;
  };
  const size_t o_xn = take((size_t)P * p * 4), o_wn = take((size_t)nviews * q * 4);
  const size_t o_vs = take(16), o_scal = take(GPP_NSCAL * 8), o_vbs = take(16);
  size_t o_x0s[2], o_v0s[2], o_ds[2], o_wsl[2], o_lvss[2], o_X[2], o_Xb[2], o_nll[2];
  for (int i = 0; i < 2; ++i) {
    o_x0s[i] = take((size_t)P * p * 4);
    o_v0s[i] = take((size_t)nviews * q * 4);
    o_ds[i] = take((size_t)n * 8);
    o_wsl[i] = take((size_t)n * 8);
    o_lvss[i] = take(16);
    o_X[i] = take((size_t)n * L * 4);
    o_Xb[i] = take((size_t)n * L * 4);
    o_nll[i] = take((size_t)n * 4);
  }
  const size_t o_V = take((size_t)n * Q * 4);
  const size_t o_GC = take((size_t)Q * (Q + L) * 4), o_W = take((size_t)Q * L * 4);
  const size_t o_pV = take(planes ? planes_bytes(n, Q) : 0), o_pX = take(planes ? planes_bytes(n, L) : 0);
  // workspace: the Gram pass (or the split) first; afterwards the factor state sits at its head and the later calls use the rest
  const size_t b_state = align_up(gpp_factor_state_bytes(Q), 256);
  size_t b_tail = gpp_solve_workspace_bytes(Q, L), b_ws;
  if (planes) {
    if (pl_pass1_workspace_bytes(n, Q, L, true) > b_tail) b_tail = pl_pass1_workspace_bytes(n, Q, L, true);
    if (pl_xb_workspace_bytes(n, Q, L) > b_tail) b_tail = pl_xb_workspace_bytes(n, Q, L);
    b_ws = b_state + align_up(b_tail, 256);
    if (pl_pass1_workspace_bytes(n, Q, 0, false) > b_ws) b_ws = pl_pass1_workspace_bytes(n, Q, 0, false);
    if (split_workspace_bytes(n, Q) > b_ws) b_ws = split_workspace_bytes(n, Q);
  } else {
    b_ws = b_state + align_up(b_tail, 256);
    if (gpp_gram_workspace_bytes(n, Q, L) > b_ws) b_ws = gpp_gram_workspace_bytes(n, Q, L);
    if (gpp_xb_workspace_bytes(n, Q, L) > b_ws) b_ws = gpp_xb_workspace_bytes(n, Q, L);
  }
  const size_t o_ws = take(b_ws);
  if (off > ctx->arena_bytes) {
    GPP_CUDA(cudaDeviceSynchronize());
    if (ctx->arena) GPP_CUDA(cudaFree(ctx->arena));
    ctx->arena = nullptr;
    ctx->arena_bytes = 0;
    ctx->used[0] = ctx->used[1] = false;
    GPP_CUDA(cudaMalloc(&ctx->arena, off));
    ctx->arena_bytes = off;
  }
  char* a = static_cast<char*>(ctx->arena);
  auto F = [&](size_t o) { return reinterpret_cast<float*>(a + o); };
  const size_t o_x0 = o_x0s[s], o_v0 = o_v0s[s], o_lvs = o_lvss[s];
  int64_t* d_dev = reinterpret_cast<int64_t*>(a + o_ds[s]);
  int64_t* w_dev = reinterpret_cast<int64_t*>(a + o_wsl[s]);
  double* scal = reinterpret_cast<double*>(a + o_scal);
  cudaStream_t st = ctx->compute;

  // copy-in stream: the inputs of slot s, once the compute that last read this slot is done; small ones first
  cudaStream_t ci = ctx->copy_in;
  if (ctx->used[s]) GPP_CUDA(cudaStreamWaitEvent(ci, ctx->comp_done[s], 0));
  GPP_CUDA(cudaMemcpyAsync(F(o_x0), x0_host, (size_t)P * p * 4, cudaMemcpyHostToDevice, ci));
  GPP_CUDA(cudaMemcpyAsync(F(o_v0), v0_host, (size_t)nviews * q * 4, cudaMemcpyHostToDevice, ci));
  GPP_CUDA(cudaMemcpyAsync(d_dev, d_host, (size_t)n * 8, cudaMemcpyHostToDevice, ci));
  GPP_CUDA(cudaMemcpyAsync(w_dev, w_host, (size_t)n * 8, cudaMemcpyHostToDevice, ci));
  GPP_CUDA(cudaMemcpyAsync(F(o_lvs), lvs_host, 8, cudaMemcpyHostToDevice, ci));
  GPP_CUDA(cudaEventRecord(ctx->small_done[s], ci));
  GPP_CUDA(cudaMemcpyAsync(F(o_X[s]), X_host, (size_t)n * L * 4, cudaMemcpyHostToDevice, ci));
  GPP_CUDA(cudaEventRecord(ctx->in_done[s], ci));

  // compute stream: everything that does not need X
  GPP_CUDA(cudaStreamWaitEvent(st, ctx->small_done[s], 0));
  GPP_TRY(gpp_normalize_rows_fwd(F(o_x0), P, p, F(o_xn), st));
  GPP_TRY(gpp_normalize_rows_fwd(F(o_v0), nviews, q, F(o_wn), st));
  softmax2_kernel<<<1, 32, 0, st>>>(F(o_lvs), F(o_vs));
  GPP_LAUNCH_CHECK();
  if (planes) {
    GPP_TRY(gpp_khatri_rao_fwd_planes(F(o_xn), P, p, F(o_wn), nviews, q, d_dev, w_dev, n, F(o_V), Q, a + o_pV,
                                      planes_bytes(n, Q), a + o_ws, b_ws, st));
    // Gram tiles alone (L = 0), then the Cholesky: X is still in flight
    GPP_TRY(gpp_gram_vtz_planes(a + o_pV, nullptr, n, Q, 0, 1, F(o_GC), Q + L, a + o_ws, b_ws, st));
    GPP_TRY(gpp_factor(F(o_GC), Q + L, Q, F(o_vs), 0, nullptr, scal, a + o_ws, b_state, st));
    GPP_CUDA(cudaStreamWaitEvent(st, ctx->in_done[s], 0));
    // the factor state occupies the head of the workspace: the rest serves the calls below
    char* ws2 = a + o_ws + b_state;
    const size_t ws2_bytes = b_ws - b_state;
    GPP_TRY(gpp_split_planes(F(o_X[s]), L, n, L, 0, a + o_pX, planes_bytes(n, L), nullptr, 0, st));
    GPP_TRY(gpp_atb_planes(a + o_pV, a + o_pX, n, Q, L, F(o_GC) + Q, Q + L, ws2, ws2_bytes, st));
    GPP_TRY(gpp_solve_w(F(o_GC) + Q, Q + L, Q, L, L, n, F(o_W), L, scal, a + o_ws, b_state, ws2, ws2_bytes, st));
    if (ctx->used[s]) GPP_CUDA(cudaStreamWaitEvent(st, ctx->out_done[s], 0));   // Xb / nll of slot s have left the device
    GPP_TRY(gpp_xb_nll_planes(a + o_pV, F(o_X[s]), L, F(o_W), L, n, Q, L, scal, F(o_Xb[s]), L, F(o_nll[s]), ws2, ws2_bytes,
                              st));
  } else {
    GPP_TRY(gpp_khatri_rao_fwd(F(o_xn), P, p, F(o_wn), nviews, q, d_dev, w_dev, n, F(o_V), Q, st));
    GPP_CUDA(cudaStreamWaitEvent(st, ctx->in_done[s], 0));
    GPP_TRY(gpp_gram_vtz(F(o_V), Q, F(o_X[s]), L, n, Q, L, F(o_GC), Q + L, a + o_ws, b_ws, st));
    GPP_TRY(gpp_factor_solve(F(o_GC), Q + L, Q, L, F(o_vs), n, 0, F(o_W), L, nullptr, scal, a + o_ws, b_ws, st));
    // (gpp_factor_solve keeps the factor state at the head of the workspace; pass 2 below must not overwrite it only if a
    //  later call needed it -- none does)
    if (ctx->used[s]) GPP_CUDA(cudaStreamWaitEvent(st, ctx->out_done[s], 0));
    GPP_TRY(gpp_xb_nll(F(o_V), Q, F(o_X[s]), L, F(o_W), L, n, Q, L, scal, F(o_Xb[s]), L, F(o_nll[s]), a + o_ws, b_ws, st));
  }
  GPP_TRY(gpp_vbs(scal, n, Q, L, F(o_vbs), st));
  if (vbs_host) GPP_CUDA(cudaMemcpyAsync(vbs_host, F(o_vbs), 8, cudaMemcpyDeviceToHost, st));
  GPP_CUDA(cudaEventRecord(ctx->comp_done[s], st));

  // copy-out stream: behind this submission's compute, beside the next one's
  GPP_CUDA(cudaStreamWaitEvent(ctx->copy_out, ctx->comp_done[s], 0));
  GPP_CUDA(cudaMemcpyAsync(nll_host, F(o_nll[s]), (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->copy_out));
  if (Xb_host) GPP_CUDA(cudaMemcpyAsync(Xb_host, F(o_Xb[s]), (size_t)n * L * 4, cudaMemcpyDeviceToHost, ctx->copy_out));
  GPP_CUDA(cudaEventRecord(ctx->out_done[s], ctx->copy_out));
  ctx->out_pending[s] = true;
  ctx->used[s] = true;
  *ticket = s;
  ++ctx->next;
  return GPP_OK;
}

extern "C" int gpp_gp_term_host(gpp_host_ctx* ctx, const float* x0_host, int64_t P, int32_t p, const float* v0_host,
                                int64_t nviews, int32_t q, const int64_t* d_host, const int64_t* w_host,
                                const float* X_host, int64_t n, int32_t L, const float* lvs_host, float* nll_host,
                                float* Xb_host, float* vbs_host) {
  int32_t ticket = 0;
  GPP_TRY(gpp_gp_term_host_submit(ctx, x0_host, P, p, v0_host, nviews, q, d_host, w_host, X_host, n, L, lvs_host,
                                  nll_host, Xb_host, vbs_host, &ticket));
  return gpp_gp_term_host_wait(ctx, ticket);
}
