/*
 * gppvae_b200.h -- C ABI of libgppvae_b200.so: the B200 (sm_100a) implementation of the
 * low-rank Gaussian-process prior term of GPPVAE.
 *
 * The reference (ahmerb/GPPVAE) has no FFI: its boundary for this path is the Python class
 * API of pysrc/faceplace/gp.py and vmod.py, whose bodies are sequences of torch library calls.
 * Every entry point below replaces one such sequence; the reference lines are cited on each.
 * gppvae_b200/gp.py and gppvae_b200/vmod.py bind these symbols with ctypes and present the
 * reference's GP / Vmodel classes on top (INTEGRATION.md shows the stub).
 *
 * Conventions
 *   - plain C types only; no torch / ATen / pybind types cross this boundary;
 *   - all matrices are float32, row-major, with an explicit leading dimension (elements);
 *     every pointer must be 16-byte aligned and every leading dimension and every column count
 *     (Q, L, p*q) a multiple of 4 (the Python layer zero-pads columns when it has to);
 *   - indices are int64 (the reference's .long(), train_gppvae.py:123-126);
 *   - pointers are DEVICE pointers unless the name ends in _host; memory is caller-owned, the
 *     library never allocates or frees user-visible memory; scratch comes from a caller-provided
 *     workspace whose size the matching *_workspace_bytes() call reports;
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*), performs no host
 *     synchronisation and never changes the current device (gpp_gp_term_host is the exception:
 *     it is the host-buffer convenience entry and synchronises before returning);
 *   - return value: 0 on success, a negative gpp_status otherwise; gpp_last_error() returns the
 *     message of the last failure on the calling thread;
 *   - the variance parameters travel as DEVICE vectors (vs = softmax(lvs), gp.py:48-50, or lvs itself
 *     for the Taylor surrogate), so no call needs a host read of a parameter.
 */
#ifndef GPPVAE_B200_H_
#define GPPVAE_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* gpp_stream_t; /* cudaStream_t */

enum gpp_status {
  GPP_OK = 0,
  GPP_ERR_INVALID_ARGUMENT = -1, /* null pointer, misaligned pointer, bad size or leading dimension */
  GPP_ERR_CUDA = -2,             /* a CUDA runtime / driver call failed; see gpp_last_error() */
  GPP_ERR_WORKSPACE = -3,        /* workspace smaller than *_workspace_bytes() */
  GPP_ERR_UNSUPPORTED = -4       /* shape outside what the kernels were built for */
};

/* Slots of the device-side double[GPP_NSCAL] scalar block shared by the GP-term calls. */
enum gpp_scalar_slot {
  GPP_S_V0 = 0,        /* softmax(lvs)[0]                         gp.py:50 */
  GPP_S_VN = 1,        /* softmax(lvs)[1]                         gp.py:50 */
  GPP_S_LOGDETB = 2,   /* log|I + (v0/vn) V^T V| = sum log Shb    gp.py:33,86 */
  GPP_S_TRBINV = 3,    /* tr B^-1 (over the Q real columns)       gp.py:79 via tr K^-1 */
  GPP_S_WNORM2 = 4,    /* ||W||_F^2, W = (v0/vn) B^-1 V^T X       gp.py:75 */
  GPP_S_ROWCONST = 5,  /* 0.5 L (log vn + logdetB / n_total)      gp.py:85-87 */
  GPP_S_XB2 = 6,       /* sum Xb^2  over the rows of this call    gp.py:80 */
  GPP_S_QUAD = 7,      /* sum_i X_i . Xb_i over the rows of this call  gp.py:84 */
  GPP_NSCAL = 8
};

/* flags for gpp_factor / gpp_factor_solve */
#define GPP_WANT_BINV 1u /* also form B^-1 (needed by gpp_vb, i.e. by the full taylor_coeff) */

int gpp_version(void);
const char* gpp_last_error(void);
/* Which GEMM engine the library was built with: "tcgen05-3xf16" (3-term split of every fp32 product on the fp16 tensor
 * pipe; the Q-space block GEMMs keep a TF32 main term) or "simt-fp32". */
const char* gpp_gemm_engine(void);
/* Number of kernels this library has launched in the process so far (bench.py reports the delta). */
uint64_t gpp_launch_count(void);

/* ---------------- Vmodel (vmod.py) ---------------- */

/* y = x / sqrt(rowsum(x^2))                                   vmod.py:10-12 (normalize_rows) */
int gpp_normalize_rows_fwd(const float* x, int64_t rows, int64_t cols, float* y, gpp_stream_t stream);
/* gx = (gy - y (y . gy)) / |x| : backward of the above        autograd of vmod.py:10-12 */
int gpp_normalize_rows_bwd(const float* x, const float* gy, int64_t rows, int64_t cols, float* gx,
                           gpp_stream_t stream);

/* V[i, j*q + k] = xn[d_i, j] * wn[w_i, k]                     vmod.py:28-35 (Vmodel.forward)
 * xn is (P x p), wn is (nviews x q), both already row-normalised; V is (n x p*q), ld = ldv.
 * An index outside its table yields a row of NaN. */
int gpp_khatri_rao_fwd(const float* xn, int64_t P, int32_t p, const float* wn, int64_t nviews, int32_t q,
                       const int64_t* d, const int64_t* w, int64_t n, float* V, int64_t ldv,
                       gpp_stream_t stream);
/* gxn[d_i, j] += sum_k gV[i, j*q+k] wn[w_i, k];  gwn[w_i, k] += sum_j gV[i, j*q+k] xn[d_i, j]
 * (backward of vmod.py:30-34; gxn and gwn must be zeroed by the caller). */
int gpp_khatri_rao_bwd(const float* gV, int64_t ldg, const float* xn, int64_t P, int32_t p, const float* wn,
                       int64_t nviews, int32_t q, const int64_t* d, const int64_t* w, int64_t n, float* gxn,
                       float* gwn, gpp_stream_t stream);

/* ---------------- GP (gp.py) ---------------- */

/* Pass 1: GC = V^T [V | X]  (Q x (Q+L), ld = ldgc); both triangles of G are written.
 * Replaces the U^T U of gp.py:30 and the U^T X of gp.py:42 (and gp.py:68) in one sweep over the rows.
 * Rows may be a shard: partial GC of different ranks are summed by the caller (NCCL all-reduce). */
size_t gpp_gram_workspace_bytes(int64_t n, int32_t Q, int32_t L);
int gpp_gram_vtz(const float* V, int64_t ldv, const float* X, int64_t ldx, int64_t n, int32_t Q, int32_t L,
                 float* GC, int64_t ldgc, void* workspace, size_t workspace_bytes, gpp_stream_t stream);

/* Same contract as gpp_gram_vtz, always on the fp32 SIMT tile engine (cross-check entry used by the tests). */
int gpp_gram_vtz_simt(const float* V, int64_t ldv, const float* X, int64_t ldx, int64_t n, int32_t Q, int32_t L,
                      float* GC, int64_t ldgc, void* workspace, size_t workspace_bytes, gpp_stream_t stream);

/* Q-space solve, replicated on every rank.  vs = [v0, vn] is the DEVICE vector softmax(lvs) (gp.py:50).
 *
 * gpp_factor:   B = I + (v0/vn) G = Lc Lc^T (blocked Cholesky; replaces svd + inverse of gp.py:33-35),
 *               Linv = Lc^-1, scal[V0, VN, LOGDETB, TRBINV]; with GPP_WANT_BINV also Binv = B^-1 (Q x Q, ld = Q).
 *               `state` (gpp_factor_state_bytes) receives the factorisation: keep it to call gpp_solve_w()
 *               for further right-hand sides (the reference factors twice per epoch on identical inputs,
 *               train_gppvae.py:235 and :166 -- cache this buffer instead).
 * gpp_solve_w:  W = (v0/vn) B^-1 C for C = V^T X (Q x L, ld = ldc), scal[WNORM2, ROWCONST].
 *               n_total is the global number of rows (all ranks); L_true <= L is the number of real latent
 *               columns when X was zero-padded to a multiple of 4 (it enters ROWCONST only).
 * gpp_factor_solve: both, with G = GC[:, :Q] and C = GC[:, Q:]; `workspace` must hold
 *               gpp_factor_state_bytes(Q) + gpp_solve_workspace_bytes(Q, L). */
size_t gpp_factor_state_bytes(int32_t Q);
size_t gpp_solve_workspace_bytes(int32_t Q, int32_t L);
int gpp_factor(const float* G, int64_t ldg, int32_t Q, const float* vs, uint32_t flags, float* Binv, double* scal,
               void* state, size_t state_bytes, gpp_stream_t stream);
int gpp_solve_w(const float* C, int64_t ldc, int32_t Q, int32_t L, int32_t L_true, int64_t n_total, float* W,
                int64_t ldw, double* scal, const void* state, size_t state_bytes, void* workspace,
                size_t workspace_bytes, gpp_stream_t stream);
int gpp_factor_solve(const float* GC, int64_t ldgc, int32_t Q, int32_t L, const float* vs, int64_t n_total,
                     uint32_t flags, float* W, int64_t ldw, float* Binv, double* scal, void* workspace,
                     size_t workspace_bytes, gpp_stream_t stream);

/* Pass 2 + epilogue: Xb = (X - V W) / vn  (= K^-1 X, gp.py:42-44), nll_i = 0.5 X_i.Xb_i + ROWCONST
 * (gp.py:84-87), and scal[XB2], scal[QUAD] for these rows (overwritten, not accumulated). */
size_t gpp_xb_workspace_bytes(int64_t n, int32_t Q, int32_t L);
int gpp_xb_nll(const float* V, int64_t ldv, const float* X, int64_t ldx, const float* W, int64_t ldw, int64_t n,
               int32_t Q, int32_t L, double* scal, float* Xb, int64_t ldxb, float* nll, void* workspace,
               size_t workspace_bytes, gpp_stream_t stream);

/* vbs = [dNLL/dv0, dNLL/dvn] (gp.py:75-76,79-81) from the scalar block; xb2_total = sum Xb^2 over ALL ranks
 * is read from scal[XB2] (the caller all-reduces that slot first when rows are sharded). */
int gpp_vbs(const double* scal, int64_t n_total, int32_t Q, int32_t L, float* vbs, gpp_stream_t stream);

/* Vb = v0 (L K^-1 V - Xb Xb^T V)  (gp.py:68-71)  computed as  (v0/vn) L_true V B^-1 - Xb W^T.
 * L is the (padded) width of Xb and W, L_true the number of real latent columns. */
size_t gpp_vb_workspace_bytes(int64_t n, int32_t Q, int32_t L);
int gpp_vb(const float* V, int64_t ldv, const float* Xb, int64_t ldxb, const float* Binv, const float* W,
           int64_t ldw, const double* scal, int64_t n, int32_t Q, int32_t L, int32_t L_true, float* Vb,
           int64_t ldvb, void* workspace, size_t workspace_bytes, gpp_stream_t stream);

/* out = alpha * (X - A M)   X:(n x m) A:(n x k) M:(k x m).  The generic form of gp.py:42-44 used by
 * GP.solve() when the caller hands in dense U / UBi tensors.  alpha is a host scalar. */
/* (workspace: gpp_rows_workspace_bytes() bytes, 16-byte aligned -- it receives the operands' exact maxima, from which
 * the fp16 operand scales of the tensor-core form are derived; may be NULL below the tensor-core tile) */
size_t gpp_rows_workspace_bytes(void);
int gpp_x_minus_am(const float* X, int64_t ldx, const float* A, int64_t lda, const float* M, int64_t ldm,
                   int64_t n, int32_t k, int32_t m, float alpha, float* out, int64_t ldo, void* workspace,
                   size_t workspace_bytes, gpp_stream_t stream);
/* ---------------- pre-split operand planes (the fast form of the two N-long sweeps) ----------------
 * The tensor cores take fp16 operands; an fp32-accurate product needs every operand as hi + lo (hi = the value rounded
 * to 11 significant bits, lo = the remainder, one power-of-two scale per matrix).  A `planes` buffer holds that form
 * of one fp32 matrix ONCE -- same 4 bytes per element -- so that gpp_gram_vtz_planes / gpp_xb_nll_planes stream it
 * with the copy engine straight into the tensor cores (no conversion inside the GEMM kernels).  The buffer is opaque,
 * caller-owned, gpp_planes_bytes(n, cols) long, 256-byte aligned; it also carries the matrix' exact column sums of
 * squares when requested (they become the diagonal of V^T V: gp.py:30's U^T U has an exactly representable
 * same-sign diagonal that the truncating tensor-core accumulator would otherwise bias).
 *   gpp_split_planes           X (n x cols, fp32) -> planes.  flags: GPP_PLANES_COLSQ, GPP_PLANES_UNIT_BOUND.
 *   gpp_khatri_rao_fwd_planes  vmod.py:28-35 writing V (fp32, what Vmodel.forward returns) AND its planes (with
 *                              column sums of squares) in one sweep.
 *   gpp_gram_vtz_planes        the contract of gpp_gram_vtz with both operands as planes (planesX may be NULL when L = 0);
 *                              use_colsq != 0 writes the exact diagonal.
 *   gpp_atb_planes             out = A^T B (ka x kb) from planes (a further right-hand side on a cached factorisation).
 *   gpp_xb_nll_planes          the contract of gpp_xb_nll with V as planes (X and W stay fp32; W is split internally). */
#define GPP_PLANES_COLSQ 1u      /* also accumulate the column sums of squares (fp64, fixed order) */
#define GPP_PLANES_UNIT_BOUND 2u /* caller guarantees |x| <= 1: skip the magnitude scan */
size_t gpp_planes_bytes(int64_t n, int32_t cols);
size_t gpp_split_workspace_bytes(int64_t n, int32_t cols);
int gpp_split_planes(const float* X, int64_t ldx, int64_t n, int32_t cols, uint32_t flags, void* planes,
                     size_t planes_bytes, void* workspace, size_t workspace_bytes, gpp_stream_t stream);
int gpp_khatri_rao_fwd_planes(const float* xn, int64_t P, int32_t p, const float* wn, int64_t nviews, int32_t q,
                              const int64_t* d, const int64_t* w, int64_t n, float* V, int64_t ldv, void* planes,
                              size_t planes_bytes, void* workspace, size_t workspace_bytes, gpp_stream_t stream);
size_t gpp_gram_planes_workspace_bytes(int64_t n, int32_t Q, int32_t L);
int gpp_gram_vtz_planes(const void* planesV, const void* planesX, int64_t n, int32_t Q, int32_t L, int32_t use_colsq,
                        float* GC, int64_t ldgc, void* workspace, size_t workspace_bytes, gpp_stream_t stream);
int gpp_atb_planes(const void* planesA, const void* planesB, int64_t n, int32_t ka, int32_t kb, float* out,
                   int64_t ldo, void* workspace, size_t workspace_bytes, gpp_stream_t stream);
size_t gpp_xb_planes_workspace_bytes(int64_t n, int32_t Q, int32_t L);
int gpp_xb_nll_planes(const void* planesV, const float* X, int64_t ldx, const float* W, int64_t ldw, int64_t n,
                      int32_t Q, int32_t L, double* scal, float* Xb, int64_t ldxb, float* nll, void* workspace,
                      size_t workspace_bytes, gpp_stream_t stream);
/* the contract of gpp_vb with V as planes (Xb, Binv, W stay fp32 and are split internally) */
size_t gpp_vb_planes_workspace_bytes(int64_t n, int32_t Q, int32_t L);
int gpp_vb_planes(const void* planesV, const float* Xb, int64_t ldxb, const float* Binv, const float* W, int64_t ldw,
                  const double* scal, int64_t n, int32_t Q, int32_t L, int32_t L_true, float* Vb, int64_t ldvb,
                  void* workspace, size_t workspace_bytes, gpp_stream_t stream);
/* 1 when the planes kernels take this shape (n >= 512, Q >= 128), else the fp32 entries must be used */
int gpp_planes_supported(int64_t n, int32_t Q, int32_t L);

/* out = A^T B   A:(n x ka) B:(n x kb) -> (ka x kb).  Generic form of gp.py:42 (U^T X). */
size_t gpp_atb_workspace_bytes(int64_t n, int32_t ka, int32_t kb);
int gpp_atb(const float* A, int64_t lda, const float* B, int64_t ldb, int64_t n, int32_t ka, int32_t kb,
            float* out, int64_t ldo, void* workspace, size_t workspace_bytes, gpp_stream_t stream);

/* out = alpha * A M   A:(n x k) M:(k x m).  (Y = xn [M_0 | M_1 | ...] of the structured path below.) */
int gpp_am(const float* A, int64_t lda, const float* M, int64_t ldm, int64_t n, int32_t k, int32_t m, float alpha,
           float* out, int64_t ldo, void* workspace, size_t workspace_bytes, gpp_stream_t stream);

/* ---------------- several random effects: GP(n_rand_effs = k)  (gp.py:21-22,27,55-95,127-133) ----------------
 * K = sum_i v_i V_i V_i^T + vn I with vs = softmax(lvs) = [v_0 .. v_{k-1}, vn] (k + 1 entries, DEVICE vector).  The
 * designs are stacked, V = [V_0 | ... | V_{k-1}] (n x Q, Q = sum Q_i; gp.py:27 concatenates sqrt(v_i) V_i), and with
 * D = diag(sqrt(v_i) on the columns of block i):
 *   B = I + D G D / vn (G = V^T V),   W = D B^-1 D C / vn (C = V^T X),   Xb = (X - V W) / vn.
 * Block column counts travel as a HOST int32 array cols_host[k] (each a positive multiple of 4, k <= GPP_MAX_DESIGNS);
 * per-block scalars as a caller-owned DEVICE double[2k]: blk[2i] = tr_i B^-1 (the diagonal of B^-1 over block i),
 * blk[2i + 1] = ||W_i||^2 (row block i of W).
 *   gpp_split_planes_stacked  planes of the concatenation written directly from the k fp32 sources (X_host: HOST array of
 *                             k device pointers, ldx_host their leading dimensions): one exact magnitude scan over all
 *                             sources (skipped with GPP_PLANES_UNIT_BOUND), every source column written once into its
 *                             column range, the column sums of squares (GPP_PLANES_COLSQ) in a fixed order.  The buffer is
 *                             what gpp_split_planes makes of the concatenation: every *_planes entry takes it.
 *   gpp_factor_blocks         gp.py:27-35 for k designs: the Cholesky of B as gpp_factor does it; writes
 *                             scal[V0] = 1, scal[VN] = vn, LOGDETB, TRBINV (all blocks), blk[2i]; with GPP_WANT_BINV,
 *                             Binv = D B^-1 D.  With scal[V0] = 1 and this Binv, gpp_xb_nll(_planes) and gpp_vb(_planes)
 *                             compute the k-design Xb, nll (gp.py:42-44,84-87) and Vb = [Vb_0 | ... ] (gp.py:68-71)
 *                             unchanged.  The state also serves gpp_solve_w (W without the per-block norms).
 *   gpp_solve_w_blocks        W = D B^-1 D C / vn, scal[WNORM2, ROWCONST] as gpp_solve_w, and blk[2i + 1].
 *   gpp_vbs_blocks            vbs (k + 1 entries, gp.py:75-81):  vbs[i] = -||W_i||^2 / (2 v_i^2) + L (Q_i - tr_i B^-1) / (2 v_i),
 *                             vbs[k] = -sum Xb^2 / 2 + L (n_total - Q + tr B^-1) / (2 vn); sum Xb^2 from scal[XB2]
 *                             (all-reduced by the caller when rows are sharded). */
#define GPP_MAX_DESIGNS 16
size_t gpp_split_stacked_workspace_bytes(int64_t n, int32_t k, const int32_t* cols_host);
int gpp_split_planes_stacked(int32_t k, const float* const* X_host, const int64_t* ldx_host, const int32_t* cols_host,
                             int64_t n, uint32_t flags, void* planes, size_t planes_bytes, void* workspace,
                             size_t workspace_bytes, gpp_stream_t stream);
size_t gpp_factor_blocks_state_bytes(int32_t Q, int32_t k);
int gpp_factor_blocks(const float* G, int64_t ldg, int32_t k, const int32_t* cols_host, const float* vs, uint32_t flags,
                      float* Binv, double* scal, double* blk, void* state, size_t state_bytes, gpp_stream_t stream);
size_t gpp_solve_blocks_workspace_bytes(int32_t Q, int32_t L, int32_t k);
int gpp_solve_w_blocks(const float* C, int64_t ldc, int32_t k, const int32_t* cols_host, int32_t L, int32_t L_true,
                       int64_t n_total, float* W, int64_t ldw, double* scal, double* blk, const void* state,
                       size_t state_bytes, void* workspace, size_t workspace_bytes, gpp_stream_t stream);
int gpp_vbs_blocks(const double* scal, const double* blk, const float* vs, int32_t k, const int32_t* cols_host,
                   int64_t n_total, int32_t L, float* vbs, gpp_stream_t stream);
/* Taylor surrogate over k designs (gp.py:127-133):  out_i = Xb_i.X_i + sum_j Vb_j,i.V_j,i + <vbs, softmax(lvs)> / n,
 * vbs and lvs of k + 1 entries; V_host / Vb_host are HOST arrays of k device pointers, Q_host the designs' column counts
 * (multiples of 4).  Backward: gX = gout_i Xb_i, gV_j = gout_i Vb_j, glvs = J_softmax^T vbs * sum(gout) / n (k + 1
 * entries); gX, glvs and any gV_host[j] may be NULL when that gradient is not needed.  One launch each whatever k is. */
int gpp_taylor_expansion_fwd_multi(const float* X, int64_t ldx, const float* Xb, int64_t ldxb, int32_t k,
                                   const float* const* V_host, const int64_t* ldv_host, const float* const* Vb_host,
                                   const int64_t* ldvb_host, const int32_t* Q_host, int64_t n, int32_t L,
                                   const float* vbs, const float* lvs, float* out, gpp_stream_t stream);
int gpp_taylor_expansion_bwd_multi(const float* gout, const float* Xb, int64_t ldxb, int32_t k,
                                   const float* const* Vb_host, const int64_t* ldvb_host, const int32_t* Q_host,
                                   int64_t n, int32_t L, const float* vbs, const float* lvs, float* gX, int64_t ldgx,
                                   float* const* gV_host, const int64_t* ldgv_host, float* glvs, gpp_stream_t stream);

/* ---------------- structured Khatri-Rao path (V never materialised; SURVEY.md 8(f) row 4) ----------------
 * V[i, j q + k] = xn[d_i, j] wn[w_i, k] (vmod.py:28-35), so V^T V, V^T X and V W (gp.py:30,42-44) factor through the
 * (object, view) slots s = o * nviews + v:
 *   gpp_kr_slot_sums   XZ (P x nviews (p + L)):  XZ[o, v p + j] = cnt[s] xn[o, j],  XZ[o, nviews p + v L + l] = sum of
 *                      X[i, l] over the rows of slot s.  `order` lists the row indices sorted by slot and
 *                      slot_start (P nviews + 1) the first position of every slot in it (both int64, device; the
 *                      caller prepares them once per (d, w)); rows of a slot are added in that order (deterministic).
 *   ST = xn^T XZ       (p x nviews (p + L)) with gpp_atb: S_v = ST[:, v p ..], T_v = ST[:, nviews p + v L ..]
 *                      (row-sharded callers all-reduce ST, 8 MB at c3, instead of GC)
 *   gpp_kr_assemble_gc GC[(j,k), (j',k')] = sum_v wn[v,k] wn[v,k'] S_v[j,j'],  GC[(j,k), Q + l] = sum_v wn[v,k] T_v[j,l]
 *                      -- the same GC = V^T [V | X] gpp_gram_vtz produces; gpp_factor / gpp_solve_w follow unchanged
 *   gpp_kr_assemble_m  M (p x nviews L):  M[j, v L + l] = sum_k wn[v,k] W[(j,k), l];  then Y = xn M with gpp_am
 *   gpp_kr_xb_nll      Xb_i = (X_i - Y[d_i, w_i L ..]) / vn, nll, scal[XB2], scal[QUAD]   (the contract of gpp_xb_nll)
 * with_x = 0 / with_g = 0: only the X part (XZ, ST are nviews L wide; GC is C alone) -- a further right-hand side on
 * a cached factorisation.  p, p*q and L must be multiples of 4. */
int gpp_kr_slot_sums(const float* X, int64_t ldx, const int64_t* order, const int64_t* slot_start, const float* xn,
                     int64_t P, int32_t p, int32_t nviews, int32_t L, int32_t with_x, float* XZ, int64_t ldxz,
                     gpp_stream_t stream);
/* The same two products on operand planes (shapes from the tensor-core tile up: P >= 512, p >= 128):
 *   gpp_kr_slot_sums_planes  XZ written directly as planes (gpp_planes_bytes(P, cols)): no fp32 copy, and no scan of
 *                            it -- the scale comes from a bound, with max_count = the largest number of rows in one slot
 *                            (the caller knows it from the index) and max|X| from one read of X (n rows):
 *                              with_x = 0  the slot sums alone, cols = nviews L, scale bound max_count max|X|;
 *                              with_x = 2  cnt (x) xn alone, cols = nviews p, scale bound max_count (X is not read and
 *                                          may be NULL; L is ignored);
 *                              with_x = 1  both, cols = nviews (p + L), ONE scale for both, max_count max(1, max|X|):
 *                                          the range far below that bound keeps fewer bits (|X| >> 1 costs cnt (x) xn
 *                                          its precision, |X| << 1 or one crowded slot the slot sums).
 *                            ST = xn^T XZ is then gpp_atb_planes; the route writes ST as two products (with_x = 2 and
 *                            0, each into its column range of ST through ldo), so that each range keeps its own scale.
 *   gpp_am_planes            out = alpha A M from the planes of A (n x k) and M (k x m): Y = xn [M_0 | M_1 | ...];
 *                            workspace: 256 bytes. */
int gpp_kr_slot_sums_planes(const float* X, int64_t ldx, int64_t n, const int64_t* order, const int64_t* slot_start,
                            const float* xn, int64_t P, int32_t p, int32_t nviews, int32_t L, int32_t with_x,
                            int32_t max_count, void* planes, size_t planes_bytes, gpp_stream_t stream);
int gpp_am_planes(const void* planesA, const void* planesB, int64_t n, int32_t k, int32_t m, float alpha, float* out,
                  int64_t ldo, void* workspace, size_t workspace_bytes, gpp_stream_t stream);
int gpp_kr_assemble_gc(const float* ST, int64_t ldst, const float* wn, int32_t p, int32_t q, int32_t nviews, int32_t L,
                       int32_t with_g, float* GC, int64_t ldgc, gpp_stream_t stream);
int gpp_kr_assemble_m(const float* W, int64_t ldw, const float* wn, int32_t p, int32_t q, int32_t nviews, int32_t L,
                      float* M, int64_t ldm, gpp_stream_t stream);
size_t gpp_kr_xb_workspace_bytes(int64_t n);
int gpp_kr_xb_nll(const float* X, int64_t ldx, const float* Y, int64_t ldy, const int64_t* d, const int64_t* w,
                  int64_t n, int64_t P, int32_t nviews, int32_t L, double* scal, float* Xb, int64_t ldxb, float* nll,
                  void* workspace, size_t workspace_bytes, gpp_stream_t stream);
/* NLL gradient to the tables (DESIGN 5.8): the Khatri-Rao backward of Vb = alpha V B^-1 - Xb W^T, alpha = (v0/vn) L_true,
 * through the slots.  With H_v = (I_p (x) wn_v)^T B^-1 (I_p (x) wn_v) (p x p) and M_v as in gpp_kr_assemble_m:
 *   gpp_kr_grad_rhs    R (nviews (p + L) x p, ld = ldr):  R[v p + j', j] = alpha H_v[j', j],
 *                      R[nviews p + v L + l, j] = -M_v[j, l], so that
 *                      gxn = [cnt (x) xn | slot sums of Xb] R  (gpp_kr_slot_sums with_x = 1 and gpp_am, or the two
 *                      ranges as planes, with_x = 2 and 0, and two gpp_am_planes summed).
 *   gpp_kr_grad_views  gw (nviews x q, ld = ldgw) from ST = xn^T [cnt (x) xn | slot sums of Xb] (p x nviews (p + L), as
 *                      gpp_atb writes it: S_v[j, j'] = ST[j, v p + j'], T_v[j, l] = ST[j, nviews p + v L + l]):
 *                      gw[v, k] = alpha sum_{j,j',k'} S_v[j,j'] wn[v,k'] B^-1[(j',k'),(j,k)] - sum_{j,l} T_v[j,l] W[(j,k),l];
 *                      workspace: gpp_kr_grad_views_workspace_bytes (p nviews q floats).
 * Padding: the rows of R for zero (padded) columns of W are exactly zero.  The alpha H_v rows and columns of padded
 * object features (p rounded up to 4) are NOT zero: there B^-1 is the identity, so R[v p + j, j] = alpha |wn_v|^2.  They
 * meet zero columns of cnt (x) xn, so gxn's padded columns come out zero, and the caller drops them.
 * Both read B^-1 (ld = ldb >= p q) once, in tiles of q rows shared by all views, and reduce in a fixed order without
 * atomics: repeats are bit-identical.  p and L must be multiples of 4; nviews q floats must fit 48 KB, and one tile of
 * B^-1 with the view table, (q (q + 1) + nviews q) floats, must fit 160 KB of shared memory (q up to about 200). */
int gpp_kr_grad_rhs(const float* Binv, int64_t ldb, const float* W, int64_t ldw, const float* wn, int32_t p, int32_t q,
                    int32_t nviews, int32_t L, double alpha, float* R, int64_t ldr, gpp_stream_t stream);
size_t gpp_kr_grad_views_workspace_bytes(int32_t p, int32_t q, int32_t nviews);
int gpp_kr_grad_views(const float* ST, int64_t ldst, const float* Binv, int64_t ldb, const float* W, int64_t ldw,
                      const float* wn, int32_t p, int32_t q, int32_t nviews, int32_t L, double alpha, float* gw,
                      int64_t ldgw, void* workspace, size_t workspace_bytes, gpp_stream_t stream);

/* ---------------- several factored designs over one slot index (GP(n_rand_effs = k), k <= 3) ----------------
 * The Khatri-Rao design V_K = xn[d] (x) wn[w], the object-only design V_O = xn[d] and the view-only design V_W = wn[w],
 * stacked in the order of a HOST int32 list kinds_host[k] of distinct GPP_EFFECT_* values.  Block widths: p q (K),
 * p (O), round4(q) (W; its padding rows and columns are exactly zero).  With the per-view first moments
 *   z_v = sum_{i: w_i = v} X_i (L),   a_v = xn^T cnt[:, v] (p),   n_v = sum_o cnt[o, v]
 * every block of GC = V^T [V | X] is a sum over v:  KK = wn_vk wn_vk' S_v,  KO = wn_vk S_v,  KW = wn_vk wn_vk' a_v,
 * OO = S_v,  OW = a_v wn_vk',  WW = n_v wn_vk wn_vk';  C_K = wn_vk T_v,  C_O = T_v,  C_W = wn_vk z_v.
 *   gpp_kr_view_sums         VM (nviews rows):  VM[v, 0 .. L) = z_v;  with_x: VM[v, L .. L + p) = a_v, VM[v, L + p] = n_v
 *                            (exact up to 2^24 rows per view), VM[v, L + p + 1 .. L + p + 4) = 0.  Partials per block of
 *                            objects (rows in slot order), then summed in a fixed order: no atomics.
 *   gpp_kr_assemble_gc_blocks  the stacked GC (with_g) or C alone from ST (as gpp_kr_assemble_gc reads it; unused and
 *                            may be NULL without K and O) and VM (unused and may be NULL without W).
 *   gpp_kr_assemble_m_blocks  M (p x nviews L): M[j, v L + l] = sum_k wn[v,k] W_K[(j,k), l] + W_O[j, l] (needed with K or O)
 *                            and R (nviews x L): R[v, l] = sum_k wn[v,k] W_W[k, l] (needed with W); then Y = xn M.
 *   gpp_kr_xb_nll_views      gpp_kr_xb_nll with the per-view row:  Xb_i = (X_i - Y[d_i, w_i L ..] - R[w_i]) / vn. */
enum gpp_effect_kind { GPP_EFFECT_KR = 0, GPP_EFFECT_OBJECT = 1, GPP_EFFECT_VIEW = 2 };
size_t gpp_kr_view_sums_workspace_bytes(int64_t P, int32_t p, int32_t nviews, int32_t L, int32_t with_x);
int gpp_kr_view_sums(const float* X, int64_t ldx, const int64_t* order, const int64_t* slot_start, const float* xn,
                     int64_t P, int32_t p, int32_t nviews, int32_t L, int32_t with_x, float* VM, int64_t ldvm,
                     void* workspace, size_t workspace_bytes, gpp_stream_t stream);
int gpp_kr_assemble_gc_blocks(const float* ST, int64_t ldst, const float* VM, int64_t ldvm, const float* wn, int32_t p,
                              int32_t q, int32_t nviews, int32_t L, int32_t k, const int32_t* kinds_host, int32_t with_g,
                              float* GC, int64_t ldgc, gpp_stream_t stream);
int gpp_kr_assemble_m_blocks(const float* W, int64_t ldw, const float* wn, int32_t p, int32_t q, int32_t nviews,
                             int32_t L, int32_t k, const int32_t* kinds_host, float* M, int64_t ldm, float* R,
                             int64_t ldr, gpp_stream_t stream);
int gpp_kr_xb_nll_views(const float* X, int64_t ldx, const float* Y, int64_t ldy, const float* R, int64_t ldr,
                        const int64_t* d, const int64_t* w, int64_t n, int64_t P, int32_t nviews, int32_t L,
                        double* scal, float* Xb, int64_t ldxb, float* nll, void* workspace, size_t workspace_bytes,
                        gpp_stream_t stream);

/* ---------------- posterior prediction at new rows (GP.predict; DESIGN 5.9) ----------------
 * For a new row u of the stacked design (the designs' Binv as gpp_factor or gpp_factor_blocks leaves it, W from
 * gpp_solve_w(_blocks)):  mean* = u W,  var* = scal[V0] u Binv u^T  -- the posterior mean and variance of the noise-free
 * latent, one variance shared by all L columns (the observation adds scal[VN]).  On factored designs the row at
 * (o, v) is u = A_v x + b_v with x = xn[o] (p) and w = wn[v] (q): A_v puts x (x) w in the K block and x in the O block,
 * b_v puts w in the W block, so  var* = scal[V0] (x^T H_v x + 2 x^T h_v + c_v)  and  mean* = Y[o, v L ..] + R[v]  (Y, R
 * from gpp_kr_assemble_m(_blocks) and gpp_am).  The kinds list is that of gpp_kr_assemble_m_blocks; a single Khatri-Rao
 * design (gpp_factor with Q = p q) is kinds = {GPP_EFFECT_KR}.
 *   gpp_kr_predict_views  H = [H_0 | ... | H_{nviews-1}] (p x nviews p, ld = ldh; NULL without K and O):
 *                           H_v[j',j] = sum_{k',k} w_k' w_k Binv[K(j',k'), K(j,k)] + sum_k' w_k' Binv[K(j',k'), O j]
 *                                       + sum_k w_k Binv[O j', K(j,k)] + Binv[O j', O j];
 *                         h (nviews x p, contiguous) and c (nviews), both NULL without W:
 *                           h_v[j] = sum_{k,k'} w_k Binv[K(j,k), W k'] w_k' + sum_k' Binv[O j, W k'] w_k',
 *                           c_v = sum_{k,k'} w_k Binv[W k, W k'] w_k'.
 *                         Binv (ld = ldb >= the stacked width) is read once, in tiles of q rows shared by every view (as
 *                         gpp_kr_grad_rhs does); fixed-order sums without atomics.  Only the q true columns of the W
 *                         block are read.  p must be a multiple of 4; nviews q floats must fit 48 KB, and one tile of
 *                         Binv with the view table must fit 160 KB of shared memory (q up to about 200).
 *   then YH = xn H (P x nviews p) with gpp_am / gpp_am_planes, the P-long product of the structured pass 2.
 *   gpp_kr_predict_rows   one warp per new row i (o = d_i, v = w_i):  mean (m x L, ld = ldmean) = Y[o, v L ..] + R[v],
 *                         var (m) = scal[V0] (xn[o] . YH[o, v p ..] + 2 xn[o] . h[v] + c[v]).  Y and YH (and xn) are NULL
 *                         when the kinds are W alone; R, h and c are NULL without W.  A row with an index outside the
 *                         tables gets NaN for mean and var.  Fixed order: repeats are bit-identical.  L % 4 == 0.
 *   gpp_rows_dot          out_i = scal[V0] sum_c A[i, c] B[i, c]  (m rows, cols % 4 == 0): the variance of dense new rows
 *                         from A = V* Binv and B = V*, one warp per row in a fixed order. */
int gpp_kr_predict_views(const float* Binv, int64_t ldb, const float* wn, int32_t p, int32_t q, int32_t nviews, int32_t k,
                         const int32_t* kinds_host, float* H, int64_t ldh, float* h, float* c, gpp_stream_t stream);
int gpp_kr_predict_rows(const float* Y, int64_t ldy, const float* R, int64_t ldr, const float* YH, int64_t ldyh,
                        const float* xn, const float* h, const float* c, const int64_t* d, const int64_t* w, int64_t m,
                        int64_t P, int32_t p, int32_t nviews, int32_t L, const double* scal, float* mean, int64_t ldmean,
                        float* var, gpp_stream_t stream);
int gpp_rows_dot(const float* A, int64_t lda, const float* B, int64_t ldb, int64_t m, int32_t cols, const double* scal,
                 float* out, gpp_stream_t stream);

/* Taylor surrogate (gp.py:127-133): out_i = Xb_i.X_i + Vb_i.V_i + <vbs, softmax(lvs)> / n      */
int gpp_taylor_expansion_fwd(const float* X, int64_t ldx, const float* Xb, int64_t ldxb, const float* V,
                             int64_t ldv, const float* Vb, int64_t ldvb, int64_t n, int32_t L, int32_t Q,
                             const float* vbs, const float* lvs, float* out, gpp_stream_t stream);
/* its backward: gX = gout_i Xb_i, gV = gout_i Vb_i, glvs = J_softmax^T vbs * sum(gout) / n.
 * gX / gV / glvs may be NULL when that gradient is not needed. */
int gpp_taylor_expansion_bwd(const float* gout, const float* Xb, int64_t ldxb, const float* Vb, int64_t ldvb,
                             int64_t n, int32_t L, int32_t Q, const float* vbs, const float* lvs, float* gX,
                             int64_t ldgx, float* gV, int64_t ldgv, float* glvs, gpp_stream_t stream);

/* ---------------- host-buffer entry (end-to-end measurement; train_gppvae.py:161-167) ---------------- */

/* One evaluation of the GP term from HOST buffers: copies x0, v0, d, w, X, lvs to the device, builds V
 * (vmod.py:22-35), runs pass 1 / factor / pass 2 (gp.py:55-60,84-87) and copies nll (n), Xb (n x L) and vbs[2] back.
 * All inputs travel on one copy stream, the small ones first, into one of two sets of device buffers: X is on the wire
 * beside the work that does not need it (the Khatri-Rao map, the Gram tiles of pass 1, the Cholesky), the inputs of a
 * second submission beside the compute of the first, and the results leave on a third stream beside the compute of the
 * NEXT submission:
 *   gpp_gp_term_host_submit  enqueues one evaluation and returns a ticket (0 or 1: two sets of host-facing device
 *                            buffers); at most two submissions are in flight -- a third first waits for the oldest;
 *   gpp_gp_term_host_wait    blocks until the results of that ticket are in the host buffers;
 *   gpp_gp_term_host         = submit + wait (synchronous).
 * The host buffers of a submission must stay valid and untouched until its wait returns.  Device buffers live in the
 * context and are reused across calls.  Xb_host or vbs_host may be NULL to skip that copy.  Host buffers should be
 * pinned (page-locked) for the copies to be asynchronous and at full PCIe speed. */
typedef struct gpp_host_ctx gpp_host_ctx;
int gpp_host_ctx_create(gpp_host_ctx** ctx);
int gpp_host_ctx_destroy(gpp_host_ctx* ctx);
int gpp_gp_term_host_submit(gpp_host_ctx* ctx, const float* x0_host, int64_t P, int32_t p, const float* v0_host,
                            int64_t nviews, int32_t q, const int64_t* d_host, const int64_t* w_host,
                            const float* X_host, int64_t n, int32_t L, const float* lvs_host, float* nll_host,
                            float* Xb_host, float* vbs_host, int32_t* ticket);
int gpp_gp_term_host_wait(gpp_host_ctx* ctx, int32_t ticket);
int gpp_gp_term_host(gpp_host_ctx* ctx, const float* x0_host, int64_t P, int32_t p, const float* v0_host,
                     int64_t nviews, int32_t q, const int64_t* d_host, const int64_t* w_host,
                     const float* X_host, int64_t n, int32_t L, const float* lvs_host, float* nll_host,
                     float* Xb_host, float* vbs_host);

#ifdef __cplusplus
}
#endif
#endif /* GPPVAE_B200_H_ */
