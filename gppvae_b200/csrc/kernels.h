// Internal launch interface between the translation units of libgppvae_b200.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include "../../include/gppvae_b200.h"

namespace gpp {

// ---- gemm_simt.cu ----
struct GemmParams {
  const float* A; int64_t lda; int64_t strideA;
  const float* B; int64_t ldb; int64_t strideB;
  float* C; int64_t ldc; int64_t strideC;
  int M, N, K;
  int M_last;      // >= 0: rows of the last batch (ragged final pair of the triangular inverse)
  int K_is_M;      // contraction length equals this batch's M
  float alpha, beta;
  int lower_only;  // skip tiles strictly above the block diagonal
  int tri_a;       // A(m, k) == 0 for k > m : stop the contraction at the tile's last row
  int tri_b;       // B(n, k) == 0 for k < n : start the contraction at the tile's first column
};
int launch_gemm(const GemmParams& p, bool a_rowc, bool b_rowc, int batches, cudaStream_t st);

size_t tn_workspace_bytes(int64_t n, int ka, int kb1, int kb2, int symmetric);
int launch_tn(const float* A, int64_t lda, int ka, const float* B1, int64_t ldb1, int kb1, const float* B2,
              int64_t ldb2, int kb2, int64_t n, int symmetric, float* out, int64_t ldo, float* out2, int64_t ldo2,
              const double* scal_for_b2, void* ws, size_t ws_bytes, cudaStream_t st);

size_t xb_workspace_bytes(int64_t n, int L);
int launch_xb(const float* V, int64_t ldv, const float* X, int64_t ldx, const float* W, int64_t ldw, int64_t n, int Q,
              int L, double* scal, float alpha_host, float* Xb, int64_t ldxb, float* nll, void* ws, size_t ws_bytes,
              cudaStream_t st);
int launch_vb(const float* V, int64_t ldv, const float* Xb, int64_t ldxb, const float* Binv, int64_t ldb,
              const float* W, int64_t ldw, const double* scal, int64_t n, int Q, int L, int L_true, float* Vb,
              int64_t ldvb, cudaStream_t st);

// ---- gemm_tc.cu (tcgen05 / TMA / TMEM) ----
bool tc_pass1_supported(int64_t n, int Q, int L);
size_t tc_pass1_workspace_bytes(int64_t n, int Q, int L, bool skip_g);
int launch_tc_pass1(const float* V, int64_t ldv, const float* X, int64_t ldx, int64_t n, int Q, int L, float* G,
                    int64_t ldg, float* C, int64_t ldc, const double* scal_c, void* ws, size_t ws_bytes,
                    bool wide_range, cudaStream_t st);

// batched block GEMM on the tensor cores (see gemm_tc.cu)
struct TcBlockGemm {
  int n, n_last, K, ncols, batches;
  int a_row0, a_row_step, a_k0, a_k_step, b_k0, b_k_step, b_col0, b_col_step, tri_a, tri_b;
  int64_t out_step;
  float alpha;
  int wide_range;   // operands span many orders of magnitude (Cholesky factor, its inverse): tf32 hi.hi split, see gemm_tc.cu
};
bool tc_blockgemm_supported(int n, int K, int ncols);
// amax (device, may be null): [0] bit pattern of max|A|, [1] of max|B| -- the magnitudes the fp16 scales of the
// correction terms are derived from (tc_absmax fills one slot)
int launch_tc_blockgemm(const float* Amat, int64_t a_rows, int64_t a_cols, int64_t lda, const float* Bmat, int64_t b_rows,
                        int64_t b_cols, int64_t ldb, float* out, int64_t ldo, const TcBlockGemm& g,
                        const uint32_t* amax, cudaStream_t st);
// C -= A A^T on the lower block triangle (C n x n in place, A n x K, At = A^T K x n); n >= 512, K >= 64
int launch_tc_syrk_sub(float* C, int64_t ldc, const float* A, int64_t lda, const float* At, int64_t ldat, int n, int K,
                       const uint32_t* amax, cudaStream_t st);
int tc_absmax(const float* X, int64_t ld, int64_t rows, int cols, uint32_t* slot, cudaStream_t st);
// the same scan folded into *slot (not zeroed first): one scale for several matrices
int tc_absmax_fold(const float* X, int64_t ld, int64_t rows, int cols, uint32_t* slot, cudaStream_t st);

bool tc_available();   // cuTensorMapEncodeTiled resolvable from this driver

// ---- gemm_planes.cu (pre-split fp16 operand planes: TMA -> shared memory -> tcgen05, no conversion in the kernel) ----
size_t planes_bytes(int64_t n, int cols);
size_t split_workspace_bytes(int64_t n, int cols);
int launch_split_planes(const float* X, int64_t ldx, int64_t n, int cols, void* planes, const void* share_scale_of,
                        int exp_hint, bool want_colsq, void* ws, size_t ws_bytes, cudaStream_t st);
int launch_kr_planes(const float* xn, int64_t P, int p, const float* wn, int64_t nviews, int q, const int64_t* d,
                     const int64_t* w, int64_t n, float* V, int64_t ldv, void* planes, void* ws, size_t ws_bytes,
                     cudaStream_t st);
bool pl_pass1_supported(int64_t n, int Q, int L);
size_t pl_pass1_workspace_bytes(int64_t n, int Q, int L, bool skip_g);
int launch_pl_pass1(const void* planesV, const void* planesX, int64_t n, int Q, int L, float* G, int64_t ldg, float* C,
                    int64_t ldc, bool use_colsq, void* ws, size_t ws_bytes, cudaStream_t st);
bool pl_rows_supported(int64_t n, int K, int ncols);
size_t pl_xb_workspace_bytes(int64_t n, int Q, int L);
int launch_pl_xb(const void* planesV, const float* X, int64_t ldx, const float* W, int64_t ldw, int64_t n, int Q, int L,
                 double* scal, float alpha_host, float* Xb, int64_t ldxb, float* nll, void* ws, size_t ws_bytes,
                 cudaStream_t st);

size_t pl_vb_workspace_bytes(int64_t n, int Q, int L);
int launch_pl_vb(const void* planesV, const float* Xb, int64_t ldxb, const float* Binv, const float* W, int64_t ldw,
                 const double* scal, int64_t n, int Q, int L, int L_true, float* Vb, int64_t ldvb, void* ws,
                 size_t ws_bytes, cudaStream_t st);

int launch_kr_slot_sums_planes(const float* X, int64_t ldx, int64_t n, const int64_t* order, const int64_t* slot_start,
                               const float* xn, int64_t P, int p, int nviews, int L, int with_x, int max_count,
                               void* planes, cudaStream_t st);
int launch_pl_am(const void* planesA, const void* planesB, int64_t n, int K, int ncols, float alpha, float* out,
                 int64_t ldo, void* ws, size_t ws_bytes, cudaStream_t st);

bool tc_rows_supported(int64_t n, int K, int ncols);
size_t tc_xb_workspace_bytes(int64_t n, int L);
int launch_tc_xb(const float* V, int64_t ldv, const float* X, int64_t ldx, const float* W, int64_t ldw, int64_t n,
                 int Q, int L, double* scal, float alpha_host, float* Xb, int64_t ldxb, float* nll, void* ws,
                 size_t ws_bytes, cudaStream_t st);
size_t tc_vb_workspace_bytes(int Q, int L);
int launch_tc_vb(const float* V, int64_t ldv, const float* Xb, int64_t ldxb, const float* Binv, const float* W,
                 int64_t ldw, const double* scal, int64_t n, int Q, int L, int L_true, float* Vb, int64_t ldvb, void* ws,
                 size_t ws_bytes, cudaStream_t st);
// gemm_simt.cu: nll_i = 0.5 sum_t quad_part[t][i] + ROWCONST; scal[XB2], scal[QUAD]
constexpr int kXbFinalizeBlocks = 296;
inline size_t xb_finalize_bytes() { return (size_t)kXbFinalizeBlocks * 2 * sizeof(double); }
int launch_xb_finalize(const float* quad_part, int tiles_n, int64_t n, const double* xb2_part, int64_t nparts,
                       double* fin, double* scal, float* nll, cudaStream_t st);

// ---- qspace.cu ----
size_t factor_workspace_bytes(int Q);
size_t solve_workspace_bytes(int Q, int L);
int launch_factor(const float* G, int64_t ldg, int Q, const float* vs, uint32_t flags, float* Binv, double* scal,
                  void* ws, size_t ws_bytes, cudaStream_t st);
int launch_solve_w(const float* C, int64_t ldc, int Q, int L, int L_true, int64_t n_total, float* W, int64_t ldw,
                   double* scal, const void* state, size_t state_bytes, void* ws, size_t ws_bytes, cudaStream_t st);
int launch_vbs(const double* scal, int64_t n_total, int Q, int L, float* vbs, cudaStream_t st);

// k stacked designs V = [V_0 | ... | V_{k-1}]: block i owns columns [start[i], start[i+1]) (start[k] = Q, every width a
// positive multiple of 4).  Passed to kernels by value.
constexpr int kMaxBlocks = GPP_MAX_DESIGNS;
struct BlockSpec {
  int k;
  int start[kMaxBlocks + 1];
};
size_t factor_blocks_workspace_bytes(int Q, int k);
size_t solve_blocks_workspace_bytes(int Q, int L, int k);
int launch_factor_blocks(const float* G, int64_t ldg, const BlockSpec& bs, const float* vs, uint32_t flags, float* Binv,
                         double* scal, double* blk, void* ws, size_t ws_bytes, cudaStream_t st);
int launch_solve_w_blocks(const float* C, int64_t ldc, const BlockSpec& bs, int L, int L_true, int64_t n_total, float* W,
                          int64_t ldw, double* scal, double* blk, const void* state, size_t state_bytes, void* ws,
                          size_t ws_bytes, cudaStream_t st);
int launch_vbs_blocks(const double* scal, const double* blk, const float* vs, const BlockSpec& bs, int64_t n_total, int L,
                      float* vbs, cudaStream_t st);

// ---- gemm_planes.cu / gemm_tc.cu: planes of a stacked design
size_t split_stacked_workspace_bytes(int64_t n, int k, const int* cols);
int launch_split_planes_stacked(int k, const float* const* X, const int64_t* ldx, const int* cols, int64_t n, void* planes,
                                bool unit_bound, bool want_colsq, void* ws, size_t ws_bytes, cudaStream_t st);

}  // namespace gpp
