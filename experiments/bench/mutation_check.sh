#!/bin/bash
# Check that the elementwise edge tests (tests/test_gpu_*kernel_edges.py, tests/test_gpu_featmap_taylor_edges.py) bite: build deliberately wrong
# variants of the library in throw-away copies of the tree and run the tests that must catch each one.  Every mutation
# writes or reads LESS than the original or changes a value; none widens a range or changes a trip count that producer
# and consumer warps must agree on.
#   last_column_group  pass-2 epilogue of tc_rows_kernel skips its last float4 column group  -> section A (sentinels)
#   last_split         tc_reduce_kernel sums splits - 1 partials                              -> section B (split knob)
#   diagonal           the exact diagonal that colsq installs is scaled by 1 + 2^-20          -> colsq cases of pass 1
#   slot_last_row      kr_slot_sum_kernel drops the last row of each slot                     -> structured A
#   view_last_chunk    kr_view_sums_reduce_kernel sums nchunks - 1 partials                   -> structured D
#   views_r_w          kr_xb_views_kernel leaves R out of the .w component                    -> structured E
#   shared_slot_scale  KhatriRao.st writes cnt (x) xn under the scale shared with the sums    -> structured B
#   grad_rhs_last_h    kr_grad_rhs drops the last view's alpha H block from R (writes zero)     -> grad edges, table grad
#   grad_rhs_m_sign    kr_grad_rhs writes +M_v^T instead of -M_v^T                             -> grad edges, table grad
#   predict_no_h       kr_predict_rows drops the 2 x^T h_v term of the variance                -> predict edges, predict
#   predict_last_h     kr_predict_views writes zero for the last view's H_v block               -> predict edges, predict
#   predict_yh_at_l    kr_predict_rows reads YH at w_i L instead of w_i p                      -> predict edges, predict
#   kr_bwd_last_view   khatri_rao_bwd_kernel skips the last view column (k < q - 1)            -> featmap D
#   kr_planes_tail     kr_planes_kernel drops the last row of a chunk's tail loop              -> featmap A planes
#   te_last_design     taylor_fwd_multi_kernel skips the last design                           -> featmap E multi
#   te_last_glvs       taylor_bwd_multi_lvs_kernel leaves the last glvs unwritten              -> featmap E multi
#   norm_bwd_sign      normalize_rows_bwd_kernel adds the projection instead of subtracting it -> featmap C
#   host_lvs_slot0     the host entry's compute reads slot 0's lvs whatever its slot            -> host entry B
#   host_nll_other     the host entry's copy-out takes nll from the other slot                  -> host entry A, B
#   vbs_no_trb         vbs_kernel drops tr B^-1 from vbs[1]                                      -> host entry F, A
#   host_planes_ltrue  the planes branch of the host entry runs solve_w with L_true = L - 4      -> host entry A
# usage: mutation_check.sh OUT_DIR      (one log per mutation in OUT_DIR; exit 0 only if every mutation was caught)
#        ONLY="name ..." mutation_check.sh OUT_DIR   runs the named mutations only
set -u
OUT=$(mkdir -p "$1" && cd "$1" && pwd)
ROOT=$(cd "$(dirname "$0")/../.." && pwd)
TMP=$(mktemp -d)
trap 'rm -rf "$TMP"' EXIT
status=0
run() {   # name file python-replacement pytest-selection...
  local name=$1 file=$2 repl=$3
  shift 3
  if [ -n "${ONLY:-}" ] && [[ " $ONLY " != *" $name "* ]]; then return; fi
  local dst=$TMP/$name
  mkdir -p "$dst"
  (cd "$ROOT" && tar --exclude=./.git --exclude="./${OUT#"$ROOT"/}" --exclude=./gppvae_b200/build -cf - .) | tar -xf - -C "$dst"
  python - "$dst/$file" "$repl" <<'EOF' || { echo "$name: mutation does not apply"; status=1; return; }
import sys
path, repl = sys.argv[1], sys.argv[2]
old, new, count = repl.split("|||")
src = open(path).read()
assert src.count(old) == int(count), f"expected {count} occurrence(s) of {old!r}, found {src.count(old)}"
open(path, "w").write(src.replace(old, new))
EOF
  (cd "$dst" && python -m gppvae_b200.build --force > "$OUT/$name.build.txt" 2>&1) || { echo "$name: build failed"; status=1; return; }
  (cd "$dst" && python -m pytest -m gpu -x -q -p no:cacheprovider "$@" > "$OUT/$name.txt" 2>&1)
  if [ $? -eq 0 ]; then
    echo "$name: NOT caught"; status=1
  else
    echo "$name: caught"; grep -E "^(E |FAILED)" "$OUT/$name.txt" | head -8
  fi
}
run last_column_group gppvae_b200/csrc/gemm_tc.cu "if (col0 + i < p.ncols) {|||if (col0 + i + 4 < p.ncols) {|||1" \
  tests/test_gpu_kernel_edges.py -k "tc and (test_row_product_entries or test_xb_nll_entries)"
run last_split gppvae_b200/csrc/gemm_tc.cu "for (int s = 0; s < p.splits; ++s) {|||for (int s = 0; s < p.splits - 1; ++s) {|||1" \
  tests/test_gpu_kernel_edges.py -k test_split_rows_knob
run diagonal gppvae_b200/csrc/gemm_tc.cu "= p.diag[row0 + r];|||= p.diag[row0 + r] * (1.0 + 0x1p-20);|||4" \
  tests/test_gpu_kernel_edges.py -k "test_pass1_gram_entries and tc"
run slot_last_row gppvae_b200/csrc/structured.cu "for (int64_t t = b; t < e; ++t) {|||for (int64_t t = b; t < e - 1; ++t) {|||1" \
  tests/test_gpu_structured_kernel_edges.py -k test_kr_slot_sums
run view_last_chunk gppvae_b200/csrc/structured.cu "for (int ch = 0; ch < nchunks; ++ch) s +=|||for (int ch = 0; ch < nchunks - 1; ++ch) s +=|||1" \
  tests/test_gpu_structured_kernel_edges.py -k test_kr_view_sums
run views_r_w gppvae_b200/csrc/structured.cu "(yy.w + r4.w)|||yy.w|||1" \
  tests/test_gpu_structured_kernel_edges.py -k "test_kr_xb_nll_entries and views"
run shared_slot_scale gppvae_b200/vmod.py "Lx, 2, self.max_count())|||Lx, 1, self.max_count())|||1" \
  tests/test_gpu_structured_kernel_edges.py -k test_kr_st_per_range_floor
run grad_rhs_last_h gppvae_b200/csrc/structured.cu "+ j0 + jj] = (float)(alpha * (double)s);|||+ j0 + jj] = v == nviews - 1 ? 0.f : (float)(alpha * (double)s);|||1" \
  tests/test_gpu_structured_grad_kernel_edges.py tests/test_gpu_structured_table_grad.py -k "grad_rhs or c1"
run grad_rhs_m_sign gppvae_b200/csrc/structured.cu "* ldr + j] = -s;|||* ldr + j] = s;|||1" \
  tests/test_gpu_structured_grad_kernel_edges.py tests/test_gpu_structured_table_grad.py -k "grad_rhs or c1"
run predict_no_h gppvae_b200/csrc/structured.cu "(double)(a + 2.f * b + |||(double)(a + |||1" \
  tests/test_gpu_predict_kernel_edges.py tests/test_gpu_predict.py -k "test_kr_predict_rows or k_designs"
run predict_last_h gppvae_b200/csrc/structured.cu "H[(int64_t)jp * ldh + (int64_t)v * p + j] = s;|||H[(int64_t)jp * ldh + (int64_t)v * p + j] = v == nviews - 1 ? 0.f : s;|||1" \
  tests/test_gpu_predict_kernel_edges.py tests/test_gpu_predict.py -k "test_kr_predict_views or trained"
run predict_yh_at_l gppvae_b200/csrc/structured.cu "YH + di * ldyh + wi * p;|||YH + di * ldyh + wi * L;|||1" \
  tests/test_gpu_predict_kernel_edges.py tests/test_gpu_predict.py -k "test_kr_predict_rows or trained"
run kr_bwd_last_view gppvae_b200/csrc/featmap.cu "for (int k = lane; k < q; k += 32) {  // d/d wn|||for (int k = lane; k < q - 1; k += 32) {  // d/d wn|||1" \
  tests/test_gpu_featmap_taylor_edges.py -k test_khatri_rao_bwd
run kr_planes_tail gppvae_b200/csrc/gemm_planes.cu "for (; r < nr; ++r) {|||for (; r < nr - 1; ++r) {|||1" \
  tests/test_gpu_featmap_taylor_edges.py -k test_khatri_rao_fwd_planes
run te_last_design gppvae_b200/csrc/taylor.cu "for (int j = 0; j < t.k; ++j) s += row_dot(|||for (int j = 0; j < t.k - 1; ++j) s += row_dot(|||1" \
  tests/test_gpu_featmap_taylor_edges.py -k test_taylor_multi
run te_last_glvs gppvae_b200/csrc/taylor.cu "      glvs[b] = (float)(scale * (exp(|||      if (b < m - 1) glvs[b] = (float)(scale * (exp(|||1" \
  tests/test_gpu_featmap_taylor_edges.py -k test_taylor_multi
run norm_bwd_sign gppvae_b200/csrc/featmap.cu "(gr[c] - xr[c] * proj)|||(gr[c] + xr[c] * proj)|||1" \
  tests/test_gpu_featmap_taylor_edges.py -k test_normalize_rows
run host_lvs_slot0 gppvae_b200/csrc/api.cu "softmax2_kernel<<<1, 32, 0, st>>>(F(o_lvs), F(o_vs));|||softmax2_kernel<<<1, 32, 0, st>>>(F(o_lvss[0]), F(o_vs));|||1" \
  tests/test_gpu_host_entry.py -k test_every_input_changes_in_flight
run host_nll_other gppvae_b200/csrc/api.cu "F(o_nll[s]), (size_t)n * 4, cudaMemcpyDeviceToHost|||F(o_nll[1 - s]), (size_t)n * 4, cudaMemcpyDeviceToHost|||1" \
  tests/test_gpu_host_entry.py -k "test_every_input_changes_in_flight or test_branch_switch"
run vbs_no_trb gppvae_b200/csrc/qspace.cu "((double)n_total - (double)Q + trb) / vn|||((double)n_total - (double)Q) / vn|||1" \
  tests/test_gpu_host_entry.py -k "test_vbs_direct or test_branch_switch"
run host_planes_ltrue gppvae_b200/csrc/api.cu "Q + L, Q, L, L, n, F(o_W)|||Q + L, Q, L, L - 4, n, F(o_W)|||1" \
  tests/test_gpu_host_entry.py -k test_branch_switch
exit $status
