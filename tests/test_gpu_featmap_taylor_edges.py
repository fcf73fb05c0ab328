"""The kernels in front of and behind the N-long products -- row normalisation, the Khatri-Rao map (fp32 kernel and the
fused V + planes writer), its backward, the stacked split of k designs and the Taylor surrogate -- against float64, entry
by entry, with the conventions of test_gpu_kernel_edges.py: C entries called directly, sentinel outputs (a NaN bit
pattern outside the written block must survive), inputs with ld > cols whose gap holds NaN, per-column spread where
magnitudes matter, and the worst bound ratio printed per case.

Row counts come from the SM count: the featmap and Taylor kernels are persistent grids of 8 CTAs x 8 warps per SM, one
row per warp, so a sweep covers 64 SMs rows; 64 SMs - 1, 64 SMs + 1 and 3 (64 SMs) + 17 rows wrap it (and exercise the
index prefetch of khatri_rao_fwd_kernel).  The planes writer runs at prime n (never a multiple of its 256-row chunk,
its 4-row batch or its rows per block, so every chunk-tail path runs).

Bounds, derived from the kernels' arithmetic in units of u = 2^-24 (gamma_k = k u / (1 - k u), the error of any sum
whose terms pass through at most k roundings):
  Khatri-Rao forward (both kernels)  one fp32 multiply per element: BIT-IDENTICAL to torch's fp32 product; rows with an
                      index outside its table are NaN in every column.  The planes writer's V is bit-identical to the fp32
                      kernel's.  Its planes are graded without decoding the buffer: pass 1 on them and on
                      gpp_split_planes(V, COLSQ | UNIT_BOUND) gives BIT-IDENTICAL off-diagonals (same scale, same split,
                      deterministic pass 1), diagonals within 2^-24 of the fp64 column sums of squares, and G within the
                      c_tc(n) bound of test_gpu_kernel_edges.py, whose floor here takes the unit bound (max|v| <= 1, the
                      scale the writer uses) instead of the observed maximum.
  stacked split       the same two checks against gpp_split_planes of the fp32 concatenation, and gpp_atb_planes with the
                      c_tc(n) bound (floor from the common scale's maximum: 1 under UNIT_BOUND).
  normalize fwd       s = sum x^2: a lane chain of ceil(cols/32) fmaf and a 5-level butterfly, so with a = ceil(cols/32)
                      + 5 the relative error of s is gamma_a; sqrtf and the divide are IEEE (no --use_fast_math in
                      build.py): |y - y64| <= (gamma_a / 2 + gamma_3) |y64|.
  normalize bwd       gx = (g - x proj) inv with proj = dot / s, inv = 1 / sqrtf(s).  dot carries gamma_a sum|x g|, proj
                      (2 gamma_a + u) sum|x g| / s, inv gamma_a / 2 + 2u, and three more roundings: 2.5 gamma_a + 6u,
                      taken as gamma_(3a + 7), times (|g| + |x| sum|x g| / ||x||^2) / ||x||.  The second term is the
                      magnitude of the projection, which cancels against g (pure cancellation for g parallel to y).
  Khatri-Rao bwd      gxn[o, j]: per row a chain of q fmaf, then cnt_o fp32 atomics in any order: gamma_(q + cnt_o) times
                      sum |g| |wn|; gwn[v, k] likewise with p and cnt_v.  Atomics make repeats differ in the last bits:
                      no bit-identity is asserted.  Rows with an index outside its table add nothing.
  Taylor fwd          out = Xb.X + sum_j Vb_j.V_j + <vbs, softmax(lvs)> / n.  Lane chains of 4 ceil(len/128) fmaf per
                      operand pair (float4 loads), one add per further pair, 5 butterflies, + cterm:
                      gamma_(m + 6) (sum|Xb X| + sum_j sum|Vb_j V_j| + |cterm|), m = sum over L and every Q_j of
                      4 ceil(len/128).
  Taylor bwd rows     gX = fl(g Xb), gV_j = fl(g Vb_j): BIT-IDENTICAL to torch's fp32 product.
  Taylor bwd lvs      double throughout, one rounding to fp32: u |ref| plus the double sums, (2n + 2m + 16) 2^-53
                      (sum|g| / n) vs_b (|vbs_b| + sum vs |vbs|) (n-term sum of g in the kernel and in the reference).
The file fails (does not skip) when the library was not built with the tensor-core engine.
"""
import math

import pytest
import torch

from edge_helpers import (DEV, FLOOR, NAN_BITS, U, c_tc, check_sentinel, gamma, grade, nan_vector, ratio_of, sentinel,
                          spread_cols, strided)
from edge_helpers import call as _call
from edge_helpers import stream as _st
from edge_helpers import workspace as _ws

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", autouse=True)
def lib():
    from gppvae_b200 import _lib
    engine = _lib.gemm_engine()
    assert engine == "tcgen05-3xf16", f"this file checks the tensor-core paths; the library was built with {engine}"
    return _lib.load()


def rows_of(label):
    """Row count of a label: the persistent grids cover 64 x SMs rows per sweep (8 CTAs of 8 warps per SM)."""
    sweep = 64 * torch.cuda.get_device_properties(0).multi_processor_count
    return {"1": 1, "64": 64, "sweep-1": sweep - 1, "sweep+1": sweep + 1, "3sweep+17": 3 * sweep + 17}[label]


def _gen(seed):
    return torch.Generator(device=DEV).manual_seed(seed)


def unit_rows(T):
    return T / T.norm(dim=1, keepdim=True)


def index(n, P, nv, seed, occ):
    """(d, w, in_table) with uniform, skewed (object 3 % P and view 1 % nv each hit by 10 % of the rows) or out-of-table
    occupancy (indices -1, P and nviews on the first, the last and about 2 % of the other rows)."""
    g = _gen(seed)
    d = torch.randint(0, P, (n,), generator=g, device=DEV)
    w = torch.randint(0, nv, (n,), generator=g, device=DEV)
    if occ == "skewed":
        d[torch.rand(n, generator=g, device=DEV) < 0.1] = 3 % P
        w[torch.rand(n, generator=g, device=DEV) < 0.1] = 1 % nv
    elif occ == "oob":
        perm = torch.randperm(n, generator=torch.Generator().manual_seed(seed))[: n // 50]
        rows = torch.cat([torch.tensor([0, n - 1]), perm]).to(DEV)
        d[rows[0::4]] = -1
        d[rows[1::4]] = P
        w[rows[2::4]] = -1
        w[rows[3::4]] = nv
    ok = (d >= 0) & (d < P) & (w >= 0) & (w < nv)
    return d.contiguous(), w.contiguous(), ok


def kr_ref(xn, wn, d, w):
    """torch's fp32 V (rows with an out-of-table index take row 0: the caller masks them)."""
    P, nv = xn.shape[0], wn.shape[0]
    dc, wc = d.clamp(0, P - 1), w.clamp(0, nv - 1)
    return (xn[dc][:, :, None] * wn[wc][:, None, :]).reshape(d.shape[0], -1)


def assert_kr_rows(tag, V, R, ok):
    """In-table rows bit-identical to torch's fp32 product; out-of-table rows NaN in every column."""
    assert torch.equal(V[ok].view(torch.int32), R[ok].view(torch.int32)), f"{tag}: V is not the fp32 product bit for bit"
    if bool((~ok).any()):
        assert bool(torch.isnan(V[~ok]).all()), f"{tag}: a row with an out-of-table index is not NaN in every column"
    print(f"[{tag}] bit-identical ({int(ok.sum())} in-table rows, {int((~ok).sum())} out-of-table rows NaN)")


# ---------------------------------------------------------------------------------- A. Khatri-Rao forward, fp32 kernel
# (p, q, rows, occupancy, pad of ldv): the fast path (q = 4 ... 128 with p % 4 == 0), the general path (q = 1, 2, 3, 9,
# 132, 256; p % 4 != 0 with p q % 4 == 0: p = 6, q = 2 and p = 3, q = 12) and p + q = 1536, the shared-memory limit
FWD = [(4, 4, "sweep+1", "oob", 8), (8, 8, "3sweep+17", "uniform", 0), (12, 16, "sweep-1", "skewed", 4),
       (4, 32, "64", "uniform", 8), (8, 64, "sweep+1", "oob", 0), (4, 128, "sweep-1", "uniform", 4),
       (8, 1, "3sweep+17", "oob", 4), (6, 2, "sweep+1", "uniform", 0), (4, 3, "sweep-1", "skewed", 8),
       (4, 9, "1", "uniform", 4), (3, 12, "sweep+1", "oob", 8), (4, 132, "64", "uniform", 0),
       (4, 256, "sweep-1", "oob", 4), (1532, 4, "sweep+1", "uniform", 8), (4, 1532, "64", "oob", 4)]


def _fast(p, q):
    q4 = q // 4
    return q % 4 == 0 and p % 4 == 0 and q4 <= 32 and 32 % q4 == 0


@pytest.mark.parametrize("case", FWD, ids=lambda c: "p{}-q{}-n{}-{}-ld+{}-".format(*c) + ("fast" if _fast(c[0], c[1])
                                                                                          else "general"))
def test_khatri_rao_fwd(lib, case):
    p, q, label, occ, pad = case
    n, P, nv, Q = rows_of(label), 97, 13, p * q
    g = _gen(p * 1000 + q)
    xn = torch.randn(P, p, generator=g, device=DEV) * 10.0 ** (torch.rand(P, 1, generator=g, device=DEV) * 4 - 2)
    wn = torch.randn(nv, q, generator=g, device=DEV)
    d, w, ok = index(n, P, nv, seed=n + Q, occ=occ)
    V, ldv = torch.full((n + 1, Q + pad), NAN_BITS, dtype=torch.int32, device=DEV).view(torch.float32), Q + pad
    _call(lib.gpp_khatri_rao_fwd(xn.data_ptr(), P, p, wn.data_ptr(), nv, q, d.data_ptr(), w.data_ptr(), n, V.data_ptr(),
                                 ldv, _st()), "khatri_rao_fwd")
    torch.cuda.synchronize()
    V = check_sentinel(V, n, Q, "khatri_rao_fwd", allow_nan=True)
    assert_kr_rows(f"khatri_rao_fwd p={p} q={q} n={n} {occ} ld+{pad}", V, kr_ref(xn, wn, d, w), ok)


def test_khatri_rao_fwd_padded_q():
    """ops.khatri_rao_fwd at p q % 4 != 0 (p = 3, q = 3): p is zero-padded to 4 for the kernel and V[:, :9] returned;
    those columns are still the fp32 products bit for bit, and out-of-table rows NaN."""
    from gppvae_b200 import ops
    n, P, nv = rows_of("sweep+1"), 41, 5
    g = _gen(33)
    xn, wn = torch.randn(P, 3, generator=g, device=DEV), torch.randn(nv, 3, generator=g, device=DEV)
    d, w, ok = index(n, P, nv, seed=34, occ="oob")
    V = ops.khatri_rao_fwd(xn, wn, d, w)
    torch.cuda.synchronize()
    assert V.shape == (n, 9)
    assert_kr_rows(f"ops.khatri_rao_fwd p=3 q=3 n={n}", V, kr_ref(xn, wn, d, w), ok)


# --------------------------------------------------------------------------- A. gpp_khatri_rao_fwd_planes (V + planes)
# (p, q, n, occupancy): the c1 design (non-QUAD), Q = 4096 (QUAD, four 1024-column blocks), the dense ObjectEffect and
# ViewEffect (q = 1 / p = 1), p odd; n prime.  The out-of-table cases check V only (their NaN rows would fill G).
PLANES_KR = [(64, 9, 7919, "uniform"), (256, 16, 4099, "skewed"), (128, 1, 521, "uniform"), (1, 128, 1031, "uniform"),
             (33, 4, 20011, "skewed"), (64, 9, 2053, "oob"), (33, 4, 1031, "oob")]


def _gram_planes(lib, pl, n, Q):
    G, ldg = sentinel(Q, Q)
    ws = _ws(lib.gpp_gram_planes_workspace_bytes(n, Q, 0))
    _call(lib.gpp_gram_vtz_planes(pl, None, n, Q, 0, 1, G.data_ptr(), ldg, ws.data_ptr(), ws.numel(), _st()),
          "gram_vtz_planes")
    return check_sentinel(G, Q, Q, "gram_vtz_planes")


def unit_floor(A, B, maxA, maxB):
    """2^-31 (max|A| ||B_:,j||_1 + max|B| ||A_:,i||_1) with the maxima of the operands' common scales."""
    return FLOOR * (maxA * B.double().abs().sum(0)[None, :] + maxB * A.double().abs().sum(0)[:, None])


def check_same_planes(tag, G1, G2, V64):
    """Off-diagonals of two pass-1 results bit-identical; each diagonal within 2^-24 of the fp64 column sums of
    squares."""
    Q = G1.shape[0]
    off = ~torch.eye(Q, dtype=torch.bool, device=DEV)
    assert torch.equal(G1.view(torch.int32)[off], G2.view(torch.int32)[off]), f"{tag}: off-diagonals differ"
    colsq = (V64 ** 2).sum(0)
    worst = 0.0
    for G in (G1, G2):
        e = float(((torch.diagonal(G).double() - colsq).abs() / colsq).max())
        worst = max(worst, e)
        assert e <= U, f"{tag}: diag(G) is {e:.2e} off the fp64 column sums of squares"
    print(f"[{tag}] off-diagonals bit-identical; diag worst relative error {worst:.2e} (bound 2^-24)")


@pytest.mark.parametrize("case", PLANES_KR, ids=lambda c: "p{}-q{}-n{}-{}-".format(*c) + ("quad" if c[1] % 4 == 0
                                                                                         else "general"))
def test_khatri_rao_fwd_planes(lib, case):
    from gppvae_b200 import ops
    from gppvae_b200._lib import GPP_PLANES_COLSQ, GPP_PLANES_UNIT_BOUND
    p, q, n, occ = case
    P, nv, Q = 211, 17, p * q
    g = _gen(p * 100 + q)
    xn = unit_rows(torch.randn(P, p, generator=g, device=DEV))
    wn = unit_rows(torch.randn(nv, q, generator=g, device=DEV))
    d, w, ok = index(n, P, nv, seed=n, occ=occ)
    tag = f"khatri_rao_fwd_planes p={p} q={q} n={n} {occ}"
    V, ldv = sentinel(n, Q)
    buf = _ws(lib.gpp_planes_bytes(n, Q))
    ws = _ws(lib.gpp_split_workspace_bytes(n, Q))
    _call(lib.gpp_khatri_rao_fwd_planes(xn.data_ptr(), P, p, wn.data_ptr(), nv, q, d.data_ptr(), w.data_ptr(), n,
                                        V.data_ptr(), ldv, buf.data_ptr(), buf.numel(), ws.data_ptr(), ws.numel(), _st()),
          "khatri_rao_fwd_planes")
    # the fp32 kernel on the same rows: V must agree bit for bit
    V32 = torch.empty(n, Q, device=DEV)
    _call(lib.gpp_khatri_rao_fwd(xn.data_ptr(), P, p, wn.data_ptr(), nv, q, d.data_ptr(), w.data_ptr(), n,
                                 V32.data_ptr(), Q, _st()), "khatri_rao_fwd")
    torch.cuda.synchronize()
    V = check_sentinel(V, n, Q, tag, allow_nan=True)
    assert_kr_rows(tag, V, kr_ref(xn, wn, d, w), ok)
    assert torch.equal(V[ok].view(torch.int32), V32[ok].view(torch.int32)), f"{tag}: V differs from the fp32 kernel's"
    assert bool(torch.isnan(V32[~ok]).all())
    if occ == "oob":
        return
    Vc = V.contiguous()
    G_kr = _gram_planes(lib, buf.data_ptr(), n, Q)
    pl = ops.split_planes(Vc, Q, n, Q, colsq=True, unit_bound=True)
    assert GPP_PLANES_COLSQ | GPP_PLANES_UNIT_BOUND == 3
    G_sp = _gram_planes(lib, pl.ptr, n, Q)
    torch.cuda.synchronize()
    V64 = Vc.double()
    check_same_planes(tag, G_kr, G_sp, V64)
    aV = V64.abs()
    grade(f"{tag} G", G_kr, V64.t() @ V64, aV.t() @ aV, unit_floor(Vc, Vc, 1.0, 1.0), c_tc(n))


# ----------------------------------------------------------------------------------------- B. gpp_split_planes_stacked
# (widths, n, unit bound, pads): k = 1, 2, 3, 16; widths from 4 to 1100 (per-source split grids of 1 or 2 column blocks
# against the concatenation's); ld gaps with NaN; neighbouring sources 1e6 apart in magnitude
STACKED = [([132], 521, False, [4]), ([4, 1028], 1031, False, [8, 0]), ([1100, 36], 2053, True, [0, 12]),
           ([12, 260, 1032], 1031, False, [4, 0, 8]), ([128, 4, 8], 4099, True, [0, 4, 8]),
           ([4 * (i + 1) for i in range(15)] + [1028], 521, False, [4 * (i % 4) for i in range(16)]),
           ([8, 4, 12, 16] * 4, 1031, True, [4, 0] * 8)]


def _stacked_sources(widths, n, unit, seed):
    srcs = []
    for i, c in enumerate(widths):
        if unit:   # |x| < 1 as the flag promises, the odd sources a million times smaller
            M = torch.randn(n, c, generator=_gen(seed + i), device=DEV)
            M = M / (1.01 * float(M.abs().max())) * (1e-6 if i % 2 else 1.0)
        else:
            M = spread_cols(n, c, seed=seed + i) * (1e-3 if i % 2 else 1e3)
        srcs.append(M)
    return srcs


@pytest.mark.parametrize("case", STACKED, ids=lambda c: f"k{len(c[0])}-Q{sum(c[0])}-n{c[1]}-" + ("unit" if c[2]
                                                                                                 else "scan"))
def test_split_planes_stacked(lib, case):
    from gppvae_b200 import ops
    widths, n, unit, pads = case
    k, Q, Lx = len(widths), sum(widths), 68
    srcs = _stacked_sources(widths, n, unit, seed=n + Q)
    mats = [strided(M, pad) for M, pad in zip(srcs, pads)]
    tag = f"split_planes_stacked k={k} Q={Q} n={n} {'unit bound' if unit else 'scanned'}"
    pS = ops.split_planes_stacked(mats, n, colsq=True, unit_bound=unit)
    cat = torch.cat(srcs, 1).contiguous()
    pC = ops.split_planes(cat, Q, n, Q, colsq=True, unit_bound=unit)
    G_s = _gram_planes(lib, pS.ptr, n, Q)
    G_c = _gram_planes(lib, pC.ptr, n, Q)
    torch.cuda.synchronize()
    C64 = cat.double()
    check_same_planes(tag, G_s, G_c, C64)
    X = spread_cols(n, Lx, seed=n + Q + 99, positive=False)
    pX = ops.split_planes(X, Lx, n, Lx)
    out, ldo = sentinel(Q, Lx)
    ws = _ws(lib.gpp_gram_planes_workspace_bytes(n, Q, Lx))
    _call(lib.gpp_atb_planes(pS.ptr, pX.ptr, n, Q, Lx, out.data_ptr(), ldo, ws.data_ptr(), ws.numel(), _st()),
          "atb_planes")
    torch.cuda.synchronize()
    out = check_sentinel(out, Q, Lx, "atb_planes")
    X64 = X.double()
    maxA = 1.0 if unit else float(cat.abs().max())
    grade(f"{tag} atb_planes", out, C64.t() @ X64, C64.abs().t() @ X64.abs(),
          unit_floor(cat, X, maxA, float(X.abs().max())), c_tc(n))


# ------------------------------------------------------------------------------------------------ C. row normalisation
NORM = [(1, "3sweep+17"), (3, "sweep-1"), (4, "sweep+1"), (31, "64"), (32, "3sweep+17"), (33, "1"), (33, "sweep+1"),
        (256, "sweep-1"), (1032, "sweep+1")]


def _norm_inputs(n, cols, seed):
    """x with rows scaled 1e-6 ... 1e6, g with rows scaled 1e-3 ... 1e3; every 7th g parallel to y; row 5 of x zero."""
    g = _gen(seed)
    x = torch.randn(n, cols, generator=g, device=DEV) * 10.0 ** (torch.rand(n, 1, generator=g, device=DEV) * 12 - 6)
    gy = torch.randn(n, cols, generator=g, device=DEV) * 10.0 ** (torch.rand(n, 1, generator=g, device=DEV) * 6 - 3)
    zero = 5 if n >= 64 else None
    if n >= 64:
        par = torch.arange(0, n, 7, device=DEV)
        y = unit_rows(x[par].double())
        gy[par] = (y * (torch.rand(par.numel(), 1, generator=g, device=DEV, dtype=torch.float64) * 4 - 2)).float()
        x[zero] = 0.0
    return x, gy, zero


def _flat_out(n, cols):
    return nan_vector(n * cols)


def _flat_check(buf, n, cols, what):
    assert int(buf.view(torch.int32)[n * cols]) == NAN_BITS, f"{what}: wrote past the {n} x {cols} output"
    return buf[: n * cols].view(n, cols)


@pytest.mark.parametrize("cols,label", NORM, ids=[f"cols{c}-n{r}" for c, r in NORM])
def test_normalize_rows(lib, cols, label):
    n = rows_of(label)
    x, gy, zero = _norm_inputs(n, cols, seed=cols * 7 + n)
    y = _flat_out(n, cols)
    gx = _flat_out(n, cols)
    _call(lib.gpp_normalize_rows_fwd(x.data_ptr(), n, cols, y.data_ptr(), _st()), "normalize_rows_fwd")
    _call(lib.gpp_normalize_rows_bwd(x.data_ptr(), gy.data_ptr(), n, cols, gx.data_ptr(), _st()), "normalize_rows_bwd")
    torch.cuda.synchronize()
    y, gx = _flat_check(y, n, cols, "normalize_rows_fwd"), _flat_check(gx, n, cols, "normalize_rows_bwd")
    keep = torch.ones(n, dtype=torch.bool, device=DEV)
    if zero is not None:
        # an all-zero row is 0 / 0, as in the reference x / (x*x).sum(1).sqrt() (and its autograd)
        x0 = x[zero:zero + 1].double().requires_grad_(True)
        ref0 = x0 / (x0 * x0).sum(1, keepdim=True).sqrt()
        ref0.backward(gy[zero:zero + 1].double())
        assert bool(torch.isnan(ref0).all()) and bool(torch.isnan(x0.grad).all())
        assert bool(torch.isnan(y[zero]).all()), "normalize_rows_fwd: an all-zero row must give NaN"
        assert bool(torch.isnan(gx[zero]).all()), "normalize_rows_bwd: an all-zero row must give NaN"
        keep[zero] = False
    a = math.ceil(cols / 32) + 5
    x64, g64 = x[keep].double(), gy[keep].double()
    s = (x64 * x64).sum(1, keepdim=True)
    nrm = s.sqrt()
    y64 = x64 / nrm
    grade(f"normalize_rows_fwd cols={cols} n={n}", y[keep], y64, y64.abs(), 0.0, 0.5 * gamma(a) + gamma(3))
    dot = (x64 * g64).sum(1, keepdim=True)
    ref = (g64 - x64 * dot / s) / nrm
    mag = (g64.abs() + x64.abs() * (x64 * g64).abs().sum(1, keepdim=True) / s) / nrm
    grade(f"normalize_rows_bwd cols={cols} n={n}", gx[keep], ref, mag, 0.0, gamma(3 * a + 7))


# ----------------------------------------------------------------------------------------------- D. Khatri-Rao backward
# (p, q, P, nviews, rows, occupancy, pad of ldg): p q = 18 and 15 not multiples of 4; q = 1 (the dense ObjectEffect);
# nviews = 1 puts every row on one view
BWD = [(4, 4, 50, 7, "sweep-1", "uniform", 0), (6, 3, 40, 9, "sweep+1", "skewed", 4),
       (32, 9, 300, 11, "3sweep+17", "oob", 12), (64, 16, 120, 20, "sweep+1", "skewed", 0),
       (3, 5, 17, 3, "64", "oob", 8), (128, 1, 100, 1, "sweep-1", "uniform", 4), (1, 128, 60, 13, "1", "uniform", 0)]


def kr_bwd_ref(G, xn, wn, d, w, ok):
    """fp64 gxn, gwn over the in-table rows and their bounds gamma(q + cnt_o) sum|g||wn|, gamma(p + cnt_v) sum|g||xn|."""
    P, p = xn.shape
    nv, q = wn.shape
    G3 = G[ok].double().view(-1, p, q)
    di, wi = d[ok], w[ok]
    X, W = xn.double()[di], wn.double()[wi]
    gx = torch.zeros(P, p, dtype=torch.float64, device=DEV).index_add_(0, di, torch.einsum("rjk,rk->rj", G3, W))
    gw = torch.zeros(nv, q, dtype=torch.float64, device=DEV).index_add_(0, wi, torch.einsum("rjk,rj->rk", G3, X))
    mx = torch.zeros(P, p, dtype=torch.float64, device=DEV).index_add_(0, di, torch.einsum("rjk,rk->rj", G3.abs(),
                                                                                         W.abs()))
    mw = torch.zeros(nv, q, dtype=torch.float64, device=DEV).index_add_(0, wi, torch.einsum("rjk,rj->rk", G3.abs(),
                                                                                          X.abs()))
    cnt_o = torch.bincount(di, minlength=P).double()[:, None]
    cnt_v = torch.bincount(wi, minlength=nv).double()[:, None]
    cx = (q + cnt_o) * U / (1 - (q + cnt_o) * U)
    cw = (p + cnt_v) * U / (1 - (p + cnt_v) * U)
    return gx, cx * mx, gw, cw * mw


def grade_kr_bwd(tag, gxn, gwn, ref):
    gx, lx, gw, lw = ref
    for name, got, R, lim in (("gxn", gxn, gx, lx), ("gwn", gwn, gw, lw)):
        assert bool(torch.isfinite(got).all()), f"{tag} {name}: non-finite output"
        r = ratio_of((got.double() - R).abs(), lim)
        print(f"[{tag} {name}] worst bound ratio {r:.3f}")
        assert r <= 1.0, f"{tag} {name}: elementwise error {r:.3g} x the fp64 bound"


@pytest.mark.parametrize("case", BWD, ids=lambda c: "p{}-q{}-P{}-nv{}-n{}-{}-ld+{}".format(*c))
def test_khatri_rao_bwd(lib, case):
    p, q, P, nv, label, occ, pad = case
    n, Q = rows_of(label), p * q
    g = _gen(p * 31 + q)
    xn = unit_rows(torch.randn(P, p, generator=g, device=DEV))
    wn = unit_rows(torch.randn(nv, q, generator=g, device=DEV))
    d, w, ok = index(n, P, nv, seed=n + 3 * Q, occ=occ)
    G0 = spread_cols(n, Q, seed=n + Q, positive=False)
    Gv, ldg = strided(G0, pad)
    gxn, gwn = torch.zeros(P + 1, p, device=DEV), torch.zeros(nv + 1, q, device=DEV)
    gxn[P], gwn[nv] = float("nan"), float("nan")      # a row past each table that must stay untouched
    _call(lib.gpp_khatri_rao_bwd(Gv.data_ptr(), ldg, xn.data_ptr(), P, p, wn.data_ptr(), nv, q, d.data_ptr(),
                                 w.data_ptr(), n, gxn.data_ptr(), gwn.data_ptr(), _st()), "khatri_rao_bwd")
    torch.cuda.synchronize()
    assert bool(torch.isnan(gxn[P]).all()) and bool(torch.isnan(gwn[nv]).all()), "khatri_rao_bwd wrote past a table"
    grade_kr_bwd(f"khatri_rao_bwd p={p} q={q} P={P} nv={nv} n={n} {occ} ld+{pad}", gxn[:P], gwn[:nv],
                 kr_bwd_ref(G0, xn, wn, d, w, ok))


# Through Vmodel: V.sum(0) hands _KhatriRao.backward a gradient with strides (0, 1), V.sum() one with strides (0, 0),
# V.mean(0) @ c a contiguous one (mean divides the expanded gradient).  p q = 12 and 9 (the padded forward).
VM_UPSTREAM = [(m, p, q, n) for m in ("sum0", "sum", "mean0") for p, q in ((4, 3), (3, 3)) for n in (301, 1)]


def _upstream(mode, V, c):
    if mode == "sum0":
        return (V.sum(0) * c).sum()
    if mode == "sum":
        return V.sum()
    return V.mean(0) @ c


@pytest.mark.parametrize("mode,p,q,n", VM_UPSTREAM, ids=[f"{m}-p{p}-q{q}-n{n}" for m, p, q, n in VM_UPSTREAM])
def test_khatri_rao_bwd_broadcast_upstream(mode, p, q, n):
    """Vmodel gradients for broadcast and contiguous upstream gradients against fp64 autograd of the torch expression."""
    from conftest import rel_err
    from gppvae_b200 import Vmodel
    from oracle import gp_oracle as O
    P, nv = 23, 7
    vm = Vmodel(P, nv, p, q).to(DEV)
    g = _gen(p * 10 + q + n)
    with torch.no_grad():
        vm.x0.copy_(torch.randn(P, p, generator=g, device=DEV))
        vm.v0.copy_(torch.randn(nv, q, generator=g, device=DEV))
    d, w, _ = index(n, P, nv, seed=n + 5, occ="uniform")
    c = torch.randn(p * q, generator=g, device=DEV)
    _upstream(mode, vm(d, w), c).backward()
    x64 = vm.x0.detach().double().requires_grad_(True)
    v64 = vm.v0.detach().double().requires_grad_(True)
    _upstream(mode, O.feature_map(x64, v64, d, w), c.double()).backward()
    ex, ev = rel_err(vm.x0.grad, x64.grad), rel_err(vm.v0.grad, v64.grad)
    print(f"[Vmodel {mode} p={p} q={q} n={n}] x0.grad {ex:.2e}  v0.grad {ev:.2e} (max-relative against fp64)")
    assert ex < 1e-4 and ev < 1e-4


def test_khatri_rao_bwd_transposed_tables():
    """_KhatriRao on transposed (dense, non-contiguous) tables: the gradients land on the right entries."""
    from gppvae_b200 import ops
    P, p, nv, q, n = 37, 4, 11, 3, 301
    g = _gen(77)
    T = torch.randn(p, P, generator=g, device=DEV).requires_grad_(True)
    S = torch.randn(q, nv, generator=g, device=DEV).requires_grad_(True)
    d, w, ok = index(n, P, nv, seed=78, occ="uniform")
    C = spread_cols(n, p * q, seed=79, positive=False)
    V = ops._KhatriRao.apply(T.t(), S.t(), d, w)
    (V * C).sum().backward()
    grade_kr_bwd(f"_KhatriRao transposed tables P={P} p={p} nv={nv} q={q} n={n}", T.grad.t(), S.grad.t(),
                 kr_bwd_ref(C, T.detach().t(), S.detach().t(), d, w, ok))


# -------------------------------------------------------------------------------------------- E. Taylor surrogate
LVS = {"mild": [0.3, -1.2, 0.8, -0.1, 1.5, -0.7, 0.2, 0.0, -2.0, 1.1, 0.4, -0.3, 0.9, -1.6, 0.6, -0.9, 1.3],
       "big": None}


def _lvs(kind, m):
    """lvs of m entries: moderate values, or +-750 (exp(750) overflows double: softmax must subtract the maximum)."""
    if kind == "big":
        v = [750.0, 0.0] if m == 2 else [-750.0, 0.0, 750.0] + [0.0] * (m - 3)
    else:
        v = LVS["mild"][:m]
    return torch.tensor(v, device=DEV)


def _mixed_gout(n, seed):
    """Upstream gradient of mixed signs whose sum nearly cancels."""
    gv = torch.randn(n, generator=_gen(seed), device=DEV)
    return (gv - 0.999 * gv.mean()).contiguous() if n > 1 else gv


def _cterm_ref(vbs, lvs, n):
    vs = torch.softmax(lvs.double(), 0)
    return float((vbs.double() * vs).sum()) / n


def grade_glvs(tag, glvs, gout, vbs, lvs, extra_u=0.0):
    """glvs_b = (sum g / n) vs_b (vbs_b - <vbs, vs>) in fp64, with the bound of the module docstring."""
    m, n = vbs.numel(), gout.numel()
    vs = torch.softmax(lvs.double(), 0)
    v = vbs.double()
    mean = (v * vs).sum()
    gs = gout.double()
    ref = gs.sum() / n * vs * (v - mean)
    lim = (U + extra_u) * ref.abs() + (2 * n + 2 * m + 16) * 2.0 ** -53 * gs.abs().sum() / n * vs * (
        v.abs() + (vs * v.abs()).sum())
    assert bool(torch.isfinite(glvs).all()), f"{tag} glvs: non-finite (softmax without the maximum subtracted?)"
    r = ratio_of((glvs.double() - ref).abs(), lim)
    print(f"[{tag} glvs] worst bound ratio {r:.3f}")
    assert r <= 1.0, f"{tag} glvs: error {r:.3g} x the bound"


def _te_fwd_ref(X, Xb, Vs, Vbs, vbs, lvs, n, L, Qs):
    ref = (Xb.double() * X.double()).sum(1)
    mag = (Xb.double() * X.double()).abs().sum(1)
    for V, Vb in zip(Vs, Vbs):
        ref = ref + (Vb.double() * V.double()).sum(1)
        mag = mag + (Vb.double() * V.double()).abs().sum(1)
    ct = _cterm_ref(vbs, lvs, n)
    m = 4 * math.ceil(L / 128) + sum(4 * math.ceil(Q / 128) for Q in Qs)
    return ref + ct, mag + abs(ct), gamma(m + 6)


def _bit_rows(tag, out, g, src):
    R = g[:, None] * src
    assert torch.equal(out.view(torch.int32), R.view(torch.int32)), f"{tag}: not fl(g * Xb) bit for bit"


# (L, Q, rows, lvs, which gradient is NULL)
SINGLE = [(4, 0, "1", "mild", ""), (128, 4, "64", "big", "gV"), (132, 576, "sweep+1", "mild", ""),
          (256, 4368, "sweep-1", "mild", "gX"), (4, 576, "3sweep+17", "big", ""), (132, 0, "sweep+1", "mild", "")]


@pytest.mark.parametrize("case", SINGLE, ids=lambda c: "L{}-Q{}-n{}-lvs_{}".format(*c[:4]) + (f"-{c[4]}_null" if c[4]
                                                                                                else ""))
def test_taylor_single(lib, case):
    L, Q, label, lk, null = case
    n = rows_of(label)
    pad = 4 * (L % 3)
    X, ldx = strided(spread_cols(n, L, seed=L + n, positive=False), pad)
    Xb, ldxb = strided(spread_cols(n, L, seed=L + n + 1, positive=False), 8 - pad)
    if Q:
        V, ldv = strided(spread_cols(n, Q, seed=Q + n + 2, positive=False), 4)
        Vb, ldvb = strided(spread_cols(n, Q, seed=Q + n + 3, positive=False), 12)
    else:
        V = Vb = None
        ldv = ldvb = 4
    vbs = torch.randn(2, generator=_gen(n + 4), device=DEV) * 10
    lvs = _lvs(lk, 2)
    tag = f"taylor_expansion L={L} Q={Q} n={n} lvs={lvs.tolist()}"
    out = nan_vector(n)
    _call(lib.gpp_taylor_expansion_fwd(X.data_ptr(), ldx, Xb.data_ptr(), ldxb, V.data_ptr() if Q else None, ldv,
                                       Vb.data_ptr() if Q else None, ldvb, n, L, Q, vbs.data_ptr(), lvs.data_ptr(),
                                       out.data_ptr(), _st()), "taylor_expansion_fwd")
    gout = _mixed_gout(n, n + 5)
    gX, ldgx = sentinel(n, L)
    gV, ldgv = sentinel(n, max(Q, 4))
    glvs = nan_vector(2)
    _call(lib.gpp_taylor_expansion_bwd(gout.data_ptr(), Xb.data_ptr(), ldxb, Vb.data_ptr() if Q else None, ldvb, n, L,
                                       Q, vbs.data_ptr(), lvs.data_ptr(), None if null == "gX" else gX.data_ptr(), ldgx,
                                       None if null == "gV" or not Q else gV.data_ptr(), ldgv, glvs.data_ptr(), _st()),
          "taylor_expansion_bwd")
    torch.cuda.synchronize()
    assert int(out.view(torch.int32)[n]) == NAN_BITS, "taylor_expansion_fwd wrote past row n"
    ref, mag, c = _te_fwd_ref(X, Xb, [V] if Q else [], [Vb] if Q else [], vbs, lvs, n, L, [Q] if Q else [])
    grade(f"{tag} fwd", out[:n], ref, mag, 0.0, c)
    if null == "gX":
        assert bool((gX.view(torch.int32) == NAN_BITS).all()), "gX = NULL: the sentinel buffer was written"
    else:
        _bit_rows(f"{tag} gX", check_sentinel(gX, n, L, "taylor_expansion_bwd gX"), gout, Xb)
    if null == "gV" or not Q:
        assert bool((gV.view(torch.int32) == NAN_BITS).all()), "gV = NULL: the sentinel buffer was written"
    else:
        _bit_rows(f"{tag} gV", check_sentinel(gV, n, Q, "taylor_expansion_bwd gV"), gout, Vb)
    assert int(glvs.view(torch.int32)[2]) == NAN_BITS, "taylor_expansion_bwd wrote past glvs[1]"
    grade_glvs(tag, glvs[:2], gout, vbs, lvs)


# (widths, L, rows, lvs, designs whose gV is NULL, gX NULL)
MULTI = [([576], 132, "sweep+1", "big", (), False), ([4, 4368], 4, "sweep-1", "big", (1,), False),
         ([132, 4, 576], 256, "3sweep+17", "mild", (0, 2), True), ([4 * (1 + i % 5) for i in range(16)], 128, "64",
                                                                     "mild", tuple(range(1, 16, 2)), False),
         ([8, 132] * 8, 4, "1", "big", (), False)]


@pytest.mark.parametrize("case", MULTI, ids=lambda c: f"k{len(c[0])}-Q{sum(c[0])}-L{c[1]}-n{c[2]}-lvs_{c[3]}")
def test_taylor_multi(lib, case):
    from gppvae_b200._lib import host_i32, host_i64, host_ptrs
    widths, L, label, lk, vnull, xnull = case
    k, n = len(widths), rows_of(label)
    X, ldx = strided(spread_cols(n, L, seed=L + n, positive=False), 4)
    Xb, ldxb = strided(spread_cols(n, L, seed=L + n + 1, positive=False), 0)
    Vs, Vbs = [], []
    for j, Qj in enumerate(widths):
        Vs.append(strided(spread_cols(n, Qj, seed=n + 10 * j + 2, positive=False), 4 * (j % 3)))
        Vbs.append(strided(spread_cols(n, Qj, seed=n + 10 * j + 3, positive=False), 4 * ((j + 1) % 3)))
    vbs = torch.randn(k + 1, generator=_gen(n + k), device=DEV) * 10
    lvs = _lvs(lk, k + 1)
    tag = f"taylor_expansion_multi k={k} Q={widths if k < 4 else sum(widths)} L={L} n={n}"
    out = nan_vector(n)
    _call(lib.gpp_taylor_expansion_fwd_multi(X.data_ptr(), ldx, Xb.data_ptr(), ldxb, k,
                                             host_ptrs([V.data_ptr() for V, _ in Vs]), host_i64([ld for _, ld in Vs]),
                                             host_ptrs([V.data_ptr() for V, _ in Vbs]), host_i64([ld for _, ld in Vbs]),
                                             host_i32(widths), n, L, vbs.data_ptr(), lvs.data_ptr(), out.data_ptr(),
                                             _st()), "taylor_expansion_fwd_multi")
    gout = _mixed_gout(n, n + 7)
    gX, ldgx = sentinel(n, L)
    gVs = [sentinel(n, Qj) for Qj in widths]
    glvs = nan_vector(k + 1)
    _call(lib.gpp_taylor_expansion_bwd_multi(gout.data_ptr(), Xb.data_ptr(), ldxb, k,
                                             host_ptrs([V.data_ptr() for V, _ in Vbs]), host_i64([ld for _, ld in Vbs]),
                                             host_i32(widths), n, L, vbs.data_ptr(), lvs.data_ptr(),
                                             None if xnull else gX.data_ptr(), ldgx,
                                             host_ptrs([None if j in vnull else b.data_ptr()
                                                        for j, (b, _) in enumerate(gVs)]),
                                             host_i64([ld for _, ld in gVs]), glvs.data_ptr(), _st()),
          "taylor_expansion_bwd_multi")
    torch.cuda.synchronize()
    assert int(out.view(torch.int32)[n]) == NAN_BITS, "taylor_expansion_fwd_multi wrote past row n"
    ref, mag, c = _te_fwd_ref(X, Xb, [V for V, _ in Vs], [V for V, _ in Vbs], vbs, lvs, n, L, widths)
    grade(f"{tag} fwd", out[:n], ref, mag, 0.0, c)
    if xnull:
        assert bool((gX.view(torch.int32) == NAN_BITS).all()), "gX = NULL: the sentinel buffer was written"
    else:
        _bit_rows(f"{tag} gX", check_sentinel(gX, n, L, "taylor_expansion_bwd_multi gX"), gout, Xb)
    for j, ((b, _), (Vb, _)) in enumerate(zip(gVs, Vbs)):
        if j in vnull:
            assert bool((b.view(torch.int32) == NAN_BITS).all()), f"gV[{j}] = NULL: the sentinel buffer was written"
        else:
            _bit_rows(f"{tag} gV[{j}]", check_sentinel(b, n, widths[j], f"taylor_expansion_bwd_multi gV[{j}]"), gout,
                      Vb)
    print(f"[{tag}] gX and {k - len(vnull)} gV bit-identical, {len(vnull) + int(xnull)} NULL outputs untouched")
    assert int(glvs.view(torch.int32)[k + 1]) == NAN_BITS, "taylor_expansion_bwd_multi wrote past glvs[k]"
    grade_glvs(tag, glvs[:k + 1], gout, vbs, lvs)


UPSTREAMS = ("sum", "mean", "weighted")


@pytest.mark.parametrize("k", [1, 2])
@pytest.mark.parametrize("how", UPSTREAMS)
def test_taylor_through_gp(k, how):
    """GP.taylor_expansion at L = 6 and Q = 9 / 5 (the padded as_matrix path) for upstream gradients from .sum() (stride
    0), .mean() and a non-uniform weighting -- the surrogate is linear per row, so every weighting is legitimate --
    against fp64 autograd of the oracle.  gX and gV are one fp32 multiply of an fp32 upstream value (2 u with the
    rounding of 1/n); glvs adds that rounding to the bound of the module docstring."""
    from gppvae_b200 import GP
    from oracle import gp_oracle as O
    n, L, widths = 517, 6, [9, 5][:k]
    gp = GP(n_rand_effs=k).to(DEV)
    with torch.no_grad():
        gp.lvs.copy_(torch.tensor([0.4, -0.9, 1.3][:k + 1], device=DEV))
    g = _gen(k * 10 + len(how))
    X = torch.randn(n, L, generator=g, device=DEV).requires_grad_(True)
    Vs = [torch.randn(n, Qj, generator=g, device=DEV).requires_grad_(True) for Qj in widths]
    Xb = torch.randn(n, L, generator=g, device=DEV)
    Vbs = [torch.randn(n, Qj, generator=g, device=DEV) for Qj in widths]
    vbs = torch.randn(k + 1, generator=g, device=DEV) * 10
    wts = torch.randn(n, 1, generator=g, device=DEV)

    def up(o, wt):
        return o.sum() if how == "sum" else o.mean() if how == "mean" else (o * wt).sum()

    up(gp.taylor_expansion(X, Vs, Xb, Vbs, vbs), wts).backward()
    X64 = X.detach().double().requires_grad_(True)
    V64 = [V.detach().double().requires_grad_(True) for V in Vs]
    l64 = gp.lvs.detach().double().requires_grad_(True)
    up(O.taylor_expansion(X64, V64, Xb.double(), [V.double() for V in Vbs], vbs.double(), l64), wts.double()).backward()
    tag = f"GP(n_rand_effs={k}).taylor_expansion L={L} Q={widths} {how}"
    grade(f"{tag} gX", X.grad, X64.grad, X64.grad.abs(), 0.0, gamma(2))
    for j, (V, Vr) in enumerate(zip(Vs, V64)):
        grade(f"{tag} gV[{j}]", V.grad, Vr.grad, Vr.grad.abs(), 0.0, gamma(2))
    gup = torch.full((n,), 1.0 / n if how == "mean" else 1.0, dtype=torch.float64, device=DEV) if how != "weighted" \
        else wts.view(-1).double()
    grade_glvs(tag, gp.lvs.grad, gup, vbs, gp.lvs.detach(), extra_u=2 * U)
