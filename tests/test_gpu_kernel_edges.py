"""The N-long product entries and the Q-space factorisation against float64, at the shapes where the kernels switch
engine, cross tile edges and split their work, with an ELEMENTWISE bound.

Every N-long entry is graded element by element,

    |C - R|_ij  <=  c (|A|^T |B|)_ij  +  2^-31 (max|A| ||B_:,j||_1 + max|B| ||A_:,i||_1)        (A^T B; |A||M| for A M)

with R and the magnitude product computed in float64 on the device.  The first term is the relative error of the
arithmetic, derived (not fitted) per engine in units of u = 2^-24:

  tensor cores (tcgen05, 3-term fp16 split, DESIGN 5.0 / 5.1)
    * the split: hi = x rounded to 11 significant bits, lo = fp16(x - hi); the products hi.hi + hi.lo + lo.hi are exact
      in fp32 and miss lo.lo (<= 2^-22 |ab|) and the rounding of each lo (<= 2^-22 |ab| twice):            12 u
    * a window of 64 k-rows accumulates in TMEM, which rounds toward zero: 3 terms x 4 MMAs of K = 16, each counted
      twice (alignment of the 16 products inside the MMA, and the accumulator), each < 1 ulp = 2 u of the window's
      magnitude sum:                                                                                          48 u
    * the m = ceil(k / 64) finished windows are added in fp32 registers, round-to-nearest:                    m u
    * the split-K partials are added in fp64 (negligible) and rounded to fp32 once:                           1 u
  fp32 SIMT tiles: a chain of at most k fused multiply-adds per partial, fp64 reduction, one rounding:     (k + 1) u
  epilogues (X - A M, the 1/vn or alpha factor, the scale of B^-1 in Vb) add a few roundings:              +4 u

k is the length of the contraction one partial covers: the rows of a split for pass 1 (bounded by n where the split
count is the cost model's), Q (+ L) for the row products.  The second term is the floor of the common power-of-two
operand scale: the planes hold x 2^(7-e) with max|x| < 2^e, so the scaled maximum lies in [2^6, 2^7) and an element too
small for a normal fp16 lo keeps the absolute precision of half an fp16 subnormal, 2^-25, i.e. 2^-32 ... 2^-31 of its
matrix' maximum (DESIGN 5.0, test_outlier_rows_do_not_saturate).  For the epilogues |X| is added to the magnitude.

The inputs multiply every column by a factor between 1e-3 and 1e3 (and make some columns all-positive, which exposes
accumulation bias), so that the elementwise bound is far stricter than a max-relative error: a wrong ragged tile corner
in a small column cannot hide under the large columns.  Where the test calls a C entry itself the output is a sentinel
buffer (one extra row, ld = cols + 8, filled with a NaN bit pattern that must survive outside the n x cols block), and
inputs with ld > cols are views of wider tensors whose extra columns hold NaN, so that a read past `cols` shows up.

Each parametrisation names the engine the documented thresholds select (csrc/gemm_tc.cu, gemm_planes.cu):
pass 1 on the tensor cores from n >= 512 and Q >= 128; the row products from n >= 512, K >= 64 and ncols >= 64.
The file fails (does not skip) when the library was not built with the tensor-core engine.
"""
import math

import numpy as np
import pytest
import torch

from edge_helpers import (DEV, FLOOR, NAN_BITS, U, am_terms, atb_terms, c_simt, c_tc, check_sentinel, grade,
                          nan_vector, ratio_of, sentinel, spread_cols, strided)
from edge_helpers import call as _call
from edge_helpers import stream as _st
from edge_helpers import workspace as _ws

pytestmark = pytest.mark.gpu

TILE = 256                     # rows / columns of a CTA-pair tile


# ----------------------------------------------------------------------------------------------------------- helpers
@pytest.fixture(scope="module", autouse=True)
def lib():
    from gppvae_b200 import _lib
    engine = _lib.gemm_engine()
    assert engine == "tcgen05-3xf16", f"this file checks the tensor-core paths; the library was built with {engine}"
    return _lib.load()


def planes(X, ld, n, cols, colsq=False):
    """Operand planes of X.  The caller must hold the returned object until the kernel that reads it has run: its buffer
    goes back to the caching allocator with it, and the next allocation on the stream may reuse it."""
    from gppvae_b200 import ops
    return ops.split_planes(X, ld, n, cols, colsq=colsq)


def pass1_engine(n, Q):
    return "tc" if n >= 512 and Q >= 128 else "simt"


def rows_engine(n, K, ncols):
    return "tc" if n >= 512 and K >= 64 and ncols >= 64 else "simt"


# ------------------------------------------------------------------------------------------- A. N-long product entries
# (n, Q, L, pad): pad is added to the leading dimension of every input.  Covers n = 511/512/513 (engine switch),
# 767/768/769 (row tile edge), 1089 (n % 64 = 1) and 1023 (n % 64 = 63), 20000 (several splits); Q = 124/128/132
# (engine switch, Q % 8 = 4 for the planes' ldp), 252/256/260 (tile edge), 516, 1028 (ragged last tile); L = 4, 8
# (narrow C tiles), 60/64/68, 252/256/260, 516 (two and three column tiles) and 0.
PASS1 = [(511, 128, 64, 0), (767, 124, 60, 4), (511, 132, 0, 0), (512, 128, 64, 4), (513, 132, 68, 12),
         (768, 252, 4, 0), (769, 256, 8, 12), (767, 260, 60, 0), (1089, 260, 252, 4), (1023, 516, 256, 12),
         (1089, 128, 516, 0), (513, 260, 0, 12), (20000, 1028, 260, 4)]


def _pass1_id(s):
    n, Q, L, pad = s
    return f"n{n}-Q{Q}-L{L}-ld+{pad}-{pass1_engine(n, Q)}"


def _run_gram(lib, entry, V, ldv, X, ldx, n, Q, L):
    GC, ldgc = sentinel(Q, Q + L)
    ws = _ws(lib.gpp_gram_workspace_bytes(n, Q, L))
    fn = lib.gpp_gram_vtz if entry == "gram_vtz" else lib.gpp_gram_vtz_simt
    _call(fn(V.data_ptr(), ldv, X.data_ptr() if L else None, ldx, n, Q, L, GC.data_ptr(), ldgc, ws.data_ptr(), ws.numel(),
             _st()), entry)
    return check_sentinel(GC, Q, Q + L, entry)


def _run_gram_planes(lib, pV, pX, n, Q, L, use_colsq):
    GC, ldgc = sentinel(Q, Q + L)
    ws = _ws(lib.gpp_gram_planes_workspace_bytes(n, Q, L))
    _call(lib.gpp_gram_vtz_planes(pV.ptr, pX.ptr if pX is not None else None, n, Q, L, int(use_colsq), GC.data_ptr(),
                                  ldgc, ws.data_ptr(), ws.numel(), _st()), "gram_vtz_planes")
    return check_sentinel(GC, Q, Q + L, "gram_vtz_planes")


def _gram_ref(V, X, L):
    Q = V.shape[1]
    B = torch.cat([V, X], 1) if L else V
    maxB = torch.cat([torch.full((Q,), float(V.abs().max()), dtype=torch.float64, device=DEV),
                      torch.full((L,), float(X.abs().max()) if L else 0.0, dtype=torch.float64, device=DEV)])
    return atb_terms(V, B, maxB)


@pytest.mark.parametrize("shape", PASS1, ids=_pass1_id)
def test_pass1_gram_entries(lib, shape):
    """gpp_gram_vtz, gpp_gram_vtz_simt and (at tensor-core shapes) gpp_gram_vtz_planes with and without colsq against
    fp64; G exactly symmetric; with colsq, diag(G) the correctly rounded fp32 of the fp64 column sums (DESIGN 5.0)."""
    n, Q, L, pad = shape
    V0 = spread_cols(n, Q, seed=n + Q)
    X0 = spread_cols(n, L, seed=n + Q + 1) if L else None
    V, ldv = strided(V0, pad)
    X, ldx = strided(X0, pad) if L else (None, 4)
    R, mag, floor = _gram_ref(V0, X0, L)
    eng = pass1_engine(n, Q)
    outs = {"gram_vtz": (_run_gram(lib, "gram_vtz", V, ldv, X, ldx, n, Q, L), c_tc(n) if eng == "tc" else c_simt(n)),
            "gram_vtz_simt": (_run_gram(lib, "gram_vtz_simt", V, ldv, X, ldx, n, Q, L), c_simt(n))}
    if eng == "tc":
        pV = planes(V, ldv, n, Q, colsq=True)
        pX = planes(X, ldx, n, L) if L else None
        outs["gram_vtz_planes colsq"] = (_run_gram_planes(lib, pV, pX, n, Q, L, True), c_tc(n))
        outs["gram_vtz_planes"] = (_run_gram_planes(lib, pV, pX, n, Q, L, False), c_tc(n))
    torch.cuda.synchronize()
    colsq = (V0.double() ** 2).sum(0)
    for name, (GC, c) in outs.items():
        tag = f"{name} n={n} Q={Q} L={L} ld+{pad} {eng if name != 'gram_vtz_simt' else 'simt'}"
        grade(tag, GC, R, mag, floor, c)
        assert torch.equal(GC[:, :Q], GC[:, :Q].t()), f"{tag}: G is not exactly symmetric"
        if name.endswith("colsq"):
            d = (torch.diagonal(GC[:, :Q]).double() - colsq).abs() / colsq
            print(f"[{tag}] diag(G) worst relative error {float(d.max()):.2e} (bound 2^-24 = {U:.2e})")
            assert float(d.max()) <= U, f"{tag}: diag(G) is not the correctly rounded column sum of squares"


ATB = [s for s in PASS1 if s[2] > 0]


def _run_atb(lib, A, lda, B, ldb, n, ka, kb):
    out, ldo = sentinel(ka, kb)
    ws = _ws(lib.gpp_atb_workspace_bytes(n, ka, kb))
    _call(lib.gpp_atb(A.data_ptr(), lda, B.data_ptr(), ldb, n, ka, kb, out.data_ptr(), ldo, ws.data_ptr(), ws.numel(),
                      _st()), "atb")
    return check_sentinel(out, ka, kb, "atb")


def _run_atb_planes(lib, pA, pB, n, ka, kb):
    out, ldo = sentinel(ka, kb)
    ws = _ws(lib.gpp_gram_planes_workspace_bytes(n, ka, kb))
    _call(lib.gpp_atb_planes(pA.ptr, pB.ptr, n, ka, kb, out.data_ptr(), ldo, ws.data_ptr(), ws.numel(), _st()),
          "atb_planes")
    return check_sentinel(out, ka, kb, "atb_planes")


@pytest.mark.parametrize("shape", ATB, ids=_pass1_id)
def test_atb_entries(lib, shape):
    """gpp_atb and (at tensor-core shapes) gpp_atb_planes: out = A^T B against fp64."""
    n, ka, kb, pad = shape
    A0, B0 = spread_cols(n, ka, seed=3 * n + ka), spread_cols(n, kb, seed=3 * n + kb + 7)
    A, lda = strided(A0, pad)
    B, ldb = strided(B0, pad)
    R, mag, floor = atb_terms(A0, B0)
    eng = pass1_engine(n, ka)
    grade(f"atb n={n} ka={ka} kb={kb} ld+{pad} {eng}", _run_atb(lib, A, lda, B, ldb, n, ka, kb), R, mag, floor,
          c_tc(n) if eng == "tc" else c_simt(n))
    if eng == "tc":
        out = _run_atb_planes(lib, planes(A, lda, n, ka), planes(B, ldb, n, kb), n, ka, kb)
        grade(f"atb_planes n={n} ka={ka} kb={kb} ld+{pad} tc", out, R, mag, floor, c_tc(n))


# (n, K, m, pad) of the row products: out (n x m) from A (n x K) and M (K x m).  m = 260 / 516 gives the row kernel
# two / three column tiles; K = 1028 a ragged last k-stage.
ROWS = [(511, 128, 64, 0), (513, 124, 60, 4), (769, 132, 8, 12), (512, 128, 64, 4), (768, 124, 68, 12),
        (767, 252, 4, 0), (1089, 256, 252, 4), (1023, 260, 256, 12), (769, 516, 260, 0), (1089, 1028, 516, 4),
        (20000, 1028, 260, 12)]


def _rows_id(s):
    n, K, m, pad = s
    return f"n{n}-K{K}-m{m}-ld+{pad}-{rows_engine(n, K, m)}"


@pytest.mark.parametrize("shape", ROWS, ids=_rows_id)
def test_row_product_entries(lib, shape):
    """gpp_x_minus_am (alpha = -0.75), gpp_am and (at tensor-core shapes) gpp_am_planes (alpha = 1.5) against fp64."""
    n, k, m, pad = shape
    A0, M0 = spread_cols(n, k, seed=n + 5 * k), spread_cols(k, m, seed=n + 5 * k + 1)
    X0 = spread_cols(n, m, seed=n + 5 * k + 2, positive=False)
    A, lda = strided(A0, pad)
    M, ldm = strided(M0, pad)
    X, ldx = strided(X0, pad)
    R, mag, floor = am_terms(A0, M0)
    eng = rows_engine(n, k, m)
    c = c_tc(k, 4) if eng == "tc" else c_simt(k, 4)
    tag = f"n={n} k={k} m={m} ld+{pad} {eng}"

    alpha = -0.75
    out, ldo = sentinel(n, m)
    ws = _ws(lib.gpp_rows_workspace_bytes())
    _call(lib.gpp_x_minus_am(X.data_ptr(), ldx, A.data_ptr(), lda, M.data_ptr(), ldm, n, k, m, alpha, out.data_ptr(), ldo,
                             ws.data_ptr(), ws.numel(), _st()), "x_minus_am")
    out = check_sentinel(out, n, m, "x_minus_am")
    grade(f"x_minus_am {tag}", out, alpha * (X0.double() - R), abs(alpha) * (X0.double().abs() + mag), abs(alpha) * floor,
          c)

    for name in (("am", "am_planes") if eng == "tc" else ("am",)):
        alpha = 1.5
        out, ldo = sentinel(n, m)
        ws = _ws(256)
        if name == "am":
            st = lib.gpp_am(A.data_ptr(), lda, M.data_ptr(), ldm, n, k, m, alpha, out.data_ptr(), ldo, ws.data_ptr(),
                            ws.numel(), _st())
        else:
            pA, pM = planes(A, lda, n, k), planes(M, ldm, k, m)   # held until the kernel has run
            st = lib.gpp_am_planes(pA.ptr, pM.ptr, n, k, m, alpha, out.data_ptr(), ldo, ws.data_ptr(), ws.numel(), _st())
        _call(st, name)
        out = check_sentinel(out, n, m, name)
        grade(f"{name} {tag}", out, alpha * R, alpha * mag, alpha * floor, c)


def _scal(v0=0.7, vn=0.3, rowconst=-1.25):
    from gppvae_b200._lib import NSCAL, S_ROWCONST, S_V0, S_VN
    s = torch.zeros(NSCAL, dtype=torch.float64, device=DEV)
    s[S_V0], s[S_VN], s[S_ROWCONST] = v0, vn, rowconst
    return s


@pytest.mark.parametrize("shape", ROWS, ids=_rows_id)
def test_xb_nll_entries(lib, shape):
    """gpp_xb_nll and (at tensor-core shapes) gpp_xb_nll_planes with the scalar block filled by hand: Xb = (X - V W)/vn
    elementwise, nll_i = X_i.Xb_i / 2 + ROWCONST per row, scal[XB2] and scal[QUAD] against fp64 sums.  The bounds of
    the three sums follow from the elementwise bound E of Xb, plus the fp32 partial sums of the epilogue (at most 128
    products and 5 shuffle levels before a partial reaches fp64: 136 u)."""
    from gppvae_b200._lib import S_QUAD, S_ROWCONST, S_VN, S_XB2
    n, Q, L, pad = shape
    V0, W0 = spread_cols(n, Q, seed=n + 11 * Q), spread_cols(Q, L, seed=n + 11 * Q + 1) * 1e-2
    X0 = spread_cols(n, L, seed=n + 11 * Q + 2, positive=False)
    V, ldv = strided(V0, pad)
    W, ldw = strided(W0, pad)
    X, ldx = strided(X0, pad)
    P, mag, floor = am_terms(V0, W0)
    eng = rows_engine(n, Q, L)
    runs = [("xb_nll", eng)] + ([("xb_nll_planes", "tc")] if eng == "tc" else [])
    for name, e in runs:
        scal = _scal()
        vn = float(scal[S_VN])
        rowconst = float(scal[S_ROWCONST])
        Xb, ldxb = sentinel(n, L)
        nll = nan_vector(n)
        if name == "xb_nll":
            ws = _ws(lib.gpp_xb_workspace_bytes(n, Q, L))
            st = lib.gpp_xb_nll(V.data_ptr(), ldv, X.data_ptr(), ldx, W.data_ptr(), ldw, n, Q, L, scal.data_ptr(),
                                Xb.data_ptr(), ldxb, nll.data_ptr(), ws.data_ptr(), ws.numel(), _st())
        else:
            ws = _ws(lib.gpp_xb_planes_workspace_bytes(n, Q, L))
            pV = planes(V, ldv, n, Q)
            st = lib.gpp_xb_nll_planes(pV.ptr, X.data_ptr(), ldx, W.data_ptr(), ldw, n, Q, L,
                                       scal.data_ptr(), Xb.data_ptr(), ldxb, nll.data_ptr(), ws.data_ptr(), ws.numel(),
                                       _st())
        _call(st, name)
        Xb = check_sentinel(Xb, n, L, name)
        assert nll.view(torch.int32)[n] == NAN_BITS, f"{name}: wrote nll past row {n}"
        tag = f"{name} n={n} Q={Q} L={L} ld+{pad} {e}"
        R = (X0.double() - P) / vn
        E = ((c_tc(Q, 4) if e == "tc" else c_simt(Q, 4)) * (X0.double().abs() + mag) + floor) / vn
        grade(tag, Xb, R, (X0.double().abs() + mag) / vn, floor / vn, c_tc(Q, 4) if e == "tc" else c_simt(Q, 4))
        x, xb = X0.double(), Xb.double()
        quad_ref = (x * R).sum(1)
        nll_ref = 0.5 * quad_ref + rowconst
        nll_lim = 0.5 * ((x.abs() * E).sum(1) + 136 * U * (x * xb).abs().sum(1)) + U * (nll_ref.abs() + abs(rowconst))
        r_nll = ratio_of((nll[:n].double() - nll_ref).abs(), nll_lim)
        xb2_ref, q_ref = float((R * R).sum()), float(quad_ref.sum())
        xb2_lim = float((2 * R.abs() * E + E * E).sum() + 136 * U * (xb * xb).sum())
        q_lim = float((x.abs() * E).sum() + 136 * U * (x * xb).abs().sum())
        sc = scal.cpu().numpy()
        r_xb2, r_q = abs(sc[S_XB2] - xb2_ref) / xb2_lim, abs(sc[S_QUAD] - q_ref) / q_lim
        print(f"[{tag}] worst bound ratio nll {r_nll:.3f}  scal[XB2] {r_xb2:.3f}  scal[QUAD] {r_q:.3f}")
        assert r_nll <= 1.0 and r_xb2 <= 1.0 and r_q <= 1.0


def _vb_engine(n, Q, L, planes_):
    if planes_:
        return "tc"
    return "tc" if n >= 512 and Q + L >= 64 and Q >= 64 else "simt"


@pytest.mark.parametrize("shape", ROWS, ids=lambda s: f"n{s[0]}-Q{s[1]}-L{s[2]}-ld+{s[3]}-{_vb_engine(s[0], s[1], s[2], False)}")
def test_vb_entries(lib, shape):
    """gpp_vb and (at tensor-core shapes with Q >= 128) gpp_vb_planes: Vb = r L_true V B^-1 - Xb W^T, r = v0/vn, graded
    against r L_true |V||B^-1| + |Xb||W|^T.  Both parts run as ONE product [V | Xb] [r L_true B^-1 ; -W^T]: the
    contraction is Q + L long, the stacked right operand shares one scale, and r L_true and its product with B^-1 are
    rounded to fp32 (2 u)."""
    from gppvae_b200._lib import S_V0, S_VN
    n, Q, L, pad = shape
    L_true = L - 2
    V0 = spread_cols(n, Q, seed=n + 13 * Q)
    Xb0 = spread_cols(n, L, seed=n + 13 * Q + 1, positive=False)
    Binv = spread_cols(Q, Q, seed=n + 13 * Q + 2) * 1e-3
    W0 = spread_cols(Q, L, seed=n + 13 * Q + 3, positive=False) * 1e-2
    V, ldv = strided(V0, pad)
    Xbv, ldxb = strided(Xb0, pad)
    W, ldw = strided(W0, pad)
    scal = _scal()
    coef = float(np.float32(float(scal[S_V0]) / float(scal[S_VN]) * L_true))
    P1, m1, _ = am_terms(V0, Binv)
    P2, m2, _ = am_terms(Xb0, W0.t())
    R = coef * P1 - P2
    mag = coef * m1 + m2
    aV, aXb, aBi, aW = V0.double().abs(), Xb0.double().abs(), Binv.double().abs(), W0.double().abs()
    maxB = max(coef * float(aBi.max()), float(aW.max()))
    floor = FLOOR * (float(aV.max()) * coef * aBi.sum(0)[None, :] + float(aXb.max()) * aW.sum(1)[None, :]
                     + maxB * (aV.sum(1) + aXb.sum(1))[:, None])
    eng = _vb_engine(n, Q, L, False)
    runs = [("vb", eng)] + ([("vb_planes", "tc")] if n >= 512 and Q >= 128 else [])
    for name, e in runs:
        Vb, ldvb = sentinel(n, Q)
        if name == "vb":
            ws = _ws(lib.gpp_vb_workspace_bytes(n, Q, L))
            st = lib.gpp_vb(V.data_ptr(), ldv, Xbv.data_ptr(), ldxb, Binv.data_ptr(), W.data_ptr(), ldw, scal.data_ptr(),
                            n, Q, L, L_true, Vb.data_ptr(), ldvb, ws.data_ptr(), ws.numel(), _st())
        else:
            ws = _ws(lib.gpp_vb_planes_workspace_bytes(n, Q, L))
            pV = planes(V, ldv, n, Q)
            st = lib.gpp_vb_planes(pV.ptr, Xbv.data_ptr(), ldxb, Binv.data_ptr(), W.data_ptr(), ldw,
                                   scal.data_ptr(), n, Q, L, L_true, Vb.data_ptr(), ldvb, ws.data_ptr(), ws.numel(), _st())
        _call(st, name)
        Vb = check_sentinel(Vb, n, Q, name)
        c = c_tc(Q + L, 2) if e == "tc" else c_simt(Q + L, 2)
        grade(f"{name} n={n} Q={Q} L={L} L_true={L_true} ld+{pad} {e}", Vb, R, mag, floor, c)


# ------------------------------------------------------------------ B. split-K and scheduling variants of pass 1
def split_geometry(n, r, kblock):
    """What pass1_geometry (csrc/gemm_tc.cu) makes of GPP_TC_SPLIT_ROWS = r: s = ceil(n / r) splits requested, rows per
    split ceil(n / s) rounded up to the k-block, and the split count that results."""
    s = -(-n // r)
    rps = -(-(-(-n // s)) // kblock) * kblock
    return rps, -(-n // rps)


# (entry, n, Q, L, r): unequal splits whose last one ends in a partial k-block (n % 64 = 63 and = 1), and r = 512 at
# n = 20033, which asks for more splits (40) than the cost model can ever pick (at most n // 512 = 39).
SPLITS = [(e, *s) for e in ("gram_vtz", "gram_vtz_planes", "atb", "atb_planes")
          for s in ((5055, 260, 68, 1500), (1089, 132, 256, 700), (20033, 516, 260, 512))]


@pytest.mark.parametrize("entry,n,Q,L,r", SPLITS, ids=[f"{e}-n{n}-Q{Q}-L{L}-r{r}-tc" for e, n, Q, L, r in SPLITS])
def test_split_rows_knob(lib, monkeypatch, entry, n, Q, L, r):
    """GPP_TC_SPLIT_ROWS moves the split-K count of pass 1: the result must meet the fp64 bound (with m = the windows
    of one split) and agree with the default split count to within both bounds.  The geometry is mirrored here; the
    planes entries' workspace query, which sizes the partial tiles as tiles x splits, confirms it."""
    planes_ = entry.endswith("planes")
    kblock = 64 if planes_ else 16
    rps, splits = split_geometry(n, r, kblock)
    last = n - (splits - 1) * rps
    assert splits >= 2 and 0 < last < rps and last % kblock != 0, (rps, splits, last)
    if r == 512:
        assert splits > n // 512
    gram = entry.startswith("gram")
    tm = -(-Q // TILE)
    tiles = tm * (tm + 1) // 2 + tm * -(-L // TILE)
    V0, X0 = spread_cols(n, Q, seed=n + 17), spread_cols(n, L, seed=n + 18)
    V, ldv = strided(V0, 4)
    X, ldx = strided(X0, 4)
    if gram:
        R, mag, floor = _gram_ref(V0, X0, L)
    else:
        R, mag, floor = atb_terms(V0, X0)

    def run():
        if entry == "gram_vtz":
            return _run_gram(lib, "gram_vtz", V, ldv, X, ldx, n, Q, L)
        if entry == "atb":
            return _run_atb(lib, V, ldv, X, ldx, n, Q, L)
        pV, pX = planes(V, ldv, n, Q, colsq=True), planes(X, ldx, n, L)
        if entry == "gram_vtz_planes":
            return _run_gram_planes(lib, pV, pX, n, Q, L, True)
        return _run_atb_planes(lib, pV, pX, n, Q, L)

    ref_out = run().clone()
    monkeypatch.setenv("GPP_TC_SPLIT_ROWS", str(r))
    if planes_:   # serves both planes entries: sized for the Gram tiles too
        wsb = lib.gpp_gram_planes_workspace_bytes(n, Q, L)
        assert wsb == tiles * splits * TILE * TILE * 4 + 256, f"workspace {wsb}: not {tiles} tiles x {splits} splits"
    else:         # the larger of the tensor-core partials and the SIMT engine's
        wsb = lib.gpp_gram_workspace_bytes(n, Q, L) if gram else lib.gpp_atb_workspace_bytes(n, Q, L)
        assert wsb >= (tiles if gram else tm * -(-L // TILE)) * splits * TILE * TILE * 4 + 256
    out = run()
    torch.cuda.synchronize()
    tag = f"{entry} n={n} Q={Q} L={L} GPP_TC_SPLIT_ROWS={r}: {splits} splits of {rps} rows, last {last}"
    grade(tag, out, R, mag, floor, c_tc(rps))
    grade(f"{entry} n={n} Q={Q} L={L} r={r} against the default split count", out, ref_out.double(), mag, 2 * floor,
          c_tc(rps) + c_tc(n))


@pytest.mark.parametrize("entry", ["gram_vtz", "gram_vtz_planes", "xb_nll", "xb_nll_planes", "vb", "vb_planes"])
def test_wave_sync_off_is_bit_identical(lib, monkeypatch, entry):
    """GPP_TC_WAVE_SYNC=0 only changes when the TMA producers issue; every reduction is fixed-order, so the outputs
    must not change by a bit.  n = 20000 rows, Q = 1028, L = 260: more units than one wave, several column tiles."""
    n, Q, L = 20000, 1028, 260
    V0, X0 = spread_cols(n, Q, seed=41), spread_cols(n, L, seed=42, positive=False)
    W0 = spread_cols(Q, L, seed=43, positive=False) * 1e-2
    Binv = spread_cols(Q, Q, seed=44) * 1e-3
    pV = planes(V0, Q, n, Q, colsq=True)

    def run():
        scal = _scal()
        if entry == "gram_vtz":
            outs = [_run_gram(lib, "gram_vtz", V0, Q, X0, L, n, Q, L)]
        elif entry == "gram_vtz_planes":
            outs = [_run_gram_planes(lib, pV, planes(X0, L, n, L), n, Q, L, True)]
        elif entry.startswith("xb_nll"):
            Xb, nll = torch.empty(n, L, device=DEV), torch.empty(n, device=DEV)
            if entry == "xb_nll":
                ws = _ws(lib.gpp_xb_workspace_bytes(n, Q, L))
                st = lib.gpp_xb_nll(V0.data_ptr(), Q, X0.data_ptr(), L, W0.data_ptr(), L, n, Q, L, scal.data_ptr(),
                                    Xb.data_ptr(), L, nll.data_ptr(), ws.data_ptr(), ws.numel(), _st())
            else:
                ws = _ws(lib.gpp_xb_planes_workspace_bytes(n, Q, L))
                st = lib.gpp_xb_nll_planes(pV.ptr, X0.data_ptr(), L, W0.data_ptr(), L, n, Q, L, scal.data_ptr(),
                                           Xb.data_ptr(), L, nll.data_ptr(), ws.data_ptr(), ws.numel(), _st())
            _call(st, entry)
            outs = [Xb, nll, scal]
        else:
            Vb = torch.empty(n, Q, device=DEV)
            if entry == "vb":
                ws = _ws(lib.gpp_vb_workspace_bytes(n, Q, L))
                st = lib.gpp_vb(V0.data_ptr(), Q, X0.data_ptr(), L, Binv.data_ptr(), W0.data_ptr(), L, scal.data_ptr(),
                                n, Q, L, L, Vb.data_ptr(), Q, ws.data_ptr(), ws.numel(), _st())
            else:
                ws = _ws(lib.gpp_vb_planes_workspace_bytes(n, Q, L))
                st = lib.gpp_vb_planes(pV.ptr, X0.data_ptr(), L, Binv.data_ptr(), W0.data_ptr(), L, scal.data_ptr(),
                                       n, Q, L, L, Vb.data_ptr(), Q, ws.data_ptr(), ws.numel(), _st())
            _call(st, entry)
            outs = [Vb]
        torch.cuda.synchronize()
        return [o.clone() for o in outs]

    base = run()
    monkeypatch.setenv("GPP_TC_WAVE_SYNC", "0")
    off = run()
    same = [torch.equal(a, b) for a, b in zip(base, off)]
    print(f"[{entry} n={n} Q={Q} L={L}] GPP_TC_WAVE_SYNC=0 bit-identical: {same}")
    assert all(same)


# ------------------------------------------------------------------------------------------------------ C. Q-space
def _qspace_problem(Q, r, L=68, L_true=65, seed=0):
    """B = I + r G from G = V^T V (a few dominant directions, as test_qspace_large_against_fp64), C with L - L_true
    zero padding columns, and the fp64 Cholesky quantities."""
    g = torch.Generator(device=DEV).manual_seed(Q + seed)
    n = 3 * Q
    V = torch.randn(n, Q, generator=g, device=DEV, dtype=torch.float64) / Q ** 0.5
    V[:, : max(1, Q // 8)] *= 4.0
    G64 = V.t() @ V
    C64 = torch.zeros(Q, L, device=DEV, dtype=torch.float64)
    C64[:, :L_true] = torch.randn(Q, L_true, generator=g, device=DEV, dtype=torch.float64)
    vn = 1.0 / (1.0 + r)
    vs = torch.tensor([1.0 - vn, vn], device=DEV, dtype=torch.float32)
    r_eff = float(vs[0].double() / vs[1].double())
    GC = torch.zeros(Q, Q + L, device=DEV)
    GC[:, :Q] = G64.float()
    GC[:, Q:] = C64.float()
    # the fp64 truth of what the kernels see: the fp32 G and C
    B64 = torch.eye(Q, device=DEV, dtype=torch.float64) + r_eff * GC[:, :Q].double()
    Lc = torch.linalg.cholesky(B64)
    ref = dict(logdet=2.0 * float(torch.log(torch.diagonal(Lc)).sum()), Binv=torch.cholesky_inverse(Lc),
               W=r_eff * torch.cholesky_solve(GC[:, Q:].double(), Lc))
    ref["tr"] = float(ref["Binv"].trace())
    return dict(Q=Q, L=L, L_true=L_true, n=n, vs=vs, GC=GC, ref=ref)


def _qspace_run(pb):
    from gppvae_b200 import ops
    Q, L = pb["Q"], pb["L"]
    fac = ops.factor(pb["GC"], Q + L, Q, pb["vs"], True)
    W, scal = ops.solve_w(fac, pb["GC"][:, Q:], Q + L, L, pb["L_true"], pb["n"])
    torch.cuda.synchronize()
    return fac.Binv.clone(), W.clone(), scal.clone()


def _qspace_check(pb, out, what):
    """The bounds of test_qspace_large_against_fp64; the padding columns of W exactly zero; ROWCONST from L_true."""
    from conftest import rel_err
    from gppvae_b200._lib import S_LOGDETB, S_ROWCONST, S_TRBINV, S_VN
    Binv, W, scal = out
    Q, L_true, ref = pb["Q"], pb["L_true"], pb["ref"]
    sc = scal.cpu().numpy()
    e_ld = abs(sc[S_LOGDETB] - ref["logdet"]) / abs(ref["logdet"])
    e_tr = abs(sc[S_TRBINV] - ref["tr"]) / ref["tr"]
    e_bi, e_w = rel_err(Binv, ref["Binv"]), rel_err(W[:, :L_true], ref["W"][:, :L_true])
    print(f"[{what}] logdet {e_ld:.2e}  trBinv {e_tr:.2e}  Binv {e_bi:.2e}  W {e_w:.2e}")
    assert e_ld < 1e-6 and e_tr < 1e-4 and e_bi < 1e-4 and e_w < 1e-4
    assert bool((W[:, L_true:] == 0).all()), f"{what}: the zero padding columns of C gave non-zero columns of W"
    rc = 0.5 * L_true * (math.log(sc[S_VN]) + sc[S_LOGDETB] / pb["n"])
    assert abs(sc[S_ROWCONST] - rc) <= 1e-12 * abs(rc), f"{what}: ROWCONST {sc[S_ROWCONST]} != {rc} (L_true = {L_true})"


@pytest.mark.parametrize("r", [1.0, 400.0])
@pytest.mark.parametrize("Q", [68, 124, 132, 508, 516, 1028, 1092, 2052])
def test_qspace_ragged_padded_q(Q, r):
    """gpp_factor + gpp_solve_w at Q that are not multiples of the 64-wide panel (partial last panel); from 1024 up the
    side-stream inverse runs, with a short trailing block after b_top."""
    pb = _qspace_problem(Q, r)
    _qspace_check(pb, _qspace_run(pb), f"qspace Q={Q} (Qp={-(-Q // 64) * 64}) r={r:g}")


def _fork_steps(Q):
    Qp = -(-Q // 64) * 64
    nb = Qp // 64
    b_top = 64
    while b_top * 2 < Qp:
        b_top *= 2
    jsplit = b_top // 64
    return jsplit, nb, max(jsplit - 1, (3 * nb) // 4)


@pytest.mark.parametrize("Q", [1028, 1988, 2052])
def test_qspace_launch_order_schedules_are_bit_identical(monkeypatch, Q):
    """PDL off, no side stream, and the side stream forked at the earliest step (jsplit - 1) and at the last (nb - 1)
    only reorder launches around the same arithmetic: B^-1, W and the scalar block must match the default to the bit.
    The earliest fork is the strongest check of the fork/join events.  (At Q = 1028 and 2052 the default fork already is
    jsplit - 1; Q = 1988 has a default fork of 3 nb / 4 = 24 against jsplit - 1 = 15.)"""
    jsplit, nb, default_fork = _fork_steps(Q)
    pb = _qspace_problem(Q, 400.0, seed=1)
    base = _qspace_run(pb)
    _qspace_check(pb, base, f"qspace Q={Q} default (fork at {default_fork})")
    for knob, val in (("GPP_CHOL_PDL", "0"), ("GPP_INV_OVERLAP", "0"), ("GPP_INV_FORK", str(jsplit - 1)),
                      ("GPP_INV_FORK", str(nb - 1))):
        monkeypatch.setenv(knob, val)
        out = _qspace_run(pb)
        monkeypatch.delenv(knob)
        same = [torch.equal(a, b) for a, b in zip(base, out)]
        print(f"[qspace Q={Q} {knob}={val}] bit-identical (Binv, W, scal): {same}")
        assert all(same), f"{knob}={val} changed the result at Q = {Q}: a missing dependency"


SUM_ORDER = [("GPP_CHOL_WIDE", "rl", 1028), ("GPP_CHOL_WIDE", "rl", 2052), ("GPP_INV_SIDE_SMS", "16", 1028),
             ("GPP_INV_SIDE_SMS", "16", 2052), ("GPP_CHOL_OUTER_MIN_Q", "1024", 1028),
             ("GPP_CHOL_OUTER_MIN_Q", "1024", 1092)]


@pytest.mark.parametrize("knob,val,Q", SUM_ORDER, ids=[f"{k}={v}-Q{q}" for k, v, q in SUM_ORDER])
def test_qspace_sum_order_schedules_against_fp64(monkeypatch, knob, val, Q):
    """Schedules that reorder sums (right-looking updates, SMs set aside for the side stream, the outer-block scheme
    with a ragged last outer block at Q = 1092) meet the fp64 bounds of the default."""
    monkeypatch.setenv(knob, val)
    for r in (1.0, 400.0):
        pb = _qspace_problem(Q, r, seed=2)
        _qspace_check(pb, _qspace_run(pb), f"qspace Q={Q} r={r:g} {knob}={val}")


@pytest.mark.parametrize("widths,scaled", [([516, 132, 12], 1), ([12, 1028], 0)], ids=["516-132-12", "12-1028"])
def test_factor_blocks_at_ragged_block_edges(widths, scaled):
    """gpp_factor_blocks / gpp_solve_w_blocks / gpp_vbs_blocks with block edges off the panel edges and one design
    scaled by 1e-3, against fp64 B = I + D G D / vn, W = D B^-1 D C / vn, the per-block tr_i B^-1 and ||W_i||^2 and the
    k + 1 vbs.  ||W_i||^2 and vbs are graded with the error they inherit from the W and tr bounds."""
    from conftest import rel_err
    from gppvae_b200 import ops
    from gppvae_b200._lib import S_LOGDETB, S_TRBINV, S_XB2
    k, Q, L = len(widths), sum(widths), 64
    n = 3 * Q
    g = torch.Generator(device=DEV).manual_seed(Q)
    V = torch.randn(n, Q, generator=g, device=DEV, dtype=torch.float64) / Q ** 0.5
    off = [sum(widths[:i]) for i in range(k + 1)]
    V[:, off[scaled]:off[scaled + 1]] *= 1e-3
    X = torch.randn(n, L, generator=g, device=DEV, dtype=torch.float64)
    GC = torch.cat([V.t() @ V, V.t() @ X], 1).float()
    vs = torch.tensor([0.5, 0.2, 0.1, 0.2] if k == 3 else [0.6, 0.1, 0.3], device=DEV, dtype=torch.float32)
    v = vs.double()
    vn = float(v[k])
    d = torch.cat([torch.full((w,), float(v[i].sqrt()), dtype=torch.float64, device=DEV) for i, w in enumerate(widths)])
    B64 = torch.eye(Q, dtype=torch.float64, device=DEV) + d[:, None] * GC[:, :Q].double() * d[None, :] / vn
    Lc = torch.linalg.cholesky(B64)
    Bi = torch.cholesky_inverse(Lc)
    W64 = d[:, None] * torch.cholesky_solve(d[:, None] * GC[:, Q:].double(), Lc) / vn
    fac = ops.factor_blocks(GC, Q + L, widths, vs, True)
    W, scal, blk = ops.solve_w_blocks(fac, GC[:, Q:], Q + L, L, L, n)
    scal[S_XB2] = 123.25
    vbs = ops.vbs_blocks(scal, blk, vs, widths, n, L)
    torch.cuda.synchronize()
    sc, bk = scal.cpu().numpy(), blk.cpu().numpy()
    logdet = 2.0 * float(torch.log(torch.diagonal(Lc)).sum())
    e_ld, e_tr = abs(sc[S_LOGDETB] - logdet) / abs(logdet), abs(sc[S_TRBINV] - float(Bi.trace())) / float(Bi.trace())
    e_bi, e_w = rel_err(fac.Binv, d[:, None] * Bi * d[None, :]), rel_err(W, W64)
    print(f"[blocks {widths}, design {scaled} x 1e-3] logdet {e_ld:.2e}  trBinv {e_tr:.2e}  DBinvD {e_bi:.2e}  W {e_w:.2e}")
    assert e_ld < 1e-6 and e_tr < 1e-4 and e_bi < 1e-4 and e_w < 1e-4
    delta = 1e-4 * float(W64.abs().max())              # the W bound, elementwise
    vbs_ref, vbs_lim = [], []
    for i in range(k):
        Wi = W64[off[i]:off[i + 1]]
        tr_i, w2_i = float(torch.diagonal(Bi)[off[i]:off[i + 1]].sum()), float((Wi * Wi).sum())
        w2_lim = float((2 * Wi.abs() * delta + delta * delta).sum())
        e_tri, r_w2 = abs(bk[2 * i] - tr_i) / tr_i, abs(bk[2 * i + 1] - w2_i) / w2_lim
        print(f"   block {i} ({widths[i]} cols): tr_i {e_tri:.2e}  ||W_i||^2 bound ratio {r_w2:.3f}")
        assert e_tri < 1e-4 and r_w2 <= 1.0
        vi = float(v[i])
        vbs_ref.append(-0.5 * w2_i / vi ** 2 + 0.5 * L * (widths[i] - tr_i) / vi)
        vbs_lim.append(0.5 * w2_lim / vi ** 2 + 0.5 * L * 1e-4 * tr_i / vi)
    trB = float(Bi.trace())
    vbs_ref.append(-0.5 * 123.25 + 0.5 * L * (n - Q + trB) / vn)
    vbs_lim.append(0.5 * L * 1e-4 * trB / vn)
    got = vbs.double().cpu().numpy()
    for i in range(k + 1):
        lim = vbs_lim[i] + U * abs(vbs_ref[i])
        print(f"   vbs[{i}] = {got[i]:.6g} (fp64 {vbs_ref[i]:.6g}) bound ratio {abs(got[i] - vbs_ref[i]) / lim:.3f}")
        assert abs(got[i] - vbs_ref[i]) <= lim
