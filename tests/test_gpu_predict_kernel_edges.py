"""The three entries of GP.predict (gpp_kr_predict_views, gpp_kr_predict_rows, gpp_rows_dot; DESIGN 5.9) against float64,
element by element, with the conventions of test_gpu_structured_kernel_edges.py: sentinel output buffers (one extra row,
ld = cols + 8, a NaN bit pattern that must survive), inputs with ld > cols whose gap holds NaN, and the worst bound ratio
printed per case.  The references are fp64 evaluations of the header formulas on the same fp32 inputs, through the
row maps u = A_v x + b_v (not the index arithmetic of the kernels).

The bounds, in units of u = 2^-24 (gamma_k = k u / (1 - k u), the error of a k-step fp32 recursive sum; a warp's
lane-strided fma chains joined by a butterfly are such a sum over the same terms in another order):
  H_v       q^2 KK terms (the weight product rounded once) + 2q KO / OK terms, then the OO entry:
            gamma_(q^2 + 2q + 3) sum |A_v|^T |Binv| |A_v|.
  h_v, c_v  q^2 terms (weight product rounded once) + q terms: gamma_(q^2 + q + 3) sum |A_v|^T |Binv| |b_v| (|b_v|).
  mean      Y + R rounded once: u |Y + R|; Y or R alone is copied exactly.
  var       two p-term chains, 2 b and c added, times v0 in double, rounded to fp32:
            gamma_(p + 5) v0 (|x| . |YH| + 2 |x| . |h| + |c|).
  rows_dot  a cols-term chain times v0: gamma_(cols + 2) v0 sum |A| |B|.
  YH = xn H the P-long product on both sides of the planes switch: the tensor-core or SIMT constant of
            tests/edge_helpers.py, c |xn| |H| + the scale floor.
"""
import pytest
import torch

from edge_helpers import (DEV, NAN_BITS, U, am_terms, c_simt, c_tc, call, check_sentinel, gamma, grade, sentinel,
                          strided, stream)

pytestmark = pytest.mark.gpu

KIND_IDS = {"kr": 0, "object": 1, "view": 2}
# (p, q, nviews, kinds): q at 1, 4, 16 and 199 (one tile of Binv with the view table near the 160 KB limit); nviews = 1
# and nviews > q; every kind alone and together
CASES = [(4, 1, 3, ("kr", "object", "view")), (8, 4, 5, ("kr",)), (8, 4, 5, ("view", "object")),
         (12, 16, 16, ("object", "view", "kr")), (4, 16, 1, ("kr", "view")), (8, 3, 7, ("object",)), (4, 5, 6, ("view",)),
         (4, 199, 2, ("kr", "object", "view")), (128, 4, 6, ("kr", "object"))]


@pytest.fixture(scope="module", autouse=True)
def lib():
    from gppvae_b200 import _lib
    return _lib.load()


def _widths(kinds, p, q):
    return [p * q if k == "kr" else p if k == "object" else (q + 3) // 4 * 4 for k in kinds]


def _row_maps(wn, p, kinds):
    nv, q = wn.shape
    widths = _widths(kinds, p, q)
    w = wn.double()
    A = torch.zeros(nv, sum(widths), p, dtype=torch.float64, device=DEV)
    b = torch.zeros(nv, sum(widths), dtype=torch.float64, device=DEV)
    for kind, o, wd in zip(kinds, [sum(widths[:i]) for i in range(len(kinds))], widths):
        if kind == "kr":
            A[:, o:o + wd] = torch.einsum("vk,ji->vjki", w, torch.eye(p, dtype=torch.float64, device=DEV)).reshape(nv, wd, p)
        elif kind == "object":
            A[:, o:o + wd] = torch.eye(p, dtype=torch.float64, device=DEV)
        else:
            b[:, o:o + q] = w
    return A, b


def _binv(Qs, widths, kinds, q, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    B = torch.randn(Qs, Qs, generator=g, device=DEV) * 10.0 ** (torch.rand(Qs, 1, generator=g, device=DEV) * 2 - 1)
    o = 0
    for k, wd in zip(kinds, widths):       # the padding rows / columns of the view block hold NaN: they must not be read
        if k == "view" and wd > q:
            B[o + q:o + wd] = float("nan")
            B[:, o + q:o + wd] = float("nan")
        o += wd
    return B


def _views(lib, Bv, ldb, wn, p, kinds):
    nv, q = wn.shape
    has_h, has_w = ("kr" in kinds or "object" in kinds), "view" in kinds
    H, ldh = sentinel(p, nv * p) if has_h else (None, 0)
    h = torch.full((nv * p + 1,), NAN_BITS, dtype=torch.int32, device=DEV).view(torch.float32) if has_w else None
    c = torch.full((nv + 1,), NAN_BITS, dtype=torch.int32, device=DEV).view(torch.float32) if has_w else None
    from gppvae_b200 import _lib
    call(lib.gpp_kr_predict_views(Bv.data_ptr(), ldb, wn.data_ptr(), p, q, nv, len(kinds),
                                  _lib.host_i32([KIND_IDS[k] for k in kinds]), H.data_ptr() if has_h else None, ldh,
                                  h.data_ptr() if has_w else None, c.data_ptr() if has_w else None, stream()),
         "kr_predict_views")
    torch.cuda.synchronize()
    out = [check_sentinel(H, p, nv * p, "kr_predict_views H") if has_h else None, None, None]
    if has_w:
        assert h.view(torch.int32)[-1] == NAN_BITS and c.view(torch.int32)[-1] == NAN_BITS, "wrote past h / c"
        out[1], out[2] = h[:-1].view(nv, p), c[:-1]
    return out


@pytest.mark.parametrize("case", CASES, ids=lambda c: "p{}-q{}-nv{}-{}".format(c[0], c[1], c[2], "-".join(c[3])))
def test_kr_predict_views(lib, case):
    p, q, nv, kinds = case
    tag = "p{}-q{}-nv{}-{}".format(p, q, nv, "-".join(kinds))
    widths = _widths(kinds, p, q)
    Qs = sum(widths)
    B = _binv(Qs, widths, kinds, q, seed=p * 1000 + q)
    g = torch.Generator(device=DEV).manual_seed(q)
    wn = torch.randn(nv, q, generator=g, device=DEV)
    wn = wn / wn.norm(dim=1, keepdim=True)
    Bv, ldb = strided(B, 4)
    H, h, c = _views(lib, Bv, ldb, wn, p, kinds)
    A, b = _row_maps(wn, p, kinds)
    B64 = torch.nan_to_num(B.double(), nan=0.0)
    if H is not None:
        ref = torch.einsum("vai,ab,vbj->ivj", A, B64, A).reshape(p, nv * p)
        mag = torch.einsum("vai,ab,vbj->ivj", A.abs(), B64.abs(), A.abs()).reshape(p, nv * p)
        grade(f"kr_predict_views H {tag}", H, ref, mag, 1e-30, gamma(q * q + 2 * q + 3))
    if h is not None:
        grade(f"kr_predict_views h {tag}", h, torch.einsum("vai,ab,vb->vi", A, B64, b),
              torch.einsum("vai,ab,vb->vi", A.abs(), B64.abs(), b.abs()), 1e-30, gamma(q * q + q + 3))
        grade(f"kr_predict_views c {tag}", c, torch.einsum("va,ab,vb->v", b, B64, b),
              torch.einsum("va,ab,vb->v", b.abs(), B64.abs(), b.abs()), 1e-30, gamma(q * q + q + 3))
    again = _views(lib, Bv, ldb, wn, p, kinds)
    for x, y in zip(again, (H, h, c)):
        assert x is None or torch.equal(x.view(torch.int32), y.view(torch.int32)), "repeats must be bit-identical"


ROW_CASES = [(64, 8, 5, 12, "YR"), (300, 128, 16, 256, "Y"), (50, 4, 3, 4, "R"), (1000, 132, 9, 68, "YR")]


@pytest.mark.parametrize("case", ROW_CASES, ids=lambda c: "P{}-p{}-nv{}-L{}-{}".format(*c))
def test_kr_predict_rows(lib, case):
    P, p, nv, L, parts = case
    g = torch.Generator(device=DEV).manual_seed(P + p)
    m = 3 * P
    xn = torch.randn(P, p, generator=g, device=DEV)
    xn = xn / xn.norm(dim=1, keepdim=True)
    Y = torch.randn(P, nv * L, generator=g, device=DEV) * 10.0 ** (torch.rand(1, nv * L, generator=g, device=DEV) * 4 - 2)
    R = torch.randn(nv, L, generator=g, device=DEV)
    YH = torch.rand(P, nv * p, generator=g, device=DEV) * 10.0
    h = torch.randn(nv, p, generator=g, device=DEV)
    c = torch.rand(nv, generator=g, device=DEV) * 3.0
    d = torch.randint(0, P, (m,), generator=g, device=DEV)
    w = torch.randint(0, nv, (m,), generator=g, device=DEV)
    d[5], w[9], d[m - 1] = P, nv, -1                                  # out of table
    use_y, use_r = "Y" in parts, "R" in parts
    scal = torch.zeros(8, dtype=torch.float64, device=DEV)
    scal[0] = 0.37
    Yv, ldy = strided(Y, 8)
    Rv, ldr = strided(R, 4)
    YHv, ldyh = strided(YH, 12)
    mean, ldm = sentinel(m, L)
    var = torch.full((m + 1,), NAN_BITS, dtype=torch.int32, device=DEV).view(torch.float32)

    def run():
        call(lib.gpp_kr_predict_rows(Yv.data_ptr() if use_y else None, ldy, Rv.data_ptr() if use_r else None, ldr,
                                     YHv.data_ptr() if use_y else None, ldyh, xn.data_ptr(),
                                     h.data_ptr() if use_r else None, c.data_ptr() if use_r else None, d.data_ptr(),
                                     w.data_ptr(), m, P, p, nv, L, scal.data_ptr(), mean.data_ptr(), ldm, var.data_ptr(),
                                     stream()), "kr_predict_rows")
        torch.cuda.synchronize()
        assert var.view(torch.int32)[m] == NAN_BITS, "wrote past var"
        return check_sentinel(mean, m, L, "kr_predict_rows", allow_nan=True).clone(), var[:m].clone()
    mo, vo = run()
    bad = (d < 0) | (d >= P) | (w < 0) | (w >= nv)
    assert bool(torch.isnan(mo[bad]).all()) and bool(torch.isnan(vo[bad]).all())
    ok = ~bad
    dd, ww = d[ok], w[ok]
    ref = torch.zeros(int(ok.sum()), L, dtype=torch.float64, device=DEV)
    if use_y:
        ref += Y.double().view(P, nv, L)[dd, ww]
    if use_r:
        ref += R.double()[ww]
    tag = "P{}-p{}-nv{}-L{}-{}".format(*case)
    grade(f"kr_predict_rows mean {tag}", mo[ok], ref, ref.abs(), 0.0, U if (use_y and use_r) else 0.0)
    x = xn.double()[dd]
    vr = torch.zeros(ref.shape[0], dtype=torch.float64, device=DEV)
    vm = torch.zeros_like(vr)
    if use_y:
        yh = YH.double().view(P, nv, p)[dd, ww]
        vr += (x * yh).sum(1)
        vm += (x.abs() * yh.abs()).sum(1)
        if use_r:
            vr += 2 * (x * h.double()[ww]).sum(1)
            vm += 2 * (x.abs() * h.double().abs()[ww]).sum(1)
    if use_r:
        vr += c.double()[ww]
        vm += c.double()[ww].abs()
    grade(f"kr_predict_rows var {tag}", vo[ok], 0.37 * vr, 0.37 * vm, 1e-30, gamma(p + 5))
    mo2, vo2 = run()
    assert torch.equal(mo2.view(torch.int32), mo.view(torch.int32)) and torch.equal(vo2.view(torch.int32), vo.view(torch.int32))


@pytest.mark.parametrize("m,cols", [(1, 4), (700, 132), (70000, 576)])
def test_rows_dot(lib, m, cols):
    g = torch.Generator(device=DEV).manual_seed(cols)
    A = torch.randn(m, cols, generator=g, device=DEV) * 10.0 ** (torch.rand(1, cols, generator=g, device=DEV) * 4 - 2)
    B = torch.randn(m, cols, generator=g, device=DEV)
    Av, lda = strided(A, 4)
    Bv, ldb = strided(B, 8)
    scal = torch.zeros(8, dtype=torch.float64, device=DEV)
    scal[0] = 0.61
    out = torch.full((m + 1,), NAN_BITS, dtype=torch.int32, device=DEV).view(torch.float32)
    call(lib.gpp_rows_dot(Av.data_ptr(), lda, Bv.data_ptr(), ldb, m, cols, scal.data_ptr(), out.data_ptr(), stream()),
         "rows_dot")
    torch.cuda.synchronize()
    assert out.view(torch.int32)[m] == NAN_BITS
    ref = 0.61 * (A.double() * B.double()).sum(1)
    mag = 0.61 * (A.double().abs() * B.double().abs()).sum(1)
    grade(f"rows_dot m{m}-cols{cols}", out[:m], ref, mag, 1e-30, gamma(cols + 2))


@pytest.mark.parametrize("P", [500, 512, 600])
def test_yh_product_across_the_planes_switch(P):
    """YH = xn H (P x nviews p) as GP.predict forms it (GP._kr_y): the SIMT engine below P = 512, the planes form from it."""
    from gppvae_b200 import GP, ops
    from gppvae_b200.vmod import KhatriRao
    p, nv = 128, 5
    g = torch.Generator(device=DEV).manual_seed(P)
    xn = torch.randn(P, p, generator=g, device=DEV)
    xn = xn / xn.norm(dim=1, keepdim=True)
    wn = torch.randn(nv, 4, generator=g, device=DEV)
    wn = wn / wn.norm(dim=1, keepdim=True)
    d = torch.arange(P, device=DEV)
    kr = KhatriRao(xn, wn, d, d % nv)
    H = torch.randn(p, nv * p, generator=g, device=DEV) * 10.0 ** (torch.rand(1, nv * p, generator=g, device=DEV) * 2 - 1)
    YH = GP._kr_y(kr, H)
    ref, mag, floor = am_terms(xn, H)
    planes = ops.planes_supported(P, p, 0)
    assert planes == (P >= 512)
    grade(f"YH = xn H P={P} ({'planes' if planes else 'simt'})", YH, ref, mag, floor, c_tc(p) if planes else c_simt(p))
