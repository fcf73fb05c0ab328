"""The entries of the structured Khatri-Rao route (csrc/structured.cu, the slot-sum planes of csrc/gemm_planes.cu and
vmod.KhatriRao.st) against float64, element by element, with the conventions of test_gpu_kernel_edges.py: a bound
derived per operation (never fitted), sentinel output buffers (one extra row, ld = cols + 8, a NaN bit pattern that
must survive), inputs with ld > cols whose gap holds NaN, and the worst bound ratio printed per case.

Every case builds its own rows (d, w) from a seed, with one of three occupancies of the (object, view) slots:
  uniform   d, w uniform over the tables;
  skewed    one slot holds 10 % of the rows, about 90 % of the slots are empty, some slots hold exactly one row;
  oob       uniform, plus a few rows whose d or w lies outside its table (they belong to no slot: NaN rows of Xb).

The bounds, in units of u = 2^-24 (gamma_k = k u / (1 - k u) is the error of a k-step fp32 recursive sum):
  slot sums         a slot's rows are added one after the other in fp32 from 0: gamma_(cnt-1) sum|x|; cnt xn is one
                    rounding, u |cnt xn|; an empty slot is exactly zero.
  ST = xn^T XZ      the P-long product of test_gpu_kernel_edges.py (c_tc(P) or c_simt(P) times |xn|^T |XZ|), whose
                    scale floor 2^-31 (max|A| ||B_j||_1 + max|B_range| ||A_i||_1) is taken PER COLUMN RANGE, as the
                    dense pass 1 gets it for G and C from the separate planes and scales of V and X: the cnt (x) xn
                    range against max|cnt (x) xn|, the slot-sum range against max_count max|X|, the bound its scale is
                    taken from (a slot sum that cancels can lie far below it; only a scan of the sums, a second read
                    of X, would find their maximum).  The slot sums' own error passes through |xn|^T.
  assembly          GC = sum over views of (row weight)(column weight)(base): one rounding of the weight product and
                    an fma chain of nviews terms, (nviews + 2) u sum_v |w_r w_c| |base|;  M and R: (q + 2) u.
  view sums         a row passes through at most (rows of its chunk) + (chunks) fp32 additions: gamma_(n_v + nchunks);
                    a_v likewise with P objects; n_v exact.
  row epilogues     Xb = (X - (Y + R)) * fp32(1/vn): 5 u (|X| + |Y| + |R|) / vn; nll, scal[XB2], scal[QUAD] as
                    test_xb_nll_entries.
The file fails (does not skip) when the library was not built with the tensor-core engine.
"""
import pytest
import torch

from conftest import rel_err
from edge_helpers import (DEV, FLOOR, NAN_BITS, U, atb_terms, c_simt, c_tc, call, check_sentinel, gamma, grade,
                          nan_vector, ratio_of, sentinel, spread_cols, strided, stream, workspace)

pytestmark = pytest.mark.gpu

KINDS = ("kr", "object", "view")


@pytest.fixture(scope="module", autouse=True)
def lib():
    from gppvae_b200 import _lib
    engine = _lib.gemm_engine()
    assert engine == "tcgen05-3xf16", f"this file checks the tensor-core paths; the library was built with {engine}"
    return _lib.load()


# ----------------------------------------------------------------------------------------------------------- helpers
def rows_of(n, P, nviews, pattern, seed):
    """(d, w) of n rows over P objects and nviews views with the given slot occupancy (see the module docstring)."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    d = torch.randint(0, P, (n,), generator=g, device=DEV)
    w = torch.randint(0, nviews, (n,), generator=g, device=DEV)
    if pattern == "skewed":
        nslots = P * nviews
        active = torch.randperm(nslots, generator=g, device=DEV)[: max(3, nslots // 10)]
        hot = n // 10
        nsingle = min((active.numel() - 1) // 2, (n - hot) // 4)
        rest = active[1 + nsingle:]
        slot = torch.empty(n, dtype=torch.int64, device=DEV)
        slot[:hot] = active[0]
        slot[hot:hot + nsingle] = active[1:1 + nsingle]
        slot[hot + nsingle:] = rest[torch.randint(0, rest.numel(), (n - hot - nsingle,), generator=g, device=DEV)]
        slot = slot[torch.randperm(n, generator=g, device=DEV)]
        d, w = slot // nviews, slot % nviews
    elif pattern == "oob":
        bad = torch.arange(0, n, 53, device=DEV)
        kind = torch.arange(bad.numel(), device=DEV) % 4
        d[bad] = torch.where(kind == 0, P, torch.where(kind == 1, -1, d[bad]))
        w[bad] = torch.where(kind == 2, nviews, torch.where(kind == 3, -3, w[bad]))
    return d.contiguous(), w.contiguous()


def valid(d, w, P, nviews):
    return (d >= 0) & (d < P) & (w >= 0) & (w < nviews)


def unit_rows(P, p, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    x = torch.randn(P, p, generator=g, device=DEV)
    return (x / x.norm(dim=1, keepdim=True)).contiguous()


def view_table(nviews, q, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return (torch.randn(nviews, q, generator=g, device=DEV) + 0.5).contiguous()


def slot_index(xn, wn, d, w):
    """(order, slot_start, max_count) as the route prepares them (vmod.KhatriRao.index)."""
    from gppvae_b200.vmod import KhatriRao
    kr = KhatriRao(xn, wn, d, w)
    order, slot_start = kr.index()
    return order, slot_start, kr.max_count()


def slot_ref(X0, d, w, P, nviews):
    """fp64 slot sums Zs (P x nviews L), slot sums of |X| and the counts (P x nviews) of the valid rows."""
    ok = valid(d, w, P, nviews)
    key = (d * nviews + w)[ok]
    L = X0.shape[1]
    X64 = X0.double()[ok]
    Zs = torch.zeros(P * nviews, L, dtype=torch.float64, device=DEV).index_add_(0, key, X64)
    Za = torch.zeros(P * nviews, L, dtype=torch.float64, device=DEV).index_add_(0, key, X64.abs())
    cnt = torch.bincount(key, minlength=P * nviews).double()
    return Zs.view(P, nviews * L), Za.view(P, nviews * L), cnt.view(P, nviews)


def cnt_x(cnt, xn):
    P, nviews = cnt.shape
    return (cnt[:, :, None] * xn.double()[:, None, :]).reshape(P, -1)


def gamma_t(k):
    """gamma_k elementwise for a tensor of step counts (k <= 0: exact)."""
    k = k.clamp(min=0)
    return k * U / (1.0 - k * U)


def round4(c):
    return (c + 3) // 4 * 4


def widths_of(kinds, p, q):
    return [p * q if k == "kr" else p if k == "object" else round4(q) for k in kinds]


def design_maps(kinds, wn64, p):
    """E (nviews x (p + 1) x Q): column t of the stacked design in view v is E[v, a, t] times object feature a (a = p:
    the constant 1).  KR (j, k) -> wn[v, k] e_j,  O j -> e_j,  W k -> wn[v, k] 1,  W padding -> 0."""
    nv, q = wn64.shape
    widths = widths_of(kinds, p, q)
    E = torch.zeros(nv, p + 1, sum(widths), dtype=torch.float64, device=DEV)
    off = 0
    for k, wd in zip(kinds, widths):
        if k == "kr":
            j = torch.arange(p, device=DEV).repeat_interleave(q)
            kk = torch.arange(q, device=DEV).repeat(p)
            E[:, j, off + torch.arange(p * q, device=DEV)] = wn64[:, kk]
        elif k == "object":
            E[:, torch.arange(p, device=DEV), off + torch.arange(p, device=DEV)] = 1.0
        else:
            E[:, p, off:off + q] = wn64
        off += wd
    return E, widths


def effects_ref(kinds, ST, VM, wn, p, L, with_g):
    """fp64 GC (with_g) or C of the stacked designs from ST (p x nviews ((with_g ? p : 0) + L)) and VM (nviews rows
    [z_v | a_v | n_v]); the same formula with |.| everywhere is the magnitude of the assembly's sums."""
    nv = wn.shape[0]
    E, _ = design_maps(kinds, wn.double(), p)
    Sx = torch.zeros(nv, p + 1, p + 1, dtype=torch.float64, device=DEV)
    Tx = torch.zeros(nv, p + 1, L, dtype=torch.float64, device=DEV)
    zcol0 = nv * p if with_g else 0
    if ST is not None:
        S = ST.double()
        if with_g:
            Sx[:, :p, :p] = S[:, :nv * p].reshape(p, nv, p).permute(1, 0, 2)
        Tx[:, :p, :] = S[:, zcol0:zcol0 + nv * L].reshape(p, nv, L).permute(1, 0, 2)
    if VM is not None:
        M = VM.double()
        Tx[:, p, :] = M[:, :L]
        if with_g:
            Sx[:, :p, p] = M[:, L:L + p]
            Sx[:, p, :p] = M[:, L:L + p]
            Sx[:, p, p] = M[:, L + p]
    C = torch.einsum("vat,val->tl", E, Tx)
    if not with_g:
        return C
    G = torch.einsum("vat,vab,vbs->ts", E, Sx, E)
    return torch.cat([G, C], 1)


def _scal(v0=0.7, vn=0.3, rowconst=-1.25):
    from gppvae_b200._lib import NSCAL, S_ROWCONST, S_V0, S_VN
    s = torch.zeros(NSCAL, dtype=torch.float64, device=DEV)
    s[S_V0], s[S_VN], s[S_ROWCONST] = v0, vn, rowconst
    return s


# ------------------------------------------------------------------------------------- A. slot sums, fp32 form
# (P, nviews, p, L): L and p in {4, 124, 128, 132, 260} (across the 128-column lane loop), P nviews not a multiple of 8
A_SHAPES = [(37, 3, 4, 4), (101, 5, 124, 132), (203, 7, 128, 260), (77, 9, 132, 128), (51, 3, 260, 124),
            (45, 7, 4, 260), (1001, 3, 128, 4)]


@pytest.mark.parametrize("pattern", ["uniform", "skewed", "oob"])
@pytest.mark.parametrize("shape", A_SHAPES, ids=lambda s: "P{}-nv{}-p{}-L{}".format(*s))
def test_kr_slot_sums(lib, shape, pattern):
    """gpp_kr_slot_sums: the slot sums within gamma_(cnt-1) sum|x|, cnt xn within u, empty slots exactly zero, nothing
    written outside the P x cols block, and two calls bit-identical."""
    P, nviews, p, L = shape
    n = 20000
    seed = P * 31 + p + L
    d, w = rows_of(n, P, nviews, pattern, seed)
    xn, wn = unit_rows(P, p, seed + 1), view_table(nviews, 3, seed + 2)
    X0 = spread_cols(n, L, seed + 3, positive=False)
    X, ldx = strided(X0, 4)
    order, slot_start, _ = slot_index(xn, wn, d, w)
    Zs, Za, cnt = slot_ref(X0, d, w, P, nviews)
    cntL = cnt.repeat_interleave(L, 1)
    for with_x in (0, 1):
        cols = nviews * ((p if with_x else 0) + L)
        zcol0 = nviews * p if with_x else 0
        outs = []
        for _ in range(2):
            XZ, ld = sentinel(P, cols)
            call(lib.gpp_kr_slot_sums(X.data_ptr(), ldx, order.data_ptr(), slot_start.data_ptr(), xn.data_ptr(), P, p,
                                      nviews, L, with_x, XZ.data_ptr(), ld, stream()), "kr_slot_sums")
            outs.append(XZ)
        torch.cuda.synchronize()
        tag = f"kr_slot_sums P={P} nviews={nviews} p={p} L={L} {pattern} with_x={with_x}"
        assert torch.equal(outs[0].view(torch.int32), outs[1].view(torch.int32)), f"{tag}: two calls differ"
        out = check_sentinel(outs[0], P, cols, tag)
        Z = out[:, zcol0:]
        assert bool((Z[cntL == 0] == 0).all()), f"{tag}: an empty slot has a non-zero sum"
        r = ratio_of((Z.double() - Zs).abs(), gamma_t(cntL - 1) * Za)
        msg = f"slot sums {r:.3f}"
        assert r <= 1.0, f"{tag}: slot sums {r:.3g} x the bound"
        if with_x:
            R = cnt_x(cnt, xn)
            S = out[:, :zcol0]
            assert bool((S[cnt.repeat_interleave(p, 1) == 0] == 0).all()), f"{tag}: cnt (x) xn of an empty slot"
            rs = ratio_of((S.double() - R).abs(), U * R.abs())
            msg += f"  cnt (x) xn {rs:.3f}"
            assert rs <= 1.0, f"{tag}: cnt (x) xn {rs:.3g} x the bound"
        print(f"[{tag}] worst bound ratio {msg}  (largest slot {int(cnt.max())} rows)")


# ------------------------------------------------------------- B. the P-long product as the route runs it: st()
B_SHAPES = [(511, 132), (512, 128), (513, 124), (513, 132), (640, 128)]       # (P, p); planes from P >= 512, p >= 128
B_SCALES = [1e-4, 1e-2, 1.0, 1e3, "spread"]


def _st_engine(P, p):
    return "tc" if P >= 512 and p >= 128 else "simt"


def _st_terms(xn, X0, d, w, nviews, with_x):
    """fp64 ST = xn^T [cnt (x) xn | Zs], the bound of the P-long product with the floor per column range, plus the
    slot sums' own error carried through |xn|^T."""
    P, p = xn.shape
    Zs, Za, cnt = slot_ref(X0, d, w, P, nviews)
    L = X0.shape[1]
    zmax = float(cnt.max()) * float(X0.abs().max())       # the scale bound of the slot-sum range
    EZ = gamma_t(cnt.repeat_interleave(L, 1) - 1) * Za
    if with_x:
        CX = cnt_x(cnt, xn)
        B = torch.cat([CX, Zs], 1)
        EB = torch.cat([U * CX.abs(), EZ], 1)
        maxB = torch.cat([torch.full((CX.shape[1],), float(CX.abs().max()), dtype=torch.float64, device=DEV),
                          torch.full((Zs.shape[1],), zmax, dtype=torch.float64, device=DEV)])
    else:
        B, EB = Zs, EZ
        maxB = torch.full((Zs.shape[1],), zmax, dtype=torch.float64, device=DEV)
    R, mag, floor = atb_terms(xn, B, maxB)
    c = c_tc(P) if _st_engine(P, p) == "tc" else c_simt(P)
    return R, mag, floor + xn.double().abs().t() @ EB, c


def _z_input(n, L, scale, seed):
    if scale == "spread":
        return spread_cols(n, L, seed, positive=True)
    g = torch.Generator(device=DEV).manual_seed(seed)
    return torch.randn(n, L, generator=g, device=DEV) * scale


@pytest.mark.parametrize("pattern", ["uniform", "skewed"])
@pytest.mark.parametrize("scale", B_SCALES, ids=lambda s: f"Z{s}" if s == "spread" else f"Zx{s:g}")
@pytest.mark.parametrize("shape", B_SHAPES, ids=lambda s: f"P{s[0]}-p{s[1]}-{_st_engine(*s)}")
def test_kr_st_per_range_floor(lib, shape, scale, pattern):
    """KhatriRao.st() on both sides of the planes switch: ST = xn^T [cnt (x) xn | Zs] against fp64, with_x 0 and 1.
    The S range (which becomes G) must meet the floor of max|cnt (x) xn| and the T range (which becomes C) that of
    its own scale bound, whatever the magnitude of Z and however crowded one slot is."""
    from gppvae_b200.vmod import KhatriRao
    P, p = shape
    n, nviews, L, q = 30000, 6, 64, 4
    seed = P + 7 * p
    d, w = rows_of(n, P, nviews, pattern, seed)
    xn, wn = unit_rows(P, p, seed + 1), view_table(nviews, q, seed + 2)
    X0 = _z_input(n, L, scale, seed + 3)
    X, ldx = strided(X0, 4)
    kr = KhatriRao(xn, wn, d, w)
    for with_x in (False, True):
        ST = kr.st(X, ldx, L, with_x)
        torch.cuda.synchronize()
        R, mag, floor, c = _st_terms(xn, X0, d, w, nviews, with_x)
        tag = (f"st P={P} p={p} Z={scale} {pattern} with_x={int(with_x)} {_st_engine(P, p)}"
               f" (largest slot {kr.max_count()})")
        if with_x:
            s = nviews * p
            rs = ratio_of((ST[:, :s].double() - R[:, :s]).abs(), c * mag[:, :s] + floor[:, :s])
            rt = ratio_of((ST[:, s:].double() - R[:, s:]).abs(), c * mag[:, s:] + floor[:, s:])
            print(f"[{tag}] worst bound ratio S range {rs:.3f}  T range {rt:.3f}")
        grade(tag, ST, R, mag, floor, c)


@pytest.mark.parametrize("pattern,scale", [("uniform", 1.0), ("skewed", 1e-3), ("uniform", 1e3)])
def test_kr_route_gc_against_dense_pass1(lib, pattern, scale):
    """The structured GC (st() then gpp_kr_assemble_gc) and the dense pass 1 (gpp_gram_vtz_planes on the materialised V)
    against the same fp64 V^T [V | X].  The structured route replaces pass 1 and owes its accuracy: its bound is the
    st() bound carried through the assembly weights, plus the assembly's own (nviews + 2) u, plus 2 u |V|^T |V| for the
    one rounding of every element of the materialised fp32 V."""
    from gppvae_b200 import ops
    from gppvae_b200.vmod import KhatriRao
    n, P, p, q, nviews, L = 30000, 640, 128, 4, 6, 64
    Q = p * q
    seed = 101
    d, w = rows_of(n, P, nviews, pattern, seed)
    xn, wn = unit_rows(P, p, seed + 1), view_table(nviews, q, seed + 2)
    X0 = _z_input(n, L, scale, seed + 3)
    kr = KhatriRao(xn, wn, d, w)
    GC_s = ops.kr_assemble_gc(kr.st(X0, L, L, True), wn, p, L, True)
    V = kr.dense()
    pV, pX = ops.split_planes(V, Q, n, Q, colsq=True), ops.split_planes(X0, L, n, L)
    GC_d = ops.gram_vtz_planes(pV, pX, n, Q, L)
    torch.cuda.synchronize()
    V64, X64 = V.double(), X0.double()
    B = torch.cat([V64, X64], 1)
    R = V64.t() @ B
    magd = V64.abs().t() @ B.abs()
    maxB = torch.cat([torch.full((Q,), float(V64.abs().max()), dtype=torch.float64, device=DEV),
                      torch.full((L,), float(X64.abs().max()), dtype=torch.float64, device=DEV)])
    floord = FLOOR * (V64.abs().max() * B.abs().sum(0)[None, :] + maxB[None, :] * V64.abs().sum(0)[:, None])
    rd = grade(f"dense gram_vtz_planes n={n} Q={Q} L={L} {pattern} Z x{scale:g}", GC_d, R, magd, floord, c_tc(n))
    # the structured bound: E_ST through |w_r w_c|, the assembly over |ST|, and the representation of V in fp32
    Rst, mag, floor, c = _st_terms(xn, X0, d, w, nviews, True)
    EST = c * mag + floor
    lim = (effects_ref(["kr"], EST, None, wn.abs(), p, L, True)
           + (nviews + 2) * U * effects_ref(["kr"], Rst.abs(), None, wn.abs(), p, L, True) + 2 * U * magd)
    r = ratio_of((GC_s.double() - R).abs(), lim)
    print(f"[structured GC n={n} Q={Q} L={L} {pattern} Z x{scale:g}] worst bound ratio {r:.3f} (dense pass 1 {rd:.3f})")
    assert bool(torch.isfinite(GC_s).all()) and r <= 1.0, f"structured GC: {r:.3g} x the composed bound"


# ----------------------------------------------------------------------------------------------- C. assembly
def _subsets():
    import itertools
    return [list(c) for k in (1, 2, 3) for c in itertools.permutations(KINDS, k)]


def _kinds_host(kinds):
    from gppvae_b200 import _lib
    from gppvae_b200.ops import EFFECT_KINDS
    return _lib.host_i32([EFFECT_KINDS[k] for k in kinds])


@pytest.mark.parametrize("q", [1, 3, 4, 5, 9, 17])
def test_kr_assembly_entries(lib, q):
    """gpp_kr_assemble_gc, gpp_kr_assemble_m and, for all 15 ordered non-empty subsets of {KR, OBJECT, VIEW},
    gpp_kr_assemble_gc_blocks and gpp_kr_assemble_m_blocks against fp64 of the same fp32 inputs; the padding rows and
    columns of the VIEW block bit-exact zeros; NULL ST without KR and OBJECT, NULL VM without VIEW; the VIEW-only
    m_blocks launch (p = 0 inside, the R blocks start at block 0)."""
    p, L = 8, 8
    nvs = sorted({1, q - 1, 3 * q} - {0})
    for nviews in nvs:
        seed = 1000 * q + nviews
        wn = view_table(nviews, q, seed)
        aw = wn.double().abs()
        for with_g in (0, 1):
            cst = nviews * ((p if with_g else 0) + L)
            ST0 = spread_cols(p, cst, seed + 1, positive=False)
            vmw = L + (p + 4 if with_g else 0)
            VM0 = spread_cols(nviews, vmw, seed + 2, positive=False)
            if with_g:
                VM0[:, L + p] = torch.randint(0, 1000, (nviews,), device=DEV).float()
                VM0[:, L + p + 1:] = 0
            ST, ldst = strided(ST0, 4)
            VM, ldvm = strided(VM0, 4)
            worst = 0.0
            for kinds in _subsets():
                has_st = "kr" in kinds or "object" in kinds
                has_vm = "view" in kinds
                widths = widths_of(kinds, p, q)
                Q = sum(widths)
                cols = (Q if with_g else 0) + L
                tag = f"assemble_gc_blocks {kinds} q={q} nviews={nviews} with_g={with_g}"
                GC, ldgc = sentinel(Q, cols)
                call(lib.gpp_kr_assemble_gc_blocks(ST.data_ptr() if has_st else None, ldst if has_st else 0,
                                                   VM.data_ptr() if has_vm else None, ldvm if has_vm else 0,
                                                   wn.data_ptr(), p, q, nviews, L, len(kinds), _kinds_host(kinds),
                                                   with_g, GC.data_ptr(), ldgc, stream()), "kr_assemble_gc_blocks")
                GC = check_sentinel(GC, Q, cols, tag)
                R = effects_ref(kinds, ST0 if has_st else None, VM0 if has_vm else None, wn, p, L, with_g)
                mag = effects_ref(kinds, ST0.abs() if has_st else None, VM0.abs() if has_vm else None, wn.abs(), p, L,
                                  with_g)
                r = ratio_of((GC.double() - R).abs(), (nviews + 2) * U * mag)
                assert r <= 1.0, f"{tag}: {r:.3g} x the bound"
                worst = max(worst, r)
                if "view" in kinds and round4(q) > q:                     # padding of the VIEW block: +0.0 exactly
                    b = kinds.index("view")
                    off = sum(widths[:b])
                    pad = torch.arange(off + q, off + round4(q), device=DEV)
                    bits = GC.contiguous().view(torch.int32)
                    assert bool((bits[pad] == 0).all()), f"{tag}: padding rows not exactly zero"
                    if with_g:
                        assert bool((bits[:, pad] == 0).all()), f"{tag}: padding columns not exactly zero"
                if kinds == ["kr"]:                                       # the one-design entry, same inputs
                    GC1, ld1 = sentinel(Q, cols)
                    call(lib.gpp_kr_assemble_gc(ST.data_ptr(), ldst, wn.data_ptr(), p, q, nviews, L, with_g,
                                                GC1.data_ptr(), ld1, stream()), "kr_assemble_gc")
                    GC1 = check_sentinel(GC1, Q, cols, "kr_assemble_gc")
                    r1 = ratio_of((GC1.double() - R).abs(), (nviews + 2) * U * mag)
                    assert r1 <= 1.0, f"kr_assemble_gc q={q} nviews={nviews} with_g={with_g}: {r1:.3g} x the bound"
                    worst = max(worst, r1)
                if with_g:
                    continue
                # M and R from a W of the stacked width, rows in the block order
                W0 = spread_cols(Q, L, seed + 3 + len(kinds), positive=False)
                W, ldw = strided(W0, 4)
                need_m, need_r = has_st, has_vm
                M, ldm = sentinel(p, nviews * L)
                Rv, ldr = sentinel(nviews, L)
                call(lib.gpp_kr_assemble_m_blocks(W.data_ptr(), ldw, wn.data_ptr(), p, q, nviews, L, len(kinds),
                                                  _kinds_host(kinds), M.data_ptr() if need_m else None,
                                                  ldm if need_m else 0, Rv.data_ptr() if need_r else None,
                                                  ldr if need_r else 0, stream()), "kr_assemble_m_blocks")
                tagm = f"assemble_m_blocks {kinds} q={q} nviews={nviews}"
                offs = {k: sum(widths[:i]) for i, k in enumerate(kinds)}
                W64 = W0.double()
                wn64 = wn.double()
                if need_m:
                    Mr = torch.zeros(p, nviews, L, dtype=torch.float64, device=DEV)
                    Mm = torch.zeros_like(Mr)
                    if "kr" in kinds:
                        WK = W64[offs["kr"]:offs["kr"] + p * q].reshape(p, q, L)
                        Mr += torch.einsum("vk,jkl->jvl", wn64, WK)
                        Mm += torch.einsum("vk,jkl->jvl", aw, WK.abs())
                    if "object" in kinds:
                        WO = W64[offs["object"]:offs["object"] + p]
                        Mr += WO[:, None, :]
                        Mm += WO.abs()[:, None, :]
                    Mo = check_sentinel(M, p, nviews * L, tagm + " M")
                    rm = ratio_of((Mo.double() - Mr.reshape(p, -1)).abs(), (q + 2) * U * Mm.reshape(p, -1))
                    assert rm <= 1.0, f"{tagm}: M {rm:.3g} x the bound"
                    worst = max(worst, rm)
                else:
                    assert bool((M.view(torch.int32) == NAN_BITS).all()), f"{tagm}: wrote M without KR or OBJECT"
                if need_r:
                    WW = W64[offs["view"]:offs["view"] + q]
                    Ro = check_sentinel(Rv, nviews, L, tagm + " R")
                    rr = ratio_of((Ro.double() - wn64 @ WW).abs(), (q + 2) * U * (aw @ WW.abs()))
                    assert rr <= 1.0, f"{tagm}: R {rr:.3g} x the bound"
                    worst = max(worst, rr)
                else:
                    assert bool((Rv.view(torch.int32) == NAN_BITS).all()), f"{tagm}: wrote R without VIEW"
                if kinds == ["kr"]:
                    M1, ld1 = sentinel(p, nviews * L)
                    call(lib.gpp_kr_assemble_m(W.data_ptr(), ldw, wn.data_ptr(), p, q, nviews, L, M1.data_ptr(), ld1,
                                               stream()), "kr_assemble_m")
                    M1 = check_sentinel(M1, p, nviews * L, "kr_assemble_m")
                    WK = W64[: p * q].reshape(p, q, L)
                    r1 = ratio_of((M1.double() - torch.einsum("vk,jkl->jvl", wn64, WK).reshape(p, -1)).abs(),
                                  (q + 2) * U * torch.einsum("vk,jkl->jvl", aw, WK.abs()).reshape(p, -1))
                    assert r1 <= 1.0, f"kr_assemble_m q={q} nviews={nviews}: {r1:.3g} x the bound"
                    worst = max(worst, r1)
            torch.cuda.synchronize()
            print(f"[assembly q={q} nviews={nviews} with_g={with_g}, 15 kind lists] worst bound ratio {worst:.3f}")


# ---------------------------------------------------------------------------------------------- D. view sums
# (nviews, P, p, L, with_x, pattern): one chunk from nviews >= 1184; p > L and L > p; L = 1028 and p = 1028 reach the
# 256-thread cap of the partial kernel
D_CASES = [(1, 1, 4, 8, 1, "uniform"), (1, 5000, 8, 4, 1, "skewed"), (9, 37, 132, 4, 1, "uniform"),
           (9, 1183, 4, 260, 1, "oob"), (9, 1185, 128, 1028, 1, "uniform"), (9, 5000, 1028, 8, 1, "uniform"),
           (1184, 1, 4, 12, 1, "uniform"), (1184, 37, 8, 4, 0, "skewed"), (1500, 37, 4, 8, 1, "oob"),
           (1500, 1185, 260, 4, 1, "uniform"), (1, 1185, 4, 1028, 0, "uniform")]


def _view_sums(lib, X, ldx, order, slot_start, xn, P, p, nviews, L, with_x):
    width = L + (p + 4 if with_x else 0)
    VM, ld = sentinel(nviews, width)
    ws = workspace(lib.gpp_kr_view_sums_workspace_bytes(P, p, nviews, L, with_x))
    call(lib.gpp_kr_view_sums(X.data_ptr(), ldx, order.data_ptr(), slot_start.data_ptr(), xn.data_ptr(), P, p, nviews,
                              L, with_x, VM.data_ptr(), ld, ws.data_ptr(), ws.numel(), stream()), "kr_view_sums")
    return VM, width


def _view_sums_check(tag, VM, width, X0, xn, d, w, P, nviews, L, with_x):
    """z_v, a_v within their summation bounds, n_v exact, the three trailing entries exactly zero; returns the ratios."""
    p = xn.shape[1]
    out = check_sentinel(VM, nviews, width, tag)
    ok = valid(d, w, P, nviews)
    X64 = X0.double()[ok]
    wv = w[ok]
    z = torch.zeros(nviews, L, dtype=torch.float64, device=DEV).index_add_(0, wv, X64)
    za = torch.zeros(nviews, L, dtype=torch.float64, device=DEV).index_add_(0, wv, X64.abs())
    nv = torch.bincount(wv, minlength=nviews).double()
    nch = min(-(-1184 // nviews), P)
    rz = ratio_of((out[:, :L].double() - z).abs(), gamma_t(nv[:, None] + nch) * za)
    assert rz <= 1.0, f"{tag}: z_v {rz:.3g} x the bound"
    if not with_x:
        return f"z_v {rz:.3f}"
    cnt = slot_ref(X0[:, :4], d, w, P, nviews)[2]                 # P x nviews
    a = cnt.t() @ xn.double()
    aa = cnt.t() @ xn.double().abs()
    ra = ratio_of((out[:, L:L + p].double() - a).abs(), gamma(P + nch) * aa)
    assert ra <= 1.0, f"{tag}: a_v {ra:.3g} x the bound"
    assert torch.equal(out[:, L + p].double(), nv), f"{tag}: n_v is not the exact count"
    assert bool((out[:, L + p + 1:].contiguous().view(torch.int32) == 0).all()), f"{tag}: VM[v, L+p+1 .. L+p+4) not zero"
    return f"z_v {rz:.3f}  a_v {ra:.3f}"


@pytest.mark.parametrize("case", D_CASES, ids=lambda c: "nv{}-P{}-p{}-L{}-x{}-{}".format(*c))
def test_kr_view_sums(lib, case):
    """gpp_kr_view_sums: one chunk (nviews >= 1184) and many, ragged chunks; z_v and a_v within their bounds, n_v exact,
    the padding of the row exactly zero, nothing written outside the nviews x width block; two calls bit-identical."""
    nviews, P, p, L, with_x, pattern = case
    n = 20000
    seed = 7 * nviews + P + p + L
    d, w = rows_of(n, P, nviews, pattern, seed)
    xn, wn = unit_rows(P, p, seed + 1), view_table(nviews, 2, seed + 2)
    X0 = spread_cols(n, L, seed + 3, positive=False)
    X, ldx = strided(X0, 8)
    order, slot_start, _ = slot_index(xn, wn, d, w)
    VM1, width = _view_sums(lib, X, ldx, order, slot_start, xn, P, p, nviews, L, with_x)
    VM2, _ = _view_sums(lib, X, ldx, order, slot_start, xn, P, p, nviews, L, with_x)
    torch.cuda.synchronize()
    tag = f"kr_view_sums nviews={nviews} P={P} p={p} L={L} with_x={with_x} {pattern}"
    assert torch.equal(VM1.view(torch.int32), VM2.view(torch.int32)), f"{tag}: two calls differ"
    print(f"[{tag}] worst bound ratio {_view_sums_check(tag, VM1, width, X0, xn, d, w, P, nviews, L, with_x)}")


def test_kr_view_sums_2_pow_24_rows_in_one_view(lib):
    """2^24 rows in one view (L = 4, 268 MB of X): n_v = 2^24 exactly, as the header promises, and with X = 1 the sum
    z_v = 2^24 exactly too (every partial sum is an integer <= 2^24)."""
    n, P, p, L = 1 << 24, 1000, 4, 4
    d = (torch.arange(n, device=DEV) % P).contiguous()
    w = torch.zeros(n, dtype=torch.int64, device=DEV)
    xn, wn = unit_rows(P, p, 5), view_table(1, 2, 6)
    X0 = torch.ones(n, L, device=DEV)
    order, slot_start, _ = slot_index(xn, wn, d, w)
    VM, width = _view_sums(lib, X0, L, order, slot_start, xn, P, p, 1, L, 1)
    torch.cuda.synchronize()
    out = check_sentinel(VM, 1, width, "kr_view_sums 2^24 rows")
    assert float(out[0, L + p]) == float(n), f"n_v = {float(out[0, L + p])}, not 2^24"
    assert bool((out[0, :L] == float(n)).all()), f"z_v = {out[0, :L].tolist()}, not 2^24"
    cnt = torch.full((P,), float(n // P), dtype=torch.float64, device=DEV)
    cnt[: n % P] += 1
    a, aa = cnt @ xn.double(), cnt @ xn.double().abs()
    r = ratio_of((out[0, L:L + p].double() - a).abs(), gamma(P + P) * aa)
    print(f"[kr_view_sums 2^24 rows in one view] n_v and z_v exact; a_v worst bound ratio {r:.3f}")
    assert r <= 1.0


# -------------------------------------------------------------------------------------------- E. row epilogues
# (n, L, P, nviews, pattern): n = 9473 > 1184 x 8 warps runs the grid-stride loop
E_CASES = [(1, 4, 3, 2, "uniform"), (7, 128, 5, 3, "oob"), (9473, 132, 300, 7, "uniform"), (9473, 4, 40, 9, "oob"),
           (20033, 260, 500, 5, "oob"), (20033, 128, 1000, 3, "uniform")]


@pytest.mark.parametrize("entry", ["kr_xb_nll", "kr_xb_nll_views"])
@pytest.mark.parametrize("case", E_CASES, ids=lambda c: "n{}-L{}-P{}-nv{}-{}".format(*c))
def test_kr_xb_nll_entries(lib, case, entry):
    """gpp_kr_xb_nll / gpp_kr_xb_nll_views with ldy > nviews L, ldr > L and ld gaps of NaN: Xb elementwise against fp64,
    the nll rows, scal[XB2] and scal[QUAD] within the bounds of test_xb_nll_entries.  Out-of-range rows give NaN rows of
    Xb and NaN nll, and NaN scal[XB2] / scal[QUAD], exactly where the dense route (gpp_khatri_rao_fwd's NaN rows of V
    through gpp_xb_nll) gives them."""
    from gppvae_b200 import ops
    from gppvae_b200._lib import S_QUAD, S_ROWCONST, S_VN, S_XB2
    n, L, P, nviews, pattern = case
    seed = n + 3 * L + P
    d, w = rows_of(n, P, nviews, pattern, seed)
    X0 = spread_cols(n, L, seed + 1, positive=False)
    Y0 = spread_cols(P, nviews * L, seed + 2, positive=False)
    R0 = spread_cols(nviews, L, seed + 3, positive=False) if entry.endswith("views") else None
    X, ldx = strided(X0, 4)
    Y, ldy = strided(Y0, 8)
    scal = _scal()
    vn, rowconst = float(scal[S_VN]), float(scal[S_ROWCONST])
    Xb, ldxb = sentinel(n, L)
    nll = nan_vector(n)
    ws = workspace(lib.gpp_kr_xb_workspace_bytes(n))
    if R0 is None:
        st = lib.gpp_kr_xb_nll(X.data_ptr(), ldx, Y.data_ptr(), ldy, d.data_ptr(), w.data_ptr(), n, P, nviews, L,
                               scal.data_ptr(), Xb.data_ptr(), ldxb, nll.data_ptr(), ws.data_ptr(), ws.numel(), stream())
    else:
        Rm, ldr = strided(R0, 4)
        st = lib.gpp_kr_xb_nll_views(X.data_ptr(), ldx, Y.data_ptr(), ldy, Rm.data_ptr(), ldr, d.data_ptr(),
                                     w.data_ptr(), n, P, nviews, L, scal.data_ptr(), Xb.data_ptr(), ldxb, nll.data_ptr(),
                                     ws.data_ptr(), ws.numel(), stream())
    call(st, entry)
    torch.cuda.synchronize()
    tag = f"{entry} n={n} L={L} P={P} nviews={nviews} {pattern}"
    Xb = check_sentinel(Xb, n, L, tag, allow_nan=True)
    assert nll.view(torch.int32)[n] == NAN_BITS, f"{tag}: wrote nll past row {n}"
    ok = valid(d, w, P, nviews)
    assert bool(torch.isnan(Xb[~ok]).all()), f"{tag}: an out-of-range row of Xb is not NaN"
    assert bool(torch.isnan(nll[:n][~ok]).all()), f"{tag}: the nll of an out-of-range row is not NaN"
    dc, wc = d.clamp(0, P - 1), w.clamp(0, nviews - 1)
    Yg = Y0.double().view(P, nviews, L)[dc, wc]
    Rg = R0.double()[wc] if R0 is not None else torch.zeros_like(Yg)
    x = X0.double()
    Rx = ((x - Yg - Rg) / vn)[ok]
    E = 5 * U * (x.abs() + Yg.abs() + Rg.abs())[ok] / vn
    grade(tag + " Xb", Xb[ok], Rx, E, torch.zeros_like(E), 1.0)
    xo, xb = x[ok], Xb[ok].double()
    quad_ref = (xo * Rx).sum(1)
    nll_ref = 0.5 * quad_ref + rowconst
    nll_lim = 0.5 * ((xo.abs() * E).sum(1) + 136 * U * (xo * xb).abs().sum(1)) + U * (nll_ref.abs() + abs(rowconst))
    r_nll = ratio_of((nll[:n][ok].double() - nll_ref).abs(), nll_lim)
    assert r_nll <= 1.0, f"{tag}: nll {r_nll:.3g} x the bound"
    sc = scal.cpu().numpy()
    if bool(ok.all()):
        xb2_ref, q_ref = float((Rx * Rx).sum()), float(quad_ref.sum())
        xb2_lim = float((2 * Rx.abs() * E + E * E).sum() + 136 * U * (xb * xb).sum())
        q_lim = float((xo.abs() * E).sum() + 136 * U * (xo * xb).abs().sum())
        r_xb2, r_q = abs(sc[S_XB2] - xb2_ref) / xb2_lim, abs(sc[S_QUAD] - q_ref) / q_lim
        print(f"[{tag}] worst bound ratio nll {r_nll:.3f}  scal[XB2] {r_xb2:.3f}  scal[QUAD] {r_q:.3f}")
        assert r_xb2 <= 1.0 and r_q <= 1.0
        return
    # the dense route on the same indices: V from gpp_khatri_rao_fwd (NaN rows where an index is out of its table)
    p, q = 8, 4
    xn, wn = unit_rows(P, p, seed + 4), view_table(nviews, q, seed + 5)
    V = ops.khatri_rao_fwd(xn, wn, d, w)
    Wd = spread_cols(p * q, L, seed + 6, positive=False) * 1e-2
    scal_d = _scal()
    Xb_d, nll_d = ops.xb_nll(V, p * q, X, ldx, Wd, n, p * q, L, scal_d)
    torch.cuda.synchronize()
    sd = scal_d.cpu().numpy()
    assert torch.equal(torch.isnan(Xb_d).any(1), ~ok) and torch.equal(torch.isnan(Xb).any(1), ~ok)
    assert torch.equal(torch.isnan(nll_d[:, 0]), torch.isnan(nll[:n])), f"{tag}: NaN nll rows differ from the dense route"
    for s, name in ((S_XB2, "XB2"), (S_QUAD, "QUAD")):
        assert bool(sc[s] != sc[s]) == bool(sd[s] != sd[s]), f"{tag}: scal[{name}] {sc[s]} vs dense route {sd[s]}"
    print(f"[{tag}] worst bound ratio nll {r_nll:.3f} ({int((~ok).sum())} out-of-range rows: NaN as on the dense route)")


# -------------------------------------------------------------------------- F. structured NLL bias at planes shapes
# (L, lvs, pattern, Z scale, kinds): P = 600 objects, p = 128, q = 8 = nviews, n = 20000 -- the planes form of st()
F_CASES = [(64, (0.4, -0.6), "uniform", 1.0, ("kr",)), (64, (0.0, 0.0), "uniform", 1.0, ("kr",)),
           (256, (1.0, -2.0), "uniform", 1.0, ("kr",)), (256, (0.4, -0.6), "uniform", 1.0, ("kr",)),
           (64, (0.4, -0.6), "skewed", 1e-3, ("kr",)),
           (64, (2.0, -3.0, 0.0, -1.0), "skewed", 1e-3, ("kr", "object", "view"))]


@pytest.mark.parametrize("case", F_CASES, ids=lambda c: "L{}-lvs{}-{}-Zx{:g}-{}".format(c[0], "_".join(map(str, c[1])),
                                                                                     c[2], c[3], "+".join(c[4])))
def test_structured_nll_bias_planes_shapes(case):
    """The twin of test_nll_bias_small_shapes on vm.lazy(d, w) / vm.lazy_effects(d, w) where st() runs on the planes
    (P >= 512, p >= 128): sum(nll) within 1e-5 and Xb within 1e-4 (max-relative) of the fp64 oracle, also with the
    latent columns scaled by 1e-3 and one slot holding 10 % of the rows.  Where the dense route on the same inputs
    misses those bounds itself (lvs = (0, 0) at L = 64: Sigma nll +3.1e-5; one row of V repeated 2000 times: Xb 3.4e-4 on
    three designs), the structured route, which replaces it, must be no worse than it."""
    import gppvae_b200
    from oracle import gp_oracle as O
    L, lvs, pattern, zscale, kinds = case
    n, P, p, q = 20000, 600, 128, 8
    seed = L + len(kinds)
    g = torch.Generator(device=DEV).manual_seed(seed)
    x0 = torch.randn(P, p, generator=g, device=DEV)
    v0 = torch.eye(q, device=DEV) + 0.5 * torch.randn(q, q, generator=g, device=DEV)
    d, w = rows_of(n, P, q, pattern, seed + 1)
    V64 = O.feature_map(x0.double(), v0.double(), d, w)
    mix = torch.randn(p * q, L, generator=g, device=DEV, dtype=torch.float64)
    Z = ((0.5 * torch.randn(n, L, generator=g, device=DEV, dtype=torch.float64) + V64 @ mix) * zscale).float()
    vm = gppvae_b200.Vmodel(P, q, p, q).to(DEV)
    gp = gppvae_b200.GP(n_rand_effs=len(kinds)).to(DEV)
    lv = torch.tensor(lvs, device=DEV)
    with torch.no_grad():
        vm.x0.copy_(x0); vm.v0.copy_(v0); gp.lvs.copy_(lv)
    Vs = [vm.lazy(d, w)] if kinds == ("kr",) else vm.lazy_effects(d, w, kinds)
    Vd = [V.dense().double() for V in Vs]                 # the fp32 designs the kernels see, in fp64
    onll, oXb = O.nll_and_grad(Z.double(), Vd, lv.double())
    Xb, _, _, nll = gp.taylor_coeff(Z, Vs, need_vb=False)
    e_nll = (nll.double().sum().item() - onll.sum().item()) / abs(onll.sum().item())
    e_xb = rel_err(Xb, oXb)
    gpd = gppvae_b200.GP(n_rand_effs=len(kinds)).to(DEV)
    with torch.no_grad():
        gpd.lvs.copy_(lv)
    Xb_d, _, _, nll_d = gpd.taylor_coeff(Z, [V.dense() for V in Vs], need_vb=False)
    e_nll_d = (nll_d.double().sum().item() - onll.sum().item()) / abs(onll.sum().item())
    print(f"[structured n={n} P={P} p={p} q={q} L={L} lvs={lvs} {pattern} Z x{zscale:g} {'+'.join(kinds)}] "
          f"rel NLL err {e_nll:+.2e}  Xb {e_xb:.2e}   (dense route: NLL {e_nll_d:+.2e}  Xb {rel_err(Xb_d, oXb):.2e})")
    assert abs(e_nll) < max(1e-5, abs(e_nll_d))
    assert e_xb < max(1e-4, rel_err(Xb_d, oXb))
