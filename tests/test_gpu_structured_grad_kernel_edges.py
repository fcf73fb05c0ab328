"""The two entries of the table gradient on the structured route (gpp_kr_grad_rhs, gpp_kr_grad_views; DESIGN 5.8)
against float64, element by element, with the conventions of test_gpu_structured_kernel_edges.py: sentinel output
buffers (one extra row, ld = cols + 8, a NaN bit pattern that must survive), inputs with ld > cols whose gap holds NaN,
and the worst bound ratio printed per case.

The bounds, in units of u = 2^-24 (gamma_k = k u / (1 - k u), the error of a k-step fp32 recursive sum; a warp's
lane-strided fma chains joined by a butterfly are such a sum over the same terms in another order):
  R, the alpha H_v range    q^2 terms wn[v,k'] wn[v,k] B^-1[..], the weight product rounded once, then alpha (double)
                            times the fp32 sum, rounded once: gamma_(q^2 + 3) |alpha| sum |wn| |B^-1| |wn|.
  R, the -M_v^T range       an fma chain of q terms: gamma_(q + 1) sum_k |wn[v,k]| |W[(j,k), l]|; rows of zero columns
                            of W are exactly zero.
  gw                        per j', p q products S wn B^-1 (one rounding for S wn) summed over the tiles, times alpha
                            (one rounding), minus an L-term chain; then p partials added: gamma_(p q + p + L + 6) times
                            |alpha| sum |S| |wn| |B^-1| + sum |T| |W|.
"""
import pytest
import torch

from edge_helpers import DEV, call, check_sentinel, gamma, grade, sentinel, strided, stream, workspace

pytestmark = pytest.mark.gpu

# (p, q, nviews, L): p at 4, 128 and 132; nviews = 1 and nviews > q; q large enough that a tile of B^-1 holds one
# object column (jc = 1) and, at q = 110, needs more than 48 KB of shared memory; the c3 block shape last
CASES = [(4, 3, 1, 8), (4, 5, 9, 12), (128, 4, 6, 16), (132, 3, 5, 8), (128, 9, 1, 64), (8, 70, 3, 12),
         (8, 110, 2, 4), (256, 16, 16, 256)]
ALPHA = 37.5


@pytest.fixture(scope="module", autouse=True)
def lib():
    from gppvae_b200 import _lib
    return _lib.load()


def _inputs(p, q, nv, L, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    Q = p * q
    B = torch.randn(Q, Q, generator=g, device=DEV) * 10.0 ** (torch.rand(Q, 1, generator=g, device=DEV) * 2 - 1)
    W = torch.randn(Q, L, generator=g, device=DEV) * 10.0 ** (torch.rand(1, L, generator=g, device=DEV) * 4 - 2)
    W[:, L - 3:] = 0.0                      # padded latent columns, as gpp_solve_w leaves them
    wn = torch.randn(nv, q, generator=g, device=DEV)
    wn = wn / wn.norm(dim=1, keepdim=True)
    ST = torch.randn(p, nv * (p + L), generator=g, device=DEV) * 10.0 ** (
        torch.rand(1, nv * (p + L), generator=g, device=DEV) * 4 - 2)
    return B, W, wn, ST


def _rhs_ref(B, W, wn, p, L, alpha):
    nv, q = wn.shape
    w, B4, W3 = wn.double(), B.double().view(p, q, p, q), W.double().view(p, q, L)
    H = torch.einsum("va,iajb,vb->vij", w, B4, w)
    Ha = torch.einsum("va,iajb,vb->vij", w.abs(), B4.abs(), w.abs())
    M = torch.einsum("vk,jkl->vlj", w, W3)
    Ma = torch.einsum("vk,jkl->vlj", w.abs(), W3.abs())
    return alpha * H.reshape(nv * p, p), abs(alpha) * Ha.reshape(nv * p, p), -M.reshape(nv * L, p), Ma.reshape(nv * L, p)


def _views_ref(ST, B, W, wn, p, L, alpha):
    nv, q = wn.shape
    w, B4, W3 = wn.double(), B.double().view(p, q, p, q), W.double().view(p, q, L)
    S = ST.double()[:, : nv * p].view(p, nv, p)
    T = ST.double()[:, nv * p:].view(p, nv, L)
    ref = alpha * torch.einsum("jvi,vc,icjk->vk", S, w, B4) - torch.einsum("jvl,jkl->vk", T, W3)
    mag = abs(alpha) * torch.einsum("jvi,vc,icjk->vk", S.abs(), w.abs(), B4.abs()) + \
        torch.einsum("jvl,jkl->vk", T.abs(), W3.abs())
    return ref, mag


def _grad_rhs(lib, B, ldb, W, ldw, wn, p, L, alpha):
    nv, q = wn.shape
    rows = nv * (p + L)
    R, ldr = sentinel(rows, p)
    call(lib.gpp_kr_grad_rhs(B.data_ptr(), ldb, W.data_ptr(), ldw, wn.data_ptr(), p, q, nv, L, alpha, R.data_ptr(), ldr,
                             stream()), "kr_grad_rhs")
    torch.cuda.synchronize()
    return check_sentinel(R, rows, p, "kr_grad_rhs")


def _grad_views(lib, ST, ldst, B, ldb, W, ldw, wn, p, L, alpha):
    nv, q = wn.shape
    gw, ldg = sentinel(nv, q)
    ws = workspace(lib.gpp_kr_grad_views_workspace_bytes(p, q, nv))
    call(lib.gpp_kr_grad_views(ST.data_ptr(), ldst, B.data_ptr(), ldb, W.data_ptr(), ldw, wn.data_ptr(), p, q, nv, L,
                               alpha, gw.data_ptr(), ldg, ws.data_ptr(), ws.numel(), stream()), "kr_grad_views")
    torch.cuda.synchronize()
    return check_sentinel(gw, nv, q, "kr_grad_views")


@pytest.mark.parametrize("case", CASES, ids=lambda c: "p{}-q{}-nv{}-L{}".format(*c))
def test_kr_grad_rhs(lib, case):
    p, q, nv, L = case
    B, W, wn, _ = _inputs(p, q, nv, L, seed=p * 1000 + q)
    Bv, ldb = strided(B, 4)
    Wv, ldw = strided(W, 8)
    R = _grad_rhs(lib, Bv, ldb, Wv, ldw, wn, p, L, ALPHA)
    H, Ha, M, Ma = _rhs_ref(B, W, wn, p, L, ALPHA)
    tag = "p{}-q{}-nv{}-L{}".format(*case)
    grade(f"kr_grad_rhs alpha H {tag}", R[: nv * p], H, Ha, 1e-30, gamma(q * q + 3))
    grade(f"kr_grad_rhs -M^T {tag}", R[nv * p:], M, Ma, 1e-30, gamma(q + 1))
    pad = R[nv * p:].reshape(nv, L, p)[:, L - 3:]
    assert bool((pad == 0).all()), "rows of the zero columns of W must be exactly zero"
    assert torch.equal(_grad_rhs(lib, Bv, ldb, Wv, ldw, wn, p, L, ALPHA).view(torch.int32), R.view(torch.int32))


@pytest.mark.parametrize("case", CASES, ids=lambda c: "p{}-q{}-nv{}-L{}".format(*c))
def test_kr_grad_views(lib, case):
    p, q, nv, L = case
    B, W, wn, ST = _inputs(p, q, nv, L, seed=p * 1000 + q + 1)
    Bv, ldb = strided(B, 8)
    Wv, ldw = strided(W, 4)
    STv, ldst = strided(ST, 12)
    gw = _grad_views(lib, STv, ldst, Bv, ldb, Wv, ldw, wn, p, L, -ALPHA)
    ref, mag = _views_ref(ST, B, W, wn, p, L, -ALPHA)
    grade("kr_grad_views p{}-q{}-nv{}-L{}".format(*case), gw, ref, mag, 1e-30, gamma(p * q + p + L + 6))
    again = _grad_views(lib, STv, ldst, Bv, ldb, Wv, ldw, wn, p, L, -ALPHA)
    assert torch.equal(again.view(torch.int32), gw.view(torch.int32)), "repeats must be bit-identical"

