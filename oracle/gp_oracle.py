"""CPU oracle for the GPPVAE low-rank GP prior term (TEST INFRASTRUCTURE ONLY).

A function-by-function restatement of the reference's algorithm for the hot
path, written with the same torch CPU primitives the reference itself calls
(``mm``, ``svd``, ``inverse``, ``softmax``, ``embedding``) so that both its
arithmetic and its cost on the host cores are the reference's.  The dtype of
every result follows the dtype of the inputs: feed float32 for the "reference
as shipped" behaviour, float64 for the ground truth used to grade quantities
the fp32 reference itself cannot pin (``Vb``, ``vbs[0]``; BASELINE.md section 2).

Pinning: ``tests/golden/make_golden.py`` imports the *unmodified* reference
classes from the reference checkout (under a three-line shim) and stores their
inputs/outputs in ``tests/golden/*.npz``; ``tests/test_oracle.py`` checks every
function below against those vectors.

Each function cites the reference lines it follows.  Symbols: ``n`` rows,
``Q`` columns of V (= p*q), ``L`` latent dimensions, ``vs = [v0, vn]``.
"""
from __future__ import annotations

from typing import List, Sequence, Tuple

import torch
import torch.nn.functional as F

Tensor = torch.Tensor


# --------------------------------------------------------------------------
# vmod.py
# --------------------------------------------------------------------------
def unit_rows(table: Tensor) -> Tensor:
    """Scale every row to unit Euclidean length (reference vmod.py:10-12)."""
    sq = (table * table).sum(dim=1, keepdim=True)
    return table / sq.sqrt()


def init_tables(P: int, nviews: int, p: int, q: int, gen: torch.Generator | None = None,
                dtype=torch.float32) -> Tuple[Tensor, Tensor]:
    """Initial object / view tables (reference vmod.py:18-19,37-40).

    Objects start as e_0 plus 1e-3 noise, views as the identity plus 1e-3
    noise.  (The random stream is not the reference's -- only the
    distribution is; tests that need identical tables copy them over.)
    """
    x0 = torch.empty(P, p, dtype=dtype)
    x0[:, 0] = 1.0
    x0[:, 1:] = 1e-3 * torch.randn(P, p - 1, generator=gen, dtype=dtype)
    v0 = torch.eye(nviews, q, dtype=dtype) + 1e-3 * torch.randn(nviews, q, generator=gen, dtype=dtype)
    return x0, v0


def feature_map(x0: Tensor, v0: Tensor, d: Tensor, w: Tensor) -> Tensor:
    """Row-wise Khatri-Rao feature map (reference vmod.py:22-35).

    ``V[i, j*q + k] = xhat[d_i, j] * what[w_i, k]`` with row-normalised tables.
    """
    xrows = F.embedding(d, unit_rows(x0))          # vmod.py:30
    wrows = F.embedding(w, unit_rows(v0))          # vmod.py:31
    outer = xrows.unsqueeze(2) * wrows.unsqueeze(1)  # vmod.py:33  (ij,ik->ijk)
    return outer.reshape(outer.shape[0], -1)       # vmod.py:34


# --------------------------------------------------------------------------
# gp.py
# --------------------------------------------------------------------------
def variances(lvs: Tensor) -> Tensor:
    """``vs = softmax(lvs)`` -> [v0, vn]  (reference gp.py:48-50; the
    ``vsum2one=False`` branch at gp.py:52 is broken upstream and not restated)."""
    return F.softmax(lvs, 0)


def woodbury_factor(Vs: Sequence[Tensor], vs: Tensor) -> Tuple[Tensor, Tensor, Tensor]:
    """``U, U B^-1, svdvals(B)`` with ``B = U^T U + I`` (reference gp.py:24-38)."""
    stacked = torch.cat([vs[i].sqrt() * Vi for i, Vi in enumerate(Vs)], 1)   # gp.py:27
    U = stacked / vs[-1].sqrt()                                               # gp.py:28
    B = U.t().mm(U) + torch.eye(U.shape[1], dtype=U.dtype, device=U.device)  # gp.py:29-30
    Shb = torch.svd(B)[1]                                                     # gp.py:33
    UBi = U.mm(torch.inverse(B))                                              # gp.py:35-36
    return U, UBi, Shb


def woodbury_solve(X: Tensor, U: Tensor, UBi: Tensor, vs: Tensor) -> Tensor:
    """``K^-1 X = (X - U B^-1 U^T X) / vn`` (reference gp.py:40-46)."""
    return (X - UBi.mm(U.t().mm(X))) / vs[-1]


def _row_nll(X: Tensor, Xb: Tensor, Shb: Tensor, vs: Tensor) -> Tensor:
    """Per-row NLL, no 2*pi constant (reference gp.py:84-87 == gp.py:105-108)."""
    n, L = X.shape
    quad = (X * Xb).sum(1, keepdim=True)
    logdet = n * L * vs[-1].log() + L * Shb.log().sum()
    return 0.5 * quad + 0.5 * logdet / n


def nll(X: Tensor, Vs: Sequence[Tensor], lvs: Tensor) -> Tensor:
    """Differentiable low-rank NLL (reference gp.py:97-110)."""
    vs = variances(lvs)
    U, UBi, Shb = woodbury_factor(Vs, vs)
    return _row_nll(X, woodbury_solve(X, U, UBi, vs), Shb, vs)


def nll_and_grad(X: Tensor, Vs: Sequence[Tensor], lvs: Tensor) -> Tuple[Tensor, Tensor]:
    """The "NLL + dNLL/dZ" evaluation BASELINE.json's metric counts: exactly the work of the reference's
    GP.nll under no_grad (gp.py:97-110) with its local Xb = K^-1 X (gp.py:102) handed back as well."""
    with torch.no_grad():
        vs = variances(lvs)
        U, UBi, Shb = woodbury_factor(Vs, vs)
        Xb = woodbury_solve(X, U, UBi, vs)
        return _row_nll(X, Xb, Shb, vs), Xb


def nll_dense(X: Tensor, Vs: Sequence[Tensor], lvs: Tensor) -> Tensor:
    """O(n^3) NLL through the dense n x n covariance (reference gp.py:112-125)."""
    vs = variances(lvs)
    stacked = torch.cat([vs[i].sqrt() * Vi for i, Vi in enumerate(Vs)], 1)
    K = stacked.mm(stacked.t()) + vs[-1] * torch.eye(X.shape[0], dtype=X.dtype)
    Shk = torch.svd(K)[1]
    Xb = torch.inverse(K).mm(X)
    quad = (X * Xb).sum(1, keepdim=True)
    return 0.5 * quad + 0.5 * X.shape[1] * Shk.log().sum() / X.shape[0]


def taylor_coeff(X: Tensor, Vs: Sequence[Tensor], lvs: Tensor
                 ) -> Tuple[Tensor, List[Tensor], Tensor, Tensor]:
    """First-order Taylor coefficients of the NLL (reference gp.py:55-95).

    Returns ``Xb = dNLL/dX``, ``[Vb = dNLL/dV]``, ``vbs = dNLL/d[v0, vn]`` and the
    per-row ``nll``; everything detached, as gp.py:90-93 does.
    """
    with torch.no_grad():
        vs = variances(lvs)
        U, UBi, Shb = woodbury_factor(Vs, vs)
        Xb = woodbury_solve(X, U, UBi, vs)
        n, L = X.shape
        vbs = torch.zeros(len(Vs) + 1, dtype=X.dtype)
        Vbs = []
        for iv, Vi in enumerate(Vs):
            XbV = Xb.t().mm(Vi)                                   # gp.py:68
            KiV = woodbury_solve(Vi, U, UBi, vs)                  # gp.py:70
            Vbs.append(vs[iv] * (L * KiV - Xb.mm(XbV)))           # gp.py:69,71
            vbs[iv] = -0.5 * (XbV * XbV).sum() + 0.5 * L * (Vi * KiV).sum()   # gp.py:75-76
        trKi = (n - (UBi * U).sum()) / vs[-1]                     # gp.py:79
        vbs[-1] = -0.5 * (Xb * Xb).sum() + 0.5 * L * trKi         # gp.py:80-81
        out = _row_nll(X, Xb, Shb, vs)
    return Xb, Vbs, vbs, out


def taylor_expansion(X: Tensor, Vs: Sequence[Tensor], Xb: Tensor, Vbs: Sequence[Tensor],
                     vbs: Tensor, lvs: Tensor) -> Tensor:
    """Linear surrogate whose gradients are the exact NLL gradients
    (reference gp.py:127-133).  Note gp.py:132 divides by the *minibatch* rows."""
    out = (Xb * X).sum(1, keepdim=True)
    for Vi, Vbi in zip(Vs, Vbs):
        out = out + (Vbi * Vi).sum(1, keepdim=True)
    return out + (vbs * variances(lvs)).sum() / float(X.shape[0])


# --------------------------------------------------------------------------
# Q-space model of what the CUDA kernels compute (SURVEY.md section 7.2).
# Not in the reference: used by tests to check kernel intermediates stage by
# stage, and itself checked against taylor_coeff() above in tests/test_oracle.py.
# --------------------------------------------------------------------------
def qspace_model(X: Tensor, V: Tensor, lvs: Tensor, n_total: int | None = None, want_vb: bool = True):
    """Woodbury terms through G = V^T V, C = V^T X and a Cholesky of
    B = I + (v0/vn) G.  Returns a dict with every intermediate the kernels expose."""
    with torch.no_grad():
        vs = variances(lvs)
        v0, vn = vs[0], vs[1]
        r = v0 / vn
        n, L = X.shape
        n_total = n if n_total is None else n_total
        Q = V.shape[1]
        G = V.t().mm(V)
        C = V.t().mm(X)
        B = torch.eye(Q, dtype=V.dtype, device=V.device) + r * G
        Lc = torch.linalg.cholesky(B)
        logdetB = 2.0 * Lc.diagonal().log().sum()
        Linv = torch.linalg.solve_triangular(Lc, torch.eye(Q, dtype=V.dtype, device=V.device), upper=False)
        Binv = Linv.t().mm(Linv)
        W = r * Binv.mm(C)
        Xb = (X - V.mm(W)) / vn
        quad = (X * Xb).sum(1, keepdim=True)
        row_const = 0.5 * L * (vn.log() + logdetB / n_total)
        trBinv = Binv.diagonal().sum()
        vbs = torch.stack([
            -0.5 * (W * W).sum() / (v0 * v0) + 0.5 * L * ((Q - trBinv) / r) / vn,
            -0.5 * (Xb * Xb).sum() + 0.5 * L * (n_total - Q + trBinv) / vn,
        ])
        out = dict(G=G, C=C, B=B, Lc=Lc, logdetB=logdetB, Linv=Linv, Binv=Binv, W=W, Xb=Xb,
                   nll=0.5 * quad + row_const, vbs=vbs, trBinv=trBinv)
        if want_vb:
            out["Vb"] = r * L * V.mm(Binv) - Xb.mm(W.t())
    return out


def qspace_model_streamed(X: Tensor, V: Tensor, lvs: Tensor, n_total: int | None = None, chunk: int = 1 << 16):
    """qspace_model() in float64 for inputs too large to hold as doubles: X and V (any float dtype, any device) are
    read in row chunks converted to float64 on the fly, so a 16 GB fp32 V never needs a 32 GB copy.  Same formulas,
    same outputs except the N x Q ones (no Vb, no G-sized extras beyond G itself).  This is the checker of the
    full-size GPU parity tests (BASELINE.json configs[1], configs[2]): it runs on the GPU box's device through stock
    torch float64 -- test infrastructure, never the product path."""
    with torch.no_grad():
        dev = V.device
        vs = variances(lvs.to(device=dev, dtype=torch.float64))
        v0, vn = vs[0], vs[1]
        r = v0 / vn
        n, L = X.shape
        n_total = n if n_total is None else n_total
        Q = V.shape[1]
        G = torch.zeros(Q, Q, dtype=torch.float64, device=dev)
        C = torch.zeros(Q, L, dtype=torch.float64, device=dev)
        for a in range(0, n, chunk):
            Vc = V[a:a + chunk].double()
            G.addmm_(Vc.t(), Vc)
            C.addmm_(Vc.t(), X[a:a + chunk].double())
        B = torch.eye(Q, dtype=torch.float64, device=dev) + r * G
        Lc = torch.linalg.cholesky(B)
        logdetB = 2.0 * Lc.diagonal().log().sum()
        Binv = torch.cholesky_inverse(Lc)
        W = r * Binv.mm(C)
        Xb = torch.empty(n, L, dtype=torch.float64, device=dev)
        for a in range(0, n, chunk):
            Xb[a:a + chunk] = (X[a:a + chunk].double() - V[a:a + chunk].double().mm(W)) / vn
        quad = (X.double() * Xb).sum(1, keepdim=True)
        row_const = 0.5 * L * (vn.log() + logdetB / n_total)
        trBinv = Binv.diagonal().sum()
        vbs = torch.stack([
            -0.5 * (W * W).sum() / (v0 * v0) + 0.5 * L * ((Q - trBinv) / r) / vn,
            -0.5 * (Xb * Xb).sum() + 0.5 * L * (n_total - Q + trBinv) / vn,
        ])
        return dict(G=G, C=C, logdetB=logdetB, W=W, Xb=Xb, nll=0.5 * quad + row_const, vbs=vbs, trBinv=trBinv)
