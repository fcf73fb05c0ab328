"""Drop-in `Vmodel` / `normalize_rows`: the reference's vmod.py API on top of the sm_100a kernels.

Same constructor `Vmodel(P, Q, p, q)`, parameters `x0 (P x p)` and `v0 (Q x q)`, methods `x()`, `v()`,
`forward(d, w)` and initialisation as /root/reference/pysrc/faceplace/vmod.py:10-40.  (In the reference
`Q` is the number of views; everywhere else in this package Q is the rank p*q.)
"""
from __future__ import annotations

import torch
from torch import nn

from . import ops
from .ops import normalize_rows  # noqa: F401  (re-exported: vmod.py:10-12)


class KhatriRao:
    """`V = Vmodel.forward(d, w)` held as its factors instead of as an N x (p q) matrix (SURVEY 8(f) row 4).

    `GP.taylor_coeff`, `GP.U_UBi_Shb` / `GP.solve` and `GP.nll` accept it in place of the dense tensor and then take
    the structured route of csrc/structured.cu: V is never written and the N-long GEMMs shrink to P-long ones.
    It is a detached snapshot of the normalised tables (what `vm(Dt, Wt).detach()` is in train_gppvae.py:161);
    `dense()` materialises the reference tensor, `t().mm(X)` is V^T X (train_gppvae.py:237), `[idx]` the dense rows.
    Made by `Vmodel.lazy(d, w, requires_grad=True)` it also keeps the attached tables (`tables`), and `GP.nll(X, [kr])`
    then sends the exact NLL gradient to x0 and v0 through the slots (DESIGN 5.8), without the N x Q matrix dNLL/dV.
    """

    def __init__(self, xn: torch.Tensor, wn: torch.Tensor, d: torch.Tensor, w: torch.Tensor):
        ops.require_cuda_f32(xn, "xn")
        ops.require_cuda_f32(wn, "wn")
        self.d = ops._check_index(d, "d", xn.device)
        self.w = ops._check_index(w, "w", xn.device)
        if self.d.shape != self.w.shape:
            raise ValueError("d and w must have the same length")
        if self.d.shape[0] == 0:
            raise ValueError("d and w are empty: there is no row of V to build")
        P, p = xn.shape
        self.P, self.p_true = P, p
        self.nviews, self.q = wn.shape
        self.wn = wn.detach().contiguous()
        if p % 4:      # the kernels want p % 4 == 0: zero columns of xn are zero columns of V
            xp = torch.zeros(P, ops.round4(p), device=xn.device, dtype=torch.float32)
            xp[:, :p] = xn.detach()
            self.xn = xp
        else:
            self.xn = xn.detach().contiguous()
        self.p = self.xn.shape[1]
        self.n = self.d.shape[0]
        self.shape = torch.Size((self.n, p * self.q))
        self.device = xn.device
        self._index = None
        self._max_count = None
        self._xn_planes = None
        self._rows_in_table = None
        self.tables = None       # (x(), v()) still attached to autograd: Vmodel.lazy(..., requires_grad=True)

    # -- index preparation (once per (d, w): the data set does not change between epochs) ------------------
    def index(self):
        """(order, slot_start): row indices sorted by slot o * nviews + v (stable) and the first position of every slot;
        rows with an index outside its table go to a trailing dummy slot (they get NaN rows of Xb, as in the dense path)."""
        if self._index is None:
            nslots = self.P * self.nviews
            bad = (self.d < 0) | (self.d >= self.P) | (self.w < 0) | (self.w >= self.nviews)
            key = torch.where(bad, torch.full_like(self.d, nslots), self.d * self.nviews + self.w)
            order = torch.argsort(key, stable=True)
            counts = torch.bincount(key, minlength=nslots + 1)[:nslots]
            slot_start = torch.zeros(nslots + 1, dtype=torch.int64, device=self.device)
            torch.cumsum(counts, 0, out=slot_start[1:])
            self._index = (order.contiguous(), slot_start)
            self._max_count = int(counts.max()) if counts.numel() else 0     # one host read per (d, w), with the index
        return self._index

    def max_count(self) -> int:
        """Rows in the fullest slot: bounds the slot sums when they are written as operand planes."""
        if self._max_count is None:
            self._index = None
            self.index()
        return self._max_count

    def rows_in_table(self) -> int:
        """Rows whose (d, w) lies inside the tables: the first rows_in_table() entries of `order` (the rest are the
        trailing dummy slot).  One host read per KhatriRao, on first use."""
        if self._rows_in_table is None:
            self._rows_in_table = int(self.index()[1][-1])
        return self._rows_in_table

    def st(self, Xm: torch.Tensor, ldx: int, Lx: int, with_x: bool) -> torch.Tensor:
        """ST = xn^T [cnt (x) xn | slot sums of X]  (p x nviews ((with_x ? p : 0) + Lx)).  From the tensor-core tile up
        (P >= 512, p >= 128) the slot sums are written as operand planes and the P-long product runs on the planes
        kernel; below that, an fp32 matrix and the kernel that splits its operands itself.  The two column ranges get
        planes of their own, each with the scale of its own bound (max_count for cnt (x) xn, max_count max|X| for the
        slot sums), as V and X have in the dense pass 1: under one shared scale the smaller range would lose bits."""
        return self.st_operands(Xm, ldx, Lx, with_x)[0]

    def st_operands(self, Xm: torch.Tensor, ldx: int, Lx: int, with_x: bool):
        """(ST, left operand) of `st`: the left operand [cnt (x) xn | slot sums of X] is the pair of planes (pS, pZ)
        (pS None without with_x) from the tensor-core tile up, else the fp32 matrix; the table gradient multiplies it
        once more (LazyVb.table_grads)."""
        order, slot_start = self.index()
        if ops.planes_supported(self.P, self.p, 0):
            ncnt = self.nviews * self.p if with_x else 0
            ST = torch.empty(self.p, ncnt + self.nviews * Lx, device=self.device, dtype=torch.float32)
            pS = None
            if with_x:
                pS = ops.kr_slot_sums_planes(Xm, ldx, order, slot_start, self.xn, self.nviews, Lx, 2, self.max_count())
                ops.atb_planes(self.xn_planes(), pS, self.P, self.p, pS.cols, out=ST[:, : pS.cols])
            pZ = ops.kr_slot_sums_planes(Xm, ldx, order, slot_start, self.xn, self.nviews, Lx, 0, self.max_count())
            ops.atb_planes(self.xn_planes(), pZ, self.P, self.p, pZ.cols, out=ST[:, ncnt:])
            return ST, (pS, pZ)
        XZ = ops.kr_slot_sums(Xm, ldx, order, slot_start, self.xn, self.nviews, Lx, with_x)
        return ops.atb(self.xn, self.p, XZ, XZ.stride(0), self.P, self.p, XZ.shape[1]), XZ

    def xn_planes(self):
        """Operand planes of the normalised object table (the left operand of both P-long products), split once."""
        if self._xn_planes is None:
            self._xn_planes = ops.split_planes(self.xn, self.p, self.P, self.p, unit_bound=True)
        return self._xn_planes

    # -- tensor-like surface the trainer touches -----------------------------------------------------------
    def detach(self) -> "KhatriRao":
        return self

    def dense(self) -> torch.Tensor:
        return ops.khatri_rao_fwd(self.xn[:, : self.p_true], self.wn, self.d, self.w)

    def __getitem__(self, idx) -> torch.Tensor:
        return ops.khatri_rao_fwd(self.xn[:, : self.p_true], self.wn, self.d[idx].contiguous(), self.w[idx].contiguous())

    def vtx(self, X: torch.Tensor) -> torch.Tensor:
        """V^T X (p q x m) through the slot sums: no N-long GEMM."""
        Xm, ldx = ops.as_matrix(X, "X")
        if Xm.shape[0] != self.n:
            raise ValueError(f"X has {Xm.shape[0]} rows but V has {self.n}")
        Lk = Xm.shape[1]
        ST = self.st(Xm, ldx, Lk, False)
        C = ops.kr_assemble_gc(ST, self.wn, self.p, Lk, False)
        q = self.q
        if self.p != self.p_true:
            C = C[: self.p_true * q]
        return C[:, : X.shape[1]]

    def t(self) -> "_KhatriRaoT":
        return _KhatriRaoT(self)


class _KhatriRaoT:
    def __init__(self, kr):
        self.kr = kr
        self.shape = torch.Size((kr.shape[1], kr.shape[0]))

    def mm(self, X: torch.Tensor) -> torch.Tensor:
        return self.kr.vtx(X)

    __matmul__ = mm


class _FactoredEffect:
    """A design over the tables and slot index of a KhatriRao `kr` (Vmodel.lazy_effects): the same tensor-like surface
    as KhatriRao.  Several of them, with `kr` itself, are the designs of GP(n_rand_effs=k) on the structured route."""

    kind = ""

    def __init__(self, kr: KhatriRao, width: int):
        self.kr = kr
        self.n = kr.n
        self.device = kr.device
        self.shape = torch.Size((kr.n, width))

    def detach(self) -> "_FactoredEffect":
        return self

    def dense(self) -> torch.Tensor:
        return self._rows(self.kr.d, self.kr.w)

    def __getitem__(self, idx) -> torch.Tensor:
        return self._rows(self.kr.d[idx].contiguous(), self.kr.w[idx].contiguous())

    def vtx(self, X: torch.Tensor) -> torch.Tensor:
        """V^T X (width x m) through the slot sums (object) or the per-view sums (view): no N-long GEMM."""
        Xm, ldx = ops.as_matrix(X, "X")
        if Xm.shape[0] != self.n:
            raise ValueError(f"X has {Xm.shape[0]} rows but V has {self.n}")
        return effects_c(self.kr, [self.kind], Xm, ldx, Xm.shape[1])[: self.shape[1], : X.shape[1]]

    def t(self) -> "_KhatriRaoT":
        return _KhatriRaoT(self)


class ObjectEffect(_FactoredEffect):
    """The object-only design V[i, j] = x()[d_i, j] (n x p), held as the factors of `kr`."""

    kind = "object"

    def __init__(self, kr: KhatriRao):
        super().__init__(kr, kr.p_true)

    def _rows(self, d, w):
        kr = self.kr   # xn (x) a one-column view table of ones is xn[d]
        return ops.khatri_rao_fwd(kr.xn[:, : kr.p_true], torch.ones(kr.nviews, 1, device=kr.device), d, w)


class ViewEffect(_FactoredEffect):
    """The view-only design V[i, k] = v()[w_i, k] (n x q), held as the factors of `kr`."""

    kind = "view"

    def __init__(self, kr: KhatriRao):
        super().__init__(kr, kr.q)

    def _rows(self, d, w):
        kr = self.kr   # a one-column object table of ones (x) wn is wn[w]
        return ops.khatri_rao_fwd(torch.ones(kr.P, 1, device=kr.device), kr.wn, d, w)


def effect_kind(V) -> str:
    return "kr" if isinstance(V, KhatriRao) else V.kind


def effect_base(V) -> KhatriRao:
    return V if isinstance(V, KhatriRao) else V.kr


def effects_st_vm(kr: KhatriRao, kinds, Xm: torch.Tensor, ldx: int, Lx: int, with_g: bool):
    """The per-rank partial sums the stacked designs `kinds` need: ST (slot sums through x^T, None without K and O) and
    VM (per-view moments, None without W)."""
    ST = kr.st(Xm, ldx, Lx, with_g) if ("kr" in kinds or "object" in kinds) else None
    VM = None
    if "view" in kinds:
        order, slot_start = kr.index()
        VM = ops.kr_view_sums(Xm, ldx, order, slot_start, kr.xn, kr.nviews, Lx, with_g)
    return ST, VM


def effects_c(kr: KhatriRao, kinds, Xm: torch.Tensor, ldx: int, Lk: int, reduce=None) -> torch.Tensor:
    """C = V^T X of the stacked designs `kinds` (padded block widths); `reduce(ST, VM)` sums the partials over row
    shards (GP._all_reduce_pair)."""
    ST, VM = effects_st_vm(kr, kinds, Xm, ldx, Lk, False)
    if reduce is not None:
        ST, VM = reduce(ST, VM)
    return ops.kr_assemble_gc_blocks(ST, VM, kr.wn, kr.p, kinds, Lk, False)


class Vmodel(nn.Module):
    def __init__(self, P: int, Q: int, p: int, q: int):
        super().__init__()
        self.x0 = nn.Parameter(torch.randn(P, p))     # vmod.py:18
        self.v0 = nn.Parameter(torch.randn(Q, q))     # vmod.py:19
        self._init_params()

    def x(self) -> torch.Tensor:
        """Row-normalised object table (vmod.py:22-23)."""
        return ops.normalize_rows(self.x0)

    def v(self) -> torch.Tensor:
        """Row-normalised view table (vmod.py:25-26)."""
        return ops.normalize_rows(self.v0)

    def forward(self, d: torch.Tensor, w: torch.Tensor) -> torch.Tensor:
        """V[i, j*q + k] = x()[d_i, j] * v()[w_i, k]  (vmod.py:28-35), differentiable w.r.t. x0 and v0."""
        return ops._KhatriRao.apply(self.x(), self.v(), d, w)

    def lazy(self, d: torch.Tensor, w: torch.Tensor, requires_grad: bool = False) -> KhatriRao:
        """The same V as `forward(d, w).detach()`, kept in factored form (see KhatriRao): the epoch-level call of
        train_gppvae.py:161 when the GP term should take the structured route.  With `requires_grad=True` the KhatriRao
        also keeps x() and v() attached, and `GP.nll(X, [kr])` sends the exact NLL gradient back to x0 and v0."""
        if requires_grad:
            xa, va = self.x(), self.v()
            kr = KhatriRao(xa, va, d, w)
            kr.tables = (xa, va)
        else:
            with torch.no_grad():
                kr = KhatriRao(self.x(), self.v(), d, w)
        # the sort of the rows by (object, view) slot depends on (d, w) alone: the trainer passes the same index
        # tensors every epoch (train_gppvae.py:123-126, 161), so keep the last one
        key = (kr.d.data_ptr(), kr.d._version, kr.w.data_ptr(), kr.w._version, kr.n, kr.P, kr.nviews)
        cached = getattr(self, "_lazy_index", None)
        if cached is not None and cached[0] == key:
            kr._index, kr._max_count = cached[1], cached[3]
        else:
            self._lazy_index = (key, kr.index(), (kr.d, kr.w), kr.max_count())   # keeps d, w alive so the addresses stay theirs
        return kr

    def lazy_effects(self, d: torch.Tensor, w: torch.Tensor, kinds=("kr", "object", "view")) -> list:
        """Factored designs of GP(n_rand_effs=len(kinds)) for the rows (d, w): "kr" is `lazy(d, w)`, "object" the
        object-only design x()[d] (ObjectEffect), "view" the view-only design v()[w] (ViewEffect).  They share one slot
        index and one snapshot of the normalised tables, so GP takes the structured route with all of them."""
        if not kinds or len(set(kinds)) != len(kinds) or any(k not in ("kr", "object", "view") for k in kinds):
            raise ValueError(f"kinds must be distinct values of 'kr', 'object', 'view' (got {kinds})")
        kr = self.lazy(d, w)
        return [kr if k == "kr" else ObjectEffect(kr) if k == "object" else ViewEffect(kr) for k in kinds]

    def _init_params(self) -> None:
        """vmod.py:37-40: objects start at e_0 (+1e-3 noise), views at the identity (+1e-3 noise)."""
        with torch.no_grad():
            self.x0[:, 0] = 1.0
            self.x0[:, 1:] = 1e-3 * torch.randn(self.x0.shape[0], self.x0.shape[1] - 1)
            self.v0.copy_(torch.eye(*self.v0.shape) + 1e-3 * torch.randn(*self.v0.shape))
