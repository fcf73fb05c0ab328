"""Tensor-level wrappers over the C ABI: argument checks, layout normalisation, workspaces.

PyTorch is used here for device memory, streams and autograd bookkeeping only; every numerical
operation of the hot path is a call into libgppvae_b200.so.
"""
from __future__ import annotations

from typing import Optional, Tuple

import torch

import collections
import weakref

from . import _lib
from ._lib import EFFECT_KINDS, GPP_PLANES_COLSQ, GPP_PLANES_UNIT_BOUND, GPP_WANT_BINV, NSCAL, check


def _stream(device=None) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def _guard(t: torch.Tensor):
    """Make `t`'s device current for the duration of a launch (the C side launches on the current device)."""
    return torch.cuda.device(t.device)


def _on_device(fn):
    """Run a wrapper with the device of its first CUDA tensor argument current, and refuse operands spread over
    several devices: the library launches on the current device and stream, whatever the pointers say."""
    import functools

    @functools.wraps(fn)
    def wrapped(*args, **kwargs):
        dev = None
        for a in list(args) + list(kwargs.values()):
            t = a.buf if isinstance(a, Planes) else (a.state if isinstance(a, Factorisation) else a)
            if isinstance(t, torch.Tensor) and t.device.type == "cuda":
                if dev is None:
                    dev = t.device
                elif t.device != dev:
                    raise ValueError(f"{fn.__name__}: operands live on different devices ({dev} and {t.device})")
        if dev is None or dev.index == torch.cuda.current_device():
            return fn(*args, **kwargs)
        with torch.cuda.device(dev):
            return fn(*args, **kwargs)
    return wrapped


def _p(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def require_cuda_f32(t: torch.Tensor, name: str, ndim: int = 2) -> None:
    if not isinstance(t, torch.Tensor):
        raise ValueError(f"{name} must be a torch.Tensor")
    if t.device.type != "cuda":
        raise ValueError(f"{name} must live on a CUDA device (got {t.device}); gppvae_b200 has no CPU path")
    if t.dtype != torch.float32:
        raise ValueError(f"{name} must be float32 (got {t.dtype})")
    if t.dim() != ndim:
        raise ValueError(f"{name} must have {ndim} dimensions (got shape {tuple(t.shape)})")


def round4(c: int) -> int:
    return (c + 3) // 4 * 4


def as_matrix(t: torch.Tensor, name: str) -> Tuple[torch.Tensor, int]:
    """Return (tensor, ld) usable by the kernels: unit column stride, 16-byte aligned rows, columns padded
    with zeros to a multiple of 4.  Tensors that already qualify are passed through without a copy."""
    require_cuda_f32(t, name)
    t = t.detach()
    n, c = t.shape
    if n == 0 or c == 0:
        raise ValueError(f"{name} is empty ({n} x {c})")
    if c % 4 == 0 and t.data_ptr() % 16 == 0:
        if t.is_contiguous():
            return t, c
        if t.stride(1) == 1 and t.stride(0) % 4 == 0 and t.stride(0) >= c:
            return t, t.stride(0)
    buf = torch.zeros(n, round4(c), device=t.device, dtype=torch.float32)
    buf[:, :c] = t
    return buf, buf.shape[1]


def _workspace(nbytes: int, device) -> torch.Tensor:
    return torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)


# ----------------------------------------------------------------------------- Vmodel
@_on_device
def normalize_rows_fwd(x: torch.Tensor) -> torch.Tensor:
    require_cuda_f32(x, "x")
    x = x.detach().contiguous()
    y = torch.empty_like(x)
    check(_lib.load().gpp_normalize_rows_fwd(_p(x), x.shape[0], x.shape[1], _p(y), _stream()), "normalize_rows_fwd")
    return y


@_on_device
def normalize_rows_bwd(x: torch.Tensor, gy: torch.Tensor) -> torch.Tensor:
    x = x.detach().contiguous()
    gy = gy.detach().contiguous()
    gx = torch.empty_like(x)
    check(_lib.load().gpp_normalize_rows_bwd(_p(x), _p(gy), x.shape[0], x.shape[1], _p(gx), _stream()),
          "normalize_rows_bwd")
    return gx


def _check_index(t: torch.Tensor, name: str, device) -> torch.Tensor:
    if t.dtype != torch.int64 or t.dim() != 1:
        raise ValueError(f"{name} must be a 1-D int64 tensor (got {t.dtype}, shape {tuple(t.shape)})")
    if t.device != device:
        raise ValueError(f"{name} is on {t.device} but the tables are on {device}")
    return t.contiguous()


# ----------------------------------------------------------------------------- operand planes
class Planes:
    """fp16 hi / lo operand planes of an fp32 matrix (include/gppvae_b200.h, "pre-split operand planes"): an opaque
    device buffer of gpp_planes_bytes(n, cols), optionally carrying the matrix' exact column sums of squares."""

    def __init__(self, buf: torch.Tensor, n: int, cols: int, colsq: bool):
        self.buf, self.n, self.cols, self.colsq = buf, n, cols, colsq

    @property
    def ptr(self) -> int:
        return self.buf.data_ptr()


_supported_cache = {}


def planes_supported(n: int, Q: int, L: int) -> bool:
    key = (n >= 512, Q >= 128, L >= 64 or L == 0)
    if key not in _supported_cache:
        _supported_cache[key] = bool(_lib.load().gpp_planes_supported(n, Q, L))
    return _supported_cache[key]


class _PlaneRegistry:
    """Planes of the most recently produced matrices, found again by storage address, layout and version.

    An entry keeps its matrix alive, so the address cannot be recycled for another tensor while the entry exists
    (`_version` catches in-place updates; writes through `.data` are invisible to it -- call `invalidate()`)."""

    def __init__(self, cap: int = 2):
        self.cap = cap
        self.entries = collections.OrderedDict()

    @staticmethod
    def key(t: torch.Tensor, ld: int):
        return (t.device.index, t.untyped_storage().data_ptr(), t.storage_offset(), t.shape[0], t.shape[1], ld)

    def put(self, t: torch.Tensor, ld: int, planes: Planes) -> None:
        k = self.key(t, ld)
        self.entries.pop(k, None)
        self.entries[k] = (t._version, planes, t)
        while len(self.entries) > self.cap:
            self.entries.popitem(last=False)

    def get(self, t: torch.Tensor, ld: int):
        e = self.entries.get(self.key(t, ld))
        if e is not None and e[0] == t._version:
            return e[1]
        return None

    def drop_shape(self, device, n: int, cols: int) -> None:
        """Forget entries of this shape: called before a new matrix of the same shape is allocated, so that last epoch's
        V (which the caller has usually dropped by then) does not stay resident next to the new one."""
        for k in [k for k in self.entries if k[0] == device.index and k[3] == n and k[4] == cols]:
            del self.entries[k]

    def invalidate(self) -> None:
        self.entries.clear()


PLANES = _PlaneRegistry()


@_on_device
def split_planes(X: torch.Tensor, ldx: int, n: int, cols: int, colsq: bool = False, unit_bound: bool = False) -> Planes:
    lib = _lib.load()
    with _guard(X):
        buf = _workspace(lib.gpp_planes_bytes(n, cols), X.device)
        ws = _workspace(lib.gpp_split_workspace_bytes(n, cols) if colsq else 0, X.device)
        flags = (GPP_PLANES_COLSQ if colsq else 0) | (GPP_PLANES_UNIT_BOUND if unit_bound else 0)
        check(lib.gpp_split_planes(_p(X), ldx, n, cols, flags, _p(buf), buf.numel(), _p(ws), ws.numel(), _stream(X.device)),
              "split_planes")
    return Planes(buf, n, cols, colsq)


def planes_of(V: torch.Tensor, ldv: int) -> Planes:
    """The planes of the dense matrix V (with its column sums of squares): from the registry when V came out of
    Vmodel.forward (or was split before and has not changed since), else split now and remembered."""
    pl = PLANES.get(V, ldv)
    if pl is None:
        pl = split_planes(V, ldv, V.shape[0], V.shape[1], colsq=True)
        PLANES.put(V, ldv, pl)
    return pl


class Stacked:
    """k designs of one evaluation as ONE n x Q operand V = [V_0 | ... | V_{k-1}] (gp.py:27 without the sqrt(v_i)
    weights, which the block-form factorisation applies): the operand planes of V at tensor-core shapes (`planes`,
    written from the k fp32 designs without an fp32 copy of V), else a zero-padded fp32 concatenation (`V`).
    Block i occupies columns [offsets[i], offsets[i] + widths[i]); its first true_widths[i] are design i's columns."""

    def __init__(self, key, n: int, widths, true_widths, planes: Optional[Planes], V: Optional[torch.Tensor]):
        self.key, self.n, self.widths, self.true_widths, self.planes, self.V = key, n, list(widths), list(true_widths), \
            planes, V
        self.offsets = [sum(self.widths[:i]) for i in range(len(self.widths))]
        self.Q = sum(self.widths)


class _StackedRegistry:
    """The stacked operand of the designs used last (one entry), found again by the designs' storage, layout and version.

    The entry refers to the designs through weak references only and is dropped when the first of them dies, so it
    never keeps a design alive, and its planes (4 bytes per element of V) go with last epoch's designs instead of
    staying resident next to the new ones."""

    def __init__(self):
        self.entry: Optional[Stacked] = None
        self._refs = ()

    @staticmethod
    def key(Vs, mats, use_planes: bool):
        return (use_planes,) + tuple((V.device.index, V.untyped_storage().data_ptr(), V.storage_offset(), tuple(V.shape),
                                      tuple(V.stride()), V._version, ld) for V, (_, ld) in zip(Vs, mats))

    def get(self, key) -> Optional[Stacked]:
        e = self.entry
        return e if e is not None and e.key == key else None

    def put(self, Vs, st: Stacked) -> None:
        def drop(_ref, st=st):
            if self.entry is st:
                self.invalidate()
        self.entry = st
        self._refs = tuple(weakref.ref(V, drop) for V in Vs)

    def invalidate(self) -> None:
        self.entry = None
        self._refs = ()


STACKED = _StackedRegistry()


def stacked(Vs, use_planes: bool, before_build=None) -> Stacked:
    """The Stacked operand of the designs Vs (CUDA float32 n x Q_i each, same n): from the registry, or built now (the
    previous entry is dropped first, and `before_build()` is called, so that the caller can release what it holds of
    the previous one: two sets of stacked planes need never coexist)."""
    mats = [as_matrix(V, f"Vs[{i}]") for i, V in enumerate(Vs)]
    n = mats[0][0].shape[0]
    for i, (Vm, _) in enumerate(mats):
        if Vm.shape[0] != n:
            raise ValueError(f"Vs[{i}] has {Vm.shape[0]} rows but Vs[0] has {n}")
        if Vm.device != mats[0][0].device:
            raise ValueError("all designs must be on the same device")
    key = STACKED.key(Vs, mats, use_planes)
    st = STACKED.get(key)
    if st is not None:
        return st
    STACKED.invalidate()
    if before_build is not None:
        before_build()
    widths, true_widths = [Vm.shape[1] for Vm, _ in mats], [V.shape[1] for V in Vs]
    if use_planes:
        st = Stacked(key, n, widths, true_widths, split_planes_stacked(mats, n, colsq=True), None)
    else:
        Vc = torch.zeros(n, sum(widths), device=mats[0][0].device, dtype=torch.float32)
        o = 0
        for V, w in zip(Vs, widths):
            Vc[:, o:o + V.shape[1]] = V.detach()
            o += w
        st = Stacked(key, n, widths, true_widths, None, Vc)
    STACKED.put(Vs, st)
    return st


def split_planes_stacked(mats, n: int, colsq: bool = False, unit_bound: bool = False) -> Planes:
    """Operand planes of [M_0 | M_1 | ...] for mats = [(M_i, ld_i)] (fp32, n rows, widths multiples of 4), written
    directly from the sources with one common scale (gpp_split_planes_stacked)."""
    lib = _lib.load()
    dev = mats[0][0].device
    cols = [M.shape[1] for M, _ in mats]
    k = len(mats)
    with torch.cuda.device(dev):
        buf = _workspace(lib.gpp_planes_bytes(n, sum(cols)), dev)
        c32 = _lib.host_i32(cols)
        ws = _workspace(lib.gpp_split_stacked_workspace_bytes(n, k, c32) if colsq else 0, dev)
        flags = (GPP_PLANES_COLSQ if colsq else 0) | (GPP_PLANES_UNIT_BOUND if unit_bound else 0)
        check(lib.gpp_split_planes_stacked(k, _lib.host_ptrs([M.data_ptr() for M, _ in mats]),
                                           _lib.host_i64([ld for _, ld in mats]), c32, n, flags, _p(buf), buf.numel(),
                                           _p(ws), ws.numel(), _stream(dev)), "split_planes_stacked")
    return Planes(buf, n, sum(cols), colsq)


@_on_device
def khatri_rao_fwd(xn: torch.Tensor, wn: torch.Tensor, d: torch.Tensor, w: torch.Tensor) -> torch.Tensor:
    """V (n x p*q) from row-normalised tables; returns a view with the reference's shape (columns are
    padded internally to a multiple of 4 when p*q is not one, by zero-padding p).  For matrices large enough for the
    tensor-core passes the same sweep also writes V's operand planes (kept in `PLANES` for GP.taylor_coeff)."""
    require_cuda_f32(xn, "xn")
    require_cuda_f32(wn, "wn")
    d = _check_index(d, "d", xn.device)
    w = _check_index(w, "w", xn.device)
    if d.shape != w.shape:
        raise ValueError("d and w must have the same length")
    if d.shape[0] == 0:
        # the reference raises here as well (vmod.py:34 reshapes 0 elements to [0, -1])
        raise ValueError("d and w are empty: there is no row of V to build")
    P, p = xn.shape
    nv, q = wn.shape
    Q = p * q
    xn_k, p_k = xn.detach().contiguous(), p
    if Q % 4:
        p_k = round4(p)
        xn_k = torch.zeros(P, p_k, device=xn.device, dtype=torch.float32)
        xn_k[:, :p] = xn.detach()
    n = d.shape[0]
    lib = _lib.load()
    Qk = p_k * q
    with _guard(xn):
        if p_k == p and planes_supported(n, Qk, 0):
            PLANES.drop_shape(xn.device, n, Qk)
            V = torch.empty(n, Qk, device=xn.device, dtype=torch.float32)
            buf = _workspace(lib.gpp_planes_bytes(n, Qk), xn.device)
            ws = _workspace(lib.gpp_split_workspace_bytes(n, Qk), xn.device)
            check(lib.gpp_khatri_rao_fwd_planes(_p(xn_k), P, p_k, _p(wn.detach().contiguous()), nv, q, _p(d), _p(w), n,
                                                _p(V), Qk, _p(buf), buf.numel(), _p(ws), ws.numel(),
                                                _stream(xn.device)), "khatri_rao_fwd_planes")
            PLANES.put(V, Qk, Planes(buf, n, Qk, True))
            return V
        V = torch.empty(n, Qk, device=xn.device, dtype=torch.float32)
        check(lib.gpp_khatri_rao_fwd(_p(xn_k), P, p_k, _p(wn.detach().contiguous()), nv, q, _p(d), _p(w), n,
                                     _p(V), V.stride(0) if n > 0 else Qk, _stream(xn.device)), "khatri_rao_fwd")
    return V[:, :Q] if p_k != p else V


@_on_device
def khatri_rao_bwd(gV: torch.Tensor, xn: torch.Tensor, wn: torch.Tensor, d: torch.Tensor, w: torch.Tensor
                   ) -> Tuple[torch.Tensor, torch.Tensor]:
    gV = gV.detach()
    n, Q = gV.shape
    # the kernel reads row r at gV + r * ldg with unit column stride: a broadcast upstream gradient (strides (0, 1) for
    # V.sum(0), (0, 0) for V.sum()) or any other overlapping layout is copied first
    if (Q > 1 and gV.stride(1) != 1) or (n > 1 and gV.stride(0) < Q):
        gV = gV.contiguous()
    ldg = gV.stride(0) if n > 1 else Q
    P, p = xn.shape
    nv, q = wn.shape
    # row-major like the kernel's writes, whatever the layout of the tables (zeros_like would keep a transposed one's)
    gxn = torch.zeros(P, p, device=xn.device, dtype=torch.float32)
    gwn = torch.zeros(nv, q, device=wn.device, dtype=torch.float32)
    # held until the launch: a copy passed as `_p(t.contiguous())` is freed before the next argument is built, whose
    # own copy may then take the same block (a transposed xn was read as wn's copy)
    xc, wc, dc, wic = xn.detach().contiguous(), wn.detach().contiguous(), d.contiguous(), w.contiguous()
    check(_lib.load().gpp_khatri_rao_bwd(_p(gV), ldg, _p(xc), P, p, _p(wc), nv, q, _p(dc), _p(wic), d.shape[0], _p(gxn),
                                         _p(gwn), _stream()), "khatri_rao_bwd")
    return gxn, gwn


# ----------------------------------------------------------------------------- GP term
@_on_device
def gram_vtz(V: torch.Tensor, ldv: int, X: Optional[torch.Tensor], ldx: int, n: int, Q: int, L: int) -> torch.Tensor:
    """GC = V^T [V | X]  ->  (Q x (Q+L)) float32."""
    lib = _lib.load()
    GC = torch.empty(Q, Q + L, device=V.device, dtype=torch.float32)
    ws = _workspace(lib.gpp_gram_workspace_bytes(n, Q, L), V.device)
    check(lib.gpp_gram_vtz(_p(V), ldv, _p(X), ldx, n, Q, L, _p(GC), Q + L, _p(ws), ws.numel(), _stream()), "gram_vtz")
    return GC


@_on_device
def gram_vtz_planes(pV: Planes, pX: Optional[Planes], n: int, Q: int, L: int) -> torch.Tensor:
    """GC = V^T [V | X] from operand planes; the diagonal of G is V's exact column sums of squares."""
    lib = _lib.load()
    dev = pV.buf.device
    with torch.cuda.device(dev):
        GC = torch.empty(Q, Q + L, device=dev, dtype=torch.float32)
        ws = _workspace(lib.gpp_gram_planes_workspace_bytes(n, Q, L), dev)
        check(lib.gpp_gram_vtz_planes(pV.ptr, pX.ptr if pX is not None else None, n, Q, L, int(pV.colsq), _p(GC), Q + L,
                                      _p(ws), ws.numel(), _stream(dev)), "gram_vtz_planes")
    return GC


@_on_device
def atb_planes(pA: Planes, pB: Planes, n: int, ka: int, kb: int, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """A^T B (ka x kb) from operand planes, into `out` when given (a ka x kb view; its row stride is the ld)."""
    lib = _lib.load()
    dev = pA.buf.device
    with torch.cuda.device(dev):
        if out is None:
            out = torch.empty(ka, kb, device=dev, dtype=torch.float32)
        ws = _workspace(lib.gpp_gram_planes_workspace_bytes(n, ka, kb), dev)
        check(lib.gpp_atb_planes(pA.ptr, pB.ptr, n, ka, kb, _p(out), out.stride(0), _p(ws), ws.numel(), _stream(dev)),
              "atb_planes")
    return out


@_on_device
def xb_nll_planes(pV: Planes, X, ldx, W, n, Q, L, scal) -> Tuple[torch.Tensor, torch.Tensor]:
    lib = _lib.load()
    dev = X.device
    with torch.cuda.device(dev):
        Xb = torch.empty(n, L, device=dev, dtype=torch.float32)
        nll = torch.empty(n, 1, device=dev, dtype=torch.float32)
        ws = _workspace(lib.gpp_xb_planes_workspace_bytes(n, Q, L), dev)
        check(lib.gpp_xb_nll_planes(pV.ptr, _p(X), ldx, _p(W), W.stride(0), n, Q, L, _p(scal), _p(Xb), L, _p(nll), _p(ws),
                                    ws.numel(), _stream(dev)), "xb_nll_planes")
    return Xb, nll


@_on_device
def vb_planes(pV: Planes, Xb, Binv, W, scal, n, Q, L, L_true) -> torch.Tensor:
    lib = _lib.load()
    Vb = torch.empty(n, Q, device=Xb.device, dtype=torch.float32)
    ws = _workspace(lib.gpp_vb_planes_workspace_bytes(n, Q, L), Xb.device)
    check(lib.gpp_vb_planes(pV.ptr, _p(Xb), Xb.stride(0), _p(Binv), _p(W), W.stride(0), _p(scal), n, Q, L, L_true, _p(Vb), Q,
                            _p(ws), ws.numel(), _stream()), "vb_planes")
    return Vb


@_on_device
def atb(A: torch.Tensor, lda: int, B: torch.Tensor, ldb: int, n: int, ka: int, kb: int) -> torch.Tensor:
    lib = _lib.load()
    out = torch.empty(ka, kb, device=A.device, dtype=torch.float32)
    ws = _workspace(lib.gpp_atb_workspace_bytes(n, ka, kb), A.device)
    check(lib.gpp_atb(_p(A), lda, _p(B), ldb, n, ka, kb, _p(out), kb, _p(ws), ws.numel(), _stream()), "atb")
    return out


class Factorisation:
    """State left by gpp_factor: Lc and Linv inside `state`, the scalar block, optionally Binv.  Block form
    (gpp_factor_blocks): `widths` are the designs' column counts, `blk` the per-block scalars, Binv = D B^-1 D."""

    def __init__(self, Q: int, state: torch.Tensor, scal: torch.Tensor, Binv: Optional[torch.Tensor],
                 widths=None, blk: Optional[torch.Tensor] = None):
        self.Q, self.state, self.scal, self.Binv, self.widths, self.blk = Q, state, scal, Binv, widths, blk


@_on_device
def factor(G: torch.Tensor, ldg: int, Q: int, vs: torch.Tensor, want_binv: bool) -> Factorisation:
    lib = _lib.load()
    dev = G.device
    state = _workspace(lib.gpp_factor_state_bytes(Q), dev)
    scal = torch.zeros(NSCAL, device=dev, dtype=torch.float64)
    Binv = torch.empty(Q, Q, device=dev, dtype=torch.float32) if want_binv else None
    vs32 = vs.detach().to(torch.float32).contiguous()
    check(lib.gpp_factor(_p(G), ldg, Q, _p(vs32), GPP_WANT_BINV if want_binv else 0, _p(Binv), _p(scal), _p(state),
                         state.numel(), _stream()), "factor")
    return Factorisation(Q, state, scal, Binv)


@_on_device
def solve_w(f: Factorisation, C: torch.Tensor, ldc: int, L: int, L_true: int, n_total: int
            ) -> Tuple[torch.Tensor, torch.Tensor]:
    """W = (v0/vn) B^-1 C and a private copy of the scalar block extended with WNORM2 / ROWCONST."""
    lib = _lib.load()
    W = torch.empty(f.Q, L, device=C.device, dtype=torch.float32)
    scal = f.scal.clone()
    ws = _workspace(lib.gpp_solve_workspace_bytes(f.Q, L), C.device)
    check(lib.gpp_solve_w(_p(C), ldc, f.Q, L, L_true, n_total, _p(W), L, _p(scal), _p(f.state), f.state.numel(),
                          _p(ws), ws.numel(), _stream()), "solve_w")
    return W, scal


@_on_device
def factor_blocks(G: torch.Tensor, ldg: int, widths, vs: torch.Tensor, want_binv: bool) -> Factorisation:
    """gpp_factor_blocks: B = I + D G D / vn for the stacked designs of column counts `widths`."""
    lib = _lib.load()
    dev = G.device
    Q, k = sum(widths), len(widths)
    state = _workspace(lib.gpp_factor_blocks_state_bytes(Q, k), dev)
    scal = torch.zeros(NSCAL, device=dev, dtype=torch.float64)
    blk = torch.zeros(2 * k, device=dev, dtype=torch.float64)
    Binv = torch.empty(Q, Q, device=dev, dtype=torch.float32) if want_binv else None
    vs32 = vs.detach().to(torch.float32).contiguous()
    check(lib.gpp_factor_blocks(_p(G), ldg, k, _lib.host_i32(widths), _p(vs32), GPP_WANT_BINV if want_binv else 0,
                                _p(Binv), _p(scal), _p(blk), _p(state), state.numel(), _stream()), "factor_blocks")
    return Factorisation(Q, state, scal, Binv, list(widths), blk)


@_on_device
def solve_w_blocks(f: Factorisation, C: torch.Tensor, ldc: int, L: int, L_true: int, n_total: int
                   ) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """W = D B^-1 D C / vn and private copies of the scalar block and of the per-block scalars (||W_i||^2 added)."""
    lib = _lib.load()
    k = len(f.widths)
    W = torch.empty(f.Q, L, device=C.device, dtype=torch.float32)
    scal, blk = f.scal.clone(), f.blk.clone()
    ws = _workspace(lib.gpp_solve_blocks_workspace_bytes(f.Q, L, k), C.device)
    check(lib.gpp_solve_w_blocks(_p(C), ldc, k, _lib.host_i32(f.widths), L, L_true, n_total, _p(W), L, _p(scal), _p(blk),
                                 _p(f.state), f.state.numel(), _p(ws), ws.numel(), _stream()), "solve_w_blocks")
    return W, scal, blk


@_on_device
def vbs_blocks(scal: torch.Tensor, blk: torch.Tensor, vs: torch.Tensor, widths, n_total: int, L: int) -> torch.Tensor:
    """vbs = dNLL/d[v_0 .. v_{k-1}, vn] (k + 1 entries)."""
    k = len(widths)
    out = torch.empty(k + 1, device=scal.device, dtype=torch.float32)
    vs32 = vs.detach().to(torch.float32).contiguous()
    check(_lib.load().gpp_vbs_blocks(_p(scal), _p(blk), _p(vs32), k, _lib.host_i32(widths), n_total, L, _p(out),
                                     _stream()), "vbs_blocks")
    return out


@_on_device
def xb_nll(V, ldv, X, ldx, W, n, Q, L, scal) -> Tuple[torch.Tensor, torch.Tensor]:
    lib = _lib.load()
    Xb = torch.empty(n, L, device=V.device, dtype=torch.float32)
    nll = torch.empty(n, 1, device=V.device, dtype=torch.float32)
    ws = _workspace(lib.gpp_xb_workspace_bytes(n, Q, L), V.device)
    check(lib.gpp_xb_nll(_p(V), ldv, _p(X), ldx, _p(W), W.stride(0), n, Q, L, _p(scal), _p(Xb), L, _p(nll), _p(ws),
                         ws.numel(), _stream()), "xb_nll")
    return Xb, nll


@_on_device
def vbs_from_scal(scal: torch.Tensor, n_total: int, Q: int, L: int) -> torch.Tensor:
    out = torch.empty(2, device=scal.device, dtype=torch.float32)
    check(_lib.load().gpp_vbs(_p(scal), n_total, Q, L, _p(out), _stream()), "vbs")
    return out


@_on_device
def vb(V, ldv, Xb, Binv, W, scal, n, Q, L, L_true) -> torch.Tensor:
    lib = _lib.load()
    Vb = torch.empty(n, Q, device=V.device, dtype=torch.float32)
    ws = _workspace(lib.gpp_vb_workspace_bytes(n, Q, L), V.device)
    check(lib.gpp_vb(_p(V), ldv, _p(Xb), Xb.stride(0), _p(Binv), _p(W), W.stride(0), _p(scal), n, Q, L,
                     L_true, _p(Vb), Q, _p(ws), ws.numel(), _stream()), "vb")
    return Vb


@_on_device
def x_minus_am(X, ldx, A, lda, M, ldm, n, k, m, alpha: float) -> torch.Tensor:
    out = torch.empty(n, m, device=X.device, dtype=torch.float32)
    ws = _workspace(256, X.device)
    check(_lib.load().gpp_x_minus_am(_p(X), ldx, _p(A), lda, _p(M), ldm, n, k, m, float(alpha), _p(out), m, _p(ws),
                                     ws.numel(), _stream()), "x_minus_am")
    return out


@_on_device
def am(A: torch.Tensor, lda: int, M: torch.Tensor, ldm: int, n: int, k: int, m: int, alpha: float = 1.0) -> torch.Tensor:
    """out = alpha * A M  (n x m)."""
    out = torch.empty(n, m, device=A.device, dtype=torch.float32)
    ws = _workspace(256, A.device)
    check(_lib.load().gpp_am(_p(A), lda, _p(M), ldm, n, k, m, float(alpha), _p(out), m, _p(ws), ws.numel(), _stream()), "am")
    return out


# ----------------------------------------------------------------------------- structured Khatri-Rao path
@_on_device
def kr_slot_sums(X: torch.Tensor, ldx: int, order: torch.Tensor, slot_start: torch.Tensor, xn: torch.Tensor,
                 nviews: int, L: int, with_x: bool) -> torch.Tensor:
    """XZ (P x nviews (p + L)) = [cnt (x) xn | per-slot sums of X]  (with_x=False: the X part alone)."""
    P, p = xn.shape
    XZ = torch.empty(P, nviews * ((p if with_x else 0) + L), device=X.device, dtype=torch.float32)
    check(_lib.load().gpp_kr_slot_sums(_p(X), ldx, _p(order), _p(slot_start), _p(xn), P, p, nviews, L, int(with_x),
                                       _p(XZ), XZ.stride(0), _stream()), "kr_slot_sums")
    return XZ


@_on_device
def kr_slot_sums_planes(X: torch.Tensor, ldx: int, order: torch.Tensor, slot_start: torch.Tensor, xn: torch.Tensor,
                        nviews: int, L: int, with_x: int, max_count: int) -> Planes:
    """The matrix of `kr_slot_sums` written directly as operand planes (no fp32 copy, no scan of it).  with_x = 2:
    the cnt (x) xn part alone, under its own scale (include/gppvae_b200.h)."""
    lib = _lib.load()
    P, p = xn.shape
    cols = nviews * (p if with_x == 2 else (p if with_x else 0) + L)
    with _guard(X):
        buf = _workspace(lib.gpp_planes_bytes(P, cols), X.device)
        check(lib.gpp_kr_slot_sums_planes(_p(X), ldx, X.shape[0], _p(order), _p(slot_start), _p(xn), P, p, nviews, L,
                                          int(with_x), int(max_count), _p(buf), buf.numel(), _stream(X.device)),
              "kr_slot_sums_planes")
    return Planes(buf, P, cols, False)


@_on_device
def am_planes(pA: Planes, pM: Planes, n: int, k: int, m: int, alpha: float = 1.0) -> torch.Tensor:
    """out (n x m) = alpha A M from operand planes."""
    lib = _lib.load()
    dev = pA.buf.device
    with torch.cuda.device(dev):
        out = torch.empty(n, m, device=dev, dtype=torch.float32)
        ws = _workspace(256, dev)
        check(lib.gpp_am_planes(pA.ptr, pM.ptr, n, k, m, float(alpha), _p(out), m, _p(ws), ws.numel(), _stream(dev)),
              "am_planes")
    return out


@_on_device
def kr_assemble_gc(ST: torch.Tensor, wn: torch.Tensor, p: int, L: int, with_g: bool) -> torch.Tensor:
    nv, q = wn.shape
    Q = p * q
    GC = torch.empty(Q, (Q if with_g else 0) + L, device=ST.device, dtype=torch.float32)
    check(_lib.load().gpp_kr_assemble_gc(_p(ST), ST.stride(0), _p(wn), p, q, nv, L, int(with_g), _p(GC), GC.stride(0),
                                         _stream()), "kr_assemble_gc")
    return GC


@_on_device
def kr_assemble_m(W: torch.Tensor, wn: torch.Tensor, p: int, L: int) -> torch.Tensor:
    nv, q = wn.shape
    M = torch.empty(p, nv * L, device=W.device, dtype=torch.float32)
    check(_lib.load().gpp_kr_assemble_m(_p(W), W.stride(0), _p(wn), p, q, nv, L, _p(M), M.stride(0), _stream()),
          "kr_assemble_m")
    return M


@_on_device
def kr_xb_nll(X: torch.Tensor, ldx: int, Y: torch.Tensor, d: torch.Tensor, w: torch.Tensor, P: int, nviews: int,
              L: int, scal: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    lib = _lib.load()
    n = X.shape[0]
    Xb = torch.empty(n, L, device=X.device, dtype=torch.float32)
    nll = torch.empty(n, 1, device=X.device, dtype=torch.float32)
    ws = _workspace(lib.gpp_kr_xb_workspace_bytes(n), X.device)
    check(lib.gpp_kr_xb_nll(_p(X), ldx, _p(Y), Y.stride(0), _p(d), _p(w), n, P, nviews, L, _p(scal), _p(Xb), L, _p(nll),
                            _p(ws), ws.numel(), _stream()), "kr_xb_nll")
    return Xb, nll


@_on_device
def kr_grad_rhs(Binv: torch.Tensor, W: torch.Tensor, wn: torch.Tensor, p: int, L: int, alpha: float) -> torch.Tensor:
    """R (nviews (p + L) x p) = [alpha H_0; ..; alpha H_{nv-1}; -M_0^T; ..; -M_{nv-1}^T]: gxn = [cnt (x) xn | Xb sums] R."""
    nv, q = wn.shape
    R = torch.empty(nv * (p + L), p, device=W.device, dtype=torch.float32)
    check(_lib.load().gpp_kr_grad_rhs(_p(Binv), Binv.stride(0), _p(W), W.stride(0), _p(wn), p, q, nv, L, float(alpha),
                                      _p(R), R.stride(0), _stream()), "kr_grad_rhs")
    return R


@_on_device
def kr_grad_views(ST: torch.Tensor, Binv: torch.Tensor, W: torch.Tensor, wn: torch.Tensor, p: int, L: int,
                  alpha: float) -> torch.Tensor:
    """The NLL gradient to the normalised view table (nviews x q) from ST = xn^T [cnt (x) xn | slot sums of Xb]."""
    lib = _lib.load()
    nv, q = wn.shape
    gw = torch.empty(nv, q, device=W.device, dtype=torch.float32)
    ws = _workspace(lib.gpp_kr_grad_views_workspace_bytes(p, q, nv), W.device)
    check(lib.gpp_kr_grad_views(_p(ST), ST.stride(0), _p(Binv), Binv.stride(0), _p(W), W.stride(0), _p(wn), p, q, nv, L,
                                float(alpha), _p(gw), gw.stride(0), _p(ws), ws.numel(), _stream()), "kr_grad_views")
    return gw


# ----------------------------------------------------------------------------- several factored designs
@_on_device
def kr_view_sums(X: torch.Tensor, ldx: int, order: torch.Tensor, slot_start: torch.Tensor, xn: torch.Tensor,
                 nviews: int, L: int, with_x: bool) -> torch.Tensor:
    """VM (nviews x (L + (p + 4 if with_x))): rows [z_v | a_v | n_v, 0, 0, 0], the per-view first moments."""
    lib = _lib.load()
    P, p = xn.shape
    VM = torch.empty(nviews, L + (p + 4 if with_x else 0), device=X.device, dtype=torch.float32)
    ws = _workspace(lib.gpp_kr_view_sums_workspace_bytes(P, p, nviews, L, int(with_x)), X.device)
    check(lib.gpp_kr_view_sums(_p(X), ldx, _p(order), _p(slot_start), _p(xn), P, p, nviews, L, int(with_x), _p(VM),
                               VM.stride(0), _p(ws), ws.numel(), _stream()), "kr_view_sums")
    return VM


def effect_widths(kinds, p: int, q: int):
    """Block widths of the stacked factored designs (p already a multiple of 4)."""
    return [p * q if k == "kr" else p if k == "object" else round4(q) for k in kinds]


@_on_device
def kr_assemble_gc_blocks(ST: Optional[torch.Tensor], VM: Optional[torch.Tensor], wn: torch.Tensor, p: int, kinds,
                          L: int, with_g: bool) -> torch.Tensor:
    """The stacked GC = V^T [V | X] (with_g) or C = V^T X of the factored designs `kinds`, from ST and VM."""
    nv, q = wn.shape
    Q = sum(effect_widths(kinds, p, q))
    dev = wn.device
    GC = torch.empty(Q, (Q if with_g else 0) + L, device=dev, dtype=torch.float32)
    check(_lib.load().gpp_kr_assemble_gc_blocks(_p(ST), ST.stride(0) if ST is not None else 0, _p(VM),
                                                VM.stride(0) if VM is not None else 0, _p(wn), p, q, nv, L, len(kinds),
                                                _lib.host_i32([EFFECT_KINDS[k] for k in kinds]), int(with_g), _p(GC),
                                                GC.stride(0), _stream()), "kr_assemble_gc_blocks")
    return GC


@_on_device
def kr_assemble_m_blocks(W: torch.Tensor, wn: torch.Tensor, p: int, kinds, L: int
                         ) -> Tuple[Optional[torch.Tensor], Optional[torch.Tensor]]:
    """(M, R): M (p x nviews L) with W_O folded in, None without K and O; R (nviews x L), None without W."""
    nv, q = wn.shape
    M = torch.empty(p, nv * L, device=W.device, dtype=torch.float32) if ("kr" in kinds or "object" in kinds) else None
    R = torch.empty(nv, L, device=W.device, dtype=torch.float32) if "view" in kinds else None
    check(_lib.load().gpp_kr_assemble_m_blocks(_p(W), W.stride(0), _p(wn), p, q, nv, L, len(kinds),
                                               _lib.host_i32([EFFECT_KINDS[k] for k in kinds]), _p(M),
                                               M.stride(0) if M is not None else 0, _p(R),
                                               R.stride(0) if R is not None else 0, _stream()), "kr_assemble_m_blocks")
    return M, R


@_on_device
def kr_xb_nll_views(X: torch.Tensor, ldx: int, Y: torch.Tensor, R: torch.Tensor, d: torch.Tensor, w: torch.Tensor,
                    P: int, nviews: int, L: int, scal: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    lib = _lib.load()
    n = X.shape[0]
    Xb = torch.empty(n, L, device=X.device, dtype=torch.float32)
    nll = torch.empty(n, 1, device=X.device, dtype=torch.float32)
    ws = _workspace(lib.gpp_kr_xb_workspace_bytes(n), X.device)
    check(lib.gpp_kr_xb_nll_views(_p(X), ldx, _p(Y), Y.stride(0), _p(R), R.stride(0), _p(d), _p(w), n, P, nviews, L,
                                  _p(scal), _p(Xb), L, _p(nll), _p(ws), ws.numel(), _stream()), "kr_xb_nll_views")
    return Xb, nll


# ----------------------------------------------------------------------------- posterior prediction (GP.predict)
@_on_device
def kr_predict_views(Binv: torch.Tensor, wn: torch.Tensor, p: int, kinds
                     ) -> Tuple[Optional[torch.Tensor], Optional[torch.Tensor], Optional[torch.Tensor]]:
    """(H, h, c) of the factored designs `kinds`: H = [H_0 | ..] (p x nviews p, None without K and O), h (nviews x p)
    and c (nviews), both None without W (include/gppvae_b200.h, gpp_kr_predict_views)."""
    nv, q = wn.shape
    dev = wn.device
    H = torch.empty(p, nv * p, device=dev, dtype=torch.float32) if ("kr" in kinds or "object" in kinds) else None
    h = torch.empty(nv, p, device=dev, dtype=torch.float32) if "view" in kinds else None
    c = torch.empty(nv, device=dev, dtype=torch.float32) if "view" in kinds else None
    check(_lib.load().gpp_kr_predict_views(_p(Binv), Binv.stride(0), _p(wn), p, q, nv, len(kinds),
                                           _lib.host_i32([EFFECT_KINDS[k] for k in kinds]), _p(H),
                                           H.stride(0) if H is not None else 0, _p(h), _p(c), _stream()),
          "kr_predict_views")
    return H, h, c


@_on_device
def kr_predict_rows(Y: Optional[torch.Tensor], R: Optional[torch.Tensor], YH: Optional[torch.Tensor], xn: torch.Tensor,
                    h: Optional[torch.Tensor], c: Optional[torch.Tensor], d: torch.Tensor, w: torch.Tensor, P: int,
                    nviews: int, L: int, scal: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """(mean (m x L), var (m x 1)) of the new rows (d, w) from the P-long products Y = xn M and YH = xn H."""
    m, p = d.shape[0], xn.shape[1]
    mean = torch.empty(m, L, device=d.device, dtype=torch.float32)
    var = torch.empty(m, 1, device=d.device, dtype=torch.float32)
    check(_lib.load().gpp_kr_predict_rows(_p(Y), Y.stride(0) if Y is not None else 0, _p(R),
                                          R.stride(0) if R is not None else 0, _p(YH),
                                          YH.stride(0) if YH is not None else 0, _p(xn), _p(h), _p(c), _p(d), _p(w), m, P,
                                          p, nviews, L, _p(scal), _p(mean), L, _p(var), _stream()), "kr_predict_rows")
    return mean, var


@_on_device
def rows_dot(A: torch.Tensor, B: torch.Tensor, cols: int, scal: torch.Tensor) -> torch.Tensor:
    """out (m x 1) = scal[V0] * sum_c A[:, c] B[:, c] over the first `cols` columns."""
    m = A.shape[0]
    out = torch.empty(m, 1, device=A.device, dtype=torch.float32)
    check(_lib.load().gpp_rows_dot(_p(A), A.stride(0), _p(B), B.stride(0), m, cols, _p(scal), _p(out), _stream()),
          "rows_dot")
    return out


# ----------------------------------------------------------------------------- autograd glue
class _NormalizeRows(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        ctx.save_for_backward(x)
        return normalize_rows_fwd(x)

    @staticmethod
    def backward(ctx, gy):
        (x,) = ctx.saved_tensors
        return normalize_rows_bwd(x, gy)


class _KhatriRao(torch.autograd.Function):
    @staticmethod
    def forward(ctx, xn, wn, d, w):
        ctx.save_for_backward(xn, wn, d, w)
        return khatri_rao_fwd(xn, wn, d, w)

    @staticmethod
    def backward(ctx, gV):
        xn, wn, d, w = ctx.saved_tensors
        gxn, gwn = khatri_rao_bwd(gV, xn, wn, d, w)
        return gxn, gwn, None, None


class _TaylorExpansion(torch.autograd.Function):
    """gp.py:127-133 as one fused forward and one fused backward launch."""

    @staticmethod
    def forward(ctx, X, V, lvs, Xb, Vb, vbs):
        lib = _lib.load()
        Xm, ldx = as_matrix(X, "X")
        Xbm, ldxb = as_matrix(Xb, "Xb")
        n, L = X.shape
        Lk = Xm.shape[1]
        if V is not None:
            Vm, ldv = as_matrix(V, "V")
            Vbm, ldvb = as_matrix(Vb, "Vb")
            Qk = Vm.shape[1]
        else:
            Vm = Vbm = None
            ldv = ldvb = 4
            Qk = 0
        vbs32 = vbs.detach().to(torch.float32).contiguous()
        lvs32 = lvs.detach().to(torch.float32).contiguous()
        out = torch.empty(n, 1, device=X.device, dtype=torch.float32)
        check(lib.gpp_taylor_expansion_fwd(_p(Xm), ldx, _p(Xbm), ldxb, _p(Vm), ldv, _p(Vbm), ldvb, n, Lk, Qk,
                                           _p(vbs32), _p(lvs32), _p(out), _stream()), "taylor_expansion_fwd")
        ctx.save_for_backward(Xbm, Vbm, vbs32, lvs32)
        ctx.dims = (n, L, Lk, ldxb, (V.shape[1] if V is not None else 0), Qk, ldvb)
        return out

    @staticmethod
    def backward(ctx, gout):
        lib = _lib.load()
        Xbm, Vbm, vbs32, lvs32 = ctx.saved_tensors
        n, L, Lk, ldxb, Q, Qk, ldvb = ctx.dims
        g = gout.detach().to(torch.float32).contiguous().view(-1)
        need_x, need_v, need_l = ctx.needs_input_grad[0], ctx.needs_input_grad[1] and Vbm is not None, \
            ctx.needs_input_grad[2]
        gX = torch.empty(n, Lk, device=g.device, dtype=torch.float32) if need_x else None
        gV = torch.empty(n, Qk, device=g.device, dtype=torch.float32) if need_v else None
        gl = torch.empty(2, device=g.device, dtype=torch.float32) if need_l else None
        check(lib.gpp_taylor_expansion_bwd(_p(g), _p(Xbm), ldxb, _p(Vbm), ldvb, n, Lk, Qk, _p(vbs32), _p(lvs32),
                                           _p(gX), Lk, _p(gV), max(Qk, 4), _p(gl), _stream()), "taylor_expansion_bwd")
        return (gX[:, :L] if need_x and Lk != L else gX, gV[:, :Q] if need_v and Qk != Q else gV, gl, None, None, None)


class _TaylorExpansionMulti(torch.autograd.Function):
    """gp.py:127-133 over k designs (k + 1 variances) as one fused forward and one fused backward launch.
    apply(X, lvs, Xb, vbs, V_0 .. V_{k-1}, Vb_0 .. Vb_{k-1})."""

    @staticmethod
    def forward(ctx, X, lvs, Xb, vbs, *VVb):
        lib = _lib.load()
        k = len(VVb) // 2
        Xm, ldx = as_matrix(X, "X")
        Xbm, ldxb = as_matrix(Xb, "Xb")
        n, L = X.shape
        Lk = Xm.shape[1]
        Vm = [as_matrix(V, f"Vs[{j}]") for j, V in enumerate(VVb[:k])]
        Vbm = [as_matrix(Vb, f"Vbs[{j}]") for j, Vb in enumerate(VVb[k:])]
        for j in range(k):
            if VVb[j].shape != VVb[k + j].shape:
                raise ValueError(f"Vs[{j}] is {tuple(VVb[j].shape)} but Vbs[{j}] is {tuple(VVb[k + j].shape)}")
        Qk = [M.shape[1] for M, _ in Vm]
        vbs32 = vbs.detach().to(torch.float32).contiguous()
        lvs32 = lvs.detach().to(torch.float32).contiguous()
        if vbs32.numel() != k + 1 or lvs32.numel() != k + 1:
            raise ValueError(f"vbs and lvs must have {k + 1} entries for {k} designs")
        out = torch.empty(n, 1, device=X.device, dtype=torch.float32)
        check(lib.gpp_taylor_expansion_fwd_multi(_p(Xm), ldx, _p(Xbm), ldxb, k, _lib.host_ptrs([_p(M) for M, _ in Vm]),
                                                 _lib.host_i64([ld for _, ld in Vm]),
                                                 _lib.host_ptrs([_p(M) for M, _ in Vbm]),
                                                 _lib.host_i64([ld for _, ld in Vbm]), _lib.host_i32(Qk), n, Lk, _p(vbs32),
                                                 _p(lvs32), _p(out), _stream()), "taylor_expansion_fwd_multi")
        ctx.save_for_backward(Xbm, vbs32, lvs32, *[M for M, _ in Vbm])
        ctx.dims = (n, L, Lk, ldxb, [V.shape[1] for V in VVb[:k]], Qk, [ld for _, ld in Vbm])
        return out

    @staticmethod
    def backward(ctx, gout):
        lib = _lib.load()
        Xbm, vbs32, lvs32, *Vbm = ctx.saved_tensors
        n, L, Lk, ldxb, Qt, Qk, ldvb = ctx.dims
        k = len(Vbm)
        g = gout.detach().to(torch.float32).contiguous().view(-1)
        need_x, need_l = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        need_v = ctx.needs_input_grad[4:4 + k]
        gX = torch.empty(n, Lk, device=g.device, dtype=torch.float32) if need_x else None
        gV = [torch.empty(n, Qk[j], device=g.device, dtype=torch.float32) if need_v[j] else None for j in range(k)]
        gl = torch.empty(k + 1, device=g.device, dtype=torch.float32) if need_l else None
        check(lib.gpp_taylor_expansion_bwd_multi(_p(g), _p(Xbm), ldxb, k, _lib.host_ptrs([_p(M) for M in Vbm]),
                                                 _lib.host_i64(ldvb), _lib.host_i32(Qk), n, Lk, _p(vbs32), _p(lvs32),
                                                 _p(gX), Lk, _lib.host_ptrs([_p(t) for t in gV]),
                                                 _lib.host_i64(Qk), _p(gl), _stream()), "taylor_expansion_bwd_multi")
        gX = gX[:, :L] if need_x and Lk != L else gX
        gV = [t[:, :Qt[j]] if t is not None and Qk[j] != Qt[j] else t for j, t in enumerate(gV)]
        return (gX, gl, None, None, *gV, *([None] * k))


def normalize_rows(x: torch.Tensor) -> torch.Tensor:
    """vmod.py:10-12 with autograd (forward and backward are CUDA kernels of this library)."""
    require_cuda_f32(x, "x")
    return _NormalizeRows.apply(x)
