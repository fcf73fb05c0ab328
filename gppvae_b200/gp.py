"""Drop-in `GP` module: the reference's gp.py API on top of the sm_100a kernels.

Same class name, constructor, parameter (`lvs`), method names, argument order, shapes and detach
semantics as /root/reference/pysrc/faceplace/gp.py:11-133, so `from gppvae_b200 import GP` can stand
where `from gp import GP` stood in train_gppvae.py:11.  Underneath, the reference's op sequence
(U, B = U^T U + I, svd, inverse, U B^-1, two GEMMs per solve) is replaced by the Q-space algorithm of
SURVEY.md section 7.2:

    pass 1    GC = V^T [V | X]                       gpp_gram_vtz     (+ NCCL all-reduce when sharded)
    factor    B = I + (v0/vn) G = Lc Lc^T, Linv      gpp_factor       (cached, see `_FactorCache`)
    solve     W = (v0/vn) B^-1 C                     gpp_solve_w
    pass 2    Xb = (X - V W)/vn, nll, sum Xb^2       gpp_xb_nll
    extras    vbs, Vb                                gpp_vbs, gpp_vb

Row sharding: construct with `process_group=` (or call `shard_rows(group)`); X and V are then this
rank's rows, GC and sum Xb^2 are all-reduced over the group and every rank holds identical W.
"""
from __future__ import annotations

import weakref
from typing import List, Optional, Sequence, Tuple

import torch
import torch.nn.functional as F
from torch import nn

from . import ops
from ._lib import GPP_MAX_DESIGNS, S_QUAD, S_V0, S_VN, S_XB2
from .vmod import KhatriRao, _FactoredEffect, effect_base, effect_kind, effects_c, effects_st_vm


class LowRankFactor:
    """What `GP.U_UBi_Shb` returns in place of the reference's dense `U` and `UBi` (gp.py:24-38).

    The reference materialises two extra N x Q tensors only to hand them back to `GP.solve`
    (train_gppvae.py:235-236).  This handle carries V, vs and the factorisation instead; `dense()`
    materialises the reference tensor on request.
    """

    def __init__(self, kind: str, V: torch.Tensor, ldv: int, Q: int, Qtrue: int, vs: torch.Tensor,
                 fac: ops.Factorisation):
        self.kind, self.V, self.ldv, self.Q, self.Qtrue, self.vs, self.fac = kind, V, ldv, Q, Qtrue, vs, fac
        self.n = V.shape[0]
        self.shape = torch.Size((self.n, Qtrue))

    def dense(self) -> torch.Tensor:
        vs = self.vs.detach()
        r = torch.sqrt(vs[0] / vs[-1])
        if self.kind == "U":
            return r * self.V[:, : self.Qtrue]
        if self.fac.Binv is None:
            raise RuntimeError("UBi.dense() needs B^-1: call GP.U_UBi_Shb(Vs, vs, want_binv=True)")
        zeros = torch.zeros(self.n, self.Q, device=self.V.device, dtype=torch.float32)
        VB = ops.x_minus_am(zeros, self.Q, self.V, self.ldv, self.fac.Binv, self.Q, self.n, self.Q, self.Q, -1.0)
        return r * VB[:, : self.Qtrue]


class BlocksFactor(LowRankFactor):
    """`U` / `UBi` of `GP.U_UBi_Shb` for k >= 2 designs: carries the designs, their stacked operand (ops.Stacked) and the
    block-form factorisation (Binv = D B^-1 D, D = diag(sqrt(v_i)) on block i)."""

    def __init__(self, kind: str, Vs, stk: ops.Stacked, vs: torch.Tensor, fac: ops.Factorisation):
        self.kind, self.Vs, self.stk, self.vs, self.fac = kind, list(Vs), stk, vs, fac
        self.Q = stk.Q
        self.n = stk.n
        self.shape = torch.Size((self.n, sum(stk.true_widths)))

    def dense(self) -> torch.Tensor:
        """The reference's U = [sqrt(v_i) V_i] / sqrt(vn) (gp.py:27-28) or UBi = U B^-1 (gp.py:35-36)."""
        vs = self.vs.detach()
        sq = torch.sqrt(vs[:-1] / vs[-1])
        if self.kind == "U":
            return torch.cat([sq[i] * V.detach() for i, V in enumerate(self.Vs)], 1)
        if self.fac.Binv is None:
            raise RuntimeError("UBi.dense() needs B^-1: call GP.U_UBi_Shb(Vs, vs, want_binv=True)")
        Vc = torch.zeros(self.n, self.Q, device=vs.device, dtype=torch.float32)
        for o, V in zip(self.stk.offsets, self.Vs):
            Vc[:, o:o + V.shape[1]] = V.detach()
        # V (D B^-1 D) D^-1 / sqrt(vn) = U B^-1 on the true columns
        VB = ops.x_minus_am(torch.zeros_like(Vc), self.Q, Vc, self.Q, self.fac.Binv, self.Q, self.n, self.Q, self.Q, -1.0)
        return torch.cat([VB[:, o:o + V.shape[1]] / torch.sqrt(vs[i] * vs[-1])
                          for i, (o, V) in enumerate(zip(self.stk.offsets, self.Vs))], 1)


class EffectsFactor(BlocksFactor):
    """`U` / `UBi` of `GP.U_UBi_Shb` for k factored designs (Vmodel.lazy_effects): carries the designs, their block
    layout (an ops.Stacked without operand) and the block-form factorisation; `GP.solve` takes the structured route with
    it.  `dense()` goes through the designs' dense()."""

    def dense(self) -> torch.Tensor:
        return BlocksFactor(self.kind, [V.dense() for V in self.Vs], self.stk, self.vs, self.fac).dense()


class KhatriRaoFactor:
    """`U` / `UBi` of `GP.U_UBi_Shb` when V was given in factored form (vmod.KhatriRao): carries the factors and the
    factorisation; `GP.solve` takes the structured route with it.  `dense()` goes through the dense handle."""

    def __init__(self, kind: str, kr: KhatriRao, vs: torch.Tensor, fac: ops.Factorisation):
        self.kind, self.kr, self.vs, self.fac = kind, kr, vs, fac
        self.n = kr.n
        self.shape = kr.shape

    def dense(self) -> torch.Tensor:
        Vm, ldv = ops.as_matrix(self.kr.dense(), "V")
        if Vm.shape[1] != self.fac.Q:       # p was padded to a multiple of 4: the extra columns of V are zero
            Vp = torch.zeros(self.n, self.fac.Q, device=Vm.device, dtype=torch.float32)
            Vp[:, : Vm.shape[1]] = Vm
            Vm, ldv = Vp, self.fac.Q
        return LowRankFactor(self.kind, Vm, ldv, self.fac.Q, self.shape[1], self.vs, self.fac).dense()


class LazyVb:
    """`Vbs[0] = dNLL/dV` (gp.py:68-71) of a structured evaluation: an N x Q matrix nobody needs whole -- the trainer only
    gathers minibatch rows from it (train_gppvae.py:283).  `[idx]` computes those rows, r L V[idx] B^-1 - Xb[idx] W^T."""

    def __init__(self, kr: KhatriRao, Xb, fac, W, scal, Q, Lk, L):
        self.kr, self.Xb, self.fac, self.W, self.scal, self.Q, self.Lk, self.L = kr, Xb, fac, W, scal, Q, Lk, L
        self.shape = kr.shape

    def __getitem__(self, idx) -> torch.Tensor:
        if not torch.is_tensor(idx):
            idx = torch.as_tensor(idx, device=self.kr.device)
        idx = idx.to(self.kr.device).reshape(-1)
        Vr = self.kr[idx]
        m = Vr.shape[0]
        Vp = torch.zeros(m, self.Q, device=Vr.device, dtype=torch.float32)
        Vp[:, : Vr.shape[1]] = Vr
        Xbr = self.Xb[idx].contiguous()
        Vb = ops.vb(Vp, self.Q, Xbr, self.fac.Binv, self.W, self.scal, m, self.Q, self.Lk, self.L)
        return Vb[:, : self.shape[1]]

    def table_grads(self) -> Tuple[torch.Tensor, torch.Tensor]:
        """The Khatri-Rao backward of this Vb (the contract of khatri_rao_bwd) through the slots, without forming Vb:
        (gxn (P x p), gwn (nviews x q)), the gradients of sum(nll) to the normalised tables (DESIGN 5.8).

            gxn = [cnt (x) xn | slot sums of Xb] R      R from kr_grad_rhs (alpha H_v over -M_v^T)
            gwn = kr_grad_views(ST)                     ST = xn^T [cnt (x) xn | slot sums of Xb]

        Only the rows of X this object was built from take part (a row shard's partial gradient), and rows with an
        index outside the tables sit in no slot, so they add nothing.  Their rows of Xb are NaN, and the slot-sum
        planes take their scale from max|Xb| over all rows, so those rows are zeroed first (a copy of Xb, made only
        when such rows exist)."""
        kr, Lk = self.kr, self.Lk
        alpha = float(self.scal[S_V0] / self.scal[S_VN]) * self.L
        Xb = self.Xb
        n_in = kr.rows_in_table()
        if n_in < kr.n:
            Xb = Xb.index_fill(0, kr.index()[0][n_in:], 0.0)
        ST, ops_left = kr.st_operands(Xb, Xb.stride(0), Lk, True)
        R = ops.kr_grad_rhs(self.fac.Binv, self.W, kr.wn, kr.p, Lk, alpha)
        ncnt = kr.nviews * kr.p
        if isinstance(ops_left, tuple):     # operand planes: each range of the left operand keeps its own scale
            pS, pZ = ops_left
            gx = ops.am_planes(pS, ops.split_planes(R[:ncnt], kr.p, ncnt, kr.p), kr.P, ncnt, kr.p)
            gx += ops.am_planes(pZ, ops.split_planes(R[ncnt:], kr.p, R.shape[0] - ncnt, kr.p), kr.P, pZ.cols, kr.p)
        else:
            gx = ops.am(ops_left, ops_left.stride(0), R, kr.p, kr.P, ops_left.shape[1], kr.p)
        gw = ops.kr_grad_views(ST, self.fac.Binv, self.W, kr.wn, kr.p, Lk, alpha)
        return gx[:, : kr.p_true], gw

    def dense(self, chunk: int = 65536) -> torch.Tensor:
        n = self.kr.n
        out = torch.empty(n, self.shape[1], device=self.kr.device, dtype=torch.float32)
        for a in range(0, n, chunk):
            idx = torch.arange(a, min(n, a + chunk), device=self.kr.device)
            out[a:a + idx.numel()] = self[idx]
        return out


class _EffectsVbRows:
    """Rows of the stacked Vb = (L/vn) V (D B^-1 D) - Xb W^T of k factored designs: the trainer gathers every Vbs[i][idx]
    with the same idx, so the m x Q product is formed once per index set and sliced per design."""

    def __init__(self, Vs, lay: ops.Stacked, Xb, fac, W, scal, Lk, L):
        self.Vs, self.lay, self.Xb, self.fac, self.W, self.scal, self.Lk, self.L = list(Vs), lay, Xb, fac, W, scal, Lk, L
        self.device = Xb.device
        self._key = self._idx = self._rows = None

    def rows(self, key) -> torch.Tensor:
        if self._key is not None and key is self._key:
            return self._rows
        idx = key if torch.is_tensor(key) else torch.as_tensor(key, device=self.device)
        idx = idx.to(self.device).reshape(-1)
        if self._idx is not None and idx.shape == self._idx.shape and torch.equal(idx, self._idx):
            self._key = key
            return self._rows
        lay = self.lay
        m = idx.numel()
        Vr = torch.zeros(m, lay.Q, device=self.device, dtype=torch.float32)
        for V, o, t in zip(self.Vs, lay.offsets, lay.true_widths):
            Vr[:, o:o + t] = V[idx]
        Xbr = self.Xb[idx].contiguous()
        self._rows = ops.vb(Vr, lay.Q, Xbr, self.fac.Binv, self.W, self.scal, m, lay.Q, self.Lk, self.L)
        self._key, self._idx = key, idx
        return self._rows


class LazyEffectVb:
    """`Vbs[i]` of a structured evaluation with k factored designs: `[idx]` returns design i's columns of the rows idx
    of the stacked Vb (see _EffectsVbRows)."""

    def __init__(self, rows: _EffectsVbRows, i: int):
        self._r, self.i = rows, i
        self.shape = rows.Vs[i].shape

    def __getitem__(self, idx) -> torch.Tensor:
        o = self._r.lay.offsets[self.i]
        return self._r.rows(idx)[:, o:o + self.shape[1]]

    def dense(self, chunk: int = 65536) -> torch.Tensor:
        n, dev = self.shape[0], self._r.device
        out = torch.empty(n, self.shape[1], device=dev, dtype=torch.float32)
        for a in range(0, n, chunk):
            idx = torch.arange(a, min(n, a + chunk), device=dev)
            out[a:a + idx.numel()] = self[idx]
        return out


class LazySingularValues:
    """`Shb` of gp.py:33 (singular values of B, descending).  The trainer discards it
    (train_gppvae.py:235), so it is only computed if somebody asks -- off the hot path, from G."""

    def __init__(self, G: torch.Tensor, Qtrue: int, vs: torch.Tensor, stk: Optional[ops.Stacked] = None):
        self._G, self._Q, self._vs, self._stk, self._val = G, Qtrue, vs, stk, None

    def value(self) -> torch.Tensor:
        if self._val is None:
            vs = self._vs.detach()
            if self._stk is not None:   # k designs: B = I + D G D / vn on the true columns of every block
                stk = self._stk
                cols = torch.cat([torch.arange(o, o + t) for o, t in zip(stk.offsets, stk.true_widths)]).to(self._G.device)
                d = torch.cat([torch.sqrt(vs[i]).expand(t) for i, t in enumerate(stk.true_widths)])
                G = self._G[:, : stk.Q][cols][:, cols]
                B = torch.eye(cols.numel(), device=G.device) + (d[:, None] * d[None, :] / vs[-1]) * G
            else:
                B = torch.eye(self._Q, device=self._G.device) + (vs[0] / vs[-1]) * self._G[: self._Q, : self._Q]
            self._val = torch.linalg.eigvalsh(B.double()).flip(0).to(torch.float32)
        return self._val

    @classmethod
    def __torch_function__(cls, func, types, args=(), kwargs=None):
        args = tuple(a.value() if isinstance(a, LazySingularValues) else a for a in args)
        return func(*args, **(kwargs or {}))


class _FactorCache:
    """One-entry cache of (G, factorisation) keyed on the identity and version of V and of the variances.

    train_gppvae.py factors the same (Vt, vs) twice per epoch (:235 via U_UBi_Shb, then :166 inside
    taylor_coeff).  What keeps V's address from being recycled while the entry is alive: for matrices that have operand
    planes, the planes registry (`ops.PLANES`) -- the entry remembers WHICH planes object it was built from and is valid
    only while the registry still returns that very object for V (so dropping the registry entry, which
    `Vmodel.forward` does before it allocates the next V of the same shape, also retires this entry, and no second
    reference keeps last epoch's 16 GB alive); for small matrices the entry holds V itself.  In-place updates of V or lvs
    bump their version counters and miss; the variances are compared value for value as well.
    """

    def __init__(self):
        self.key = None
        self.keep = None
        self.token = None
        self.G = None
        self.ldg = 0
        self.C = None                # V^T X of the evaluation that built the entry (bench.run_check reads it)
        self.fac: Optional[ops.Factorisation] = None

    def lookup(self, key, want_binv: bool, vs: torch.Tensor, token=None):
        if self.key is not None and self.key == key and token is self.token and \
                (self.fac.Binv is not None or not want_binv):
            # version counters do not see writes through `.data` (the reference itself initialises parameters that way,
            # vmod.py:37-40): a hit also needs the variances the factorisation was built with, value for value
            if torch.equal(self.vs_snapshot, vs.detach().to(torch.float32)):
                return self.fac
        return None

    def store(self, key, keep, G, ldg, fac, vs: torch.Tensor, token=None):
        self.key, self.keep, self.G, self.ldg, self.fac, self.token = key, keep, G, ldg, fac, token
        self.vs_snapshot = vs.detach().to(torch.float32).clone()

    def clear(self):
        self.key = self.keep = self.G = self.C = self.fac = self.token = None


class GP(nn.Module):
    def __init__(self, n_rand_effs: int = 1, vsum2one: bool = True, process_group=None):
        super().__init__()
        if not vsum2one:
            # the reference's other branch is broken (gp.py:52 uses an undefined name)
            raise NotImplementedError("vsum2one=False is not implemented (it raises NameError in the reference too)")
        if int(n_rand_effs) != n_rand_effs or not 1 <= n_rand_effs <= GPP_MAX_DESIGNS:
            raise ValueError(f"n_rand_effs must be an integer in 1..{GPP_MAX_DESIGNS} (got {n_rand_effs})")
        self.n_rand_effs = n_rand_effs
        self.vsum2one = vsum2one
        self.lvs = nn.Parameter(torch.zeros([n_rand_effs + 1]))      # gp.py:21-22
        self._group = process_group
        self._sharded = process_group is not None
        self._cache = _FactorCache()
        self._n_total_given = None
        self._vs_ref = None          # weakref to the tensor last returned by get_vs()
        self._vs_version = -1
        self.cache_hits = 0
        self.stage_hook = None       # optional callable(name): bench.py records CUDA events at stage boundaries
        self.overlap_exchange = True  # row shards: all-reduce G beside V^T X, C beside the Cholesky (see _factorise)

    # ------------------------------------------------------------------ sharding
    def shard_rows(self, process_group=None, n_total: Optional[int] = None) -> "GP":
        """Treat the rows handed to every method as this rank's shard of the N rows (SURVEY 8(e)).

        `n_total` is the global number of rows.  Pass it when it is known (it usually is: the size of the data set):
        otherwise every evaluation all-reduces its local row count first, which costs a host synchronisation."""
        import torch.distributed as dist
        self._group = process_group if process_group is not None else dist.group.WORLD
        self._sharded = True
        self._n_total_given = n_total
        return self

    def invalidate_cache(self) -> None:
        """Forget the cached factorisation and operand planes.  Needed only after writes the version counters cannot
        see (`V.data[...] = ...`); in-place tensor operations and optimiser steps are detected."""
        self._cache.clear()
        ops.PLANES.invalidate()
        ops.STACKED.invalidate()

    def _all_reduce(self, t: torch.Tensor, async_op: bool = False):
        """SUM over the row shards.  `async_op=True` returns the collective's work handle (None when not sharded): the
        caller keeps launching on its stream and calls `.wait()` where the result is first needed."""
        if self._sharded:
            import torch.distributed as dist
            return dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self._group, async_op=async_op)
        return None

    def _n_total(self, n: int, device) -> int:
        if not self._sharded:
            return n
        if self._n_total_given is not None:
            return int(self._n_total_given)
        # every rank takes part in this collective on every call (a per-rank cache keyed on the local row count would
        # let ranks disagree about whether to communicate)
        t = torch.tensor([n], device=device, dtype=torch.int64)
        self._all_reduce(t)
        return int(t.item())

    def _stage(self, name: str) -> None:
        if self.stage_hook is not None:
            self.stage_hook(name)

    # ------------------------------------------------------------------ reference API
    def get_vs(self) -> torch.Tensor:
        """softmax(lvs) = [v0, vn]  (gp.py:48-50)."""
        vs = F.softmax(self.lvs, 0)
        self._vs_ref, self._vs_version = weakref.ref(vs), self.lvs._version
        return vs

    def _vs_token(self, vs: torch.Tensor):
        """Cache token for a variance vector: tensors that came out of get_vs() for the current lvs are
        all the same value; anything else is identified by object and version (and kept alive)."""
        mine = self._vs_ref() if self._vs_ref is not None else None
        if mine is not None and vs is mine and self._vs_version == self.lvs._version:
            return ("lvs", id(self.lvs), self.lvs._version), None
        return ("tensor", id(vs), vs._version), vs

    def _cat(self, Vs: Sequence[torch.Tensor], vs: torch.Tensor) -> Tuple[torch.Tensor, int, int, int]:
        """gp.py:27 for the single design the trainer uses: V passes through untouched (the sqrt(vs[0])
        weight folds into the v0/vn factor inside the kernels).  Returns (V, ldv, Q padded, Q)."""
        if len(Vs) != 1:
            raise NotImplementedError(f"expected one design matrix in Vs, got {len(Vs)}")
        Vm, ldv = ops.as_matrix(Vs[0], "V")
        return Vm, ldv, Vm.shape[1], Vs[0].shape[1]

    def _stack(self, Vs: Sequence[torch.Tensor], Lk: int) -> ops.Stacked:
        """k >= 2 designs: check them and return their stacked operand (planes at tensor-core shapes)."""
        k = self.n_rand_effs
        if len(Vs) != k:
            raise ValueError(f"GP(n_rand_effs={k}) expects {k} design matrices in Vs, got {len(Vs)}")
        n, Q = Vs[0].shape[0], sum(ops.round4(V.shape[1]) for V in Vs)
        use_planes = ops.planes_supported(n, Q, Lk)

        def before_build():   # new stacked planes are about to be built: a cache entry on the previous ones lets them go
            if isinstance(self._cache.token, ops.Stacked):
                self._cache.clear()
        return ops.stacked(Vs, use_planes, before_build)

    def _factor(self, G, ldg, Q, vs, want_binv, stk):
        if stk is None:
            return ops.factor(G, ldg, Q, vs, want_binv)
        return ops.factor_blocks(G, ldg, stk.widths, vs, want_binv)

    def _factorise(self, Vm, ldv, Q, vs, want_binv: bool, Xm=None, ldx=0, Lk=0, vs_origin=None, stk=None):
        """Pass 1 (+ all-reduce) and the factorisation, through the cache.
        Returns (fac, C, pV) with C = V^T X (Q x Lk, summed over ranks) or None when no X was given, and pV the operand
        planes of V (None for shapes below the tensor-core tile, which run on the fp32 engine).  With `stk` (k >= 2
        designs) V is the stacked operand and the factorisation is the block form."""
        tok, keep_vs = self._vs_token(vs if vs_origin is None else vs_origin)
        if stk is None:
            n = Vm.shape[0]
            key = (Vm.untyped_storage().data_ptr(), Vm.storage_offset(), Vm._version, n, Q, ldv, tok)
            use_planes = ops.planes_supported(n, Q, Lk)
            pV = ops.planes_of(Vm, ldv) if use_planes else None
            token, keep_v = pV, (None if use_planes else Vm)
        else:
            n = stk.n
            key = ("blocks", stk.key, tok)
            use_planes = stk.planes is not None
            pV = stk.planes
            token, keep_v = stk, None          # the stacked operand (held by the entry's token) pins what it needs

        def vtx():
            if use_planes:
                return ops.atb_planes(pV, ops.split_planes(Xm, ldx, n, Lk), n, Q, Lk)
            return ops.atb(Vm, ldv, Xm, ldx, n, Q, Lk)

        fac = self._cache.lookup(key, want_binv, vs, token=token)
        if fac is not None:
            self.cache_hits += 1
            C = None
            if Lk:
                C = vtx()
                self._all_reduce(C)
            return fac, C, pV
        if self._sharded and Lk and self.overlap_exchange:
            # Row shards: the exchange step rides beside the work that does not need it.  Gram tiles -> all-reduce of G on
            # the collective's own stream WHILE this stream splits X and forms V^T X -> all-reduce of the small C WHILE
            # the Cholesky runs.  Only the tail of the first collective and nothing of the second stay exposed.
            self._stage("pass1:start")
            G = ops.gram_vtz_planes(pV, None, n, Q, 0) if use_planes else ops.gram_vtz(Vm, ldv, None, 0, n, Q, 0)
            hG = self._all_reduce(G, async_op=True)
            C = vtx()
            self._stage("pass1:end")
            hC = self._all_reduce(C, async_op=True)
            hG.wait()
            self._stage("allreduce:end")
            fac = self._factor(G, Q, Q, vs, want_binv, stk)
            hC.wait()
            self._stage("factor:end")
            self._cache.store(key, (keep_v, keep_vs), G, Q, fac, vs, token=token)
            self._cache.C = C
            return fac, C, pV
        pX = ops.split_planes(Xm, ldx, n, Lk) if (use_planes and Lk) else None
        self._stage("pass1:start")
        GC = ops.gram_vtz_planes(pV, pX, n, Q, Lk) if use_planes else ops.gram_vtz(Vm, ldv, Xm, ldx, n, Q, Lk)
        self._stage("pass1:end")
        self._all_reduce(GC)
        self._stage("allreduce:end")
        fac = self._factor(GC, Q + Lk, Q, vs, want_binv, stk)
        self._stage("factor:end")
        # with planes the registry entry pins V (see _FactorCache); without, the cache entry does
        self._cache.store(key, (keep_v, keep_vs), GC, Q + Lk, fac, vs, token=token)
        self._cache.C = GC[:, Q:] if Lk else None
        return fac, (GC[:, Q:] if Lk else None), pV

    # ------------------------------------------------------------------ structured route (vmod.KhatriRao)
    def _kr_c(self, kr: KhatriRao, Xm, ldx, Lk) -> torch.Tensor:
        """C = V^T X (Q x Lk) through the slot sums, summed over the ranks."""
        ST = kr.st(Xm, ldx, Lk, False)
        self._all_reduce(ST)
        return ops.kr_assemble_gc(ST, kr.wn, kr.p, Lk, False)

    def _kr_factorise(self, kr: KhatriRao, vs, want_binv: bool, Xm=None, ldx=0, Lk=0, vs_origin=None):
        """Structured pass 1 (+ all-reduce of the small ST instead of GC) and the factorisation, through the cache."""
        tok, keep_vs = self._vs_token(vs if vs_origin is None else vs_origin)
        key = ("kr", id(kr), tok)
        Q = kr.p * kr.q
        fac = self._cache.lookup(key, want_binv, vs)
        if fac is not None:
            self.cache_hits += 1
            return fac, (self._kr_c(kr, Xm, ldx, Lk) if Lk else None)
        if not Lk:      # factorisation alone (U_UBi_Shb): the slot sums still need a right-hand side to walk
            Xm = torch.zeros(kr.n, 4, device=kr.device, dtype=torch.float32)
            ldx, Lx = 4, 4
        else:
            Lx = Lk
        kr.index()
        self._stage("pass1:start")
        ST = kr.st(Xm, ldx, Lx, True)
        self._stage("pass1:end")
        self._all_reduce(ST)
        self._stage("allreduce:end")
        GC = ops.kr_assemble_gc(ST, kr.wn, kr.p, Lx, True)
        fac = ops.factor(GC, Q + Lx, Q, vs, want_binv)
        self._stage("factor:end")
        self._cache.store(key, (kr, keep_vs), GC, Q + Lx, fac, vs)
        return fac, (GC[:, Q:] if Lk else None)

    @staticmethod
    def _kr_y(kr: KhatriRao, M: torch.Tensor) -> torch.Tensor:
        """Y = xn [M_0 | M_1 | ...], the P-long product of the structured pass 2."""
        if ops.planes_supported(kr.P, kr.p, 0):
            pM = ops.split_planes(M, M.stride(0), kr.p, M.shape[1])
            return ops.am_planes(kr.xn_planes(), pM, kr.P, kr.p, M.shape[1])
        return ops.am(kr.xn, kr.p, M, M.stride(0), kr.P, kr.p, M.shape[1])

    def _kr_solve(self, kr: KhatriRao, fac, C, Xm, ldx, Lk, L, n_total):
        """W, the scalar block, Xb = (X - V W)/vn and nll for the rows of X, V in factored form."""
        W, scal = ops.solve_w(fac, C, C.stride(0), Lk, L, n_total)
        self._stage("solve:end")
        M = ops.kr_assemble_m(W, kr.wn, kr.p, Lk)
        Y = self._kr_y(kr, M)
        Xb, nll = ops.kr_xb_nll(Xm, ldx, Y, kr.d, kr.w, kr.P, kr.nviews, Lk, scal)
        self._stage("pass2:end")
        return W, scal, Xb, nll

    # ------------------------------------------------------------------ structured route, k factored designs
    def _effects(self, Vs) -> Optional[KhatriRao]:
        """k >= 2 designs: the KhatriRao whose slot index and tables the designs share when they are all factored
        (Vmodel.lazy_effects), None when they are all dense."""
        k = self.n_rand_effs
        if len(Vs) != k:
            raise ValueError(f"GP(n_rand_effs={k}) expects {k} design matrices in Vs, got {len(Vs)}")
        factored = [isinstance(V, (KhatriRao, _FactoredEffect)) for V in Vs]
        if not any(factored):
            return None
        if not all(factored):
            raise NotImplementedError("factored designs (vmod.KhatriRao, ObjectEffect, ViewEffect) and dense designs "
                                      "cannot be mixed: pass every design factored (Vmodel.lazy_effects) or every one "
                                      "dense (.dense())")
        base = effect_base(Vs[0])
        if any(effect_base(V) is not base for V in Vs):
            raise ValueError("the factored designs are built over different d, w or tables: make them with one "
                             "Vmodel.lazy_effects call")
        kinds = [effect_kind(V) for V in Vs]
        if len(set(kinds)) != k:
            raise ValueError(f"each kind of factored design may appear once, got {kinds}")
        return base

    @staticmethod
    def _effects_layout(base: KhatriRao, kinds) -> ops.Stacked:
        """Block layout of the stacked factored designs: widths p q, p, round4(q) (p already padded to 4)."""
        true = [base.p_true * base.q if k == "kr" else base.p_true if k == "object" else base.q for k in kinds]
        return ops.Stacked(None, base.n, ops.effect_widths(kinds, base.p, base.q), true, None, None)

    def _all_reduce_pair(self, ST, VM):
        """SUM of the slot-sum products and the per-view moments over the row shards, in one collective."""
        if not self._sharded:
            return ST, VM
        parts = [t for t in (ST, VM) if t is not None]
        flat = torch.cat([t.reshape(-1) for t in parts])
        self._all_reduce(flat)
        out, o = [], 0
        for t in (ST, VM):
            if t is None:
                out.append(None)
            else:
                out.append(flat[o:o + t.numel()].view(t.shape))
                o += t.numel()
        return tuple(out)

    def _effects_factorise(self, Vs, base: KhatriRao, kinds, lay, vs, want_binv: bool, Xm=None, ldx=0, Lk=0,
                           vs_origin=None):
        """Structured pass 1 of the stacked factored designs (+ one all-reduce of ST and the moments instead of GC) and
        the block-form factorisation, through the cache (keyed on the designs and the variances)."""
        tok, keep_vs = self._vs_token(vs if vs_origin is None else vs_origin)
        key = ("effects", tuple(id(V) for V in Vs), tok)
        fac = self._cache.lookup(key, want_binv, vs)
        if fac is not None:
            self.cache_hits += 1
            return fac, (effects_c(base, kinds, Xm, ldx, Lk, self._all_reduce_pair) if Lk else None)
        if not Lk:      # factorisation alone (U_UBi_Shb): the slot sums still need a right-hand side to walk
            Xm = torch.zeros(base.n, 4, device=base.device, dtype=torch.float32)
            ldx, Lx = 4, 4
        else:
            Lx = Lk
        base.index()
        self._stage("pass1:start")
        ST, VM = effects_st_vm(base, kinds, Xm, ldx, Lx, True)
        self._stage("pass1:end")
        ST, VM = self._all_reduce_pair(ST, VM)
        self._stage("allreduce:end")
        GC = ops.kr_assemble_gc_blocks(ST, VM, base.wn, base.p, kinds, Lx, True)
        fac = ops.factor_blocks(GC, lay.Q + Lx, lay.widths, vs, want_binv)
        self._stage("factor:end")
        self._cache.store(key, (tuple(Vs), keep_vs), GC, lay.Q + Lx, fac, vs)
        return fac, (GC[:, lay.Q:] if Lk else None)

    def _effects_solve(self, base: KhatriRao, kinds, fac, C, Xm, ldx, Lk, L, n_total):
        """W, the scalar blocks, Xb = (X - V W)/vn and nll for the rows of X, the k designs in factored form:
        (V W)_i = Y[d_i, w_i] + R[w_i]."""
        W, scal, blk = ops.solve_w_blocks(fac, C, C.stride(0), Lk, L, n_total)
        self._stage("solve:end")
        M, R = ops.kr_assemble_m_blocks(W, base.wn, base.p, kinds, Lk)
        Y = self._kr_y(base, M)
        if R is None:
            Xb, nll = ops.kr_xb_nll(Xm, ldx, Y, base.d, base.w, base.P, base.nviews, Lk, scal)
        else:
            Xb, nll = ops.kr_xb_nll_views(Xm, ldx, Y, R, base.d, base.w, base.P, base.nviews, Lk, scal)
        self._stage("pass2:end")
        return W, scal, blk, Xb, nll

    def _effects_coefficients(self, X, Vs, base: KhatriRao, vs, vs_attached, want_vb: bool):
        Xm, ldx = ops.as_matrix(X, "X")
        n, L = X.shape
        if base.n != n:
            raise ValueError(f"X has {n} rows but the designs have {base.n}")
        if base.device != Xm.device:
            raise ValueError("X and V must be on the same device")
        Lk = Xm.shape[1]
        kinds = [effect_kind(V) for V in Vs]
        lay = self._effects_layout(base, kinds)
        n_total = self._n_total(n, X.device)
        fac, C = self._effects_factorise(Vs, base, kinds, lay, vs, want_vb, Xm, ldx, Lk, vs_origin=vs_attached)
        W, scal, blk, Xb, nll = self._effects_solve(base, kinds, fac, C, Xm, ldx, Lk, L, n_total)
        return dict(vs=vs, Vm=None, effects=list(Vs), Q=lay.Q, Qtrue=lay.Q, n=n, L=L, Lk=Lk, n_total=n_total, fac=fac,
                    W=W, scal=scal, Xb=Xb, nll=nll, pV=None, stk=lay, blk=blk)

    def U_UBi_Shb(self, Vs: Sequence[torch.Tensor], vs: torch.Tensor, want_binv: bool = False):
        """gp.py:24-38.  Returns handles (see LowRankFactor) that `solve` accepts."""
        if self.n_rand_effs == 1 and len(Vs) == 1 and isinstance(Vs[0], KhatriRao):
            kr = Vs[0]
            fac, _ = self._kr_factorise(kr, vs, want_binv)
            return (KhatriRaoFactor("U", kr, vs, fac), KhatriRaoFactor("UBi", kr, vs, fac),
                    LazySingularValues(self._cache.G, kr.p * kr.q, vs))
        if self.n_rand_effs > 1:
            base = self._effects(Vs)
            if base is not None:
                kinds = [effect_kind(V) for V in Vs]
                lay = self._effects_layout(base, kinds)
                fac, _ = self._effects_factorise(Vs, base, kinds, lay, vs, want_binv)
                return (EffectsFactor("U", Vs, lay, vs, fac), EffectsFactor("UBi", Vs, lay, vs, fac),
                        LazySingularValues(self._cache.G, lay.Q, vs, stk=lay))
            stk = self._stack(Vs, 0)
            fac, _, _ = self._factorise(stk.V, stk.Q, stk.Q, vs, want_binv, stk=stk)
            return (BlocksFactor("U", Vs, stk, vs, fac), BlocksFactor("UBi", Vs, stk, vs, fac),
                    LazySingularValues(self._cache.G, stk.Q, vs, stk=stk))
        Vm, ldv, Q, Qtrue = self._cat(Vs, vs)
        fac, _, _ = self._factorise(Vm, ldv, Q, vs, want_binv)
        U = LowRankFactor("U", Vm, ldv, Q, Qtrue, vs, fac)
        UBi = LowRankFactor("UBi", Vm, ldv, Q, Qtrue, vs, fac)
        return U, UBi, LazySingularValues(self._cache.G, Qtrue, vs)

    def solve(self, X: torch.Tensor, U, UBi, vs: torch.Tensor) -> torch.Tensor:
        """K^-1 X  (gp.py:40-46)."""
        Xm, ldx = ops.as_matrix(X, "X")
        n, L = X.shape
        Lk = Xm.shape[1]
        if isinstance(U, EffectsFactor):
            if n != U.n:
                raise ValueError(f"X has {n} rows but the factorisation was built for {U.n}")
            base, kinds = effect_base(U.Vs[0]), [effect_kind(V) for V in U.Vs]
            C = effects_c(base, kinds, Xm, ldx, Lk, self._all_reduce_pair)
            _, _, _, Xb, _ = self._effects_solve(base, kinds, U.fac, C, Xm, ldx, Lk, L, self._n_total(n, X.device))
        elif isinstance(U, KhatriRaoFactor):
            if n != U.n:
                raise ValueError(f"X has {n} rows but the factorisation was built for {U.n}")
            C = self._kr_c(U.kr, Xm, ldx, Lk)
            _, _, Xb, _ = self._kr_solve(U.kr, U.fac, C, Xm, ldx, Lk, L, self._n_total(n, X.device))
        elif isinstance(U, BlocksFactor):
            if n != U.n:
                raise ValueError(f"X has {n} rows but the factorisation was built for {U.n}")
            # the stacked operand in the form this X needs (the factorisation holds for the same designs either way)
            stk = U.stk if (U.stk.planes is not None) == ops.planes_supported(n, U.Q, Lk) else self._stack(U.Vs, Lk)
            if stk.planes is not None:
                C = ops.atb_planes(stk.planes, ops.split_planes(Xm, ldx, n, Lk), n, U.Q, Lk)
            else:
                C = ops.atb(stk.V, U.Q, Xm, ldx, n, U.Q, Lk)
            self._all_reduce(C)
            W, scal = ops.solve_w(U.fac, C, Lk, Lk, L, self._n_total(n, X.device))
            if stk.planes is not None:
                Xb, _ = ops.xb_nll_planes(stk.planes, Xm, ldx, W, n, U.Q, Lk, scal)
            else:
                Xb, _ = ops.xb_nll(stk.V, U.Q, Xm, ldx, W, n, U.Q, Lk, scal)
        elif isinstance(U, LowRankFactor):
            if n != U.n:
                raise ValueError(f"X has {n} rows but the factorisation was built for {U.n}")
            if ops.planes_supported(n, U.Q, Lk):
                pV = ops.planes_of(U.V, U.ldv)
                C = ops.atb_planes(pV, ops.split_planes(Xm, ldx, n, Lk), n, U.Q, Lk)
            else:
                pV = None
                C = ops.atb(U.V, U.ldv, Xm, ldx, n, U.Q, Lk)
            self._all_reduce(C)
            W, scal = ops.solve_w(U.fac, C, Lk, Lk, L, self._n_total(n, X.device))
            if pV is not None:
                Xb, _ = ops.xb_nll_planes(pV, Xm, ldx, W, n, U.Q, Lk, scal)
            else:
                Xb, _ = ops.xb_nll(U.V, U.ldv, Xm, ldx, W, n, U.Q, Lk, scal)
        else:
            # dense tensors, exactly gp.py:42-44: (X - UBi (U^T X)) / vn
            Um, ldu = ops.as_matrix(U, "U")
            UBm, ldub = ops.as_matrix(UBi, "UBi")
            UX = ops.atb(Um, ldu, Xm, ldx, n, Um.shape[1], Lk)
            self._all_reduce(UX)
            Xb = ops.x_minus_am(Xm, ldx, UBm, ldub, UX, Lk, n, Um.shape[1], Lk, 1.0 / float(vs.detach()[-1]))
        return Xb[:, :L] if Lk != L else Xb

    def _coefficients(self, X: torch.Tensor, Vs: Sequence[torch.Tensor], want_vb: bool):
        """Shared body of taylor_coeff and nll: returns a dict of everything computed."""
        vs_attached = self.get_vs()
        vs = vs_attached.detach()
        if self.n_rand_effs == 1 and len(Vs) == 1 and isinstance(Vs[0], KhatriRao):
            kr = Vs[0]
            Xm, ldx = ops.as_matrix(X, "X")
            n, L = X.shape
            if kr.n != n:
                raise ValueError(f"X has {n} rows but V has {kr.n}")
            if kr.device != Xm.device:
                raise ValueError("X and V must be on the same device")
            Lk = Xm.shape[1]
            n_total = self._n_total(n, X.device)
            fac, C = self._kr_factorise(kr, vs, want_vb, Xm, ldx, Lk, vs_origin=vs_attached)
            W, scal, Xb, nll = self._kr_solve(kr, fac, C, Xm, ldx, Lk, L, n_total)
            return dict(vs=vs, Vm=None, kr=kr, ldv=0, Q=kr.p * kr.q, Qtrue=kr.p_true * kr.q, n=n, L=L, Lk=Lk,
                        n_total=n_total, fac=fac, W=W, scal=scal, Xb=Xb, nll=nll)
        if self.n_rand_effs > 1:
            base = self._effects(Vs)
            if base is not None:
                return self._effects_coefficients(X, Vs, base, vs, vs_attached, want_vb)
            Xm, ldx = ops.as_matrix(X, "X")
            n, L = X.shape
            Lk = Xm.shape[1]
            if any(V.shape[0] != n for V in Vs if torch.is_tensor(V)):
                raise ValueError(f"X has {n} rows but the designs have {[V.shape[0] for V in Vs]}")
            self._stage("stack:start")
            stk = self._stack(Vs, Lk)
            self._stage("stack:end")
            if (stk.planes.buf if stk.planes is not None else stk.V).device != Xm.device:
                raise ValueError("X and V must be on the same device")
            n_total = self._n_total(n, X.device)
            fac, C, pV = self._factorise(stk.V, stk.Q, stk.Q, vs, want_vb, Xm, ldx, Lk, vs_origin=vs_attached, stk=stk)
            W, scal, blk = ops.solve_w_blocks(fac, C, C.stride(0), Lk, L, n_total)
            self._stage("solve:end")
            if pV is not None:
                Xb, nll = ops.xb_nll_planes(pV, Xm, ldx, W, n, stk.Q, Lk, scal)
            else:
                Xb, nll = ops.xb_nll(stk.V, stk.Q, Xm, ldx, W, n, stk.Q, Lk, scal)
            self._stage("pass2:end")
            return dict(vs=vs, Vm=stk.V, ldv=stk.Q, Q=stk.Q, Qtrue=stk.Q, n=n, L=L, Lk=Lk, n_total=n_total, fac=fac,
                        W=W, scal=scal, Xb=Xb, nll=nll, pV=pV, stk=stk, blk=blk)
        Vm, ldv, Q, Qtrue = self._cat(Vs, vs)
        Xm, ldx = ops.as_matrix(X, "X")
        n, L = X.shape
        if Vm.shape[0] != n:
            raise ValueError(f"X has {n} rows but V has {Vm.shape[0]}")
        if Vm.device != Xm.device:
            raise ValueError("X and V must be on the same device")
        Lk = Xm.shape[1]
        n_total = self._n_total(n, X.device)
        fac, C, pV = self._factorise(Vm, ldv, Q, vs, want_vb, Xm, ldx, Lk, vs_origin=vs_attached)
        W, scal = ops.solve_w(fac, C, C.stride(0), Lk, L, n_total)
        self._stage("solve:end")
        if pV is not None:
            Xb, nll = ops.xb_nll_planes(pV, Xm, ldx, W, n, Q, Lk, scal)
        else:
            Xb, nll = ops.xb_nll(Vm, ldv, Xm, ldx, W, n, Q, Lk, scal)
        self._stage("pass2:end")
        return dict(vs=vs, Vm=Vm, ldv=ldv, Q=Q, Qtrue=Qtrue, n=n, L=L, Lk=Lk, n_total=n_total, fac=fac, W=W,
                    scal=scal, Xb=Xb, nll=nll, pV=pV)

    def taylor_coeff(self, X: torch.Tensor, Vs: Sequence[torch.Tensor], need_vb: bool = True
                     ) -> Tuple[torch.Tensor, List[torch.Tensor], torch.Tensor, torch.Tensor]:
        """gp.py:55-95: Xb = dNLL/dX, [Vb = dNLL/dV], vbs = dNLL/d[v0, vn], nll (n x 1); all detached.

        `need_vb=False` (an extension) skips B^-1 and the N x Q matrix Vb and returns `[None]` in its place:
        that is the "NLL + dNLL/dZ" evaluation BASELINE.json's metric counts."""
        c = self._coefficients(X, Vs, need_vb)
        scal, Q, L, Lk = c["scal"], c["Q"], c["L"], c["Lk"]
        if self._sharded:
            self._all_reduce(scal[S_XB2:S_QUAD + 1])
        stk = c.get("stk")
        if stk is not None:
            vbs = ops.vbs_blocks(scal, c["blk"], c["vs"], stk.widths, c["n_total"], L)
        else:
            vbs = ops.vbs_from_scal(scal, c["n_total"], Q, L)
        if need_vb and c.get("effects") is not None:
            rows = _EffectsVbRows(c["effects"], stk, c["Xb"], c["fac"], c["W"], scal, Lk, L)
            Vbs = [LazyEffectVb(rows, i) for i in range(len(stk.widths))]
        elif need_vb and stk is not None:
            # one N x Q matrix; Vb_i is the view of block i at design i's true width
            if c["pV"] is not None:
                Vb = ops.vb_planes(c["pV"], c["Xb"], c["fac"].Binv, c["W"], scal, c["n"], Q, Lk, L)
            else:
                Vb = ops.vb(stk.V, Q, c["Xb"], c["fac"].Binv, c["W"], scal, c["n"], Q, Lk, L)
            Vbs = [Vb[:, o:o + t] for o, t in zip(stk.offsets, stk.true_widths)]
            self._stage("vb:end")
        elif stk is not None:
            Vbs = [None] * len(stk.widths)
        elif need_vb and c["Vm"] is None:
            Vbs = [LazyVb(c["kr"], c["Xb"], c["fac"], c["W"], scal, Q, Lk, L)]
        elif need_vb:
            if c.get("pV") is not None:
                Vb = ops.vb_planes(c["pV"], c["Xb"], c["fac"].Binv, c["W"], scal, c["n"], Q, Lk, L)
            else:
                Vb = ops.vb(c["Vm"], c["ldv"], c["Xb"], c["fac"].Binv, c["W"], scal, c["n"], Q, Lk, L)
            Vbs = [Vb[:, : c["Qtrue"]] if c["Qtrue"] != Q else Vb]
            self._stage("vb:end")
        else:
            Vbs = [None]
        self.last_scalars = scal
        Xb = c["Xb"][:, :L] if Lk != L else c["Xb"]
        return Xb, Vbs, vbs, c["nll"]

    # ------------------------------------------------------------------ posterior prediction (DESIGN 5.9)
    def predict(self, X: torch.Tensor, Vs: Sequence, Vs_new: Sequence) -> Tuple[torch.Tensor, torch.Tensor]:
        """Posterior mean (m x L) and variance (m x 1) of the noise-free latents at the new rows `Vs_new`, given the
        training latents X and designs Vs (what taylor_coeff / nll take); float32, detached.

            mean* = u W = v0 u V^T K^-1 X,    var* = scal[V0] u Binv u^T = v0 (u u^T - v0 u V^T K^-1 V u^T)

        for a new stacked row u (W and Binv of the factorisation, Binv = D B^-1 D and scal[V0] = 1 for k designs).  One
        variance per row, shared by the L columns; the observation z* has variance var* + vn.

        `Vs_new` has the form of Vs: dense tensors of the same widths, or factored designs over the same (equal) tables
        with the same kinds in the same order (`vm.lazy(dv, wv)`, `vm.lazy_effects(dv, wv, kinds)`); of those only d and w
        are read.  Note that `vm.lazy(dv, wv)` replaces Vmodel's one-entry slot-index cache, so the next
        `vm.lazy(Dt, Wt)` sorts the training rows again.  The factorisation goes through the cache with B^-1: after
        taylor_coeff(X, Vs) it is a hit, and only C, the solve and the prediction stages run.  With row shards X and Vs
        are this rank's rows and every rank predicts its own new rows without further communication.  New rows with an
        index outside the tables get NaN.  Factored new rows form nothing of size m x Q (DESIGN 5.9)."""
        with torch.no_grad():
            return self._predict(X, list(Vs), list(Vs_new))

    def _predict(self, X, Vs, Vs_new):
        is_f = [isinstance(V, (KhatriRao, _FactoredEffect)) for V in Vs + Vs_new]
        if any(is_f) and not all(is_f):
            raise ValueError("predict: dense and factored designs cannot be mixed in Vs and Vs_new")
        if len(Vs_new) != len(Vs):
            raise ValueError(f"predict: Vs has {len(Vs)} designs but Vs_new has {len(Vs_new)}")
        for i, (V, Vn) in enumerate(zip(Vs, Vs_new)):
            if V.shape[1] != Vn.shape[1]:
                raise ValueError(f"predict: Vs_new[{i}] has {Vn.shape[1]} columns but Vs[{i}] has {V.shape[1]}")
        if not torch.is_tensor(X):
            raise ValueError("predict: X must be a tensor")
        devs = {X.device} | {V.device for V in Vs + Vs_new}
        if len(devs) != 1:
            raise ValueError(f"predict: X, Vs and Vs_new must be on one device (got {sorted(map(str, devs))})")
        if all(is_f):
            return self._predict_factored(X, Vs, Vs_new)
        m = Vs_new[0].shape[0]
        if m == 0 or any(Vn.shape[0] != m for Vn in Vs_new):
            raise ValueError(f"predict: the new designs must have the same, positive number of rows "
                             f"(got {[Vn.shape[0] for Vn in Vs_new]})")
        return self._predict_dense(X, Vs, Vs_new, m)

    def _predict_factored(self, X, Vs, Vs_new):
        vs_attached = self.get_vs()
        vs = vs_attached.detach()
        if self.n_rand_effs == 1:
            if len(Vs) != 1 or not isinstance(Vs[0], KhatriRao) or not isinstance(Vs_new[0], KhatriRao):
                raise ValueError("predict: GP(n_rand_effs=1) takes one Khatri-Rao design (Vmodel.lazy) in Vs and Vs_new")
            base, new, kinds = Vs[0], Vs_new[0], ["kr"]
        else:
            base, new = self._effects(Vs), self._effects(Vs_new)
            kinds = [effect_kind(V) for V in Vs]
            if [effect_kind(V) for V in Vs_new] != kinds:
                raise ValueError(f"predict: Vs_new has kinds {[effect_kind(V) for V in Vs_new]} but Vs has {kinds}")
        if new.n == 0:
            raise ValueError("predict: Vs_new has no rows")
        for name in ("xn", "wn"):
            a, b = getattr(base, name), getattr(new, name)
            if a.shape != b.shape or not torch.equal(a, b):
                raise ValueError(f"predict: the tables of Vs_new differ from those of Vs ({name}): build both from the "
                                 "same Vmodel state")
        Xm, ldx = ops.as_matrix(X, "X")
        n, L = X.shape
        if base.n != n:
            raise ValueError(f"X has {n} rows but the designs have {base.n}")
        Lk = Xm.shape[1]
        n_total = self._n_total(n, X.device)
        if self.n_rand_effs == 1:
            fac, C = self._kr_factorise(base, vs, True, Xm, ldx, Lk, vs_origin=vs_attached)
            W, scal = ops.solve_w(fac, C, C.stride(0), Lk, L, n_total)
            M, R = ops.kr_assemble_m(W, base.wn, base.p, Lk), None
        else:
            lay = self._effects_layout(base, kinds)
            fac, C = self._effects_factorise(Vs, base, kinds, lay, vs, True, Xm, ldx, Lk, vs_origin=vs_attached)
            W, scal, _ = ops.solve_w_blocks(fac, C, C.stride(0), Lk, L, n_total)
            M, R = ops.kr_assemble_m_blocks(W, base.wn, base.p, kinds, Lk)
        self._stage("solve:end")
        Y = self._kr_y(base, M) if M is not None else None
        H, h, c = ops.kr_predict_views(fac.Binv, base.wn, base.p, kinds)
        YH = self._kr_y(base, H) if H is not None else None
        mean, var = ops.kr_predict_rows(Y, R, YH, base.xn, h, c, new.d, new.w, base.P, base.nviews, Lk, scal)
        self._stage("predict:end")
        return (mean[:, :L] if Lk != L else mean), var

    def _predict_dense(self, X, Vs, Vs_new, m, chunk: int = 65536):
        vs_attached = self.get_vs()
        vs = vs_attached.detach()
        Xm, ldx = ops.as_matrix(X, "X")
        n, L = X.shape
        Lk = Xm.shape[1]
        if any(V.shape[0] != n for V in Vs):
            raise ValueError(f"X has {n} rows but the designs have {[V.shape[0] for V in Vs]}")
        n_total = self._n_total(n, X.device)
        if self.n_rand_effs == 1:
            Vm, ldv, Q, _ = self._cat(Vs, vs)
            fac, C, _ = self._factorise(Vm, ldv, Q, vs, True, Xm, ldx, Lk, vs_origin=vs_attached)
            W, scal = ops.solve_w(fac, C, C.stride(0), Lk, L, n_total)
            offsets = [0]
        else:
            stk = self._stack(Vs, Lk)
            Q, offsets = stk.Q, stk.offsets
            fac, C, _ = self._factorise(stk.V, stk.Q, stk.Q, vs, True, Xm, ldx, Lk, vs_origin=vs_attached, stk=stk)
            W, scal, _ = ops.solve_w_blocks(fac, C, C.stride(0), Lk, L, n_total)
        self._stage("solve:end")
        mean = torch.empty(m, Lk, device=X.device, dtype=torch.float32)
        var = torch.empty(m, 1, device=X.device, dtype=torch.float32)
        pW = pB = None
        for a in range(0, m, chunk):
            b = min(m, a + chunk)
            if len(Vs_new) == 1:
                Vc, ldc = ops.as_matrix(Vs_new[0][a:b], "Vs_new[0]")
            else:     # the stacked rows, zero-padded per block as the training operand is
                Vc, ldc = torch.zeros(b - a, Q, device=X.device, dtype=torch.float32), Q
                for o, Vn in zip(offsets, Vs_new):
                    Vc[:, o:o + Vn.shape[1]] = Vn[a:b].detach()
            mc = b - a
            pV = ops.split_planes(Vc, ldc, mc, Q) if ops.planes_supported(mc, Q, Q) else None
            if pV is not None and ops.planes_supported(mc, Q, Lk):
                pW = pW or ops.split_planes(W, W.stride(0), Q, Lk)
                mean[a:b] = ops.am_planes(pV, pW, mc, Q, Lk)
            else:
                mean[a:b] = ops.am(Vc, ldc, W, W.stride(0), mc, Q, Lk)
            if pV is not None:
                pB = pB or ops.split_planes(fac.Binv, Q, Q, Q)
                VB = ops.am_planes(pV, pB, mc, Q, Q)
            else:
                VB = ops.am(Vc, ldc, fac.Binv, Q, mc, Q, Q)
            var[a:b] = ops.rows_dot(VB, Vc, Q, scal)
        self._stage("predict:end")
        return (mean[:, :L] if Lk != L else mean), var

    def nll(self, X: torch.Tensor, Vs: Sequence[torch.Tensor]) -> torch.Tensor:
        """gp.py:97-110.  Differentiable: backward applies the Taylor coefficients (the exact gradients
        of sum(nll), gp.py:185-221), i.e. it is exact for a uniform upstream gradient (`.sum()`,
        `.mean()`) -- the only way the reference ever differentiates it; any other upstream gradient raises.  With a
        KhatriRao from `Vmodel.lazy(d, w, requires_grad=True)` the gradient also reaches the tables (LazyVb.table_grads).
        """
        tables = ()
        if self.n_rand_effs == 1 and len(Vs) == 1 and isinstance(Vs[0], KhatriRao) and Vs[0].tables is not None:
            tables = Vs[0].tables     # Vmodel.lazy(..., requires_grad=True): the gradient reaches x0 and v0
        return _NllFunction.apply(self, X, self.lvs, len(Vs), *Vs, *tables)

    def nll_ineff(self, X: torch.Tensor, Vs: Sequence[torch.Tensor]) -> torch.Tensor:
        """gp.py:112-125: O(N^3) cross-check through the dense N x N covariance.  Test utility, stock torch."""
        vs = self.get_vs()
        V = torch.cat([torch.sqrt(vs[i]) * Vi for i, Vi in enumerate(Vs)], 1)
        K = V.mm(V.t()) + vs[-1] * torch.eye(X.shape[0], device=X.device, dtype=X.dtype)
        quad = (X * torch.linalg.solve(K, X)).sum(1, keepdim=True)
        return 0.5 * quad + 0.5 * X.shape[1] * torch.linalg.slogdet(K)[1] / X.shape[0]

    def taylor_expansion(self, X: torch.Tensor, Vs: Sequence[torch.Tensor], Xb: torch.Tensor,
                         Vbs: Sequence[torch.Tensor], vbs: torch.Tensor) -> torch.Tensor:
        """gp.py:127-133: (n x 1) surrogate with gradients to X, each V and lvs."""
        if self.n_rand_effs > 1:
            k = self.n_rand_effs
            if len(Vs) != k or len(Vbs) != k:
                raise ValueError(f"GP(n_rand_effs={k}) expects {k} designs in Vs and Vbs, got {len(Vs)} / {len(Vbs)}")
            if any(isinstance(V, (KhatriRao, _FactoredEffect)) for V in Vs):
                raise NotImplementedError("taylor_expansion takes dense designs: pass the minibatch rows (V[idx]) of "
                                          "each factored design")
            return ops._TaylorExpansionMulti.apply(X, self.lvs, Xb, vbs, *Vs, *Vbs)
        if len(Vs) != 1 or len(Vbs) != 1:
            raise NotImplementedError(f"expected one design matrix in Vs / Vbs, got {len(Vs)} / {len(Vbs)}")
        return ops._TaylorExpansion.apply(X, Vs[0], self.lvs, Xb, Vbs[0], vbs)


class _NllFunction(torch.autograd.Function):
    """gp.py:97-110 with the Taylor coefficients as its backward.

    The coefficients are the exact gradients of sum_i nll_i (gp.py:185-221).  nll_i couples all rows through K^-1, so a
    NON-uniform upstream gradient (a weighted sum of the rows) has a different gradient, which this class does not
    implement: it raises instead of returning the uniform-weight one.  `.sum()`, `.mean()` and any constant multiple --
    every way the reference ever differentiates nll -- are exact."""

    @staticmethod
    def forward(ctx, gp: GP, X, lvs, nV, *Vs_tables):
        Vs, tables = Vs_tables[:nV], Vs_tables[nV:]
        want_grad = any(ctx.needs_input_grad[1:])
        dense = [torch.is_tensor(V) for V in Vs]
        ctx.dense = dense
        ctx.nV = nV
        ctx.lazy_vb = None
        with torch.no_grad():
            if want_grad:
                # a factored V (vmod.KhatriRao) has no Vb to form: its tables (given after Vs when they are attached)
                # get theirs through the slots, which needs B^-1 as the dense Vb does
                want_tables = any(ctx.needs_input_grad[4 + nV:])
                need_vb = want_tables or any(d and ng for d, ng in zip(dense, ctx.needs_input_grad[4:4 + nV]))
                Xb, Vbs, vbs, nll = gp.taylor_coeff(X, list(Vs), need_vb=need_vb)
                saved = [Vb for Vb, d in zip(Vbs, dense) if d and torch.is_tensor(Vb)]
                ctx.n_vb = len(saved)
                if want_tables:
                    ctx.lazy_vb = Vbs[0]
                ctx.save_for_backward(Xb, vbs, gp.get_vs().detach(), *saved)
            else:
                nll = gp._coefficients(X, list(Vs), False)["nll"]
        return nll

    @staticmethod
    def backward(ctx, g):
        Xb, vbs, vs, *Vbs = ctx.saved_tensors
        gmin, gmax = torch.aminmax(g.detach())
        gbar = float(gmax)
        if float(gmin) != gbar:
            raise NotImplementedError(
                "GP.nll: backward is implemented for a uniform upstream gradient only (nll.sum(), nll.mean(), or a "
                "constant multiple); a per-row weighting couples the rows through K^-1 and needs a second solve")
        gX = gbar * Xb if ctx.needs_input_grad[1] else None
        glvs = gbar * vs * (vbs - (vbs * vs).sum()) if ctx.needs_input_grad[2] else None
        it = iter(Vbs)
        gVs = []
        for d, need in zip(ctx.dense, ctx.needs_input_grad[4:4 + ctx.nV]):
            Vb = next(it) if (d and ctx.n_vb) else None
            gVs.append(gbar * Vb if (need and Vb is not None) else None)
        n_tables = len(ctx.needs_input_grad) - 4 - ctx.nV
        gtables = [None] * n_tables
        if ctx.lazy_vb is not None:
            gx, gw = ctx.lazy_vb.table_grads()
            gtables = [gbar * gx if ctx.needs_input_grad[4 + ctx.nV] else None,
                       gbar * gw if ctx.needs_input_grad[5 + ctx.nV] else None]
        return (None, gX, glvs, None, *gVs, *gtables)
