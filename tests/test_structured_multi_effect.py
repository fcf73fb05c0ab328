"""GP(n_rand_effs=k) on factored designs (the Khatri-Rao, object-only and view-only designs of Vmodel.lazy_effects)
without a GPU: the host logic of the structured k-design route on the CPU stand-in engine (tests/fake_engine.py, the
k-design stand-ins of tests/test_multi_effect.py, and fp64 stand-ins for the new entries defined here, written from the
block table of DESIGN 5.7) against the oracle on the dense designs, and argument validation of the new C entries."""
import os

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import test_multi_effect as k_designs
from conftest import rel_err
from gppvae_b200 import ops as real_ops
from gppvae_b200._lib import S_QUAD, S_ROWCONST, S_VN, S_XB2
from oracle import gp_oracle as oracle

LVS3 = (2.0, -3.0, 0.0, -1.0)
LVS2 = (0.5, -2.0, -1.0)


# ---------------------------------------------------------------- stand-ins for the new entries (fp64, CPU)
def _wpad(wn):
    nv, q = wn.shape
    w = torch.zeros(nv, real_ops.round4(q), dtype=torch.float64)
    w[:, :q] = wn.double()
    return w


def kr_view_sums(X, ldx, order, slot_start, xn, nviews, L, with_x):
    P, p = xn.shape
    counts = slot_start[1:] - slot_start[:-1]
    slot = torch.repeat_interleave(torch.arange(P * nviews), counts)
    z = torch.zeros(nviews, L, dtype=torch.float64)
    z.index_add_(0, slot % nviews, X.double()[order[: slot.numel()]][:, :L])
    if not with_x:
        return z.to(torch.float32)
    cnt = counts.view(P, nviews).double()
    return torch.cat([z, cnt.t() @ xn.double(), cnt.sum(0)[:, None], torch.zeros(nviews, 3, dtype=torch.float64)],
                     1).to(torch.float32)


def kr_assemble_gc_blocks(ST, VM, wn, p, kinds, L, with_g):
    nv, q = wn.shape
    w, wp = wn.double(), _wpad(wn)
    off = nv * p if with_g else 0
    C = {}
    if ST is not None:
        T = ST.double()[:, off:].view(p, nv, L)
        C["kr"] = torch.einsum("vk,jvl->jkl", w, T).reshape(p * q, L)
        C["object"] = T.sum(1)
    if VM is not None:
        C["view"] = wp.t() @ VM.double()[:, :L]
    if not with_g:
        return torch.cat([C[k] for k in kinds]).to(torch.float32)
    S = ST.double()[:, :off].view(p, nv, p) if ST is not None else None
    if VM is not None:
        a, cnt = VM.double()[:, L:L + p], VM.double()[:, L + p]
    G = {}
    if S is not None:
        G["kr", "kr"] = torch.einsum("vk,vm,jvi->jkim", w, w, S).reshape(p * q, p * q)
        G["kr", "object"] = torch.einsum("vk,jvi->jki", w, S).reshape(p * q, p)
        G["object", "object"] = S.sum(1)
    if VM is not None:
        G["view", "view"] = torch.einsum("v,vk,vm->km", cnt, wp, wp)
        if S is not None:
            G["kr", "view"] = torch.einsum("vk,vm,vj->jkm", w, wp, a).reshape(p * q, -1)
            G["object", "view"] = a.t() @ wp

    def block(r, c):
        return G[r, c] if (r, c) in G else G[c, r].t()
    rows = [torch.cat([block(r, c) for c in kinds] + [C[r]], 1) for r in kinds]
    return torch.cat(rows).to(torch.float32)


def kr_assemble_m_blocks(W, wn, p, kinds, L):
    nv, q = wn.shape
    widths = real_ops.effect_widths(kinds, p, q)
    offs = dict(zip(kinds, [sum(widths[:i]) for i in range(len(kinds))]))
    Wd = W.double()
    M = torch.zeros(p, nv, L, dtype=torch.float64)
    if "kr" in offs:
        M += torch.einsum("vk,jkl->jvl", wn.double(), Wd[offs["kr"]:offs["kr"] + p * q].view(p, q, L))
    if "object" in offs:
        M += Wd[offs["object"]:offs["object"] + p][:, None, :]
    R = None
    if "view" in offs:
        R = (_wpad(wn) @ Wd[offs["view"]:offs["view"] + real_ops.round4(q)]).to(torch.float32)
    return M.reshape(p, nv * L).to(torch.float32), R


def kr_xb_nll_views(X, ldx, Y, R, d, w, P, nviews, L, scal):
    Yg = Y.double().view(P, nviews, L)[d, w] + R.double()[w]
    Xb = (X.double() - Yg) / scal[S_VN]
    quad = (X.double() * Xb).sum(1, keepdim=True)
    scal[S_XB2] = (Xb * Xb).sum()
    scal[S_QUAD] = quad.sum()
    return Xb.to(torch.float32), (0.5 * quad + scal[S_ROWCONST]).to(torch.float32)


def install(monkeypatch):
    k_designs.install(monkeypatch)
    for name, fn in (("kr_view_sums", kr_view_sums), ("kr_assemble_gc_blocks", kr_assemble_gc_blocks),
                     ("kr_assemble_m_blocks", kr_assemble_m_blocks), ("kr_xb_nll_views", kr_xb_nll_views)):
        monkeypatch.setattr(real_ops, name, fn)


def _tables(n=60, p=3, q=9, L=6, seed=0, rows=None):
    """Z, (xn, wn, d, w) and the dense designs {kind: V}; p = 3 and q = 9 exercise the padding of every block."""
    g = torch.Generator().manual_seed(seed)
    xn = oracle.unit_rows(torch.randn(n // 3 + 1, p, generator=g))
    wn = oracle.unit_rows(torch.eye(q) + 0.5 * torch.randn(q, q, generator=g))
    d = torch.randint(0, xn.shape[0], (n,), generator=g)     # some objects have no rows: empty slots
    w = torch.randint(0, q, (n,), generator=g)
    dense = dict(kr=oracle.feature_map(xn, wn, d, w), object=xn[d], view=wn[w])
    Z = 0.5 * torch.randn(n, L, generator=g) + dense["kr"] @ torch.randn(p * q, L, generator=g) + \
        dense["view"] @ torch.randn(q, L, generator=g)
    return Z, (xn, wn, d, w), dense


def _factored(tables, kinds, rows=slice(None)):
    from gppvae_b200.vmod import KhatriRao, ObjectEffect, ViewEffect
    xn, wn, d, w = tables
    kr = KhatriRao(xn, wn, d[rows].contiguous(), w[rows].contiguous())
    return [kr if k == "kr" else ObjectEffect(kr) if k == "object" else ViewEffect(kr) for k in kinds]


def _gp(k, lvs):
    from gppvae_b200 import GP
    gp = GP(n_rand_effs=k)
    with torch.no_grad():
        gp.lvs.copy_(torch.tensor(lvs))
    return gp


KIND_LISTS = [("kr", "object", "view"), ("kr", "view"), ("object", "view"), ("view", "kr", "object"), ("kr", "object")]


@pytest.mark.parametrize("kinds", KIND_LISTS, ids=["-".join(k) for k in KIND_LISTS])
def test_structured_k_designs_against_oracle(monkeypatch, kinds):
    install(monkeypatch)
    Z, tables, dense = _tables()
    k = len(kinds)
    lvs = LVS3 if k == 3 else LVS2
    Vs = _factored(tables, kinds)
    Vd = [dense[kd] for kd in kinds]
    assert [V.shape for V in Vs] == [V.shape for V in Vd]
    for V, D in zip(Vs, Vd):
        assert rel_err(V.dense(), D) < 1e-6
    gp = _gp(k, lvs)
    Xb, Vbs, vbs, nll = gp.taylor_coeff(Z, Vs)
    oXb, oVbs, ovbs, onll = oracle.taylor_coeff(Z.double(), [V.double() for V in Vd], torch.tensor(lvs).double())
    assert rel_err(Xb, oXb) < 1e-5 and rel_err(nll, onll) < 1e-5 and rel_err(vbs, ovbs) < 1e-5
    idx = torch.tensor([5, 0, 17, 5, 59])
    for i in range(k):
        assert Vbs[i].shape == Vd[i].shape
        assert rel_err(Vbs[i][idx], oVbs[i][idx]) < 1e-4, i
        assert rel_err(Vbs[i].dense(chunk=16), oVbs[i]) < 1e-4, i
    _, Vbs0, vbs0, nll0 = gp.taylor_coeff(Z, Vs, need_vb=False)
    assert Vbs0 == [None] * k and torch.equal(vbs0, vbs) and torch.equal(nll0, nll)
    # nll: backward to X and the k + 1 log-variances (no gradient flows to a factored design)
    Zl = Z.clone().requires_grad_(True)
    gp.zero_grad()
    gp.nll(Zl, Vs).sum().backward()
    Zd = Z.double().requires_grad_(True)
    lvd = torch.tensor(lvs, dtype=torch.float64, requires_grad=True)
    oracle.nll(Zd, [V.double() for V in Vd], lvd).sum().backward()
    assert rel_err(Zl.grad, Zd.grad) < 1e-5 and rel_err(gp.lvs.grad, lvd.grad) < 1e-5


def test_vb_rows_are_formed_once_per_index(monkeypatch):
    install(monkeypatch)
    calls = []
    vb = real_ops.vb
    monkeypatch.setattr(real_ops, "vb", lambda *a: calls.append(1) or vb(*a))
    Z, tables, _ = _tables()
    Vs = _factored(tables, ("kr", "object", "view"))
    _, Vbs, _, _ = _gp(3, LVS3).taylor_coeff(Z, Vs)
    idx = torch.arange(10, 20)
    [Vb[idx] for Vb in Vbs]
    assert len(calls) == 1
    [Vb[idx.clone()] for Vb in Vbs]
    assert len(calls) == 1
    Vbs[0][idx + 1]
    assert len(calls) == 2


def test_u_ubi_shb_then_solve_hits_the_cache(monkeypatch):
    install(monkeypatch)
    Z, tables, dense = _tables()
    kinds = ("view", "kr", "object")
    Vs = _factored(tables, kinds)
    gp = _gp(3, LVS3)
    vs = gp.get_vs()
    U, UBi, Shb = gp.U_UBi_Shb(Vs, vs, want_binv=True)
    assert gp.cache_hits == 0
    Xs = gp.solve(Z, U, UBi, vs)
    Xb, _, _, _ = gp.taylor_coeff(Z, Vs)
    assert gp.cache_hits == 1
    Vd = [dense[k].double() for k in kinds]
    Ur, UBir, Shbr = oracle.woodbury_factor(Vd, vs.detach().double())
    assert U.shape == Ur.shape and rel_err(U.dense(), Ur) < 1e-6 and rel_err(UBi.dense(), UBir) < 1e-5
    assert rel_err(torch.sort(Shb.value(), descending=True).values, Shbr) < 1e-5
    assert rel_err(Xs, Xb) < 1e-5
    oXb, _, _, _ = oracle.taylor_coeff(Z.double(), Vd, torch.tensor(LVS3).double())
    assert rel_err(Xs, oXb) < 1e-5
    # other designs (even over the same tables) miss
    gp.taylor_coeff(Z, _factored(tables, kinds))
    assert gp.cache_hits == 1


def test_transpose_products(monkeypatch):
    from gppvae_b200.vmod import effect_kind
    install(monkeypatch)
    Z, tables, dense = _tables(L=7)
    for V in _factored(tables, ("kr", "object", "view")):
        kind = effect_kind(V)
        ref = dense[kind].double().t() @ Z.double()
        out = V.t().mm(Z)
        assert out.shape == ref.shape and rel_err(out, ref) < 1e-6, kind


def test_lazy_effects_and_argument_errors(monkeypatch):
    from gppvae_b200 import GP, ObjectEffect, ViewEffect, Vmodel
    from gppvae_b200.vmod import KhatriRao
    install(monkeypatch)
    torch.manual_seed(0)
    Z, tables, dense = _tables()
    xn, wn, d, w = tables
    vm = Vmodel(xn.shape[0], wn.shape[0], xn.shape[1], wn.shape[1])
    Vs = vm.lazy_effects(d, w)
    assert isinstance(Vs[0], KhatriRao) and isinstance(Vs[1], ObjectEffect) and isinstance(Vs[2], ViewEffect)
    assert Vs[1].kr is Vs[0] and Vs[2].kr is Vs[0]
    assert vm.lazy_effects(d, w)[0]._index is Vs[0]._index          # the slot index is built once per (d, w)
    assert torch.equal(Vs[2].dense(), vm.v().detach()[w]) and torch.equal(Vs[1][d[:4] * 0 + 2], vm.x().detach()[d[2:3]].expand(4, -1))
    for bad in ((), ("kr", "kr"), ("object", "time")):
        with pytest.raises(ValueError):
            vm.lazy_effects(d, w, kinds=bad)
    gp = GP(n_rand_effs=3)
    other = _factored(tables, ("kr", "object", "view"))
    with pytest.raises(ValueError):       # built over different slot indices / tables
        gp.taylor_coeff(Z, [Vs[0], other[1], Vs[2]])
    with pytest.raises(ValueError):
        gp.U_UBi_Shb([Vs[0], Vs[1], other[2]], gp.get_vs())
    with pytest.raises(ValueError):       # a kind twice
        gp.taylor_coeff(Z, [Vs[0], Vs[1], ObjectEffect(Vs[0])])
    with pytest.raises(ValueError):       # wrong number of designs
        gp.taylor_coeff(Z, Vs[:2])
    with pytest.raises(NotImplementedError):   # factored and dense mixed
        gp.taylor_coeff(Z, [Vs[0], Vs[1], dense["view"]])
    with pytest.raises(NotImplementedError):
        gp.U_UBi_Shb([dense["kr"], Vs[1], Vs[2]], gp.get_vs())
    with pytest.raises(NotImplementedError):
        gp.taylor_expansion(Z, Vs, Z, [dense[k] for k in ("kr", "object", "view")], torch.zeros(4))
    with pytest.raises(ValueError):
        gp.taylor_coeff(Z[:10], Vs)


def _shard_worker(rank, world, port, out):
    from _pytest.monkeypatch import MonkeyPatch
    from gppvae_b200 import GP
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    mpch = MonkeyPatch()
    install(mpch)
    try:
        Z, tables, _ = _tables()
        n = Z.shape[0]
        rows = slice(0, 37) if rank == 0 else slice(37, n)         # unequal shards
        Vs = _factored(tables, ("kr", "object", "view"), rows)
        gp = GP(n_rand_effs=3).shard_rows()
        with torch.no_grad():
            gp.lvs.copy_(torch.tensor(LVS3))
        Xb, Vbs, vbs, nll = gp.taylor_coeff(Z[rows].contiguous(), Vs)
        idx = torch.arange(Z[rows].shape[0])
        torch.save(dict(Xb=Xb, Vbs=[Vb[idx] for Vb in Vbs], vbs=vbs, nll=nll), os.path.join(out, f"r{rank}.pt"))
    finally:
        mpch.undo()
        dist.destroy_process_group()


def test_row_sharding_world2_gloo(tmp_path, monkeypatch):
    port = 29500 + (os.getpid() % 2000) + 11
    mp.spawn(_shard_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    install(monkeypatch)
    Z, tables, dense = _tables()
    oXb, oVbs, ovbs, onll = oracle.taylor_coeff(Z.double(), [dense[k].double() for k in ("kr", "object", "view")],
                                                torch.tensor(LVS3).double())
    r0, r1 = (torch.load(os.path.join(tmp_path, f"r{r}.pt")) for r in (0, 1))
    assert torch.equal(r0["vbs"], r1["vbs"]) and rel_err(r0["vbs"], ovbs) < 1e-5
    assert rel_err(torch.cat([r0["Xb"], r1["Xb"]]), oXb) < 1e-5
    assert rel_err(torch.cat([r0["nll"], r1["nll"]]), onll) < 1e-5
    for i in range(3):
        assert rel_err(torch.cat([r0["Vbs"][i], r1["Vbs"][i]]), oVbs[i]) < 1e-4, i


# ---------------------------------------------------------------- C entries: validation before any device work
@pytest.fixture(scope="module")
def lib():
    from gppvae_b200 import _lib, build
    build.build()
    return _lib.load(build_if_missing=False)


def test_new_c_entries_validate_without_a_device(lib):
    from gppvae_b200._lib import host_i32
    p = 1 << 12   # a non-null, 16-byte aligned fake device address: validation must fail before it is used
    big = 1 << 30
    three, dup, bad_kind = host_i32([0, 1, 2]), host_i32([0, 2, 0]), host_i32([0, 3])
    # view sums: shapes, leading dimensions, alignment, workspace
    assert lib.gpp_kr_view_sums(p, 64, p, p, p, 100, 6, 9, 64, 1, p, 80, p, big, None) == -1          # p % 4
    assert lib.gpp_kr_view_sums(p, 64, p, p, None, 100, 8, 9, 64, 1, p, 80, p, big, None) == -1       # xn with with_x
    assert lib.gpp_kr_view_sums(p, 64, p, p, p, 100, 8, 9, 64, 1, p, 72, p, big, None) == -1          # ldvm < L + p + 4
    assert lib.gpp_kr_view_sums(p, 64, p, p, p, 100, 8, 9, 64, 1, p + 4, 76, p, big, None) == -1      # misaligned VM
    assert lib.gpp_kr_view_sums(p, 64, p, p, p, 100, 8, 9, 64, 1, p, 76, p, 16, None) == -3           # workspace
    assert b"kr_view_sums" in lib.gpp_last_error()
    assert lib.gpp_kr_view_sums_workspace_bytes(0, 8, 9, 64, 1) == 0
    assert lib.gpp_kr_view_sums_workspace_bytes(100, 8, 9, 64, 1) > lib.gpp_kr_view_sums_workspace_bytes(100, 8, 9, 64, 0)
    # block assembly (p = 8, q = 9, nviews = 9, L = 64: ldst >= 648, ldvm >= 76, Q = 72 + 8 + 12, ldgc >= 156)
    assert lib.gpp_kr_assemble_gc_blocks(p, 648, p, 76, p, 8, 9, 9, 64, 3, dup, 1, p, 156, None) == -1
    assert lib.gpp_kr_assemble_gc_blocks(p, 648, p, 76, p, 8, 9, 9, 64, 2, bad_kind, 1, p, 156, None) == -1
    assert lib.gpp_kr_assemble_gc_blocks(p, 648, p, 76, p, 8, 9, 9, 64, 4, three, 1, p, 156, None) == -1
    assert lib.gpp_kr_assemble_gc_blocks(p, 648, None, 0, p, 8, 9, 9, 64, 3, three, 1, p, 156, None) == -1   # VM for view
    assert lib.gpp_kr_assemble_gc_blocks(None, 0, p, 76, p, 8, 9, 9, 64, 3, three, 1, p, 156, None) == -1    # ST for kr
    assert lib.gpp_kr_assemble_gc_blocks(p, 644, p, 76, p, 8, 9, 9, 64, 3, three, 1, p, 156, None) == -1    # ldst
    assert lib.gpp_kr_assemble_gc_blocks(p, 648, p, 72, p, 8, 9, 9, 64, 3, three, 1, p, 156, None) == -1    # ldvm
    assert lib.gpp_kr_assemble_gc_blocks(p, 648, p, 76, p, 8, 9, 9, 64, 3, three, 1, p, 152, None) == -1    # ldgc < Q + L
    assert b"kr_assemble_gc_blocks" in lib.gpp_last_error()
    # pass-2 pieces
    assert lib.gpp_kr_assemble_m_blocks(p, 64, p, 8, 9, 9, 64, 3, dup, p, 576, p, 64, None) == -1
    assert lib.gpp_kr_assemble_m_blocks(p, 64, p, 8, 9, 9, 64, 3, three, p, 576, None, 64, None) == -1     # R for view
    assert lib.gpp_kr_assemble_m_blocks(p, 64, p, 8, 9, 9, 64, 3, three, p, 512, p, 64, None) == -1        # ldm
    assert lib.gpp_kr_xb_nll_views(p, 64, p, 576, None, 64, p, p, 10, 5, 9, 64, p, p, 64, p, p, big, None) == -1
    assert lib.gpp_kr_xb_nll_views(p, 64, p, 576, p, 60, p, p, 10, 5, 9, 64, p, p, 64, p, p, big, None) == -1  # ldr
    assert lib.gpp_kr_xb_nll_views(p, 64, p, 576, p, 64, p, p, 10, 5, 9, 64, p, p, 64, p, p, 16, None) == -3
