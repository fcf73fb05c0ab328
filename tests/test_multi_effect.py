"""GP(n_rand_effs=k) without a GPU: the oracle's k-design Taylor coefficients against fp64 autograd (they pin the
specification: there are no golden vectors for k > 1), the host logic of the drop-in class on the CPU stand-in engine
(tests/fake_engine.py plus stand-ins for the k-design entries, defined here), and argument validation of the new C
entries."""
import os

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import fake_engine
from conftest import rel_err
from gppvae_b200 import ops as real_ops
from gppvae_b200._lib import NSCAL, S_LOGDETB, S_TRBINV, S_V0, S_VN, S_XB2
from oracle import gp_oracle as oracle

LVS3 = (2.0, -3.0, 0.0, -1.0)
LVS2 = (0.5, -2.0, -1.0)


# ---------------------------------------------------------------- stand-ins for the k-design entries (fp64, CPU)
def factor_blocks(G, ldg, widths, vs, want_binv):
    vs = vs.detach().double()
    Q = sum(widths)
    d = torch.cat([vs[i].sqrt().expand(w) for i, w in enumerate(widths)])
    B = torch.eye(Q, dtype=torch.float64) + d[:, None] * d[None, :] * G[:, :Q].double() / vs[-1]
    Lc = torch.linalg.cholesky(B)
    Binv = torch.cholesky_inverse(Lc)
    DBD = d[:, None] * Binv * d[None, :]
    scal = torch.zeros(NSCAL, dtype=torch.float64)
    scal[S_V0], scal[S_VN] = 1.0, vs[-1]
    scal[S_LOGDETB] = 2 * Lc.diagonal().log().sum()
    scal[S_TRBINV] = Binv.diagonal().sum()
    blk = torch.zeros(2 * len(widths), dtype=torch.float64)
    o = 0
    for i, w in enumerate(widths):
        blk[2 * i] = Binv.diagonal()[o:o + w].sum()
        o += w
    # the state plays Linv'^T Linv' = D B^-1 D for fake_engine.solve_w
    return real_ops.Factorisation(Q, DBD, scal, DBD.to(torch.float32) if want_binv else None, list(widths), blk)


def solve_w_blocks(f, C, ldc, L, L_true, n_total):
    W, scal = fake_engine.solve_w(f, C, ldc, L, L_true, n_total)
    blk = f.blk.clone()
    o = 0
    for i, w in enumerate(f.widths):
        blk[2 * i + 1] = (W[o:o + w].double() ** 2).sum()
        o += w
    return W, scal, blk


def vbs_blocks(scal, blk, vs, widths, n_total, L):
    vs = vs.detach().double()
    out = [-0.5 * blk[2 * i + 1] / vs[i] ** 2 + 0.5 * L * (w - blk[2 * i]) / vs[i] for i, w in enumerate(widths)]
    out.append(-0.5 * scal[S_XB2] + 0.5 * L * (n_total - sum(widths) + scal[S_TRBINV]) / vs[-1])
    return torch.stack(out).to(torch.float32)


def x_minus_am(X, ldx, A, lda, M, ldm, n, k, m, alpha):
    return (alpha * (X.double() - A.double()[:, :k] @ M.double())).to(torch.float32)


def install(monkeypatch):
    fake_engine.install(monkeypatch)
    for name, fn in (("factor_blocks", factor_blocks), ("solve_w_blocks", solve_w_blocks), ("vbs_blocks", vbs_blocks),
                     ("x_minus_am", x_minus_am)):
        monkeypatch.setattr(real_ops, name, fn)
    real_ops.STACKED.invalidate()


def _problem(n=60, p=3, q=9, L=6, seed=0, k=3):
    """Z and the designs [Khatri-Rao p*q, xn[d] p, wn[w] q][:k] (q = 9 views: widths 27 -> 28, 9 -> 12)."""
    g = torch.Generator().manual_seed(seed)
    xn = oracle.unit_rows(torch.randn(n // 3 + 1, p, generator=g))
    wn = oracle.unit_rows(torch.eye(q) + 0.5 * torch.randn(q, q, generator=g))
    d = torch.randint(0, xn.shape[0], (n,), generator=g)
    w = torch.randint(0, q, (n,), generator=g)
    Vs = [oracle.feature_map(xn, wn, d, w), xn[d], wn[w]][:k]
    Z = 0.5 * torch.randn(n, L, generator=g) + Vs[0] @ torch.randn(Vs[0].shape[1], L, generator=g)
    return Z, Vs


# ---------------------------------------------------------------- the specification: oracle vs fp64 autograd
@pytest.mark.parametrize("k", [2, 3])
def test_oracle_taylor_coeff_is_the_gradient_of_nll(k):
    Z, Vs = _problem(k=k)
    lvs = torch.tensor((LVS3 if k == 3 else LVS2), dtype=torch.float64)
    Zd = Z.double().requires_grad_(True)
    Vd = [V.double().requires_grad_(True) for V in Vs]
    vs = torch.softmax(lvs, 0).requires_grad_(True)
    U, UBi, Shb = oracle.woodbury_factor(Vd, vs)
    nll = oracle._row_nll(Zd, oracle.woodbury_solve(Zd, U, UBi, vs), Shb, vs)
    nll.sum().backward()
    Xb, Vbs, vbs, out = oracle.taylor_coeff(Z.double(), [V.double() for V in Vs], lvs)
    assert vbs.shape == (k + 1,) and len(Vbs) == k
    assert rel_err(out, nll.detach()) < 1e-12
    assert rel_err(Xb, Zd.grad) < 1e-10
    for i in range(k):
        assert rel_err(Vbs[i], Vd[i].grad) < 1e-10, i
    assert rel_err(vbs, vs.grad) < 1e-10
    assert rel_err(oracle.nll(Z.double(), [V.double() for V in Vs], lvs),
                   oracle.nll_dense(Z.double(), [V.double() for V in Vs], lvs)) < 1e-10


# ---------------------------------------------------------------- host logic on the stand-in engine
@pytest.mark.parametrize("k", [2, 3])
def test_gp_k_designs_against_oracle(monkeypatch, k):
    from gppvae_b200 import GP
    install(monkeypatch)
    Z, Vs = _problem(k=k)
    lvs = LVS3 if k == 3 else LVS2
    gp = GP(n_rand_effs=k)
    assert gp.lvs.shape == (k + 1,) and list(gp.state_dict()) == ["lvs"]
    with torch.no_grad():
        gp.lvs.copy_(torch.tensor(lvs))
    Xb, Vbs, vbs, nll = gp.taylor_coeff(Z, Vs)
    oXb, oVbs, ovbs, onll = oracle.taylor_coeff(Z.double(), [V.double() for V in Vs], torch.tensor(lvs).double())
    assert [Vb.shape for Vb in Vbs] == [V.shape for V in Vs]        # 27 and 9 columns: padded inside, true width out
    assert rel_err(Xb, oXb) < 1e-5 and rel_err(nll, onll) < 1e-5 and rel_err(vbs, ovbs) < 1e-5
    for i in range(k):
        assert rel_err(Vbs[i], oVbs[i]) < 1e-4, i
    _, Vbs0, vbs0, nll0 = gp.taylor_coeff(Z, Vs, need_vb=False)
    assert Vbs0 == [None] * k and torch.equal(vbs0, vbs) and torch.equal(nll0, nll)
    # nll: backward applies the coefficients to X, every design and all k + 1 log-variances
    Zl = Z.clone().requires_grad_(True)
    Vl = [V.clone().requires_grad_(True) for V in Vs]
    gp.zero_grad()
    gp.nll(Zl, Vl).sum().backward()
    Zd = Z.double().requires_grad_(True)
    Vd = [V.double().requires_grad_(True) for V in Vs]
    lvd = torch.tensor(lvs, dtype=torch.float64, requires_grad=True)
    oracle.nll(Zd, Vd, lvd).sum().backward()
    assert rel_err(Zl.grad, Zd.grad) < 1e-5 and rel_err(gp.lvs.grad, lvd.grad) < 1e-5
    for i in range(k):
        assert rel_err(Vl[i].grad, Vd[i].grad) < 1e-4, i
    assert rel_err(gp.nll_ineff(Z, Vs).detach(), onll) < 1e-4


def test_u_ubi_shb_then_taylor_coeff_hits_the_cache(monkeypatch):
    from gppvae_b200 import GP
    install(monkeypatch)
    Z, Vs = _problem()
    gp = GP(n_rand_effs=3)
    with torch.no_grad():
        gp.lvs.copy_(torch.tensor(LVS3))
    vs = gp.get_vs()
    U, UBi, Shb = gp.U_UBi_Shb(Vs, vs, want_binv=True)
    assert gp.cache_hits == 0
    Xb, _, _, _ = gp.taylor_coeff(Z, Vs)
    assert gp.cache_hits == 1
    Ur, UBir, Shbr = oracle.woodbury_factor([V.double() for V in Vs], vs.detach().double())
    assert U.shape == Ur.shape and rel_err(U.dense(), Ur) < 1e-6 and rel_err(UBi.dense(), UBir) < 1e-5
    assert rel_err(torch.sort(Shb.value(), descending=True).values, Shbr) < 1e-5
    assert rel_err(gp.solve(Z, U, UBi, vs), Xb) < 1e-5
    # a new version of one design misses; so does a new design of the same shape
    Vs[2].mul_(1.0)
    gp.taylor_coeff(Z, Vs)
    assert gp.cache_hits == 1
    gp.taylor_coeff(Z, [Vs[0], Vs[1], Vs[2].clone()])
    assert gp.cache_hits == 1


def test_stacked_entry_does_not_keep_designs_alive(monkeypatch):
    import weakref
    from gppvae_b200 import GP
    install(monkeypatch)
    Z, Vs = _problem()
    gp = GP(n_rand_effs=3)
    gp.taylor_coeff(Z, Vs)
    assert real_ops.STACKED.entry is not None
    ref = weakref.ref(Vs[1])
    del Vs
    assert ref() is None and real_ops.STACKED.entry is None


def test_argument_errors(monkeypatch):
    from gppvae_b200 import GP
    from gppvae_b200.vmod import KhatriRao
    install(monkeypatch)
    Z, Vs = _problem()
    gp = GP(n_rand_effs=3)
    for bad in (Vs[:2], Vs + [Vs[1]]):
        with pytest.raises(ValueError):
            gp.taylor_coeff(Z, bad)
        with pytest.raises(ValueError):
            gp.U_UBi_Shb(bad, gp.get_vs())
    g = torch.Generator().manual_seed(1)
    kr = KhatriRao(oracle.unit_rows(torch.randn(21, 3, generator=g)), oracle.unit_rows(torch.randn(9, 9, generator=g)),
                   torch.randint(0, 21, (60,), generator=g), torch.randint(0, 9, (60,), generator=g))
    with pytest.raises(NotImplementedError):
        gp.taylor_coeff(Z, [kr, Vs[1], Vs[2]])
    with pytest.raises(NotImplementedError):
        gp.taylor_expansion(Z, [kr, Vs[1], Vs[2]], Z, Vs, torch.zeros(4))
    with pytest.raises(ValueError):
        gp.taylor_expansion(Z, Vs[:2], Z, Vs[:2], torch.zeros(4))
    for n_bad in (0, 17, 1.5):
        with pytest.raises(ValueError):
            GP(n_rand_effs=n_bad)
    with pytest.raises(NotImplementedError):
        GP(n_rand_effs=2, vsum2one=False)
    with pytest.raises(NotImplementedError):      # k = 1 keeps its errors
        GP().taylor_coeff(Z, Vs[:2])


def _shard_worker(rank, world, port, out):
    from _pytest.monkeypatch import MonkeyPatch
    from gppvae_b200 import GP
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    mpch = MonkeyPatch()
    install(mpch)
    try:
        Z, Vs = _problem()
        n = Z.shape[0]
        rows = slice(0, 37) if rank == 0 else slice(37, n)         # unequal shards
        gp = GP(n_rand_effs=3).shard_rows()
        with torch.no_grad():
            gp.lvs.copy_(torch.tensor(LVS3))
        Xb, Vbs, vbs, nll = gp.taylor_coeff(Z[rows].contiguous(), [V[rows].contiguous() for V in Vs])
        torch.save(dict(Xb=Xb, Vbs=Vbs, vbs=vbs, nll=nll), os.path.join(out, f"r{rank}.pt"))
    finally:
        mpch.undo()
        dist.destroy_process_group()


def test_row_sharding_world2_gloo(tmp_path, monkeypatch):
    from gppvae_b200 import GP
    port = 29500 + (os.getpid() % 2000) + 7
    mp.spawn(_shard_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    install(monkeypatch)
    Z, Vs = _problem()
    gp = GP(n_rand_effs=3)
    with torch.no_grad():
        gp.lvs.copy_(torch.tensor(LVS3))
    Xb, Vbs, vbs, nll = gp.taylor_coeff(Z, Vs)
    r0, r1 = (torch.load(os.path.join(tmp_path, f"r{r}.pt")) for r in (0, 1))
    assert torch.equal(r0["vbs"], r1["vbs"]) and rel_err(r0["vbs"], vbs) < 1e-5
    assert rel_err(torch.cat([r0["Xb"], r1["Xb"]]), Xb) < 1e-5 and rel_err(torch.cat([r0["nll"], r1["nll"]]), nll) < 1e-5
    for i in range(3):
        assert rel_err(torch.cat([r0["Vbs"][i], r1["Vbs"][i]]), Vbs[i]) < 1e-4, i


# ---------------------------------------------------------------- C entries: validation before any device work
@pytest.fixture(scope="module")
def lib():
    from gppvae_b200 import _lib, build
    build.build()
    return _lib.load(build_if_missing=False)


def test_new_c_entries_validate_without_a_device(lib):
    from gppvae_b200._lib import host_i32, host_i64, host_ptrs
    c_ok, c_odd = host_i32([128, 16, 8]), host_i32([128, 6, 8])
    p = 1 << 12   # a non-null, 16-byte aligned fake device address: validation must fail before it is used
    assert lib.gpp_split_planes_stacked(3, host_ptrs([p, p, p]), host_i64([128, 16, 8]), c_odd, 1536, 0, 256, 1 << 30,
                                        None, 0, None) == -1
    assert b"split_planes_stacked" in lib.gpp_last_error()
    assert lib.gpp_split_planes_stacked(0, None, None, None, 1536, 0, 256, 1 << 30, None, 0, None) == -1
    assert lib.gpp_split_planes_stacked(3, host_ptrs([p, None, p]), host_i64([128, 16, 8]), c_ok, 1536, 0, 256,
                                        1 << 30, None, 0, None) == -1
    assert lib.gpp_split_planes_stacked(3, host_ptrs([p, p, p]), host_i64([128, 16, 8]), c_ok, 1536, 0, 256, 16, None, 0,
                                        None) == -1                                       # planes buffer too small
    assert lib.gpp_factor_blocks(p, 152, 3, c_odd, p, 0, None, p, p, p, 1 << 30, None) == -1
    assert lib.gpp_factor_blocks(p, 152, 17, c_ok, p, 0, None, p, p, p, 1 << 30, None) == -1
    assert lib.gpp_factor_blocks(p, 100, 3, c_ok, p, 0, None, p, p, p, 1 << 30, None) == -1   # ldg < Q
    assert lib.gpp_factor_blocks(p, 152, 3, c_ok, p, 0, None, p, None, p, 1 << 30, None) == -1  # null blk
    assert lib.gpp_factor_blocks(p, 152, 3, c_ok, p, 1, None, p, p, p, 1 << 30, None) == -1     # Binv missing
    assert lib.gpp_factor_blocks(p, 152, 3, c_ok, p, 0, None, p, p, p, 16, None) == -3          # state too small
    assert lib.gpp_solve_w_blocks(p, 64, 3, c_ok, 64, 65, 100, p, 64, p, p, p, 1 << 30, p, 1 << 30, None) == -1
    assert lib.gpp_solve_w_blocks(p, 64, 3, c_ok, 64, 64, 100, p, 64, p, None, p, 1 << 30, p, 1 << 30, None) == -1
    assert lib.gpp_solve_w_blocks(p, 64, 3, c_ok, 64, 64, 100, p, 64, p, p, p, 16, p, 1 << 30, None) == -3
    assert lib.gpp_vbs_blocks(p, p, p, 3, c_odd, 100, 64, p, None) == -1
    assert lib.gpp_vbs_blocks(p, None, p, 3, c_ok, 100, 64, p, None) == -1
    assert lib.gpp_taylor_expansion_fwd_multi(p, 64, p, 64, 17, host_ptrs([p] * 17), host_i64([4] * 17),
                                              host_ptrs([p] * 17), host_i64([4] * 17), host_i32([4] * 17), 8, 64, p, p, p,
                                              None) == -1
    assert lib.gpp_taylor_expansion_fwd_multi(p, 64, p, 64, 2, host_ptrs([p, p]), host_i64([8, 8]), host_ptrs([p, p + 4]),
                                              host_i64([8, 8]), host_i32([8, 8]), 8, 64, p, p, p, None) == -1  # misaligned
    assert lib.gpp_taylor_expansion_bwd_multi(p, p, 64, 2, host_ptrs([p, p]), host_i64([8, 8]), host_i32([8, 6]), 8, 64, p,
                                              p, None, 64, None, None, None, None) == -1
    assert lib.gpp_taylor_expansion_bwd_multi(p, p, 64, 2, host_ptrs([p, p]), host_i64([8, 8]), host_i32([8, 8]), 8, 64, p,
                                              p, None, 64, host_ptrs([p, p]), host_i64([4, 8]), None, None) == -1  # ldgv
    # workspace queries: 0 for bad arguments, enough for the state / solve otherwise
    assert lib.gpp_factor_blocks_state_bytes(152, 0) == 0 and lib.gpp_solve_blocks_workspace_bytes(152, 64, 17) == 0
    assert lib.gpp_factor_blocks_state_bytes(152, 3) > lib.gpp_factor_state_bytes(152)
    assert lib.gpp_solve_blocks_workspace_bytes(152, 64, 3) > lib.gpp_solve_workspace_bytes(152, 64)
    assert lib.gpp_split_stacked_workspace_bytes(1536, 3, c_ok) >= lib.gpp_split_workspace_bytes(1536, 128)
