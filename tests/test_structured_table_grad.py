"""The NLL gradient to the tables on the structured route (Vmodel.lazy(..., requires_grad=True), DESIGN 5.8) without a
GPU: the host logic of LazyVb.table_grads and _NllFunction on the CPU stand-in engine (tests/fake_engine.py plus fp64
stand-ins for the two new entries, defined here from the formulas of the header) against the fp64 oracle, a two-rank
gloo run on unequal shards, and argument validation of the new C entries."""
import os

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import fake_engine
from conftest import rel_err
from gppvae_b200 import ops as real_ops
from oracle import gp_oracle as oracle


# ---------------------------------------------------------------- stand-ins for the new entries (fp64, CPU)
def kr_grad_rhs(Binv, W, wn, p, L, alpha):
    nv, q = wn.shape
    w, B4, W3 = wn.double(), Binv.double().view(p, q, p, q), W.double().view(p, q, L)
    H = torch.einsum("va,iajb,vb->vij", w, B4, w)                 # H_v[j', j]
    M = torch.einsum("vk,jkl->vjl", w, W3)                         # M_v[j, l]
    return torch.cat([alpha * H.reshape(nv * p, p), -M.transpose(1, 2).reshape(nv * L, p)]).to(torch.float32)


def kr_grad_views(ST, Binv, W, wn, p, L, alpha):
    nv, q = wn.shape
    w, B4, W3 = wn.double(), Binv.double().view(p, q, p, q), W.double().view(p, q, L)
    S = ST.double()[:, : nv * p].view(p, nv, p)                   # S[j, v, j'] = S_v[j, j']
    T = ST.double()[:, nv * p:].view(p, nv, L)                    # T[j, v, l] = T_v[j, l]
    gw = alpha * torch.einsum("jvi,vc,icjk->vk", S, w, B4) - torch.einsum("jvl,jkl->vk", T, W3)
    return gw.to(torch.float32)


def install(monkeypatch):
    fake_engine.install(monkeypatch)
    monkeypatch.setattr(real_ops, "kr_grad_rhs", kr_grad_rhs)
    monkeypatch.setattr(real_ops, "kr_grad_views", kr_grad_views)


def _problem(n=90, P=25, nv=6, p=3, q=5, L=7, seed=0):
    """A Vmodel with random tables, rows with repeated and empty slots, and latents with structure; p, q and L are not
    multiples of 4."""
    from gppvae_b200 import Vmodel
    g = torch.Generator().manual_seed(seed)
    vm = Vmodel(P, nv, p, q)
    with torch.no_grad():
        vm.x0.copy_(torch.randn(P, p, generator=g))
        vm.v0.copy_(torch.eye(nv, q) + 0.5 * torch.randn(nv, q, generator=g))
    d = torch.randint(0, P - 3, (n,), generator=g)        # the last objects have no rows: empty slots
    w = torch.randint(0, nv, (n,), generator=g)
    V = oracle.feature_map(vm.x0.detach().double(), vm.v0.detach().double(), d, w)
    Z = (0.5 * torch.randn(n, L, generator=g, dtype=torch.float64) + V @ torch.randn(p * q, L, generator=g,
                                                                                      dtype=torch.float64)).float()
    return vm, d, w, Z


def _gp(lvs):
    from gppvae_b200 import GP
    gp = GP()
    with torch.no_grad():
        gp.lvs.copy_(torch.tensor(lvs))
    return gp


def _oracle_table_grads(vm, d, w, Z, lvs, rows=slice(None)):
    """fp64 ground truth: the Khatri-Rao backward of the oracle's Vb (gp.py:185-221), chained through unit_rows."""
    x0 = vm.x0.detach().double().requires_grad_(True)
    v0 = vm.v0.detach().double().requires_grad_(True)
    V64 = oracle.feature_map(x0, v0, d[rows], w[rows])
    _, Vbs, _, _ = oracle.taylor_coeff(Z[rows].double(), [V64.detach()], torch.tensor(lvs, dtype=torch.float64))
    return torch.autograd.grad(V64, (x0, v0), Vbs[0])


@pytest.mark.parametrize("lvs", [(0.3, -0.5), (2.0, -4.0)])
def test_table_grads_against_oracle(monkeypatch, lvs):
    install(monkeypatch)
    vm, d, w, Z = _problem()
    gp = _gp(lvs)
    Zl = Z.clone().requires_grad_(True)
    gp.nll(Zl, [vm.lazy(d, w, requires_grad=True)]).sum().backward()
    gx, gv = _oracle_table_grads(vm, d, w, Z, lvs)
    assert rel_err(vm.x0.grad, gx) < 1e-5 and rel_err(vm.v0.grad, gv) < 1e-5
    # the gradients to X and lvs are those of the path without table gradients, value for value
    Z0 = Z.clone().requires_grad_(True)
    gp2 = _gp(lvs)
    gp2.nll(Z0, [vm.lazy(d, w)]).sum().backward()
    assert torch.equal(Zl.grad, Z0.grad) and torch.equal(gp.lvs.grad, gp2.lvs.grad)


def test_default_lazy_gives_the_tables_no_gradient(monkeypatch):
    install(monkeypatch)
    vm, d, w, Z = _problem()
    kr = vm.lazy(d, w)
    assert kr.tables is None
    _gp((0.3, -0.5)).nll(Z.clone().requires_grad_(True), [kr]).sum().backward()
    assert vm.x0.grad is None and vm.v0.grad is None


def test_tables_only_mean_and_nonuniform(monkeypatch):
    install(monkeypatch)
    vm, d, w, Z = _problem(seed=1)
    lvs = (0.3, -0.5)
    _gp(lvs).nll(Z, [vm.lazy(d, w, requires_grad=True)]).sum().backward()   # Z and lvs need no gradient here
    gx, gv = vm.x0.grad.clone(), vm.v0.grad.clone()
    ox, ov = _oracle_table_grads(vm, d, w, Z, lvs)
    assert rel_err(gx, ox) < 1e-5 and rel_err(gv, ov) < 1e-5
    vm.zero_grad()
    _gp(lvs).nll(Z, [vm.lazy(d, w, requires_grad=True)]).mean().backward()
    assert rel_err(vm.x0.grad * Z.shape[0], gx) < 1e-6 and rel_err(vm.v0.grad * Z.shape[0], gv) < 1e-6
    nll = _gp(lvs).nll(Z, [vm.lazy(d, w, requires_grad=True)])
    with pytest.raises(NotImplementedError):
        (nll * torch.arange(Z.shape[0], dtype=torch.float32)[:, None]).sum().backward()


def _shard_worker(rank, world, port, out):
    from _pytest.monkeypatch import MonkeyPatch
    from gppvae_b200 import GP
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    mpch = MonkeyPatch()
    install(mpch)
    try:
        vm, d, w, Z = _problem()
        n = Z.shape[0]
        rows = slice(0, 31) if rank == 0 else slice(31, n)          # unequal shards
        gp = GP().shard_rows(n_total=n)
        with torch.no_grad():
            gp.lvs.copy_(torch.tensor((0.3, -0.5)))
        Zl = Z[rows].clone().requires_grad_(True)
        gp.nll(Zl, [vm.lazy(d[rows].contiguous(), w[rows].contiguous(), requires_grad=True)]).sum().backward()
        torch.save(dict(gx=vm.x0.grad, gv=vm.v0.grad, gZ=Zl.grad), os.path.join(out, f"r{rank}.pt"))
    finally:
        mpch.undo()
        dist.destroy_process_group()


def test_row_sharding_world2_gloo(tmp_path, monkeypatch):
    port = 29500 + (os.getpid() % 2000) + 23
    mp.spawn(_shard_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    install(monkeypatch)
    vm, d, w, Z = _problem()
    lvs = (0.3, -0.5)
    Zl = Z.clone().requires_grad_(True)
    _gp(lvs).nll(Zl, [vm.lazy(d, w, requires_grad=True)]).sum().backward()
    r0, r1 = (torch.load(os.path.join(tmp_path, f"r{r}.pt")) for r in (0, 1))
    # each rank returns its rows' part; their sum (what epoch._all_reduce_grads forms) is the single-process gradient
    assert rel_err(r0["gx"] + r1["gx"], vm.x0.grad) < 1e-5 and rel_err(r0["gv"] + r1["gv"], vm.v0.grad) < 1e-5
    assert rel_err(r0["gx"], vm.x0.grad) > 1e-2
    assert rel_err(torch.cat([r0["gZ"], r1["gZ"]]), Zl.grad) < 1e-5


# ---------------------------------------------------------------- C entries: validation before any device work
@pytest.fixture(scope="module")
def lib():
    from gppvae_b200 import _lib, build
    build.build()
    return _lib.load(build_if_missing=False)


def test_grad_entries_validate_without_a_device(lib):
    a = 1 << 12   # a non-null, 16-byte aligned fake device address: validation must fail before it is used
    p, q, nv, L = 8, 5, 7, 12     # Q = 40, ST ld >= nv (p + L) = 140
    assert lib.gpp_kr_grad_rhs(None, 40, a, 12, a, p, q, nv, L, 1.0, a, 8, None) == -1
    assert b"kr_grad_rhs: null pointer" in lib.gpp_last_error()
    assert lib.gpp_kr_grad_rhs(a, 40, a, 12, a, 6, q, nv, L, 1.0, a, 8, None) == -1            # p % 4
    assert lib.gpp_kr_grad_rhs(a, 40, a, 12, a, p, q, nv, 10, 1.0, a, 8, None) == -1           # L % 4
    assert lib.gpp_kr_grad_rhs(a, 36, a, 12, a, p, q, nv, L, 1.0, a, 8, None) == -1            # ldb < p q
    assert lib.gpp_kr_grad_rhs(a, 40, a, 8, a, p, q, nv, L, 1.0, a, 8, None) == -1             # ldw < L
    assert lib.gpp_kr_grad_rhs(a, 40, a, 12, a, p, q, nv, L, 1.0, a, 4, None) == -1            # ldr < p
    assert lib.gpp_kr_grad_rhs(a, 40, a, 12, a, p, q, 4096, L, 1.0, a, 8, None) == -1          # view table > 48 KB
    assert lib.gpp_kr_grad_rhs(a, 1200, a, 12, a, 4, 300, 1, L, 1.0, a, 8, None) == -1          # q (q + 1) > 160 KB
    assert b"q too large" in lib.gpp_last_error()
    assert b"kr_grad_rhs" in lib.gpp_last_error()
    ws = lib.gpp_kr_grad_views_workspace_bytes(p, q, nv)
    assert ws >= p * q * nv * 4 and lib.gpp_kr_grad_views_workspace_bytes(0, q, nv) == 0
    args = lambda **k: [k.get("ST", a), k.get("ldst", 140), a, k.get("ldb", 40), a, k.get("ldw", 12), k.get("wn", a),
                        k.get("p", p), q, nv, k.get("L", L), 1.0, k.get("gw", a), k.get("ldgw", 8), a, k.get("ws", ws),
                        None]
    assert lib.gpp_kr_grad_views(*args(ST=None)) == -1
    assert lib.gpp_kr_grad_views(*args(gw=None)) == -1
    assert lib.gpp_kr_grad_views(*args(wn=None)) == -1
    assert b"kr_grad_views: null pointer" in lib.gpp_last_error()
    assert lib.gpp_kr_grad_views(*args(p=6)) == -1
    assert lib.gpp_kr_grad_views(*args(ldst=136)) == -1                                          # ldst < nv (p + L)
    assert lib.gpp_kr_grad_views(*args(ldb=39)) == -1
    assert lib.gpp_kr_grad_views(*args(ldw=11)) == -1
    assert lib.gpp_kr_grad_views(*args(ldgw=4)) == -1                                            # ldgw < q
    assert b"kr_grad_views" in lib.gpp_last_error()
    assert lib.gpp_kr_grad_views(*args(ws=ws - 1)) == -3
    assert b"workspace too small" in lib.gpp_last_error()
