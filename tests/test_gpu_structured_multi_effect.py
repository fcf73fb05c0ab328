"""GP(n_rand_effs=k) on factored designs (Vmodel.lazy_effects: the object x view Khatri-Rao product, the object-only
design xn[d] and the view-only design wn[w], never materialised) against the fp64 oracle on their dense() forms and
against the dense k-design path on the same inputs."""
import math
import os
import subprocess
import sys

import pytest
import torch

from conftest import rel_err
from gppvae_b200 import GP, Vmodel, synth
from oracle import gp_oracle as oracle

pytestmark = pytest.mark.gpu
DEV = "cuda"
LVS = (2.0, -3.0, 0.0, -1.0)     # vs ~ (0.84, 0.0057, 0.11, 0.042): widely unequal variances
LVS2 = (2.0, -3.0, -1.0)
SHAPES = {
    "planes_q152": (1536, 16, 8, 64),      # stacked Q = 128 + 16 + 8; P = 192 objects: the P-long products in fp32 form
    "simt_q80": (1024, 8, 8, 32),          # stacked Q = 64 + 8 + 8
    "c1": (4005, 64, 9, 256),              # stacked Q = 576 + 64 + 12 (9 views padded to 12)
}


def _gp(k, lvs=None):
    gp = GP(n_rand_effs=k).to(DEV)
    with torch.no_grad():
        gp.lvs.copy_(torch.tensor(lvs if lvs is not None else (LVS if k == 3 else LVS2)))
    return gp


def _problem(N, p, q, L, kinds=("kr", "object", "view"), seed=0, lvs=None):
    """The GP, Z, the factored designs and their dense() forms of a seeded synthetic problem."""
    pr = synth.make_problem(N, p, q, L, seed=seed, device=DEV)
    vm = Vmodel(pr.x0.shape[0], pr.v0.shape[0], p, q).to(DEV)
    with torch.no_grad():
        vm.x0.copy_(pr.x0)
        vm.v0.copy_(pr.v0)
    Vs = vm.lazy_effects(pr.d, pr.w, kinds)
    return _gp(len(kinds), lvs), pr.Z, Vs, [V.dense() for V in Vs]


def _oracle(Z, Vd, lvs, dtype):
    return oracle.taylor_coeff(Z.cpu().to(dtype), [V.cpu().to(dtype) for V in Vd], torch.tensor(lvs, dtype=dtype))


def _check_against_oracle(gp, Z, Vs, Vd, lvs):
    Xb, Vbs, vbs, nll = gp.taylor_coeff(Z, Vs)
    o64 = _oracle(Z, Vd, lvs, torch.float64)
    o32 = _oracle(Z, Vd, lvs, torch.float32)
    assert vbs.shape == (len(Vs) + 1,) and [Vb.shape for Vb in Vbs] == [V.shape for V in Vd]
    ref = float(o64[3].sum())
    assert abs(float(nll.double().sum()) - ref) <= 1e-5 * abs(ref)
    assert rel_err(Xb, o64[0]) <= 1e-4
    idx = torch.randperm(Z.shape[0], generator=torch.Generator().manual_seed(1))[:257].to(DEV)
    for i in range(len(Vs)):
        assert rel_err(Vbs[i][idx], o64[1][i][idx.cpu()]) < max(5 * rel_err(o32[1][i], o64[1][i]), 2e-3), i
    assert rel_err(vbs, o64[2]) < max(5 * rel_err(o32[2], o64[2]), 1e-4)
    return Xb, Vbs, vbs, nll


@pytest.mark.parametrize("shape", sorted(SHAPES))
def test_parity_against_fp64_oracle_and_dense_path(shape):
    gp, Z, Vs, Vd = _problem(*SHAPES[shape])
    Xb, Vbs, vbs, nll = _check_against_oracle(gp, Z, Vs, Vd, LVS)
    Xb2, Vbs2, vbs2, nll2 = gp.taylor_coeff(Z, Vs, need_vb=False)
    assert Vbs2 == [None] * 3 and torch.equal(Xb2, Xb) and torch.equal(vbs2, vbs) and torch.equal(nll2, nll)
    Xbd, _, vbsd, nlld = _gp(3).taylor_coeff(Z, Vd, need_vb=False)
    assert rel_err(Xb, Xbd) <= 1e-4
    assert abs(float(nll.double().sum()) - float(nlld.double().sum())) <= 1e-5 * abs(float(nlld.double().sum()))
    assert rel_err(vbs, vbsd) <= 1e-4


@pytest.mark.parametrize("kinds", [("kr", "view"), ("object", "view"), ("view", "kr", "object"), ("object", "kr")])
def test_kind_orders_and_subsets(kinds):
    gp, Z, Vs, Vd = _problem(*SHAPES["c1"], kinds=kinds)
    _check_against_oracle(gp, Z, Vs, Vd, LVS if len(kinds) == 3 else LVS2)


@pytest.mark.parametrize("n,P,nv,p,q,L", [(700, 37, 5, 8, 4, 12), (3000, 50, 7, 16, 7, 260), (6000, 640, 6, 128, 4, 72),
                                          (5000, 1500, 3, 130, 3, 64)])
def test_repeated_and_empty_slots(n, P, nv, p, q, L):
    """Random (object, view) indices: slots with several rows and slots with none, widths that need padding, more views
    than view features; the last two shapes take the operand-planes form of the P-long products."""
    g = torch.Generator().manual_seed(n)
    x0 = torch.randn(P, p, generator=g)
    v0 = torch.eye(nv, q) + 0.5 * torch.randn(nv, q, generator=g)
    d, w = torch.randint(0, P, (n,), generator=g), torch.randint(0, nv, (n,), generator=g)
    vm = Vmodel(P, nv, p, q).to(DEV)
    with torch.no_grad():
        vm.x0.copy_(x0.to(DEV))
        vm.v0.copy_(v0.to(DEV))
    Vs = vm.lazy_effects(d.to(DEV), w.to(DEV))
    Vd = [V.dense() for V in Vs]
    Z = (0.5 * torch.randn(n, L, generator=g).to(DEV) + Vd[0] @ torch.randn(Vd[0].shape[1], L, generator=g).to(DEV))
    _check_against_oracle(_gp(3), Z, Vs, Vd, LVS)


def test_bad_index_gives_nan_row():
    vm = Vmodel(10, 4, 8, 4).to(DEV)
    d = torch.tensor([0, 3, 99, 5] * 8, device=DEV)
    w = torch.tensor([0, 1, 2, 3] * 8, device=DEV)
    Z = torch.randn(32, 8, device=DEV)
    Xb, _, _, _ = _gp(3).taylor_coeff(Z, vm.lazy_effects(d, w), need_vb=False)
    bad = torch.arange(2, 32, 4, device=DEV)
    good = torch.tensor([i for i in range(32) if i % 4 != 2], device=DEV)
    assert torch.isnan(Xb[bad]).all() and torch.isfinite(Xb[good]).all()


def test_eval_step_calls():
    """train_gppvae.py:235-237: U_UBi_Shb -> solve (the cached factorisation) and V.t().mm(Kiz) of every design."""
    gp, Z, Vs, Vd = _problem(*SHAPES["c1"])
    vs = gp.get_vs()
    U, UBi, Shb = gp.U_UBi_Shb(Vs, vs, want_binv=True)
    Kiz = gp.solve(Z, U, UBi, vs)
    hits = gp.cache_hits
    Xb, _, _, _ = gp.taylor_coeff(Z, Vs, need_vb=False)
    assert gp.cache_hits == hits + 1
    assert rel_err(Kiz, Xb) <= 1e-5
    gpd = _gp(3)
    Ud, UBid, Shbd = gpd.U_UBi_Shb(Vd, vs, want_binv=True)
    assert rel_err(Kiz, gpd.solve(Z, Ud, UBid, vs)) <= 1e-4
    assert rel_err(U.dense(), Ud.dense()) < 1e-6 and rel_err(UBi.dense(), UBid.dense()) < 1e-4
    assert rel_err(Shb.value(), Shbd.value()) < 1e-4
    # the view-only product adds ~N / nviews rows of Kiz per view in fp32, and they largely cancel
    for V, D, tol in zip(Vs, Vd, (1e-5, 1e-5, 1e-4)):
        assert rel_err(V.t().mm(Kiz), D.double().t() @ Kiz.double()) < tol


def test_nll_gradients_against_fp64_autograd():
    gp, Z, Vs, Vd = _problem(*SHAPES["c1"])
    Zl = Z.clone().requires_grad_(True)
    gp.nll(Zl, Vs).sum().backward()
    Zd = Z.cpu().double().requires_grad_(True)
    lvs = torch.tensor(LVS, dtype=torch.float64, requires_grad=True)
    oracle.nll(Zd, [V.cpu().double() for V in Vd], lvs).sum().backward()
    assert rel_err(Zl.grad, Zd.grad) <= 1e-4
    assert rel_err(gp.lvs.grad, lvs.grad) < 1e-4


def test_taylor_expansion_minibatch_from_lazy_vb():
    gp, Z, Vs, _ = _problem(*SHAPES["c1"])
    Xb, Vbs, vbs, _ = gp.taylor_coeff(Z, Vs)
    idx = torch.randperm(Z.shape[0], generator=torch.Generator().manual_seed(3))[:64].to(DEV)
    xm = Z[idx].clone().requires_grad_(True)
    vm = [V[idx].clone().requires_grad_(True) for V in Vs]
    Vbm = [Vb[idx] for Vb in Vbs]
    te = gp.taylor_expansion(xm, vm, Xb[idx], Vbm, vbs)
    te.sum().backward()
    xd = xm.detach().cpu().double().requires_grad_(True)
    vd = [v.detach().cpu().double().requires_grad_(True) for v in vm]
    lvs = torch.tensor(LVS, dtype=torch.float64, requires_grad=True)
    ted = oracle.taylor_expansion(xd, vd, Xb[idx].cpu().double(), [Vb.cpu().double() for Vb in Vbm],
                                  vbs.cpu().double(), lvs)
    ted.sum().backward()
    assert rel_err(te, ted) < 1e-5
    assert rel_err(xm.grad, xd.grad) < 1e-6
    for i in range(3):
        assert rel_err(vm[i].grad, vd[i].grad) < 1e-6, i
    assert rel_err(gp.lvs.grad, lvs.grad) < 1e-5


def test_determinism_bit_identical():
    gp, Z, Vs, _ = _problem(*SHAPES["c1"])
    idx = torch.arange(0, Z.shape[0], 13, device=DEV)
    a = gp.taylor_coeff(Z, Vs)
    ra = [Vb[idx] for Vb in a[1]]
    gp.invalidate_cache()
    b = gp.taylor_coeff(Z, Vs)
    assert torch.equal(a[0], b[0]) and torch.equal(a[2], b[2]) and torch.equal(a[3], b[3])
    assert all(torch.equal(x, Vb[idx]) for x, Vb in zip(ra, b[1]))


def test_full_size_250k_against_streamed_oracle():
    """N = 250k, designs [4096, 256, 16]: the structured k-design evaluation against the fp64 streamed Q-space model of
    the single design V' = [sqrt(v_i / s) V_i], s = 1 - vn, lvs' = (log s, log vn) (the same covariance)."""
    N, p, q, L = 250_000, 256, 16, 256
    gp, Z, Vs, _ = _problem(N, p, q, L)
    Xb, _, _, nll = gp.taylor_coeff(Z, Vs, need_vb=False)
    vs = torch.softmax(torch.tensor(LVS, dtype=torch.float64), 0)
    s = 1.0 - float(vs[-1])
    Vp = torch.cat([math.sqrt(float(vs[i]) / s) * V.dense() for i, V in enumerate(Vs)], 1)
    m = oracle.qspace_model_streamed(Z, Vp, torch.tensor((math.log(s), math.log(float(vs[-1]))), dtype=torch.float64))
    ref = float(m["nll"].sum())
    assert abs(float(nll.double().sum()) - ref) <= 1e-5 * abs(ref)
    assert rel_err(Xb, m["Xb"]) <= 1e-4


def test_full_size_1m_against_dense_path_without_n_by_q_buffers():
    """N = 1M, designs [4096, 256, 16] (Q = 4368): the structured step allocates less than half an N x Q fp32 matrix at
    its peak, and agrees with the dense k-design path."""
    N, p, q, L = 1_000_000, 256, 16, 256
    gp, Z, Vs, _ = _problem(N, p, q, L)
    Vs[0].index()
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    Xb, _, vbs, nll = gp.taylor_coeff(Z, Vs, need_vb=False)
    torch.cuda.synchronize()
    grown = torch.cuda.max_memory_allocated() - base
    Q = 4096 + 256 + 16
    assert grown < N * Q * 4 / 2, grown
    Vd = [V.dense() for V in Vs]
    Xbd, _, vbsd, nlld = _gp(3).taylor_coeff(Z, Vd, need_vb=False)
    assert rel_err(Xb, Xbd) <= 1e-4
    assert abs(float(nll.double().sum()) - float(nlld.double().sum())) <= 1e-5 * abs(float(nlld.double().sum()))
    assert rel_err(vbs, vbsd) <= 1e-4


# ---- two ranks (NCCL): run as a torchrun worker by the test below
def _worker():
    import torch.distributed as dist
    dist.init_process_group("nccl")
    rank, world = dist.get_rank(), dist.get_world_size()
    torch.cuda.set_device(rank)
    global DEV
    DEV = f"cuda:{rank}"
    N, p, q, L = 4005, 64, 9, 256
    pr = synth.make_problem(N, p, q, L, seed=0, device=DEV)
    vm = Vmodel(pr.x0.shape[0], pr.v0.shape[0], p, q).to(DEV)
    with torch.no_grad():
        vm.x0.copy_(pr.x0)
        vm.v0.copy_(pr.v0)
    Xb_full, _, vbs_full, nll_full = _gp(3).taylor_coeff(pr.Z, vm.lazy_effects(pr.d, pr.w))
    cut = [0, 1700, N][rank:rank + 2]          # unequal shards
    gps = _gp(3).shard_rows(n_total=N)
    Vs = vm.lazy_effects(pr.d[cut[0]:cut[1]].contiguous(), pr.w[cut[0]:cut[1]].contiguous())
    Xb, _, vbs, nll = gps.taylor_coeff(pr.Z[cut[0]:cut[1]].contiguous(), Vs)
    ok = True
    for t in (gps._cache.G, vbs):
        ts = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(ts, t.contiguous())
        ok &= all(torch.equal(ts[0], x) for x in ts)
    s = nll.double().sum().reshape(1)
    dist.all_reduce(s)
    ok &= abs(float(s) - float(nll_full.double().sum())) <= 1e-6 * abs(float(nll_full.double().sum()))
    ok &= rel_err(Xb, Xb_full[cut[0]:cut[1]]) <= 1e-5 and rel_err(vbs, vbs_full) <= 1e-5
    print("STRUCTURED_MULTI_EFFECT_OK" if ok else "STRUCTURED_MULTI_EFFECT_FAIL", flush=True)
    dist.destroy_process_group()


def test_two_rank_nccl_parity():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([root, os.path.join(root, "tests")]))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", "29549", os.path.abspath(__file__)]
    res = subprocess.run(cmd, cwd=root, env=env, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-2000:]
    assert res.stdout.count("STRUCTURED_MULTI_EFFECT_OK") == 2, res.stdout[-2000:]


if __name__ == "__main__":
    _worker()
