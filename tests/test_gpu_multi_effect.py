"""GP(n_rand_effs=k): k random-effect designs K = sum_i v_i V_i V_i^T + vn I on the tensor-core path, against the fp64
oracle (oracle/gp_oracle.py restates gp.py:24-133 for any number of designs) and against the single-design path through
the identity  V' = [sqrt(v_i / s) V_i], s = 1 - vn,  lvs' = (log s, log vn)  (same covariance).

The designs are the additive models of the Face-Place data: the object x view Khatri-Rao product, an object-only
effect xn[d] and a view-only effect wn[w]."""
import math
import os
import subprocess
import sys

import pytest
import torch

from conftest import rel_err
from gppvae_b200 import GP, ops, synth
from oracle import gp_oracle as oracle

pytestmark = pytest.mark.gpu
DEV = "cuda"
LVS = (2.0, -3.0, 0.0, -1.0)     # vs ~ (0.84, 0.0057, 0.11, 0.042): widely unequal variances


def _designs(N, p, q, L, seed=0, kind="trained", lvs=LVS, scale=None):
    """Z and the designs [Khatri-Rao, xn[d], wn[w]] (fresh tensors) of a seeded synthetic problem."""
    pr = synth.make_problem(N, p, q, L, kind=kind, seed=seed, device=DEV)
    xn = ops.normalize_rows(pr.x0)
    wn = ops.normalize_rows(pr.v0)
    Vs = [ops.khatri_rao_fwd(xn, wn, pr.d, pr.w), xn[pr.d].contiguous(), wn[pr.w].contiguous()]
    if scale is not None:
        Vs[scale[0]] = Vs[scale[0]] * scale[1]
    gp = GP(n_rand_effs=len(Vs)).to(DEV)
    with torch.no_grad():
        gp.lvs.copy_(torch.tensor(lvs))
    return gp, pr.Z, Vs


def _oracle(Z, Vs, lvs, dtype):
    return oracle.taylor_coeff(Z.cpu().to(dtype), [V.cpu().to(dtype) for V in Vs], torch.tensor(lvs, dtype=dtype))


SHAPES = {
    "planes_q152": (1536, 16, 8, 64),      # stacked Q = 128 + 16 + 8 = 152: tensor-core planes, not a multiple of 64
    "simt_q80": (1024, 8, 8, 32),          # stacked Q = 80: below the tensor-core tile
    "c1": (4005, 64, 9, 256),              # stacked Q = 576 + 64 + 12 (9 views padded to 12)
}


@pytest.mark.parametrize("shape", sorted(SHAPES))
def test_parity_against_fp64_oracle(shape):
    gp, Z, Vs = _designs(*SHAPES[shape])
    Xb, Vbs, vbs, nll = gp.taylor_coeff(Z, Vs)
    o64 = _oracle(Z, Vs, LVS, torch.float64)
    o32 = _oracle(Z, Vs, LVS, torch.float32)
    assert vbs.shape == (4,) and [Vb.shape for Vb in Vbs] == [V.shape for V in Vs]
    assert abs(float(nll.double().sum()) - float(o64[3].sum())) <= 1e-5 * abs(float(o64[3].sum()))
    assert rel_err(Xb, o64[0]) <= 1e-4
    for i in range(3):
        assert rel_err(Vbs[i], o64[1][i]) < max(5 * rel_err(o32[1][i], o64[1][i]), 2e-3), i
    assert rel_err(vbs, o64[2]) < max(5 * rel_err(o32[2], o64[2]), 1e-4)
    # need_vb=False: the same Xb, nll and vbs, no Vb
    Xb2, Vbs2, vbs2, nll2 = gp.taylor_coeff(Z, Vs, need_vb=False)
    assert Vbs2 == [None] * 3 and torch.equal(Xb2, Xb) and torch.equal(vbs2, vbs) and torch.equal(nll2, nll)


def test_one_design_scaled_by_1e3():
    """One common power-of-two scale for the stacked planes: a design 1e-3 below the others costs 2^-32 of the largest
    magnitude in absolute terms, which stays inside the bounds."""
    gp, Z, Vs = _designs(*SHAPES["planes_q152"], scale=(1, 1e-3))
    Xb, Vbs, vbs, nll = gp.taylor_coeff(Z, Vs)
    o64 = _oracle(Z, Vs, LVS, torch.float64)
    o32 = _oracle(Z, Vs, LVS, torch.float32)
    assert abs(float(nll.double().sum()) - float(o64[3].sum())) <= 1e-5 * abs(float(o64[3].sum()))
    assert rel_err(Xb, o64[0]) <= 1e-4
    for i in range(3):
        assert rel_err(Vbs[i], o64[1][i]) < max(5 * rel_err(o32[1][i], o64[1][i]), 2e-3), i
    assert rel_err(vbs, o64[2]) < max(5 * rel_err(o32[2], o64[2]), 1e-4)


def test_nll_gradients_against_fp64_autograd():
    gp, Z, Vs = _designs(*SHAPES["planes_q152"])
    Vl = [V.clone().requires_grad_(True) for V in Vs]
    Zl = Z.clone().requires_grad_(True)
    gp.nll(Zl, Vl).sum().backward()
    Vd = [V.detach().cpu().double().requires_grad_(True) for V in Vs]
    Zd = Z.cpu().double().requires_grad_(True)
    lvs = torch.tensor(LVS, dtype=torch.float64, requires_grad=True)
    oracle.nll(Zd, Vd, lvs).sum().backward()
    assert rel_err(Zl.grad, Zd.grad) <= 1e-4
    for i in range(3):
        assert rel_err(Vl[i].grad, Vd[i].grad) < 2e-3, i
    assert rel_err(gp.lvs.grad, lvs.grad) < 1e-4


def test_taylor_expansion_minibatch_against_oracle():
    gp, Z, Vs = _designs(*SHAPES["planes_q152"])
    Xb, Vbs, vbs, _ = gp.taylor_coeff(Z, Vs)
    idx = torch.randperm(Z.shape[0], generator=torch.Generator().manual_seed(3))[:64].to(DEV)
    xm = Z[idx].clone().requires_grad_(True)
    vm = [V[idx].clone().requires_grad_(True) for V in Vs]
    te = gp.taylor_expansion(xm, vm, Xb[idx], [Vb[idx] for Vb in Vbs], vbs)
    te.sum().backward()
    xd = xm.detach().cpu().double().requires_grad_(True)
    vd = [v.detach().cpu().double().requires_grad_(True) for v in vm]
    lvs = torch.tensor(LVS, dtype=torch.float64, requires_grad=True)
    ted = oracle.taylor_expansion(xd, vd, Xb[idx].cpu().double(), [Vb[idx].cpu().double() for Vb in Vbs],
                                  vbs.cpu().double(), lvs)
    ted.sum().backward()
    assert rel_err(te, ted) < 1e-5
    assert rel_err(xm.grad, xd.grad) < 1e-6
    for i in range(3):
        assert rel_err(vm[i].grad, vd[i].grad) < 1e-6, i
    assert rel_err(gp.lvs.grad, lvs.grad) < 1e-5


def test_taylor_coeff_nll_and_nll_ineff_agree():
    gp, Z, Vs = _designs(*SHAPES["planes_q152"])
    Xb, Vbs, vbs, nll = gp.taylor_coeff(Z, Vs)
    Vl = [V.clone().requires_grad_(True) for V in Vs]
    Zl = Z.clone().requires_grad_(True)
    out = gp.nll(Zl, Vl)
    out.sum().backward()
    assert torch.equal(out.detach(), nll)
    assert torch.equal(Zl.grad, Xb)
    for i in range(3):
        assert torch.equal(Vl[i].grad, Vbs[i])
    vs = gp.get_vs().detach()
    assert torch.allclose(gp.lvs.grad, vs * (vbs - (vbs * vs).sum()), rtol=1e-6, atol=1e-6)
    ineff = gp.nll_ineff(Z, Vs)
    assert abs(float(ineff.detach().sum()) - float(nll.sum())) <= 1e-3 * abs(float(nll.sum()))


def test_u_ubi_shb_dense_and_solve_match_the_reference_form():
    gp, Z, Vs = _designs(*SHAPES["planes_q152"])
    vs = gp.get_vs()
    U, UBi, Shb = gp.U_UBi_Shb(Vs, vs, want_binv=True)
    hits = gp.cache_hits
    Xb, _, _, _ = gp.taylor_coeff(Z, Vs)
    assert gp.cache_hits == hits + 1
    Ur, UBir, Shbr = oracle.woodbury_factor([V.cpu().double() for V in Vs], vs.detach().cpu().double())
    assert rel_err(U.dense(), Ur) < 1e-6
    assert rel_err(UBi.dense(), UBir) < 1e-4
    assert rel_err(torch.sort(Shb.value(), descending=True).values, Shbr) < 1e-4
    assert rel_err(gp.solve(Z, U, UBi, vs), Xb) < 1e-5


def test_determinism_bit_identical():
    gp, Z, Vs = _designs(*SHAPES["c1"])
    a = gp.taylor_coeff(Z, Vs)
    gp.invalidate_cache()
    b = gp.taylor_coeff(Z, Vs)
    assert torch.equal(a[0], b[0]) and torch.equal(a[2], b[2]) and torch.equal(a[3], b[3])
    assert all(torch.equal(x, y) for x, y in zip(a[1], b[1]))


def _identity_check(N, p, q, L, lvs):
    """k-design evaluation == single-design evaluation on V' == fp64 oracle on V'."""
    gp, Z, Vs = _designs(N, p, q, L, lvs=lvs)
    Xb, _, _, nll = gp.taylor_coeff(Z, Vs, need_vb=False)
    vs = torch.softmax(torch.tensor(lvs, dtype=torch.float64), 0)
    s = 1.0 - float(vs[-1])
    Vp = torch.cat([math.sqrt(float(vs[i]) / s) * V for i, V in enumerate(Vs)], 1)
    del Vs
    lvs1 = (math.log(s), math.log(float(vs[-1])))
    gp1 = GP().to(DEV)
    with torch.no_grad():
        gp1.lvs.copy_(torch.tensor(lvs1))
    Xb1, _, _, nll1 = gp1.taylor_coeff(Z, [Vp], need_vb=False)
    m = oracle.qspace_model_streamed(Z, Vp, torch.tensor(lvs1, dtype=torch.float64))
    ref = float(m["nll"].sum())
    for x, n_ in ((Xb, nll), (Xb1, nll1)):
        assert abs(float(n_.double().sum()) - ref) <= 1e-5 * abs(ref)
        assert rel_err(x, m["Xb"]) <= 1e-4
    assert abs(float(nll.double().sum()) - float(nll1.double().sum())) <= 1e-5 * abs(ref)
    assert rel_err(Xb, Xb1) <= 1e-4


def test_full_size_identity_c2():
    _identity_check(100_000, 64, 16, 256, LVS)      # designs [1024, 64, 16]


def test_full_size_identity_250k():
    _identity_check(250_000, 256, 16, 256, LVS)     # designs [4096, 256, 16]


def test_fresh_designs_every_epoch_do_not_accumulate():
    """Each "epoch" builds new designs: the stacked planes and the cached factorisation of the previous epoch go with
    them, so memory_allocated() returns to one epoch's set."""
    N, p, q, L = 100_000, 64, 16, 256
    pr = synth.make_problem(N, p, q, L, seed=1, device=DEV)
    gp = GP(n_rand_effs=3).to(DEV)
    mem = []
    for epoch in range(4):
        xn = ops.normalize_rows(pr.x0 * (1 + 0.01 * epoch))
        wn = ops.normalize_rows(pr.v0)
        Vs = [ops.khatri_rao_fwd(xn, wn, pr.d, pr.w), xn[pr.d].contiguous(), wn[pr.w].contiguous()]
        out = gp.taylor_coeff(pr.Z, Vs, need_vb=False)
        del out, Vs, xn, wn
        torch.cuda.synchronize()
        mem.append(torch.cuda.memory_allocated())
    assert max(mem[1:]) <= mem[1] + (1 << 20), mem


def test_argument_errors():
    gp, Z, Vs = _designs(*SHAPES["simt_q80"])
    with pytest.raises(ValueError):
        gp.taylor_coeff(Z, Vs[:2])
    with pytest.raises(ValueError):
        gp.taylor_coeff(Z, Vs + [Vs[0]])
    with pytest.raises(NotImplementedError):
        GP(vsum2one=False)


# ---- two ranks (NCCL): run as a torchrun worker by the test below
def _worker():
    import torch.distributed as dist
    dist.init_process_group("nccl")
    rank, world = dist.get_rank(), dist.get_world_size()
    torch.cuda.set_device(rank)
    global DEV
    DEV = f"cuda:{rank}"
    N, p, q, L = 4005, 64, 9, 256
    gp, Z, Vs = _designs(N, p, q, L)
    Xb_full, _, vbs_full, nll_full = gp.taylor_coeff(Z, Vs)
    cut = [0, 1700, N][rank:rank + 2]          # unequal shards
    gps = GP(n_rand_effs=3).to(DEV).shard_rows(n_total=N)
    with torch.no_grad():
        gps.lvs.copy_(gp.lvs)
    Xb, _, vbs, nll = gps.taylor_coeff(Z[cut[0]:cut[1]].contiguous(), [V[cut[0]:cut[1]].contiguous() for V in Vs])
    G, C = gps._cache.G, gps._cache.C
    W = ops.solve_w_blocks(gps._cache.fac, C, C.stride(0), L, L, N)[0]
    ok = True
    for t in (G, C, W):
        ts = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(ts, t.contiguous())
        ok &= all(torch.equal(ts[0], x) for x in ts)
    s = nll.double().sum().reshape(1)
    dist.all_reduce(s)
    ok &= abs(float(s) - float(nll_full.double().sum())) <= 1e-6 * abs(float(nll_full.double().sum()))
    ok &= rel_err(Xb, Xb_full[cut[0]:cut[1]]) <= 1e-5 and rel_err(vbs, vbs_full) <= 1e-5
    print("MULTI_EFFECT_OK" if ok else "MULTI_EFFECT_FAIL", flush=True)
    dist.destroy_process_group()


def test_two_rank_nccl_parity():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([root, os.path.join(root, "tests")]))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", "29547", os.path.abspath(__file__)]
    res = subprocess.run(cmd, cwd=root, env=env, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-2000:]
    assert res.stdout.count("MULTI_EFFECT_OK") == 2, res.stdout[-2000:]


if __name__ == "__main__":
    _worker()
