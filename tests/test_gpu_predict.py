"""GP.predict (posterior mean and variance at new rows, DESIGN 5.9) on the dense and structured routes against fp64.

Ground truth: tests/predict_oracle.py (the textbook n x n forms) where n allows it (c1), else the fp64 Woodbury form on
the device (tests/test_predict.py checks the two agree).  Errors are max-relative: max |mean - mean64| / max |mean64| and
max |var - var64| / max var64."""
import os
import subprocess
import sys

import pytest
import torch

from conftest import rel_err

pytestmark = pytest.mark.gpu

DEV = "cuda:0"


def _models(x0, v0, lvs, k=1):
    import gppvae_b200
    vm = gppvae_b200.Vmodel(x0.shape[0], v0.shape[0], x0.shape[1], v0.shape[1]).to(DEV)
    gp = gppvae_b200.GP(n_rand_effs=k).to(DEV)
    with torch.no_grad():
        vm.x0.copy_(x0); vm.v0.copy_(v0); gp.lvs.copy_(torch.as_tensor(lvs))
    return vm, gp


def _dense_designs(vm, d, w, kinds):
    with torch.no_grad():
        xn, wn = vm.x(), vm.v()
        return [vm(d, w) if k == "kr" else xn[d].contiguous() if k == "object" else wn[w].contiguous() for k in kinds]


def _fp64(Z, Vs, Vs_new, lvs):
    """fp64 prediction: the textbook forms on the CPU for small n, the Woodbury form on the device otherwise."""
    from predict_oracle import predict
    lv = torch.as_tensor(lvs, dtype=torch.float64)
    if Z.shape[0] <= 6000:
        return predict(Z.double().cpu(), [V.double().cpu() for V in Vs], [V.double().cpu() for V in Vs_new], lv)
    vs = torch.softmax(lv, 0).to(Z.device)
    Vt = torch.cat([vs[i].sqrt() * V.double() for i, V in enumerate(Vs)], 1)
    Binv = torch.linalg.inv(torch.eye(Vt.shape[1], dtype=torch.float64, device=Z.device) + Vt.t() @ Vt / vs[-1])
    W = Binv @ (Vt.t() @ Z.double()) / vs[-1]
    del Vt
    Vn = torch.cat([vs[i].sqrt() * V.double() for i, V in enumerate(Vs_new)], 1)
    return Vn @ W, ((Vn @ Binv) * Vn).sum(1, keepdim=True)


def _grid(P, nv, m=None, seed=0):
    """New rows over the (object, view) grid: all of it, or m slots of it at random."""
    g = torch.arange(P * nv, device=DEV)
    if m is not None:
        g = g[torch.randperm(P * nv, generator=torch.Generator(device=DEV).manual_seed(seed), device=DEV)[:m]]
    return (g // nv).contiguous(), (g % nv).contiguous()


def _errors(tag, pr, lvs, dn, wn_, kinds=("kr",)):
    k = len(kinds)
    vm, gp = _models(pr.x0, pr.v0, lvs, k)
    Z = pr.Z.to(DEV)
    d, w = pr.d.to(DEV), pr.w.to(DEV)
    Vd, Vnd = _dense_designs(vm, d, w, kinds), _dense_designs(vm, dn, wn_, kinds)
    rm, rv = _fp64(Z, Vd, Vnd, lvs)
    rm, rv = rm.to(DEV), rv.to(DEV)
    lazy = (lambda dd, ww: [vm.lazy(dd, ww)]) if k == 1 else (lambda dd, ww: vm.lazy_effects(dd, ww, kinds))
    sm, sv = gp.predict(Z, lazy(d, w), lazy(dn, wn_))
    dm, dv = _models(pr.x0, pr.v0, lvs, k)[1].predict(Z, Vd, Vnd)
    es = (rel_err(sm, rm), rel_err(sv, rv))
    ed = (rel_err(dm, rm), rel_err(dv, rv))
    print(f"[predict {tag}] vs fp64: mean structured {es[0]:.2e} dense {ed[0]:.2e}   "
          f"var structured {es[1]:.2e} dense {ed[1]:.2e}   structured vs dense: mean {rel_err(sm, dm):.2e} "
          f"var {rel_err(sv, dv):.2e}")
    return es, ed


@pytest.mark.parametrize("cfg", ["c1", "c2"])
def test_trained_tables_against_fp64(cfg):
    from gppvae_b200.synth import CONFIGS, make_problem
    c = CONFIGS[cfg]
    pr = make_problem(c["N"], c["p"], c["q"], c["L"], kind="trained", lvs=(0.0, 0.0), seed=11)
    P = pr.x0.shape[0]
    dn, wn_ = _grid(P, c["q"], None if cfg == "c1" else 20000, seed=1)
    es, ed = _errors(cfg, pr, (0.0, 0.0), dn, wn_)
    assert max(es + ed) <= 1e-4


@pytest.mark.parametrize("kind,zscale,lvs", [("init", 1.0, (0.0, 0.0)), ("trained", 1e-3, (0.0, 0.0)),
                                             ("trained", 1e3, (0.0, 0.0)), ("trained", 1.0, (2.0, -4.0))])
def test_init_tables_and_scaled_latents(kind, zscale, lvs):
    """The structured route within 3x of the dense CUDA route's error (no worse than it where the dense route misses
    1e-4)."""
    from gppvae_b200.synth import make_problem
    pr = make_problem(4005, 64, 9, 256, kind=kind, lvs=lvs, seed=3)
    pr.Z.mul_(zscale)
    dn, wn_ = _grid(pr.x0.shape[0], 9)
    es, ed = _errors(f"c1 {kind} Z x {zscale:g} lvs={lvs}", pr, lvs, dn, wn_)
    for s, dd in zip(es, ed):
        assert s <= max(3 * dd, 1e-6) if dd <= 1e-4 else s <= dd


@pytest.mark.parametrize("kinds", [("kr", "object", "view"), ("view", "kr"), ("object", "view")],
                         ids=["kr-object-view", "view-kr", "object-view"])
def test_k_designs_structured_against_dense(kinds):
    from gppvae_b200.synth import make_problem
    pr = make_problem(4005, 64, 9, 256, kind="trained", seed=5)
    lvs = (0.5, -2.0, -1.0) if len(kinds) == 2 else (2.0, -3.0, 0.0, -1.0)
    es, ed = _errors("-".join(kinds), pr, lvs, *_grid(pr.x0.shape[0], 9), kinds=kinds)
    assert max(es + ed) <= 1e-4


def test_mean_at_least_as_accurate_as_the_eval_step_expression():
    """eval_step's Zo = vs[0] vm(Dv, Wv) (Vt^T K^-1 Zm) against predict's mean, both against fp64."""
    from gppvae_b200.synth import make_problem
    out = []
    for kind in ("trained", "init"):
        pr = make_problem(4005, 64, 9, 256, kind=kind, seed=7)
        lvs = (0.0, 0.0)
        vm, gp = _models(pr.x0, pr.v0, lvs)
        Z, d, w = pr.Z.to(DEV), pr.d.to(DEV), pr.w.to(DEV)
        dn, wn_ = _grid(pr.x0.shape[0], 9)
        with torch.no_grad():
            vs = gp.get_vs()
            Vt, Vv = vm(d, w), vm(dn, wn_)
            U, UBi, _ = gp.U_UBi_Shb([Vt], vs)
            Zo = vs[0] * Vv.mm(Vt.t().mm(gp.solve(Z, U, UBi, vs)))
        mean, _ = gp.predict(Z, [vm.lazy(d, w)], [vm.lazy(dn, wn_)])
        rm, _ = _fp64(Z, [Vt], [Vv], lvs)
        ee, ep = rel_err(Zo, rm), rel_err(mean, rm)
        print(f"[predict vs eval-step expression, {kind}] vs fp64: predict {ep:.2e}  eval step {ee:.2e}")
        out.append((ep, ee))
    assert all(ep <= ee for ep, ee in out)


def test_out_of_table_rows_are_nan_and_the_rest_unaffected():
    from gppvae_b200.synth import make_problem
    pr = make_problem(4005, 64, 9, 256, seed=2)
    vm, gp = _models(pr.x0, pr.v0, (2.0, -3.0, 0.0, -1.0), 3)
    Z, d, w = pr.Z.to(DEV), pr.d.to(DEV), pr.w.to(DEV)
    dn, wn_ = _grid(pr.x0.shape[0], 9, 3000)
    kinds = ("kr", "object", "view")
    m0, v0 = gp.predict(Z, vm.lazy_effects(d, w, kinds), vm.lazy_effects(dn, wn_, kinds))
    dn2, wn2 = dn.clone(), wn_.clone()
    dn2[[4, 100]] = pr.x0.shape[0]
    wn2[[7, 2999]] = -1
    m1, v1 = gp.predict(Z, vm.lazy_effects(d, w, kinds), vm.lazy_effects(dn2, wn2, kinds))
    bad = torch.zeros(3000, dtype=torch.bool, device=DEV)
    bad[[4, 100, 7, 2999]] = True
    assert bool(torch.isnan(m1[bad]).all()) and bool(torch.isnan(v1[bad]).all())
    assert torch.equal(m1[~bad], m0[~bad]) and torch.equal(v1[~bad], v0[~bad])


@pytest.mark.parametrize("route", ["structured", "dense"])
def test_cache_hit_after_taylor_coeff_and_bit_identical_repeats(route, monkeypatch):
    from gppvae_b200 import _lib, ops
    from gppvae_b200.synth import make_problem
    pr = make_problem(4005, 64, 9, 256, seed=4)
    vm, gp = _models(pr.x0, pr.v0, (0.3, -0.5))
    Z, d, w = pr.Z.to(DEV), pr.d.to(DEV), pr.w.to(DEV)
    # fewer new rows than training rows: Vmodel.forward retires the planes of the previous V of the same shape, and with
    # them a factorisation cached on that V
    dn, wn_ = _grid(pr.x0.shape[0], 9, 3000)
    Vs = [vm.lazy(d, w)] if route == "structured" else [vm(d, w)]
    Vn = (lambda: [vm.lazy(dn, wn_)]) if route == "structured" else (lambda: [vm(dn, wn_)])
    gp.taylor_coeff(Z, Vs)
    factor_calls = []
    real_factor = ops.factor
    monkeypatch.setattr(ops, "factor", lambda *a, **k: factor_calls.append(1) or real_factor(*a, **k))
    hits, n0 = gp.cache_hits, _lib.launch_count()
    out1 = gp.predict(Z, Vs, Vn())
    torch.cuda.synchronize()
    n_hit = _lib.launch_count() - n0
    assert gp.cache_hits == hits + 1 and not factor_calls
    out2 = gp.predict(Z, Vs, Vn())
    assert torch.equal(out1[0], out2[0]) and torch.equal(out1[1], out2[1])
    gp.invalidate_cache()
    n0 = _lib.launch_count()
    gp.predict(Z, Vs, Vn())
    n_miss = _lib.launch_count() - n0
    assert len(factor_calls) == 1 and n_miss > n_hit
    print(f"[predict {route}] library launches: {n_hit} on a cache hit, {n_miss} on a miss")


def test_structured_against_dense_c3_and_full_grid_memory():
    from gppvae_b200.synth import CONFIGS, make_problem
    c = CONFIGS["c3"]
    pr = make_problem(c["N"], c["p"], c["q"], c["L"], kind="trained", lvs=(0.0, 0.0), seed=7, device=DEV)
    vm, gp = _models(pr.x0, pr.v0, (0.0, 0.0))
    P, nv = pr.x0.shape[0], c["q"]
    kr = vm.lazy(pr.d, pr.w)
    gp.taylor_coeff(pr.Z, [kr])
    dn, wn_ = _grid(P, nv)
    new = vm.lazy(dn, wn_)
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    mean, var = gp.predict(pr.Z, [kr], [new])
    torch.cuda.synchronize()
    growth = torch.cuda.max_memory_allocated() - base
    nq = P * nv * c["p"] * c["q"] * 4
    print(f"[predict c3 full grid] m = {P * nv}, peak allocation growth {growth / 1e9:.2f} GB "
          f"(one fp32 m x Q matrix: {nq / 1e9:.2f} GB)")
    assert growth < 4.5e9
    sel = torch.randperm(P * nv, generator=torch.Generator(device=DEV).manual_seed(0), device=DEV)[:65536]
    sel = sel.sort().values
    gpd = _models(pr.x0, pr.v0, (0.0, 0.0))[1]
    dm, dv = gpd.predict(pr.Z, [vm(pr.d, pr.w)], [vm(dn[sel], wn_[sel])])
    em, ev = rel_err(mean[sel], dm), rel_err(var[sel], dv)
    print(f"[predict c3] structured vs dense CUDA on 65536 rows: mean {em:.2e}  var {ev:.2e}")
    assert em < 2e-4 and ev < 2e-4


# ---- two ranks (NCCL): run as a torchrun worker by the test below
def _worker():
    import torch.distributed as dist
    from gppvae_b200.synth import make_problem
    dist.init_process_group("nccl")
    rank = dist.get_rank()
    torch.cuda.set_device(rank)
    dev = f"cuda:{rank}"
    N = 4005
    lvs = (0.3, -0.5)
    pr = make_problem(N, 64, 9, 256, seed=0, device=dev)
    import gppvae_b200

    def models():
        vm = gppvae_b200.Vmodel(pr.x0.shape[0], 9, 64, 9).to(dev)
        gp = gppvae_b200.GP().to(dev)
        with torch.no_grad():
            vm.x0.copy_(pr.x0); vm.v0.copy_(pr.v0); gp.lvs.copy_(torch.tensor(lvs))
        return vm, gp
    g = torch.arange(pr.x0.shape[0] * 9, device=dev)
    dn, wn_ = (g // 9).contiguous(), (g % 9).contiguous()
    vm, gp = models()
    ref = gp.predict(pr.Z, [vm.lazy(pr.d, pr.w)], [vm.lazy(dn, wn_)])
    cut = [0, 1700, N][rank:rank + 2]          # unequal shards
    vms, gps = models()
    gps.shard_rows(n_total=N)
    mean, var = gps.predict(pr.Z[cut[0]:cut[1]].contiguous(),
                            [vms.lazy(pr.d[cut[0]:cut[1]].contiguous(), pr.w[cut[0]:cut[1]].contiguous())],
                            [vms.lazy(dn, wn_)])
    other = [torch.empty_like(mean) for _ in range(2)], [torch.empty_like(var) for _ in range(2)]
    dist.all_gather(other[0], mean)
    dist.all_gather(other[1], var)
    ok = torch.equal(other[0][0], other[0][1]) and torch.equal(other[1][0], other[1][1]) and \
        rel_err(mean, ref[0]) <= 1e-4 and rel_err(var, ref[1]) <= 1e-4
    print("PREDICT_SHARDS_OK" if ok else "PREDICT_SHARDS_FAIL", flush=True)
    dist.destroy_process_group()


def test_two_rank_nccl_ranks_agree():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([root, os.path.join(root, "tests")]))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", "29553", os.path.abspath(__file__)]
    res = subprocess.run(cmd, cwd=root, env=env, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-2000:]
    assert res.stdout.count("PREDICT_SHARDS_OK") == 2, res.stdout[-2000:]


if __name__ == "__main__":
    _worker()
