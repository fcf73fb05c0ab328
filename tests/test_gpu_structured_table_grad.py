"""The exact NLL gradient to the object and view tables on the structured route (Vmodel.lazy(d, w, requires_grad=True),
DESIGN 5.8) against fp64 ground truth and the dense CUDA route.

Ground truth: V64 = oracle.feature_map(x0, v0, d, w) in fp64, Vb64 from oracle.taylor_coeff, then
torch.autograd.grad(V64, (x0, v0), Vb64) -- the Khatri-Rao backward of dNLL/dV chained through unit_rows.  (Not the
backward of oracle.nll: its svd backward is undefined at the repeated singular values of init-like tables.)  Each case
grades x0.grad and v0.grad with rel_err and requires the structured error to be at most max(2e-3, 2 x the dense CUDA
route's error against the same reference)."""
import os
import subprocess
import sys

import pytest
import torch

from conftest import rel_err

pytestmark = pytest.mark.gpu

DEV = "cuda:0"


def _fp64_table_grads(x0, v0, d, w, Z, lvs, keep=None):
    from oracle import gp_oracle as O
    x = x0.detach().double().cpu().requires_grad_(True)
    v = v0.detach().double().cpu().requires_grad_(True)
    d, w, Z = d.cpu(), w.cpu(), Z.detach().double().cpu()
    if keep is not None:
        d, w, Z = d[keep], w[keep], Z[keep]
    V64 = O.feature_map(x, v, d, w)
    _, Vbs, _, _ = O.taylor_coeff(Z, [V64.detach()], torch.as_tensor(lvs).double().cpu())
    return torch.autograd.grad(V64, (x, v), Vbs[0])


def _models(x0, v0, lvs):
    import gppvae_b200
    vm = gppvae_b200.Vmodel(x0.shape[0], v0.shape[0], x0.shape[1], v0.shape[1]).to(DEV)
    gp = gppvae_b200.GP().to(DEV)
    with torch.no_grad():
        vm.x0.copy_(x0); vm.v0.copy_(v0); gp.lvs.copy_(torch.as_tensor(lvs))
    return vm, gp


def _structured(x0, v0, d, w, Z, lvs, reduce="sum"):
    vm, gp = _models(x0, v0, lvs)
    out = gp.nll(Z.to(DEV), [vm.lazy(d.to(DEV), w.to(DEV), requires_grad=True)])
    getattr(out, reduce)().backward()
    return vm.x0.grad, vm.v0.grad


def _dense(x0, v0, d, w, Z, lvs):
    vm, gp = _models(x0, v0, lvs)
    gp.nll(Z.to(DEV), [vm(d.to(DEV), w.to(DEV))]).sum().backward()
    return vm.x0.grad, vm.v0.grad


def _grade(tag, x0, v0, d, w, Z, lvs):
    rx, rv = _fp64_table_grads(x0, v0, d, w, Z, lvs)
    sx, sv = _structured(x0, v0, d, w, Z, lvs)
    dx, dv = _dense(x0, v0, d, w, Z, lvs)
    es = (rel_err(sx, rx), rel_err(sv, rv))
    ed = (rel_err(dx, rx), rel_err(dv, rv))
    print(f"[table grad {tag}] vs fp64: x0 structured {es[0]:.2e} dense {ed[0]:.2e} (ratio {es[0] / ed[0]:.2f})  "
          f"v0 structured {es[1]:.2e} dense {ed[1]:.2e} (ratio {es[1] / ed[1]:.2f})")
    assert es[0] <= max(2e-3, 2 * ed[0]) and es[1] <= max(2e-3, 2 * ed[1])


@pytest.mark.parametrize("kind,lvs", [("trained", (0.0, 0.0)), ("init", (0.0, 0.0)), ("trained", (2.0, -4.0))])
def test_c1_against_fp64_and_dense(kind, lvs):
    from gppvae_b200.synth import make_problem
    pr = make_problem(4005, 64, 9, 256, kind=kind, lvs=lvs, seed=11)
    _grade(f"c1 {kind} lvs={lvs}", pr.x0, pr.v0, pr.d, pr.w, pr.Z, lvs)


def _random_problem(n, P, nv, p, q, L, zscale=1.0, bad=0):
    from oracle import gp_oracle as O
    g = torch.Generator().manual_seed(n)
    x0 = torch.randn(P, p, generator=g); v0 = torch.eye(nv, q) + 0.5 * torch.randn(nv, q, generator=g)
    d = torch.randint(0, P, (n,), generator=g); w = torch.randint(0, nv, (n,), generator=g)
    V64 = O.feature_map(x0.double(), v0.double(), d, w)
    Z = (0.5 * torch.randn(n, L, generator=g).double() + V64 @ torch.randn(p * q, L, generator=g).double()).float()
    d[:bad] = P + 5
    return x0, v0, d, w, zscale * Z


SHAPES = [(700, 37, 5, 8, 4, 12), (3000, 50, 7, 16, 7, 260), (513, 600, 3, 33, 4, 8), (6000, 640, 6, 128, 4, 72),
          (5000, 1500, 3, 130, 3, 64)]


@pytest.mark.parametrize("n,P,nv,p,q,L", SHAPES)
def test_repeated_and_empty_slots(n, P, nv, p, q, L):
    """p % 4 != 0, repeated and empty slots, more views than view features; the last two shapes take the planes form."""
    _grade(f"n={n} P={P} nv={nv} p={p} q={q} L={L}", *_random_problem(n, P, nv, p, q, L), (0.3, -0.5))


@pytest.mark.parametrize("zscale", [1e-3, 1e3])
def test_scaled_latents(zscale):
    _grade(f"Z x {zscale:g}", *_random_problem(6000, 640, 6, 128, 4, 72, zscale=zscale), (0.3, -0.5))


@pytest.mark.parametrize("shape", ["c1", "planes"])
def test_other_gradients_unchanged_and_default_has_none(shape):
    """requires_grad=True asks the factorisation for B^-1 as well: X and lvs still get bit-identical gradients, below the
    tensor-core tile (c1, P = 445) and on the operand-planes form (P = 640, p = 128)."""
    from gppvae_b200.synth import make_problem
    if shape == "c1":
        pr = make_problem(4005, 64, 9, 256, kind="trained", lvs=(0.5, -1.0), seed=3)
        x0, v0, d, w, Z0 = pr.x0, pr.v0, pr.d, pr.w, pr.Z
    else:
        x0, v0, d, w, Z0 = _random_problem(6000, 640, 6, 128, 4, 72)
    lvs = (0.5, -1.0)
    grads = []
    for rg in (True, False):
        vm, gp = _models(x0, v0, lvs)
        Z = Z0.to(DEV).requires_grad_(True)
        gp.nll(Z, [vm.lazy(d.to(DEV), w.to(DEV), requires_grad=rg)]).sum().backward()
        grads.append((Z.grad, gp.lvs.grad, vm.x0.grad, vm.v0.grad))
    assert torch.equal(grads[0][0], grads[1][0]) and torch.equal(grads[0][1], grads[1][1])
    assert grads[0][2] is not None and grads[0][3] is not None
    assert grads[1][2] is None and grads[1][3] is None


def test_tables_only_mean_and_nonuniform_upstream():
    x0, v0, d, w, Z = _random_problem(3000, 50, 7, 16, 7, 260)
    lvs = (0.3, -0.5)
    sx, sv = _structured(x0, v0, d, w, Z, lvs)               # Z does not require grad
    mx, mv = _structured(x0, v0, d, w, Z, lvs, reduce="mean")
    n = Z.shape[0]
    assert rel_err(mx * n, sx) < 1e-6 and rel_err(mv * n, sv) < 1e-6
    vm, gp = _models(x0, v0, lvs)
    out = gp.nll(Z.to(DEV), [vm.lazy(d.to(DEV), w.to(DEV), requires_grad=True)])
    with pytest.raises(NotImplementedError):
        (out * torch.arange(n, device=DEV, dtype=torch.float32)[:, None]).sum().backward()


@pytest.mark.parametrize("shape", [(700, 37, 5, 8, 4, 12), (6000, 640, 6, 128, 4, 72)], ids=["fp32", "planes"])
def test_out_of_table_rows_add_nothing(shape):
    """Out-of-table rows are NaN rows of Xb; on the planes form (second shape) they must not reach the scale of the
    slot-sum planes either."""
    x0, v0, d, w, Z = _random_problem(*shape, bad=40)
    lvs = (0.3, -0.5)
    sx, sv = _structured(x0, v0, d, w, Z, lvs)
    keep = torch.arange(40, d.shape[0])
    rx, rv = _fp64_table_grads(x0, v0, d, w, Z, lvs, keep=keep)
    ex, ev = rel_err(sx, rx), rel_err(sv, rv)
    print(f"[table grad out-of-table rows {shape}] vs fp64 over the in-table rows: x0 {ex:.2e}  v0 {ev:.2e}")
    assert ex < 2e-3 and ev < 2e-3


def test_repeats_are_bit_identical():
    x0, v0, d, w, Z = _random_problem(6000, 640, 6, 128, 4, 72)
    vm, gp = _models(x0, v0, (0.3, -0.5))
    out = []
    for _ in range(2):
        vm.zero_grad()
        gp.nll(Z.to(DEV), [vm.lazy(d.to(DEV), w.to(DEV), requires_grad=True)]).sum().backward()
        out.append((vm.x0.grad.clone(), vm.v0.grad.clone()))
    assert torch.equal(out[0][0], out[1][0]) and torch.equal(out[0][1], out[1][1])


def _full_size(cfg_name, seed):
    from gppvae_b200.synth import CONFIGS, make_problem
    cfg = CONFIGS[cfg_name]
    pr = make_problem(cfg["N"], cfg["p"], cfg["q"], cfg["L"], kind="trained", lvs=(0.0, 0.0), seed=seed, device=DEV)
    lvs = (0.0, 0.0)
    vm, gp = _models(pr.x0, pr.v0, lvs)
    out = gp.nll(pr.Z, [vm.lazy(pr.d, pr.w, requires_grad=True)])
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    out.sum().backward()
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated()
    sx, sv = vm.x0.grad.clone(), vm.v0.grad.clone()
    del vm, gp, out
    dx, dv = _dense(pr.x0, pr.v0, pr.d, pr.w, pr.Z, lvs)
    ex, ev = rel_err(sx, dx), rel_err(sv, dv)
    nq = cfg["N"] * cfg["p"] * cfg["q"] * 4
    print(f"[table grad {cfg_name}] structured vs dense CUDA: x0 {ex:.2e}  v0 {ev:.2e};  peak allocation over the "
          f"structured backward {peak / 1e9:.2f} GB (one fp32 N x Q matrix: {nq / 1e9:.2f} GB)")
    assert ex < 2e-3 and ev < 2e-3
    return peak, nq


def test_full_size_c2():
    _full_size("c2", seed=5)


def test_full_size_c3_memory():
    peak, nq = _full_size("c3", seed=7)
    assert peak < nq / 2


# ---- two ranks (NCCL): run as a torchrun worker by the test below
def _worker():
    import torch.distributed as dist
    from gppvae_b200.synth import make_problem
    dist.init_process_group("nccl")
    rank = dist.get_rank()
    torch.cuda.set_device(rank)
    dev = f"cuda:{rank}"
    N, p, q, L = 4005, 64, 9, 256
    lvs = (0.3, -0.5)
    pr = make_problem(N, p, q, L, seed=0, device=dev)
    import gppvae_b200

    def models():
        vm = gppvae_b200.Vmodel(pr.x0.shape[0], pr.v0.shape[0], p, q).to(dev)
        gp = gppvae_b200.GP().to(dev)
        with torch.no_grad():
            vm.x0.copy_(pr.x0); vm.v0.copy_(pr.v0); gp.lvs.copy_(torch.tensor(lvs))
        return vm, gp
    vm, gp = models()
    gp.nll(pr.Z, [vm.lazy(pr.d, pr.w, requires_grad=True)]).sum().backward()
    cut = [0, 1700, N][rank:rank + 2]          # unequal shards
    vms, gps = models()
    gps.shard_rows(n_total=N)
    gps.nll(pr.Z[cut[0]:cut[1]].contiguous(), [vms.lazy(pr.d[cut[0]:cut[1]].contiguous(), pr.w[cut[0]:cut[1]].contiguous(),
                                                         requires_grad=True)]).sum().backward()
    gx, gv = vms.x0.grad.clone(), vms.v0.grad.clone()
    dist.all_reduce(gx)
    dist.all_reduce(gv)
    ok = rel_err(gx, vm.x0.grad) <= 1e-4 and rel_err(gv, vm.v0.grad) <= 1e-4
    print("TABLE_GRAD_SHARDS_OK" if ok else "TABLE_GRAD_SHARDS_FAIL", flush=True)
    dist.destroy_process_group()


def test_two_rank_nccl_partial_gradients_sum():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([root, os.path.join(root, "tests")]))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", "29551", os.path.abspath(__file__)]
    res = subprocess.run(cmd, cwd=root, env=env, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-2000:]
    assert res.stdout.count("TABLE_GRAD_SHARDS_OK") == 2, res.stdout[-2000:]


if __name__ == "__main__":
    _worker()
