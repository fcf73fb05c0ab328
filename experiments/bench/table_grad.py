"""The NLL with its gradient to the object and view tables at c3 (N = 1M, L = 256, Q = 4096; synth.make_problem, trained
tables): `gp.nll(Z, [V]).sum().backward()` on three arms, alternated step by step in one process:

  structured_tables  V = vm.lazy(d, w, requires_grad=True): gradients to Z, lvs, x0 and v0 through the slots (DESIGN 5.8)
  structured         V = vm.lazy(d, w): gradients to Z and lvs only (the path before table gradients existed)
  dense              V = vm(d, w): gradients to Z, lvs, x0 and v0 through Vb = dNLL/dV and khatri_rao_bwd

    python experiments/bench/table_grad.py [--steps K] [--warmup W] [--n N] [--structured-only] [--out PATH]

Every step builds V anew (a new epoch's V: the factorisation cache misses); the slot index, built once per (d, w), is
reused.  A step is timed with CUDA events from before V is built to after the backward, followed by a synchronise;
the median over the steps is reported.  The backward of the structured_tables arm is split into its stages in a
separate loop that calls the pieces of LazyVb.table_grads one by one with events between them.  `--structured-only`
(e.g. --n 4000000, where the dense route does not fit one GPU) times the structured_tables arm alone.  Prints one JSON
line and writes it to --out."""
import argparse
import json
import os
import statistics
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", ".."))
from gppvae_b200 import GP, Vmodel, ops, synth  # noqa: E402
from gppvae_b200._lib import S_V0, S_VN  # noqa: E402
from multi_effect import gpu_info  # noqa: E402


def models(pr, p, q, dev):
    vm = Vmodel(pr.x0.shape[0], pr.v0.shape[0], p, q).to(dev)
    gp = GP().to(dev)
    with torch.no_grad():
        vm.x0.copy_(pr.x0); vm.v0.copy_(pr.v0); gp.lvs.copy_(pr.lvs)
    return vm, gp


def step(arm, vm, gp, pr):
    vm.zero_grad(set_to_none=True)
    gp.zero_grad(set_to_none=True)
    Z = pr.Z.detach().requires_grad_(True)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    if arm == "dense":
        V = vm(pr.d, pr.w)
    else:
        V = vm.lazy(pr.d, pr.w, requires_grad=(arm == "structured_tables"))
    gp.nll(Z, [V]).sum().backward()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b)


def backward_stages(vm, gp, pr):
    """One structured_tables forward, then the pieces of LazyVb.table_grads timed one by one."""
    kr = vm.lazy(pr.d, pr.w, requires_grad=True)
    with torch.no_grad():
        _, Vbs, _, _ = gp.taylor_coeff(pr.Z, [kr], need_vb=True)
    lz = Vbs[0]
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
    ev[0].record()
    alpha = float(lz.scal[S_V0] / lz.scal[S_VN]) * lz.L
    ST, left = kr.st_operands(lz.Xb, lz.Xb.stride(0), lz.Lk, True)
    ev[1].record()
    R = ops.kr_grad_rhs(lz.fac.Binv, lz.W, kr.wn, kr.p, lz.Lk, alpha)
    ev[2].record()
    ncnt = kr.nviews * kr.p
    if isinstance(left, tuple):
        pS, pZ = left
        gx = ops.am_planes(pS, ops.split_planes(R[:ncnt], kr.p, ncnt, kr.p), kr.P, ncnt, kr.p)
        gx += ops.am_planes(pZ, ops.split_planes(R[ncnt:], kr.p, R.shape[0] - ncnt, kr.p), kr.P, pZ.cols, kr.p)
    else:
        gx = ops.am(left, left.stride(0), R, kr.p, kr.P, left.shape[1], kr.p)
    ev[3].record()
    ops.kr_grad_views(ST, lz.fac.Binv, lz.W, kr.wn, kr.p, lz.Lk, alpha)
    ev[4].record()
    torch.cuda.synchronize()
    names = ["slot_sums_and_st", "grad_rhs", "object_products", "grad_views"]
    return {k: ev[i].elapsed_time(ev[i + 1]) for i, k in enumerate(names)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--n", type=int, default=1_000_000)
    ap.add_argument("--structured-only", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    p, q, L = 256, 16, 256
    pr = synth.make_problem(args.n, p, q, L, kind="trained", lvs=(0.0, 0.0), seed=3, device=dev)
    arms = ["structured_tables"] if args.structured_only else ["structured_tables", "structured", "dense"]
    mods = {arm: models(pr, p, q, dev) for arm in arms}
    times = {arm: [] for arm in arms}
    for i in range(args.warmup + args.steps):
        for arm in arms:
            t = step(arm, *mods[arm], pr)
            if i >= args.warmup:
                times[arm].append(t)
    split = [backward_stages(*mods["structured_tables"], pr) for _ in range(args.steps)]
    out = dict(bench="table_grad", n=args.n, p=p, q=q, L=L, steps=args.steps, warmup=args.warmup, **gpu_info(),
               median_ms={arm: statistics.median(v) for arm, v in times.items()},
               all_ms={arm: [round(t, 3) for t in v] for arm, v in times.items()},
               structured_tables_backward_stages_median_ms={k: statistics.median(s[k] for s in split) for k in split[0]})
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
