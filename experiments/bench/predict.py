"""GP.predict at c3 (N = 1M training rows, L = 256, Q = 4096; synth.make_problem, trained tables), on a cache hit after
taylor_coeff, four arms alternated call by call in one process:

  structured_full   vm.lazy over every (object, view) slot: m = P nviews = 1M new rows (DESIGN 5.9)
  structured_4005   vm.lazy over 4 005 random slots
  dense_65536       dense new rows vm(dv, wv), m = 65 536 (the training design dense as well)
  eval_step         the expression of epoch.eval_step on the same 65 536 rows: vs[0] vm(dv, wv) (Vt^T K^-1 Z), Vt = vm.lazy

    python experiments/bench/predict.py [--steps K] [--warmup W] [--out PATH]

A call is timed with CUDA events followed by a synchronise; the median over the steps is reported.  The stages of the
structured full-grid arm (C and the solve, the views entry, the two P-long products, the rows kernel) are timed in a
separate loop that calls the pieces of GP._predict_factored one by one with events between them.  Prints one JSON
line and writes it to --out."""
import argparse
import json
import os
import statistics
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", ".."))
from gppvae_b200 import GP, Vmodel, ops, synth  # noqa: E402
from multi_effect import gpu_info  # noqa: E402


def models(pr, p, q, dev):
    vm = Vmodel(pr.x0.shape[0], pr.v0.shape[0], p, q).to(dev)
    gp = GP().to(dev)
    with torch.no_grad():
        vm.x0.copy_(pr.x0); vm.v0.copy_(pr.v0); gp.lvs.copy_(pr.lvs)
    return vm, gp


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b)


def eval_step_expr(gp, Vt, Vv, Z):
    with torch.no_grad():
        vs = gp.get_vs()
        U, UBi, _ = gp.U_UBi_Shb([Vt], vs)
        return vs[0] * Vv.mm(Vt.t().mm(gp.solve(Z, U, UBi, vs)))


def structured_stages(gp, kr, new, Z):
    """The pieces of GP._predict_factored (single Khatri-Rao design), with events between them."""
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(6)]
    with torch.no_grad():
        vs_a = gp.get_vs()
        Xm, ldx = ops.as_matrix(Z, "X")
        ev[0].record()
        fac, C = gp._kr_factorise(kr, vs_a.detach(), True, Xm, ldx, Xm.shape[1], vs_origin=vs_a)
        W, scal = ops.solve_w(fac, C, C.stride(0), Xm.shape[1], Z.shape[1], kr.n)
        M = ops.kr_assemble_m(W, kr.wn, kr.p, Xm.shape[1])
        ev[1].record()
        H, _, _ = ops.kr_predict_views(fac.Binv, kr.wn, kr.p, ["kr"])
        ev[2].record()
        Y = gp._kr_y(kr, M)
        ev[3].record()
        YH = gp._kr_y(kr, H)
        ev[4].record()
        ops.kr_predict_rows(Y, None, YH, kr.xn, None, None, new.d, new.w, kr.P, kr.nviews, Xm.shape[1], scal)
        ev[5].record()
    torch.cuda.synchronize()
    names = ["c_solve_m", "predict_views", "y_product", "yh_product", "predict_rows"]
    return {k: ev[i].elapsed_time(ev[i + 1]) for i, k in enumerate(names)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    N, p, q, L = 1_000_000, 256, 16, 256
    pr = synth.make_problem(N, p, q, L, kind="trained", lvs=(0.0, 0.0), seed=3, device=dev)
    P, nv = pr.x0.shape[0], q
    vm, gp_s = models(pr, p, q, dev)
    _, gp_d = models(pr, p, q, dev)
    kr = vm.lazy(pr.d, pr.w)
    Vt = vm(pr.d, pr.w).detach()
    gp_s.taylor_coeff(pr.Z, [kr])
    gp_d.taylor_coeff(pr.Z, [Vt])
    g = torch.arange(P * nv, device=dev)
    full = vm.lazy((g // nv).contiguous(), (g % nv).contiguous())
    sel = torch.randperm(P * nv, generator=torch.Generator(device=dev).manual_seed(0), device=dev)
    s4 = sel[:4005]
    small = vm.lazy((s4 // nv).contiguous(), (s4 % nv).contiguous())
    s64 = sel[:65536]
    Vv = vm(s64 // nv, s64 % nv).detach()
    kr.index()
    arms = {
        "structured_full": lambda: gp_s.predict(pr.Z, [kr], [full]),
        "structured_4005": lambda: gp_s.predict(pr.Z, [kr], [small]),
        "dense_65536": lambda: gp_d.predict(pr.Z, [Vt], [Vv]),
        "eval_step": lambda: eval_step_expr(gp_s, kr, Vv, pr.Z),
    }
    times = {a: [] for a in arms}
    hits0 = gp_s.cache_hits, gp_d.cache_hits
    for i in range(args.warmup + args.steps):
        for a, fn in arms.items():
            t = timed(fn)
            if i >= args.warmup:
                times[a].append(t)
    hits = (gp_s.cache_hits - hits0[0], gp_d.cache_hits - hits0[1])
    stages = [structured_stages(gp_s, kr, full, pr.Z) for _ in range(args.warmup + args.steps)][args.warmup:]
    out = dict(bench="predict", n=N, p=p, q=q, L=L, P=P, nviews=nv, m_full=P * nv, steps=args.steps,
               warmup=args.warmup, cache_hits_structured_dense=hits, **gpu_info(),
               median_ms={a: statistics.median(v) for a, v in times.items()},
               all_ms={a: [round(t, 3) for t in v] for a, v in times.items()},
               structured_full_stages_median_ms={k: statistics.median(s[k] for s in stages) for k in stages[0]})
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
