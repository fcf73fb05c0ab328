"""GP(n_rand_effs=3) at full size: N = 1M rows, L = 256, designs [Khatri-Rao 4096, xn[d] 256, wn[w] 16] (Q = 4368),
on the dense k-design route and on the structured one (the designs in factored form, Vmodel.lazy_effects), against the
single-design c3 step (Q = 4096) measured in the same process, the three alternated step by step.

    python experiments/bench/multi_effect.py [--steps K] [--warmup W] [--n N] [--structured-only]

`--structured-only` (e.g. with --n 4000000, where the dense designs and their planes do not fit one GPU) times the
structured k-design arm alone.

One step is "NLL + dNLL/dZ" (taylor_coeff with need_vb=False) on designs that are new to the GP: the factorisation cache
(and, for k designs, the stacked planes) is dropped before every step, as a new epoch's designs would; the Khatri-Rao
map itself is not in the step (its planes are written by Vmodel.forward before the GP sees V, for both arms); the
structured arm gets new factored designs before every step (the slot index, built once per (d, w), is reused).  Stage
times come from GP.stage_hook with CUDA events.  Prints one JSON line."""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", ".."))
from gppvae_b200 import GP, Vmodel, ops, synth  # noqa: E402

STAGES = [("stacked_planes", "stack:start", "stack:end"), ("pass1", "pass1:start", "pass1:end"),
          ("factor", "allreduce:end", "factor:end"), ("solve", "factor:end", "solve:end"),
          ("pass2", "solve:end", "pass2:end")]


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        power, clock = [s.strip() for s in out.split(",")]
    except Exception:   # no nvidia-smi: name only
        power = clock = None
    return dict(gpu=name, power_limit=power, max_sm_clock=clock)


class Timer:
    def __init__(self, gp):
        self.ev = {}
        gp.stage_hook = self.hook

    def hook(self, name):
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        self.ev[name] = e

    def stages(self):
        return {k: self.ev[a].elapsed_time(self.ev[b]) for k, a, b in STAGES if a in self.ev and b in self.ev}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--n", type=int, default=1_000_000)
    ap.add_argument("--structured-only", action="store_true")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("multi_effect.py measures the GPU: no CUDA device")
    dev = "cuda"
    N, p, q, L = a.n, 256, 16, 256
    pr = synth.make_problem(N, p, q, L, seed=0, device=dev)
    vm = Vmodel(pr.x0.shape[0], pr.v0.shape[0], p, q).to(dev)
    with torch.no_grad():
        vm.x0.copy_(pr.x0)
        vm.v0.copy_(pr.v0)
    Z = pr.Z
    if a.structured_only:
        V = Vs = None
    else:
        xn, wn = ops.normalize_rows(pr.x0), ops.normalize_rows(pr.v0)
        V = ops.khatri_rao_fwd(xn, wn, pr.d, pr.w)
        Vs = [V, xn[pr.d].contiguous(), wn[pr.w].contiguous()]
    gpk = GP(n_rand_effs=3).to(dev)
    gps = GP(n_rand_effs=3).to(dev)
    gp1 = GP().to(dev)
    with torch.no_grad():
        gpk.lvs.copy_(torch.tensor([0.0, -1.0, -2.0, -1.0]))
        gps.lvs.copy_(gpk.lvs)
    tk, ts, t1 = Timer(gpk), Timer(gps), Timer(gp1)
    vm.lazy_effects(pr.d, pr.w)      # the slot index, once per (d, w)

    def step(gp, tm, designs):
        gp._cache.clear()
        ops.STACKED.invalidate()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        gp.taylor_coeff(Z, designs, need_vb=False)
        e.record()
        torch.cuda.synchronize()
        return s.elapsed_time(e), tm.stages()

    arms = [("k_structured", gps, ts)] + ([] if a.structured_only else [("k", gpk, tk), ("single", gp1, t1)])
    res = {arm: [] for arm, _, _ in arms}
    check = None
    for i in range(a.warmup + a.steps):
        for arm, gp, tm in arms:
            designs = vm.lazy_effects(pr.d, pr.w) if arm == "k_structured" else Vs if arm == "k" else [V]
            r = step(gp, tm, designs)
            if i >= a.warmup:
                res[arm].append(r)
    if not a.structured_only:   # the two k-design routes on the same inputs
        Xs, _, vbs_s, nll_s = gps.taylor_coeff(Z, vm.lazy_effects(pr.d, pr.w), need_vb=False)
        Xd, _, vbs_d, nll_d = gpk.taylor_coeff(Z, Vs, need_vb=False)
        check = dict(Xb_max_rel=float(((Xs - Xd).abs().max() / Xd.abs().max())),
                     nll_sum_rel=abs(float(nll_s.double().sum() - nll_d.double().sum())) / abs(float(nll_d.double().sum())),
                     vbs_max_rel=float(((vbs_s - vbs_d).abs().max() / vbs_d.abs().max())))
        del Xs, Xd, nll_s, nll_d

    def summary(rows):
        ts = sorted(t for t, _ in rows)
        st = {k: sorted(s[k] for _, s in rows if k in s) for k, _, _ in STAGES}
        return dict(step_ms_median=ts[len(ts) // 2], step_ms_min=ts[0], step_ms_max=ts[-1],
                    stages_ms_median={k: v[len(v) // 2] for k, v in st.items() if v})

    # the full taylor_coeff (Vb of all three designs as well) of the k-design workload
    full = []
    for i in range(0 if a.structured_only else a.warmup + max(3, a.steps // 2)):
        gpk._cache.clear()
        ops.STACKED.invalidate()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        out = gpk.taylor_coeff(Z, Vs)
        e.record()
        torch.cuda.synchronize()
        del out
        if i >= a.warmup:
            full.append(s.elapsed_time(e))
    full.sort()
    out = dict(benchmark="multi_effect", **gpu_info(), N=N, L=L, designs=[p * q, p, q], Q_stacked=p * q + p + q,
               steps=a.steps, warmup=a.warmup, k_structured=summary(res["k_structured"]))
    if not a.structured_only:
        out.update(k_designs=summary(res["k"]), single_design_c3=summary(res["single"]),
                   k_taylor_coeff_full_ms_median=full[len(full) // 2], structured_vs_dense_k=check)
    out["note"] = ("CUDA events; need_vb=False step with the factorisation cache and the stacked planes dropped before "
                   "each step, new factored designs for the structured arm; arms alternated")
    print(json.dumps(out))


if __name__ == "__main__":
    main()
