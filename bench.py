#!/usr/bin/env python
"""Benchmark of the GP prior term (Woodbury NLL + dNLL/dZ) -- BASELINE.json's metric.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c3|c2|c1] [--impl ours|reference]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

One "step" = one evaluation of the GP term over the whole latent matrix, as train_gppvae.py:161-167 does
once per epoch: normalise tables -> Khatri-Rao map V -> pass 1 (V^T[V|Z]) -> all-reduce (N>1) ->
Cholesky/solve -> pass 2 + epilogue, producing nll (N x 1), Xb = dNLL/dZ (N x L) and vbs.  The workload is
BASELINE.json configs[2] (N=1M, L=256, Q=4096: the configuration the north-star target is quoted on; it
fits one B200), row-sharded over the ranks (strong scaling).  Rank 0 prints ONE JSON line.

`--impl reference` times the reference's own CPU implementation of the path on the host cores: the UNMODIFIED
gp.py / vmod.py from the git-ignored copy under baseline/_ref/ (`__graft_entry__.build()` makes it where the reference
checkout named by BASELINE.json's reference_path exists), falling back to the op-for-op port in oracle/gp_oracle.py
(`kind: "port"`).  Each step evaluates a fixed 100k-row sample of the workload (BASELINE.md 3).

`--dump-outputs DIR` writes what the last timed step of the device-resident leg returned (see dump_outputs), so that
two builds can be compared output for output: the inputs are generated from fixed seeds.

`--check` (any --gpus): parity of the multi-GPU path on the real collective -- all ranks' all-reduced G, C and W
bit-identical, sum(nll) / Xb rows against the unsharded evaluation on rank 0; a failure fails the run.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from gppvae_b200.synth import CONFIGS, make_problem  # noqa: E402

# dram__bytes_read.sum + dram__bytes_write.sum of pl_pass1_kernel per launch, from profiles/ (ncu --set full, 1 GPU);
# filled in by profiles/summarize.py output of the round (None where no capture exists for the shape)
TRAFFIC = {}
TRAFFIC_SOURCE = None
_tr = os.path.join(ROOT, "profiles", "r02_pass1_traffic.json")
if os.path.exists(_tr):
    with open(_tr) as _f:
        _t = json.load(_f)
    TRAFFIC = {(k.split(":")[0], int(k.split(":")[1])): v for k, v in _t["bytes"].items()}
    TRAFFIC_SOURCE = _t.get("source")

METRIC = "gp_term_samples_per_s"
UNIT = "samples/s"


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        out = dict(hbm_gbs=p["hbm_gbs"], bf16_burst=p["bf16_tflops"],
                   bf16_sustained=p.get("bf16_tflops_sustained", p["bf16_tflops"]), source="measured")
    else:
        out = dict(hbm_gbs=6650.0, bf16_burst=1590.0, bf16_sustained=1400.0, source="fallback")
    # round-2 yard-sticks measured on this pool (experiments/bench/peaks.py, experiments/tc/exp3_f16_planes.cu)
    alt = os.path.join(ROOT, "profiles", "r02_peaks.json")
    if os.path.exists(alt):
        with open(alt) as f:
            a = json.load(f)
        out["alt"] = {"tf32_cublas_sustained": a["tf32"]["sustained_tflops"], "tf32_cublas_burst": a["tf32"]["burst_tflops"],
                      "fp16_cublas_sustained": a["fp16"]["sustained_tflops"], "fp16_cublas_burst": a["fp16"]["burst_tflops"],
                      "umma_ss_fp16_burst_own_kernel": 2201.3, "umma_ss_tf32_burst_own_kernel": 1037.1,
                      "source": "profiles/r02_peaks.json (torch.matmul 8192^3), profiles/r02_exp3_tma_box_rate.txt "
                                "(own SS-form MMA-only kernel)"}
    return out


# ------------------------------------------------------------------------------------------- CPU arm
REF_DIR = os.path.join(ROOT, "baseline", "_ref")
CPU_SAMPLE_ROWS = 100_000        # BASELINE.md section 3: N in {100k, 250k}; fixed, not sized by a time budget


class _CpuShim:
    """Import the UNMODIFIED reference modules for a CPU run: stub the unused `h5py` import (gp.py:5) and make the
    hard-coded `.cuda()` calls (gp.py:29,64,115) the identity while the reference runs.  Restored on exit."""

    def __enter__(self):
        import types
        self._saved = (torch.Tensor.cuda, torch.nn.Module.cuda, sys.modules.get("h5py"))
        torch.Tensor.cuda = lambda self_, *a, **k: self_
        torch.nn.Module.cuda = lambda self_, *a, **k: self_
        if "h5py" not in sys.modules:
            sys.modules["h5py"] = types.ModuleType("h5py")
        return self

    def __exit__(self, *exc):
        torch.Tensor.cuda, torch.nn.Module.cuda = self._saved[0], self._saved[1]
        if self._saved[2] is None:
            sys.modules.pop("h5py", None)
        return False


def _load_reference():
    """(gp module, vmod module) of the unmodified reference from baseline/_ref/, or None."""
    if not (os.path.exists(os.path.join(REF_DIR, "gp.py")) and os.path.exists(os.path.join(REF_DIR, "vmod.py"))):
        return None
    import importlib.util
    mods = []
    for name in ("gp", "vmod"):
        spec = importlib.util.spec_from_file_location(f"_gppvae_ref_{name}", os.path.join(REF_DIR, name + ".py"))
        m = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(m)
        mods.append(m)
    return tuple(mods)


def cpu_reference_timing(cfg, rows: int = CPU_SAMPLE_ROWS, fixed_cost: float | None = None):
    """Time ONE evaluation of the reference path (Vmodel.forward + GP.nll under no_grad: NLL + K^-1 Z, gp.py:97-110)
    on `rows` rows of the workload, on all host threads.

    The reference's cost is a*N + b with b the N-independent Q x Q work (svd + inverse, gp.py:33-35): b is measured at
    256 rows, a on the sample, and `value` is the throughput extrapolated to the full N of the workload, N / (a*N + b)
    -- what the sample measured directly is reported beside it."""
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    N, p, q, L = cfg["N"], cfg["p"], cfg["q"], cfg["L"]
    Q = p * q
    rows = min(rows, N)
    with _CpuShim():
        ref = _load_reference()
        if ref is not None:
            ref_gp, ref_vmod = ref
            kind = "reference"
        else:
            from oracle import gp_oracle as O
            kind = "port"

        def run(n):
            pr = make_problem(N, p, q, L, kind="trained", lvs=(0.0, 0.0), seed=0, n_rows=n)
            if kind == "reference":
                vm = ref_vmod.Vmodel(pr.x0.shape[0], q, p, q)
                gp = ref_gp.GP(n_rand_effs=1)
                with torch.no_grad():
                    vm.x0.copy_(pr.x0); vm.v0.copy_(pr.v0); gp.lvs.copy_(pr.lvs)
                t0 = time.perf_counter()
                with torch.no_grad():
                    V = vm(pr.d, pr.w)
                    nll = gp.nll(pr.Z, [V])
            else:
                t0 = time.perf_counter()
                with torch.no_grad():
                    V = O.feature_map(pr.x0, pr.v0, pr.d, pr.w)
                    nll, _ = O.nll_and_grad(pr.Z, [V], pr.lvs)
            return time.perf_counter() - t0, float(nll.sum())

        small = min(256, N)
        if fixed_cost is None:
            run(small)                       # thread-pool / MKL warm-up
            fixed_cost, _ = run(small)       # ~ the N-independent cost b
        ts, _ = run(rows)
    a = max(ts - fixed_cost, 1e-9) / max(rows - small, 1)
    full = a * N + fixed_cost if rows < N else ts
    return dict(value=N / full, unit=UNIT, cores=threads, kind=kind,
                sample=f"{rows} of {N} rows (Q={Q}, L={L}): Vmodel.forward + GP.nll under no_grad in {ts:.2f} s "
                       f"({rows / ts:.0f} samples/s on the sample itself); Q x Q cost b={fixed_cost:.2f} s measured at "
                       f"{small} rows; value = N/(a*N+b), linear in N" if rows < N else
                       f"all {N} rows (Q={Q}, L={L}): Vmodel.forward + GP.nll under no_grad in {ts:.2f} s",
                sample_rows=rows, sample_seconds=ts, sample_samples_per_s=rows / ts, fixed_cost_seconds=fixed_cost,
                seconds_full_extrapolated=full, extrapolated=rows < N, torch=torch.__version__)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = CONFIGS[args.workload]
    # every step evaluates the same fixed sample; the N-independent cost is measured once, before the warm-up
    first = cpu_reference_timing(cfg)
    b = first["fixed_cost_seconds"]
    vals, secs, last = [], [], first
    for i in range(args.warmup + args.steps):
        last = cpu_reference_timing(cfg, fixed_cost=b)
        if i >= args.warmup:
            vals.append(last["value"])
            secs.append(last["sample_seconds"])
    v = statistics.median(vals) if vals else last["value"]
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus,
            "steps": len(vals), "warmup": args.warmup,
            # wall time of what one step actually ran (the sample); the full-N time is in cpu_baseline
            "ms_per_step": 1e3 * (statistics.median(secs) if secs else last["sample_seconds"]),
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args.workload, args.gpus),
            "value_is": "throughput on the full workload extrapolated from the per-step sample (cpu_baseline.sample)",
            "cpu_baseline": dict(last, value=v),
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def workload_config(name, gpus):
    c = CONFIGS[name]
    return {"workload": f"{name}: GP term N={c['N']} L={c['L']} Q={c['p'] * c['q']} (p={c['p']}, q={c['q']}), "
                        f"NLL + dNLL/dZ incl. Khatri-Rao map, rows sharded over {gpus} GPU(s)",
            "N": c["N"], "L": c["L"], "Q": c["p"] * c["q"], "p": c["p"], "q": c["q"], "tables": "trained-like",
            "lvs": [0.0, 0.0], "seed": 0, "parallelism": f"rows/{gpus}",
            "l2_policy": "inputs larger than L2 (V alone is N*Q*4 bytes per rank; no explicit flush)"}


# ------------------------------------------------------------------------------------------- clocks
class ClockSampler(threading.Thread):
    def __init__(self, index: int, period: float = 0.05):
        super().__init__(daemon=True)
        self.index, self.period, self.samples, self.reasons = index, period, [], set()
        self._stop_evt = threading.Event()
        self.max_mhz = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        return {"sm_mhz": statistics.median(self.samples) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------- GPU arm
def _pin_to_local_numa(index: int) -> None:
    """Bind this process to the CPUs NVML reports as local to GPU `index` before the pinned host buffers of the
    end-to-end leg are allocated (first touch then places them on the GPU's own NUMA node: at 8 ranks the round-1 run
    moved 258 MB per rank at ~14 GB/s, far below a PCIe 5 x16 link)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = {64 * wi + b for wi, wv in enumerate(words) for b in range(64) if (wv >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
    except Exception:
        pass


def run_check(args, gp, vm, pr, cfg, world, rank, dev):
    """Real-collective parity of the row-sharded path (SURVEY section 4 item 5): after the all-reduce every rank must
    hold bit-identical GC and W; sum(nll) and this rank's rows of Xb must agree with the UNSHARDED evaluation of the
    whole problem (computed on every rank's own GPU from the same seeded generator) to 1e-6 / 1e-5."""
    import torch.distributed as dist
    from gppvae_b200 import ops
    N, p, q, L = cfg["N"], cfg["p"], cfg["q"], cfg["L"]
    with torch.no_grad():
        V = vm(pr.d, pr.w)
        Xb, _, vbs, nll = gp.taylor_coeff(pr.Z, [V], need_vb=False)
    G, C = gp._cache.G[:, : p * q], gp._cache.C
    W = ops.solve_w(gp._cache.fac, C, C.stride(0), L, L, N)[0]
    ok = True
    report = {}
    if world > 1:
        for name, t in (("G", G.contiguous()), ("C", C.contiguous()), ("W", W)):
            lo, hi = t.clone(), t.clone()
            dist.all_reduce(lo, op=dist.ReduceOp.MIN)
            dist.all_reduce(hi, op=dist.ReduceOp.MAX)
            same = bool(torch.equal(lo, hi))       # min over ranks == max over ranks, element by element
            report[name + "_bit_identical_across_ranks"] = same
            ok &= same
    # the unsharded evaluation (a plain 1-GPU GP on the full problem; needs the whole problem on this GPU)
    full = make_problem(N, p, q, L, kind="trained", lvs=(0.0, 0.0), seed=0, device=dev)
    import gppvae_b200
    gp1 = gppvae_b200.GP().to(dev)
    with torch.no_grad():
        gp1.lvs.copy_(full.lvs)
        V1 = vm(full.d, full.w)
        Xb1, _, vbs1, nll1 = gp1.taylor_coeff(full.Z, [V1], need_vb=False)
    off = pr.meta["row_offset"]
    n = pr.meta["n_rows"]
    tot = nll.double().sum().reshape(1)
    if world > 1:
        dist.all_reduce(tot)
    e_nll = abs(float(tot) - float(nll1.double().sum())) / abs(float(nll1.double().sum()))
    e_xb = float((Xb - Xb1[off:off + n]).abs().max() / Xb1.abs().max()) if n else 0.0
    e_vbs = float((vbs - vbs1).abs().max() / vbs1.abs().max())
    errs = torch.tensor([e_nll, e_xb, e_vbs], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(errs, op=dist.ReduceOp.MAX)
    report.update(nll_sum_rel_vs_1gpu=float(errs[0]), xb_max_rel_vs_1gpu=float(errs[1]), vbs_max_rel_vs_1gpu=float(errs[2]))
    ok &= float(errs[0]) <= 1e-6 and float(errs[1]) <= 1e-5 and float(errs[2]) <= 1e-5
    report["ok"] = bool(ok)
    del full, V1, Xb1, nll1, gp1
    gp.invalidate_cache()
    torch.cuda.empty_cache()
    return report


DUMP_XB_ROWS = 1 << 15       # 32 MB of Xb at L = 256; nll is written whole (4 MB at N = 1M)


def dump_outputs(out_dir, result, N, off, n, world, rank, dev):
    """Write what one step returned to its caller, as float32 .npy files in out_dir: nll (N x 1) and vbs whole, and Xb
    (N x L) on DUMP_XB_ROWS rows drawn with a fixed seed, in ascending row order (all of Xb where N is not larger).
    Ranks contribute their own rows to zero-filled buffers summed over the ranks, so the files do not depend on --gpus."""
    import numpy as np
    Xb, _, vbs, nll = result
    nll_all = torch.zeros(N, 1, device=dev, dtype=nll.dtype)
    nll_all[off:off + n] = nll
    rows = torch.arange(N) if N <= DUMP_XB_ROWS else \
        torch.randperm(N, generator=torch.Generator().manual_seed(0))[:DUMP_XB_ROWS].sort().values
    rows = rows.to(dev)
    mine = (rows >= off) & (rows < off + n)
    xb_rows = torch.zeros(rows.numel(), Xb.shape[1], device=dev, dtype=Xb.dtype)
    xb_rows[mine] = Xb[rows[mine] - off]
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(nll_all)
        dist.all_reduce(xb_rows)
    if rank == 0:
        os.makedirs(out_dir, exist_ok=True)
        for name, t in (("nll", nll_all), ("vbs", vbs), ("Xb", xb_rows)):
            np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())


def run_ours(args):
    import torch.distributed as dist
    import gppvae_b200
    from gppvae_b200 import _lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; gppvae_b200 has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    if args.gpus != world and rank == 0:
        print(f"bench.py: --gpus {args.gpus} but WORLD_SIZE={world}; using {world}", file=sys.stderr)

    cfg = CONFIGS[args.workload]
    N, p, q, L = cfg["N"], cfg["p"], cfg["q"], cfg["L"]
    Q = p * q
    per = -(-N // world)
    off = rank * per
    n = max(0, min(per, N - off))
    pr = make_problem(N, p, q, L, kind="trained", lvs=(0.0, 0.0), seed=0, device=dev, row_offset=off, n_rows=n)

    vm = gppvae_b200.Vmodel(pr.x0.shape[0], q, p, q).to(dev)
    gp = gppvae_b200.GP().to(dev)
    with torch.no_grad():
        vm.x0.copy_(pr.x0); vm.v0.copy_(pr.v0); gp.lvs.copy_(pr.lvs)
    if world > 1:
        gp.shard_rows(n_total=N)

    events = []

    def hook(name):
        ev = torch.cuda.Event(enable_timing=True)
        ev.record()
        events.append((name, ev))

    def step(d, w, Z):
        with torch.no_grad():
            if gp.stage_hook is not None:
                gp.stage_hook("kr:start")
            V = vm(d, w)
            return gp.taylor_coeff(Z, [V], need_vb=False)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = _lib.launch_count()
        e0.record()
        for _ in range(steps - 1):
            fn()
        out = fn()      # only the last step's results are held: earlier ones are freed as in an ordinary loop
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1) / steps], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), _lib.launch_count() - l0, out

    # ---- device-resident throughput (inputs already in HBM)
    sampler = ClockSampler(local)
    for _ in range(max(args.warmup, 3)):
        step(pr.d, pr.w, pr.Z)
    barrier()
    sampler.start()
    gp.stage_hook = hook
    ms, launches, last = timed(lambda: step(pr.d, pr.w, pr.Z), args.steps, 0)
    gp.stage_hook = None
    clocks = sampler.stop()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last, N, off, n, world, rank, dev)
    del last
    stages = {}
    for (na, ea), (nb, eb) in zip(events[:-1], events[1:]):
        if nb.endswith(":end"):
            stages.setdefault(nb[:-4], []).append(ea.elapsed_time(eb))
        elif na == "kr:start" and nb == "pass1:start":
            stages.setdefault("khatri_rao", []).append(ea.elapsed_time(eb))
    stage_ms = {k: sum(v) / len(v) for k, v in stages.items()}

    # ---- the same step replayed from a CUDA graph (launch-bound shapes; reported beside the eager number)
    ms_graph = None
    if world == 1 and args.workload != "c3":
        from gppvae_b200.graph import CapturedGPTerm
        cap = CapturedGPTerm(vm, gp, pr.d, pr.w, pr.Z)
        ms_graph, _ = timed(lambda: cap(), args.steps, 3)[:2]
        del cap
        gp.invalidate_cache()

    # ---- full taylor_coeff (adds B^-1, Vb): reported, not the headline
    def full_step():
        with torch.no_grad():
            V = vm(pr.d, pr.w)
            return gp.taylor_coeff(pr.Z, [V], need_vb=True)
    ms_full = None
    if not args.skip_full:
        ms_full, _ = timed(full_step, max(1, min(args.steps, 3)), 1)[:2]
        gp.invalidate_cache()      # drop the cached V / Binv / planes before the next leg
        torch.cuda.empty_cache()

    # ---- structured route (SURVEY 8(f) row 4): same inputs, same outputs, V never materialised.  Reported beside
    #      the dense path, which stays the headline (it is the path BASELINE.json's north_star names).
    structured = None
    if not args.skip_structured:
        def kr_step():
            with torch.no_grad():
                if gp.stage_hook is not None:
                    gp.stage_hook("kr:start")
                return gp.taylor_coeff(pr.Z, [vm.lazy(pr.d, pr.w)], need_vb=False)
        gp.invalidate_cache()
        torch.cuda.empty_cache()
        for _ in range(3):
            kr_step()
        events.clear()
        gp.stage_hook = hook
        ms_kr, launches_kr = timed(kr_step, args.steps, 0)[:2]
        gp.stage_hook = None
        st_kr = {}
        for (na, ea), (nb, eb) in zip(events[:-1], events[1:]):
            if nb.endswith(":end"):
                st_kr.setdefault(nb[:-4], []).append(ea.elapsed_time(eb))
            elif na == "kr:start" and nb == "pass1:start":
                st_kr.setdefault("index_and_tables", []).append(ea.elapsed_time(eb))
        Xb_s, _, vbs_s, nll_s = kr_step()
        Xb_d, _, vbs_d, nll_d = step(pr.d, pr.w, pr.Z)
        structured = {"ms_per_step": ms_kr, "value": N / (ms_kr * 1e-3), "gpu_launches": launches_kr,
                      "stage_ms": {k: sum(v) / len(v) for k, v in st_kr.items()},
                      "vs_dense_route": {"xb_max_rel": float((Xb_s - Xb_d).abs().max() / Xb_d.abs().max()),
                                         "nll_sum_rel": float(((nll_s.double().sum() - nll_d.double().sum()) /
                                                               nll_d.double().sum()).abs())},
                      "api": "GP.taylor_coeff(Z, [Vmodel.lazy(d, w)], need_vb=False)"}
        del Xb_s, Xb_d, nll_s, nll_d
        gp.invalidate_cache()
        torch.cuda.empty_cache()

    # ---- parity of the sharded path on the real collective (--check; always on when more than one rank runs)
    check = None
    if args.check or world > 1:
        check = run_check(args, gp, vm, pr, cfg, world, rank, dev)

    # ---- end to end: inputs start in pinned host memory, results end in pinned host memory, every step.
    # Pipelined leg: the inputs of step i+1 (d, w, Z) ride a copy stream beside the compute of step i (two sets of device
    # buffers), the results of step i leave on a third stream beside the compute of step i+1 (two sets of host buffers) --
    # every step still moves its own inputs and its own results inside the timed region (the last step's results are waited
    # for before the clock stops), and the evaluation is the plain `vm(d, w)` + `gp.taylor_coeff(Z, [V])` of the
    # device-resident leg.
    # `sync_ms_per_step` is the same work with nothing pipelined across steps (submit, wait for the results, submit):
    # there Z travels beside the work that does not need it (Khatri-Rao map, Gram tiles, Cholesky: GP.U_UBi_Shb, what
    # train_gppvae.py:235 calls first anyway) and V^T Z follows as a launch of its own.
    _pin_to_local_numa(local)
    hd, hw, hZ = (t.cpu().pin_memory() for t in (pr.d, pr.w, pr.Z))
    h_out = [(torch.empty(n, 1).pin_memory(), torch.empty(n, L).pin_memory(), torch.empty(2).pin_memory())
             for _ in range(2)]
    s_in, s_out = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    # device landing buffers of the inputs, double-buffered.  ALL of a step's inputs travel on the copy stream: the 16 MB
    # of d, w issued on the compute stream queued behind the 1 GB of Z on the one host -> device copy engine and held the
    # step's first kernel back by 8 ms (experiments/bench/e2e_trace.py).
    Zd = [torch.empty_like(pr.Z) for _ in range(2)]
    dd = [torch.empty_like(pr.d) for _ in range(2)]
    wd = [torch.empty_like(pr.w) for _ in range(2)]
    in_ready = [None, None]                                   # upload of buffer set k finished (recorded on s_in)
    in_free = [None, None]                                    # last compute that read buffer set k finished (on main)
    out_done = [None, None]
    step_no = [0]

    def upload(k):
        with torch.cuda.stream(s_in):
            if in_free[k] is not None:
                s_in.wait_event(in_free[k])
            dd[k].copy_(hd, non_blocking=True); wd[k].copy_(hw, non_blocking=True)
            ev_dw = torch.cuda.Event(); ev_dw.record(s_in)
            Zd[k].copy_(hZ, non_blocking=True)
            ev = torch.cuda.Event(); ev.record(s_in)
        in_ready[k] = (ev_dw, ev)

    def finish(i, main, Xb, vbs, nll):
        if out_done[i] is not None:
            out_done[i].synchronize()               # host buffers of slot i are ours again
        ev_c = torch.cuda.Event(); ev_c.record(main)
        with torch.cuda.stream(s_out):
            s_out.wait_event(ev_c)
            for t in (Xb, vbs, nll):
                t.record_stream(s_out)
            h_out[i][0].copy_(nll, non_blocking=True); h_out[i][1].copy_(Xb, non_blocking=True)
            h_out[i][2].copy_(vbs, non_blocking=True)
            ev = torch.cuda.Event(); ev.record(s_out)
        out_done[i] = ev
        return ev_c

    def e2e_submit(prefetch_next=True):
        i = step_no[0] & 1
        step_no[0] += 1
        main = torch.cuda.current_stream()
        if in_ready[i] is None:                     # first step of a run: nothing was prefetched
            upload(i)
        ev_dw, ev_z = in_ready[i]
        with torch.no_grad():
            main.wait_event(ev_dw)
            V = vm(dd[i], wd[i])
            main.wait_event(ev_z)
            Xb, _, vbs, nll = gp.taylor_coeff(Zd[i], [V], need_vb=False)
        in_ready[i] = None
        in_free[i] = finish(i, main, Xb, vbs, nll)
        if prefetch_next:                           # step i+1's inputs start their way now, beside this step's compute
            upload(i ^ 1)
        return i

    def e2e_sync_step():
        i = step_no[0] & 1
        step_no[0] += 1
        main = torch.cuda.current_stream()
        upload(i)
        ev_dw, ev_z = in_ready[i]
        with torch.no_grad():
            main.wait_event(ev_dw)
            V = vm(dd[i], wd[i])
            gp.U_UBi_Shb([V], gp.get_vs())          # pass 1 (Gram) + Cholesky while Z is still on the wire
            main.wait_event(ev_z)
            Xb, _, vbs, nll = gp.taylor_coeff(Zd[i], [V], need_vb=False)   # factorisation reused: V^T Z, W, pass 2
        in_ready[i] = None
        in_free[i] = finish(i, main, Xb, vbs, nll)
        out_done[i].synchronize()

    def e2e_drain():
        for ev in out_done:
            if ev is not None:
                ev.synchronize()

    def timed_wall(fn, steps, warmup, drain, last_arg=False):
        """Wall time per step of `steps` calls of fn (+ the drain of whatever they left in flight).  With last_arg the
        final call gets prefetch_next=False: no input is uploaded for a step that never runs."""
        for _ in range(warmup):
            fn()
        if last_arg:
            fn(False)
        drain()
        barrier()
        t0 = time.perf_counter()
        for k in range(steps):
            fn(k + 1 < steps) if last_arg else fn()
        drain()
        torch.cuda.synchronize()
        ms = torch.tensor([1e3 * (time.perf_counter() - t0) / steps], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    ms_e2e = timed_wall(e2e_submit, args.steps, 2, e2e_drain, last_arg=True)
    ms_e2e_sync = timed_wall(e2e_sync_step, max(2, min(args.steps, 5)), 1, e2e_drain)
    last = (step_no[0] - 1) & 1
    h_nll, h_Xb, h_vbs = h_out[last]
    h2d = hd.numel() * 8 + hw.numel() * 8 + hZ.numel() * 4
    d2h = h_nll.numel() * 4 + h_Xb.numel() * 4 + 8
    # checksum of the result over ALL ranks (comparable across --gpus: the synthetic rows do not depend on sharding)
    chk = torch.stack([h_nll.double().sum(), h_Xb.double().pow(2).sum()]).to(dev)
    if world > 1:
        dist.all_reduce(chk)
    nll_mean = float(chk[0]) / N
    xb_sq = float(chk[1])
    vbs_host = [float(v) for v in h_vbs]

    # ---- pure C entry with host buffers (1 GPU only): the same pipeline without Python between the calls
    ms_c = ms_c_sync = None
    if world == 1 and not args.skip_c_entry:
        import ctypes
        lib = _lib.load()
        ctx = ctypes.c_void_p()
        _lib.check(lib.gpp_host_ctx_create(ctypes.byref(ctx)), "host_ctx_create")
        hx0, hv0, hl = (t.detach().cpu().contiguous().pin_memory() for t in (pr.x0, pr.v0, pr.lvs))
        torch.cuda.synchronize()
        gp.invalidate_cache()
        torch.cuda.empty_cache()
        pending = []

        def c_submit():
            i = len(pending) & 1
            tk = ctypes.c_int32(-1)
            _lib.check(lib.gpp_gp_term_host_submit(ctx, hx0.data_ptr(), hx0.shape[0], p, hv0.data_ptr(), q, q,
                                                   hd.data_ptr(), hw.data_ptr(), hZ.data_ptr(), n, L, hl.data_ptr(),
                                                   h_out[i][0].data_ptr(), h_out[i][1].data_ptr(), h_out[i][2].data_ptr(),
                                                   ctypes.byref(tk)), "gp_term_host_submit")
            pending.append(tk.value)

        def c_drain():
            for tk in set(pending[-2:]):
                _lib.check(lib.gpp_gp_term_host_wait(ctx, tk), "gp_term_host_wait")

        def c_sync_step():
            c_submit()
            _lib.check(lib.gpp_gp_term_host_wait(ctx, pending[-1]), "gp_term_host_wait")

        ms_c = timed_wall(c_submit, args.steps, 2, c_drain)
        ms_c_sync = timed_wall(c_sync_step, max(2, min(args.steps, 5)), 1, c_drain)
        lib.gpp_host_ctx_destroy(ctx)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    pk = peaks()
    # Denominator of the roofline: the dense TF32 rate.  MEASURED_PEAKS.json holds bf16 only; dense TF32 is half the
    # dense bf16 rate by construction of the tensor pipe, and that figure (sustained: the kernel is timed inside a long,
    # power-capped step) is HIGHER than what cuBLAS' own TF32 GEMM sustains on this pool (profiles/r02_peaks.json), so
    # it is the more demanding of the two; fractions against the alternatives are listed beside it.
    tf32_peak = pk["bf16_sustained"] / 2.0
    flops_pass1 = float(n) * Q * (Q + 1) + 2.0 * n * Q * L          # algorithmic: symmetric Gram + V^T Z
    t_pass1 = stage_ms.get("pass1", float("nan"))
    achieved = flops_pass1 / (t_pass1 * 1e-3) / 1e12 if t_pass1 == t_pass1 and t_pass1 > 0 else None
    flops_total = float(n) * (Q * (Q + 1) + 4.0 * Q * L + Q + 3 * L)
    bytes_total = float(n) * (12 * Q + 12 * L + 20)
    t_roof = max(flops_total / (tf32_peak * 1e12), bytes_total / (pk["hbm_gbs"] * 1e9)) * 1e3
    # executed tensor work: every product is issued as three fp16 MMAs (hi.hi, hi.lo, lo.hi; K = 16), each half the
    # tensor-pipe time of a TF32 one: 1.5 TF32-pass equivalents
    passes = 1.5
    t_q = -(-Q // 256)
    stream_bytes = float(n) * 512 * 4 * (t_q * (t_q + 1) / 2 + t_q * -(-L // 256))
    flops_gemm = float(n) * (Q * (Q + 1) + 4.0 * Q * L)
    t_roof_k3 = max(passes * flops_gemm / (tf32_peak * 1e12), bytes_total / (pk["hbm_gbs"] * 1e9)) * 1e3
    traffic = TRAFFIC.get((args.workload, world))
    alt = pk.get("alt")
    frac_alt = None
    if alt and achieved:
        frac_alt = {"vs_tf32_cublas_sustained": achieved / alt["tf32_cublas_sustained"],
                    "vs_tf32_cublas_burst": achieved / alt["tf32_cublas_burst"],
                    "executed_fp16_vs_fp16_cublas_sustained": 3.0 * achieved / alt["fp16_cublas_sustained"],
                    "executed_fp16_vs_own_mma_only_kernel_burst": 3.0 * achieved / alt["umma_ss_fp16_burst_own_kernel"]}
    line = {
        "metric": METRIC, "value": N / (ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(args.workload, world),
        "clocks": clocks, "gpu_launches": launches, "engine": _lib.gemm_engine(),
        "e2e": {"value": N / (ms_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": ms_e2e, "sync_ms_per_step": ms_e2e_sync, "pipelined_steps_in_flight": 2,
                "api": "Vmodel.forward + GP.taylor_coeff(need_vb=False) from pinned host tensors, every step: d, w, Z host -> "
                       "device (step i+1's Z on a copy stream beside the compute of step i, two device buffers), nll, Xb, vbs "
                       "device -> pinned host on a third stream beside the next step's compute; the last step's results are "
                       "waited for inside the timed region.  sync_ms_per_step: nothing pipelined across steps (Z beside "
                       "Vmodel.forward + GP.U_UBi_Shb, then GP.taylor_coeff on the cached factorisation; each step waits "
                       "for its own results before the next one is submitted)",
                "c_entry_ms_per_step": ms_c, "c_entry_sync_ms_per_step": ms_c_sync,
                "c_entry": "gpp_gp_term_host_submit / _wait (same pipeline inside libgppvae_b200.so)"},
        "roofline": {"bound": "tensor", "kernel": "pass 1: V^T[V|Z] (pl_pass1_kernel + tc_reduce_kernel + tc_mirror_kernel; "
                                                  "operands as pre-split fp16 planes)",
                     "achieved": achieved, "peak": tf32_peak, "unit": "TFLOP/s",
                     "frac": (achieved / tf32_peak) if achieved else None, "traffic": traffic,
                     "traffic_source": TRAFFIC_SOURCE if traffic else None,
                     "algorithmic_bytes_per_launch": float(n) * (4 * Q + 4 * L) + 4.0 * Q * (Q + L),
                     "peak_source": f"{pk['source']} bf16_tflops_sustained / 2 (dense TF32), k=1 algorithmic flops",
                     "peak_alternatives": alt, "frac_alternatives": frac_alt,
                     "algorithmic_flops_per_launch": flops_pass1, "ms_per_launch": t_pass1,
                     "split_terms": "hi.hi, hi.lo and lo.hi as kind::f16 SS-form MMAs (K=16) on operand planes split once "
                                    "per matrix, common power-of-two scale: 1.5 TF32-pass equivalents",
                     "operand_stream": {"l2_to_smem_bytes_per_launch": stream_bytes,
                                        "achieved_tbs": (stream_bytes / (t_pass1 * 1e-3) / 1e12) if achieved else None,
                                        "ceiling_tbs": 24.6,
                                        "ceiling_source": "pure TMA stream of the same 8 KB boxes at 1.9 GHz: 3.0 G boxes/s "
                                                          "chip-wide whatever the box size (profiles/r02_exp3_tma_box_rate.txt)"},
                     "tf32_pass_equivalents": passes,
                     "executed_tflops_tf32_equivalent": passes * achieved if achieved else None,
                     "executed_frac": (passes * achieved / tf32_peak) if achieved else None,
                     "whole_step_frac_of_roofline": t_roof / ms, "whole_step_roofline_ms": t_roof,
                     "whole_step_frac_of_roofline_at_executed_passes": t_roof_k3 / ms,
                     "whole_step_roofline_ms_at_executed_passes": t_roof_k3},
        "stage_ms": stage_ms, "cuda_graph_ms_per_step": ms_graph, "nll_mean": nll_mean, "xb_sumsq": xb_sq, "vbs": vbs_host,
        "full_taylor_coeff": None if ms_full is None else {"ms_per_step": ms_full, "value": N / (ms_full * 1e-3)},
        "structured_route": structured, "multi_gpu_check": check,
    }
    if structured is not None:
        # roofline of the structured route (V never materialised): what is left per row is streaming -- read Z twice, write
        # Xb and nll, read the indices -- 12 L + 36 bytes per row, plus the P-long GEMMs and the replicated Q-space stage
        sb = float(n) * (12 * L + 36)
        structured["roofline"] = {"bound": "hbm", "algorithmic_bytes": sb, "hbm_floor_ms": sb / (pk["hbm_gbs"] * 1e9) * 1e3,
                                  "p_long_gemm_macs": float(pr.x0.shape[0]) * p * q * (p + 2 * L),
                                  "frac_of_hbm_floor": sb / (pk["hbm_gbs"] * 1e9) * 1e3 / structured["ms_per_step"],
                                  "note": "the replicated Q x Q Cholesky (stage_ms.factor) is the floor of this route"}
    if world == 1 and not args.skip_cpu:
        line["cpu_baseline"] = cpu_reference_timing(cfg)
    if check is not None and not check["ok"]:
        line["error"] = "multi-GPU parity check failed"
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    if check is not None and not check["ok"]:
        raise SystemExit(3)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(CONFIGS))
    ap.add_argument("--skip-cpu", action="store_true", help="omit the cpu_baseline leg")
    ap.add_argument("--skip-full", action="store_true", help="omit the full taylor_coeff (Vb) leg")
    ap.add_argument("--skip-c-entry", action="store_true", help="omit the pure-C host-buffer leg")
    ap.add_argument("--skip-structured", action="store_true", help="omit the structured-route leg")
    ap.add_argument("--check", action="store_true",
                    help="run the sharded-vs-unsharded parity check (always on when more than one rank runs)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the results of the last timed step as DIR/<name>.npy (nll, vbs, a seeded row sample of Xb)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours), not those of --impl reference")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
