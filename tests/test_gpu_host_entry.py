"""The host-buffer GP-term entry (gpp_gp_term_host_submit / _wait, gpp_gp_term_host) and the two entries only it
reaches, gpp_factor_solve and gpp_vbs, against float64.

Conventions of the edge files (tests/edge_helpers.py): the host output buffers are pinned, one row (nll, Xb) or one
element (vbs) longer than the entry writes and filled with the NaN pattern NAN_BITS; the tail must survive every call.
Bars are those of tests/test_gpu_parity.py: relative error of sum(nll) <= 1e-5, max-relative error of Xb <= 1e-4 and of
vbs <= 1e-4 (what the Python route meets in the stage-by-stage parity test), against the fp64 oracle
(oracle.gp_oracle.qspace_model, streamed on the device at c2 / c3).  Each case prints its ratio to each bar.

Beside the oracle, every case runs the "twin": the same C entries the host entry issues, called one by one through
gppvae_b200.ops on the same operands (planes branch: the factorisation of GP.U_UBi_Shb and the right-hand-side path of
GP.solve; fp32 branch: gpp_gram_vtz -> gpp_factor -> gpp_solve_w -> gpp_xb_nll -> gpp_vbs).  The twin gets the entry's
vs = [v0, vn], the softmax of lvs formed in double and rounded once (softmax2_kernel); GP.get_vs forms it in fp32 through
torch, which can differ in the last bit (the cases print whether it does), so the twin is handed the entry's vs and the
Python route proper (GP.taylor_coeff) is graded, not compared bit for bit: where it misses a bar itself, the entry's
fp64 error must be no worse than its error (see grade()).  nll, Xb and vbs of the entry must equal the twin's bit for
bit, which also pins every submission in flight to its own inputs.

Groups: A the branch switch inside the entry (gpp_planes_supported(n, Q, L) on both sides of n = 512, Q = 128, L = 64),
B every input changing between three submissions in flight, C a change of shape between submissions in flight (the
arena is carved per shape), D NULL outputs and reuse of the context, E the bench workloads c1 / c2 / c3, F
gpp_factor_solve and gpp_vbs called directly."""
import ctypes
import math

import numpy as np
import pytest
import torch

from conftest import rel_err
from edge_helpers import DEV, NAN_BITS, U, stream, workspace

pytestmark = pytest.mark.gpu

NLL_TOL, GRAD_TOL, VBS_TOL = 1e-5, 1e-4, 1e-4
GPP_ERR_WORKSPACE = -3


def _lib():
    from gppvae_b200 import _lib as L
    return L.load()


class HostCtx:
    def __init__(self):
        self.lib = _lib()
        self.h = ctypes.c_void_p()
        assert self.lib.gpp_host_ctx_create(ctypes.byref(self.h)) == 0, self.lib.gpp_last_error()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        assert self.lib.gpp_host_ctx_destroy(self.h) == 0

    def args(self, h, o, xb=True, vbs=True):
        return (self.h, h["x0"].data_ptr(), h["P"], h["p"], h["v0"].data_ptr(), h["nviews"], h["q"], h["d"].data_ptr(),
                h["w"].data_ptr(), h["X"].data_ptr(), h["n"], h["L"], h["lvs"].data_ptr(), o["nll"].data_ptr(),
                o["Xb"].data_ptr() if xb else None, o["vbs"].data_ptr() if vbs else None)

    def run(self, h, o, **kw):
        assert self.lib.gpp_gp_term_host(*self.args(h, o, **kw)) == 0, self.lib.gpp_last_error()

    def submit(self, h, o):
        tk = ctypes.c_int32(-1)
        assert self.lib.gpp_gp_term_host_submit(*self.args(h, o), ctypes.byref(tk)) == 0, self.lib.gpp_last_error()
        return tk.value

    def wait(self, tk):
        assert self.lib.gpp_gp_term_host_wait(self.h, tk) == 0, self.lib.gpp_last_error()


def host_problem(n, p, q, L, lvs, seed, kind="trained", gen_device="cpu"):
    """make_problem's inputs in pinned host memory (nviews = q)."""
    from gppvae_b200.synth import make_problem
    pr = make_problem(n, p, q, L, kind=kind, lvs=lvs, seed=seed, device=gen_device)
    pin = lambda t: t.cpu().contiguous().pin_memory()
    return dict(x0=pin(pr.x0), v0=pin(pr.v0), d=pin(pr.d), w=pin(pr.w), X=pin(pr.Z), lvs=pin(pr.lvs), n=n, p=p, q=q,
                L=L, P=pr.x0.shape[0], nviews=pr.v0.shape[0], Q=p * q, lv=tuple(lvs))


def host_outputs(n, L):
    nan = lambda *shape: torch.full(shape, NAN_BITS, dtype=torch.int32).pin_memory().view(torch.float32)
    return dict(nll=nan(n + 1), Xb=nan(n + 1, L), vbs=nan(3))


def results(o, n, L, what):
    """(nll, Xb, vbs) of a host output set, after checking that the sentinel tail survived."""
    assert int(o["nll"].view(torch.int32)[n]) == NAN_BITS, f"{what}: nll written past row {n}"
    assert bool((o["Xb"].view(torch.int32)[n] == NAN_BITS).all()), f"{what}: Xb written past row {n}"
    assert int(o["vbs"].view(torch.int32)[2]) == NAN_BITS, f"{what}: vbs written past element 2"
    return o["nll"][:n].clone(), o["Xb"][:n].clone(), o["vbs"][:2].clone()


def entry_vs(lvs):
    """vs as softmax2_kernel forms it from the fp32 lvs: in double with the maximum subtracted, rounded once to fp32."""
    a, b = float(lvs[0]), float(lvs[1])
    m = max(a, b)
    ea, eb = math.exp(a - m), math.exp(b - m)
    return torch.tensor([ea / (ea + eb), eb / (ea + eb)], dtype=torch.float32)


def device_V(h):
    """V as the drop-in Vmodel builds it (the same normalisation and Khatri-Rao kernels as the entry)."""
    import gppvae_b200
    vm = gppvae_b200.Vmodel(h["P"], h["nviews"], h["p"], h["q"]).to(DEV)
    with torch.no_grad():
        vm.x0.copy_(h["x0"]); vm.v0.copy_(h["v0"])
        return vm(h["d"].to(DEV), h["w"].to(DEV))


def oracle(h, streamed=False, V=None):
    """fp64 (nll, Xb, vbs) on the device: the Q-space model on the fp64 feature map, or (streamed, c2 / c3) on the fp32
    V of the drop-in Vmodel read in fp64 chunks, as tests/test_gpu_fullsize.py does."""
    from oracle import gp_oracle as O
    X = h["X"].to(DEV)
    lvs = h["lvs"].to(DEV).double()
    if streamed:
        m = O.qspace_model_streamed(X, V, lvs)
    else:
        V64 = O.feature_map(h["x0"].to(DEV).double(), h["v0"].to(DEV).double(), h["d"].to(DEV), h["w"].to(DEV))
        m = O.qspace_model(X.double(), V64, lvs, want_vb=False)
    return m["nll"][:, 0], m["Xb"], m["vbs"]


def twin(h, V):
    """The C entries the host entry issues, called one by one through gppvae_b200.ops with the entry's vs."""
    import gppvae_b200
    from gppvae_b200 import ops
    n, Q, L = h["n"], h["Q"], h["L"]
    Z = h["X"].to(DEV)
    vs = entry_vs(h["lvs"]).to(DEV)
    with torch.no_grad():
        if ops.planes_supported(n, Q, L):
            gp = gppvae_b200.GP().to(DEV)
            Uf, UBi, _ = gp.U_UBi_Shb([V], vs)
            Xb_solve = gp.solve(Z, Uf, UBi, vs)
            pV = ops.planes_of(V, Q)
            C = ops.atb_planes(pV, ops.split_planes(Z, L, n, L), n, Q, L)
            W, scal = ops.solve_w(Uf.fac, C, L, L, L, n)
            Xb, nll = ops.xb_nll_planes(pV, Z, L, W, n, Q, L, scal)
            assert torch.equal(Xb, Xb_solve)
        else:
            GC = ops.gram_vtz(V, Q, Z, L, n, Q, L)
            fac = ops.factor(GC, Q + L, Q, vs, False)
            W, scal = ops.solve_w(fac, GC[:, Q:], Q + L, L, L, n)
            Xb, nll = ops.xb_nll(V, Q, Z, L, W, n, Q, L, scal)
        vbs = ops.vbs_from_scal(scal, n, Q, L)
    return nll[:, 0].cpu(), Xb.cpu(), vbs.cpu()


def python_route(h, V):
    import gppvae_b200
    gp = gppvae_b200.GP().to(DEV)
    with torch.no_grad():
        gp.lvs.copy_(h["lvs"])
        Xb, _, vbs, nll = gp.taylor_coeff(h["X"].to(DEV), [V], need_vb=False)
    return nll[:, 0], Xb, vbs


def errors(got, ref):
    """(relative error of sum(nll), max-relative error of Xb, of vbs).  Where sum(nll) nearly cancels (small n) it is
    graded against the typical magnitude of its terms instead (as test_host_entry_matches_oracle does)."""
    nll, Xb, vbs = got
    rn, rX, rv = ref
    s = float(rn.sum())
    den = max(abs(s), 0.05 * float(rn.abs().sum()))
    return abs(float(nll.double().sum()) - s) / den, rel_err(Xb, rX), rel_err(vbs, rv)


def grade(tag, got, ref, py=None):
    """Ratios to the bars.  Where GP.taylor_coeff misses a bar itself (the two form V^T X in different calls, so their
    roundings differ), the entry's error must be no worse than taylor_coeff's."""
    e = errors(got, ref)
    bars = (NLL_TOL, GRAD_TOL, VBS_TOL)
    ep = errors(py, ref) if py is not None else (0.0, 0.0, 0.0)
    r = [x / b for x, b in zip(e, bars)]
    print(f"[{tag}] ratio to bar: nll {r[0]:.3f}  Xb {r[1]:.3f}  vbs {r[2]:.3f}   (errors {e[0]:.2e} {e[1]:.2e} {e[2]:.2e};"
          f" Python route {ep[0]:.2e} {ep[1]:.2e} {ep[2]:.2e})")
    for name, x, b, xp in zip(("sum(nll)", "Xb", "vbs"), e, bars, ep):
        if x > b:
            print(f"[{tag}] {name} over its bar: entry / Python route error = {x / xp:.3f}")
        assert x <= max(b, xp), f"{tag}: {name} error {x:.3g} over the bar {b:g} (Python route {xp:.3g})"
    return r


def bits_equal(tag, got, tw):
    same = [torch.equal(a.view(torch.int32), b.contiguous().view(torch.int32)) for a, b in zip(got, tw)]
    assert all(same), f"{tag}: (nll, Xb, vbs) bit-identical to the twin: {same}"


def check_case(h, o, tag, streamed=False):
    """Grade one finished run against fp64, the twin (bit for bit) and the Python route."""
    got = results(o, h["n"], h["L"], tag)
    V = device_V(h)
    tw = twin(h, V)
    bits_equal(tag, got, tw)
    ref = oracle(h, streamed, V)
    py = python_route(h, V)
    same_vs = torch.equal(torch.softmax(h["lvs"], 0), entry_vs(h["lvs"]))
    print(f"[{tag}] planes branch {bool(_lib().gpp_planes_supported(h['n'], h['Q'], h['L']))}; "
          f"GP.get_vs equals the entry's vs bit for bit: {same_vs}")
    return grade(tag, got, ref, py)


# ------------------------------------------------------------------------------ A. the branch switch inside the entry
# (n, p, q, L): n = 511 / 512 / 513 at Q = 128; Q = 124 / 128 / 132 at n = 4096; L = 60 / 64 / 68; n < 512 (fp32 SIMT
# engine on the fp32 branch); q = 9 (the c1 design) and q = 1.
A_CASES = [(511, 16, 8, 64), (512, 16, 8, 64), (513, 16, 8, 64),
           (4096, 31, 4, 64), (4096, 16, 8, 64), (4096, 33, 4, 64),
           (4096, 16, 8, 60), (4096, 16, 8, 68),
           (300, 8, 4, 32), (2000, 64, 9, 64), (1024, 128, 1, 64)]


@pytest.mark.parametrize("lvs", [(0.3, -0.3), (1.0, -2.0)])
@pytest.mark.parametrize("shape", A_CASES, ids=lambda s: "n{}-p{}-q{}-L{}".format(*s))
def test_branch_switch(shape, lvs):
    """gpp_planes_supported(n, Q, L) picks the pipeline inside the entry: split planes -> Gram tiles -> factor ->
    atb_planes -> solve_w -> xb_nll_planes, or gram_vtz -> factor_solve -> xb_nll.  Both sides of every boundary."""
    n, p, q, L = shape
    lib = _lib()
    planes = bool(lib.gpp_planes_supported(n, p * q, L))
    assert planes == (n >= 512 and p * q >= 128 and L >= 64)
    h = host_problem(n, p, q, L, lvs, seed=n + p + q + L)
    o = host_outputs(n, L)
    with HostCtx() as ctx:
        ctx.run(h, o)
    check_case(h, o, f"A n={n} Q={p * q} (p={p} q={q}) L={L} lvs={lvs}")


# ------------------------------------------------------------------------------ B. every input changes in flight
def _with_out_of_table(h):
    """A copy of the indices with one object and one view index past their tables."""
    h = dict(h)
    d, w = h["d"].clone(), h["w"].clone()
    d[5], w[h["n"] // 2] = h["P"], h["nviews"] + 3
    h["d"], h["w"] = d.pin_memory(), w.pin_memory()
    return h


def nan_reference(h):
    """The fp64 Q-space formulas on the fp64 feature map, with NaN rows of V where an index is out of its table (as the
    dense route has them).  O.qspace_model refuses such a V (its Cholesky raises on the NaN B), so the same formulas are
    run here through cholesky_ex, which returns what it got instead of raising."""
    from oracle import gp_oracle as O
    d, w = h["d"].to(DEV), h["w"].to(DEV)
    ok = (d >= 0) & (d < h["P"]) & (w >= 0) & (w < h["nviews"])
    V = O.feature_map(h["x0"].to(DEV).double(), h["v0"].to(DEV).double(), torch.where(ok, d, 0), torch.where(ok, w, 0))
    V[~ok] = float("nan")
    X = h["X"].to(DEV).double()
    vs = O.variances(h["lvs"].to(DEV).double())
    v0, vn = vs[0], vs[1]
    r, n, L, Q = v0 / vn, X.shape[0], X.shape[1], V.shape[1]
    B = torch.eye(Q, dtype=torch.float64, device=DEV) + r * (V.t() @ V)
    Lc = torch.linalg.cholesky_ex(B).L
    W = r * torch.cholesky_solve(V.t() @ X, Lc)
    Xb = (X - V @ W) / vn
    trB = torch.cholesky_inverse(Lc).diagonal().sum()
    nll = 0.5 * (X * Xb).sum(1) + 0.5 * L * (vn.log() + 2.0 * Lc.diagonal().log().sum() / n)
    vbs = torch.stack([-0.5 * (W * W).sum() / (v0 * v0) + 0.5 * L * (Q - trB) / v0,
                       -0.5 * (Xb * Xb).sum() + 0.5 * L * (n - Q + trB) / vn])
    return int((~ok).sum()), nll, Xb, vbs


def test_every_input_changes_in_flight():
    """Four submissions in flight over the two buffer sets, each with its own x0, v0, d, w, lvs and X.  The third and
    fourth reuse a buffer set (their submit waits for the results of the first and second internally).  The first three
    are graded against their own fp64 references and bit for bit against their twins; the fourth has an object and a view
    index out of their tables and must be NaN exactly where the fp64 formulas on the same indices are."""
    n, p, q, L = 2048, 16, 8, 64
    hs = [host_problem(n, p, q, L, (0.3, -0.3), seed=21), host_problem(n, p, q, L, (1.0, -1.5), seed=22),
          host_problem(n, p, q, L, (-0.5, 0.2), seed=23),
          _with_out_of_table(host_problem(n, p, q, L, (0.8, 0.1), seed=24))]
    outs = [host_outputs(n, L) for _ in hs]
    with HostCtx() as ctx:
        tickets = [ctx.submit(hs[0], outs[0]), ctx.submit(hs[1], outs[1])]
        tickets.append(ctx.submit(hs[2], outs[2]))       # waits for the first submission's results internally
        got0 = results(outs[0], n, L, "B submission 0")  # already in the host buffers: no wait on ticket 0
        tickets.append(ctx.submit(hs[3], outs[3]))       # and this one for the second's
        got1 = results(outs[1], n, L, "B submission 1")
        assert tickets == [0, 1, 0, 1]
        ctx.wait(tickets[2])
        ctx.wait(tickets[3])
    for i in range(3):
        check_case(hs[i], outs[i], f"B submission {i} lvs={hs[i]['lv']}")
    for i, g in ((0, got0), (1, got1)):
        assert all(torch.equal(a.view(torch.int32), b.view(torch.int32))
                   for a, b in zip(g, results(outs[i], n, L, f"B submission {i}")))
    bad, *ref = nan_reference(hs[3])
    got = results(outs[3], n, L, "B submission 3")
    for name, a, b in zip(("nll", "Xb", "vbs"), got, ref):
        assert torch.equal(torch.isnan(a), torch.isnan(b).cpu()), f"B submission 3: NaN pattern of {name} differs"
    print(f"[B submission 3] {bad} rows with an out-of-table index: NaN pattern of nll, Xb and vbs equal to the fp64 "
          f"formulas' ({int(torch.isnan(got[0]).sum())} of {n} nll rows NaN)")


# ------------------------------------------------------------------------------ C. shape change in flight
def arena_layout(n, p, q, L, P, nviews):
    """The carving of the context's device arena in gpp_gp_term_host_submit (gppvae_b200/csrc/api.cu): offsets of
    the two slots' buffers and of V, and the whole footprint.  The pass-1 workspace of the planes branch is read from
    gpp_gram_planes_workspace_bytes, which covers both pass-1 forms, so there the footprint is an upper bound."""
    lib = _lib()
    Q = p * q
    planes = bool(lib.gpp_planes_supported(n, Q, L))
    a256 = lambda b: (b + 255) // 256 * 256
    off = 0

    def take(b):
        nonlocal off
        o = off
        off += a256(b)
        return o
    take(P * p * 4); take(nviews * q * 4); take(16); take(9 * 8); take(16)
    slots = []
    for _ in range(2):
        s = dict(x0=take(P * p * 4), v0=take(nviews * q * 4), d=take(n * 8), w=take(n * 8), lvs=take(16),
                 X=take(n * L * 4), Xb=take(n * L * 4), nll=take(n * 4))
        s["end"] = off
        slots.append(s)
    o_V = take(n * Q * 4)
    take(Q * (Q + L) * 4); take(Q * L * 4)
    take(lib.gpp_planes_bytes(n, Q) if planes else 0); take(lib.gpp_planes_bytes(n, L) if planes else 0)
    b_state = a256(lib.gpp_factor_state_bytes(Q))
    b_tail = lib.gpp_solve_workspace_bytes(Q, L)
    if planes:
        b_tail = max(b_tail, lib.gpp_gram_planes_workspace_bytes(n, Q, L), lib.gpp_xb_planes_workspace_bytes(n, Q, L))
        b_ws = max(b_state + a256(b_tail), lib.gpp_gram_planes_workspace_bytes(n, Q, 0), lib.gpp_split_workspace_bytes(n, Q))
    else:
        b_ws = max(b_state + a256(b_tail), lib.gpp_gram_workspace_bytes(n, Q, L), lib.gpp_xb_workspace_bytes(n, Q, L))
    take(b_ws)
    return dict(slots=slots, V=o_V, total=off, planes=planes)


def test_shape_change_in_flight():
    """A large shape, then at once a smaller one that fits the arena, then one that grows it; all three in flight
    before any wait, each graded against fp64 and bit for bit against its twin.  The second shape's whole footprint
    lies below the first's V, so an unordered copy or kernel of it can reach only the first submission's tables,
    indices, X, Xb and nll (wrong numbers, never the workspace in which the Cholesky spin-waits), and its slot-1 X lies
    inside the first submission's X.  Each shape runs once in a throwaway context first, so every kernel is loaded and
    a submit only enqueues, and the first shape reads its short X (L = 64) only after the Gram tiles of 65536 rows and
    the Cholesky of Q = 4096, long after the second shape's copies queued behind it have landed.  Without the wait that
    gpp_gp_term_host_submit adds for a change of shape, the first submission's nll, Xb and vbs all differ from its twin
    on a B200; with it they are bit-identical.  (Without the warm-up and the long first phase the race went the other
    way and the case passed on the unordered code.)"""
    shapes = [(65536, 256, 16, 64), (6144, 16, 8, 256), (131072, 256, 16, 64)]
    hs = [host_problem(n, p, q, L, lv, seed=31 + i)
          for i, ((n, p, q, L), lv) in enumerate(zip(shapes, [(0.3, -0.3), (1.0, -1.5), (-0.5, 0.2)]))]
    lay = [arena_layout(h["n"], h["p"], h["q"], h["L"], h["P"], h["nviews"]) for h in hs]
    a, b, c = lay
    assert b["total"] <= a["V"], (b["total"], a["V"])
    xa, xb = a["slots"][0]["X"], b["slots"][1]["X"]
    assert xa <= xb and xb + hs[1]["n"] * hs[1]["L"] * 4 <= xa + hs[0]["n"] * hs[0]["L"] * 4
    assert c["total"] > a["total"]
    print(f"[C] arena {a['total'] / 2**20:.1f} MB; second shape's footprint {b['total'] / 2**20:.2f} MB below the "
          f"first's V at {a['V'] / 2**20:.1f} MB; its slot-1 X at {xb / 2**20:.2f} MB inside the first's X "
          f"[{xa / 2**20:.2f}, {(xa + hs[0]['n'] * hs[0]['L'] * 4) / 2**20:.2f}) MB; third grows the arena to "
          f"{c['total'] / 2**20:.1f} MB")
    with HostCtx() as warm:
        for h in hs:
            warm.run(h, host_outputs(h["n"], h["L"]))
    outs = [host_outputs(h["n"], h["L"]) for h in hs]
    with HostCtx() as ctx:
        tickets = [ctx.submit(h, o) for h, o in zip(hs, outs)]
        assert tickets == [0, 1, 0]
        ctx.wait(tickets[1])
        ctx.wait(tickets[2])
    for i, (h, o) in enumerate(zip(hs, outs)):
        check_case(h, o, f"C submission {i} n={h['n']} Q={h['Q']} L={h['L']}")


# ------------------------------------------------------------------------------ D. optional outputs and reuse
@pytest.mark.parametrize("shape", [(1024, 16, 8, 64), (300, 8, 4, 32)], ids=["planes", "fp32"])
def test_optional_outputs_and_reuse(shape):
    """Xb_host / vbs_host = NULL leave those buffers untouched and nll unchanged; waiting twice on a ticket, or on a
    ticket of a fresh context, returns 0; the synchronous form reuses the arena bit-identically; a context destroyed
    and created again gives the same bits."""
    n, p, q, L = shape
    h = host_problem(n, p, q, L, (0.4, -0.6), seed=41)
    bits = lambda r: [t.view(torch.int32).clone() for t in r]
    with HostCtx() as ctx:
        for tk in (0, 1):
            ctx.wait(tk)                                  # nothing submitted yet
        o = host_outputs(n, L)
        ctx.run(h, o)
        first = bits(results(o, n, L, "D first"))
        ctx.wait(0)
        ctx.wait(0)                                       # waiting twice
        o2 = host_outputs(n, L)
        ctx.run(h, o2)                                    # the same arena again
        assert all(torch.equal(x, y) for x, y in zip(first, bits(results(o2, n, L, "D second"))))
        for xb, vb in ((False, True), (True, False), (False, False)):
            o3 = host_outputs(n, L)
            ctx.run(h, o3, xb=xb, vbs=vb)
            nll, Xb, vbs = bits(results(o3, n, L, "D NULL outputs"))
            assert torch.equal(nll, first[0])
            assert torch.equal(Xb, first[1]) if xb else bool((o3["Xb"].view(torch.int32) == NAN_BITS).all())
            assert torch.equal(vbs, first[2]) if vb else bool((o3["vbs"].view(torch.int32) == NAN_BITS).all())
    with HostCtx() as ctx:
        o4 = host_outputs(n, L)
        ctx.run(h, o4)
        assert all(torch.equal(x, y) for x, y in zip(first, bits(results(o4, n, L, "D new context"))))
    check_case(h, o, f"D n={n} Q={p * q} L={L}")


# ------------------------------------------------------------------------------ E. the bench workloads
@pytest.mark.parametrize("cfg", ["c1", "c2", "c3"])
def test_bench_workloads(cfg):
    """c1 against the fp64 feature map; c2 and c3 (the shape bench.py times as c_entry_ms_per_step) against the
    Q-space model streamed in fp64 on the device, as tests/test_gpu_fullsize.py grades the Python route."""
    from gppvae_b200.synth import CONFIGS
    c = CONFIGS[cfg]
    n, p, q, L = c["N"], c["p"], c["q"], c["L"]
    h = host_problem(n, p, q, L, (0.0, 0.0), seed=7, gen_device=DEV)
    torch.cuda.empty_cache()
    free0, total = torch.cuda.mem_get_info()
    o = host_outputs(n, L)
    with HostCtx() as ctx:
        ctx.run(h, o)
        free1, _ = torch.cuda.mem_get_info()
    lay = arena_layout(n, p, q, L, h["P"], h["nviews"])
    check_case(h, o, f"E {cfg} n={n} Q={p * q} L={L}", streamed=cfg != "c1")
    print(f"[E {cfg}] arena {lay['total'] / 2**30:.2f} GiB (upper bound from the layout), device memory taken by the "
          f"context {(free0 - free1) / 2**30:.2f} GiB; torch peak (inputs, checker, twin) "
          f"{torch.cuda.max_memory_allocated() / 2**30:.2f} GiB of {total / 2**30:.0f} GiB")
    torch.cuda.empty_cache()


# ------------------------------------------------------------------------------ F. gpp_factor_solve and gpp_vbs
@pytest.mark.parametrize("r", [1.0, 400.0])
@pytest.mark.parametrize("Q", [128, 576, 1028])
def test_factor_solve_direct(Q, r):
    """gpp_factor_solve on a GC with ld = Q + L: bit for bit gpp_factor followed by gpp_solve_w on the same operands,
    within the Q-space fp64 bounds of test_gpu_kernel_edges.py; a workspace one byte short is refused
    (GPP_ERR_WORKSPACE) and W left untouched."""
    from gppvae_b200 import ops
    from gppvae_b200._lib import GPP_WANT_BINV, NSCAL
    from edge_helpers import check_sentinel, sentinel
    from test_gpu_kernel_edges import _qspace_check, _qspace_problem
    lib = _lib()
    L = 68
    pb = _qspace_problem(Q, r, L=L, L_true=L)
    n, GC, vs = pb["n"], pb["GC"], pb["vs"]
    fac = ops.factor(GC, Q + L, Q, vs, True)
    W_ref, scal_ref = ops.solve_w(fac, GC[:, Q:], Q + L, L, L, n)
    need = (lib.gpp_factor_state_bytes(Q) + 255) // 256 * 256 + lib.gpp_solve_workspace_bytes(Q, L)
    W, ldw = sentinel(Q, L)
    Binv = torch.empty(Q, Q, device=DEV)
    scal = torch.zeros(NSCAL, device=DEV, dtype=torch.float64)
    ws = workspace(need)
    call = lambda nbytes: lib.gpp_factor_solve(GC.data_ptr(), Q + L, Q, L, vs.data_ptr(), n, GPP_WANT_BINV,
                                               W.data_ptr(), ldw, Binv.data_ptr(), scal.data_ptr(), ws.data_ptr(), nbytes,
                                               stream())
    assert call(need - 1) == GPP_ERR_WORKSPACE and b"workspace too small" in lib.gpp_last_error()
    torch.cuda.synchronize()
    assert bool((W.view(torch.int32) == NAN_BITS).all()), "a refused call wrote W"
    assert call(need) == 0, lib.gpp_last_error()
    torch.cuda.synchronize()
    Wb = check_sentinel(W, Q, L, f"factor_solve Q={Q}")
    assert torch.equal(Wb, W_ref) and torch.equal(scal, scal_ref) and torch.equal(Binv, fac.Binv)
    _qspace_check(pb, (Binv, Wb, scal), f"F factor_solve Q={Q} r={r:g}")


# (v0, vn, tr B^-1 as an offset from Q, ||W||^2, ||Xb||^2, n_total, Q, L)
VBS_CASES = [(0.5, 0.5, -3.25, 17.0, 1234.5, 4096, 128, 64),
             (0.5, 0.5, -7e-7, 2.5e-3, 80.0, 4096, 576, 256),                   # tr B^-1 within 1e-6 of Q
             (0.7, 0.3, -100.0, 3.0e4, 2.0e9, 3_000_000_123, 4096, 256),        # n_total past 2^31
             (1e-30, 1.0 - 1e-30, -5e-7, 1e-56, 300.0, 100_000, 1024, 256),     # v0 near 1e-30
             (1.0 - 1e-30, 1e-30, -900.0, 5.0, 1e-28, 100_000, 1024, 256)]      # vn near 1e-30


@pytest.mark.parametrize("case", VBS_CASES, ids=lambda c: f"v0={c[0]:g}-trb{c[2]:+g}-N{c[5]}")
def test_vbs_direct(case):
    """gpp_vbs on a crafted scalar block: the fp64 formula (gp.py:75-76, 79-81 in Q-space form) rounded once to fp32.
    The bound is half an fp32 ulp plus the double rounding of the two terms (the kernel may contract to FMA)."""
    from gppvae_b200._lib import NSCAL, S_TRBINV, S_V0, S_VN, S_WNORM2, S_XB2
    lib = _lib()
    v0, vn, dtr, w2, xb2, n_total, Q, L = case
    sc = np.zeros(NSCAL)
    sc[S_V0], sc[S_VN], sc[S_TRBINV], sc[S_WNORM2], sc[S_XB2] = v0, vn, Q + dtr, w2, xb2
    trb = sc[S_TRBINV]
    scal = torch.tensor(sc, device=DEV, dtype=torch.float64)
    out = torch.full((3,), NAN_BITS, dtype=torch.int32, device=DEV).view(torch.float32)
    assert lib.gpp_vbs(scal.data_ptr(), n_total, Q, L, out.data_ptr(), stream()) == 0, lib.gpp_last_error()
    got = out.cpu()
    assert int(got.view(torch.int32)[2]) == NAN_BITS
    terms = [(-0.5 * w2 / (v0 * v0), 0.5 * L * (Q - trb) / v0),
             (-0.5 * xb2, 0.5 * L * (float(n_total) - Q + trb) / vn)]
    worst = 0.0
    for i, (t1, t2) in enumerate(terms):
        ref = t1 + t2
        lim = U * abs(ref) + 2.0 ** -50 * (abs(t1) + abs(t2))
        err = abs(float(got[i]) - ref)
        worst = max(worst, err / lim)
        assert err <= lim, f"vbs[{i}] = {float(got[i])!r}, fp64 {ref!r}: error {err:.3g} over {lim:.3g}"
    print(f"[F vbs {case}] worst ratio {worst:.3f}")
