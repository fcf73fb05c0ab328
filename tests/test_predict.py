"""GP.predict (posterior mean and variance at new rows, DESIGN 5.9) without a GPU: the textbook prediction
(tests/predict_oracle.py) against the Woodbury forms, the host logic of the dense and structured routes on the CPU stand-in engine
(tests/fake_engine.py, the k-design stand-ins of tests/test_structured_multi_effect.py, and fp64 stand-ins for the three
new entries written here from the formulas of the header), a two-rank gloo run on unequal shards, the argument errors,
and argument validation of the new C entries."""
import itertools
import os

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import test_structured_multi_effect as k_struct
from conftest import rel_err
from gppvae_b200 import ops as real_ops
from gppvae_b200._lib import S_V0
from oracle import gp_oracle as oracle
from predict_oracle import predict as textbook_predict

ALL_KINDS = [kk for r in (1, 2, 3) for kk in itertools.permutations(("kr", "object", "view"), r)]   # 15 lists
LVS = {1: (0.3, -0.5), 2: (0.5, -2.0, -1.0), 3: (2.0, -3.0, 0.0, -1.0)}


# ---------------------------------------------------------------- stand-ins for the new entries (fp64, CPU)
def _row_maps(wn, p, kinds):
    """A (nviews x Qs x p) and b (nviews x Qs): the stacked new row at (o, v) is A[v] xn[o] + b[v]."""
    nv, q = wn.shape
    widths = real_ops.effect_widths(kinds, p, q)
    w = wn.double()
    A = torch.zeros(nv, sum(widths), p, dtype=torch.float64)
    b = torch.zeros(nv, sum(widths), dtype=torch.float64)
    for kind, o, wd in zip(kinds, [sum(widths[:i]) for i in range(len(kinds))], widths):
        if kind == "kr":
            A[:, o:o + wd] = torch.einsum("vk,ji->vjki", w, torch.eye(p, dtype=torch.float64)).reshape(nv, p * q, p)
        elif kind == "object":
            A[:, o:o + wd] = torch.eye(p, dtype=torch.float64)
        else:
            b[:, o:o + q] = w
    return A, b


def kr_predict_views(Binv, wn, p, kinds):
    nv, _ = wn.shape
    A, b = _row_maps(wn, p, kinds)
    B = Binv.double()
    H = torch.einsum("vai,ab,vbj->ivj", A, B, A).reshape(p, nv * p) if ("kr" in kinds or "object" in kinds) else None
    if "view" not in kinds:
        return H.float(), None, None
    h = torch.einsum("vai,ab,vb->vi", A, B, b)
    c = torch.einsum("va,ab,vb->v", b, B, b)
    return (H.float() if H is not None else None), h.float(), c.float()


def kr_predict_rows(Y, R, YH, xn, h, c, d, w, P, nviews, L, scal):
    p = xn.shape[1]
    bad = (d < 0) | (d >= P) | (w < 0) | (w >= nviews)
    dd, ww = d.clamp(0, P - 1), w.clamp(0, nviews - 1)
    mean = torch.zeros(d.shape[0], L, dtype=torch.float64)
    if Y is not None:
        mean += Y.double().view(P, nviews, L)[dd, ww]
    if R is not None:
        mean += R.double()[ww]
    x = xn.double()[dd]
    var = torch.zeros(d.shape[0], dtype=torch.float64)
    if YH is not None:
        var += (x * YH.double().view(P, nviews, p)[dd, ww]).sum(1)
        if h is not None:
            var += 2 * (x * h.double()[ww]).sum(1)
    if c is not None:
        var += c.double()[ww]
    var = scal[S_V0] * var[:, None]
    mean[bad] = float("nan")
    var[bad] = float("nan")
    return mean.float(), var.float()


def rows_dot(A, B, cols, scal):
    return (scal[S_V0] * (A.double()[:, :cols] * B.double()[:, :cols]).sum(1, keepdim=True)).float()


def install(monkeypatch):
    k_struct.install(monkeypatch)
    for name, fn in (("kr_predict_views", kr_predict_views), ("kr_predict_rows", kr_predict_rows),
                     ("rows_dot", rows_dot)):
        monkeypatch.setattr(real_ops, name, fn)


# ---------------------------------------------------------------- problems
def _tables(n=60, P=21, nv=9, p=3, q=9, L=6, seed=0):
    """Z, (xn, wn, d, w) of the training rows and (dn, wn_) of new rows over every slot, including the slots of the
    objects that have no training rows; p, q and L are not multiples of 4."""
    g = torch.Generator().manual_seed(seed)
    xn = oracle.unit_rows(torch.randn(P, p, generator=g))
    wn = oracle.unit_rows(torch.eye(nv, q) + 0.5 * torch.randn(nv, q, generator=g))
    d = torch.randint(0, P - 3, (n,), generator=g)          # the last three objects have no rows: empty slots
    w = torch.randint(0, nv, (n,), generator=g)
    grid = torch.arange(P * nv)
    dn, wn_idx = grid // nv, grid % nv
    Vk = oracle.feature_map(xn, wn, d, w)
    Z = 0.5 * torch.randn(n, L, generator=g) + Vk @ torch.randn(p * q, L, generator=g) + \
        wn[w] @ torch.randn(q, L, generator=g)
    return Z, (xn, wn, d, w), (dn, wn_idx)


def _dense(xn, wn, d, w):
    return dict(kr=oracle.feature_map(xn, wn, d, w), object=xn[d], view=wn[w])


def _factored(xn, wn, d, w, kinds):
    from gppvae_b200.vmod import KhatriRao, ObjectEffect, ViewEffect
    kr = KhatriRao(xn, wn, d.contiguous(), w.contiguous())
    return [kr if k == "kr" else ObjectEffect(kr) if k == "object" else ViewEffect(kr) for k in kinds]


def _gp(k, lvs):
    from gppvae_b200 import GP
    gp = GP(n_rand_effs=k)
    with torch.no_grad():
        gp.lvs.copy_(torch.tensor(lvs))
    return gp


def _woodbury(Z, Vs, Vs_new, lvs):
    """mean = u W and var = u D B^-1 D u^T (B = I + D G D / vn) for the stacked new rows u, in fp64."""
    vs = torch.softmax(torch.tensor(lvs, dtype=torch.float64), 0)
    Vt = torch.cat([vs[i].sqrt() * V.double() for i, V in enumerate(Vs)], 1)
    Vn = torch.cat([vs[i].sqrt() * V.double() for i, V in enumerate(Vs_new)], 1)
    Binv = torch.linalg.inv(torch.eye(Vt.shape[1], dtype=torch.float64) + Vt.t() @ Vt / vs[-1])
    W = Binv @ Vt.t() @ Z.double() / vs[-1]
    return Vn @ W, ((Vn @ Binv) * Vn).sum(1, keepdim=True)


# ---------------------------------------------------------------- the oracle against the Woodbury forms
@pytest.mark.parametrize("case", ["dense", "kr", "k2", "k3"])
def test_oracle_prediction_is_the_woodbury_form(case):
    Z, (xn, wn, d, w), (dn, wnn) = _tables()
    tr, new = _dense(xn, wn, d, w), _dense(xn, wn, dn, wnn)
    if case == "dense":
        g = torch.Generator().manual_seed(3)
        Vs, Vs_new = [torch.randn(60, 7, generator=g)], [torch.randn(11, 7, generator=g)]
    else:
        kinds = {"kr": ["kr"], "k2": ["kr", "view"], "k3": ["object", "kr", "view"]}[case]
        Vs, Vs_new = [tr[k] for k in kinds], [new[k] for k in kinds]
    lvs = LVS[len(Vs)]
    mean, var = textbook_predict(Z.double(), [V.double() for V in Vs], [V.double() for V in Vs_new],
                               torch.tensor(lvs, dtype=torch.float64))
    wm, wv = _woodbury(Z, Vs, Vs_new, lvs)
    assert rel_err(mean, wm) < 1e-10 and rel_err(var, wv) < 1e-10
    assert bool((var > 0).all())


@pytest.mark.parametrize("kinds", ALL_KINDS, ids=["-".join(k) for k in ALL_KINDS])
def test_header_forms_against_the_oracle(kinds):
    """u = A_v x + b_v: mean = Y[o, v] + R[v] and var = scal[V0] (x^T H_v x + 2 x^T h_v + c_v) through the three stand-ins,
    for every ordered kinds list, against the textbook prediction."""
    Z, (xn, wn, d, w), (dn, wnn) = _tables()
    k = len(kinds)
    lvs = LVS[k]
    p = real_ops.round4(xn.shape[1])
    xp = torch.zeros(xn.shape[0], p)
    xp[:, : xn.shape[1]] = xn
    tr = _dense(xp, wn, d, w)
    vs = torch.softmax(torch.tensor(lvs, dtype=torch.float64), 0)
    widths = real_ops.effect_widths(kinds, p, wn.shape[1])
    Vt = torch.zeros(d.shape[0], sum(widths), dtype=torch.float64)
    for i, (kd, o) in enumerate(zip(kinds, [sum(widths[:i]) for i in range(k)])):
        Vt[:, o:o + tr[kd].shape[1]] = tr[kd].double()
    D = torch.cat([vs[i].sqrt().expand(wd) for i, wd in enumerate(widths)])
    Binv = D[:, None] * torch.linalg.inv(torch.eye(Vt.shape[1], dtype=torch.float64) +
                                         D[:, None] * (Vt.t() @ Vt) * D[None, :] / vs[-1]) * D[None, :]
    W = (Binv @ Vt.t() @ Z.double() / vs[-1]).float()
    M, R = k_struct.kr_assemble_m_blocks(W, wn, p, kinds, Z.shape[1])
    Y = xp.double() @ M.double() if M is not None else None
    H, h, c = kr_predict_views(Binv.float(), wn, p, kinds)
    YH = xp.double() @ H.double() if H is not None else None
    scal = torch.zeros(8, dtype=torch.float64)
    scal[S_V0] = 1.0
    mean, var = kr_predict_rows(Y, R, YH, xp, h, c, dn, wnn, xn.shape[0], wn.shape[0], Z.shape[1], scal)
    dense = _dense(xn, wn, d, w)
    new = _dense(xn, wn, dn, wnn)
    om, ov = textbook_predict(Z.double(), [dense[kd].double() for kd in kinds], [new[kd].double() for kd in kinds],
                            torch.tensor(lvs, dtype=torch.float64))
    assert rel_err(mean, om) < 1e-5 and rel_err(var, ov) < 1e-5


# ---------------------------------------------------------------- GP.predict on the stand-in engine
def _check(mean, var, om, ov, tol=1e-5):
    assert mean.shape == om.shape and var.shape == ov.shape
    assert rel_err(mean, om) < tol and rel_err(var, ov) < tol


def test_gp_predict_dense_and_khatri_rao(monkeypatch):
    install(monkeypatch)
    Z, (xn, wn, d, w), (dn, wnn) = _tables()
    lvs = LVS[1]
    om, ov = textbook_predict(Z.double(), [oracle.feature_map(xn, wn, d, w).double()],
                            [oracle.feature_map(xn, wn, dn, wnn).double()], torch.tensor(lvs, dtype=torch.float64))
    gp = _gp(1, lvs)
    _check(*gp.predict(Z, [oracle.feature_map(xn, wn, d, w)], [oracle.feature_map(xn, wn, dn, wnn)]), om, ov)
    gp = _gp(1, lvs)
    _check(*gp.predict(Z, _factored(xn, wn, d, w, ["kr"]), _factored(xn, wn, dn, wnn, ["kr"])), om, ov)


def test_gp_predict_dense_in_chunks(monkeypatch):
    install(monkeypatch)
    Z, (xn, wn, d, w), (dn, wnn) = _tables()
    gp = _gp(1, LVS[1])
    V, Vn = oracle.feature_map(xn, wn, d, w), oracle.feature_map(xn, wn, dn, wnn)
    m1, v1 = gp.predict(Z, [V], [Vn])
    m2, v2 = gp._predict_dense(Z, [V], [Vn], Vn.shape[0], chunk=16)
    assert rel_err(m2, m1) < 1e-6 and rel_err(v2, v1) < 1e-6


@pytest.mark.parametrize("kinds", [k for k in ALL_KINDS if len(k) > 1], ids=["-".join(k) for k in ALL_KINDS if len(k) > 1])
def test_gp_predict_k_designs(monkeypatch, kinds):
    """k factored designs and the same k dense designs against the textbook prediction."""
    install(monkeypatch)
    Z, (xn, wn, d, w), (dn, wnn) = _tables()
    k = len(kinds)
    tr, new = _dense(xn, wn, d, w), _dense(xn, wn, dn, wnn)
    om, ov = textbook_predict(Z.double(), [tr[kd].double() for kd in kinds], [new[kd].double() for kd in kinds],
                            torch.tensor(LVS[k], dtype=torch.float64))
    _check(*_gp(k, LVS[k]).predict(Z, _factored(xn, wn, d, w, kinds), _factored(xn, wn, dn, wnn, kinds)), om, ov)
    real_ops.STACKED.invalidate()
    _check(*_gp(k, LVS[k]).predict(Z, [tr[kd] for kd in kinds], [new[kd] for kd in kinds]), om, ov)


def test_out_of_table_rows_are_nan(monkeypatch):
    install(monkeypatch)
    Z, (xn, wn, d, w), (dn, wnn) = _tables()
    dn, wnn = dn.clone(), wnn.clone()
    dn[3], wnn[7] = xn.shape[0], -1
    kinds = ("kr", "object", "view")
    mean, var = _gp(3, LVS[3]).predict(Z, _factored(xn, wn, d, w, kinds), _factored(xn, wn, dn, wnn, kinds))
    bad = torch.zeros(dn.shape[0], dtype=torch.bool)
    bad[[3, 7]] = True
    assert bool(torch.isnan(mean[bad]).all()) and bool(torch.isnan(var[bad]).all())
    assert bool(torch.isfinite(mean[~bad]).all()) and bool(torch.isfinite(var[~bad]).all())


def test_cache_hit_after_taylor_coeff_and_no_index_of_new_rows(monkeypatch):
    install(monkeypatch)
    Z, (xn, wn, d, w), (dn, wnn) = _tables()
    for kinds in (["kr"], ["view", "kr", "object"]):
        k = len(kinds)
        gp = _gp(k, LVS[k])
        Vs = _factored(xn, wn, d, w, kinds)
        gp.taylor_coeff(Z, Vs)
        hits = gp.cache_hits
        Vn = _factored(xn, wn, dn, wnn, kinds)
        base = Vn[0] if kinds[0] == "kr" else Vn[0].kr

        def refuse(*a, **kw):
            raise AssertionError("predict must not call index() on the new rows")
        base.index = base.max_count = base.rows_in_table = refuse
        gp.predict(Z, Vs, Vn)
        assert gp.cache_hits == hits + 1


def test_argument_errors(monkeypatch):
    install(monkeypatch)
    Z, (xn, wn, d, w), (dn, wnn) = _tables()
    V, Vn = oracle.feature_map(xn, wn, d, w), oracle.feature_map(xn, wn, dn, wnn)
    gp = _gp(1, LVS[1])
    with pytest.raises(ValueError, match="positive number of rows"):
        gp.predict(Z, [V], [Vn[:0]])
    with pytest.raises(ValueError, match="columns"):
        gp.predict(Z, [V], [Vn[:, :-1]])
    with pytest.raises(ValueError, match="mixed"):
        gp.predict(Z, [V], _factored(xn, wn, dn, wnn, ["kr"]))
    with pytest.raises(ValueError, match="mixed"):
        gp.predict(Z, _factored(xn, wn, d, w, ["kr"]), [Vn])
    with pytest.raises(ValueError, match="tables"):
        gp.predict(Z, _factored(xn, wn, d, w, ["kr"]), _factored(xn * 0.5, wn, dn, wnn, ["kr"]))
    with pytest.raises(ValueError, match="tables"):
        gp.predict(Z, _factored(xn, wn, d, w, ["kr"]), _factored(xn, wn[:-1], dn % (wn.shape[0] - 1),
                                                                  wnn % (wn.shape[0] - 1), ["kr"]))
    with pytest.raises(ValueError, match="device"):
        gp.predict(Z.to("meta"), [V], [Vn])
    gp3 = _gp(3, LVS[3])
    kinds = ["kr", "object", "view"]
    with pytest.raises(ValueError, match="kinds|columns"):
        gp3.predict(Z, _factored(xn, wn, d, w, kinds), _factored(xn, wn, dn, wnn, ["kr", "view", "object"]))
    with pytest.raises(ValueError, match="designs"):
        gp3.predict(Z, _factored(xn, wn, d, w, kinds), _factored(xn, wn, dn, wnn, kinds[:2]))


# ---------------------------------------------------------------- two ranks (gloo)
def _shard_worker(rank, world, port, out):
    from _pytest.monkeypatch import MonkeyPatch
    from gppvae_b200 import GP
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    mpch = MonkeyPatch()
    install(mpch)
    try:
        Z, (xn, wn, d, w), (dn, wnn) = _tables()
        n = Z.shape[0]
        rows = slice(0, 23) if rank == 0 else slice(23, n)          # unequal shards
        res = {}
        for kinds in (["kr"], ["kr", "object", "view"]):
            k = len(kinds)
            gp = GP(n_rand_effs=k).shard_rows(n_total=n)
            with torch.no_grad():
                gp.lvs.copy_(torch.tensor(LVS[k]))
            res["-".join(kinds)] = gp.predict(Z[rows], _factored(xn, wn, d[rows], w[rows], kinds),
                                              _factored(xn, wn, dn, wnn, kinds))
        gp = GP().shard_rows(n_total=n)
        with torch.no_grad():
            gp.lvs.copy_(torch.tensor(LVS[1]))
        res["dense"] = gp.predict(Z[rows], [oracle.feature_map(xn, wn, d[rows], w[rows])],
                                  [oracle.feature_map(xn, wn, dn, wnn)])
        torch.save(res, os.path.join(out, f"r{rank}.pt"))
    finally:
        mpch.undo()
        dist.destroy_process_group()


def test_row_sharding_world2_gloo(tmp_path, monkeypatch):
    port = 29500 + (os.getpid() % 2000) + 31
    mp.spawn(_shard_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    install(monkeypatch)
    Z, (xn, wn, d, w), (dn, wnn) = _tables()
    r0, r1 = (torch.load(os.path.join(tmp_path, f"r{r}.pt")) for r in (0, 1))
    for key in r0:
        assert torch.equal(r0[key][0], r1[key][0]) and torch.equal(r0[key][1], r1[key][1]), key
    for kinds in (["kr"], ["kr", "object", "view"]):
        k = len(kinds)
        m, v = _gp(k, LVS[k]).predict(Z, _factored(xn, wn, d, w, kinds), _factored(xn, wn, dn, wnn, kinds))
        assert rel_err(r0["-".join(kinds)][0], m) < 1e-5 and rel_err(r0["-".join(kinds)][1], v) < 1e-5
    m, v = _gp(1, LVS[1]).predict(Z, [oracle.feature_map(xn, wn, d, w)], [oracle.feature_map(xn, wn, dn, wnn)])
    assert rel_err(r0["dense"][0], m) < 1e-5 and rel_err(r0["dense"][1], v) < 1e-5


# ---------------------------------------------------------------- C entries: validation before any device work
@pytest.fixture(scope="module")
def lib():
    from gppvae_b200 import _lib, build
    build.build()
    return _lib.load(build_if_missing=False)


def test_predict_entries_validate_without_a_device(lib):
    from gppvae_b200 import _lib
    a = 1 << 12   # a non-null, 16-byte aligned fake device address: validation must fail before it is used
    p, q, nv = 8, 5, 7
    kall = _lib.host_i32([0, 1, 2])          # Binv width p q + p + round4(q) = 56
    kv = _lib.host_i32([2])
    views = lambda **k: [k.get("B", a), k.get("ldb", 56), k.get("wn", a), k.get("p", p), k.get("q", q), nv, k.get("k", 3),
                         k.get("kinds", kall), k.get("H", a), k.get("ldh", nv * p), k.get("h", a), k.get("c", a), None]
    assert lib.gpp_kr_predict_views(*views(B=None)) == -1
    assert b"kr_predict_views: null pointer" in lib.gpp_last_error()
    assert lib.gpp_kr_predict_views(*views(H=None)) == -1
    assert lib.gpp_kr_predict_views(*views(h=None)) == -1
    assert lib.gpp_kr_predict_views(*views(p=6)) == -1                                   # p % 4
    assert lib.gpp_kr_predict_views(*views(ldb=52)) == -1                                # ldb < stacked width
    assert lib.gpp_kr_predict_views(*views(ldh=nv * p - 4)) == -1                        # ldh < nviews p
    assert lib.gpp_kr_predict_views(*views(kinds=_lib.host_i32([0, 0, 2]))) == -1        # repeated kind
    assert b"kinds" in lib.gpp_last_error()
    assert lib.gpp_kr_predict_views(*views(q=300, ldb=4000)) == -1                       # q (q + 1) > 160 KB
    assert b"q too large" in lib.gpp_last_error()
    # the view kind alone needs no H; without the view kind h and c may be NULL -- both get past the pointer checks
    assert lib.gpp_kr_predict_views(*views(k=1, kinds=kv, H=None, ldb=4, ldh=0, p=6)) == -1
    assert b"p must be" in lib.gpp_last_error()
    L = 12
    rows = lambda **k: [k.get("Y", a), k.get("ldy", nv * L), k.get("R", a), k.get("ldr", L), k.get("YH", a),
                        k.get("ldyh", nv * p), k.get("xn", a), a, k.get("c", a), k.get("d", a), a, 10, 20, p, nv,
                        k.get("L", L), k.get("scal", a), k.get("mean", a), k.get("ldm", L), k.get("var", a), None]
    assert lib.gpp_kr_predict_rows(*rows(d=None)) == -1
    assert lib.gpp_kr_predict_rows(*rows(Y=None, R=None)) == -1
    assert lib.gpp_kr_predict_rows(*rows(xn=None)) == -1                                 # YH without xn
    assert lib.gpp_kr_predict_rows(*rows(c=None)) == -1                                  # R without c
    assert lib.gpp_kr_predict_rows(*rows(var=None)) == -1
    assert b"kr_predict_rows: null pointer" in lib.gpp_last_error()
    assert lib.gpp_kr_predict_rows(*rows(L=10, ldm=12)) == -1                            # L % 4
    assert lib.gpp_kr_predict_rows(*rows(ldy=nv * L - 4)) == -1
    assert lib.gpp_kr_predict_rows(*rows(ldr=8)) == -1
    assert lib.gpp_kr_predict_rows(*rows(ldyh=nv * p - 1)) == -1
    assert lib.gpp_kr_predict_rows(*rows(ldm=8)) == -1
    assert lib.gpp_kr_predict_rows(*rows(mean=a + 4)) == -1                              # misaligned
    assert b"kr_predict_rows: bad leading dimension" in lib.gpp_last_error()
    assert lib.gpp_rows_dot(None, 8, a, 8, 10, 8, a, a, None) == -1
    assert b"rows_dot: null pointer" in lib.gpp_last_error()
    assert lib.gpp_rows_dot(a, 8, a, 8, 10, 6, a, a, None) == -1                         # cols % 4
    assert lib.gpp_rows_dot(a, 4, a, 8, 10, 8, a, a, None) == -1                         # lda < cols
    assert lib.gpp_rows_dot(a, 8, a + 4, 8, 10, 8, a, a, None) == -1                     # misaligned
    assert b"rows_dot: bad leading dimension" in lib.gpp_last_error()
