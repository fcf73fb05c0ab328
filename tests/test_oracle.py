"""The oracle (oracle/gp_oracle.py) against the reference's own outputs.

Pins every oracle function to the golden vectors produced by the unmodified
reference classes (tests/golden/make_golden.py), in float32 and float64.
"""
import numpy as np
import pytest
import torch

from conftest import rel_err
from oracle import gp_oracle as O

DT = {"f32": torch.float32, "f64": torch.float64}
# fp32 runs of the *same* op sequence on the same MKL differ only by threading/blocking noise
TOL = {"f32": 2e-4, "f64": 1e-10}


def _inputs(g, tag):
    dt = DT[tag]
    X = torch.as_tensor(g["Z"], dtype=dt)
    lvs = torch.as_tensor(g["lvs"], dtype=dt)
    if "Vdirect" in g:
        V = torch.as_tensor(g["Vdirect"], dtype=dt)
    else:
        V = O.feature_map(torch.as_tensor(g["x0"], dtype=dt), torch.as_tensor(g["v0"], dtype=dt),
                          torch.as_tensor(g["d"]), torch.as_tensor(g["w"]))
    return X, V, lvs


@pytest.mark.parametrize("tag", ["f32", "f64"])
def test_feature_map_matches_reference(golden, tag):
    if "Vdirect" in golden:
        pytest.skip("case has no Vmodel")
    dt = DT[tag]
    x0, v0 = torch.as_tensor(golden["x0"], dtype=dt), torch.as_tensor(golden["v0"], dtype=dt)
    assert rel_err(O.unit_rows(x0), golden[f"{tag}_xn"]) < 1e-6
    assert rel_err(O.unit_rows(v0), golden[f"{tag}_wn"]) < 1e-6
    V = O.feature_map(x0, v0, torch.as_tensor(golden["d"]), torch.as_tensor(golden["w"]))
    assert V.shape == golden[f"{tag}_V"].shape
    assert rel_err(V, golden[f"{tag}_V"]) < 1e-6
    # layout: column j*q+k, unit row norms (SURVEY 3.4)
    q = v0.shape[1]
    xn, wn = O.unit_rows(x0), O.unit_rows(v0)
    i, j, k = 3, x0.shape[1] - 1, q - 1
    assert V[i, j * q + k].item() == pytest.approx((xn[golden["d"][i], j] * wn[golden["w"][i], k]).item(), rel=1e-6)
    assert np.allclose((V * V).sum(1).numpy(), 1.0, atol=1e-5)


@pytest.mark.parametrize("tag", ["f32", "f64"])
def test_factor_and_solve_match_reference(golden, tag):
    X, V, lvs = _inputs(golden, tag)
    vs = O.variances(lvs)
    assert rel_err(vs, golden[f"{tag}_vs"]) < 1e-6
    U, UBi, Shb = O.woodbury_factor([V], vs)
    tol = TOL[tag]
    assert rel_err(U, golden[f"{tag}_U"]) < tol
    assert rel_err(UBi, golden[f"{tag}_UBi"]) < 50 * tol
    assert rel_err(Shb, golden[f"{tag}_Shb"]) < tol
    assert rel_err(O.woodbury_solve(X, U, UBi, vs), golden[f"{tag}_KiX"]) < 50 * tol


@pytest.mark.parametrize("tag", ["f32", "f64"])
def test_taylor_coeff_matches_reference(golden, tag):
    X, V, lvs = _inputs(golden, tag)
    Xb, Vbs, vbs, nll = O.taylor_coeff(X, [V], lvs)
    tol = TOL[tag]
    assert nll.shape == (X.shape[0], 1)
    assert abs(nll.sum().item() - golden[f"{tag}_nll"].sum()) / abs(golden[f"{tag}_nll"].sum()) < tol
    assert rel_err(nll, golden[f"{tag}_nll"]) < 10 * tol
    assert rel_err(Xb, golden[f"{tag}_Xb"]) < 50 * tol
    if tag == "f64":   # fp32 Vb / vbs[0] cancel catastrophically in the reference itself (BASELINE.md s.2)
        assert rel_err(Vbs[0], golden["f64_Vb"]) < 1e-8
        assert rel_err(vbs, golden["f64_vbs"]) < 1e-9
    else:
        assert rel_err(vbs[-1:], golden["f32_vbs"][-1:]) < 1e-3
    assert not any(t.requires_grad for t in (Xb, Vbs[0], vbs, nll))


@pytest.mark.parametrize("tag", ["f32", "f64"])
def test_three_way_nll(golden, tag):
    """The reference's own check 1 (gp.py:175-183): taylor_coeff / nll / nll_ineff agree."""
    X, V, lvs = _inputs(golden, tag)
    a = O.taylor_coeff(X, [V], lvs)[3]
    b = O.nll(X, [V], lvs)
    c = O.nll_dense(X, [V], lvs)
    tol = 5e-4 if tag == "f32" else 1e-9
    assert rel_err(a, b) < tol and rel_err(a, c) < tol
    assert rel_err(b, golden[f"{tag}_nll_attached"]) < tol
    assert rel_err(c, golden[f"{tag}_nll_ineff"]) < tol


def test_taylor_expansion_and_gradients(golden):
    """The reference's own check 2 (gp.py:185-221), in float64."""
    tag = "f64"
    X, V, lvs = _inputs(golden, tag)
    Xb, Vbs, vbs, _ = O.taylor_coeff(X, [V], lvs)
    idx = torch.as_tensor(golden["mb"])
    xm = X[idx].clone().requires_grad_(True)
    vm = V[idx].clone().requires_grad_(True)
    lv = lvs.clone().requires_grad_(True)
    te = O.taylor_expansion(xm, [vm], Xb[idx], [Vbs[0][idx]], vbs, lv)
    te.sum().backward()
    assert rel_err(te, golden["f64_te"]) < 1e-9
    assert rel_err(xm.grad, golden["f64_te_gX"]) < 1e-9
    assert rel_err(vm.grad, golden["f64_te_gV"]) < 1e-9
    assert rel_err(lv.grad, golden["f64_te_glvs"]) < 1e-9
    # full-batch surrogate gradients == exact gradients of sum(nll)
    xf = X.clone().requires_grad_(True)
    vf = V.clone().requires_grad_(True)
    lf = lvs.clone().requires_grad_(True)
    O.taylor_expansion(xf, [vf], Xb, Vbs, vbs, lf).sum().backward()
    assert rel_err(xf.grad, golden["f64_nll_gX"]) < 1e-8
    assert rel_err(vf.grad, golden["f64_nll_gV"]) < 1e-7
    assert rel_err(lf.grad, golden["f64_nll_glvs"]) < 1e-8


def test_qspace_model_equals_reference_form(golden):
    """The Q-space algorithm the kernels implement (SURVEY 7.2) == the reference form, in float64."""
    X, V, lvs = _inputs(golden, "f64")
    m = O.qspace_model(X, V, lvs)
    assert rel_err(m["Xb"], golden["f64_Xb"]) < 1e-9
    assert rel_err(m["nll"], golden["f64_nll"]) < 1e-10
    assert rel_err(m["Vb"], golden["f64_Vb"]) < 1e-8
    assert rel_err(m["vbs"], golden["f64_vbs"]) < 1e-9
    assert abs(m["logdetB"].item() - np.log(golden["f64_Shb"]).sum()) < 1e-9 * max(1.0, abs(m["logdetB"].item()))


def test_init_tables_distribution():
    x0, v0 = O.init_tables(50, 9, 16, 9, torch.Generator().manual_seed(1))
    assert torch.all(x0[:, 0] == 1) and x0[:, 1:].abs().max() < 1e-2
    assert (v0 - torch.eye(9)).abs().max() < 1e-2

