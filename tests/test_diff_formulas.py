"""torchcde_b200/_diff.py (the torch-operator restatements that serve BACKWARD passes of the kernel-backed builders)
against the reference: same values and the same gradients with respect to the data and the knots, with and without
missing values.  CPU, fp64.  The reference's values and gradients are tests/golden/diff_formulas.npz
(oracle/make_golden.py)."""
import pytest
import torch

from conftest import Golden
from torchcde_b200 import _diff

_OURS = {"hermite": _diff.hermite, "natural1": lambda a, b: _diff.natural(a, b, 1),
         "natural0": lambda a, b: _diff.natural(a, b, 0), "linear_fill": _diff.linear_fill}


def _compare(g, k, ours, x, t):
    xa = x.clone().requires_grad_(True)
    ta = None if t is None else t.clone().requires_grad_(True)
    got, want = ours(xa, ta), g.t(k + "_ref_out")
    assert got.shape == want.shape
    nan_same = torch.isnan(got) == torch.isnan(want)
    assert bool(nan_same.all())
    ok = ~torch.isnan(want)
    assert torch.allclose(got[ok], want[ok], rtol=1e-9, atol=1e-11), float((got[ok] - want[ok]).abs().max())
    if not bool(g.z[k + "_ref_has_grad"]):          # e.g. linear coefficients without NaN return their input
        return
    cot = g.t(k + "_in_cot").double()
    ins_a = [xa] + ([ta] if t is not None else [])
    ga = torch.autograd.grad(torch.where(ok, got, torch.zeros_like(got)), ins_a, cot, allow_unused=True)
    for a, label in zip(ga, ("x", "t")):
        a = torch.zeros(1, dtype=torch.float64) if a is None else torch.nan_to_num(a)
        b = g.t(k + "_ref_grad_" + label)
        assert torch.allclose(a, b, rtol=1e-7, atol=1e-9), float((a - b).abs().max())


@pytest.mark.parametrize("nan", [0.0, 0.35])
@pytest.mark.parametrize("irregular", [False, True])
def test_builders_values_and_gradients_match_the_reference(nan, irregular):
    g = Golden("diff_formulas")
    checked = 0
    for i in range(g.count):
        k = "d{:03d}".format(i)
        group = g.s(k + "_group")
        if g.f(group + "_nan") != nan or g.has(group + "_in_t") != irregular:
            continue
        x = g.t(group + "_in_x")
        t = g.t(group + "_in_t") if irregular else None
        name = g.s(k + "_fn")
        if name == "forward_fill":
            ff = g.t(k + "_ref_out")
            mine = _diff.forward_fill(x)
            assert bool(((ff == mine) | (torch.isnan(ff) & torch.isnan(mine))).all())
        else:
            _compare(g, k, _OURS[name], x, t)
        checked += 1
    assert checked == (20 if nan else 12)


def test_rectilinear_matches_the_reference():
    g = Golden("diff_formulas")
    x = g.t("rect_in_x")
    want = g.t("rect_ref")
    got = _diff.linear_fill(_diff.rectilinear(x, 0), None)
    assert torch.allclose(got, want)


def test_evaluation_formulas_match_the_reference():
    g = Golden("diff_formulas")
    x, t, coeffs = g.t("ev_in_x"), g.t("ev_in_t"), g.t("ev_ref_coeffs")
    c = x.size(-1)
    a, b, two_c, three_d = coeffs[..., :c], coeffs[..., c:2 * c], coeffs[..., 2 * c:3 * c], coeffs[..., 3 * c:]
    for i in range(3):
        k = "ev{}".format(i)
        q = g.t(k + "_in_query")
        index, lindex = g.t(k + "_ref_index"), g.t(k + "_ref_linear_index")
        for deriv in (False, True):
            want = g.t(k + ("_ref_cubic_deriv" if deriv else "_ref_cubic_eval"))
            got = _diff.cubic_eval(a, b, two_c, three_d, t, q, index, deriv)
            assert torch.allclose(got, want, rtol=1e-12, atol=1e-12)
            want = g.t(k + ("_ref_linear_deriv" if deriv else "_ref_linear_eval"))
            got = _diff.linear_eval(x, t, q, lindex, deriv)
            assert torch.allclose(got, want, rtol=1e-12, atol=1e-12)
