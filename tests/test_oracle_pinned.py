"""Pin the CPU oracle (oracle/cde_oracle.py) to the reference, bit for bit.

The fixtures in tests/golden/ are outputs of the unmodified reference
(oracle/make_golden.py).
"""
import warnings

import pytest
import torch

from conftest import Golden, same
from oracle import cde_oracle as O
from oracle.make_golden import bit_digest


def test_builders_match_reference_fixtures():
    g = Golden("builders")
    assert g.count == 96
    for i in range(g.count):
        k = "c{:03d}".format(i)
        x = g.t(k + "_in_x")
        t = g.t(k + "_in_t") if g.has(k + "_in_t") else None
        assert same(O.linear_knots(x, t), g.t(k + "_ref_linear")), k
        assert same(O.hermite_backward_difference_coeffs(x, t), g.t(k + "_ref_hermite")), k
        assert same(O.natural_cubic_coeffs(x, t, version=1), g.t(k + "_ref_natural_v1")), k
        assert same(O.natural_cubic_coeffs(x, t, version=0), g.t(k + "_ref_natural_v0")), k
        assert same(O.carry_forward(x), g.t(k + "_ref_ffill")), k


def test_linear_knots_returns_input_object_when_dense():
    # interpolation_linear.py:169-171: no NaN -> the very same tensor comes back
    x = torch.randn(3, 5, 2)
    assert O.linear_knots(x) is x


def test_rectilinear_known_answers_and_fixtures():
    g = Golden("rectilinear")
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        x = g.t("k_in_x")
        # the tensors written out in the reference's test_linear_interpolation.py:125-137
        assert torch.equal(O.linear_knots(x, rectilinear=0), g.t("k_known"))
        assert torch.equal(O.linear_knots(x[:, :, [1, 0]], rectilinear=1), g.t("k_ref_swapped"))
        assert torch.equal(O.linear_knots(x[0], rectilinear=0), g.t("k_known")[0])
        bad = x.clone()
        bad[0, 1, 0] = float("nan")
        with pytest.raises(AssertionError):
            O.linear_knots(bad, rectilinear=0)
        for i in range(g.count):
            k = "r{:02d}".format(i)
            got = O.linear_knots(g.t(k + "_in_x"), rectilinear=int(g.z[k + "_time_index"]))
            assert same(got, g.t(k + "_ref")), k


def test_evaluation_and_interval_indices_bit_exact():
    g = Golden("evaluation")
    for i in range(g.count):
        k = "e{:02d}".format(i)
        x = g.t(k + "_in_x")
        t = g.t(k + "_in_t") if g.has(k + "_in_t") else O.knot_times(x.size(-2), x.dtype)
        q = g.t(k + "_in_query")
        coeffs = g.t(k + "_ref_coeffs")
        frac, index = O.locate(t, q, coeffs.size(-2))
        assert torch.equal(index, g.t(k + "_ref_index")), k          # integer work: bit exact
        assert torch.equal(frac, g.t(k + "_ref_frac")), k
        assert same(O.cubic_evaluate(coeffs, t, q), g.t(k + "_ref_cubic_eval")), k
        assert same(O.cubic_derivative(coeffs, t, q), g.t(k + "_ref_cubic_deriv")), k
        assert same(O.linear_evaluate(x, t, q), g.t(k + "_ref_linear_eval")), k
        assert same(O.linear_derivative(x, t, q), g.t(k + "_ref_linear_deriv")), k


def test_interval_semantics_at_knots():
    # SURVEY 8(a) row 2: a knot t_n (n > 0) belongs to interval n-1 with fraction = width
    knots = O.knot_times(256, torch.float32)
    for value, want_idx, want_frac in ((0.0, 0, 0.0), (0.5, 0, 0.5), (1.0, 0, 1.0), (255.0, 254, 1.0),
                                       (256.0, 254, 2.0), (-1.0, 0, -1.0)):
        frac, idx = O.locate(knots, torch.tensor(value), 255)
        assert int(idx) == want_idx and float(frac) == want_frac
    frac, idx = O.locate(knots, torch.nextafter(torch.tensor(1.0), torch.tensor(2.0)), 255)
    assert int(idx) == 1


def test_solve_fixtures_vector_field_and_call_site():
    g = Golden("solves")
    assert g.s("stepping") == "odeint_port"
    for i in range(g.count):
        k = "s{:02d}".format(i)
        control = g.t(k + "_in_control")
        kind = g.s(k + "_kind")
        n_knots = control.size(-2) + (1 if kind == "cubic" else 0)
        knots = g.t(k + "_in_knots") if g.has(k + "_in_knots") else O.knot_times(n_knots, control.dtype)
        w, b, z0, t = g.t(k + "_in_weight"), g.t(k + "_in_bias"), g.t(k + "_in_z0"), g.t(k + "_in_t")
        probe = g.t(k + "_in_probe")
        dxdt = O.cubic_derivative(control, knots, probe) if kind == "cubic" else O.linear_derivative(control, knots, probe)
        # reference _VectorField.forward (solver.py:117-135), no stepping involved: pinned
        assert same(O.linear_field(w, b, z0, dxdt), g.t(k + "_ref_field")), k
        step = g.f(k + "_step")
        out = O.cdeint_linear(control, knots, w, b, z0, t, g.s(k + "_method"), None if step < 0 else step, kind)
        assert same(out, g.t(k + "_ref_out")), k


def test_oracle_against_live_reference_fresh_inputs():
    # tests/golden/builders_fresh.npz: a second seeded set of inputs and the SHA-256 of the reference's outputs on them
    g = Golden("builders_fresh")
    assert g.count == 36
    assert list(g.z["ref_names"]) == ["linear", "hermite", "natural_v1", "natural_v0", "ffill"]
    for i in range(g.count):
        k = "c{:03d}".format(i)
        xin = g.t(k + "_in_x")
        tt = g.t(k + "_in_t") if g.has(k + "_in_t") else None
        got = (O.linear_knots(xin, tt), O.hermite_backward_difference_coeffs(xin, tt), O.natural_cubic_coeffs(xin, tt, 1),
               O.natural_cubic_coeffs(xin, tt, 0), O.carry_forward(xin))
        assert [bit_digest(out) for out in got] == list(g.z["ref_digests"][i]), k


def test_validation_messages_follow_reference():
    with pytest.raises(ValueError, match="floating point"):
        O.linear_knots(torch.zeros(3, 2, dtype=torch.int64))
    with pytest.raises(ValueError, match="at least two dimensions"):
        O.linear_knots(torch.zeros(3))
    with pytest.raises(ValueError, match="monotonically increasing"):
        O.linear_knots(torch.zeros(3, 2), torch.tensor([0.0, 2.0, 1.0]))
    with pytest.raises(ValueError, match="one dimensional"):
        O.linear_knots(torch.zeros(3, 2), torch.zeros(3, 1))
    with pytest.raises(ValueError, match="time dimension of X must equal"):
        O.linear_knots(torch.zeros(3, 2), torch.tensor([0.0, 1.0]))
    with pytest.raises(ValueError, match="at least 2"):
        O.linear_knots(torch.zeros(1, 2))
