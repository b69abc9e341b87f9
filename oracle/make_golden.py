"""Generate tests/golden/*.npz from the LIVE reference -- run in the build container only.

    python -m oracle.make_golden [fixture ...]      (default: every fixture in FIXTURES)

Every array under ``ref_*`` keys is an output of the unmodified reference code imported
from /root/reference (``oracle/reference_loader.py``); the ``in_*`` arrays are the seeded
inputs that produced them.  Nothing here is computed by the oracle or by the CUDA path.
The only non-reference arithmetic involved is the fixed-grid stepping inside the
``cdeint`` fixtures, which is ``oracle/odeint_port.py`` standing where torchdiffeq would
(those files are named ``solve_*`` and carry ``stepping='odeint_port'``).

The first fixture re-states the known-answer tensors hard-coded in the reference's own
test (test/test_linear_interpolation.py:125-137) so that they are pinned even if the
reference tree is not around.
"""
import math
import os
import warnings

import numpy as np
import torch

from . import reference_loader

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
NAN = float("nan")


def _np(x):
    return x.detach().cpu().numpy()


def _holes(x, frac, gen, keep_ends=False, kill_channel=None):
    mask = torch.rand(x.shape, generator=gen) < frac
    if keep_ends:
        mask[..., 0, :] = False
        mask[..., -1, :] = False
    x = x.clone()
    x[mask] = NAN
    if kill_channel is not None:
        x[0, :, kill_channel] = NAN          # one series with no observation at all
    return x


def builders(ref):
    """Coefficient builders: every (dtype, t, NaN pattern) combination, small shapes."""
    gen = torch.Generator().manual_seed(1234)
    cases = {}
    n = 0
    for dtype in (torch.float32, torch.float64):
        for shape in ((3, 9, 2), (2, 2, 6, 3), (4, 2, 1), (5, 2, 2), (7, 4), (2, 33, 8)):
            length = shape[-2]
            for own_t in (False, True):
                x = torch.randn(shape, generator=gen, dtype=torch.float64).to(dtype)
                t = ((torch.rand(length, generator=gen, dtype=torch.float64) + 0.1).cumsum(0)).to(dtype) \
                    if own_t else None
                for pattern in ("dense", "interior", "ragged", "sparse"):
                    if pattern == "dense":
                        xin = x
                    elif pattern == "interior":
                        xin = _holes(x, 0.3, gen, keep_ends=True)
                    elif pattern == "ragged":
                        xin = _holes(x, 0.4, gen, kill_channel=0 if len(shape) > 2 else None)
                    else:
                        xin = _holes(x, 0.85, gen)
                    key = "c{:03d}".format(n)
                    n += 1
                    cases[key + "_in_x"] = _np(xin)
                    if t is not None:
                        cases[key + "_in_t"] = _np(t)
                    cases[key + "_ref_linear"] = _np(ref.linear_interpolation_coeffs(xin, t))
                    cases[key + "_ref_hermite"] = _np(ref.hermite_cubic_coefficients_with_backward_differences(xin, t))
                    cases[key + "_ref_natural_v1"] = _np(ref.natural_cubic_coeffs(xin, t))
                    cases[key + "_ref_natural_v0"] = _np(ref.natural_cubic_spline_coeffs(xin, t))
                    cases[key + "_ref_ffill"] = _np(ref.misc.forward_fill(xin))
    cases["count"] = np.array(n)
    np.savez_compressed(os.path.join(OUT, "builders.npz"), **cases)
    return n


def rectilinear(ref):
    cases = {}
    # known answers written out in the reference's own test (test_linear_interpolation.py:125-137)
    x = torch.tensor([[[0.1, 0.4], [0.2, NAN], [0.9, 1.1]],
                      [[0.2, NAN], [0.3, 2.0], [0.3, NAN]]])
    known = torch.tensor([[[0.1, 0.4], [0.2, 0.4], [0.2, 0.4], [0.9, 0.4], [0.9, 1.1]],
                          [[0.2, 2.0], [0.3, 2.0], [0.3, 2.0], [0.3, 2.0], [0.3, 2.0]]])
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        got = ref.linear_interpolation_coeffs(x, rectilinear=0)
        assert torch.equal(got, known)
        cases["k_in_x"] = _np(x)
        cases["k_known"] = _np(known)
        cases["k_ref_swapped"] = _np(ref.linear_interpolation_coeffs(x[:, :, [1, 0]], rectilinear=1))
        gen = torch.Generator().manual_seed(99)
        n = 0
        for dtype in (torch.float32, torch.float64):
            for shape, tc in (((4, 7, 3), 0), ((2, 3, 5, 4), 2), ((6, 2), 1), ((3, 20, 5), 4)):
                x = torch.randn(shape, generator=gen, dtype=torch.float64).to(dtype)
                x[..., tc] = x[..., tc].abs().cumsum(-1) if x.dim() == 2 else x[..., tc].abs().cumsum(-1)
                xin = _holes(x, 0.35, gen)
                xin[..., tc] = x[..., tc]
                key = "r{:02d}".format(n)
                n += 1
                cases[key + "_in_x"] = _np(xin)
                cases[key + "_time_index"] = np.array(tc)
                cases[key + "_ref"] = _np(ref.linear_interpolation_coeffs(xin, rectilinear=tc))
    cases["count"] = np.array(n)
    np.savez_compressed(os.path.join(OUT, "rectilinear.npz"), **cases)
    return n


def evaluation(ref):
    """CubicSpline / LinearInterpolation evaluate, derivative and (bit-exact) interval indices."""
    gen = torch.Generator().manual_seed(7)
    cases = {}
    n = 0
    for dtype in (torch.float32, torch.float64):
        for shape in ((3, 9, 2), (2, 2, 6, 3), (5, 1), (2, 257, 4)):
            length = shape[-2]
            for own_t in (False, True):
                x = torch.randn(shape, generator=gen, dtype=torch.float64).to(dtype)
                t = ((torch.rand(length, generator=gen, dtype=torch.float64) + 0.1).cumsum(0)).to(dtype) \
                    if own_t else None
                coeffs = ref.natural_cubic_coeffs(x, t)
                spline = ref.CubicSpline(coeffs, t)
                knots_x = ref.linear_interpolation_coeffs(x, t)
                linear = ref.LinearInterpolation(knots_x, t)
                grid = spline.grid_points
                span = float(grid[-1] - grid[0])
                inside = torch.rand(40, generator=gen, dtype=torch.float64) * span * 1.2 + float(grid[0]) - 0.1 * span
                thirds = (grid[:-1, None] + (grid[1:] - grid[:-1])[:, None]
                          * torch.tensor([1 / 3, 2 / 3], dtype=dtype)).flatten()[:60]
                just_above = torch.nextafter(grid, grid + 1)[:30]
                query = torch.cat([grid[:30], just_above, thirds, inside.to(dtype)])
                frac, index = spline._interpret_t(query)
                key = "e{:02d}".format(n)
                n += 1
                cases[key + "_in_x"] = _np(x)
                if t is not None:
                    cases[key + "_in_t"] = _np(t)
                cases[key + "_in_query"] = _np(query)
                cases[key + "_ref_coeffs"] = _np(coeffs)
                cases[key + "_ref_index"] = _np(index)
                cases[key + "_ref_frac"] = _np(frac)
                cases[key + "_ref_cubic_eval"] = _np(spline.evaluate(query))
                cases[key + "_ref_cubic_deriv"] = _np(spline.derivative(query))
                cases[key + "_ref_linear_eval"] = _np(linear.evaluate(query))
                cases[key + "_ref_linear_deriv"] = _np(linear.derivative(query))
    cases["count"] = np.array(n)
    np.savez_compressed(os.path.join(OUT, "evaluation.npz"), **cases)
    return n


class _ReadmeFunc(torch.nn.Module):
    """The README's vector field (README.md:42-49), batch-shape agnostic."""

    def __init__(self, hidden, channels, dtype, seed):
        super().__init__()
        torch.manual_seed(seed)
        self.hidden, self.channels = hidden, channels
        self.linear = torch.nn.Linear(hidden, hidden * channels).to(dtype)

    def forward(self, t, z):
        return self.linear(z).view(*z.shape[:-1], self.hidden, self.channels)


def solves(ref):
    """Reference ``cdeint`` + ``_VectorField`` run end to end, stepping by oracle/odeint_port.py."""
    gen = torch.Generator().manual_seed(2024)
    cases = {"stepping": np.array("odeint_port")}
    n = 0
    plans = (
        # (batch shape, L, C, H, builder, control, method, step, t kind)
        ((6,), 12, 3, 4, "hermite", "cubic", "rk4", 1.0, "interval"),
        ((6,), 12, 3, 4, "hermite", "cubic", "rk4", 0.5, "inner64"),
        ((2, 3), 9, 2, 5, "natural", "cubic", "midpoint", 1.0, "knots"),
        ((4,), 17, 8, 32, "hermite", "cubic", "rk4", 1.0, "interval"),
        ((4,), 17, 8, 32, "hermite", "cubic", "euler", 0.25, "inner"),
        ((3,), 10, 2, 3, "linear", "linear", "rk4", 1.0, "interval"),
        ((3,), 10, 2, 3, "linear", "linear", "midpoint", 0.5, "inner"),
        ((5,), 8, 4, 6, "hermite", "cubic", "rk4", None, "knots"),
        ((5,), 8, 4, 6, "hermite_t", "cubic", "rk4", 0.3, "inner"),
        ((1,), 10, 2, 3, "hermite", "cubic", "rk4", 1.0, "reversed"),
    )
    with torch.no_grad():
        for dtype in (torch.float32, torch.float64):
            for bshape, length, chan, hid, builder, kind, method, step, tkind in plans:
                x = (torch.randn(*bshape, length, chan, generator=gen, dtype=torch.float64).cumsum(-2)
                     / math.sqrt(length)).to(dtype)
                t_knots = None
                if builder == "hermite":
                    control = ref.hermite_cubic_coefficients_with_backward_differences(x)
                elif builder == "hermite_t":
                    t_knots = ((torch.rand(length, generator=gen, dtype=torch.float64) + 0.2).cumsum(0)).to(dtype)
                    control = ref.hermite_cubic_coefficients_with_backward_differences(x, t_knots)
                elif builder == "natural":
                    control = ref.natural_cubic_coeffs(x)
                else:
                    control = ref.linear_interpolation_coeffs(x)
                X = ref.CubicSpline(control, t_knots) if kind == "cubic" else ref.LinearInterpolation(control, t_knots)
                lo, hi = X.interval
                if tkind == "interval":
                    t = X.interval
                elif tkind == "knots":
                    t = X.grid_points
                elif tkind == "inner":
                    w = torch.rand(5, generator=gen, dtype=torch.float64).sort().values.to(dtype)
                    t = torch.cat([lo.view(1), lo + (hi - lo) * w, hi.view(1)])
                elif tkind == "inner64":      # float64 output times with a float32 state (test_cdeint.py:43)
                    w = torch.rand(5, generator=gen, dtype=torch.float64).sort().values
                    t = torch.cat([lo.view(1).double(), lo.double() + (hi - lo).double() * w, hi.view(1).double()])
                else:
                    t = torch.stack([hi, lo])
                func = _ReadmeFunc(hid, chan, dtype, seed=100 + n)
                z0 = torch.randn(*bshape, hid, generator=gen, dtype=torch.float64).to(dtype)
                options = {} if step is None else {"step_size": step}
                out = ref.cdeint(X, func, z0, t, adjoint=False, method=method, options=options)
                # one bare vector-field evaluation straight from the reference (solver.py:117-135)
                vf = ref.solver._VectorField(X, func, True, False)
                probe = torch.as_tensor(float(lo) + 0.37 * float(hi - lo), dtype=dtype)
                key = "s{:02d}".format(n)
                n += 1
                cases[key + "_in_control"] = _np(control)
                if t_knots is not None:
                    cases[key + "_in_knots"] = _np(t_knots)
                cases[key + "_in_weight"] = _np(func.linear.weight)
                cases[key + "_in_bias"] = _np(func.linear.bias)
                cases[key + "_in_z0"] = _np(z0)
                cases[key + "_in_t"] = _np(t)
                cases[key + "_kind"] = np.array(kind)
                cases[key + "_method"] = np.array(method)
                cases[key + "_step"] = np.array(-1.0 if step is None else step)
                cases[key + "_ref_out"] = _np(out)
                cases[key + "_in_probe"] = _np(probe)
                cases[key + "_ref_field"] = _np(vf(probe, z0))
    cases["count"] = np.array(n)
    np.savez_compressed(os.path.join(OUT, "solves.npz"), **cases)
    return n


def bit_digest(x):
    """SHA-256 of a tensor's dtype, shape and values, with every NaN made the same NaN and -0 made +0: two tensors
    have the same digest exactly when ``conftest.same`` calls them equal (up to hash collisions)."""
    import hashlib
    x = x.detach().cpu().contiguous()
    x = torch.where(torch.isnan(x), torch.full_like(x, NAN), x) + 0
    head = "{}{}".format(x.dtype, tuple(x.shape)).encode()
    return hashlib.sha256(head + x.numpy().tobytes()).hexdigest()


def builders_fresh(ref):
    """The builders once more on a second seeded set of shapes (4-d batches, a single channel, length 2).  The
    comparison is bit for bit, so each reference output is stored as its ``bit_digest``: row n of ``ref_digests``
    holds case n's, in the order of ``ref_names``."""
    gen = torch.Generator().manual_seed(31337)
    cases = {}
    digests = []
    n = 0
    for dtype in (torch.float32, torch.float64):
        for shape in ((4, 11, 3), (2, 2, 5, 2), (6, 2, 1)):
            x = torch.randn(shape, generator=gen, dtype=torch.float64).to(dtype)
            t = (torch.rand(shape[-2], generator=gen, dtype=torch.float64) + 0.05).cumsum(0).to(dtype)
            for frac in (0.0, 0.25, 0.7):
                xin = x.clone()
                xin[torch.rand(shape, generator=gen) < frac] = NAN
                for tt in (None, t):
                    key = "c{:03d}".format(n)
                    n += 1
                    cases[key + "_in_x"] = _np(xin)
                    if tt is not None:
                        cases[key + "_in_t"] = _np(tt)
                    digests.append([bit_digest(out) for out in (
                        ref.linear_interpolation_coeffs(xin, tt),
                        ref.hermite_cubic_coefficients_with_backward_differences(xin, tt),
                        ref.natural_cubic_coeffs(xin, tt), ref.natural_cubic_spline_coeffs(xin, tt),
                        ref.misc.forward_fill(xin))])
    cases["ref_names"] = np.array(["linear", "hermite", "natural_v1", "natural_v0", "ffill"])
    cases["ref_digests"] = np.array(digests)
    cases["count"] = np.array(n)
    np.savez_compressed(os.path.join(OUT, "builders_fresh.npz"), **cases)
    return n


def _diff_data(seed, batch=(3,), length=9, channels=2, nan=0.0, irregular=True):
    gen = torch.Generator().manual_seed(seed)
    x = torch.randn(*batch, length, channels, generator=gen, dtype=torch.float64)
    if nan:
        hole = torch.rand(x.shape, generator=gen) < nan
        x = x.masked_fill(hole, NAN)
    t = torch.rand(length, generator=gen, dtype=torch.float64).add(0.2).cumsum(0) if irregular else None
    return x, t


def diff_formulas(ref):
    """Values and gradients (with respect to the data and the knots) of the reference builders, fp64, with and
    without missing values, for the torch-operator backward passes of torchcde_b200/_diff.py.  Input ``g*``: data
    (and knots) with the missing-value pattern ``g*_nan`` on a regular or irregular grid.  Case ``d*``: one builder
    on input ``d*_group``, its output, a seeded cotangent and the reference's gradients of <cotangent, output> (NaN
    outputs masked out; an input the output does not depend on gets a gradient of zeros(1))."""
    cases = {}
    n = 0
    groups = 0
    builders_by_name = {"hermite": ref.hermite_cubic_coefficients_with_backward_differences,
                        "natural1": ref.natural_cubic_coeffs, "natural0": ref.natural_cubic_spline_coeffs,
                        "linear_fill": ref.linear_interpolation_coeffs}
    for nan in (0.0, 0.35):
        for irregular in (False, True):
            for seed, batch, length in ((0, (3,), 9), (1, (2, 2), 6), (2, (), 2), (3, (4,), 3)):
                x, t = _diff_data(seed, batch, length, 2, nan, irregular)
                if nan:
                    x[..., 1, :] = NAN if length > 2 else x[..., 1, :]      # a fully missing knot row
                    if batch:
                        x[0] = NAN                                             # an all-NaN path
                        x[-1][..., 0, :] = NAN                                 # leading NaN
                        x[-1][..., -1, 0] = NAN                                # trailing NaN
                group = "g{:02d}".format(groups)
                groups += 1
                cases[group + "_nan"] = np.array(nan)
                cases[group + "_in_x"] = _np(x)
                if t is not None:
                    cases[group + "_in_t"] = _np(t)
                names = ["hermite", "natural1", "natural0"] + (["linear_fill", "forward_fill"] if nan else [])
                for name in names:
                    key = "d{:03d}".format(n)
                    n += 1
                    cases[key + "_fn"] = np.array(name)
                    cases[key + "_group"] = np.array(group)
                    if name == "forward_fill":
                        cases[key + "_ref_out"] = _np(ref.misc.forward_fill(x))
                        continue
                    xb = x.clone().requires_grad_(True)
                    tb = None if t is None else t.clone().requires_grad_(True)
                    want = builders_by_name[name](xb, tb)
                    ok = ~torch.isnan(want)
                    # float32-representable, so that it is stored exactly in half the bytes
                    cot = (torch.randn(want.shape, generator=torch.Generator().manual_seed(seed)) * ok).double()
                    cases[key + "_ref_out"] = _np(want)
                    cases[key + "_in_cot"] = _np(cot.float())
                    cases[key + "_ref_has_grad"] = np.array(want.requires_grad)
                    if not want.requires_grad:      # linear coefficients without NaN return their input
                        continue
                    ins = [xb] + ([tb] if t is not None else [])
                    grads = torch.autograd.grad(torch.where(ok, want, torch.zeros_like(want)), ins, cot, allow_unused=True)
                    for label, g in zip(("x", "t"), grads):
                        g = torch.zeros(1, dtype=torch.float64) if g is None else torch.nan_to_num(g)
                        cases[key + "_ref_grad_" + label] = _np(g)

    # rectilinear: a time channel without NaN and no leading NaN
    x, _ = _diff_data(5, (3,), 7, 3, 0.3, False)
    x[..., 0] = torch.arange(7, dtype=torch.float64)
    x[:, 0, :] = 1.0
    cases["rect_in_x"] = _np(x)
    cases["rect_ref"] = _np(ref.linear_interpolation_coeffs(x, rectilinear=0))

    # spline evaluation: natural cubic + linear interpolation on irregular knots, queries outside, on and between knots
    x, t = _diff_data(7, (2, 3), 8, 2, 0.0, True)
    coeffs = ref.natural_cubic_coeffs(x, t)
    spline = ref.CubicSpline(coeffs, t)
    linear = ref.LinearInterpolation(x, t)
    query = torch.tensor([t[0] - 0.3, t[0], t[2], 0.5 * (t[3] + t[4]), t[-1], t[-1] + 1.0], dtype=torch.float64)
    cases["ev_in_x"] = _np(x)
    cases["ev_in_t"] = _np(t)
    cases["ev_ref_coeffs"] = _np(coeffs)
    for i, q in enumerate((query, query[3], query.view(2, 3))):
        key = "ev{}".format(i)
        cases[key + "_in_query"] = _np(q)
        cases[key + "_ref_index"] = _np(spline._interpret_t(q)[1])
        cases[key + "_ref_linear_index"] = _np(linear._interpret_t(q)[1])
        cases[key + "_ref_cubic_eval"] = _np(spline.evaluate(q))
        cases[key + "_ref_cubic_deriv"] = _np(spline.derivative(q))
        cases[key + "_ref_linear_eval"] = _np(linear.evaluate(q))
        cases[key + "_ref_linear_deriv"] = _np(linear.derivative(q))
    cases["count"] = np.array(n)
    np.savez_compressed(os.path.join(OUT, "diff_formulas.npz"), **cases)
    return n


def _oracle_signatory():
    """A ``signatory`` module whose Logsignature is oracle/logsig_oracle.py (signatory itself is not installed)."""
    import types
    from . import logsig_oracle

    mod = types.ModuleType("signatory")

    class Logsignature:
        def __init__(self, depth):
            self.depth = depth

        def __call__(self, paths):
            out = [logsig_oracle.logsignature(p.detach().cpu().double().numpy(), self.depth) for p in paths]
            return torch.tensor(np.stack(out), dtype=paths.dtype)

    mod.Logsignature = Logsignature
    mod.logsignature_channels = lambda channels, depth: len(logsig_oracle.lyndon_words(channels, depth))
    return mod


def logsig_windows(ref):
    """The reference's own log_ode.py (window construction, NaN knots, linear fill, scaling, cumsum) with the oracle
    standing in for signatory: ``logsig_windows`` and ``logsignature_windows``, fp64."""
    import sys
    log_ode = sys.modules[ref.__name__ + ".log_ode"]
    saved = getattr(log_ode, "signatory", None)
    log_ode.signatory = _oracle_signatory()
    cases = {}
    n = 0
    try:
        torch.manual_seed(1)
        for batch, length, channels, depth, window, irregular, nan in (
                ((2,), 11, 2, 3, 2.5, False, 0.0), ((3,), 9, 3, 2, 4.0, True, 0.3),
                ((2, 2), 7, 1, 4, 1.0, False, 0.2), ((1,), 6, 2, 2, 10.0, True, 0.0)):
            x = torch.randn(*batch, length, channels, dtype=torch.float64)
            if nan:
                hole = torch.rand(x.shape) < nan
                hole[..., 0, :] = False
                hole[..., -1, :] = False
                x = x.masked_fill(hole, NAN)
            t = (torch.rand(length, dtype=torch.float64) + 0.3).cumsum(0) if irregular else None
            key = "w{:02d}".format(n)
            n += 1
            cases[key + "_in_x"] = _np(x)
            if t is not None:
                cases[key + "_in_t"] = _np(t)
            cases[key + "_depth"] = np.array(depth)
            cases[key + "_window"] = np.array(window)
            cases[key + "_ref_logsig"] = _np(ref.logsig_windows(x, depth, window, t))
            values, times = ref.logsignature_windows(x, depth, window, t)
            cases[key + "_ref_values"] = _np(values)
            cases[key + "_ref_times"] = _np(times)
    finally:
        log_ode.signatory = saved
    cases["count"] = np.array(n)
    np.savez_compressed(os.path.join(OUT, "logsig_windows.npz"), **cases)
    return n


FIXTURES = {"builders": builders, "rectilinear": rectilinear, "evaluation": evaluation, "solves": solves,
            "builders_fresh": builders_fresh, "diff_formulas": diff_formulas, "logsig_windows": logsig_windows}


def main(names=None):
    torch.set_num_threads(1)
    os.makedirs(OUT, exist_ok=True)
    ref = reference_loader.load_reference()
    for name in names or FIXTURES:
        print("{:15s}: {}".format(name, FIXTURES[name](ref)))
    for name in sorted(os.listdir(OUT)):
        print("  {:20s} {:8d} B".format(name, os.path.getsize(os.path.join(OUT, name))))


if __name__ == "__main__":
    import sys
    main(sys.argv[1:])
