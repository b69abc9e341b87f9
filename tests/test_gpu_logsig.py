"""SURVEY 8(f)4: ``logsig_windows`` / ``logsignature_windows`` on the device.  (1) the kernel against the independent fp64
oracle; (2) the whole transform against the REFERENCE's own log_ode.py executed on the CPU with the oracle plugged in as
``signatory`` (so the window construction, NaN knots, linear fill, scaling and cumsum are the reference's code; its
outputs are tests/golden/logsig_windows.npz, oracle/make_golden.py); (3) the reference's test_log_ode.py:8-36 with the
oracle in signatory's place."""
import numpy as np
import pytest
import torch

import torchcde_b200 as cde
from conftest import Golden
from oracle import logsig_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda"


@pytest.mark.parametrize("dtype,tol", [(torch.float64, 1e-11), (torch.float32, 2e-5)])
def test_kernel_against_the_oracle(dtype, tol):
    torch.manual_seed(0)
    for channels, depth, length, window in ((3, 4, 13, 4.0), (1, 3, 6, 2.0), (8, 3, 9, 3.0), (2, 5, 10, 5.0), (4, 1, 5, 1.0)):
        x = torch.randn(3, length, channels, dtype=torch.float64).cumsum(1)
        got = cde.logsig_windows(x.to(DEV).to(dtype), depth, window).cpu().double()
        n_words = len(O.lyndon_words(channels, depth))
        want = [torch.zeros(3, n_words, dtype=torch.float64)]
        want[0][:, :channels] = x[:, 0]
        edges = list(range(0, length - 1, int(window))) + [length - 1]
        for lo, hi in zip(edges[:-1], edges[1:]):
            want.append(torch.tensor(np.stack([O.logsignature(p[lo:hi + 1].numpy(), depth) for p in x])))
        want = torch.stack(want, dim=-2).cumsum(-2)
        assert got.shape == want.shape
        scale = float(want.abs().max())
        assert float((got - want).abs().max()) <= tol * max(1.0, scale), (channels, depth)


def test_whole_transform_against_the_reference_code_with_the_oracle_as_signatory():
    g = Golden("logsig_windows")
    assert g.count == 4
    for i in range(g.count):
        k = "w{:02d}".format(i)
        x = g.t(k + "_in_x")
        t = g.t(k + "_in_t").to(DEV) if g.has(k + "_in_t") else None
        depth, window = int(g.z[k + "_depth"]), g.f(k + "_window")
        want = g.t(k + "_ref_logsig")
        got = cde.logsig_windows(x.to(DEV), depth, window, t)
        assert got.shape == want.shape
        assert torch.allclose(got.cpu(), want, rtol=1e-9, atol=1e-10), (tuple(x.shape), depth)
        want_v, want_t = g.t(k + "_ref_values"), g.t(k + "_ref_times")
        got_v, got_t = cde.logsignature_windows(x.to(DEV), depth, window, t)
        assert torch.allclose(got_v.cpu(), want_v, rtol=1e-9, atol=1e-10) and torch.allclose(got_t.cpu(), want_t)


def test_with_linear_interpolation():
    """test/test_log_ode.py:8-36 (the reference's only test of this transform), the oracle standing in for signatory."""
    window_length = 4
    torch.manual_seed(2)
    for depth in (1, 2, 3, 4):
        for pieces in (1, 2, 3, 5, 10):
            num_channels = torch.randint(low=1, high=4, size=(1,)).item()
            x_ = [torch.randn(1, num_channels, dtype=torch.float64)]
            logsignatures = []
            for _ in range(pieces):
                x = torch.randn(window_length, num_channels, dtype=torch.float64)
                logsignatures.append(torch.tensor(O.logsignature(torch.cat([x_[-1][-1:], x]).numpy(), depth)))
                x_.append(x)
            x = torch.cat(x_).to(DEV)
            logsig_x = cde.logsig_windows(x, depth, window_length)
            coeffs = cde.linear_interpolation_coeffs(logsig_x)
            X = cde.LinearInterpolation(coeffs)
            point = 0.5
            for logsignature in logsignatures:
                interp_logsignature = X.derivative(torch.tensor(point, device=DEV, dtype=torch.float64))
                assert interp_logsignature.cpu().allclose(logsignature)
                point += 1
