"""CPU tests of the respaced (DDIM) schedules: the C ABI's host-only builder against the reference bit for bit, the
special rows, argument validation of the new entry points without a device, and an exact fp64 round trip of
inversion followed by deterministic sampling."""
import ctypes as C

import numpy as np
import pytest
import torch

import oracle
from ddim_reference import constant_eps_params, ddim_invert, ddim_sample, ddim_schedule, ddim_timesteps


@pytest.mark.parametrize("inverse", [False, True])
@pytest.mark.parametrize("eta", [0.0, 0.5, 1.0])
@pytest.mark.parametrize("S", [1, 7, 50, 999, 1000])
def test_library_schedule_equals_reference(pkg, S, eta, inverse):
    ts, coef = pkg.ddim_schedule(S, eta, inverse=inverse)
    rts, rcoef = ddim_schedule(S, eta, inverse=inverse)
    assert ts.dtype == np.int32 and coef.dtype == np.float32 and coef.shape == (S, 8)
    assert np.array_equal(ts, rts)
    assert np.array_equal(coef.view(np.uint32), rcoef.view(np.uint32))
    assert np.array_equal(np.sort(ts), ddim_timesteps(S)) and (np.diff(ts) > 0 if inverse else np.diff(ts) < 0).all()


def _ulp_distance(a, b):
    return np.abs(a.astype(np.float32).view(np.int32).astype(np.int64) - b.astype(np.float32).view(np.int32).astype(np.int64))


def test_full_length_eta_one_is_the_ddpm_posterior(pkg):
    ts, coef = pkg.ddim_schedule(1000, 1.0)
    assert np.array_equal(ts, np.arange(999, -1, -1))
    d = oracle.ddpm_schedule()
    for j, k in enumerate(("sra", "srm1", "c1", "c2")):
        assert _ulp_distance(coef[:, j], d[k][ts]).max() <= 1, k
    assert _ulp_distance(coef[:, 5], d["sigma"][ts]).max() <= 1
    assert (coef[:, 4] == 0).all() and (coef[:, 6] == 1).all()


@pytest.mark.parametrize("S", [1, 7, 50, 1000])
def test_boundary_rows(pkg, S):
    for eta in (0.0, 1.0):
        _, coef = pkg.ddim_schedule(S, eta)
        assert coef[-1, 2] == 1 and coef[-1, 3] == 0 and coef[-1, 5] == 0          # last sampling step returns x0
        if eta == 0:
            assert (coef[:, 5] == 0).all()
    _, inv = pkg.ddim_schedule(S, 0.0, inverse=True)
    assert inv[0, 0] == 1 and inv[0, 1] == 0                                      # the first inversion step starts from x0
    assert (inv[:, 3] == 0).all() and (inv[:, 5] == 0).all() and np.isinf(inv[:, 6]).all() and (inv[:, 4] > 0).all()


def test_argument_validation_without_device(pkg):
    lib = pkg.load_library()
    ts = np.zeros(1000, np.int32)
    coef = np.zeros((1000, 8), np.float32)
    for steps, eta in ((0, 0.0), (1001, 0.0), (-3, 0.5), (10, -0.1), (10, 1.5), (10, float("nan")), (10, float("inf"))):
        for inverse in (0, 1):
            assert lib.sdfb_ddim_schedule(steps, eta, inverse, ts.ctypes.data, coef.ctypes.data) == -1, (steps, eta)
    assert lib.sdfb_ddim_schedule(10, 0.0, 0, None, coef.ctypes.data) == -1
    assert lib.sdfb_ddim_schedule(10, 0.0, 0, ts.ctypes.data, None) == -1
    assert lib.sdfb_ddim_schedule(10, 0.0, 0, ts.ctypes.data, coef.ctypes.data) == 0
    x = C.c_void_p(16)      # never dereferenced: every call below is refused before it touches a device
    assert lib.sdfb_ddpm_sample_ddim(None, x, None, 4, 10, 0.0, 0, None) == -1
    assert lib.sdfb_ddpm_sample_ddim_philox(None, x, 0, 0, 4, 10, 0.0, 1, 0, None) == -1
    assert lib.sdfb_ddpm_invert_ddim(None, x, 4, 10, 0, None) == -1
    with pytest.raises(pkg.SdfbError):
        pkg.ddim_schedule(0, 0.0)
    with pytest.raises(pkg.SdfbError):
        pkg.ddim_schedule(50, 2.0)


@pytest.mark.parametrize("S", [10, 100, 1000])
def test_fp64_round_trip_with_a_constant_noise_prediction(S):
    """eps_hat is the same constant everywhere, so every state of the inversion lies on the line through x0 and that
    constant, x0-hat is x0 at every step (|x0| < 0.5: the clamp never engages), and deterministic sampling walks the
    line back: exact up to fp64 rounding."""
    params = constant_eps_params()
    x0 = np.random.RandomState(S).uniform(-0.5, 0.5, (6, 256))
    x_T = ddim_invert(x0, S, params=params, dtype=torch.float64)
    assert np.abs(x_T - x0).max() > 0.1
    back = ddim_sample(6, x_T, None, S, 0.0, params=params, dtype=torch.float64)
    assert np.abs(back - x0).max() < 1e-12
