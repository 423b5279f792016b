"""CPU checks of the float64 censoring reference (tests/censor_reference.py) the GPU censoring tests compare with:
an all-zero mask gives the pinned oracle's outputs bit for bit, x = A w on every scan, the censored Lipschitz constant
is that of the dense A^T M A, and the censored noise level reads only the kept detail coefficients."""
import numpy as np
import pytest

from oracle import pybold_oracle as orc
from tests import censor_reference as cref


def _problem(T=120, K=20, seed=0):
    rs = np.random.RandomState(seed)
    h = orc.spm_hrf(1.0, 1.0, 20.0, True)[0][:K]
    z = np.zeros(T)
    z[20:35] = 1.0
    z[70:80] = -0.5
    y = orc.conv_causal(h, z) + 0.1 * rs.randn(T)
    return y, h, rs.randn(T)


def _mask(T, seed=3):
    m = np.zeros(T, dtype=np.uint8)
    m[0] = m[-1] = 1
    m[np.random.RandomState(seed).choice(T, T // 10, replace=False)] = 1
    return m


@pytest.mark.parametrize("es", [False, True])
def test_all_zero_mask_is_the_oracle_bit_for_bit(es):
    y, h, x0 = _problem()
    zero = np.zeros(len(y), dtype=np.uint8)
    a = cref.deconv_fixed_lbda(y, h, 0.3, x0_power=x0, nb_iter=80, early_stopping=es, tol=1e-3, censor=zero)
    b = orc.deconv_fixed_lbda(y, h, 0.3, x0_power=x0, nb_iter=80, early_stopping=es, tol=1e-3)
    for u, v in zip(a, b):
        assert np.array_equal(u, v)
    a = cref.deconv_auto_lbda(y, h, 0.1, x0_power=x0, nb_iter=6, nb_sub_iter=40, censor=zero)
    b = orc.deconv_auto_lbda(y, h, 0.1, x0_power=x0, nb_iter=6, nb_sub_iter=40)
    for u, v in zip(a, b):
        assert np.array_equal(u, v)
    assert cref.mad_daub_noise_est(y, zero) == orc.mad_daub_noise_est(y)


def test_x_is_the_model_on_every_scan_and_ignores_censored_values():
    y, h, x0 = _problem(seed=1)
    m = _mask(len(y))
    x, z, w, J, n = cref.deconv_fixed_lbda(y, h, 0.3, x0_power=x0, nb_iter=60, censor=m)
    assert np.array_equal(x, orc.conv_causal(h, np.cumsum(w)))
    assert np.abs(x[m != 0]).max() > 0
    for bad in (np.nan, np.inf, 1e30):
        out = cref.deconv_fixed_lbda(np.where(m != 0, bad, y), h, 0.3, x0_power=x0, nb_iter=60, censor=m)
        for u, v in zip(out, (x, z, w, J, n)):
            assert np.array_equal(u, v)


def test_censored_lipschitz_is_the_dense_power_iteration():
    y, h, x0 = _problem(T=90, seed=2)
    T = len(y)
    m = _mask(T)
    A = orc.toeplitz_from_kernel(h, T).dot(np.tril(np.ones((T, T))))
    G = A.T.dot(np.diag(1.0 - m)).dot(A)
    x_old = x0.copy()
    x_new = x_old
    for _ in range(30):
        x_new = G.dot(x_old) / np.linalg.norm(x_old)
        if abs(np.linalg.norm(x_new) - np.linalg.norm(x_old)) < 1e-6:
            break
        x_old = x_new
    dense = np.linalg.norm(x_new)
    assert abs(cref.spectral_radius_est(h, x0, m) - dense) <= 1e-12 * dense
    assert cref.spectral_radius_est(h, x0, m) < orc.spectral_radius_est(orc.HrfIntegOperator(h, T), x0)


def test_censored_noise_level_reads_only_kept_coefficients():
    y, _, _ = _problem(T=64, seed=4)
    m = np.zeros(64, dtype=np.uint8)
    m[30] = 1
    kept = cref.kept_detail_coefficients(y, m)
    full = orc.db3_detail_level1(y)
    # scan 30 is read by the coefficients o with 2 o + 1 - j = 30, j < 6: o = 15, 16, 17
    assert np.array_equal(kept, np.delete(full, [15, 16, 17]))
    y2 = y.copy()
    y2[30] = 1e6
    assert cref.mad_daub_noise_est(y2, m) == cref.mad_daub_noise_est(y, m) == orc.mad(kept)
