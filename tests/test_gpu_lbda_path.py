"""Regularisation path with per-voxel HRFs, early stopping and the fit-only mode
(``deconv_lbda_path``, ``deconv_lbda_path_fit``, ``pb_deconv_lbda_path_ex_*``).

The path must be exactly a loop of ``deconv(y, t_r, h, lbda=l, ...)`` calls on the batch: same kernel, same
inputs, so the results are compared bit for bit.  Shapes are chosen to reach every deconv kernel family
(pb_fast_registry.cu, gen_fast_instances.py): the group early-stopping kernel (T = 300, K = 20), the
warp-per-voxel tier (T = 600 / K = 20, T = 1200 / K = 28) and the generic kernel (K = 40; T = 1500; FP64 with
T = 3300, whose early-stopping ring spills into the output rows).
"""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import pybold_oracle as orc  # noqa: E402
from pybold_b200.synth import gen_voxels  # noqa: E402

THETAS = (0.8, 1.0, 1.25, 1.5, 1.9)
T_R = {20: 1.0, 28: 0.72, 40: 0.5}          # hrf_dur 20 s -> K taps
# early stop: tol 1e-2 stops these signals after 170-220 iterations (oracle), so nb_iter = 200 gives both
# stopped problems and problems that run to the end
ES = dict(early_stopping=True, tol=1.0e-2, wind=6)


def rel(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return np.max(np.abs(a - b)) / (np.max(np.abs(b)) + 1e-300)


def case(V, T, K, dtype, seed=0):
    t_r = T_R[K]
    y = gen_voxels(V, T, t_r, 20.0, seed0=5000 + seed).astype(dtype)
    h = np.stack([orc.spm_hrf(THETAS[v % len(THETAS)], t_r, 20.0, True)[0] for v in range(V)]).astype(dtype)
    assert h.shape == (V, K)
    x0 = np.random.RandomState(seed).randn(T)
    return y, t_r, h, x0


def n_valid(J):
    return np.sum(~np.isnan(J), axis=-1)


def same(a, b):
    return np.array_equal(a, b, equal_nan=True)


SHAPES = [(300, 20), (600, 20), (1200, 28), (600, 40), (1500, 20)]


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("T,K", SHAPES)
def test_path_per_voxel_hrf_equals_deconv_calls(T, K, dtype):
    import pybold_b200 as pb
    from pybold_b200.bold_signal import deconv_lbda_path
    V, nb = 9, 60
    y, t_r, h, x0 = case(V, T, K, dtype, seed=T + K)
    lbdas = [0.3, 1.0, 3.0]
    x, z, dz, J = deconv_lbda_path(y, t_r, h, lbdas, nb_iter=nb, x0=x0)
    assert z.shape == (3, V, T) and J.shape == (3, V, nb) and z.dtype == dtype
    for i, lb in enumerate(lbdas):
        x1, z1, dz1, J1, _, _ = pb.deconv(y, t_r, h, lbda=lb, x0=x0, early_stopping=False, nb_iter=nb)
        assert same(x[i], x1) and same(z[i], z1) and same(dz[i], dz1) and same(J[i], J1), (i, lb)


def test_path_per_voxel_hrf_vs_oracle_fp64():
    from pybold_b200.bold_signal import deconv_lbda_path
    V, T, K, nb = 5, 300, 20, 80
    y, t_r, h, x0 = case(V, T, K, np.float64, seed=1)
    lbdas = [0.5, 2.0]
    x, z, dz, J = deconv_lbda_path(y, t_r, h, lbdas, nb_iter=nb, x0=x0)
    for l, v in ((0, 3), (1, 4)):
        Lc = 0.9 * orc.spectral_radius_est(orc.HrfIntegOperator(h[v], T), x0)
        xo, zo, wo, Jo, n = orc.deconv_fixed_lbda(y[v], h[v], lbdas[l], lipschitz=Lc, early_stopping=False,
                                                  nb_iter=nb)
        assert rel(dz[l, v], wo) < 1e-9 and rel(z[l, v], zo) < 1e-9 and rel(x[l, v], xo) < 1e-9
        assert rel(J[l, v], Jo) < 1e-9


ES_SHAPES = [(300, 20, np.float32), (300, 20, np.float64), (600, 20, np.float32), (1200, 28, np.float32),
             (600, 40, np.float32), (1500, 20, np.float32), (600, 20, np.float64), (3300, 20, np.float64)]


@pytest.mark.parametrize("T,K,dtype", ES_SHAPES)
def test_path_early_stopping_equals_deconv_calls(T, K, dtype):
    import pybold_b200 as pb
    from pybold_b200.bold_signal import deconv_lbda_path, deconv_lbda_path_fit
    V, nb = (3 if T > 3200 else 9), 200
    y, t_r, h, x0 = case(V, T, K, dtype, seed=7 * T + K)
    lbdas = [0.3, 3.0]
    x, z, dz, J = deconv_lbda_path(y, t_r, h, lbdas, nb_iter=nb, x0=x0, **ES)
    n_path = n_valid(J)
    assert np.all(n_path >= 1) and np.all(n_path <= nb)
    for i, lb in enumerate(lbdas):
        x1, z1, dz1, J1, _, _ = pb.deconv(y, t_r, h, lbda=lb, x0=x0, nb_iter=nb, **ES)
        assert same(x[i], x1) and same(z[i], z1) and same(dz[i], dz1) and same(J[i], J1), (i, lb)
        assert np.array_equal(n_path[i], n_valid(J1))
        assert np.all(np.isnan(J[i][np.arange(nb)[None, :] >= n_path[i][:, None]]))
    R, G, n_fit = deconv_lbda_path_fit(y, t_r, h, lbdas, nb_iter=nb, x0=x0, **ES)
    assert np.array_equal(n_fit, n_path)
    if dtype == np.float64:
        for l, v in ((0, 0), (1, V - 1)):
            Lc = 0.9 * orc.spectral_radius_est(orc.HrfIntegOperator(h[v], T), x0)
            _, _, wo, Jo, n = orc.deconv_fixed_lbda(y[v], h[v], lbdas[l], lipschitz=Lc, nb_iter=nb, **ES)
            assert n_path[l, v] == n, (l, v, n_path[l, v], n)
            assert rel(dz[l, v], wo) < 1e-9 and rel(J[l, v, :n], Jo) < 1e-9


def test_early_stopping_stops_some_problems():
    """The ES tests above are only meaningful if problems do stop before nb_iter."""
    from pybold_b200.bold_signal import deconv_lbda_path_fit
    y, t_r, h, x0 = case(9, 300, 20, np.float32, seed=3)
    _, _, n = deconv_lbda_path_fit(y, t_r, h, [0.3, 3.0], nb_iter=200, x0=x0, **ES)
    assert np.all(n < 200)
    _, _, n = deconv_lbda_path_fit(y, t_r, h, [0.3, 3.0], nb_iter=200, x0=x0)
    assert np.all(n == 200)


@pytest.mark.parametrize("T,K", [(300, 20), (1200, 28), (600, 40)])
def test_shuffling_voxels_shuffles_results(T, K):
    from pybold_b200.bold_signal import deconv_lbda_path
    V = 10
    y, t_r, h, x0 = case(V, T, K, np.float32, seed=11)
    perm = np.random.RandomState(4).permutation(V)
    a = deconv_lbda_path(y, t_r, h, [0.5, 2.0], nb_iter=200, x0=x0, **ES)
    b = deconv_lbda_path(y[perm], t_r, h[perm], [0.5, 2.0], nb_iter=200, x0=x0, **ES)
    for ta, tb in zip(a, b):
        assert same(ta[:, perm], tb)


@pytest.mark.parametrize("dtype,tol", [(np.float64, 1e-12), (np.float32, 1e-5)])
@pytest.mark.parametrize("T,K,es", [(300, 20, True), (600, 20, False), (1200, 28, True), (600, 40, True)])
def test_fit_terms_match_path_solutions(T, K, es, dtype, tol):
    from pybold_b200.bold_signal import deconv_lbda_path, deconv_lbda_path_fit
    V, nb = 8, 200
    y, t_r, h, x0 = case(V, T, K, dtype, seed=13 + T)
    lbdas = [0.2, 1.0, 5.0]
    kw = ES if es else {}
    x, z, dz, J = deconv_lbda_path(y, t_r, h, lbdas, nb_iter=nb, x0=x0, **kw)
    R, G, n = deconv_lbda_path_fit(y, t_r, h, lbdas, nb_iter=nb, x0=x0, **kw)
    assert R.shape == G.shape == n.shape == (3, V) and R.dtype == dtype
    assert np.array_equal(n, n_valid(J))
    R_ref = np.sum((x.astype(np.float64) - y.astype(np.float64)[None]) ** 2, axis=-1)
    G_ref = np.sum(np.abs(dz.astype(np.float64)), axis=-1)
    assert np.max(np.abs(R - R_ref) / R_ref) < tol
    assert np.max(np.abs(G - G_ref) / G_ref) < tol


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_two_stage_choice_reproduces_path_rows(dtype):
    """The docstring's two-stage use: choose lambda per voxel from R, then solve once at it."""
    import pybold_b200 as pb
    from pybold_b200.bold_signal import deconv_lbda_path, deconv_lbda_path_fit
    from pybold_b200.utils import mad_daub_noise_est
    V, T, K, nb = 12, 300, 20, 200
    y, t_r, h, x0 = case(V, T, K, dtype, seed=21)
    lbdas = np.geomspace(0.05, 20.0, 8)
    R, G, n_it = deconv_lbda_path_fit(y, t_r, h, lbdas, nb_iter=nb, x0=x0, **ES)
    sigma = mad_daub_noise_est(y)
    best = np.argmin(np.abs(R - y.shape[1] * sigma ** 2), axis=0)
    lbda_v = np.asarray(lbdas)[best]
    x1, z1, dz1, J1, _, _ = pb.deconv(y, t_r, h, lbda=lbda_v, nb_iter=nb, x0=x0, **ES)
    x, z, dz, J = deconv_lbda_path(y, t_r, h, lbdas, nb_iter=nb, x0=x0, **ES)
    v = np.arange(V)
    assert same(x[best, v], x1) and same(z[best, v], z1) and same(dz[best, v], dz1) and same(J[best, v], J1)


def test_fit_memory_stays_within_scratch_bound():
    """64 lambdas x 50 000 voxels x 600 scans: 23 GB of solutions, never held at once."""
    from pybold_b200.bold_signal import FIT_SCRATCH_BYTES, deconv_lbda_path_fit
    V, T, n_l = 50000, 600, 64
    g = torch.Generator(device="cuda").manual_seed(0)
    y = torch.randn((V, T), device="cuda", dtype=torch.float32, generator=g)
    h = torch.as_tensor(orc.spm_hrf(1.0, 1.0, 20.0, True)[0], device="cuda", dtype=torch.float32)
    lbdas = np.geomspace(0.1, 10.0, n_l)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    R, G, n = deconv_lbda_path_fit(y, 1.0, h, lbdas, nb_iter=5, x0=np.random.RandomState(0).randn(T))
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    summaries = 3 * n_l * V * 4
    assert R.shape == (n_l, V) and bool(torch.all(n == 5))
    assert 3 * n_l * V * T * 4 > 20e9
    assert peak <= FIT_SCRATCH_BYTES + 2 * summaries + (64 << 20), peak


def test_hrf_with_wrong_row_count_raises():
    from pybold_b200.bold_signal import deconv_lbda_path, deconv_lbda_path_fit
    y, t_r, h, x0 = case(6, 300, 20, np.float32)
    for fn in (deconv_lbda_path, deconv_lbda_path_fit):
        with pytest.raises(ValueError):
            fn(y, t_r, h[:4], [1.0], nb_iter=5, x0=x0)
        with pytest.raises(ValueError):
            fn(y, t_r, h[None], [1.0], nb_iter=5, x0=x0)
