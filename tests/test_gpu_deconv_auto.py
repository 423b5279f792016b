"""``deconv(lbda=None)`` in one launch: ``deconv_auto_batch`` / ``pb_deconv_auto_*`` (csrc/pb_noise_loop.cuh).

Every voxel runs the noise-constrained outer loop of pybold/bold_signal.py:99-214 inside the deconv kernels.
Shapes reach every kernel family the picker serves (pb_fast_registry.cu): the group early-stopping kernel
(T = 300, K = 20), the warp-per-voxel tier (T = 600 / K = 20) and the generic kernel (T = 1200 / K = 28 and
K = 40 in FP64, T = 1500; FP64 T = 3300, whose early-stopping ring spills into the output rows).
"""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import pybold_oracle as orc  # noqa: E402
from pybold_b200.synth import gen_voxels  # noqa: E402

THETAS = (0.8, 1.0, 1.25, 1.5, 1.9)
T_R = {20: 1.0, 28: 0.72, 40: 0.5}          # hrf_dur 20 s -> K taps
SHAPES = [(300, 20), (600, 20), (1200, 28), (600, 40), (1500, 20), (3300, 20)]
# tol = 0.1 with nb_iter = 10 outer iterations: the alpha-window stop ends some of these voxels before the last
# outer iteration and not others (oracle: outer counts 7 ... 10); the inner passes stop on the same tol
NB, NB_SUB, WIND, TOL = 10, 30, 4, 0.1
# FP32 against FP64 on the same cases: 10x the largest difference measured on a B200 at 1000 W, 9.9e-6 (DESIGN.md
# section 4.1)
FP32_GATE = 1e-4


def rel(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return np.max(np.abs(a - b)) / (np.max(np.abs(b)) + 1e-300)


def case(V, T, K, seed=0):
    """y [V, T], per-voxel taps [V, K], per-voxel sigma [V] (the db3 MAD estimate), Lipschitz constants [V]."""
    t_r = T_R[K]
    y = gen_voxels(V, T, t_r, 20.0, seed0=7000 + seed)
    h = np.stack([orc.spm_hrf(THETAS[v % len(THETAS)], t_r, 20.0, True)[0] for v in range(V)])
    x0 = np.random.RandomState(seed).randn(T)
    L = np.array([0.9 * orc.spectral_radius_est(orc.HrfIntegOperator(h[v], T), x0) for v in range(V)])
    sigma = np.array([orc.mad_daub_noise_est(v) for v in y])
    return y, h, sigma, L


def run(y, h, sigma, L, dtype, es=True, nb=NB):
    from pybold_b200.bold_signal import deconv_auto_batch
    dev = lambda a: torch.as_tensor(np.ascontiguousarray(a), dtype=dtype, device="cuda")  # noqa: E731
    out = deconv_auto_batch(dev(y), dev(h), dev(sigma), dev(L), nb_iter=nb, nb_sub_iter=NB_SUB,
                            early_stopping=es, tol=TOL, wind=WIND)
    return {k: v.cpu().numpy() for k, v in out.items()}


@pytest.mark.parametrize("es", [True, False])
@pytest.mark.parametrize("T,K", SHAPES)
def test_fp64_vs_oracle(T, K, es):
    V = 3
    y, h, sigma, L = case(V, T, K, seed=T + K)
    o = run(y, h, sigma, L, torch.float64, es)
    counts = []
    for v in range(V):
        xo, zo, wo, Jo, Ro, Go, lo = orc.deconv_auto_lbda(y[v], h[v], sigma[v], lipschitz=L[v], early_stopping=es,
                                                          tol=TOL, wind=WIND, nb_iter=NB, nb_sub_iter=NB_SUB)
        n = len(Jo)
        counts.append(n)
        assert o["n_outer"][v] == n, (v, o["n_outer"][v], n)
        assert rel(o["x"][v], xo) < 1e-9 and rel(o["z"][v], zo) < 1e-9 and rel(o["diff_z"][v], wo) < 1e-9, v
        assert rel(o["J"][v, :n], Jo) < 1e-9 and rel(o["R"][v, :n], Ro) < 1e-9 and rel(o["G"][v, :n], Go) < 1e-9
        assert abs(o["lbda"][v] / lo - 1) < 1e-9, v
        assert np.all(np.isnan(o["J"][v, n:])) and np.all(np.isnan(o["R"][v, n:])) and np.all(np.isnan(o["G"][v, n:]))
    if not es:
        assert counts == [NB] * V


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("T,K", [(300, 20), (600, 20), (1500, 20)])
def test_batch_equals_single_and_permutation(T, K, dtype):
    """A voxel's results do not depend on the batch around it: per-voxel sigma and hrf [V, K], bit for bit."""
    V = 7
    y, h, sigma, L = case(V, T, K, seed=2 * T + K)
    sigma = sigma * np.linspace(0.8, 1.2, V)
    a = run(y, h, sigma, L, dtype)
    assert len(set(a["n_outer"].tolist())) > 1
    for v in (0, 3, V - 1):
        b = run(y[v:v + 1], h[v:v + 1], sigma[v:v + 1], L[v:v + 1], dtype)
        for k in a:
            assert np.array_equal(a[k][v], b[k][0], equal_nan=True), (v, k)
    perm = np.random.RandomState(T).permutation(V)
    c = run(y[perm], h[perm], sigma[perm], L[perm], dtype)
    for k in a:
        assert np.array_equal(a[k][perm], c[k], equal_nan=True), k


@pytest.mark.parametrize("T,K", [(300, 20), (600, 20), (1200, 28), (1500, 20)])
def test_fp32_vs_fp64(T, K):
    V = 6
    y, h, sigma, L = case(V, T, K, seed=3 * T + K)
    a = run(y, h, sigma, L, torch.float64, nb=6)
    b = run(y, h, sigma, L, torch.float32, nb=6)
    err = max(rel(b[k][v, :a["n_outer"][v]], a[k][v, :a["n_outer"][v]]) if k in ("J", "R", "G")
              else rel(b[k][v], a[k][v]) for v in range(V) for k in ("x", "z", "diff_z", "J", "R", "G"))
    print("fp32 vs fp64, T = %d, K = %d: %.2e" % (T, K, err))
    assert np.array_equal(a["n_outer"], b["n_outer"])
    assert err < FP32_GATE


def test_c_entry_nan_tails():
    """J / R / G rows are complete from the C entry itself: NaN past each voxel's outer count."""
    from pybold_b200 import _lib
    V, T, K = 5, 300, 20
    y, h, sigma, L = case(V, T, K, seed=11)
    d = lambda a: torch.as_tensor(np.ascontiguousarray(a), device="cuda")  # noqa: E731
    yd, hd, sd, Ld = d(y), d(h), d(sigma), d(L)
    J, R, G = (torch.zeros((V, 40), dtype=torch.float64, device="cuda") for _ in range(3))
    x, z, dz = (torch.empty((V, T), dtype=torch.float64, device="cuda") for _ in range(3))
    lb = torch.empty(V, dtype=torch.float64, device="cuda")
    n = torch.full((V,), -1, dtype=torch.int32, device="cuda")
    rc = _lib.lib.pb_deconv_auto_f64(yd.data_ptr(), hd.data_ptr(), K, Ld.data_ptr(), 1, sd.data_ptr(), 1, 40, NB_SUB,
                                     1, WIND, TOL, x.data_ptr(), z.data_ptr(), dz.data_ptr(), J.data_ptr(),
                                     R.data_ptr(), G.data_ptr(), lb.data_ptr(), n.data_ptr(), V, T, K, None)
    assert rc == 0
    torch.cuda.synchronize()
    n = n.cpu().numpy()
    assert np.all((n >= WIND + 2) & (n < 40)), n
    for t in (J, R, G):
        t = t.cpu().numpy()
        for v in range(V):
            assert np.all(np.isfinite(t[v, :n[v]])) and np.all(np.isnan(t[v, n[v]:])), v


def test_device_inputs_no_host_sync():
    from pybold_b200.bold_signal import deconv_auto_batch
    V, T, K = 64, 300, 20
    y, h, sigma, L = case(V, T, K, seed=5)
    d = lambda a: torch.as_tensor(np.ascontiguousarray(a), dtype=torch.float32, device="cuda")  # noqa: E731
    yd, hd, sd, Ld = d(y), d(h), d(sigma), d(L)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        out = deconv_auto_batch(yd, hd, sd, Ld, nb_iter=NB, nb_sub_iter=NB_SUB, tol=TOL, wind=WIND)
    finally:
        torch.cuda.set_sync_debug_mode("default")
    assert out["x"].shape == (V, T) and out["J"].shape == (V, NB)
    assert bool(torch.all(out["n_outer"] >= 1))


def test_error_codes():
    from pybold_b200 import _lib
    from pybold_b200.bold_signal import deconv_auto_batch
    V, T, K = 3, 300, 20
    y, h, sigma, L = case(V, T, K, seed=6)
    d = lambda a: torch.as_tensor(np.ascontiguousarray(a), device="cuda")  # noqa: E731
    yd, hd, sd, Ld = d(y), d(h), d(sigma), d(L)
    x, z, dz = (torch.empty((V, T), dtype=torch.float64, device="cuda") for _ in range(3))

    def call(sigma_stride=1, nb_sub_iter=NB_SUB):
        return _lib.lib.pb_deconv_auto_f64(yd.data_ptr(), hd.data_ptr(), K, Ld.data_ptr(), 1, sd.data_ptr(),
                                           sigma_stride, NB, nb_sub_iter, 1, WIND, TOL, x.data_ptr(), z.data_ptr(),
                                           dz.data_ptr(), None, None, None, None, None, V, T, K, None)
    assert call() == _lib.PB_OK
    assert call(sigma_stride=-1) == _lib.PB_ERR_INVALID_ARG
    assert call(nb_sub_iter=_lib.lib.pb_max_iter() + 1) == _lib.PB_ERR_UNSUPPORTED
    torch.cuda.synchronize()
    with pytest.raises(ValueError):
        deconv_auto_batch(yd, hd[:2], sd, Ld)                 # [V', K] taps with V' != V
    with pytest.raises(ValueError):
        deconv_auto_batch(yd, hd, sd[:2], Ld)                 # sigma neither a scalar nor [V]
