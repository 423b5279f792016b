"""Scan censoring for deconv, deconv(lbda=None) and the lambda path (pybold_b200/censor.py).

Censored calls run on the CTA-per-problem rows (``fast_deconvc_kernel<..., CENSOR = true>``) wherever one fits, else
on the generic kernel (``generic_deconv_kernel<..., CENSOR = true>``); ``pb_deconv_censored_variant`` reports which.
The float64 reference is tests/censor_reference.py, itself tied to the pinned oracle bit for bit when nothing is
censored (tests/test_censor_reference.py).
"""
import ctypes

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle import pybold_oracle as orc  # noqa: E402
from tests import censor_reference as cref  # noqa: E402

GENERIC, CTA = 0, 3
T_R = {20: 1.0, 28: 0.72, 40: 0.5, 63: 0.32}          # hrf_dur 20 s -> K taps
ES = dict(early_stopping=True, tol=1.0e-2, wind=6)


def rel(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return np.max(np.abs(a - b)) / (np.max(np.abs(b)) + 1e-300)


def cvariant(T, K, f64=False, nb_iter=200, es=False, wind=6, auto=False):
    from pybold_b200 import _lib
    fam = ctypes.c_int(-1)
    vid = _lib.lib.pb_deconv_censored_variant(T, K, int(f64), nb_iter, int(es), wind, int(auto), ctypes.byref(fam))
    assert vid >= 0, (T, K, vid)
    return vid, fam.value


def mask(T, seed, frac=0.1):
    """About `frac` of the scans censored in runs of 1-5, plus the first and the last scan."""
    rs = np.random.RandomState(seed)
    m = np.zeros(T, dtype=np.uint8)
    m[0] = m[-1] = 1
    while m.mean() < frac:
        a = rs.randint(0, T)
        m[a:a + rs.randint(1, 6)] = 1
    return m


def signal(T, K, seed):
    from pybold_b200.synth import gen_voxels
    t_r = T_R[K]
    y = gen_voxels(1, T, t_r, 20.0, seed0=7000 + seed)[0]
    h = orc.spm_hrf(1.0, t_r, 20.0, True)[0]
    assert h.shape == (K,)
    return y, h


def dev(a, dtype):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=dtype, device="cuda")


def batch(y, h, lbda, L, dtype, nb_iter, censor, **kw):
    from pybold_b200.bold_signal import deconv_batch
    kw = {"early_stopping": False, **kw}
    x, z, dz, J, n = deconv_batch(dev(y, dtype), dev(h, dtype), dev(lbda, dtype), dev(L, dtype), None,
                                  nb_iter=nb_iter, censor=censor, **kw)
    return tuple(t.cpu().numpy() for t in (x, z, dz, J, n))


# ---- routing --------------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_every_fp32_shape_runs_on_a_cta_row():
    Ts = sorted(set(range(1, 4097, 13)) | {1, 2, 4, 100, 128, 129, 180, 181, 256, 1280, 1281, 4095, 4096})
    for m in (dict(), dict(es=True, wind=6), dict(auto=True)):
        for T in Ts:
            for K in (1, 8, 20, 21, 28, 29, 32, 33, 40, 41, 63, 64):
                assert cvariant(T, K, **m)[1] == CTA, (T, K, m)


@pytest.mark.gpu
def test_fp64_rows_and_query_errors():
    from pybold_b200 import _lib
    assert cvariant(1200, 28, f64=True) == (64020028, CTA)
    assert cvariant(600, 20, f64=True) == (32020020, CTA)
    assert cvariant(300, 20, f64=True)[1] == GENERIC
    assert cvariant(3000, 28, f64=True)[1] == GENERIC
    fam = ctypes.c_int()
    q = _lib.lib.pb_deconv_censored_variant
    assert q(0, 20, 0, 200, 0, 6, 0, ctypes.byref(fam)) == _lib.PB_ERR_INVALID_ARG
    assert q(300, 20, 0, 200, 0, 6, 0, None) == _lib.PB_ERR_INVALID_ARG
    assert q(4097, 20, 0, 200, 0, 6, 0, ctypes.byref(fam)) == _lib.PB_ERR_UNSUPPORTED


# ---- FP64 against the float64 reference -----------------------------------------------------------------------

SHAPES = [(T, K) for T in (300, 600, 1200, 3000) for K in (20, 28, 40)]


@pytest.mark.gpu
def test_fp64_cases_reach_both_cta_rows_and_the_generic_kernel():
    ids = {cvariant(T, K, f64=True, nb_iter=150, es=es)[0] for T, K in SHAPES for es in (False, True)}
    assert {64020028, 32020020, 0} <= ids, ids


@pytest.mark.gpu
@pytest.mark.parametrize("T,K", SHAPES)
@pytest.mark.parametrize("es", [False, True])
def test_fp64_fixed_lbda_matches_reference(T, K, es):
    import pybold_b200 as pb
    y, h = signal(T, K, T + K)
    cm = mask(T, T * K)
    y = np.where(cm != 0, np.nan, y)                    # censored frames stored as NaN
    x0 = np.random.RandomState(T).randn(T)
    kw = ES if es else dict(early_stopping=False)
    x, z, dz, J, _, _ = pb.deconv(y, T_R[K], h, lbda=0.5, nb_iter=150, x0=x0, censor=cm, **kw)
    xo, zo, wo, Jo, no = cref.deconv_fixed_lbda(y, h, 0.5, x0_power=x0, nb_iter=150, censor=cm, **kw)
    assert len(J) == no
    for a, b in ((x, xo), (z, zo), (dz, wo), (J, Jo)):
        assert rel(a, b) < 1e-9, (rel(a, b), T, K, es)


@pytest.mark.gpu
@pytest.mark.parametrize("T,K", [(300, 20), (600, 20), (1200, 28), (1200, 40), (3000, 28)])
def test_fp64_auto_lbda_matches_reference(T, K):
    from pybold_b200.bold_signal import deconv_auto_batch
    y, h = signal(T, K, 3 * T + K)
    cm = mask(T, T + 5 * K)
    y = np.where(cm != 0, np.nan, y)
    L = 0.9 * cref.spectral_radius_est(h, np.random.RandomState(T + 1).randn(T), cm)
    sigma = 0.8 * cref.mad_daub_noise_est(y, cm)
    out = deconv_auto_batch(dev(y[None], torch.float64), dev(h, torch.float64), sigma, L, nb_iter=12,
                            nb_sub_iter=60, early_stopping=True, tol=1e-3, wind=4, censor=cm)
    out = {k: v.cpu().numpy() for k, v in out.items()}
    xo, zo, wo, Jo, Ro, Go, lo = cref.deconv_auto_lbda(y, h, sigma, lipschitz=L, nb_iter=12, nb_sub_iter=60,
                                                       censor=cm, early_stopping=True, tol=1e-3, wind=4)
    n = int(out["n_outer"][0])
    assert n == len(Jo)
    assert rel(out["lbda"][0], lo) < 1e-9
    for k, b in (("x", xo), ("z", zo), ("diff_z", wo)):
        assert rel(out[k][0], b) < 1e-9, (k, rel(out[k][0], b), T, K)
    for k, b in (("J", Jo), ("R", Ro), ("G", Go)):
        assert rel(out[k][0, :n], b) < 1e-9, (k, rel(out[k][0, :n], b), T, K)


# ---- FP32 against FP64 on every CTA row the censored picker chooses -----------------------------------------------

def _rows():
    """{variant id: (shortest T, longest T, K)} of the censored picker over T <= 4096 for four tap counts."""
    rows = {}
    for K in (20, 28, 40, 63):
        for T in range(1, 4097):
            vid, fam = cvariant(T, K, nb_iter=100)
            assert fam == CTA
            lo, hi, _ = rows.get((vid, K), (T, T, K))
            rows[(vid, K)] = (min(lo, T), max(hi, T), K)
    return rows


@pytest.mark.gpu
def test_fp32_matches_fp64_on_every_censored_cta_row():
    worst = 0.0
    for (vid, K), (t_lo, t_hi, _) in sorted(_rows().items()):
        for T in sorted({t_lo, t_hi}):
            if T < 16:
                continue
            from pybold_b200.synth import gen_voxels
            rs = np.random.RandomState(T * 7 + K)
            y = gen_voxels(2, T, T_R[K], 20.0, seed0=9000 + T) if T >= 64 else rs.randn(2, T)
            h = np.stack([orc.spm_hrf(1.0, T_R[K], 20.0, True)[0]] * 2)
            cm = np.stack([mask(T, T + v) for v in range(2)])
            L = np.array([0.9 * cref.spectral_radius_est(h[v], rs.randn(T), cm[v]) for v in range(2)])
            x32 = batch(y, h, np.array([0.3, 0.6]), L, torch.float32, 100, dev(cm, torch.uint8))
            x64 = batch(y, h, np.array([0.3, 0.6]), L, torch.float64, 100, dev(cm, torch.uint8))
            for a, b in zip(x32[:4], x64[:4]):
                e = rel(a, b)
                worst = max(worst, e)
                assert e < 1e-4, (vid, K, T, e)
    print("worst FP32 / FP64 relative difference: %.2e" % worst)


# ---- bit-for-bit checks ---------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("T,K,dtype", [(1500, 28, torch.float32), (400, 40, torch.float32),
                                       (1200, 28, torch.float64), (300, 20, torch.float64)])
def test_values_at_censored_scans_are_ignored(T, K, dtype):
    rs = np.random.RandomState(T)
    y = rs.randn(3, T)
    h = orc.spm_hrf(1.0, T_R[K], 20.0, True)[0]
    cm = np.stack([mask(T, T + v) for v in range(3)])
    L = np.full(3, 0.9 * cref.spectral_radius_est(h, rs.randn(T), cm[0]))
    ref = batch(np.where(cm != 0, 0.0, y), h, 0.4, L, dtype, 120, cm, **ES)
    for bad in (np.nan, np.inf, 1e30):
        out = batch(np.where(cm != 0, bad, y), h, 0.4, L, dtype, 120, cm, **ES)
        for a, b in zip(out, ref):
            assert np.array_equal(a, b, equal_nan=True), bad


@pytest.mark.gpu
@pytest.mark.parametrize("T,K", [(1500, 20), (3000, 28), (600, 40), (2000, 63)])
@pytest.mark.parametrize("es", [False, True])
def test_all_zero_mask_equals_uncensored_call(T, K, es):
    from pybold_b200 import _lib
    fam = ctypes.c_int()
    assert _lib.lib.pb_deconv_variant(T, K, 0, 150, int(es), 6, 0, ctypes.byref(fam)) == cvariant(T, K, nb_iter=150,
                                                                                                 es=es)[0]
    rs = np.random.RandomState(T + K)
    y = rs.randn(4, T)
    h = orc.spm_hrf(1.0, T_R[K], 20.0, True)[0]
    L = np.full(4, 0.9 * orc.spectral_radius_est(orc.HrfIntegOperator(h, T), rs.randn(T)))
    kw = ES if es else {}
    a = batch(y, h, 0.4, L, torch.float32, 150, np.zeros(T, np.uint8), **kw)
    b = batch(y, h, 0.4, L, torch.float32, 150, None, **kw)
    for u, v in zip(a, b):
        assert np.array_equal(u, v, equal_nan=True)


@pytest.mark.gpu
def test_per_voxel_masks_on_the_work_queue():
    """A batch larger than one grid wave, early stopping on the work queue, one mask per voxel: single-voxel calls and
    a permuted batch give the same rows bit for bit."""
    T, K, V = 1500, 28, 1300
    rs = np.random.RandomState(5)
    y = rs.randn(V, T)
    h = orc.spm_hrf(1.0, T_R[K], 20.0, True)[0]
    cm = np.stack([mask(T, v, frac=0.05 + 0.1 * (v % 3)) for v in range(V)])
    lb = 0.2 + rs.rand(V)
    L = np.full(V, 0.9 * orc.spectral_radius_est(orc.HrfIntegOperator(h, T), rs.randn(T)))
    full = batch(y, h, lb, L, torch.float32, 150, cm, **ES)
    assert len(set(full[4].tolist())) > 1
    for v in (0, 1, 700, V - 1):
        one = batch(y[v:v + 1], h, lb[v:v + 1], L[v:v + 1], torch.float32, 150, cm[v:v + 1], **ES)
        for a, b in zip(one, full):
            assert np.array_equal(a[0], b[v], equal_nan=True), v
    perm = rs.permutation(V)
    pm = batch(y[perm], h, lb[perm], L[perm], torch.float32, 150, cm[perm], **ES)
    for a, b in zip(pm, full):
        assert np.array_equal(a, b[perm], equal_nan=True)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_path_rows_equal_censored_deconv_calls(dtype):
    from pybold_b200 import bold_signal as pb
    T, K, V = 1200, 28, 5
    rs = np.random.RandomState(11)
    y = rs.randn(V, T)
    h = orc.spm_hrf(1.0, T_R[K], 20.0, True)[0]
    cm = np.stack([mask(T, 40 + v) for v in range(V)])
    x0 = rs.randn(T)
    lbdas = [0.2, 0.5, 1.0]
    np_dtype = np.float32 if dtype == torch.float32 else np.float64
    x, z, dz, J = pb.deconv_lbda_path(y.astype(np_dtype), T_R[K], h.astype(np_dtype), lbdas, nb_iter=120, x0=x0,
                                      censor=cm, **ES)
    R, G, n = pb.deconv_lbda_path_fit(y.astype(np_dtype), T_R[K], h.astype(np_dtype), lbdas, nb_iter=120, x0=x0,
                                      censor=cm, **ES)
    for li, lb in enumerate(lbdas):
        xs, zs, ws, Js, _, _ = pb.deconv(y.astype(np_dtype), T_R[K], h.astype(np_dtype), lbda=lb, nb_iter=120, x0=x0,
                                         censor=cm, **ES)
        assert np.array_equal(x[li], xs) and np.array_equal(z[li], zs) and np.array_equal(dz[li], ws)
        assert np.array_equal(J[li], Js, equal_nan=True)
        Rv = np.sum(np.where(cm != 0, 0.0, xs.astype(np.float64) - y) ** 2, axis=1)
        assert rel(R[li], Rv) < (1e-4 if dtype == torch.float32 else 1e-10)
        assert rel(G[li], np.abs(ws.astype(np.float64)).sum(axis=1)) < (1e-4 if dtype == torch.float32 else 1e-10)


# ---- sigma, host synchronisation, errors ------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("T", [9, 64, 301, 1200])
def test_censored_mad_equals_numpy_median(T):
    from pybold_b200.censor import mad_daub_noise_est_censored
    rs = np.random.RandomState(T)
    y = rs.randn(4, T)
    cm = np.stack([mask(T, T + v, frac=0.2) for v in range(4)])
    got = mad_daub_noise_est_censored(dev(y, torch.float64), dev(cm, torch.uint8), T).cpu().numpy()
    ref = [orc.mad(cref.kept_detail_coefficients(y[v], cm[v])) for v in range(4)]
    # the coefficients are formed with fused multiply-adds on the device: equal to NumPy's up to rounding
    np.testing.assert_allclose(got, np.array(ref), rtol=1e-12, atol=0)


@pytest.mark.gpu
def test_auto_batch_with_device_censor_makes_no_host_sync():
    from pybold_b200.bold_signal import deconv_auto_batch
    T, K, V = 1200, 28, 8
    y = dev(np.random.RandomState(1).randn(V, T), torch.float32)
    h = dev(orc.spm_hrf(1.0, T_R[K], 20.0, True)[0], torch.float32)
    cm = dev(np.stack([mask(T, v) for v in range(V)]), torch.uint8)
    sigma = torch.full((V,), 0.9, dtype=torch.float32, device="cuda")
    L = torch.full((V,), 0.9 * cref.spectral_radius_est(orc.spm_hrf(1.0, T_R[K], 20.0, True)[0],
                                                        np.random.RandomState(2).randn(T), np.ones(T) * 0),
                   dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        out = deconv_auto_batch(y, h, sigma, L, nb_iter=5, nb_sub_iter=20, censor=cm)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert torch.isfinite(out["x"]).all()


@pytest.mark.gpu
def test_errors():
    import pybold_b200 as pb
    from pybold_b200 import _lib
    T, K = 300, 20
    y, h = signal(T, K, 1)
    with pytest.raises(ValueError):
        pb.deconv(y, 1.0, h, lbda=0.5, nb_iter=10, censor=np.zeros(T - 1, np.uint8))
    with pytest.raises(ValueError):
        pb.deconv(np.stack([y, y]), 1.0, h, lbda=0.5, nb_iter=10, censor=np.zeros((3, T), np.uint8))
    with pytest.raises(ValueError):
        pb.deconv(y, 1.0, h, lbda=0.5, nb_iter=10, censor=np.ones(T, np.uint8))
    with pytest.raises(ValueError):
        pb.deconv(np.stack([y, y]), 1.0, h, lbda=0.5, nb_iter=10,
                  censor=np.stack([np.zeros(T, np.uint8), np.ones(T, np.uint8)]))
    alt = np.zeros(T, np.uint8)
    alt[::2] = 1                                        # every detail coefficient reads a censored scan
    with pytest.raises(ValueError, match="sigma"):
        pb.deconv(y, 1.0, h, lbda=None, nb_iter=3, censor=alt)
    # a negative mask stride from C
    yd = dev(y[None], torch.float32)
    o = torch.empty_like(yd)
    J = torch.empty((1, 10), dtype=torch.float32, device="cuda")
    n = torch.empty(1, dtype=torch.int32, device="cuda")
    hd, L, lb = dev(h, torch.float32), dev([5.0], torch.float32), dev([0.5], torch.float32)
    cm = dev(np.zeros(T), torch.uint8)
    rc = _lib.lib.pb_deconv_censored_f32(yd.data_ptr(), hd.data_ptr(), 0, L.data_ptr(), 0, lb.data_ptr(), 0, None,
                                         cm.data_ptr(), -1, 10, 0, 6, 1e-6, o.data_ptr(), o.data_ptr(), o.data_ptr(),
                                         J.data_ptr(), n.data_ptr(), 1, T, K, None)
    assert rc == _lib.PB_ERR_INVALID_ARG
