"""Deconvolution on the CTA-per-problem kernels (``fast_deconvc_kernel``, csrc/pb_fastc.cuh).

A deconvolution runs on the group rows, else the warp rows, else the CTA rows, else the generic kernel
(pb_fast_registry.cu).  The CTA rows take the long series (T > 1280 scans in FP32) and the short-TR HRFs (K > 32
taps): ``deconv``, ``deconv(lbda=None)``, the lambda path and the masked entry.  ``pb_deconv_variant`` reports the
kernel a call runs on, by the launch's own routing, so that a fall-back to the generic kernel cannot pass unseen.
"""
import ctypes
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle import pybold_oracle as orc  # noqa: E402

GENERIC, GROUP, WARP, CTA = 0, 1, 2, 3
T_R = {20: 1.0, 28: 0.72, 40: 0.5, 63: 0.32}          # hrf_dur 20 s -> K taps
ES = dict(early_stopping=True, tol=1.0e-2, wind=6)     # stops these signals at different iterations below 200
# FP32 against the float64 oracle on every CTA variant the deconv picker chooses (78 cases): the largest error this
# test printed on a B200 at 1000 W was 4.6e-5 (T = 4096 and the 63-tap variants); the gate stays at the 1e-4 of the
# other FP32 tests, below 10x that figure
FP32_GATE = 1e-4


def rel(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return np.max(np.abs(a - b)) / (np.max(np.abs(b)) + 1e-300)


def variant(T, K, f64=False, nb_iter=200, es=False, wind=6, auto=False):
    from pybold_b200 import _lib
    fam = ctypes.c_int(-1)
    vid = _lib.lib.pb_deconv_variant(T, K, int(f64), nb_iter, int(es), wind, int(auto), ctypes.byref(fam))
    assert vid >= 0, (T, K, vid)
    return vid, fam.value


def signals(V, T, K, seed):
    """y [V, T] (block design + noise, or noise for very short series) and SPM taps [V, K] of varied shape."""
    from pybold_b200.synth import gen_voxels
    t_r = T_R[K]
    y = gen_voxels(V, T, t_r, 20.0, seed0=9000 + seed) if T >= 64 else np.random.RandomState(seed).randn(V, T)
    h = np.stack([orc.spm_hrf((0.8, 1.0, 1.3)[v % 3], t_r, 20.0, True)[0] for v in range(V)])
    assert h.shape == (V, K)
    return y, h


def lipschitz(h, T, seed=0):
    x0 = np.random.RandomState(seed).randn(T)
    return np.array([0.9 * orc.spectral_radius_est(orc.HrfIntegOperator(hv, T), x0) for hv in h])


def dev(a, dtype):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=dtype, device="cuda")


def solve(y, h, lbda, L, dtype, nb_iter, w0=None, active=None, **kw):
    from pybold_b200.bold_signal import deconv_batch
    kw = {"early_stopping": False, **kw}
    x, z, dz, J, n = deconv_batch(dev(y, dtype), dev(h, dtype), dev(lbda, dtype), dev(L, dtype),
                                  None if w0 is None else dev(w0, dtype), nb_iter=nb_iter, active=active, **kw)
    return tuple(t.cpu().numpy() for t in (x, z, dz, J, n))


# ---- routing --------------------------------------------------------------------------------------------------

def test_solver_variant_table_unchanged():
    """pb_solver_variant (bd) over T <= 4096, K <= 64: the ids of the build before the deconv CTA kernels."""
    from pybold_b200 import _lib
    ref = np.load(os.path.join(os.path.dirname(__file__), "golden", "solver_variant_ids.npz"))["ids"]
    f = _lib.lib.pb_solver_variant
    ids = np.array([[[f(T, K, d) for K in range(1, 65)] for T in range(1, 4097)] for d in (0, 1)], dtype=np.int32)
    assert np.array_equal(ids, ref), np.argwhere(ids != ref)[:10]


MODES = [dict(), dict(es=True, wind=6), dict(auto=True)]


@pytest.mark.gpu
@pytest.mark.parametrize("f64,t_max", [(False, 1280), (True, 640)])
def test_short_series_stay_on_group_and_warp_kernels(f64, t_max):
    """Every shape a warp variant serves (FP32: T <= 1280, FP64: T <= 640; K <= 32) keeps its group or warp kernel."""
    for T in list(range(1, t_max, 9)) + [t_max]:
        for K in range(1, 33):
            for m in MODES:
                assert variant(T, K, f64=f64, **m)[1] in (GROUP, WARP), (T, K, m)


@pytest.mark.gpu
def test_long_series_and_short_tr_run_on_cta_kernels():
    for m in MODES:
        for T in list(range(1281, 4096, 23)) + [4096]:
            for K in (1, 20, 28, 32, 40, 63, 64):
                assert variant(T, K, **m)[1] == CTA, (T, K, m)
        for T in list(range(1, 4096, 31)) + [4096]:
            for K in range(33, 65):
                assert variant(T, K, **m)[1] == CTA, (T, K, m)
    # the FP64 parity row: two warps of R = 20, 28 taps
    for T in (641, 700, 1000, 1280):
        assert variant(T, 28, f64=True) == (64020028, CTA)
        assert variant(T, 29, f64=True)[1] == GENERIC


@pytest.mark.gpu
def test_variant_query_errors():
    from pybold_b200 import _lib
    fam = ctypes.c_int()
    q = _lib.lib.pb_deconv_variant
    assert q(0, 20, 0, 200, 0, 6, 0, ctypes.byref(fam)) == _lib.PB_ERR_INVALID_ARG
    assert q(300, 20, 0, 0, 0, 6, 0, ctypes.byref(fam)) == _lib.PB_ERR_INVALID_ARG
    assert q(300, 20, 0, 200, 0, 6, 0, None) == _lib.PB_ERR_INVALID_ARG
    assert q(4097, 20, 0, 200, 0, 6, 0, ctypes.byref(fam)) == _lib.PB_ERR_UNSUPPORTED
    assert q(300, 65, 0, 200, 0, 6, 0, ctypes.byref(fam)) == _lib.PB_ERR_UNSUPPORTED


# ---- every CTA variant the picker chooses, FP32 against the float64 oracle -----------------------------------------

def _cta_cases():
    if not torch.cuda.is_available():
        return []
    seen = {}
    for K in (20, 28, 40, 63):
        for T in range(1, 4097):
            vid, fam = variant(T, K)
            if fam == CTA:
                lo, hi = seen.get((vid, K), (T, T))
                seen[(vid, K)] = (min(lo, T), max(hi, T))
    return sorted({(T, K, vid) for (vid, K), ends in seen.items() for T in ends})


@pytest.mark.gpu
def test_cta_variants_cover_the_picker():
    cases = _cta_cases()
    assert len({vid for _, _, vid in cases}) >= 20, cases


@pytest.mark.gpu
@pytest.mark.parametrize("T,K,vid", _cta_cases())
def test_every_cta_variant_fp32_vs_oracle(T, K, vid):
    V, nb = 2, 40
    y, h = signals(V, T, K, seed=T + K)
    L = lipschitz(h, T)
    lbda = np.array([0.5, 2.0])
    assert variant(T, K, nb_iter=nb) == (vid, CTA)
    x, z, dz, J, n = solve(y, h, lbda, L, torch.float32, nb)
    err = 0.0
    for v in range(V):
        xo, zo, wo, Jo, no = orc.deconv_fixed_lbda(y[v], h[v], lbda[v], lipschitz=L[v], early_stopping=False,
                                                   nb_iter=nb)
        assert n[v] == no == nb
        err = max(err, rel(x[v], xo), rel(z[v], zo), rel(dz[v], wo), rel(J[v] / J[v, 0], Jo))
    print("T = %d, K = %d, variant %d: fp32 vs oracle %.2e" % (T, K, vid, err))
    assert err < FP32_GATE


# ---- FP64 through the double CTA row ------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("T", [700, 1280])
def test_fp64_parity_row_vs_oracle(T):
    K, V, nb = 28, 3, 200
    assert variant(T, K, f64=True)[1] == CTA and variant(T, K, f64=True, es=True)[1] == CTA
    assert variant(T, K, f64=True, auto=True)[1] == CTA
    y, h = signals(V, T, K, seed=T)
    L = lipschitz(h, T)
    lbda = np.array([0.3, 1.0, 3.0])
    for kw in (dict(), ES):
        x, z, dz, J, n = solve(y, h, lbda, L, torch.float64, nb, **kw)
        for v in range(V):
            xo, zo, wo, Jo, no = orc.deconv_fixed_lbda(y[v], h[v], lbda[v], lipschitz=L[v], nb_iter=nb,
                                                       **({"early_stopping": False} if not kw else kw))
            assert n[v] == no, (kw, v, n[v], no)
            assert rel(x[v], xo) < 1e-9 and rel(z[v], zo) < 1e-9 and rel(dz[v], wo) < 1e-9
            assert rel(J[v, :no] / J[v, 0], Jo) < 1e-9
    from pybold_b200.bold_signal import deconv_auto_batch
    sigma = np.array([orc.mad_daub_noise_est(v) for v in y])
    o = deconv_auto_batch(dev(y, torch.float64), dev(h, torch.float64), dev(sigma, torch.float64),
                          dev(L, torch.float64), nb_iter=10, nb_sub_iter=30, early_stopping=True, tol=0.1, wind=4)
    o = {k: t.cpu().numpy() for k, t in o.items()}
    for v in range(V):
        xo, zo, wo, Jo, Ro, Go, lo = orc.deconv_auto_lbda(y[v], h[v], sigma[v], lipschitz=L[v], early_stopping=True,
                                                      tol=0.1, wind=4, nb_iter=10, nb_sub_iter=30)
        m = len(Jo)
        assert o["n_outer"][v] == m, (v, o["n_outer"][v], m)
        assert rel(o["x"][v], xo) < 1e-9 and rel(o["z"][v], zo) < 1e-9 and rel(o["diff_z"][v], wo) < 1e-9
        assert rel(o["J"][v, :m], Jo) < 1e-9 and rel(o["R"][v, :m], Ro) < 1e-9 and rel(o["G"][v, :m], Go) < 1e-9
        assert abs(o["lbda"][v] / lo - 1) < 1e-9


# ---- Q5 early stop on the work queue ------------------------------------------------------------------------------

@pytest.mark.gpu
def test_early_stop_counts_match_oracle_fp64():
    T, K, V, nb = 1000, 28, 6, 200
    y, h = signals(V, T, K, seed=3)
    L = lipschitz(h, T)
    lbda = np.geomspace(0.2, 5.0, V)
    _, _, dz, _, n = solve(y, h, lbda, L, torch.float64, nb, **ES)
    counts = []
    for v in range(V):
        _, _, wo, _, no = orc.deconv_fixed_lbda(y[v], h[v], lbda[v], lipschitz=L[v], nb_iter=nb, **ES)
        counts.append(no)
        assert n[v] == no and rel(dz[v], wo) < 1e-9, (v, n[v], no)
    assert len(set(counts)) > 1, counts


@pytest.mark.gpu
@pytest.mark.parametrize("T,K", [(2000, 28), (900, 40), (4096, 63)])
def test_batch_beyond_one_wave_equals_single_and_permutation(T, K):
    """Per-voxel lbda, HRF and warm start; a batch larger than one wave of the persistent grid, so that problems
    come from the work queue: a voxel's results do not depend on the batch around it."""
    vid, fam = variant(T, K, es=True)
    assert fam == CTA
    # one wave holds at most SMs x min(32, 2048 threads / CTA size) CTAs of one problem each, whatever the launch
    # bounds and the shared memory allow
    nt = vid // 1000000
    wave_max = torch.cuda.get_device_properties(0).multi_processor_count * min(32, 2048 // nt)
    V, nb = wave_max + 64, 200
    base_y, base_h = signals(8, T, K, seed=K)
    rs = np.random.RandomState(T)
    pick = rs.randint(0, 8, V)
    y = base_y[pick] * rs.uniform(0.5, 2.0, (V, 1))
    h, L = base_h[pick], lipschitz(base_h, T)[pick]
    lbda = rs.uniform(0.2, 4.0, V)
    w0 = 1e-4 * rs.randn(V, T)
    a = solve(y, h, lbda, L, torch.float32, nb, w0=w0, **ES)
    assert len(set(a[4].tolist())) > 1 and a[4].min() < nb
    for v in (0, V // 2, V - 1):
        b = solve(y[v:v + 1], h[v:v + 1], lbda[v:v + 1], L[v:v + 1], torch.float32, nb, w0=w0[v:v + 1], **ES)
        for ta, tb in zip(a, b):
            assert np.array_equal(ta[v], tb[0], equal_nan=True), v
    perm = rs.permutation(V)
    c = solve(y[perm], h[perm], lbda[perm], L[perm], torch.float32, nb, w0=w0[perm], **ES)
    for ta, tc in zip(a, c):
        assert np.array_equal(ta[perm], tc, equal_nan=True)


# ---- arbitrary taps: tap 0 is not zero ----------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("T,K,dtype,gate", [(2000, 40, torch.float32, FP32_GATE), (1500, 63, torch.float32, FP32_GATE),
                                            (1000, 28, torch.float64, 1e-9)])
def test_random_taps_vs_oracle(T, K, dtype, gate):
    V, nb = 2, 60
    y, _ = signals(V, T, K, seed=5)
    h = np.random.RandomState(K).randn(V, K)
    h[:, 0] = 1.5                                    # a large tap 0
    L = lipschitz(h, T)
    lbda = np.array([0.5, 2.0])
    assert variant(T, K, f64=dtype == torch.float64, nb_iter=nb)[1] == CTA
    x, z, dz, J, n = solve(y, h, lbda, L, dtype, nb)
    for v in range(V):
        xo, zo, wo, Jo, _ = orc.deconv_fixed_lbda(y[v], h[v], lbda[v], lipschitz=L[v], early_stopping=False,
                                                  nb_iter=nb)
        err = max(rel(x[v], xo), rel(z[v], zo), rel(dz[v], wo))
        print("random taps T = %d, K = %d, %s: %.2e" % (T, K, dtype, err))
        assert err < gate


# ---- deconv(lbda=None) ----------------------------------------------------------------------------------------------

AUTO_SHAPES = [(2000, 28), (900, 40), (4096, 63)]


@pytest.mark.gpu
@pytest.mark.parametrize("T,K", AUTO_SHAPES)
def test_auto_fp32_vs_fp64(T, K):
    from pybold_b200.bold_signal import deconv_auto_batch
    V = 4
    y, h = signals(V, T, K, seed=2 * T + K)
    L = lipschitz(h, T)
    sigma = np.array([orc.mad_daub_noise_est(v) for v in y])
    assert variant(T, K, nb_iter=30, es=True, wind=4, auto=True)[1] == CTA

    def run(dtype):
        o = deconv_auto_batch(dev(y, dtype), dev(h, dtype), dev(sigma, dtype), dev(L, dtype), nb_iter=6,
                              nb_sub_iter=30, early_stopping=True, tol=0.1, wind=4)
        return {k: t.cpu().numpy() for k, t in o.items()}
    a, b = run(torch.float64), run(torch.float32)
    assert np.array_equal(a["n_outer"], b["n_outer"])
    err = max(rel(b[k][v, :a["n_outer"][v]], a[k][v, :a["n_outer"][v]]) if k in ("J", "R", "G")
              else rel(b[k][v], a[k][v]) for v in range(V) for k in ("x", "z", "diff_z", "J", "R", "G"))
    print("deconv(lbda=None) fp32 vs fp64, T = %d, K = %d: %.2e" % (T, K, err))
    assert err < FP32_GATE


@pytest.mark.gpu
def test_auto_c_entry_nan_tails():
    from pybold_b200 import _lib
    V, T, K, nb = 5, 2000, 28, 40
    y, h = signals(V, T, K, seed=11)
    L = lipschitz(h, T)
    sigma = np.array([orc.mad_daub_noise_est(v) for v in y])
    d = lambda a: dev(a, torch.float32)  # noqa: E731
    yd, hd, sd, Ld = d(y), d(h), d(sigma), d(L)
    J, R, G = (torch.zeros((V, nb), dtype=torch.float32, device="cuda") for _ in range(3))
    x, z, dz = (torch.empty((V, T), dtype=torch.float32, device="cuda") for _ in range(3))
    lb = torch.empty(V, dtype=torch.float32, device="cuda")
    n = torch.full((V,), -1, dtype=torch.int32, device="cuda")
    assert variant(T, K, nb_iter=30, es=True, wind=4, auto=True)[1] == CTA
    rc = _lib.lib.pb_deconv_auto_f32(yd.data_ptr(), hd.data_ptr(), K, Ld.data_ptr(), 1, sd.data_ptr(), 1, nb, 30,
                                     1, 4, 0.1, x.data_ptr(), z.data_ptr(), dz.data_ptr(), J.data_ptr(),
                                     R.data_ptr(), G.data_ptr(), lb.data_ptr(), n.data_ptr(), V, T, K, None)
    assert rc == 0
    torch.cuda.synchronize()
    n = n.cpu().numpy()
    assert np.all((n >= 6) & (n < nb)), n
    for t in (J, R, G):
        t = t.cpu().numpy()
        for v in range(V):
            assert np.all(np.isfinite(t[v, :n[v]])) and np.all(np.isnan(t[v, n[v]:])), v


# ---- lambda path, fit-only mode -----------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("T,K", [(2000, 28), (900, 40)])
def test_path_with_per_voxel_hrf_and_early_stop(T, K):
    import pybold_b200 as pb
    from pybold_b200.bold_signal import deconv_lbda_path, deconv_lbda_path_fit
    V = 6
    y, h = signals(V, T, K, seed=7 * T)
    y, h = y.astype(np.float32), h.astype(np.float32)
    t_r, x0 = T_R[K], np.random.RandomState(1).randn(T)
    lbdas = [0.3, 3.0]
    x, z, dz, J = deconv_lbda_path(y, t_r, h, lbdas, nb_iter=200, x0=x0, **ES)
    for i, lb in enumerate(lbdas):
        x1, z1, dz1, J1, _, _ = pb.deconv(y, t_r, h, lbda=lb, x0=x0, nb_iter=200, **ES)
        for a, b in ((x[i], x1), (z[i], z1), (dz[i], dz1), (J[i], J1)):
            assert np.array_equal(a, b, equal_nan=True), (i, lb)
    R, G, n = deconv_lbda_path_fit(y, t_r, h, lbdas, nb_iter=200, x0=x0, **ES)
    assert np.array_equal(n, np.sum(~np.isnan(J), axis=-1))
    R_ref = np.sum((x.astype(np.float64) - y.astype(np.float64)[None]) ** 2, axis=-1)
    G_ref = np.sum(np.abs(dz.astype(np.float64)), axis=-1)
    assert np.max(np.abs(R - R_ref) / R_ref) < 1e-5 and np.max(np.abs(G - G_ref) / G_ref) < 1e-5


# ---- masked entry -------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("es", [False, True])
@pytest.mark.parametrize("T,K", [(2000, 28), (600, 63)])
def test_masked_rows(T, K, es):
    from pybold_b200.bold_signal import deconv_batch
    V, nb = 10, 120
    y, h = signals(V, T, K, seed=T + es)
    L = lipschitz(h, T)
    lbda = np.linspace(0.3, 3.0, V)
    kw = ES if es else dict(early_stopping=False)
    full = solve(y, h, lbda, L, torch.float32, nb, **kw)
    active = torch.tensor([v % 3 != 1 for v in range(V)], dtype=torch.uint8, device="cuda")
    out = tuple(torch.full((V, T), 7.0, device="cuda") for _ in range(3)) + (
        torch.full((V,), -5, dtype=torch.int32, device="cuda"),)
    x, z, dz, J, n = deconv_batch(dev(y, torch.float32), dev(h, torch.float32), dev(lbda, torch.float32),
                                  dev(L, torch.float32), nb_iter=nb, active=active, out=out, **kw)
    got = tuple(t.cpu().numpy() for t in (x, z, dz, J, n))
    on = active.cpu().numpy().astype(bool)
    for g, f in zip(got, full):
        assert np.array_equal(g[on], f[on], equal_nan=True)
    for g in got[:3]:
        assert np.all(g[~on] == 7.0)
    assert np.all(got[4][~on] == -5) and np.all(np.isnan(got[3][~on]))
