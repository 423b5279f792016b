"""bd(early_stopping=True) on the CTA-per-voxel kernel (``fast_bdc_kernel<..., ES = true>``, csrc/pb_fastc.cuh).

Every group and CTA row has an early-stopping bd entry point, so an early-stopping bd call runs on the row
``pb_solver_variant`` reports for the shape; the warp-per-voxel and generic kernels remain the fall-back where no
such row exists.  ``pb_bd_variant`` reports the kernel a call runs on, by the launch's own routing.  Q6 is the
reference's inner stop, Q7 its signed outer stop on the windowed means of J (pybold/bold_signal.py:267-273,
:350-362).
"""
import ctypes
import math

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle import pybold_oracle as orc  # noqa: E402

GENERIC, GROUP, WARP, CTA = 0, 1, 2, 3
KS = (1, 20, 27, 28, 32, 33, 40, 63, 64)


def rel(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return np.max(np.abs(a - b)) / (np.max(np.abs(b)) + 1e-300)


def bd_variant(T, K, f64=False, nb_iter=100, es=False, wind=4):
    from pybold_b200 import _lib
    fam = ctypes.c_int(-1)
    vid = _lib.lib.pb_bd_variant(T, K, int(f64), nb_iter, int(es), wind, ctypes.byref(fam))
    assert vid >= 0, (T, K, vid)
    return vid, fam.value


def gen(V, T, t_r, seed):
    from pybold_b200.synth import gen_voxels
    return gen_voxels(V, T, t_r, 20.0, seed0=seed)


def inner_stops(y, w0, hrf, lbda, nb_iter, tol):
    """Iterations the reference's inner loop runs from w0 with early stopping (its Q6 break), as
    orc.loops_deconv computes them."""
    T = len(y)
    A = orc.toeplitz_from_kernel(hrf, T).dot(np.tril(np.ones((T, T))))
    AtA, Aty = A.T.dot(A), A.T.dot(y)
    lip = np.linalg.norm(AtA)
    w, t_old = np.array(w0, dtype=np.float64), 1.0
    for j in range(nb_iter):
        u = w - (AtA.dot(w) - Aty) / lip
        v = orc._soft(u, lbda / lip)
        t = 0.5 * (1.0 + math.sqrt(1.0 + 4.0 * t_old * t_old))
        p = np.zeros(T) if j == 0 else u
        w = v + (t_old - 1.0) / t * (v - p)
        if j > 2 and np.linalg.norm(w - p) / (np.linalg.norm(w) + 1.0e-10) < tol:
            return j + 1
        t_old = t
    return nb_iter


# ---- routing --------------------------------------------------------------------------------------------------

def _t_grid(K):
    """A stride over 1..4096 plus both sides of every change of pb_solver_variant (the edges of every range)."""
    from pybold_b200 import _lib
    ids = [_lib.lib.pb_solver_variant(T, K, 0) for T in range(1, 4097)]
    edges = {T for T in range(2, 4097) if ids[T - 1] != ids[T - 2]}
    return sorted(set(range(1, 4097, 37)) | {4096} | edges | {T - 1 for T in edges})


@pytest.mark.gpu
def test_es_calls_run_on_the_reported_variant_fp32():
    from pybold_b200 import _lib
    n_warp = 0
    for K in KS:
        for T in _t_grid(K):
            vid, fam = bd_variant(T, K)
            assert vid == _lib.lib.pb_solver_variant(T, K, 0), (T, K)
            es = bd_variant(T, K, es=True, wind=4)
            if fam in (GROUP, CTA):
                assert es == (vid, fam), (T, K, es, vid, fam)
            if T > 352 or K > 28:                  # the shapes that ran on the warp or generic kernel before
                assert es[1] == CTA, (T, K, es)
            if fam == WARP:                        # the shortest series: only a warp row serves them
                assert es == (vid, WARP), (T, K, es)
                n_warp += 1
    assert n_warp > 0


@pytest.mark.gpu
def test_es_fp64_parity_rows_run_on_cta():
    for T in (305, 400, 640):
        for K in (1, 20):
            assert bd_variant(T, K, f64=True, es=True) == bd_variant(T, K, f64=True) == (32020020, CTA), (T, K)
    for T in (641, 1000, 1280):
        for K in (20, 28):
            assert bd_variant(T, K, f64=True, es=True) == bd_variant(T, K, f64=True) == (64020028, CTA), (T, K)
    assert bd_variant(1000, 29, f64=True, es=True)[1] == GENERIC


@pytest.mark.gpu
def test_bd_variant_query_errors():
    from pybold_b200 import _lib
    fam = ctypes.c_int()
    q = _lib.lib.pb_bd_variant
    for es in (0, 1):
        assert q(0, 20, 0, 100, es, 4, ctypes.byref(fam)) == _lib.PB_ERR_INVALID_ARG
        assert q(300, 0, 0, 100, es, 4, ctypes.byref(fam)) == _lib.PB_ERR_INVALID_ARG
        assert q(300, 20, 0, 0, es, 4, ctypes.byref(fam)) == _lib.PB_ERR_INVALID_ARG
        assert q(300, 20, 0, 100, es, -1, ctypes.byref(fam)) == _lib.PB_ERR_INVALID_ARG
        assert q(300, 20, 0, 100, es, 4, None) == _lib.PB_ERR_INVALID_ARG
        assert q(4097, 20, 0, 100, es, 4, ctypes.byref(fam)) == _lib.PB_ERR_UNSUPPORTED
        assert q(300, 65, 0, 100, es, 4, ctypes.byref(fam)) == _lib.PB_ERR_UNSUPPORTED


# ---- FP64 CTA rows against the oracle ------------------------------------------------------------------------------

ES_ORACLE = dict(lbda=1.7, theta_0=2.0, hrf_dur=20.0, nb_iter=30, early_stopping=True, wind=4, tol=2.0e-3)


@pytest.mark.gpu
@pytest.mark.parametrize("T,t_r", [(305, 1.0), (640, 1.0), (641, 0.72), (1000, 0.72), (1280, 0.72)])
def test_es_fp64_cta_vs_oracle(T, t_r):
    """Both stops fire: Q6 after a different number of inner iterations per voxel and pass, Q7 before nb_iter."""
    import pybold_b200 as pb
    V = 3
    y = gen(V, T, t_r, 2600 + T) * np.linspace(0.5, 2.0, V)[:, None]
    K = pb.hrf_model.hrf_len(t_r, 20.0)
    assert bd_variant(T, K, f64=True, nb_iter=30, es=True)[1] == CTA
    x, z, dz, h, d = pb.bd(y, t_r, **ES_ORACLE)
    n_tr = d["n_trace"]
    nb = ES_ORACLE["nb_iter"]
    assert np.all(n_tr < nb + 2)                               # Q7 ended every run early
    stops = []
    for v in range(V):
        tr = {}
        xo, zo, wo, ho, do = orc.bd(y[v], t_r, theta_solver="exact", trace=tr, **ES_ORACLE)
        assert len(do["J"]) == n_tr[v], v
        assert rel(z[v], zo) < 1e-7 and rel(dz[v], wo) < 1e-7 and rel(h[v], ho) < 1e-7, v
        assert rel(d["J"][v, :n_tr[v]], do["J"]) < 1e-8, v
        stops.append(tuple(inner_stops(y[v], tr["w_in"][i], tr["h"][i], ES_ORACLE["lbda"], nb, ES_ORACLE["tol"])
                           for i in range(len(tr["w_in"]))))
    print("T = %d: inner iterations per pass %s, n_trace %s" % (T, stops, n_tr))
    assert all(min(s) < nb for s in stops)                     # Q6 fired for every voxel
    assert len(set(stops)) > 1                                 # ... not in the same passes


# ---- FP32 CTA against the FP64 generic kernel ----------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("T,t_r", [(1300, 0.72), (2000, 0.72), (4096, 0.72), (600, 0.5), (1500, 0.32), (3000, 1.0)])
def test_es_fp32_cta_vs_fp64_generic(T, t_r):
    """The default tol = 1e-12: Q6 never fires, Q7 alone decides the trace length."""
    import pybold_b200 as pb
    K = pb.hrf_model.hrf_len(t_r, 20.0)
    assert bd_variant(T, K, nb_iter=12, es=True)[1] == CTA
    assert bd_variant(T, K, f64=True, nb_iter=12, es=True)[1] == GENERIC
    y = gen(3, T, t_r, 7700 + T)
    kw = dict(lbda=1.4, theta_0=2.0, hrf_dur=20.0, nb_iter=12, early_stopping=True, wind=4)
    x, z, dz, h, d = pb.bd(y, t_r, **kw)
    x32, z32, dz32, h32, d32 = pb.bd(y.astype(np.float32), t_r, **kw)
    assert np.array_equal(d32["n_trace"], d["n_trace"]) and np.all(d["n_trace"] < 14)
    # FP32 and FP64 drift apart with the series length through the theta step (test_gpu_solvers.py,
    # test_bd_short_tr_and_long_series_variants): the same bounds
    tol = 1e-4 if T <= 1300 else (4e-4 if T <= 2600 else 2.5e-3)
    assert rel(z32, z) < tol and rel(x32, x) < tol and rel(h32, h) < tol
    assert np.max(np.abs(d32["theta"] - d["theta"])) < tol
    for v in range(3):
        n = d["n_trace"][v]
        assert rel(d32["J"][v, :n], d["J"][v, :n]) < 1e-4


# ---- batch against single voxel, through the work queue ------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("T,t_r,nw", [(600, 1.0, 1), (2000, 0.72, 4)])
def test_es_batch_equals_single_and_permutation(T, t_r, nw):
    """A batch larger than one wave of the grid: the CTAs take their later voxels from the work queue.  Every ninth
    voxel has lambda = 1e4 and no warm start: its cost rises from pass to pass, so the signed Q7 test never stops it
    (n_trace = nb_iter + 2), while the others stop at the first test: the voxels finish at different outer counts."""
    import pybold_b200 as pb
    from pybold_b200 import _lib
    K = pb.hrf_model.hrf_len(t_r, 20.0)
    vid, fam = bd_variant(T, K, nb_iter=10, es=True)
    assert fam == CTA and vid // 1000000 == 32 * nw
    wave = _lib.lib.pb_bd_wave_voxels(T, K, 0, 10)
    V = wave + 37
    rs = np.random.RandomState(T)
    y = (gen(V, T, t_r, 8100 + T) * rs.uniform(0.3, 3.0, (V, 1))).astype(np.float32)
    lb = rs.uniform(0.5, 3.0, V)
    lb[::9] = 1.0e4
    lb = lb.astype(np.float32)
    th0 = rs.uniform(0.8, 2.0, V).astype(np.float32)
    z0 = (0.2 * y * rs.uniform(0.0, 1.0, (V, 1))).astype(np.float32)
    z0[::9] = 0.0
    kw = dict(hrf_dur=20.0, nb_iter=10, early_stopping=True, wind=4, tol=1.0e-3)

    def run(idx):
        out = pb.bd(torch.as_tensor(y[idx], device="cuda"), t_r, lbda=torch.as_tensor(lb[idx], device="cuda"),
                    theta_0=torch.as_tensor(th0[idx], device="cuda"), z_0=torch.as_tensor(z0[idx], device="cuda"),
                    **kw)
        x, z, dz, h, d = (t.cpu().numpy() if isinstance(t, torch.Tensor) else t for t in out)
        return x, z, dz, h, {k: d[k].cpu().numpy() for k in ("J", "r", "g", "theta", "n_trace")}

    full = run(np.arange(V))
    n_tr = full[4]["n_trace"]
    assert len(set(n_tr.tolist())) >= 2 and np.all(n_tr[::9] == 12), sorted(set(n_tr.tolist()))
    perm = rs.permutation(V)
    permuted = run(perm)
    for a, b in zip(full[:4], permuted[:4]):
        assert np.array_equal(a[perm], b)
    for k in ("J", "r", "g", "theta", "n_trace"):       # (trace rows past n_trace hold bd_alloc's NaN fill)
        assert np.array_equal(full[4][k][perm], permuted[4][k], equal_nan=True), k
    for v in list(range(0, V, 97)) + [V - 1]:
        one = run(np.array([v]))
        for a, b in zip(full[:4], one[:4]):
            assert np.array_equal(a[v:v + 1], b), v
        n = n_tr[v]
        for k in ("J", "r", "g"):
            assert np.array_equal(full[4][k][v, :n], one[4][k][0, :n]), (v, k)
        assert one[4]["n_trace"][0] == n


# ---- the C entry: trace entries past out_ntrace are not written -----------------------------------------------------

@pytest.mark.gpu
def test_es_c_entry_trace_tail_untouched():
    """pb_bd_f32 through bd_batch, the ctypes call with caller-owned output buffers (``out=``): the J / r / g rows are
    filled with a sentinel first, and the entries past out_ntrace must still hold it after the call."""
    from pybold_b200.bold_signal import bd_alloc, bd_batch
    T, t_r, V = 1200, 0.72, 6
    K = 28
    assert bd_variant(T, K, nb_iter=20, es=True)[1] == CTA
    y = torch.as_tensor(gen(V, T, t_r, 8300), dtype=torch.float32, device="cuda")
    bounds = [(0.6, 1.9)]
    sentinel = -12345.0
    for nb_iter, wind in ((20, 4), (5, 4), (4, 4), (3, 8)):
        out = bd_alloc(V, T, K, nb_iter, torch.float32, y.device)
        for k in ("J", "r", "g"):
            out[k].fill_(sentinel)
        bd_batch(y, t_r, 1.5, 2.0, None, 20.0, bounds, nb_iter, True, wind, 1.0e-12, out=out)
        n = out["n_trace"].cpu().numpy()
        if nb_iter <= wind + 1:                    # Q7 tests after passes idx > wind only
            assert np.all(n == nb_iter + 2), (nb_iter, wind, n)
        else:
            assert np.all(n < nb_iter + 2), n
        for k in ("J", "r", "g"):
            a = out[k].cpu().numpy()
            for v in range(V):
                assert np.all(a[v, n[v]:] == sentinel), (k, v)
                assert np.all(np.isfinite(a[v, :n[v]])) and not np.any(a[v, :n[v]] == sentinel), (k, v)
