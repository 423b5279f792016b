"""Degenerate and scanner-unit voxels through every deconvolution entry point and kernel family.

A whole-brain batch does not hold clean voxels only: all-zero voxels outside the brain mask, constant voxels, series in
raw scanner units (a DC level near 1e4, fluctuations near 1e2) and single NaN or Inf scans nobody censored.  Each case
below is pinned, through the routing queries, to the kernel family it runs on (group, warp, CTA, generic), and checks:

* isolation: in a batch larger than one grid wave, a good voxel gives the same bits with or without bad voxels around
  it, and a permuted batch gives permuted rows;
* the float64 reference on the degenerate voxels themselves (oracle/pybold_oracle.py, tests/censor_reference.py):
  FP64 at 1e-9 with the same iteration and outer counts, FP32 directly against it;
* exact symmetries: y -> -y everywhere, (y, lbda) -> 2^k (y, lbda) where no absolute constant enters;
* the MAD kernels on rows that hold NaN or Inf, and deconv(lbda=None) with a NaN noise level.
"""
import ctypes
import functools

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle import pybold_oracle as orc  # noqa: E402
from tests import censor_reference as cref  # noqa: E402

GENERIC, GROUP, WARP, CTA = 0, 1, 2, 3
F32, F64 = torch.float32, torch.float64
T_R = {20: 1.0, 28: 0.72, 40: 0.5, 63: 0.32}            # hrf_dur 20 s -> K taps
NB = 60                                                 # deconv iterations
ES = dict(early_stopping=True, tol=1.0e-2, wind=6)      # Q5 fires within NB on the good voxels
AUTO = dict(nb_iter=10, nb_sub_iter=30, early_stopping=True, tol=0.1, wind=4)
LBDAS = [0.3, 1.5]
BD = dict(theta_0=2.0, hrf_dur=20.0, nb_iter=8, wind=4, tol=1.0e-3)

# name: (T, K, dtype, family of deconv / deconv(lbda=None) / the path, family of the censored calls)
CASES = {
    "group-f32": (300, 20, F32, GROUP, CTA),
    "group-f64": (300, 20, F64, GROUP, GENERIC),
    "warp-600": (600, 20, F32, WARP, CTA),
    "warp-1200": (1200, 28, F32, WARP, CTA),
    "cta-1500": (1500, 28, F32, CTA, CTA),
    "cta-2000-k63": (2000, 63, F32, CTA, CTA),
    "cta-600-k40": (600, 40, F32, CTA, CTA),
    "generic-f64": (300, 40, F64, GENERIC, GENERIC),
}
ENTRIES = ("deconv", "deconv-es", "auto-sigma", "auto-est", "path", "fit", "censored", "censored-auto")
# name: (T, t_r, family of bd with early stopping)
BD_CASES = {"bd-group": (300, 1.0, GROUP), "bd-cta": (2000, 0.72, CTA), "bd-cta-k40": (600, 0.5, CTA)}

KINDS = ("zero", "const", "const1e4", "scanner", "tiny", "huge", "nan", "inf")


def same_nan(a, b, zeros_ok=False):
    """The NaN pattern of the float64 reference.  zeros_ok: the dense reference also multiplies NaN by the exact zeros
    of its Toeplitz matrices (and by the SPM HRF's tap 0, which is 0); the kernels never form those products, so a scan
    that no data reaches -- a censored tail, x[0] and diff_z[T - 1] of bd -- may stay 0 where the reference has NaN."""
    na, nb = np.isnan(np.asarray(a, dtype=np.float64)), np.isnan(np.asarray(b, dtype=np.float64))
    if not zeros_ok:
        return np.array_equal(na, nb)
    return bool(np.all(nb | ~na) and np.all(na | ~nb | (np.asarray(a) == 0)))


def rel(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return np.max(np.abs(a - b)) / (np.max(np.abs(b)) + 1e-300)


def dev(a, dtype):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=dtype, device="cuda")


def same(a, b):
    """Bit for bit up to the sign of zero (like np.array_equal), NaN equal to NaN."""
    if not a.dtype.is_floating_point:
        return torch.equal(a, b)
    return a.shape == b.shape and bool(((a == b) | (torch.isnan(a) & torch.isnan(b))).all())


def routed(T, K, dtype, entry):
    """(variant id, family) the routing query reports for an entry point at this shape."""
    from pybold_b200 import _lib
    f64, fam = int(dtype == F64), ctypes.c_int(-1)
    auto = entry in ("auto-sigma", "auto-est", "censored-auto")
    nb, es, wind = (AUTO["nb_sub_iter"], 1, AUTO["wind"]) if auto else (NB, int(entry != "deconv"), ES["wind"])
    q = _lib.lib.pb_deconv_censored_variant if entry.startswith("censored") else _lib.lib.pb_deconv_variant
    vid = q(T, K, f64, nb, es, wind, int(auto), ctypes.byref(fam))
    assert vid >= 0, (T, K, entry, vid)
    return vid, fam.value


def bd_routed(T, t_r, dtype, es):
    from pybold_b200 import _lib
    from pybold_b200.hrf_model import hrf_len
    fam = ctypes.c_int(-1)
    vid = _lib.lib.pb_bd_variant(T, hrf_len(t_r, 20.0), int(dtype == F64), BD["nb_iter"], int(es), BD["wind"],
                                 ctypes.byref(fam))
    assert vid >= 0
    return vid, fam.value


def wave_max(vid, fam):
    """An upper bound on the problems one wave of the persistent grid holds: ids are lanes per problem * 1e6 + ..."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    if fam == GENERIC or vid == 0:
        return sms * 64
    lanes = vid // 1000000
    return sms * (min(32, 2048 // lanes) if fam == CTA else 2048 // lanes)


@functools.lru_cache(maxsize=None)
def taps(K):
    return orc.spm_hrf(1.0, T_R[K], 20.0, True)[0]


@functools.lru_cache(maxsize=None)
def lipschitz(T, K):
    return 0.9 * orc.spectral_radius_est(orc.HrfIntegOperator(taps(K), T), np.random.RandomState(T).randn(T))


def bad_row(kind, g):
    T = len(g)
    if kind == "zero":
        return np.zeros(T)
    if kind == "const":
        return np.full(T, 3.5)
    if kind == "const1e4":
        return np.full(T, 1.0e4)
    if kind == "scanner":
        return 1.0e4 + 100.0 * g
    if kind == "tiny":
        return g * 2.0 ** -40
    if kind == "huge":
        return g * 2.0 ** 40
    r = g.copy()
    r[T // 3] = np.nan if kind == "nan" else np.inf
    return r


def good_voxels(V, T, t_r, seed):
    from pybold_b200.synth import gen_voxels
    rs = np.random.RandomState(seed)
    base = gen_voxels(16, T, t_r, 20.0, seed0=seed)
    return base[rs.randint(0, 16, V)] * rs.uniform(0.5, 2.0, (V, 1))


def mixed(n_good, T, t_r, seed):
    """n_good good voxels with copies of every bad kind among them: some at random places, a run of consecutive
    ones early in the batch (they share warps and CTA rows with good voxels) and some in the tail (from the work
    queue).  Returns (y, is_bad)."""
    rs = np.random.RandomState(seed + 1)
    n = n_good + 3 * len(KINDS)
    run0 = min(40, n // 3)
    pos = set(rs.choice(n, len(KINDS), replace=False).tolist()) | set(range(run0, run0 + len(KINDS)))
    pos |= set(range(n - 3 * len(KINDS), n, 3))
    for i in rs.permutation(n):                         # where the sets overlap, fill up to three of each kind
        if len(pos) == 3 * len(KINDS):
            break
        pos.add(int(i))
    pos = sorted(pos)
    is_bad = np.zeros(n, dtype=bool)
    is_bad[pos] = True
    good = good_voxels(n_good, T, t_r, seed)
    y = np.empty((n, T))
    y[~is_bad] = good
    y[is_bad] = np.stack([bad_row(KINDS[i % len(KINDS)], good[i % n_good]) for i in range(len(pos))])
    return y, is_bad


def censor_rows(V, T, seed):
    """About 5 % of the scans of every voxel censored, a different pattern per voxel."""
    cm = np.zeros((V, T), dtype=np.uint8)
    for v in range(V):
        cm[v, (np.arange(max(1, T // 20)) * 19 + 7 * (v + seed)) % T] = 1
    return cm


def run(entry, T, K, dtype, y, lb, cm):
    """One entry point on the rows of y (NumPy), per-voxel lbda / sigma `lb` and per-voxel mask `cm`; returns a dict
    of device tensors with the voxel on axis 0."""
    import pybold_b200 as pb
    from pybold_b200 import bold_signal as bs
    from pybold_b200.censor import mad_daub_noise_est_censored
    yd, h, L = dev(y, dtype), dev(taps(K), dtype), lipschitz(T, K)
    cmd = dev(cm, torch.uint8) if entry.startswith("censored") else None
    if entry in ("deconv", "deconv-es", "censored"):
        kw = dict(early_stopping=False) if entry == "deconv" else ES
        x, z, dz, J, n = bs.deconv_batch(yd, h, dev(lb, dtype), L, None, nb_iter=NB, censor=cmd, **kw)
        return dict(x=x, z=z, diff_z=dz, J=J, n=n)
    if entry in ("auto-sigma", "auto-est", "censored-auto"):
        if entry == "auto-sigma":
            # small enough that lambda stays positive on the zero voxels: their alpha falls by 1e-4 T sigma^2 a pass
            sg = dev(0.05 * lb, dtype)
        elif entry == "auto-est":
            sg = pb.noise.mad_daub_noise_est(yd)
        else:
            sg = mad_daub_noise_est_censored(yd, cmd, T)
        o = bs.deconv_auto_batch(yd, h, sg, L, censor=cmd, **AUTO)
        o["sigma"] = sg
        return o
    f = bs.deconv_lbda_path if entry == "path" else bs.deconv_lbda_path_fit
    out = f(yd, T_R[K], h, LBDAS, nb_iter=NB, x0=np.random.RandomState(T).randn(T), **ES)
    keys = ("x", "z", "diff_z", "J") if entry == "path" else ("R", "G", "n")
    return {k: t.transpose(0, 1) for k, t in zip(keys, out)}


def run_bd(T, t_r, dtype, y, lb, es):
    import pybold_b200 as pb
    x, z, dz, h, d = pb.bd(dev(y, dtype), t_r, lbda=dev(lb, dtype), early_stopping=es, **BD)
    return dict(x=x, z=z, diff_z=dz, h=h, theta=d["theta"], J=d["J"], r=d["r"], g=d["g"], n=d["n_trace"])


def check_isolation(go, y, is_bad, lb, cm):
    full = go(y, lb, cm)
    alone = go(y[~is_bad], lb[~is_bad], cm[~is_bad])
    gi = torch.as_tensor(np.flatnonzero(~is_bad), device="cuda")
    for k in full:
        assert same(full[k][gi], alone[k]), k
    perm = np.random.RandomState(len(y)).permutation(len(y))
    pm = go(y[perm], lb[perm], cm[perm])
    pt = torch.as_tensor(perm, device="cuda")
    for k in full:
        assert same(full[k][pt], pm[k]), k
    return full


# ---- routing ------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_every_family_is_reached():
    """Each case runs on the family of its row in CASES / BD_CASES, and every family appears."""
    seen = set()
    for name, (T, K, dtype, fam, cfam) in CASES.items():
        for entry in ENTRIES:
            got = routed(T, K, dtype, entry)[1]
            assert got == (cfam if entry.startswith("censored") else fam), (name, entry, got)
            seen.add(got)
    for name, (T, t_r, fam) in BD_CASES.items():
        assert bd_routed(T, t_r, F32, True)[1] == fam, name
        assert bd_routed(T, t_r, F32, False)[1] == fam, name
    assert seen == {GENERIC, GROUP, WARP, CTA}, seen


# ---- isolation and permutation in batches beyond one grid wave -----------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("entry", ENTRIES)
@pytest.mark.parametrize("case", list(CASES))
def test_bad_voxels_stay_in_their_rows(case, entry):
    T, K, dtype, fam, cfam = CASES[case]
    vid, got = routed(T, K, dtype, entry)
    assert got == (cfam if entry.startswith("censored") else fam)
    y, is_bad = mixed(wave_max(vid, got) + 37, T, T_R[K], T + K)
    rs = np.random.RandomState(3)
    lb = rs.uniform(0.2, 2.0, len(y))
    cm = censor_rows(len(y), T, K)
    full = check_isolation(lambda a, b, c: run(entry, T, K, dtype, a, b, c), y, is_bad, lb, cm)
    # the bad voxels are there: the NaN voxel is NaN, the zero voxel stays zero
    kinds = np.array([KINDS[i % len(KINDS)] for i in range(is_bad.sum())])
    bad = np.flatnonzero(is_bad)
    first = full["x" if "x" in full else "R"]
    assert bool(torch.isnan(first[int(bad[kinds == "nan"][0])]).all())
    assert not bool(torch.isnan(first[torch.as_tensor(np.flatnonzero(~is_bad), device="cuda")]).any())
    if "x" in full:
        assert bool((first[int(bad[kinds == "zero"][0])] == 0).all())
    if "n" in full and entry != "deconv" and entry != "fit":    # early stopping: the counts differ in the batch
        assert len(set(full["n"].reshape(-1).tolist())) > 1


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(BD_CASES))
def test_bd_bad_voxels_stay_in_their_rows(case):
    from pybold_b200 import _lib
    from pybold_b200.hrf_model import hrf_len
    T, t_r, fam = BD_CASES[case]
    assert bd_routed(T, t_r, F32, True)[1] == fam
    wave = _lib.lib.pb_bd_wave_voxels(T, hrf_len(t_r, 20.0), 0, BD["nb_iter"])
    y, is_bad = mixed(wave + 37, T, t_r, T)
    lb = np.random.RandomState(4).uniform(0.5, 3.0, len(y))
    full = check_isolation(lambda a, b, c: run_bd(T, t_r, F32, a, b, True), y, is_bad, lb, np.zeros(len(y)))
    assert len(set(full["n"].tolist())) > 1


# ---- degenerate voxels against the float64 reference ------------------------------------------------------------

DEGEN = ("zero", "const", "const1e4", "scanner", "nan", "inf")
# (T, K, dtype): every family in both builds where it exists; the dense oracle up to 1200 scans, the censor reference
# (all-zero mask: the oracle bit for bit) beyond
# (T, K, dtype, family of the uncensored calls, family of the censored ones)
REF_CASES = [(300, 20, F64, GROUP, GENERIC), (600, 28, F64, WARP, GENERIC), (1200, 28, F64, CTA, CTA),
             (300, 40, F64, GENERIC, GENERIC), (1500, 28, F64, GENERIC, GENERIC),
             (300, 20, F32, GROUP, CTA), (600, 20, F32, WARP, CTA), (1200, 28, F32, WARP, CTA),
             (1500, 28, F32, CTA, CTA), (600, 40, F32, CTA, CTA), (2000, 63, F32, CTA, CTA)]
REF_ENTRIES = ("deconv", "deconv-es", "auto", "censored", "censored-auto")
# FP32 against the float64 reference, largest relative error over REF_CASES, REF_ENTRIES and the path cases measured
# on a B200 at 1000 W: scanner units (1e4 + 100 good) 2.2e-5, constant 3.5 1.6e-5, constant 1e4 2.0e-5, a good voxel
# 3.5e-5; the all-zero voxel is exactly zero.  Gates at no more than 10x those values.
FP32_GATE = {"zero": 0.0, "const": 5e-5, "const1e4": 1.4e-4, "scanner": 4e-5, "good": 1.9e-4}
_fp32_worst = {}


def ref_inputs(T, K, dtype):
    """Degenerate voxels plus one good voxel, rounded to the build's type (so the reference sees what the device
    sees), the taps and Lipschitz constant likewise, and one censor mask."""
    np_t = np.float32 if dtype == F32 else np.float64
    g = good_voxels(1, T, T_R[K], 100 + T)[0]
    y = np.stack([bad_row(k, g) for k in DEGEN] + [g]).astype(np_t).astype(np.float64)
    h = taps(K).astype(np_t).astype(np.float64)
    L = float(np_t(lipschitz(T, K)))
    return y, h, L, ref_mask(T)


def ref_mask(T):
    """Every odd scan of the first half censored: the last sample of every tile there, thread 0's included (R is even),
    between kept scans, so the fit is not zero there.  Plus a stride-19 pattern and the last 5 % of the series.  The
    second half keeps clean detail coefficients for sigma, and the NaN / Inf scan of DEGEN stays in the fit."""
    cm = censor_rows(1, T, 1)[0]
    cm[1:T // 2:2] = 1
    cm[T - max(1, T // 20):] = 1
    cm[T // 3] = 0
    return cm


def ref_solve(entry, y, h, L, sigma, cm):
    """(outputs, count) of the float64 reference for one voxel."""
    kw = dict(lipschitz=L, nb_iter=NB)
    with np.errstate(all="ignore"):      # 0 / 0 and inf - inf on purpose
        if entry in ("deconv", "deconv-es"):
            kw.update(ES if entry == "deconv-es" else dict(early_stopping=False))
            x, z, w, J, n = cref.deconv_fixed_lbda(y, h, 0.7, **kw)
            return dict(x=x, z=z, diff_z=w, J=J), n
        if entry == "censored":
            x, z, w, J, n = cref.deconv_fixed_lbda(y, h, 0.7, censor=cm, **kw, **ES)
            return dict(x=x, z=z, diff_z=w, J=J), n
        x, z, w, J, R, G, lb = cref.deconv_auto_lbda(y, h, sigma, lipschitz=L, censor=cm if entry != "auto" else None,
                                                     **AUTO)
        return dict(x=x, z=z, diff_z=w, J=np.array(J), R=np.array(R), G=np.array(G), lbda=np.array(lb)), len(J)


def dev_solve(entry, y, h, L, sigma, cm, dtype):
    from pybold_b200 import bold_signal as bs
    yd, hd = dev(y, dtype), dev(h, dtype)
    cmd = dev(cm, torch.uint8) if entry.startswith("censored") else None
    if entry in ("deconv", "deconv-es", "censored"):
        kw = dict(early_stopping=False) if entry == "deconv" else ES
        x, z, dz, J, n = bs.deconv_batch(yd, hd, 0.7, L, None, nb_iter=NB, censor=cmd, **kw)
        J = J / (J[:, :1] + 1.0e-30)
        out = dict(x=x, z=z, diff_z=dz, J=J)
    else:
        out = bs.deconv_auto_batch(yd, hd, dev(sigma, dtype), L, censor=cmd, **AUTO)
        n = out.pop("n_outer")
    return {k: v.double().cpu().numpy() for k, v in out.items()}, n.cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("entry", REF_ENTRIES)
@pytest.mark.parametrize("T,K,dtype,fam,cfam", REF_CASES)
def test_degenerate_voxels_match_reference(T, K, dtype, fam, cfam, entry):
    y, h, L, cm = ref_inputs(T, K, dtype)
    q = entry if entry in ("deconv", "deconv-es", "censored", "censored-auto") else "auto-sigma"
    assert routed(T, K, dtype, q)[1] == (cfam if entry.startswith("censored") else fam)
    with np.errstate(all="ignore"):
        sigma = np.array([cref.mad_daub_noise_est(v, cm if entry == "censored-auto" else None) for v in y])
    sigma = sigma.astype(np.float32 if dtype == F32 else np.float64).astype(np.float64)
    got, n = dev_solve(entry, y, h, L, sigma, cm, dtype)
    kinds = DEGEN + ("good",)
    for v, kind in enumerate(kinds):
        ref, n_ref = ref_solve(entry, y[v], h, L, sigma[v], cm)
        if kind == "zero" and entry != "deconv":        # 0 / (0 + 1e-10): the first iteration where a stop can fire
            first = (ES["wind"] if entry in ("deconv-es", "censored") else AUTO["wind"]) + 2
            assert n_ref == first, (entry, n_ref)
        if kind == "nan":                               # never stops
            assert n_ref == (NB if entry in ("deconv", "deconv-es", "censored") else AUTO["nb_iter"])
        if dtype == F64 or kind in ("zero", "nan"):
            assert n[v] == n_ref, (kind, n[v], n_ref)
        for k, b in ref.items():
            a = got[k][v] if k != "lbda" else got[k][v:v + 1]
            if k in ("J", "R", "G"):
                a = a[:n_ref]
            b = np.atleast_1d(b)
            if kind in ("nan", "inf"):
                assert same_nan(a, b, zeros_ok=entry.startswith("censored")), (kind, k)
                continue
            e = rel(a, b)
            if dtype == F64:
                assert e < 1e-9, (kind, k, e)
            else:
                _fp32_worst[kind] = max(_fp32_worst.get(kind, 0.0), e)
                assert e <= FP32_GATE[kind], (kind, k, e)
    if dtype == F32:
        print("FP32 worst so far: %s" % _fp32_worst)


@pytest.mark.gpu
@pytest.mark.parametrize("T,K,dtype,fam", [(300, 20, F64, GROUP), (600, 28, F64, WARP), (1200, 28, F64, CTA),
                                           (300, 40, F64, GENERIC), (1500, 28, F32, CTA)])
def test_path_degenerate_voxels_match_reference(T, K, dtype, fam):
    """The lambda path and its fit-only mode on the degenerate voxels: every (lambda, voxel) problem against the
    reference's deconv with early stopping, same stop iteration, same NaN pattern."""
    from pybold_b200 import bold_signal as bs
    assert routed(T, K, dtype, "path")[1] == fam and routed(T, K, dtype, "fit")[1] == fam
    y, h, _, _ = ref_inputs(T, K, dtype)
    x0 = np.random.RandomState(T + 1).randn(T)
    L = 0.9 * orc.spectral_radius_est(orc.HrfIntegOperator(h, T), x0)
    yd, hd = dev(y, dtype), dev(h, dtype)
    x, z, dz, J = (t.double().cpu().numpy() for t in bs.deconv_lbda_path(yd, T_R[K], hd, LBDAS, nb_iter=NB, x0=x0,
                                                                            **ES))
    R, G, n = (t.cpu().numpy() for t in bs.deconv_lbda_path_fit(yd, T_R[K], hd, LBDAS, nb_iter=NB, x0=x0, **ES))
    gate = 1e-9 if dtype == F64 else FP32_GATE
    for li, lb in enumerate(LBDAS):
        for v, kind in enumerate(DEGEN + ("good",)):
            with np.errstate(all="ignore"):
                xo, zo, wo, Jo, no = cref.deconv_fixed_lbda(y[v], h, lb, lipschitz=L, nb_iter=NB, **ES)
                Ro, Go = np.sum(np.square(xo - y[v])), np.sum(np.abs(wo))
            if dtype == F64 or kind in ("zero", "nan"):
                assert n[li, v] == no, (lb, kind, n[li, v], no)
            pairs = ((x[li, v], xo), (z[li, v], zo), (dz[li, v], wo), (J[li, v, :no], Jo), (R[li, v], Ro),
                     (G[li, v], Go))
            for a, b in pairs:
                if kind in ("nan", "inf"):
                    assert np.array_equal(np.isnan(a), np.isnan(b)), (lb, kind)
                else:
                    e = rel(a, b)
                    assert e <= (gate if dtype == F64 else gate[kind]), (lb, kind, e)


# bd against the oracle running the device's theta algorithm (theta_solver="exact").  The gates are the bd parity
# gates of DESIGN.md section 2: the theta step ends on a Newton step of at most 1e-7 (THETA_XTOL_NEWTON), so FP64
# agrees with the oracle to ~1e-7 on the iterates and ~1e-8 on the normalised traces, not to 1e-9.
BD_REF = dict(lbda=1.7, theta_0=2.0, hrf_dur=20.0, nb_iter=8, wind=4, tol=2.0e-3)
BD_GATE = {F64: dict(x=1e-7, z=1e-7, diff_z=1e-7, h=1e-7, J=1e-8, r=1e-8, g=1e-7),
           # FP32: largest relative error over every key and voxel kind, measured on a B200 at 1000 W: 7.0e-6 (a good
           # voxel; scanner units 8.3e-7, constants 6.7e-7, zero 2.5e-8); the gate is 10x that
           F32: dict(x=7e-5, z=7e-5, diff_z=7e-5, h=7e-5, J=7e-5, r=7e-5, g=7e-5)}
_bd_fp32_worst = {}


@pytest.mark.gpu
@pytest.mark.parametrize("es", [False, True])
@pytest.mark.parametrize("T,t_r,dtype,fam", [(300, 1.0, F64, GROUP), (400, 1.0, F64, CTA), (300, 1.0, F32, GROUP),
                                             (600, 0.5, F32, CTA)])
def test_bd_degenerate_voxels_match_reference(T, t_r, dtype, fam, es):
    """bd on zero, constant, scanner-unit, NaN and Inf voxels against orc.bd.  A zero voxel has j_0 = 0: the
    reference's normalised J is NaN and Q7 never fires, so it runs every outer iteration; so does a NaN voxel."""
    import pybold_b200 as pb
    assert bd_routed(T, t_r, dtype, es)[1] == fam
    np_t = np.float32 if dtype == F32 else np.float64
    g = good_voxels(1, T, t_r, 200 + T)[0]
    y = np.stack([bad_row(k, g) for k in DEGEN] + [g]).astype(np_t)
    x, z, dz, h, d = pb.bd(y, t_r, early_stopping=es, **BD_REF)
    got = dict(x=x, z=z, diff_z=dz, h=h, J=d["J"], r=d["r"], g=d["g"])
    for v, kind in enumerate(DEGEN + ("good",)):
        with np.errstate(all="ignore"):
            xo, zo, wo, ho, do = orc.bd(y[v].astype(np.float64), t_r, theta_solver="exact", early_stopping=es,
                                        **BD_REF)
        n = len(do["J"])
        if kind in ("zero", "nan"):
            assert n == BD_REF["nb_iter"] + 2, (kind, n)
        if dtype == F64 or kind in ("zero", "nan"):
            assert d["n_trace"][v] == n, (kind, d["n_trace"][v], n)
        ref = dict(x=xo, z=zo, diff_z=wo, h=ho, J=do["J"], r=do["r"], g=do["g"])
        for k, b in ref.items():
            a = got[k][v][:n] if k in ("J", "r", "g") else got[k][v]
            if kind in ("nan", "inf") or k in ("J", "r") and kind == "zero":
                assert same_nan(a, b, zeros_ok=k in ("x", "z", "diff_z")), (kind, k, a, b)
                continue
            e = rel(a, b)
            if dtype == F32:
                _bd_fp32_worst[kind] = max(_bd_fp32_worst.get(kind, 0.0), e)
            assert e <= BD_GATE[dtype][k], (kind, k, e)
    if dtype == F32:
        print("bd FP32 worst so far: %s" % _bd_fp32_worst)


@pytest.mark.gpu
@pytest.mark.xfail(strict=True, reason="open divergence (DESIGN.md section 2): with a negative lambda the kernels' "
                                       "clamp moves every entry by -th, the reference's soft threshold keeps 0 at 0")
def test_auto_negative_lambda_keeps_a_zero_voxel_at_zero():
    """deconv(lbda=None) with a given sigma on an all-zero voxel: r = 0 every pass, so alpha falls by 1e-4 T sigma^2
    per outer iteration and turns negative after nine; the reference then still returns x = 0."""
    from pybold_b200 import bold_signal as bs
    T, K = 1200, 28
    L = lipschitz(T, K)
    kw = dict(nb_iter=12, nb_sub_iter=30, early_stopping=False)
    xo, zo, wo, Jo, Ro, Go, lo = cref.deconv_auto_lbda(np.zeros(T), taps(K), 1.0, lipschitz=L, **kw)
    assert lo < 0 and np.all(xo == 0)
    o = bs.deconv_auto_batch(dev(np.zeros((1, T)), F64), dev(taps(K), F64), 1.0, L, **kw)
    assert float(o["lbda"][0]) < 0
    assert bool((o["x"] == 0).all())


# ---- exact symmetries ---------------------------------------------------------------------------------------------

ODD = ("x", "z", "diff_z")


@pytest.mark.gpu
@pytest.mark.parametrize("entry", ENTRIES)
@pytest.mark.parametrize("case", list(CASES))
def test_sign_symmetry(case, entry):
    """y -> -y negates x, z, diff_z and leaves everything else alone, bit for bit: IEEE rounding and the median are
    sign-symmetric."""
    T, K, dtype, fam, cfam = CASES[case]
    assert routed(T, K, dtype, entry)[1] == (cfam if entry.startswith("censored") else fam)
    y, _ = mixed(12, T, T_R[K], 7 * T + K)
    lb = np.random.RandomState(5).uniform(0.2, 2.0, len(y))
    cm = censor_rows(len(y), T, 3)
    a = run(entry, T, K, dtype, y, lb, cm)
    b = run(entry, T, K, dtype, -y, lb, cm)
    for k in a:
        assert same(-a[k] if k in ODD else a[k], b[k]), k


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(BD_CASES))
@pytest.mark.parametrize("es", [False, True])
def test_bd_sign_symmetry(case, es):
    T, t_r, fam = BD_CASES[case]
    assert bd_routed(T, t_r, F32, es)[1] == fam
    y, _ = mixed(12, T, t_r, 3 * T)
    lb = np.random.RandomState(6).uniform(0.5, 3.0, len(y))
    a = run_bd(T, t_r, F32, y, lb, es)
    b = run_bd(T, t_r, F32, -y, lb, es)
    for k in a:
        assert same(-a[k] if k in ODD else a[k], b[k]), k


@pytest.mark.gpu
@pytest.mark.parametrize("k", [-64, -40, -20, 20, 40])
@pytest.mark.parametrize("case", list(CASES))
def test_scale_symmetry_deconv(case, k):
    """(y, lbda) -> 2^k (y, lbda): x, z, diff_z scale by 2^k and the cost by 2^2k, bit for bit.  Only without early
    stopping: the reference's Q5 test adds an absolute 1e-10.  At k = -64 the threshold lbda / L is 1e-29 to 1e-26
    (L ~ 1e7 to 1e8 here), where an absolute offset of 1e-30 would show; the squares of the residual then fall below
    FP32's normal range, so the cost is left out there."""
    T, K, dtype, fam, _ = CASES[case]
    assert routed(T, K, dtype, "deconv")[1] == fam
    y = good_voxels(12, T, T_R[K], 11 * T + K)
    lb = np.random.RandomState(7).uniform(0.2, 2.0, len(y))
    a = run("deconv", T, K, dtype, y, lb, None)
    b = run("deconv", T, K, dtype, y * 2.0 ** k, lb * 2.0 ** k, None)
    for key in ODD:
        assert same(a[key] * 2.0 ** k, b[key]), key
    assert same(a["n"], b["n"])
    if k > -64:
        assert same(a["J"] * 2.0 ** (2 * k), b["J"])


@pytest.mark.gpu
@pytest.mark.parametrize("k", [-40, -20, 20, 40])
@pytest.mark.parametrize("case", list(BD_CASES))
def test_scale_symmetry_bd(case, k):
    """bd without early stopping: x, z, diff_z and g = ||diff_z||_1 scale by 2^k; h, theta and the traces normalised
    by the first cost (J, r) do not change."""
    T, t_r, fam = BD_CASES[case]
    assert bd_routed(T, t_r, F32, False)[1] == fam
    y = good_voxels(12, T, t_r, 13 * T)
    lb = np.random.RandomState(8).uniform(0.5, 3.0, len(y))
    a = run_bd(T, t_r, F32, y, lb, False)
    b = run_bd(T, t_r, F32, y * 2.0 ** k, lb * 2.0 ** k, False)
    for key in a:
        assert same(a[key] * 2.0 ** k if key in ODD + ("g",) else a[key], b[key]), key


# ---- the MAD with non-finite values -------------------------------------------------------------------------------

def mad_rows(n, seed):
    """Rows of n values with NaN (sign bit clear and set), +inf, -inf, both, and more than half +inf."""
    rs = np.random.RandomState(seed)
    rows = []
    for fill in ("nan", "-nan", "inf", "-inf", "both", "most_inf", "half_each", "two_inf"):
        r = rs.randn(n)
        i = rs.permutation(n)
        if fill == "nan":
            r[i[0]] = np.nan
        elif fill == "-nan":
            r[i[0]] = -np.nan
        elif fill == "inf":
            r[i[0]] = np.inf
        elif fill == "-inf":
            r[i[0]] = -np.inf
        elif fill == "both":
            r[i[0]], r[i[1]] = np.inf, -np.inf
        elif fill == "most_inf":
            r[i[:n // 2 + 1]] = np.inf
        elif fill == "half_each":
            r[i[:n // 2]], r[i[n // 2:]] = -np.inf, np.inf
        else:
            r[i[:2]] = np.inf
        rows.append(r)
    assert np.signbit(rows[1][np.isnan(rows[1])]).all() and not np.signbit(rows[0][np.isnan(rows[0])]).any()
    return np.stack(rows)


def check_mad(got, ref, rtol=1e-12):
    got, ref = np.asarray(got, dtype=np.float64), np.asarray(ref, dtype=np.float64)
    assert np.array_equal(np.isnan(got), np.isnan(ref)), (got, ref)
    assert np.array_equal(np.isinf(got), np.isinf(ref)), (got, ref)
    fin = np.isfinite(ref)
    np.testing.assert_allclose(got[fin], ref[fin], rtol=rtol, atol=0)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [7, 8, 64, 301, 1200])
def test_mad_with_non_finite_values(n):
    import pybold_b200 as pb
    x = mad_rows(n, n)
    with np.errstate(all="ignore"):
        ref = [orc.mad(r) for r in x]
        ref_daub = [orc.mad_daub_noise_est(r) for r in x]
    assert np.isnan(ref).sum() >= 4                      # NaN, -NaN, most_inf, half_each
    check_mad(pb.noise.mad(dev(x, F64)).cpu().numpy(), ref)
    check_mad(pb.noise.mad_daub_noise_est(dev(x, F64)).cpu().numpy(), ref_daub)
    with np.errstate(all="ignore"):                     # FP32 rows: the medians in double, rounded once
        ref32 = [orc.mad(r) for r in x.astype(np.float32).astype(np.float64)]
    check_mad(pb.noise.mad(dev(x, F32)).cpu().numpy(), ref32, rtol=1e-7)


@pytest.mark.gpu
@pytest.mark.parametrize("T", [9, 64, 301, 1200])
def test_censored_mad_with_non_finite_values(T):
    from pybold_b200.censor import mad_daub_noise_est_censored
    x = mad_rows(T, T + 1)
    cm = censor_rows(len(x), T, 5)
    kept, cens = np.flatnonzero(cm[0] == 0), np.flatnonzero(cm[0] != 0)
    extra = []
    for bad in (np.nan, -np.nan, np.inf):               # at a censored scan: ignored; at a kept scan: like the others
        r = np.random.RandomState(T).randn(T)
        r[cens[len(cens) // 2]] = bad
        extra.append(r)
        r = r.copy()
        r[kept[len(kept) // 2]] = bad
        extra.append(r)
    x = np.concatenate([x, np.stack(extra)])
    cm = np.concatenate([cm, np.repeat(cm[:1], len(extra), axis=0)])
    got = mad_daub_noise_est_censored(dev(x, F64), dev(cm, torch.uint8), T).cpu().numpy()
    with np.errstate(all="ignore"):
        ref = [orc.mad(cref.kept_detail_coefficients(x[v], cm[v])) for v in range(len(x))]
    check_mad(got, ref)
    assert np.isfinite(got[-6]) and np.isnan(got[-5]) and np.isfinite(got[-4]) and np.isnan(got[-3])


# ---- deconv(lbda=None) with a NaN noise level -------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("T,K,dtype", [(300, 20, F64), (600, 20, F32), (1200, 28, F64), (300, 40, F64),
                                       (1500, 28, F32)])
@pytest.mark.parametrize("censored", [False, True])
def test_auto_with_nan_sigma(T, K, dtype, censored):
    """A NaN sigma (given, or from a NaN among the kept scans) gives that voxel the reference's outputs: x, z, diff_z,
    J and lambda NaN, R and G NaN after the first outer iteration, every outer iteration run.  The other voxels are
    bit for bit what they are with a finite sigma in its place, and the call makes no host synchronisation."""
    from pybold_b200 import bold_signal as bs
    y = good_voxels(4, T, T_R[K], 17 * T)
    h, L = taps(K), lipschitz(T, K)
    cm = censor_rows(4, T, 2) if censored else None
    sigma = np.array([0.3, np.nan, 0.5, 0.4])
    yd, hd, sd = dev(y, dtype), dev(h, dtype), dev(sigma, dtype)
    Ld = torch.full((4,), L, dtype=dtype, device="cuda")
    cmd = dev(cm, torch.uint8) if censored else None
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        o = bs.deconv_auto_batch(yd, hd, sd, Ld, censor=cmd, **AUTO)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    o = {k: v.cpu().numpy() for k, v in o.items()}
    fin = bs.deconv_auto_batch(yd, hd, dev(np.where(np.isnan(sigma), 0.6, sigma), dtype), Ld, censor=cmd, **AUTO)
    for k, v in fin.items():
        assert np.array_equal(np.delete(v.cpu().numpy(), 1, axis=0), np.delete(o[k], 1, axis=0), equal_nan=True), k
    assert o["n_outer"][1] == AUTO["nb_iter"]
    for k in ("x", "z", "diff_z", "J", "lbda"):
        assert np.isnan(o[k][1]).all(), k
    for k in ("R", "G"):
        assert np.isfinite(o[k][1, 0]) and np.isnan(o[k][1, 1:]).all(), k
    if dtype == F64:
        np_h = h
        with np.errstate(all="ignore"):
            ref = cref.deconv_auto_lbda(y[1], np_h, np.nan, lipschitz=L, censor=None if cm is None else cm[1], **AUTO)
        x, z, w, J, R, G, lb = ref
        assert len(J) == AUTO["nb_iter"] and np.isnan(lb)
        for a, b in ((o["x"][1], x), (o["z"][1], z), (o["diff_z"][1], w), (o["J"][1], J), (o["R"][1], R),
                     (o["G"][1], G)):
            assert np.array_equal(np.isnan(a), np.isnan(np.asarray(b))), (a, b)
        assert rel(o["R"][1, 0], R[0]) < 1e-9 and rel(o["G"][1, 0], G[0]) < 1e-9


@pytest.mark.gpu
def test_deconv_auto_nan_scan_voxel_is_nan_without_raising():
    """deconv(lbda=None) with the estimated sigma: a voxel with a NaN at a kept scan gets a NaN sigma and NaN outputs,
    with or without censoring, and its neighbours are what they are alone; a NaN at a censored scan is ignored."""
    import pybold_b200 as pb
    T, K = 600, 20
    y = good_voxels(3, T, T_R[K], 23)
    y[1, 100] = np.nan
    x0 = np.random.RandomState(0).randn(T)
    kw = dict(nb_iter=6, nb_sub_iter=20, x0=x0)
    for cm in (None, np.zeros(T, np.uint8), censor_rows(1, T, 0)[0]):
        x, z, dz, J, R, G = pb.deconv(y, T_R[K], taps(K), lbda=None, censor=cm, **kw)
        assert np.isnan(x[1]).all() and np.isfinite(x[[0, 2]]).all()
        xs, *_ = pb.deconv(y[2], T_R[K], taps(K), lbda=None, censor=cm, **kw)
        assert np.array_equal(xs, x[2])
    cm = np.zeros(T, np.uint8)
    cm[100] = 1
    x, *_ = pb.deconv(y, T_R[K], taps(K), lbda=None, censor=cm, **kw)
    assert np.isfinite(x).all()

