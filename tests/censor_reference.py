"""Dense float64 statement of scan censoring for the deconvolution solvers (pybold_b200/censor.py).

The pinned oracle (oracle/pybold_oracle.py) has no censoring; these functions restate its ``deconv_fixed_lbda``,
``deconv_auto_lbda``, ``spectral_radius_est`` and ``mad_daub_noise_est`` with the mask M = diag(1 - censor):

    min_w  1/2 || M (A w - y) ||^2 + lbda ||w||_1

y is read as 0 on censored scans, the gradient is A^T M (A w - y), every cost term uses the masked residual,
x = A w on every scan, the Lipschitz constant is 0.9 x the power estimate of A^T M A, and deconv(lbda=None) targets
n_kept sigma^2.  With an all-zero mask every function returns the oracle's outputs bit for bit
(tests/test_censor_reference.py), which ties the censored path to the pinned one.
"""
import math

import numpy as np

from oracle import pybold_oracle as orc


def _keep(censor, T):
    keep = np.ones(T, dtype=bool) if censor is None else np.asarray(censor).reshape(T) == 0
    return keep


def _masked(keep, r):
    return np.where(keep, r, 0.0)


class CensoredOperator:
    """``M A`` with ``A = HrfIntegOperator``: op = M K cumsum(x), adj = revcumsum(K^T M x)."""

    def __init__(self, hrf, keep):
        self.H = orc.HrfIntegOperator(hrf, len(keep))
        self.keep = keep

    def op(self, x):
        return _masked(self.keep, self.H.op(x))

    def adj(self, x):
        return self.H.adj(_masked(self.keep, x))


def spectral_radius_est(hrf, x0, censor=None, nb_iter=30, tol=1.0e-6):
    """Power estimate of ``A^T M A`` from ``x0`` (the oracle's iteration on the censored operator)."""
    keep = _keep(censor, len(x0))
    return orc.spectral_radius_est(CensoredOperator(hrf, keep), x0, nb_iter, tol)


def deconv_fixed_lbda(y, hrf, lbda, x0_power=None, lipschitz=None, early_stopping=True,
                      tol=1.0e-6, wind=6, nb_iter=1000, censor=None):
    """``oracle.deconv_fixed_lbda`` with ``censor``.  Returns (x, z, w, J / (J[0] + 1e-30), n_done)."""
    y = np.asarray(y, dtype=np.float64)
    T = len(y)
    keep = _keep(censor, T)
    y0 = np.where(keep, y, 0.0)
    H = orc.HrfIntegOperator(hrf, T)
    Aty = H.adj(y0)
    if lipschitz is None:
        lipschitz = 0.9 * spectral_radius_est(hrf, x0_power, censor)
    step = 1.0 / lipschitz
    th = lbda / lipschitz
    w = np.zeros(T)
    t_old = 1.0
    J = []
    hist = []
    sub = int(wind / 2)
    x = z = None
    for k in range(nb_iter):
        grad = H.adj(_masked(keep, H.op(w))) - Aty
        u = w - step * grad
        v = orc._soft(u, th)
        t = 0.5 * (1.0 + math.sqrt(1.0 + 4.0 * t_old * t_old))
        p = np.zeros(T) if k == 0 else u
        w = v + (t_old - 1.0) / t * (v - p)
        t_old = t
        z = np.cumsum(w)
        x = orc.conv_causal(hrf, z)
        J.append(0.5 * np.sum(np.square(_masked(keep, x - y0))) + lbda * np.sum(np.abs(w)))
        if hist:
            hist[-1] = u
        hist.append(w)
        if len(hist) > wind:
            hist = hist[1:]
        if early_stopping and k > wind:
            old_iter = np.mean(hist[:-sub], axis=0)
            new_iter = np.mean(hist[-sub:], axis=0)
            crit = np.linalg.norm(new_iter - old_iter) / (np.linalg.norm(new_iter) + 1.0e-10)
            if crit < tol:
                break
    J = np.array(J)
    return x, z, w, J / (J[0] + 1.0e-30), len(J)


def deconv_auto_lbda(y, hrf, sigma, x0_power=None, lipschitz=None, early_stopping=True,
                     tol=1.0e-6, wind=6, nb_iter=1000, nb_sub_iter=1000, censor=None):
    """``oracle.deconv_auto_lbda`` with ``censor``: target ``n_kept sigma^2``.  Returns (x, z, w, J, R, G, lbda)."""
    y = np.asarray(y, dtype=np.float64)
    T = len(y)
    keep = _keep(censor, T)
    n_kept = int(np.count_nonzero(keep)) if censor is not None else T
    y0 = np.where(keep, y, 0.0)
    H = orc.HrfIntegOperator(hrf, T)
    Aty = H.adj(y0)
    if lipschitz is None:
        lipschitz = 0.9 * spectral_radius_est(hrf, x0_power, censor)
    step = 1.0 / lipschitz
    sub = int(wind / 2)
    state = {'w': np.zeros(T), 'p': np.zeros(T)}

    def inner(lbda):
        th = lbda / lipschitz
        w = state['w']
        p_prev = state['p']
        t_old = 1.0
        hist = []
        for j in range(nb_sub_iter):
            u = w - step * (H.adj(_masked(keep, H.op(w))) - Aty)
            v = orc._soft(u, th)
            t = 0.5 * (1.0 + math.sqrt(1.0 + 4.0 * t_old * t_old))
            p = p_prev if j == 0 else u
            w = v + (t_old - 1.0) / t * (v - p)
            t_old = t
            if hist:
                hist[-1] = u
            hist.append(w)
            if len(hist) > wind:
                hist = hist[1:]
            if early_stopping and j > wind:
                old_iter = np.mean(hist[:-sub], axis=0)
                new_iter = np.mean(hist[-sub:], axis=0)
                crit = (np.linalg.norm(new_iter - old_iter)
                        / (np.linalg.norm(new_iter) + 1.0e-10))
                if crit < tol:
                    break
        state['w'] = w
        state['p'] = w

    l_alpha, J, R, G = [], [], [], []
    alpha = 1.0
    lbda = 1.0 / (2.0 * alpha)
    mu = 1.0e-4
    for i in range(nb_iter):
        inner(lbda)
        w = state['w']
        z = np.cumsum(w)
        x = orc.conv_causal(hrf, z)
        grad = np.sum(np.square(_masked(keep, x - y0))) - n_kept * sigma ** 2
        alpha += mu * grad
        lbda = 1.0 / (2.0 * alpha)
        l_alpha.append(alpha)
        if len(l_alpha) > wind:
            l_alpha = l_alpha[1:]
        r = np.sum(np.square(_masked(keep, x - y0)))
        g = np.sum(np.abs(w))
        R.append(r)
        G.append(g)
        J.append(0.5 * r + lbda * g)
        if early_stopping and i > wind:
            old_iter = np.mean(l_alpha[:-sub])
            new_iter = np.mean(l_alpha[-sub:])
            if abs(new_iter - old_iter) / abs(new_iter) < tol:
                break
    inner(lbda)
    w = state['w']
    z = np.cumsum(w)
    x = orc.conv_causal(hrf, z)
    return x, z, w, J, R, G, lbda


def kept_detail_coefficients(y, censor):
    """The level-1 db3 detail coefficients (the oracle's convention) whose six samples, after the symmetric extension,
    are all kept; for T < 10 the kept samples themselves."""
    y = np.asarray(y, dtype=np.float64)
    T = len(y)
    keep = _keep(censor, T)
    if T < 10:
        return y[keep]
    cD = orc.db3_detail_level1(np.where(keep, y, 0.0))
    ok = np.ones(len(cD), dtype=bool)
    for o in range(len(cD)):
        for j in range(6):
            i = 2 * o + 1 - j
            i = -i - 1 if i < 0 else (2 * T - 1 - i if i >= T else i)
            ok[o] &= bool(keep[i])
    return cD[ok]


def mad_daub_noise_est(y, censor=None, c=0.6744):
    """db3 MAD over the kept detail coefficients (``oracle.mad_daub_noise_est`` when nothing is censored)."""
    if censor is None or not np.any(censor):
        return orc.mad_daub_noise_est(y, c)
    return orc.mad(kept_detail_coefficients(y, censor), c)
