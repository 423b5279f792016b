"""``deconv(lbda=None)``: noise-constrained regularisation (pybold/bold_signal.py:99-214).

Row N1 of SURVEY.md 8(f).  The whole loop -- inner prox-gradient passes and the scalar alpha / lambda update of
every outer iteration -- runs per voxel inside the persistent deconv kernels (``pb_deconv_auto``,
csrc/pb_noise_loop.cuh): one launch per call.

The noise level sigma is the MAD of the level-1 db3 detail coefficients in the reference
(pybold/utils.py:10-25, PyWavelets); here one kernel (``pb_mad_daub_noise_est_*``).  The loop itself
is pinned on the live reference with sigma injected (tests/golden/deconv_auto.npz); the wavelet
convention is pinned on PyWavelets' documented Haar examples only (PyWavelets is not installed where
this was built) -- pass ``sigma=`` to ``deconv`` to bypass it.
"""
from __future__ import annotations

import torch

from . import _lib
from ._array import like_input, pick_dtype, ptr, stream_ptr, to_device

# the analysis high-pass the kernel applies (csrc/pb_noise.cuh holds the same six numbers)
_DB3_DEC_HI = (-0.3326705529509569, 0.8068915093133388, -0.4598775021193313,
               -0.13501102001039084, 0.08544127388224149, 0.035226291882100656)


_warned_sigma = False


def _mad_rows(x, c, entry):
    dtype = pick_dtype(x)
    xd = to_device(x, dtype)
    one_d = xd.dim() <= 1
    x2 = xd.reshape(1, -1) if one_d else xd.reshape(xd.shape[0], -1)
    V, n = x2.shape
    if n == 0:
        raise ValueError("%s: empty series" % entry)
    out = torch.empty(V, dtype=dtype, device=x2.device)
    with torch.cuda.device(x2.device):
        rc = _lib.fn(entry, dtype)(ptr(x2), float(c), ptr(out), V, n, stream_ptr())
    _lib.check(rc, entry)
    if one_d:
        return float(out[0])
    return like_input(out, x)


def mad(x, c=0.6744):
    """Median absolute deviation ``median(|x - median(x)|) / c`` (pybold/utils.py:10-13).

    A 1-D array (NumPy or torch) gives a float like the reference; a ``[V, n]`` batch gives one
    value per row.  Exact order statistics on the device (``pb_mad_*``).
    """
    return _mad_rows(x, c, "pb_mad")


def mad_daub_noise_est(x, c=0.6744):
    """Noise level from the MAD of the level-1 db3 detail coefficients (pybold/utils.py:16-25),
    1-D -> float, ``[V, T]`` -> one sigma per voxel (``pb_mad_daub_noise_est_*``).

    The wavelet step follows PyWavelets' ``wavedec(x, 'db3', level=1)`` convention (symmetric
    extension); PyWavelets is not installed where this was built, so that convention is pinned on
    PyWavelets' documented Haar examples and on the defining properties of the db3 filter only
    (tests/test_boundary.py), not on a PyWavelets db3 output.
    """
    return _mad_rows(x, c, "pb_mad_daub_noise_est")


def deconv_auto_lbda(y_in, yb, one_d, hrf, lipschitz, sigma, early_stopping, tol, wind,
                     nb_iter, nb_sub_iter, censor=None):
    """``deconv(lbda=None)`` (pybold/bold_signal.py:99-214) for a batch: the noise level (given, or estimated
    like the reference does), then the whole noise-constrained loop of every voxel in ONE persistent kernel
    launch (:func:`~pybold_b200.bold_signal.deconv_auto_batch`): outer iterations, alpha / lambda updates, the
    alpha-window stop and the final inner pass all run on the device, nothing goes through the host between
    outer iterations.  Returns the reference's tuple (x, z, diff_z, J, R, G): lists for one voxel, rows cut at
    the largest outer count (NaN past each voxel's own) for a batch.  ``censor``: a uint8 device mask from
    :func:`~pybold_b200.censor.censor_mask`; sigma then comes from the detail coefficients that touch no censored scan.
    """
    from .bold_signal import deconv_auto_batch
    if sigma is None:
        # bold_signal.py:103.  The wavelet convention of this estimate could not be compared with PyWavelets
        # itself (see mad_daub_noise_est): say so once, `sigma=` makes the run independent of it
        global _warned_sigma
        if not _warned_sigma:
            import warnings
            warnings.warn("pybold_b200.deconv(lbda=None): sigma comes from the on-device db3 MAD estimate, whose "
                          "boundary convention is pinned on PyWavelets' documented examples only; pass sigma= for "
                          "a run that does not depend on it", UserWarning, stacklevel=3)
            _warned_sigma = True
        if censor is None:
            sigma = mad_daub_noise_est(yb)
        else:
            from .censor import mad_daub_noise_est_censored
            sigma = mad_daub_noise_est_censored(yb, censor, 0 if censor.dim() == 1 else yb.shape[1])
    out = deconv_auto_batch(yb, hrf, sigma, lipschitz, nb_iter, nb_sub_iter, early_stopping, tol, wind,
                            censor=censor)
    x, z, w, J, R, G = (out[k] for k in ("x", "z", "diff_z", "J", "R", "G"))
    if one_d:
        n = int(out["n_outer"][0])
        conv = lambda t: like_input(t[0], y_in)  # noqa: E731
        return (conv(x), conv(z), conv(w), [float(v) for v in J[0, :n]], [float(v) for v in R[0, :n]],
                [float(v) for v in G[0, :n]])
    n_max = int(out["n_outer"].max())
    conv = lambda t: like_input(t, y_in)  # noqa: E731
    return conv(x), conv(z), conv(w), conv(J[:, :n_max]), conv(R[:, :n_max]), conv(G[:, :n_max])
