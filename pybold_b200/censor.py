"""Scan censoring ("scrubbing") for the deconvolution solvers.

Volumes flagged for head motion must not count in the fit, but a convolution model needs a uniform time grid, so
they stay in the model and leave the data term only::

    min_w  1/2 || M (A w - y) ||^2 + lbda ||w||_1,      M = diag(1 - censor)

``censor`` is a 0/1 mask of the scans to leave out, ``[T]`` (shared by the batch) or ``[V, T]``.  ``y`` is read as 0
on censored scans (NaN there is ignored), ``x = A w`` is returned on every scan.  The Lipschitz constant is
``0.9 x`` the power estimate of ``A^T M A``; the noise level of ``deconv(lbda=None)`` is the db3 MAD over the detail
coefficients that touch no censored scan, and its target ``n_kept sigma^2``.  The solvers take the mask through the
``censor=`` keyword of :func:`~pybold_b200.bold_signal.deconv` and its batch and path variants.
"""
from __future__ import annotations

import numpy as np
import torch

from . import _lib
from ._array import ptr, stream_ptr, to_device


def censor_mask(censor, V, T, device, check=True):
    """``censor`` (NumPy or torch, bool or integer, ``[T]`` or ``[V, T]``; non-zero = leave the scan out) -> (uint8
    device tensor, element stride of the C ABI: 0 shared, T per voxel).

    Raises ``ValueError`` on a shape that is neither, and on a voxel whose every scan is censored (its operator is
    zero).  That check reads the mask on the host: it is free for a host mask, and ``check=False`` skips it for a
    device mask so that the call makes no host synchronisation."""
    on_host = not (isinstance(censor, torch.Tensor) and censor.is_cuda)
    if isinstance(censor, torch.Tensor):
        c = censor.detach()
    else:
        c = torch.from_numpy(np.ascontiguousarray(np.asarray(censor)))
    if c.dtype.is_floating_point or c.dtype.is_complex:
        raise ValueError("censor must be a bool or integer mask, got %s" % c.dtype)
    if c.dim() == 2 and c.shape[0] == 1 and V != 1:
        c = c[0]
    if c.dim() == 1 and c.shape[0] == T:
        stride = 0
    elif c.dim() == 2 and tuple(c.shape) == (V, T):
        stride = T
    elif c.dim() == 2 and V == 1 and tuple(c.shape) == (1, T):
        stride = 0
    else:
        raise ValueError("censor must be [T] (shared) or [V, T] with V = %d voxels and T = %d scans, got %s"
                         % (V, T, tuple(c.shape)))
    c = c != 0
    if (on_host or check) and bool(c.reshape(-1, T).all(dim=1).any()):
        raise ValueError("censor leaves a voxel with every scan censored: its operator is zero, nothing to fit")
    return c.to(device=device, dtype=torch.uint8).contiguous(), stride


def lipschitz_censored(h, x0, cm, c_stride, dtype, T):
    """``0.9 x`` the power estimate of ``A^T M A`` (the rule of bold_signal.py:52 applied to the censored operator),
    from the start ``x0`` shared by every voxel; one constant per mask row and taps row.  Returns (tensor, stride)."""
    hd = to_device(h, dtype)
    k2 = hd.reshape(1, -1) if hd.dim() == 1 else hd
    xd = to_device(x0, dtype).reshape(1, -1)
    V = max(k2.shape[0], cm.shape[0] if c_stride else 1)
    K = k2.shape[1]
    out = torch.empty(V, dtype=dtype, device=xd.device)
    with torch.cuda.device(xd.device):
        rc = _lib.fn("pb_lipschitz_power_censored", dtype)(
            ptr(k2), K if k2.shape[0] > 1 else 0, ptr(xd), 0, ptr(cm), c_stride, 30, 1.0e-6, ptr(out), V, T, K,
            stream_ptr())
    _lib.check(rc, "pb_lipschitz_power_censored")
    L = (0.9 * out.double()).to(dtype)
    return (L, 0) if V == 1 else (L, 1)


def mad_daub_noise_est_censored(yb, cm, c_stride, c=0.6744):
    """db3 MAD noise level of every row of ``yb`` ``[V, T]`` over the level-1 detail coefficients that touch no
    censored scan.  Raises ``ValueError`` when a voxel has no such coefficient: pass ``sigma=`` then.  A voxel with a
    NaN or an Inf among its kept scans may get a NaN sigma, like NumPy's median gives; that is not an error, and such
    a voxel gets NaN without the error even when it has no clean coefficient either (its fit is NaN whatever sigma
    is)."""
    V, T = yb.shape
    out = torch.empty(V, dtype=yb.dtype, device=yb.device)
    with torch.cuda.device(yb.device):
        rc = _lib.fn("pb_mad_daub_noise_est_censored", yb.dtype)(ptr(yb), ptr(cm), c_stride, float(c), ptr(out), V, T,
                                                                  stream_ptr())
    _lib.check(rc, "pb_mad_daub_noise_est_censored")
    # with finite kept scans every kept coefficient is finite: a NaN sigma then means that none was left
    finite_kept = (torch.isfinite(yb) | (cm != 0)).all(dim=1)
    if bool((torch.isnan(out) & finite_kept).any()):
        raise ValueError("censor leaves no db3 detail coefficient free of censored scans in some voxel, so the "
                         "noise level cannot be estimated: pass sigma=")
    return out
