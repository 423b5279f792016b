"""Batched device solvers behind the signatures of ``pybold/bold_signal.py``.

``deconv`` and ``bd`` keep the reference's arguments, defaults and return tuples for a 1-D
voxel; a ``[V, T]`` input solves V voxels in ONE persistent kernel launch (the reference
fans out one process per voxel with joblib, examples/icassp_2019/validation.py:43-47).
NumPy in -> NumPy out (float64 unless everything passed is float32); torch CUDA tensors in ->
torch tensors out with no host round trip.

Deliberate, documented differences from the reference:
 * nothing is printed per iteration (the reference prints unconditionally, bold_signal.py:79-80);
 * the theta step is an exact bounded 1-D minimisation instead of SciPy's finite-difference
   L-BFGS-B (bold_signal.py:329-333): the two agree to ~1e-7 on theta (DESIGN.md, parity);
 * ``deconv`` needs the power-iteration start: it is drawn from ``np.random`` exactly like the
   reference (utils.py:97) unless ``x0=`` is passed.
"""
from __future__ import annotations

import numpy as np
import torch

from . import _lib
from ._array import like_input, per_voxel, pick_dtype, ptr, stream_ptr, to_device, upload
from .hrf_model import MAX_DELTA, MIN_DELTA, hrf_len
from .linear import ConvAndLinear, DiscretInteg
from .utils import spectral_radius_est


def _as_batch(y, dtype):
    yd = to_device(y, dtype)
    if yd.dim() == 1:
        return yd.reshape(1, -1), True
    if yd.dim() != 2:
        raise ValueError("y must be 1-D (one voxel) or [V, T]")
    return yd, False


def deconv_batch(y, hrf, lbda, lipschitz, w0=None, early_stopping=True, tol=1.0e-6, wind=6,
                 nb_iter=1000, events=None, active=None, out=None, trace=True, censor=None):
    """Device entry point: tensors in, tensors out.  Returns (x, z, diff_z, J_raw, n_iter).

    ``J_raw[v, k]`` is the un-normalised cost of iteration k (NaN past ``n_iter[v]``);
    ``lipschitz`` is the constant actually used (0.9 x power estimate in ``deconv``).
    ``events=(e0, e1)``: CUDA events recorded immediately around the solver launch (benchmarks).
    ``active`` (uint8 ``[V]``): voxels with 0 are skipped, their rows of the outputs stay as they are;
    ``out=(x, z, diff_z, n_iter)`` reuses output tensors; ``trace=False`` skips the cost trace (J is None).
    ``censor`` (``[T]`` or ``[V, T]``, non-zero = scan left out of the data term, :mod:`pybold_b200.censor`): J is
    the cost of the masked residual and ``lipschitz`` should be the censored operator's; it does not combine with
    ``active``.  A device mask is not checked for all-censored voxels (that would wait on the device).
    """
    V, T = y.shape
    dtype, dev = y.dtype, y.device
    hrf = hrf.to(device=dev, dtype=dtype).contiguous()
    K = hrf.shape[-1]
    if hrf.dim() > 2 or (hrf.dim() == 2 and hrf.shape[0] not in (1, V)):
        raise ValueError("hrf must be [K] (shared) or [V, K] with V = %d voxels, got %s"
                         % (V, tuple(hrf.shape)))
    h_stride = 0 if hrf.dim() == 1 or hrf.shape[0] == 1 else K
    if w0 is not None:
        if tuple(w0.shape) != (V, T) or w0.dtype != dtype or w0.device != dev:
            raise ValueError("w0 must be a %s tensor of shape (%d, %d) on %s" % (dtype, V, T, dev))
        w0 = w0.contiguous()
    y = y.contiguous()
    lb, lb_stride = per_voxel(lbda, V, dtype, dev, "lbda")
    Lc, L_stride = per_voxel(lipschitz, V, dtype, dev, "lipschitz")
    if out is not None:
        x, z, dz, n_iter = out
        for t in (x, z, dz):
            if tuple(t.shape) != (V, T) or t.dtype != dtype or t.device != dev or not t.is_contiguous():
                raise ValueError("out tensors must be contiguous %s tensors of shape (%d, %d) on %s" % (dtype, V, T, dev))
    else:
        x = torch.empty_like(y)
        z = torch.empty_like(y)
        dz = torch.empty_like(y)
        n_iter = torch.zeros(V, dtype=torch.int32, device=dev)
    J = torch.full((V, nb_iter), float("nan"), dtype=dtype, device=dev) if trace else None
    if active is not None and (active.dtype != torch.uint8 or active.numel() != V or active.device != dev):
        raise ValueError("active must be a uint8 tensor with one entry per voxel on %s" % dev)
    if censor is not None:
        from .censor import censor_mask
        if active is not None:
            raise ValueError("censor does not combine with active")
        cm, c_stride = censor_mask(censor, V, T, dev, check=False)
        if J is None:                   # the censored entry always writes a trace
            J_buf = torch.empty((V, nb_iter), dtype=dtype, device=dev)
    with torch.cuda.device(dev):        # the C side sizes its grid for, and launches on, the current device
        if events is not None:
            events[0].record()
        if censor is not None:
            rc = _lib.fn("pb_deconv_censored", dtype)(
                ptr(y), ptr(hrf), h_stride, ptr(Lc), L_stride, ptr(lb), lb_stride, ptr(w0), ptr(cm), c_stride,
                int(nb_iter), int(bool(early_stopping)), int(wind), float(tol),
                ptr(x), ptr(z), ptr(dz), ptr(J if J is not None else J_buf), ptr(n_iter), V, T, K, stream_ptr())
        elif active is None and trace:
            rc = _lib.fn("pb_deconv", dtype)(
                ptr(y), ptr(hrf), h_stride, ptr(Lc), L_stride, ptr(lb), lb_stride, ptr(w0),
                int(nb_iter), int(bool(early_stopping)), int(wind), float(tol),
                ptr(x), ptr(z), ptr(dz), ptr(J), ptr(n_iter), V, T, K, stream_ptr())
        else:
            rc = _lib.fn("pb_deconv_masked", dtype)(
                ptr(y), ptr(hrf), h_stride, ptr(Lc), L_stride, ptr(lb), lb_stride, ptr(w0), ptr(active),
                int(nb_iter), int(bool(early_stopping)), int(wind), float(tol),
                ptr(x), ptr(z), ptr(dz), ptr(J), ptr(n_iter), V, T, K, stream_ptr())
        if events is not None:
            events[1].record()
    _lib.check(rc, "pb_deconv")
    return x, z, dz, J, n_iter


def deconv_auto_batch(y, hrf, sigma, lipschitz, nb_iter=1000, nb_sub_iter=1000, early_stopping=True, tol=1.0e-6,
                      wind=6, censor=None):
    """Device entry point of ``deconv(lbda=None)`` (pybold/bold_signal.py:99-214): tensors in, dict of tensors out.

    ``y`` is ``[V, T]`` on the device, ``hrf`` ``[K]`` (shared) or ``[V, K]``, ``sigma`` (noise level) and
    ``lipschitz`` scalars or ``[V]``.  Every voxel runs its whole outer loop -- at most ``nb_iter`` outer iterations
    of at most ``nb_sub_iter`` inner ones, then the final inner pass -- inside ONE persistent kernel launch
    (``pb_deconv_auto_*``); with every input already on the device the call makes no host synchronisation.

    Returns ``{x, z, diff_z}`` (``[V, T]``, final pass), ``{J, R, G}`` (``[V, nb_iter]``, one entry per outer
    iteration, NaN past the voxel's outer count), ``lbda`` (``[V]``, the lambda of the final pass) and
    ``n_outer`` (``[V]`` int32, outer iterations done).

    ``censor`` (``[T]`` or ``[V, T]``, :mod:`pybold_b200.censor`): R is ``||M (x - y)||^2`` and the noise target
    ``n_kept sigma^2``; a device mask keeps the call free of host synchronisation (it is then not checked for
    all-censored voxels).

    A voxel whose sigma is NaN (the estimate is NaN when a NaN is among the kept scans, like NumPy's median) gets the
    reference's result: x, z, diff_z, J and lbda NaN, R and G NaN after the first outer iteration, and all
    ``nb_iter`` outer iterations.  The other voxels are not affected.
    """
    V, T = y.shape
    dtype, dev = y.dtype, y.device
    hrf = hrf.to(device=dev, dtype=dtype).contiguous()
    K = hrf.shape[-1]
    if hrf.dim() > 2 or (hrf.dim() == 2 and hrf.shape[0] not in (1, V)):
        raise ValueError("hrf must be [K] (shared) or [V, K] with V = %d voxels, got %s"
                         % (V, tuple(hrf.shape)))
    h_stride = 0 if hrf.dim() == 1 or hrf.shape[0] == 1 else K
    y = y.contiguous()
    sg, sg_stride = per_voxel(sigma, V, dtype, dev, "sigma")
    Lc, L_stride = per_voxel(lipschitz, V, dtype, dev, "lipschitz")
    out = {k: torch.empty((V, T), dtype=dtype, device=dev) for k in ("x", "z", "diff_z")}
    out.update({k: torch.empty((V, nb_iter), dtype=dtype, device=dev) for k in ("J", "R", "G")})
    out["lbda"] = torch.empty(V, dtype=dtype, device=dev)
    out["n_outer"] = torch.empty(V, dtype=torch.int32, device=dev)
    if censor is not None:
        from .censor import censor_mask
        cm, c_stride = censor_mask(censor, V, T, dev, check=False)
        with torch.cuda.device(dev):
            rc = _lib.fn("pb_deconv_auto_censored", dtype)(
                ptr(y), ptr(hrf), h_stride, ptr(Lc), L_stride, ptr(sg), sg_stride, ptr(cm), c_stride, int(nb_iter),
                int(nb_sub_iter), int(bool(early_stopping)), int(wind), float(tol), ptr(out["x"]), ptr(out["z"]),
                ptr(out["diff_z"]), ptr(out["J"]), ptr(out["R"]), ptr(out["G"]), ptr(out["lbda"]),
                ptr(out["n_outer"]), V, T, K, stream_ptr())
        _lib.check(rc, "pb_deconv_auto_censored")
        return out
    with torch.cuda.device(dev):
        rc = _lib.fn("pb_deconv_auto", dtype)(
            ptr(y), ptr(hrf), h_stride, ptr(Lc), L_stride, ptr(sg), sg_stride, int(nb_iter), int(nb_sub_iter),
            int(bool(early_stopping)), int(wind), float(tol), ptr(out["x"]), ptr(out["z"]), ptr(out["diff_z"]),
            ptr(out["J"]), ptr(out["R"]), ptr(out["G"]), ptr(out["lbda"]), ptr(out["n_outer"]), V, T, K,
            stream_ptr())
    _lib.check(rc, "pb_deconv_auto")
    return out


def _lipschitz_cst(est, dtype):
    """``0.9 * spectral_radius_est`` (bold_signal.py:52), the product taken in double like the reference does
    and rounded once to the build's type: the same constant on every path that solves the same problem."""
    if isinstance(est, torch.Tensor):
        return (0.9 * est.double()).to(dtype)
    est = np.asarray(est, dtype=np.float64)
    return 0.9 * float(est) if est.ndim == 0 else 0.9 * est       # scalars stay host floats (cached on the device)


def deconv(y, t_r, hrf, lbda=None, early_stopping=True, tol=1.0e-6,  # noqa
           wind=6, nb_iter=1000, nb_sub_iter=1000, verbose=0, x0=None, sigma=None, dtype=None, censor=None):
    """Sparse deconvolution with a known HRF (pybold/bold_signal.py:13-214).

    Returns ``(x, z, diff_z, J, R, G)`` like the reference: with a float ``lbda`` J is the cost
    trace normalised by its first entry and R, G are None (bold_signal.py:97).  ``lbda=None``
    (noise-constrained lambda, bold_signal.py:99-214) estimates the noise level like the reference
    (db3 MAD, utils.py:16-25, on the device) unless ``sigma=`` is given.
    Extra keyword arguments: ``x0`` (power-iteration start), ``sigma``, ``dtype``, ``censor``.  float64 input
    (the reference's type) selects the FP64 build, float32 input or ``dtype=np.float32`` the FP32 one.

    ``censor`` (``[T]`` or ``[V, T]`` 0/1 mask, NumPy or torch; :mod:`pybold_b200.censor`) leaves the flagged scans
    out of the data term: ``J = 1/2 ||M (A w - y)||^2 + lbda ||w||_1``, y may hold NaN there, x = A w on every scan,
    the Lipschitz constant is the censored operator's, and ``lbda=None`` targets ``n_kept sigma^2`` with sigma from
    the detail coefficients that touch no censored scan.  ``ValueError`` for a voxel with every scan censored.
    """
    dtype = pick_dtype(y, hrf, dtype=dtype)
    yb, one_d = _as_batch(y, dtype)
    V, T = yb.shape
    hd = to_device(hrf, dtype)
    H = ConvAndLinear(DiscretInteg(), hd, dim_in=T, dim_out=T)
    # bold_signal.py:52 -- 0.9 x power-iteration estimate, start vector from the global RNG
    if x0 is None:
        x0 = np.random.randn(T)
    cm = None
    if censor is not None:
        from .censor import censor_mask, lipschitz_censored
        cm, c_stride = censor_mask(censor, V, T, yb.device)
        lipschitz, _ = lipschitz_censored(hd, x0, cm, c_stride, dtype, T)
    else:
        est = spectral_radius_est(H, (T,), x0=to_device(x0, dtype))
        lipschitz = _lipschitz_cst(est, dtype)

    if lbda is None:
        from .noise import deconv_auto_lbda
        return deconv_auto_lbda(y, yb, one_d, hd, lipschitz, sigma, early_stopping, tol, wind,
                                nb_iter, nb_sub_iter, censor=cm)

    x, z, dz, J, n_iter = deconv_batch(yb, hd, lbda, lipschitz, None, early_stopping, tol, wind,
                                       nb_iter, censor=cm)
    Jn = J / (J[:, :1] + 1.0e-30)                                  # bold_signal.py:97
    if one_d:
        n = int(n_iter[0])
        return (like_input(x[0], y), like_input(z[0], y), like_input(dz[0], y),
                like_input(Jn[0, :n], y), None, None)
    return (like_input(x, y), like_input(z, y), like_input(dz, y), like_input(Jn, y), None, None)


# deconv_lbda_path_fit keeps no solution: each launch writes its (x, z, diff_z) into one scratch of at most this
# many bytes, reused voxel range after voxel range.  4 GiB holds about 290 000 (lambda, voxel) problems at 1200
# scans in FP32 (580 000 at 600): tens of waves of the persistent grid per launch, so the partly idle end of each
# launch (early-stopped problems finish at different times) costs a few per cent at most, while the scratch stays
# small beside the 180 GB of the card and a whole-brain y (1.1 GB at 230 000 x 1200 in FP32).
FIT_SCRATCH_BYTES = 4 << 30


def _path_problem(y, hrf, lbdas, x0, dtype, censor=None):
    """Device inputs of the regularisation path: the rows of ``y``, the taps (``[K]`` shared or ``[V, K]``), the
    Lipschitz constants ``0.9 x spectral_radius_est`` from ``x0`` -- per voxel with ``[V, K]`` taps, the constants
    ``deconv(y, t_r, hrf, x0=x0)`` uses -- and the lambdas, with the element strides of the C ABI.  With ``censor``
    also the mask and its stride, and the constants of the censored operators."""
    dtype = pick_dtype(y, hrf, dtype=dtype)
    yb, _ = _as_batch(y, dtype)
    yb = yb.contiguous()
    V, T = yb.shape
    hd = to_device(hrf, dtype)
    if hd.dim() > 2 or (hd.dim() == 2 and hd.shape[0] not in (1, V)):
        raise ValueError("hrf must be [K] (shared) or [V, K] with V = %d voxels, got %s"
                         % (V, tuple(hd.shape)))
    if hd.dim() == 2 and hd.shape[0] == 1:
        hd = hd[0]
    hd = hd.contiguous()
    h_stride = hd.shape[-1] if hd.dim() == 2 else 0
    lb = upload(np.asarray(lbdas, dtype=np.float64).reshape(-1), dtype, yb.device)
    if x0 is None:
        x0 = np.random.randn(T)
    if censor is not None:
        from .censor import censor_mask, lipschitz_censored
        cm, c_stride = censor_mask(censor, V, T, yb.device)
        Lc, L_stride = lipschitz_censored(hd, x0, cm, c_stride, dtype, T)
        return yb, hd, h_stride, Lc, L_stride, lb, (cm, c_stride)
    est = spectral_radius_est(ConvAndLinear(DiscretInteg(), hd, dim_in=T), (T,), x0=to_device(x0, dtype))
    Lc, L_stride = per_voxel(_lipschitz_cst(est, dtype), V, dtype, yb.device, "lipschitz")
    return yb, hd, h_stride, Lc, L_stride, lb, None


def _path_launch(yb, hd, h_stride, Lc, L_stride, lb, nb_iter, early_stopping, wind, tol, sol, J, r, g, n_iter,
                 censor=None):
    """One ``pb_deconv_lbda_path_ex`` launch: every lambda of ``lb`` x every row of ``yb``, problem (l, v) at
    flat index l * V + v of the outputs.  ``sol`` = (x, z, diff_z) buffers of n_lbda * V * T elements; ``J``
    (n_lbda * V * nb_iter), ``r`` and ``g`` may be None; ``n_iter`` holds n_lbda * V int32.  ``censor`` = (mask,
    stride) of the rows of ``yb``: ``pb_deconv_lbda_path_censored`` instead."""
    V, T = yb.shape
    if censor is not None:
        with torch.cuda.device(yb.device):
            rc = _lib.fn("pb_deconv_lbda_path_censored", yb.dtype)(
                ptr(yb), ptr(hd), h_stride, ptr(Lc), L_stride, ptr(lb), lb.numel(), ptr(censor[0]), censor[1],
                int(nb_iter), int(bool(early_stopping)), int(wind), float(tol), ptr(sol[0]), ptr(sol[1]),
                ptr(sol[2]), ptr(J), ptr(r), ptr(g), ptr(n_iter), V, T, hd.shape[-1], stream_ptr())
        _lib.check(rc, "pb_deconv_lbda_path_censored")
        return
    with torch.cuda.device(yb.device):
        rc = _lib.fn("pb_deconv_lbda_path_ex", yb.dtype)(
            ptr(yb), ptr(hd), h_stride, ptr(Lc), L_stride, ptr(lb), lb.numel(), int(nb_iter),
            int(bool(early_stopping)), int(wind), float(tol), ptr(sol[0]), ptr(sol[1]), ptr(sol[2]),
            ptr(J), ptr(r), ptr(g), ptr(n_iter), V, T, hd.shape[-1], stream_ptr())
    _lib.check(rc, "pb_deconv_lbda_path_ex")


def deconv_lbda_path(y, t_r, hrf, lbdas, nb_iter=200, x0=None, dtype=None, max_problems=1 << 21,
                     early_stopping=False, tol=1.0e-6, wind=6, censor=None):
    """Regularisation path: ``deconv(y, t_r, hrf, lbda=l, nb_iter=nb_iter, x0=x0, early_stopping=...,
    tol=..., wind=...)`` for every lambda of ``lbdas`` and every voxel of ``y[V, T]`` -- the grid search of
    examples/icassp_2019/validation.py batched over (lambda, voxel) instead of looping (BASELINE.json configs[4]).

    ``hrf`` is ``[K]`` (shared) or ``[V, K]`` (one HRF per voxel, e.g. from ``bd``); with ``[V, K]`` the
    Lipschitz constants are per voxel, from the same ``x0``.  Early stopping is off by default (the cfg5 grid
    runs every iteration); with ``early_stopping=True`` each problem stops like the reference's ``deconv``.

    Returns ``(x, z, diff_z, J)`` with a leading lambda axis: ``[n_lbda, V, T]`` and
    ``[n_lbda, V, nb_iter]`` (J normalised by its first entry like ``deconv``, NaN past a problem's stop
    iteration).  Every (lambda, voxel) pair is an independent problem of ONE persistent launch
    (``pb_deconv_lbda_path_ex_*``) that reads the rows of ``y`` in place -- nothing is replicated per lambda --
    and writes straight into the results; more than ``max_problems`` pairs are cut into launches of whole
    lambdas.  The solutions take ``3 n_lbda V T`` elements on the device: to choose lambda at whole-brain size,
    use :func:`deconv_lbda_path_fit`.

    ``censor`` (``[T]`` or ``[V, T]``): every problem is the censored ``deconv(..., censor=censor)`` of its voxel.
    """
    yb, hd, h_stride, Lc, L_stride, lb, cz = _path_problem(y, hrf, lbdas, x0, dtype, censor)
    V, T = yb.shape
    n_l = lb.numel()
    outs = [torch.empty((n_l, V, T), dtype=yb.dtype, device=yb.device) for _ in range(3)]
    if early_stopping:
        J = torch.full((n_l, V, nb_iter), float("nan"), dtype=yb.dtype, device=yb.device)
    else:                                                         # every entry is written
        J = torch.empty((n_l, V, nb_iter), dtype=yb.dtype, device=yb.device)
    n_iter = torch.empty((n_l, V), dtype=torch.int32, device=yb.device)
    per = max(1, min(n_l, max_problems // max(V, 1)))
    for l0 in range(0, n_l, per):
        l1 = min(l0 + per, n_l)
        _path_launch(yb, hd, h_stride, Lc, L_stride, lb[l0:l1], nb_iter, early_stopping, wind, tol,
                     [o[l0:l1] for o in outs], J[l0:l1], None, None, n_iter[l0:l1], cz)
    J /= (J[:, :, :1] + 1.0e-30)                                   # bold_signal.py:97, in place
    return tuple(like_input(t, y) for t in outs) + (like_input(J, y),)


def deconv_lbda_path_fit(y, t_r, hrf, lbdas, nb_iter=200, early_stopping=False, tol=1.0e-6, wind=6, x0=None,
                         dtype=None, censor=None):
    """Data-fit and penalty terms of every (lambda, voxel) problem of :func:`deconv_lbda_path`, without
    keeping the solutions: what choosing lambda needs, at any number of voxels.

    Returns ``(R, G, n_iter)``, each ``[n_lbda, V]``: ``R = ||x - y||^2`` and ``G = ||diff_z||_1`` of the
    solution ``deconv(y, t_r, hrf, lbda=l, ...)`` returns (the reference's own ``R`` and ``G``,
    bold_signal.py:139-145; its cost is ``0.5 R + l G``), in the working precision, and the number of
    iterations each problem ran.  Arguments as in :func:`deconv_lbda_path`.

    The batch is cut into voxel ranges; one launch solves every lambda of a range, so the rows of ``y`` are
    still read once per voxel, and its solutions go to one scratch of at most ``FIT_SCRATCH_BYTES`` reused
    from range to range.  Device memory is ``y``, ``hrf``, the three ``[n_lbda, V]`` results and that scratch,
    whatever V is.  The library does not choose lambda; a two-stage use, picking per voxel the lambda whose
    data fit is nearest the noise level (the target the reference's ``lbda=None`` loop steers toward), then
    solving once at it -- the same kernel, so the rows equal the path's rows at the chosen lambdas::

        R, G, n_iter = deconv_lbda_path_fit(y, t_r, h, lbdas, nb_iter=200, early_stopping=True, x0=x0)
        sigma = mad_daub_noise_est(y)                              # [V]
        lbda_v = np.asarray(lbdas)[np.argmin(np.abs(R - y.shape[1] * sigma ** 2), axis=0)]
        x, z, diff_z, J, _, _ = deconv(y, t_r, h, lbda=lbda_v, nb_iter=200, early_stopping=True, x0=x0)

    With ``censor`` (``[T]`` or ``[V, T]``), ``R = ||M (x - y)||^2`` counts the kept scans only, so the target is
    ``n_kept * sigma ** 2`` with ``n_kept = (censor == 0).sum(-1)`` and sigma from the kept detail coefficients::

        R, G, n_iter = deconv_lbda_path_fit(y, t_r, h, lbdas, early_stopping=True, x0=x0, censor=censor)
        sigma = mad_daub_noise_est_censored(yb, cm, stride)        # pybold_b200.censor
        lbda_v = np.asarray(lbdas)[np.argmin(np.abs(R - n_kept * sigma ** 2), axis=0)]
        x, z, diff_z, J, _, _ = deconv(y, t_r, h, lbda=lbda_v, early_stopping=True, x0=x0, censor=censor)
    """
    yb, hd, h_stride, Lc, L_stride, lb, cz = _path_problem(y, hrf, lbdas, x0, dtype, censor)
    V, T = yb.shape
    n_l = lb.numel()
    dev = yb.device
    R = torch.empty((n_l, V), dtype=yb.dtype, device=dev)
    G = torch.empty((n_l, V), dtype=yb.dtype, device=dev)
    n_iter = torch.empty((n_l, V), dtype=torch.int32, device=dev)
    if V == 0 or n_l == 0:
        return like_input(R, y), like_input(G, y), like_input(n_iter, y)
    # voxels per launch: three solution planes [n_lbda, vc, T] within the scratch budget
    vc = max(1, min(V, FIT_SCRATCH_BYTES // (3 * n_l * T * yb.element_size())))
    scratch = torch.empty((3, n_l * vc * T), dtype=yb.dtype, device=dev)
    r = torch.empty(n_l * vc, dtype=yb.dtype, device=dev)
    g = torch.empty_like(r)
    n_it = torch.empty(n_l * vc, dtype=torch.int32, device=dev)
    for v0 in range(0, V, vc):
        v1 = min(v0 + vc, V)
        n = v1 - v0
        czr = None if cz is None else (cz[0][v0:v1] if cz[1] else cz[0], cz[1])
        _path_launch(yb[v0:v1], hd[v0:v1] if h_stride else hd, h_stride, Lc[v0:v1] if L_stride else Lc,
                     L_stride, lb, nb_iter, early_stopping, wind, tol, scratch, None, r, g, n_it, czr)
        R[:, v0:v1] = r[:n_l * n].view(n_l, n)
        G[:, v0:v1] = g[:n_l * n].view(n_l, n)
        n_iter[:, v0:v1] = n_it[:n_l * n].view(n_l, n)
    return like_input(R, y), like_input(G, y), like_input(n_iter, y)


def bd_alloc(V, T, K, nb_iter, dtype, dev):
    """Output buffers of :func:`bd_batch` (reusable across calls via ``out=``)."""
    return {
        "x": torch.empty((V, T), dtype=dtype, device=dev),
        "z": torch.empty((V, T), dtype=dtype, device=dev),
        "diff_z": torch.empty((V, T), dtype=dtype, device=dev),
        "h": torch.empty((V, K), dtype=dtype, device=dev),
        "theta": torch.empty(V, dtype=dtype, device=dev),
        "J": torch.full((V, nb_iter + 2), float("nan"), dtype=dtype, device=dev),
        "r": torch.full((V, nb_iter + 2), float("nan"), dtype=dtype, device=dev),
        "g": torch.full((V, nb_iter + 2), float("nan"), dtype=dtype, device=dev),
        "n_trace": torch.zeros(V, dtype=torch.int32, device=dev),
    }


def bd_batch(y, t_r, lbda, theta_0, z_0, hrf_dur, bounds, nb_iter, early_stopping, wind, tol,
             out=None):
    """Device entry point of :func:`bd`: tensors in, dict of tensors out (all ``[V, ...]``).

    ``out`` (from :func:`bd_alloc`) lets a caller reuse the output buffers; ``lbda`` / ``theta_0``
    given as device tensors are used in place (no host round trip): the call is then a single
    asynchronous kernel launch.
    """
    V, T = y.shape
    dtype, dev = y.dtype, y.device
    K = hrf_len(t_r, hrf_dur)
    lb, lb_stride = per_voxel(lbda, V, dtype, dev, "lbda")
    th0, th_stride = per_voxel(theta_0, V, dtype, dev, "theta_0")
    lo, hi = bounds[0]
    if out is None:
        out = bd_alloc(V, T, K, nb_iter, dtype, dev)
    if z_0 is not None and (tuple(z_0.shape) != (V, T) or z_0.dtype != dtype or z_0.device != dev):
        raise ValueError("z_0 must be a %s tensor of shape (%d, %d) on %s" % (dtype, V, T, dev))
    with torch.cuda.device(dev):        # grid sizing and the launch stream follow the current device
        rc = _lib.fn("pb_bd", dtype)(
            ptr(y), float(t_r), float(hrf_dur), ptr(lb), lb_stride, ptr(th0), th_stride, ptr(z_0),
            float(lo), float(hi), int(nb_iter), int(bool(early_stopping)), int(wind), float(tol),
            ptr(out["x"]), ptr(out["z"]), ptr(out["diff_z"]), ptr(out["h"]), ptr(out["theta"]),
            ptr(out["J"]), ptr(out["r"]), ptr(out["g"]), ptr(out["n_trace"]), V, T, K, stream_ptr())
    _lib.check(rc, "pb_bd")
    return out


# ---- host-resident batches: chunked, double-buffered streaming ------------------------------
_STREAM_MIN_VOXELS = 8192      # below this a single launch is used
_STREAM_TARGET_CHUNK = 32768   # approximate chunk size, rounded to whole waves of the grid
_PINNED_RESULT_LIMIT = 4 << 30  # results up to this many bytes are returned in pinned host memory
_staging_cache = {}


def _staging(key, shapes, dtype):
    """Pinned staging buffers, cached across calls (cudaHostAlloc is expensive).  The cache is keyed
    by thread and device: one thread per GPU in the same process must not share staging slots."""
    import threading
    key = (threading.get_ident(), torch.cuda.current_device()) + tuple(key)
    bufs = _staging_cache.get(key)
    if bufs is None:
        if len(_staging_cache) > 8:
            _staging_cache.clear()
        bufs = {k: torch.empty(shp, dtype=(torch.int32 if k == "n_trace" else dtype), pin_memory=True)
                for k, shp in shapes.items()}
        _staging_cache[key] = bufs
    return bufs


def _bd_streamed(yh, dtype, t_r, lbda, theta_0, z_0, hrf_dur, bounds, nb_iter, early_stopping, wind,
                 tol):
    """``bd`` for a HOST ``[V, T]`` batch: the batch is cut into chunks of whole grid waves; while
    the kernel solves chunk i, chunk i+1 is uploaded and chunk i-1 is downloaded (two CUDA streams,
    pinned staging), so that the host<->device copies hide behind the solve.  Returns CPU tensors.
    """
    V, T = yh.shape
    dev = torch.device("cuda", torch.cuda.current_device())
    K = hrf_len(t_r, hrf_dur)
    ntr = nb_iter + 2
    # Chunks of whole waves of the persistent grid (no partially filled last wave inside a chunk).  Equal,
    # non-wave-aligned chunks were measured in round 2 and rejected: the kernels of consecutive chunks (two
    # streams) do not overlap at their tails, 4 x 25 000 voxels took 631 ms against 591-599 for 3 x 31 968 + 4 096.
    wave = _lib.lib.pb_bd_wave_voxels(T, K, int(dtype == torch.float64), int(nb_iter))
    chunk = _STREAM_TARGET_CHUNK
    if wave > 0:
        chunk = max(wave, (chunk // wave) * wave)
    chunk = min(chunk, V)
    shapes = {"x": (chunk, T), "z": (chunk, T), "diff_z": (chunk, T), "h": (chunk, K),
              "theta": (chunk,), "J": (chunk, ntr), "r": (chunk, ntr), "g": (chunk, ntr),
              "n_trace": (chunk,)}
    # Results of moderate size are written by the device straight into pinned host tensors (PyTorch
    # caches pinned blocks, so repeated calls do not pay cudaHostAlloc again); larger ones go through
    # two pinned staging slots and a host copy into pageable memory.
    esize = torch.empty((), dtype=dtype).element_size()
    out_bytes = sum(V * int(np.prod(shp[1:], dtype=np.int64)) * esize for shp in shapes.values())
    pin_out = out_bytes <= _PINNED_RESULT_LIMIT

    def alloc_final(pinned):
        return {k: torch.empty((V,) + shp[1:], dtype=(torch.int32 if k == "n_trace" else dtype),
                               pin_memory=pinned)
                for k, shp in shapes.items()}

    try:
        final = alloc_final(pin_out)
    except RuntimeError:            # the host refuses to lock that much memory: pageable + staging
        if not pin_out:
            raise
        pin_out = False
        final = alloc_final(False)

    def host_vec(val):
        if isinstance(val, torch.Tensor):
            val = val.detach().cpu().numpy()
        return np.asarray(val, dtype=np.float64).reshape(-1)

    lb_all, th_all = host_vec(lbda), host_vec(theta_0)
    z0h = None
    if z_0 is not None:
        z0h = (z_0 if isinstance(z_0, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(z_0)))
        z0h = z0h.reshape(V, T)
    slots = []
    for s_idx in range(2):
        slots.append({
            "stream": torch.cuda.Stream(device=dev),
            "event": torch.cuda.Event(),
            "y": torch.empty((chunk, T), dtype=dtype, device=dev),
            "z0": torch.empty((chunk, T), dtype=dtype, device=dev) if z0h is not None else None,
            "out": bd_alloc(chunk, T, K, nb_iter, dtype, dev),
            "stage_in": _staging(("in", s_idx, chunk, T, dtype, z0h is not None),
                                 {"y": (chunk, T), "z0": (chunk, T)} if z0h is not None else {"y": (chunk, T)},
                                 dtype),
            "stage_out": None if pin_out else _staging(("out", s_idx, chunk, T, K, ntr, dtype), shapes, dtype),
            "range": None,
        })

    def drain(slot):
        if slot["range"] is None:
            return
        lo, hi = slot["range"]
        slot["event"].synchronize()
        if not pin_out:
            for k in final:
                final[k][lo:hi].copy_(slot["stage_out"][k][:hi - lo])
        slot["range"] = None

    main = torch.cuda.current_stream()
    n_chunks = (V + chunk - 1) // chunk
    for i in range(n_chunks):
        lo, hi = i * chunk, min((i + 1) * chunk, V)
        n = hi - lo
        slot = slots[i % 2]
        drain(slot)
        src = yh[lo:hi]
        if not (src.is_pinned() and src.dtype == dtype):
            slot["stage_in"]["y"][:n].copy_(src)
            src = slot["stage_in"]["y"][:n]
        z0src = None
        if z0h is not None:
            slot["stage_in"]["z0"][:n].copy_(z0h[lo:hi])
            z0src = slot["stage_in"]["z0"][:n]
        st = slot["stream"]
        st.wait_stream(main)
        with torch.cuda.stream(st):
            slot["y"][:n].copy_(src, non_blocking=True)
            if z0src is not None:
                slot["z0"][:n].copy_(z0src, non_blocking=True)
            lb = lb_all if lb_all.size == 1 else lb_all[lo:hi]
            th = th_all if th_all.size == 1 else th_all[lo:hi]
            out = {k: v[:n] for k, v in slot["out"].items()}
            bd_batch(slot["y"][:n], t_r, lb, th, slot["z0"][:n] if z0src is not None else None,
                     hrf_dur, bounds, nb_iter, early_stopping, wind, tol, out=out)
            for k in final:
                dst = final[k][lo:hi] if pin_out else slot["stage_out"][k][:n]
                dst.copy_(out[k], non_blocking=True)
            slot["event"].record(st)
        slot["range"] = (lo, hi)
    for slot in slots:
        drain(slot)
    main.wait_stream(slots[0]["stream"])
    main.wait_stream(slots[1]["stream"])
    return final


def bd(y, t_r, lbda=1.0, theta_0=None, z_0=None, hrf_dur=20.0,  # noqa
       bounds=None, nb_iter=100, nb_sub_iter=1000, nb_last_iter=10000,
       print_period=50, early_stopping=False, wind=4, tol=1.0e-12, verbose=0, dtype=None):
    """Semi-blind deconvolution with the dilated SPM HRF (pybold/bold_signal.py:281-382).

    Precision follows the input like NumPy would: float64 arrays (what the reference computes in,
    bold_signal.py:288) run the FP64 build -- the parity build, about 2.3x slower -- and float32
    arrays the FP32 build the throughput figures are quoted on (1e-4 of the reference, DESIGN.md);
    ``dtype=np.float32`` forces the fast build for float64 input.

    Returns ``(x, z, diff_z, h, d)``; ``d`` has the reference's keys ``'J'``, ``'r'``, ``'g'``
    (length ``nb_iter + 2``, shorter after an early stop) and ``'l_alpha'`` (empty list), plus
    ``'theta'`` (final dilation).  Like the reference, ``nb_iter`` is also the inner iteration
    count and ``nb_sub_iter`` / ``nb_last_iter`` are accepted and ignored (bold_signal.py:324,366).
    """
    dtype = pick_dtype(y, dtype=dtype)
    theta_0 = MAX_DELTA if theta_0 is None else theta_0                    # bold_signal.py:291
    th_chk = np.asarray(theta_0.detach().cpu() if isinstance(theta_0, torch.Tensor) else theta_0,
                        dtype=np.float64)
    if np.any(th_chk < MIN_DELTA) or np.any(th_chk > MAX_DELTA):           # hrf_model.py:17-21
        raise ValueError("delta should belong in [{0}, {1}], got delta = {2}".format(
            MIN_DELTA, MAX_DELTA, th_chk))
    if bounds is None:
        bounds = [(MIN_DELTA + 1.0e-1, MAX_DELTA - 1.0e-1)]                # bold_signal.py:303-304
    host_in = not (isinstance(y, torch.Tensor) and y.is_cuda)
    if host_in and np.ndim(y) == 2 and len(y) >= _STREAM_MIN_VOXELS:
        from ._array import require_cuda
        require_cuda()
        yh = y if isinstance(y, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(y))
        out = _bd_streamed(yh.contiguous(), dtype, t_r, lbda, theta_0, z_0, hrf_dur, bounds, nb_iter,
                           early_stopping, wind, tol)
        conv = (lambda t: t) if isinstance(y, torch.Tensor) else (lambda t: t.numpy())
        d = {k: conv(out[k]) for k in ("J", "r", "g", "theta", "n_trace")}
        d["l_alpha"] = []
        return conv(out["x"]), conv(out["z"]), conv(out["diff_z"]), conv(out["h"]), d
    yb, one_d = _as_batch(y, dtype)
    z0 = None
    if z_0 is not None:
        z0 = to_device(z_0, dtype).reshape(yb.shape)
    out = bd_batch(yb, t_r, lbda, theta_0, z0, hrf_dur, bounds, nb_iter, early_stopping, wind, tol)
    if one_d:
        n = int(out["n_trace"][0])
        d = {k: like_input(out[k][0, :n], y) for k in ("J", "r", "g")}
        d["l_alpha"] = []
        d["theta"] = float(out["theta"][0])
        return (like_input(out["x"][0], y), like_input(out["z"][0], y),
                like_input(out["diff_z"][0], y), like_input(out["h"][0], y), d)
    d = {k: like_input(out[k], y) for k in ("J", "r", "g", "theta", "n_trace")}
    d["l_alpha"] = []
    return (like_input(out["x"], y), like_input(out["z"], y), like_input(out["diff_z"], y),
            like_input(out["h"], y), d)


def hrf_estim_batch(z, y, t_r, dur, theta_0=MAX_DELTA, bounds=None):
    """Device entry point: bounded theta minimisation for ``[V, T]`` tensors."""
    V, T = y.shape
    dtype, dev = y.dtype, y.device
    K = hrf_len(t_r, dur)
    if bounds is None:
        bounds = [(MIN_DELTA + 1.0e-1, MAX_DELTA - 1.0e-1)]               # bold_signal.py:229
    th0, th_stride = per_voxel(theta_0, V, dtype, dev, "theta_0")
    theta = torch.empty(V, dtype=dtype, device=dev)
    h = torch.empty((V, K), dtype=dtype, device=dev)
    cost = torch.empty(V, dtype=dtype, device=dev)
    rc = _lib.fn("pb_hrf_estim", dtype)(
        ptr(z), ptr(y), float(t_r), float(dur), ptr(th0), th_stride, float(bounds[0][0]),
        float(bounds[0][1]), ptr(theta), ptr(h), ptr(cost), V, T, K, stream_ptr())
    _lib.check(rc, "pb_hrf_estim")
    return theta, h, cost


def hrf_estim(z, y, t_r, dur, verbose=0):
    """HRF estimation for a known block signal (pybold/bold_signal.py:225-239).

    Returns ``(h, J)``.  The reference's J lists the cost after every L-BFGS-B iterate (its
    ``Tracker`` callback); the device solver is not an iterate-by-iterate port, so J holds the
    cost at the start point and at the minimiser.
    """
    dtype = pick_dtype(z, y)
    yb, one_d = _as_batch(y, dtype)
    zb, _ = _as_batch(z, dtype)
    theta, h, cost = hrf_estim_batch(zb, yb, t_r, dur)
    start_cost = hrf_fit_err(MAX_DELTA - 1.0e-1, z, y, t_r, dur)
    if one_d:
        return like_input(h[0], y), [float(np.asarray(start_cost).reshape(-1)[0]), float(cost[0])]
    return like_input(h, y), [like_input(torch.as_tensor(start_cost), y), like_input(cost, y)]


def hrf_fit_err(theta, z, y, t_r, hrf_dur):
    """0.5 * || y - h(theta) * z ||^2 (pybold/bold_signal.py:217-222), evaluated on the device."""
    from .convolution import spectral_convolve
    from .hrf_model import spm_hrf
    dtype = pick_dtype(z, y)
    yb, one_d = _as_batch(y, dtype)
    zb, _ = _as_batch(z, dtype)
    th = torch.as_tensor(np.asarray(theta, dtype=np.float64).reshape(-1))
    h, _ = spm_hrf(th.to(yb.device), t_r, hrf_dur, False)
    h = h.to(dtype)
    res = yb - spectral_convolve(h if h.shape[0] > 1 else h[0], zb)
    val = 0.5 * torch.sum(res * res, dim=1)
    if one_d:
        return float(val[0])
    return like_input(val, y)
