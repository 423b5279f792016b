"""``deconv(lbda=None)``: the host-driven outer loop of the previous release against the single launch
(``deconv_auto_batch``, ``pb_deconv_auto_*``), alternated in one run, one JSON line per timed call.

Both arms are the public ``deconv(y, t_r, h, lbda=None, sigma=sigma, x0=x0, ...)`` on device inputs, timed with a
host clock to a device synchronise (power iteration, noise loop, the final pass, the tuple the call returns); the
host-loop arm swaps in a statement of the previous loop: per outer iteration one ``pb_deconv_masked`` launch
(through ``deconv_batch(active=...)``) and one ``pb_noise_step`` launch, the alpha window in torch, a host check
of "anything still running" every 4 outer iterations.  sigma is the reference's ``mad_daub_noise_est``, computed
once outside the timed calls.  Reference defaults (``nb_iter=1000``, ``nb_sub_iter=1000``, ``early_stopping``,
``tol=1e-6``, ``wind=6``) at cfg1; the two batch shapes cap the outer and inner counts (see ``SHAPES``) so that
the host-loop arm finishes in seconds.  The card's name and power limit are read in the same run.

Usage: python tools/bench_deconv_auto.py [--reps 3]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import pybold_b200 as pb  # noqa: E402
from pybold_b200.utils import mad_daub_noise_est  # noqa: E402
from pybold_b200 import _lib, noise  # noqa: E402
from pybold_b200._array import like_input, ptr, stream_ptr  # noqa: E402
from pybold_b200.bold_signal import deconv_batch  # noqa: E402
from pybold_b200.hrf_model import spm_hrf  # noqa: E402
from pybold_b200.synth import gen_voxels_device  # noqa: E402

# (name, V, T, t_r (K = 30, 20, 28 taps), dtype, nb_iter (outer), nb_sub_iter)
SHAPES = [
    ("cfg1", 1, 600, 0.68, torch.float64, 1000, 1000),
    ("100k x 300", 100000, 300, 1.0, torch.float32, 20, 200),
    ("whole brain 230k x 1200", 230000, 1200, 0.72, torch.float32, 10, 200),
]
STATS = {}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=False)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def host_loop(y_in, yb, one_d, hrf, lipschitz, sigma, early_stopping, tol, wind, nb_iter, nb_sub_iter):
    """The outer loop of the previous release (pybold_b200/noise.py), plus inner-iteration counts for STATS."""
    V, T = yb.shape
    dtype, dev = yb.dtype, yb.device
    sigma = torch.as_tensor(sigma, dtype=dtype, device=dev).reshape(-1).expand(V).clone()
    alpha = torch.ones(V, dtype=dtype, device=dev)
    lbda = 1.0 / (2.0 * alpha)
    w, x, z = torch.zeros_like(yb), torch.zeros_like(yb), torch.zeros_like(yb)
    scratch = (torch.empty_like(yb), torch.empty_like(yb), torch.empty_like(yb),
               torch.zeros(V, dtype=torch.int32, device=dev))
    active = torch.ones(V, dtype=torch.uint8, device=dev)
    n_outer = torch.full((V,), nb_iter, dtype=torch.int64, device=dev)
    n_inner = torch.zeros(V, dtype=torch.int64, device=dev)
    sub = int(wind / 2)
    hist = []
    J, R, G = (torch.full((V, nb_iter), float("nan"), dtype=dtype, device=dev) for _ in range(3))
    step = _lib.fn("pb_noise_step", dtype)
    check_every = 1 if V == 1 else 4
    for i in range(nb_iter):
        x_n, z_n, w_n, _, n_it = deconv_batch(yb, hrf, lbda, lipschitz, w, early_stopping, tol, wind,
                                              nb_sub_iter, active=active, out=scratch, trace=False)
        n_inner += torch.where(active.bool(), n_it.long(), 0)
        r = torch.empty(V, dtype=dtype, device=dev)
        g = torch.empty(V, dtype=dtype, device=dev)
        with torch.cuda.device(dev):
            rc = step(ptr(x_n), ptr(z_n), ptr(w_n), ptr(yb), ptr(sigma), ptr(active), 1.0e-4, ptr(x), ptr(z), ptr(w),
                      ptr(alpha), ptr(lbda), ptr(r), ptr(g), V, T, stream_ptr())
        _lib.check(rc, "pb_noise_step")
        hist.append(alpha.clone())
        if len(hist) > wind:
            hist = hist[1:]
        live = active.bool()
        R[:, i] = torch.where(live, r, R[:, i])
        G[:, i] = torch.where(live, g, G[:, i])
        J[:, i] = torch.where(live, 0.5 * r + lbda * g, J[:, i])
        if early_stopping and i > wind and sub > 0:
            old_it = torch.stack(hist[:-sub]).mean(dim=0)
            new_it = torch.stack(hist[-sub:]).mean(dim=0)
            stop = ((new_it - old_it).abs() / new_it.abs() < tol) & live
            n_outer = torch.where(stop, torch.full_like(n_outer, i + 1), n_outer)
            active = active & (~stop).to(torch.uint8)
            if (i % check_every == 0 or i == nb_iter - 1) and not bool(active.any()):
                break
    x, z, w, _, n_it = deconv_batch(yb, hrf, lbda, lipschitz, w, early_stopping, tol, wind, nb_sub_iter, trace=False)
    STATS["inner"] = (n_inner + n_it.long()).cpu().numpy()
    if one_d:
        n = int(n_outer[0])
        conv = lambda t: like_input(t[0], y_in)  # noqa: E731
        return (conv(x), conv(z), conv(w), [float(v) for v in J[0, :n]], [float(v) for v in R[0, :n]],
                [float(v) for v in G[0, :n]])
    n_max = int(n_outer.max())
    conv = lambda t: like_input(t, y_in)  # noqa: E731
    return conv(x), conv(z), conv(w), conv(J[:, :n_max]), conv(R[:, :n_max]), conv(G[:, :n_max])


def outer_counts(J):
    J = np.atleast_2d(np.asarray(J.cpu() if isinstance(J, torch.Tensor) else J, dtype=np.float64))
    return np.sum(~np.isnan(J), axis=1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    print(json.dumps({"card": card()}), flush=True)
    new_loop = noise.deconv_auto_lbda
    for name, V, T, t_r, dtype, nb, nb_sub in SHAPES:
        y = gen_voxels_device(V, T, t_r, 20.0, seed=V + T, dtype=dtype)
        h = spm_hrf(torch.tensor([1.0], dtype=torch.float64).cuda(), t_r, 20.0, True)[0][0].to(dtype)
        sigma = mad_daub_noise_est(y)
        x0 = np.random.RandomState(0).randn(T)
        yy = y[0] if V == 1 else y
        kw = dict(lbda=None, sigma=sigma[0] if V == 1 else sigma, x0=x0, nb_iter=nb, nb_sub_iter=nb_sub,
                  early_stopping=True, tol=1.0e-6, wind=6)
        res = {}
        for rep in range(a.reps + 1):                  # rep 0 warms both arms up
            for arm, loop in (("host loop", host_loop), ("one launch", new_loop)):
                noise.deconv_auto_lbda = loop
                try:
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    out = pb.deconv(yy, t_r, h, **kw)
                    torch.cuda.synchronize()
                    dt = time.perf_counter() - t0
                finally:
                    noise.deconv_auto_lbda = new_loop
                res[arm] = out
                if rep == 0:
                    continue
                n_out = outer_counts(out[3])
                rec = {"shape": name, "V": V, "T": T, "K": int(h.shape[0]), "dtype": str(dtype).split(".")[-1],
                       "nb_iter": nb, "nb_sub_iter": nb_sub, "arm": arm, "rep": rep, "seconds": round(dt, 4),
                       "voxels_per_s": round(V / dt, 1), "outer_median": float(np.median(n_out)),
                       "outer_max": int(n_out.max())}
                if arm == "host loop":
                    rec["inner_total_median"] = float(np.median(STATS["inner"]))
                    rec["inner_total_max"] = int(STATS["inner"].max())
                print(json.dumps(rec), flush=True)
        zo, zn = (torch.as_tensor(res[k][1]).double() for k in ("host loop", "one launch"))
        no, nn = outer_counts(res["host loop"][3]), outer_counts(res["one launch"][3])
        print(json.dumps({"shape": name, "z_max_rel_diff": float((zo - zn).abs().max() / zo.abs().max()),
                          "outer_counts_equal": float(np.mean(no == nn))}), flush=True)
        del y, res
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
