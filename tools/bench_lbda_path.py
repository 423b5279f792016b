"""Regularisation-path figures in (lambda, voxel) problems per second, one JSON line each:

  * fit mode (``deconv_lbda_path_fit``) at the whole-brain HCP shape, 230 000 voxels x 1200 scans, K = 28
    (t_r 0.72 s), 64 lambdas, 200 iterations, without and with early stopping (reference defaults tol 1e-6,
    wind 6);
  * the per-voxel-HRF path (``deconv_lbda_path`` with ``hrf[V, K]``) at the cfg5 shape, 64 x 20 000 x 600.

Every figure is a host clock around the public call ending in a device synchronise, after an untimed call
of the same shape (for the whole-brain fit: of its first 2048 voxels).  The card's name and power limit are read in the same run and printed first.
Usage: python tools/bench_lbda_path.py [--voxels-hcp 230000] [--reps 1]
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
from pybold_b200.bold_signal import FIT_SCRATCH_BYTES, deconv_lbda_path, deconv_lbda_path_fit  # noqa: E402
from pybold_b200.hrf_model import spm_hrf  # noqa: E402
from pybold_b200.synth import gen_voxels_device  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=False)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def timed(fn, reps, warm=True):
    if warm:
        fn()
    torch.cuda.synchronize()
    out = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        out.append(time.perf_counter() - t0)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--voxels-hcp", type=int, default=230000)
    ap.add_argument("--reps", type=int, default=1)
    a = ap.parse_args()
    print(json.dumps({"card": card(), "fit_scratch_bytes": FIT_SCRATCH_BYTES}), flush=True)
    n_l, nb = 64, 200

    # fit mode, whole brain
    V, T, t_r = a.voxels_hcp, 1200, 0.72
    y = gen_voxels_device(V, T, t_r, 20.0, seed=230, dtype=torch.float32)
    thetas = torch.linspace(0.8, 1.6, V, dtype=torch.float64)
    h = spm_hrf(thetas.cuda(), t_r, 20.0, True)[0].to(torch.float32)
    lbdas = np.geomspace(0.05, 20.0, n_l)
    x0 = np.random.RandomState(0).randn(T)
    for es in (False, True):
        kw = dict(nb_iter=nb, early_stopping=es, tol=1.0e-6, wind=6, x0=x0)
        warm = lambda: deconv_lbda_path_fit(y[:2048], t_r, h[:2048], lbdas, **kw)  # noqa: E731
        warm()
        torch.cuda.synchronize()
        res = {}

        def run():
            res["out"] = deconv_lbda_path_fit(y, t_r, h, lbdas, **kw)
        torch.cuda.reset_peak_memory_stats()
        ts = timed(run, a.reps, warm=False)            # warmed on the first 2048 voxels above
        n_iter = res["out"][2]
        print(json.dumps({
            "what": "deconv_lbda_path_fit", "voxels": V, "n_scans": T, "K": int(h.shape[1]), "n_lbda": n_l,
            "nb_iter": nb, "early_stopping": es, "dtype": "f32", "hrf": "per voxel",
            "seconds": [round(t, 3) for t in ts], "problems_per_s": n_l * V / min(ts),
            "mean_iterations": float(n_iter.double().mean()),
            "peak_alloc_GB": torch.cuda.max_memory_allocated() / 1e9,
            "note": "host clock around the whole public call: power iteration, every launch, summary copies"}),
            flush=True)
    del y, h, res
    torch.cuda.empty_cache()

    # per-voxel-HRF path, cfg5 shape
    V, T, t_r = 20000, 600, 1.0
    y = gen_voxels_device(V, T, t_r, 20.0, seed=5, dtype=torch.float32)
    h = spm_hrf(torch.linspace(0.8, 1.6, V, dtype=torch.float64).cuda(), t_r, 20.0, True)[0].to(torch.float32)
    x0 = np.random.RandomState(0).randn(T)
    for per_voxel in (False, True):
        hh = h if per_voxel else h[V // 2]
        ts = timed(lambda: deconv_lbda_path(y, t_r, hh, lbdas, nb_iter=nb, x0=x0), max(2, a.reps))
        print(json.dumps({
            "what": "deconv_lbda_path", "voxels": V, "n_scans": T, "K": int(h.shape[1]), "n_lbda": n_l,
            "nb_iter": nb, "dtype": "f32", "hrf": "per voxel" if per_voxel else "shared",
            "seconds": [round(t, 4) for t in ts], "problems_per_s": n_l * V / min(ts)}), flush=True)


if __name__ == "__main__":
    main()
