"""Censored (about 10 % of scans) against uncensored deconvolution, alternated in one run.

    python tools/bench_deconv_censor.py [--reps 3] [--out bench_deconv_censor.json]

Shapes: 50 000 x 300 (K = 20) and 230 000 x 1200 (K = 28, the HCP cfg4 shape), both with early stopping, and
deconv(lbda=None) at 20 000 x 900 (K = 40).  Both arms get the same y, taps, lambda and Lipschitz constant, so the
difference is the kernel: an uncensored call at T = 300 runs on the group kernel, a censored one on a CTA row
(pb_deconv_variant / pb_deconv_censored_variant are printed).  The card's name and power limit are read in the same
run.  Times are CUDA events around the launch, after one warm-up call of each arm.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pybold_b200 import _lib  # noqa: E402
from pybold_b200.bold_signal import deconv_auto_batch, deconv_batch  # noqa: E402
from pybold_b200.synth import gen_voxels  # noqa: E402
from oracle import pybold_oracle as orc  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def mask(V, T, seed):
    rs = np.random.RandomState(seed)
    m = np.zeros((V, T), dtype=np.uint8)
    starts = rs.randint(0, T, size=(V, max(1, T // 30)))
    for k in range(3):                                   # runs of three scans: ~10 % of the series
        np.put_along_axis(m, np.minimum(starts + k, T - 1), 1, axis=1)
    return torch.from_numpy(m).cuda()


def timed(fn, reps):
    out = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        out.append(e0.elapsed_time(e1) / 1e3)
    return out


def variant(q, T, K, es, auto):
    fam = ctypes.c_int()
    vid = q(T, K, 0, 200, int(es), 6, int(auto), ctypes.byref(fam))
    return [vid, fam.value]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--scale", type=float, default=1.0, help="fraction of the voxel counts (smoke runs)")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    res = {"card": card(), "cases": []}
    for V, T, K, t_r, auto in ((50000, 300, 20, 1.0, False), (230000, 1200, 28, 0.72, False),
                               (20000, 900, 40, 0.5, True)):
        V = max(1, int(V * a.scale))
        y = torch.from_numpy(gen_voxels(min(V, 4096), T, t_r, 20.0, seed0=31).astype(np.float32)).cuda()
        y = y.repeat((V + y.shape[0] - 1) // y.shape[0], 1)[:V].contiguous()
        h = torch.from_numpy(orc.spm_hrf(1.0, t_r, 20.0, True)[0].astype(np.float32)).cuda()
        assert h.numel() == K
        cm = mask(V, T, 7)
        if auto:
            arms = {c: (lambda c=c: deconv_auto_batch(y, h, 0.5, 8.0, nb_iter=20, nb_sub_iter=100, censor=c))
                    for c in (None, cm)}
        else:
            arms = {c: (lambda c=c: deconv_batch(y, h, 0.5, 8.0, nb_iter=200, early_stopping=True, tol=1e-4,
                                                 wind=6, censor=c))
                    for c in (None, cm)}
        for fn in arms.values():
            fn()
        torch.cuda.synchronize()
        t = {"plain": [], "censored": []}
        for _ in range(a.reps):                          # alternated
            t["plain"] += timed(arms[None], 1)
            t["censored"] += timed(arms[cm], 1)
        case = {"V": V, "T": T, "K": K, "auto": auto, "censored_frac": float(cm.float().mean()),
                "plain_s": min(t["plain"]), "censored_s": min(t["censored"]),
                "plain_all": t["plain"], "censored_all": t["censored"],
                "plain_variant": variant(_lib.lib.pb_deconv_variant, T, K, not auto, auto),
                "censored_variant": variant(_lib.lib.pb_deconv_censored_variant, T, K, not auto, auto)}
        case["ratio"] = case["censored_s"] / case["plain_s"]
        res["cases"].append(case)
        print(json.dumps({k: v for k, v in case.items() if not k.endswith("_all")}), flush=True)
        del y, cm, arms
        torch.cuda.empty_cache()
    print(json.dumps({"card": res["card"]}))
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
