"""Deconvolution at long series and short-TR HRFs: a build without the CTA deconv kernels (``--old``, a tree whose
library is built) against this tree, alternated old, new, old, new in one run, one JSON line per timed call.

Each arm is a subprocess importing its tree's ``pybold_b200``; it times every shape with a host clock to a device
synchronise after one warm-up call, and saves a sample of its outputs (seeded inputs, the same for both arms) so that
the driver reports the largest relative difference between the builds.  The rate is the deconv flop count of
SURVEY.md section 8(d), ``F_it + F_J`` per iteration actually run, over the call time, as a fraction of the nominal
FP32 rate (74.5 Tflop/s): the same convention as cfg2 and cfg5.  The card's name and power limit are read in the
same run.

After each arm's shapes the same tree runs ``bench.py --gpus 1`` (``--bench-steps`` / ``--bench-warmup``), so that the
headline, cfg2, cfg4 and cfg5 of both builds are compared in the same run; its JSON line is printed as is.

Usage: python tools/bench_deconv_long.py --old DIR [--reps 2] [--scale 1.0] [--bench-steps 5] [--bench-warmup 3]
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

NOMINAL_FP32 = 74.5e12
# (name, kind, V, T, t_r (K = 28, 40, 63 taps), extra); `--scale` multiplies V
SHAPES = [
    ("deconv 50k x 2400 K28", "deconv", 50000, 2400, 0.72, {}),
    ("deconv es 50k x 2400 K28", "deconv", 50000, 2400, 0.72, {"es": True}),
    ("deconv 100k x 600 K40", "deconv", 100000, 600, 0.5, {}),
    ("deconv es 100k x 600 K40", "deconv", 100000, 600, 0.5, {"es": True}),
    ("deconv 20k x 4096 K63", "deconv", 20000, 4096, 0.32, {}),
    ("deconv es 20k x 4096 K63", "deconv", 20000, 4096, 0.32, {"es": True}),
    # V shrunk so that the generic kernel of the old build finishes in seconds
    ("lbda=None 20k x 900 K40, 10 x 200", "auto", 20000, 900, 0.5, {}),
    ("path fit 64 lambdas x 5k x 2400 K28", "fit", 5000, 2400, 0.72, {}),
]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=False)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def flops_per_iter(T, K):
    mac = T * K - K * (K - 1) // 2
    return (4 * mac + 11 * T) + (2 * mac + 6 * T)


def worker(out_path, scale):
    import torch
    import pybold_b200  # noqa: F401  (the tree on PYTHONPATH)
    from pybold_b200.bold_signal import deconv_auto_batch, deconv_batch, deconv_lbda_path_fit
    from pybold_b200.hrf_model import spm_hrf
    from pybold_b200.synth import gen_voxels_device
    from oracle import pybold_oracle as orc
    saved = {}
    for name, kind, V, T, t_r, extra in SHAPES:
        V = max(1, int(V * scale))
        y = gen_voxels_device(V, T, t_r, 20.0, seed=V + T, dtype=torch.float32)
        h = spm_hrf(torch.tensor([1.0], dtype=torch.float64).cuda(), t_r, 20.0, True)[0][0].float()
        K = h.shape[0]
        Lc = 0.9 * orc.spectral_radius_est(orc.HrfIntegOperator(h.double().cpu().numpy(), T),
                                           np.random.RandomState(0).randn(T))
        lbda = torch.linspace(0.2, 4.0, V, device="cuda")

        def call():
            if kind == "deconv":
                es = extra.get("es", False)
                return deconv_batch(y, h, lbda, Lc, early_stopping=es, tol=1.0e-2, wind=6, nb_iter=200)
            if kind == "auto":
                sigma = torch.full((V,), 0.3, device="cuda")
                return deconv_auto_batch(y, h, sigma, Lc, nb_iter=10, nb_sub_iter=200, early_stopping=False)
            return deconv_lbda_path_fit(y, t_r, h, np.geomspace(0.05, 20.0, 64), nb_iter=200,
                                        x0=np.random.RandomState(0).randn(T))
        call()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = call()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if kind == "deconv":
            iters = float(out[4].double().sum())
            sample = out[1][:256].cpu().numpy()
        elif kind == "auto":
            iters = float(V) * 11 * 200
            sample = out["z"][:256].cpu().numpy()
        else:
            iters = 64.0 * V * 200
            sample = out[0].cpu().numpy()
        saved[name] = sample
        print(json.dumps({"shape": name, "V": V, "T": T, "K": K, "seconds": round(dt, 4),
                          "voxels_per_s": round(V / dt, 1),
                          "fp32_fraction": round(iters * flops_per_iter(T, K) / dt / NOMINAL_FP32, 4)}), flush=True)
        del y, out
        torch.cuda.empty_cache()
    np.savez(out_path, **{k.replace(" ", "_"): v for k, v in saved.items()})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--old", help="tree of the build to compare with (library built); required")
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--bench-steps", type=int, default=5)
    ap.add_argument("--bench-warmup", type=int, default=3)
    ap.add_argument("--worker", help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.worker:
        worker(a.worker, a.scale)
        return
    if not a.old:
        ap.error("--old DIR is required")
    new = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    print(json.dumps({"card": card()}), flush=True)
    tmp = tempfile.mkdtemp(prefix="bench_deconv_long_")
    try:
        for rep in range(a.reps):
            for arm, tree in (("old", os.path.abspath(a.old)), ("new", new)):
                env = dict(os.environ, PYTHONPATH=tree)
                print(json.dumps({"arm": arm, "rep": rep, "scale": a.scale}), flush=True)
                r = subprocess.run([sys.executable, os.path.abspath(__file__), "--worker",
                                    os.path.join(tmp, "%s.npz" % arm), "--scale", str(a.scale)], env=env, cwd=tree,
                                   check=False)
                if r.returncode != 0:
                    sys.exit("arm %s failed (%d)" % (arm, r.returncode))
                b = subprocess.run([sys.executable, "bench.py", "--gpus", "1", "--steps", str(a.bench_steps),
                                    "--warmup", str(a.bench_warmup)], env=env, cwd=tree, capture_output=True,
                                   text=True, check=False)
                lines = b.stdout.strip().splitlines()
                print(json.dumps({"arm": arm, "rep": rep, "bench.py": json.loads(lines[-1]) if b.returncode == 0
                                  and lines else "failed (%d): %s" % (b.returncode, b.stderr[-500:])}), flush=True)
        o, n = np.load(os.path.join(tmp, "old.npz")), np.load(os.path.join(tmp, "new.npz"))
        for k in o.files:
            a64, b64 = o[k].astype(np.float64), n[k].astype(np.float64)
            print(json.dumps({"shape": k.replace("_", " "), "max_rel_diff_old_new":
                              float(np.max(np.abs(a64 - b64)) / (np.max(np.abs(a64)) + 1e-300))}), flush=True)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)

if __name__ == "__main__":
    main()
