"""bd(early_stopping=True) at long series and short-TR HRFs: a build without the early-stopping CTA bd kernel (``--old``,
a tree whose library is built) against this tree, alternated old, new, old, new in one run, one JSON line per timed
call.

Each arm is a subprocess importing its tree's ``pybold_b200``; it times every shape with a host clock to a device
synchronise after one warm-up call, and saves a sample of its outputs (seeded inputs, the same for both arms): z of
the first 256 voxels and every voxel's n_trace, so that the driver reports the largest relative difference of z and
whether the trace lengths agree.  The card's name and power limit are read in the same run.

The last two shapes time, in each build, the cfg4 shape with early stopping switched on but unable to fire (tol = 0,
wind above nb_iter) against early stopping off: the cost of the early-stopping code itself (norm sums, extra
registers and spills) on the same iterations.

After each arm's shapes the same tree runs ``bench.py --gpus 1`` (``--bench-steps`` / ``--bench-warmup``), so that the
headline, cfg2, cfg4 and cfg5 of both builds are compared in the same run; its JSON line is printed as is.

Usage: python tools/bench_bd_es_long.py --old DIR [--reps 2] [--scale 1.0] [--bench-steps 5] [--bench-warmup 3]
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

ES = dict(early_stopping=True, wind=4, tol=1.0e-12)       # the reference's defaults besides early_stopping
# (name, dtype, V, T, t_r (K = 20, 28, 40, 63 taps), nb_iter, bd keywords); `--scale` multiplies V
SHAPES = [
    ("es 230k x 1200 K28", "float32", 230000, 1200, 0.72, 100, ES),
    ("es 50k x 2400 K28", "float32", 50000, 2400, 0.72, 100, ES),
    ("es 100k x 600 K40", "float32", 100000, 600, 0.5, 100, ES),
    # V shrunk so that the generic kernel of the old build finishes in seconds
    ("es 20k x 4096 K63", "float32", 20000, 4096, 0.32, 100, ES),
    ("es 50k x 300 K20 (control, group kernel)", "float32", 50000, 300, 1.0, 100, ES),
    ("es fp64 20k x 1200 K28", "float64", 20000, 1200, 0.72, 100, ES),
    ("no es 50k x 1200 K28, 20 x 20", "float32", 50000, 1200, 0.72, 20, dict(early_stopping=False)),
    ("es never fires 50k x 1200 K28, 20 x 20", "float32", 50000, 1200, 0.72, 20,
     dict(early_stopping=True, wind=25, tol=0.0)),
]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=False)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def worker(out_path, scale):
    import torch
    import pybold_b200 as pb  # (the tree on PYTHONPATH)
    from pybold_b200.synth import gen_voxels_device
    saved = {}
    for name, dt, V, T, t_r, nb_iter, kw in SHAPES:
        V = max(1, int(V * scale))
        dtype = getattr(torch, dt)
        y = gen_voxels_device(V, T, t_r, 20.0, seed=V + T, dtype=dtype)
        lbda = torch.linspace(0.5, 3.0, V, device="cuda", dtype=dtype)

        def call():
            return pb.bd(y, t_r, lbda=lbda, theta_0=2.0, hrf_dur=20.0, nb_iter=nb_iter, **kw)
        call()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = call()
        torch.cuda.synchronize()
        dt_s = time.perf_counter() - t0
        n_tr = out[4]["n_trace"]
        saved[name + " z"] = out[1][:256].cpu().numpy()
        saved[name + " n_trace"] = n_tr.cpu().numpy()
        print(json.dumps({"shape": name, "V": V, "T": T, "K": out[3].shape[1], "seconds": round(dt_s, 4),
                          "voxels_per_s": round(V / dt_s, 1), "n_trace_min": int(n_tr.min()),
                          "n_trace_max": int(n_tr.max())}), flush=True)
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
    tmp = tempfile.mkdtemp(prefix="bench_bd_es_long_")
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
        for name, *_ in SHAPES:
            kz, kn = (name + " z").replace(" ", "_"), (name + " n_trace").replace(" ", "_")
            a64, b64 = o[kz].astype(np.float64), n[kz].astype(np.float64)
            print(json.dumps({"shape": name, "max_rel_diff_z_old_new":
                              float(np.max(np.abs(a64 - b64)) / (np.max(np.abs(a64)) + 1e-300)),
                              "n_trace_equal": bool(np.array_equal(o[kn], n[kn]))}), flush=True)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


if __name__ == "__main__":
    main()
