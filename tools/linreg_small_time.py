"""Poisson and KL regression at the notebook shapes: BPG, ABPG or ABPG_gain as one launch (config.fused_small,
csrc/linreg_small.cu) against the operator-by-operator loop, alternated in one process after a warm-up, and the reference
on the host cores.

    python tools/linreg_small_time.py [--reps 3] [--out profiles/linreg_small_r01.json]
    python tools/linreg_small_time.py --drivers abpg,abpg_gain --out profiles/linreg_small_accel_r01.json

Instances: ipynb/ex_Poisson_L2 (Poisson_regrL1(200, 100, noise=1e-4, lamda=0, randseed=1), BPG with line search, 9000
iterations), ipynb/ex_KL_regr_L1 (KL_nonneg_regr(1000, 100, noise=0.01, lamdaL1=0.001, randseed=1), BPG with line
search, 4000 iterations) and a KL instance of the same shape on the simplex (ShannonEntropySimplex, 4000 iterations;
epsilon=0, because at the default 1e-14 it converges and stops after 170).
ABPG and ABPG_gain run with gamma = 2 and their defaults on the same instances and iteration budgets; ABPG_gain may stop
earlier on D(z+, z) < epsilon, so every record carries the number of iterations actually run.
The CPU arm is the unmodified reference package when oracle/_ref holds it, else the NumPy oracle port (labelled so).
"""
import argparse
import contextlib
import io
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402


def simplex_kl_data(m, n, seed):
    """A with unit column sums, b = A x_true (x_true on the simplex) with 1% multiplicative noise."""
    rs = np.random.RandomState(seed)
    A = rs.rand(m, n)
    A = A / A.sum(axis=0)
    xt = rs.rand(n)
    xt = xt / xt.sum()
    b = (A @ xt) * (1 + 0.01 * (rs.rand(m) - 0.5))
    return A, b


def workloads(mod, oracle_port):
    """name -> (description, (f, h, L, x0), maxitrs, epsilon) built with `mod` (this package, the reference or the
    oracle port)."""
    out = {}
    out["poisson_200x100"] = ("Poisson_regrL1(200,100,noise=1e-4,lamda=0,randseed=1), BPG ls_ratio=1.2, maxitrs=9000",
                              mod.Poisson_regrL1(200, 100, noise=1e-4, lamda=0, randseed=1), 9000, 1e-14)
    out["kl_1000x100"] = ("KL_nonneg_regr(1000,100,noise=0.01,lamdaL1=0.001,randseed=1), BPG ls_ratio=1.2, maxitrs=4000",
                          mod.KL_nonneg_regr(1000, 100, noise=0.01, lamdaL1=0.001, randseed=1), 4000, 1e-14)
    A, b = simplex_kl_data(1000, 100, seed=1)
    if oracle_port:
        f, h = mod.make_kl(A, b), mod.make_shannon("simplex")
    else:
        f, h = mod.KLdivRegression(A, b), mod.ShannonEntropySimplex()
    out["kl_simplex_1000x100"] = ("KLdivRegression(1000 x 100, unit column sums) + ShannonEntropySimplex, BPG "
                                  "ls_ratio=1.2, maxitrs=4000, epsilon=0",
                                  (f, h, max(A.sum(axis=0)), np.ones(100) / 100), 4000, 0.0)
    return out


def solve(mod, drv, f, h, L, x0, its, eps, **kw):
    """(F, the discrete sequence: L_k for BPG, G_k for ABPG, the gain for ABPG_gain) of one solve."""
    if drv == "bpg":
        r = mod.BPG(f, h, L, x0, maxitrs=its, epsilon=eps, **kw)
    elif drv == "abpg":
        r = mod.ABPG(f, h, L, x0, 2, its, epsilon=eps, **kw)
    else:
        r = mod.ABPG_gain(f, h, L, x0, 2, its, epsilon=eps, **kw)
    return r[1], r[2]


DRIVER_NAMES = {"bpg": "BPG ls_ratio=1.2", "abpg": "ABPG gamma=2", "abpg_gain": "ABPG_gain gamma=2"}


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        power = q.stdout.strip() or "unknown"
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return name, power


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "linreg_small_r01.json"))
    ap.add_argument("--drivers", default="bpg", help="comma-separated: bpg, abpg, abpg_gain")
    args = ap.parse_args()
    drivers_run = args.drivers.split(",")
    if not set(drivers_run) <= set(DRIVER_NAMES):
        sys.exit(f"--drivers: choose from {sorted(DRIVER_NAMES)}")
    if not torch.cuda.is_available():
        sys.exit("linreg_small_time.py measures the GPU paths and needs a CUDA device")
    import accbpg_and_fw_b200 as acc
    from accbpg_and_fw_b200 import config, drivers
    info = {"bpg": lambda: (drivers._bpg_small.last_info[3], drivers._bpg_small.last_info[1]),
            "abpg": lambda: (drivers._abpg_small.last_info[2], drivers._abpg_small.last_info[1])}
    info["abpg_gain"] = info["abpg"]
    name, power = card()
    print(f"card: {name}, power limit {power}", flush=True)
    result = {"card": name, "power_limit": power, "reps": args.reps, "workloads": {}}
    try:
        from oracle import ref_loader
        cpu_mod, cpu_kind = ref_loader.import_reference(), "reference package (oracle/_ref), host cores"
        cpu_port = False
    except ImportError:
        from oracle import accbpg_oracle as cpu_mod
        cpu_kind, cpu_port = "NumPy oracle port (the reference package is absent), host cores", True
    cpu = workloads(cpu_mod, cpu_port)
    old = config.fused_small
    try:
        for drv in drivers_run:
            for key, (desc, (f, h, L, x0), its, eps) in workloads(acc, False).items():
                if drv != "bpg":
                    desc = desc.replace("BPG ls_ratio=1.2", DRIVER_NAMES[drv])
                rec = {"workload": desc, "driver": drv}
                walls = {True: [], False: []}
                res = {}
                for fused in (True, False):                      # warm-up: modules, workspaces, pinned buffers
                    config.fused_small = fused
                    solve(acc, drv, f, h, L, x0, 50, eps, verbose=False)
                for _ in range(args.reps):
                    for fused in (True, False):
                        config.fused_small = fused
                        torch.cuda.synchronize()
                        t0 = time.perf_counter()
                        res[fused] = solve(acc, drv, f, h, L, x0, its, eps, verbose=False)
                        walls[fused].append(time.perf_counter() - t0)
                        if fused:
                            cl, trips = info[drv]()
                            rec["cluster_size"] = int(cl)
                            rec["line_search_trials" if drv == "bpg" else "trips"] = int(trips)
                for fused, tag in ((True, "fused"), (False, "operator_loop")):
                    F, D = res[fused]
                    best = min(walls[fused])
                    rec[tag] = {"iterations": len(F), "wall_s": walls[fused], "it_per_s_best": len(F) / best,
                                "F_last": float(F[-1]), "L_last" if drv == "bpg" else "G_last": float(D[-1])}
                (Ff, Df), (Fo, Do) = res[True], res[False]
                k = min(len(Ff), len(Fo))
                rec["fused_vs_operator_max_rel_dF"] = float(np.max(np.abs(Ff[:k] - Fo[:k]) /
                                                                   np.maximum(np.abs(Fo[:k]), 1e-3)))
                rec["speedup"] = rec["fused"]["it_per_s_best"] / rec["operator_loop"]["it_per_s_best"]
                cdesc, (fc, hc, Lc, x0c), _, _ = cpu[key]
                t0 = time.perf_counter()
                with contextlib.redirect_stdout(io.StringIO()):
                    rr = solve(cpu_mod, drv, fc, hc, Lc, x0c, its, eps, **({} if cpu_port else {"verbskip": 10 ** 9}))
                wall = time.perf_counter() - t0
                rec["cpu"] = {"what": cpu_kind, "iterations": len(rr[0]), "wall_s": wall, "it_per_s": len(rr[0]) / wall}
                result["workloads"][key if drv == "bpg" else f"{drv}_{key}"] = rec
                print(f"{drv} {key}: fused {rec['fused']['it_per_s_best']:.0f} it/s (cluster {rec['cluster_size']}), "
                      f"operator loop {rec['operator_loop']['it_per_s_best']:.0f} it/s, speed-up {rec['speedup']:.1f}x, "
                      f"{len(Ff)} vs {len(Fo)} iterations, max rel dF {rec['fused_vs_operator_max_rel_dF']:.1e}; "
                      f"CPU ({cpu_kind}) {rec['cpu']['it_per_s']:.0f} it/s, {len(rr[0])} iterations", flush=True)
    finally:
        config.fused_small = old
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(result, fh, indent=1)
    print(f"wrote {args.out}")


if __name__ == "__main__":
    main()
