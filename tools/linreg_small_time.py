"""Poisson and KL regression at the notebook shapes: BPG as one launch (config.fused_small, csrc/linreg_small.cu) against
the operator-by-operator loop, alternated in one process after a warm-up, and the reference on the host cores.

    python tools/linreg_small_time.py [--reps 3] [--out profiles/linreg_small_r01.json]

Instances: ipynb/ex_Poisson_L2 (Poisson_regrL1(200, 100, noise=1e-4, lamda=0, randseed=1), BPG with line search, 9000
iterations), ipynb/ex_KL_regr_L1 (KL_nonneg_regr(1000, 100, noise=0.01, lamdaL1=0.001, randseed=1), BPG with line
search, 4000 iterations) and a KL instance of the same shape on the simplex (ShannonEntropySimplex, 4000 iterations;
epsilon=0, because at the default 1e-14 it converges and stops after 170).
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
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("linreg_small_time.py measures the GPU paths and needs a CUDA device")
    import accbpg_and_fw_b200 as acc
    from accbpg_and_fw_b200 import config, drivers
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
        for key, (desc, (f, h, L, x0), its, eps) in workloads(acc, False).items():
            rec = {"workload": desc}
            walls = {True: [], False: []}
            res = {}
            for fused in (True, False):                      # warm-up: modules, workspaces, pinned buffers
                config.fused_small = fused
                acc.BPG(f, h, L, x0, maxitrs=50, verbose=False)
            for _ in range(args.reps):
                for fused in (True, False):
                    config.fused_small = fused
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    x, F, Ls, T = acc.BPG(f, h, L, x0, maxitrs=its, epsilon=eps, verbose=False)
                    walls[fused].append(time.perf_counter() - t0)
                    res[fused] = (F, Ls)
                    if fused:
                        rec["cluster_size"] = int(drivers._bpg_small.last_info[3])
                        rec["line_search_trials"] = int(drivers._bpg_small.last_info[1])
            for fused, tag in ((True, "fused"), (False, "operator_loop")):
                F, Ls = res[fused]
                best = min(walls[fused])
                rec[tag] = {"iterations": len(F), "wall_s": walls[fused], "it_per_s_best": len(F) / best,
                            "F_last": float(F[-1]), "L_last": float(Ls[-1])}
            (Ff, Lf), (Fo, Lo) = res[True], res[False]
            k = min(len(Ff), len(Fo))
            rec["fused_vs_operator_max_rel_dF"] = float(np.max(np.abs(Ff[:k] - Fo[:k]) / np.maximum(np.abs(Fo[:k]), 1e-3)))
            rec["speedup"] = rec["fused"]["it_per_s_best"] / rec["operator_loop"]["it_per_s_best"]
            cdesc, (fc, hc, Lc, x0c), _, _ = cpu[key]
            t0 = time.perf_counter()
            with contextlib.redirect_stdout(io.StringIO()):
                if cpu_port:
                    rr = cpu_mod.BPG(fc, hc, Lc, x0c, maxitrs=its, epsilon=eps)
                else:
                    rr = cpu_mod.BPG(fc, hc, Lc, x0c, maxitrs=its, epsilon=eps, verbskip=10 ** 9)
            wall = time.perf_counter() - t0
            rec["cpu"] = {"what": cpu_kind, "iterations": len(rr[1]), "wall_s": wall, "it_per_s": len(rr[1]) / wall}
            result["workloads"][key] = rec
            print(f"{key}: fused {rec['fused']['it_per_s_best']:.0f} it/s (cluster {rec['cluster_size']}), "
                  f"operator loop {rec['operator_loop']['it_per_s_best']:.0f} it/s, speed-up {rec['speedup']:.1f}x, "
                  f"{len(Ff)} vs {len(Fo)} iterations, max rel dF {rec['fused_vs_operator_max_rel_dF']:.1e}; "
                  f"CPU ({cpu_kind}) {rec['cpu']['it_per_s']:.0f} it/s", flush=True)
    finally:
        config.fused_small = old
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(result, fh, indent=1)
    print(f"wrote {args.out}")


if __name__ == "__main__":
    main()
