"""Small D-optimal designs: BPG, ABPG or ABPG_gain as one launch (config.fused_small, csrc/small.cu) against the
operator-by-operator loop, alternated in one process after a warm-up, and the reference on the host cores.

    python tools/c1_time.py                      # C1: D_opt_design(80, 200), BPG with line search, 1000 iterations
    python tools/c1_time.py --drivers bpg,abpg,abpg_gain --out profiles/dopt_small_accel_r01.json

Workloads:
  bpg        D_opt_design(80, 200, randseed=10), BPG with line search (ls_ratio=1.2), 1000 iterations (BASELINE configs[0])
  abpg       the same instance, ABPG gamma=2 theta_eq=False, 1000 iterations (ipynb/ex_Dopt_random)
  abpg_gain  the same instance, ABPG_gain gamma=2 G0=0.1, 1000 iterations (ipynb/ex_Dopt_random), and housing
             (tests/golden/housing_libsvm.txt, 13 x 506), ABPG_gain gamma=2, 4000 iterations (ipynb/ex_Dopt_LIBSVM)
A solve may stop early on its stopping test, so every record carries the number of iterations actually run.
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

HOUSING = os.path.join(ROOT, "tests", "golden", "housing_libsvm.txt")


def workloads(mod, oracle_port, drivers_run):
    """key -> (description, driver, instance builder, keyword arguments, maxitrs) for the drivers asked for."""
    def design():
        return mod.D_opt_design(80, 200, randseed=10)

    def housing():
        if oracle_port:
            from accbpg_and_fw_b200.problems import load_libsvm_dense
            X, _ = load_libsvm_dense(HOUSING)
            return mod.D_opt_from_matrix(X)
        return mod.D_opt_libsvm(HOUSING)
    out = {}
    if "bpg" in drivers_run:
        out["bpg_80x200"] = ("D_opt_design(80,200,randseed=10), BPG ls_ratio=1.2, maxitrs=1000", "bpg", design,
                             dict(linesearch=True, ls_ratio=1.2), 1000)
    if "abpg" in drivers_run:
        out["abpg_80x200"] = ("D_opt_design(80,200,randseed=10), ABPG gamma=2 theta_eq=False, maxitrs=1000", "abpg",
                              design, dict(theta_eq=False), 1000)
    if "abpg_gain" in drivers_run:
        out["abpg_gain_80x200"] = ("D_opt_design(80,200,randseed=10), ABPG_gain gamma=2 G0=0.1, maxitrs=1000",
                                   "abpg_gain", design, dict(G0=0.1), 1000)
        out["abpg_gain_housing"] = ("D_opt_libsvm(housing) 13 x 506, ABPG_gain gamma=2, maxitrs=4000", "abpg_gain",
                                    housing, dict(), 4000)
    return out


def solve(mod, drv, inst, its, kw):
    """(F, the discrete sequence: L_k for BPG, G_k for ABPG, the gain for ABPG_gain) of one solve."""
    f, h, L, x0 = inst
    if drv == "bpg":
        r = mod.BPG(f, h, L, x0, maxitrs=its, **kw)
    elif drv == "abpg":
        r = mod.ABPG(f, h, L, x0, 2, its, **kw)
    else:
        r = mod.ABPG_gain(f, h, L, x0, 2, its, **kw)
    return r[1], r[2]


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
    ap.add_argument("--out", default=None, help="JSON file for the records (none by default)")
    ap.add_argument("--drivers", default="bpg", help="comma-separated: bpg, abpg, abpg_gain")
    args = ap.parse_args()
    drivers_run = args.drivers.split(",")
    if not set(drivers_run) <= {"bpg", "abpg", "abpg_gain"}:
        sys.exit("--drivers: choose from bpg, abpg, abpg_gain")
    if not torch.cuda.is_available():
        sys.exit("c1_time.py measures the GPU paths and needs a CUDA device")
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
    cpu = workloads(cpu_mod, cpu_port, drivers_run)
    old = config.fused_small
    try:
        for key, (desc, drv, build, kw, its) in workloads(acc, False, drivers_run).items():
            inst = build()
            kw = dict(kw, verbose=False)
            rec = {"workload": desc, "driver": drv}
            walls = {True: [], False: []}
            res = {}
            for fused in (True, False):                      # warm-up: modules, workspaces, pinned buffers
                config.fused_small = fused
                solve(acc, drv, inst, 50, kw)
            for _ in range(args.reps):
                for fused in (True, False):
                    config.fused_small = fused
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    res[fused] = solve(acc, drv, inst, its, kw)
                    walls[fused].append(time.perf_counter() - t0)
                    if fused:
                        inf = drivers._bpg_small.last_info if drv == "bpg" else drivers._abpg_small.last_info
                        if drv == "bpg":
                            rec["line_search_trials"] = int(inf[1])
                        else:
                            rec["cluster_size"], rec["trips"] = int(inf[2]), int(inf[1])
            for fused, tag in ((True, "fused"), (False, "operator_loop")):
                F, D = res[fused]
                best = min(walls[fused])
                rec[tag] = {"iterations": len(F), "wall_s": walls[fused], "it_per_s_best": len(F) / best,
                            "F_last": float(F[-1]), "L_last" if drv == "bpg" else "G_last": float(D[-1])}
            (Ff, Df), (Fo, Do) = res[True], res[False]
            k = min(len(Ff), len(Fo))
            rec["fused_vs_operator_max_rel_dF"] = float(np.max(np.abs(Ff[:k] - Fo[:k]) / np.maximum(np.abs(Fo[:k]), 1e-3)))
            rec["speedup"] = rec["fused"]["it_per_s_best"] / rec["operator_loop"]["it_per_s_best"]
            _, _, cbuild, ckw, _ = cpu[key]
            cinst = cbuild()
            t0 = time.perf_counter()
            with contextlib.redirect_stdout(io.StringIO()):
                rr = solve(cpu_mod, drv, cinst, its, ckw if cpu_port else dict(ckw, verbskip=10 ** 9))
            wall = time.perf_counter() - t0
            rec["cpu"] = {"what": cpu_kind, "iterations": len(rr[0]), "wall_s": wall, "it_per_s": len(rr[0]) / wall}
            result["workloads"][key] = rec
            print(f"{key}: fused {rec['fused']['it_per_s_best']:.0f} it/s"
                  f"{' (cluster %d)' % rec['cluster_size'] if 'cluster_size' in rec else ''}, "
                  f"operator loop {rec['operator_loop']['it_per_s_best']:.0f} it/s, speed-up {rec['speedup']:.1f}x, "
                  f"{len(Ff)} vs {len(Fo)} iterations, max rel dF {rec['fused_vs_operator_max_rel_dF']:.1e}; "
                  f"CPU ({cpu_kind}) {rec['cpu']['it_per_s']:.0f} it/s, {len(rr[0])} iterations", flush=True)
    finally:
        config.fused_small = old
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            json.dump(result, fh, indent=1)
        print(f"wrote {args.out}")


if __name__ == "__main__":
    main()
