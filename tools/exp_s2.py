"""Round-2 session experiments at 500x50000 (run once per environment setting; prints one line each):
   FW-away iterations per second and the last F (bit comparison between settings), Burg-simplex prox time and its
   multiplier, ABPG iterations per second."""
import os, sys, time
import numpy as np, torch
sys.path.insert(0, ".")
import accbpg_and_fw_b200 as acc

what = sys.argv[1] if len(sys.argv) > 1 else "all"
tag = " ".join(f"{k}={v}" for k, v in sorted(os.environ.items()) if k.startswith("ACCBPG_"))
f, h, L, x0 = acc.D_opt_design(500, 50000, randseed=1)
x0d = torch.tensor(x0, device="cuda")

if what in ("fw", "all"):
    acc.D_opt_FW_away(f._Hd, x0d, 1e-12, 64, verbose=False)
    best = 0.0
    for rep in range(3):
        xa, Fa, SPa, SNa, Ta = acc.D_opt_FW_away(f._Hd, x0d, 1e-12, 1500, verbose=False)
        best = max(best, (len(Ta) - 1) / (Ta[-1] - Ta[0]))
    print(f"[fw] {tag} it/s {best:.0f} F_last {Fa[-1]!r} sum {float(np.sum(Fa))!r}", flush=True)

if what in ("burg", "all"):
    rt = f.rt
    g = f.gradient(x0d)
    out = torch.empty_like(g)
    for _ in range(5):
        z = h.div_prox_map(x0d, g, 1.0)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(200):
        z = h.div_prox_map(x0d, g, 1.0)
    b.record()
    torch.cuda.synchronize()
    print(f"[burg] {tag} us/call {a.elapsed_time(b) / 200 * 1e3:.1f} sum {float(z.sum())!r} z0 {float(z[0])!r}", flush=True)

if what in ("abpg", "all"):
    acc.ABPG(f, h, 1.0, x0d, gamma=2, maxitrs=5, verbose=False)
    best = 1e9
    for rep in range(3):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        x, F, G, T = acc.ABPG(f, h, 1.0, x0d, gamma=2, maxitrs=200, verbose=False)
        torch.cuda.synchronize()
        best = min(best, (time.perf_counter() - t0) / 200)
    print(f"[abpg] {tag} ms/it {best * 1e3:.4f} F_last {F[-1]!r}", flush=True)

if what == "fwc5":
    # D_opt_FW_away at 2000 x 1e6 (device-generated): iterations per second and a bit comparison between settings
    del f
    torch.cuda.empty_cache()
    gen = torch.Generator(device="cuda"); gen.manual_seed(5)
    m5, n5 = 2000, 1000000
    H5 = torch.randn(m5, n5, dtype=torch.float64, device="cuda", generator=gen)
    x5 = torch.full((n5,), 1.0 / n5, dtype=torch.float64, device="cuda")
    acc.D_opt_FW_away(H5, x5, 1e-12, 8, verbose=False)
    xa, Fa, SPa, SNa, Ta = acc.D_opt_FW_away(H5, x5, 1e-12, 130, verbose=False)
    print(f"[fwc5] {tag} it/s {(len(Ta) - 1) / (Ta[-1] - Ta[0]):.1f} F_last {Fa[-1]!r} sum {float(np.sum(Fa))!r}", flush=True)
