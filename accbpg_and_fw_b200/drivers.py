"""BPG, ABPG, ABPG_expo, ABPG_gain and ABDA over GPU-resident iterates.

Signatures, keyword defaults, return tuples and the host-side scalar control flow (theta
schedule, line search on L / gain / exponent, restart, stopping tests) are those of
accbpg/algorithms.py:11-514; the per-iteration arithmetic (oracles, Bregman steps, axpby,
dot products) is enqueued on the GPU through the asynchronous operator forms and the scalars a
decision needs come back in one pinned read per line-search trip.  Iterates stay in HBM: x0
is uploaded once, the last iterate is returned in the form x0 was given (NumPy or CUDA tensor).
History arrays are host NumPy float64, truncated to k+1 like the reference's.
"""
import time

import numpy as np
import torch

from . import _native as nat
from . import config
from .runtime import is_host, like_input

lib = nat.lib


def solve_theta(theta, gamma, gainratio=1):
    """Newton solve of (1-t)/t^gamma = gainratio/theta^gamma starting at theta.   algorithms.py:75-91."""
    ckg = theta ** gamma / gainratio
    cta = theta
    tol = 1e-6 * theta
    phi = cta ** gamma - ckg * (1 - cta)
    while abs(phi) > tol:
        cta = cta - phi / (gamma * cta ** (gamma - 1) + ckg)
        phi = cta ** gamma - ckg * (1 - cta)
    return cta


class _Loop:
    """Device-side helpers shared by the drivers (one instance per solve)."""

    def __init__(self, f, h, x0):
        self.f, self.h = f, h
        self.rt = f.rt
        self.host = is_host(x0)
        self.shard = getattr(f, "shard", None)
        self.x0 = self.rt.to_device(x0).clone()
        self.n = self.x0.numel()
        self.t0 = time.time()
        # carry the objective's linear image (M(x) for D-opt, A x for Poisson / KL) along with the iterates
        self.lin = bool(config.linear_images and getattr(f, "_lin_capable", False))
        self.reanchor = max(int(config.reanchor_every), 1)
        # column-sharded runs: the partial scalars of a trip (divergences, dot product, Psi) are summed over the
        # ranks by ONE all-reduce at fetch time instead of one per scalar
        self.sharded = self.shard is not None and self.shard.world > 1
        h._defer_reduce = self.sharded

    # ---- linear images (all no-ops returning None when the switch is off) -----------------------------------
    def img(self, x):
        return self.f._img_compute(x) if self.lin else None

    def img_combo(self, a, Ia, b, Ib):
        return self.f._img_axpby(a, Ia, b, Ib) if self.lin else None

    def img_refresh(self, k, x, Ix):
        """Every `reanchor_every` iterations the image of x is re-formed from x itself."""
        if self.lin and (k + 1) % self.reanchor == 0:
            return self.f._img_compute(x)
        return Ix

    def enq_f_img(self, x, Ix, slot):
        """f(x) -> slot, from the image when it is carried."""
        if self.lin:
            self.f._enqueue_img_pair(None, 0, Ix, 0, slot, None)
        else:
            self.f._enqueue(x, 0, slot, None)

    def enq_start(self, x, Ix, slot_x, y, Iy, flag_y, slot_y):
        """What an accelerated iteration starts with: f(x) -> slot_x (skipped when x is None) and
        (f(y), grad f(y)) -> (slot_y, g).  Returns g."""
        g = self.rt.empty(self.n)
        if self.lin:
            self.f._enqueue_img_pair(Ix if x is not None else None, slot_x, Iy, flag_y, slot_y, g)
        elif x is None:
            self.f._enqueue(y, flag_y, slot_y, g)
        elif hasattr(self.f, "_enqueue_pair"):
            self.f._enqueue_pair(x, slot_x, y, flag_y, slot_y, g)
        else:
            self.f._enqueue(x, 0, slot_x, None)
            self.f._enqueue(y, flag_y, slot_y, g)
        return g

    # vectors
    def combo(self, a, x, b, y):
        """a*x + b*y as a new vector (algorithms.py:147,150,243,250,369,374,478,483)."""
        rt = self.rt
        out = rt.empty(self.n)
        nat.check(lib.accbpg_vec_axpby(rt.ctx, rt.stream, self.n, float(a), x.data_ptr(), float(b), y.data_ptr(),
                                       out.data_ptr()))
        return out

    def div_prox(self, y, g, L):
        out = self.rt.empty(self.n)
        self.h._enq_div_prox(y, g, float(L), out)
        return out

    def prox(self, g, L):
        out = self.rt.empty(self.n)
        self.h._enq_prox(g, float(L), out)
        return out

    # scalars (enqueue only; `fetch` brings slots 0..5 back in one synchronising read)
    def enq_f(self, x, slot):
        self.f._enqueue(x, 0, slot, None)

    def enq_fg(self, x, slot):
        g = self.rt.empty(self.n)
        self.f._enqueue(x, 2, slot, g)
        return g

    def enq_f_and_grad(self, x, slot_x, y, flag_y, slot_y):
        """f(x) -> slot_x and (f(y), grad f(y)) -> slot_y: the two evaluations an accelerated iteration starts
        with (algorithms.py:135+148, :231+245, :347+371).  Objectives that can overlap the two chains do so."""
        g = self.rt.empty(self.n)
        if hasattr(self.f, "_enqueue_pair"):
            self.f._enqueue_pair(x, slot_x, y, flag_y, slot_y, g)
        else:
            self.f._enqueue(x, 0, slot_x, None)
            self.f._enqueue(y, flag_y, slot_y, g)
        return g

    def enq_psi(self, x):
        if self.h.has_psi:
            self.h._enq_extra_psi(x, self.rt.S_PSI)

    def enq_dot_diff(self, g, a, b):
        rt = self.rt
        nat.check(lib.accbpg_vec_dot_diff(rt.ctx, rt.stream, self.n, g.data_ptr(), a.data_ptr(), b.data_ptr(),
                                          rt.slot(rt.S_DOT)))

    def enq_div(self, x, y, slot):
        self.h._enq_divergence(x, y, slot)

    def _sum_partials(self):
        """Column-sharded runs: S_DXY, S_DZZ, S_DOT, S_PSI hold per-rank partials.  Their sums over the ranks go to the
        separate slots S_SUM.. (so a second fetch without new partials cannot add them up twice), and the same exchange
        makes the device status word the union over the ranks: one small kernel over NVLink peer memory, else collectives."""
        rt = self.rt
        src = rt.scal[rt.S_DXY:rt.S_PSI + 1]
        dst = rt.scal[rt.S_SUM:rt.S_SUM + 4]
        if self.shard.sum_scalars_into(src, dst):
            return
        dst.copy_(src)
        self.shard.sum_(dst)
        st = rt.scal[rt.S_SUM + 4:rt.S_SUM + 5]
        nat.check(lib.accbpg_ctx_status_export(rt.ctx, rt.stream, st.data_ptr()))
        self.shard.max_(st)
        nat.check(lib.accbpg_ctx_status_import(rt.ctx, rt.stream, st.data_ptr()))

    def _merge(self, vals):
        rt = self.rt
        vals[rt.S_DXY:rt.S_PSI + 1] = vals[rt.S_SUM:rt.S_SUM + 4]
        return vals

    def fetch(self):
        if not self.sharded:
            return self.rt.read(0, 7)      # S_F .. S_PSI and S_AUX0 in one pinned read
        self._sum_partials()
        return self._merge(self.rt.read(0, self.rt.S_SUM + 4))

    def fetch_async(self):
        """Deferred fetch: the copy is enqueued now, `fetch_wait(ticket)` collects it later."""
        if not self.sharded:
            return self.rt.read_async(0, 7)
        self._sum_partials()
        return self.rt.read_async(0, self.rt.S_SUM + 4)

    def fetch_wait(self, ticket):
        if not self.sharded:
            return self.rt.read_wait(ticket, 7)
        return self._merge(self.rt.read_wait(ticket, self.rt.S_SUM + 4))

    def pipeline_depth(self, verbose, restart=False):
        """How many iterations may be enqueued beyond the one whose scalars the host has seen (config.pipeline)."""
        return 1 if (config.pipeline and not verbose and not restart) else 0

    def psi(self, vals):
        return vals[self.rt.S_PSI] if self.h.has_psi else 0

    def now(self):
        return time.time() - self.t0

    def result(self, x):
        return like_input(x, self.host)


def _small_hkind(h):
    """ACCBPG_SMALL_H_* of the Legendre kernel h, or None when the linear-inverse fused solve does not cover its type."""
    from . import bregman as br
    names = {br.BurgEntropy: "BURG", br.BurgEntropyL1: "BURG_L1", br.BurgEntropyL2: "BURG_L2",
             br.ShannonEntropy: "SHANNON", br.ShannonEntropyL1: "SHANNON_L1",
             br.ShannonEntropySimplex: "SHANNON_SIMPLEX"}
    name = names.get(type(h))
    return None if name is None else nat.MACROS["ACCBPG_SMALL_H_" + name]


def _dopt_bpg_small(f, h, L, x, maxitrs, epsilon, linesearch, ls_ratio, t0):
    """accbpg_dopt_bpg_small: F, Ls, and T stamped evenly over the solve's wall time; None when H does not fit."""
    if lib.accbpg_dopt_bpg_small_smem_bytes(f.m, f.n) == 0:
        return None
    rt = f.rt
    hist = torch.empty(2 * maxitrs + 16, dtype=torch.float64, device=rt.device)
    H = f._Hd
    with rt.on_device():
        nat.check(lib.accbpg_dopt_bpg_small(rt.ctx, rt.stream, H.data_ptr(), f.m, f.n, H.stride(0), x.data_ptr(), float(L),
                                            float(ls_ratio), 1 if linesearch else 0, int(maxitrs), float(epsilon),
                                            float(h.eps), hist.data_ptr(), hist.data_ptr() + 8 * maxitrs,
                                            hist.data_ptr() + 16 * maxitrs))
    rt.read(rt.S_F, 1)                                   # synchronises and raises on a status bit
    hh = hist.cpu().numpy()
    k = int(hh[2 * maxitrs])
    _bpg_small.last_info = hh[2 * maxitrs:2 * maxitrs + 14].copy()
    F = hh[0:k].copy()
    Ls = hh[maxitrs:maxitrs + k].copy() if linesearch else np.ones(k) * L
    T = np.linspace(0.0, time.time() - t0, k + 1)[1:]
    return F, Ls, T


def _linreg_bpg_small(f, h, L, x, maxitrs, epsilon, linesearch, ls_ratio, t0):
    """accbpg_linreg_bpg_small: F, Ls, and T from the device clock at the top of each iteration, offset by the host time
    at which the solve was launched; None when A does not fit."""
    if lib.accbpg_linreg_bpg_small_smem_bytes(f.m, f.n) == 0:
        return None
    rt = f.rt
    hist = torch.empty(3 * maxitrs + 16, dtype=torch.float64, device=rt.device)
    A = f._Ad
    base = hist.data_ptr()
    with rt.on_device():
        t_launch = time.time() - t0
        nat.check(lib.accbpg_linreg_bpg_small(rt.ctx, rt.stream, f._kind, A.data_ptr(), f.m, f.n, A.stride(0),
                                              f._bd.data_ptr(), _small_hkind(h), float(h.lamda),
                                              float(getattr(h, "delta", 0.0)), x.data_ptr(), float(L), float(ls_ratio),
                                              1 if linesearch else 0, int(maxitrs), float(epsilon), base,
                                              base + 8 * maxitrs, base + 16 * maxitrs, base + 24 * maxitrs))
    rt.read(rt.S_F, 1)                                   # synchronises and raises on a status bit
    hh = hist.cpu().numpy()
    k = int(hh[3 * maxitrs])
    _bpg_small.last_info = hh[3 * maxitrs:3 * maxitrs + 4].copy()
    F = hh[0:k].copy()
    Ls = hh[maxitrs:maxitrs + k].copy()
    T = t_launch + hh[2 * maxitrs:2 * maxitrs + k] * 1e-9
    return F, Ls, T


def _bpg_small(f, h, L, x0, maxitrs, epsilon, linesearch, ls_ratio, verbose, verbskip):
    """config.fused_small: the whole BPG solve as one kernel launch when the instance is dense, unsharded and fits the
    shared memory of one SM (or of a small cluster): a D-optimal design with the Burg kernel on the simplex
    (accbpg_dopt_bpg_small), or Poisson / KL regression with a Burg or Shannon kernel (accbpg_linreg_bpg_small).
    Returns None when no fused solve applies.  `_bpg_small.last_info` keeps the kernel's info array."""
    from .objectives import DOptimalObj, PoissonRegression, KLdivRegression
    from .bregman import BurgEntropySimplex
    if not config.fused_small or maxitrs < 1 or not (L > 0) or not (ls_ratio > 1):
        return None
    if type(f) is DOptimalObj and type(h) is BurgEntropySimplex:
        solve = _dopt_bpg_small
    elif type(f) in (PoissonRegression, KLdivRegression) and _small_hkind(h) is not None:
        solve = _linreg_bpg_small
    else:
        return None
    if f.shard is not None or h.shard is not None:
        return None
    t0 = time.time()
    host = is_host(x0)
    x = f.rt.to_device(x0).clone()
    out = solve(f, h, L, x, maxitrs, epsilon, linesearch, ls_ratio, t0)
    if out is None:
        return None
    F, Ls, T = out
    if verbose:
        for i in range(0, len(F), max(int(verbskip), 1)):
            print("{0:6d}  {1:10.3e}  {2:10.3e}  {3:6.1f}".format(i, F[i], Ls[i], T[i]))
    return like_input(x, host), F, Ls, T


def _abpg_small(gain, f, h, L, x0, gamma, maxitrs, epsilon, theta_eq, restart, restart_rule, G0=1.0, ls_inc=1.2,
                ls_dec=1.2, checkdiv=False):
    """config.fused_small: the whole ABPG / ABPG_gain solve as one kernel launch on an unsharded instance that fits:
    - a DOptimalObj with BurgEntropySimplex whose H fits the shared memory of one SM or of a cluster of 2 or 4
      (accbpg_dopt_abpg_small).  It evaluates every point from scratch, which is what config.linear_images = False
      asks for; the operator loop's carried Gram images agree with that to rounding, so it is taken under both
      settings of config.linear_images;
    - a PoissonRegression / KLdivRegression instance whose A fits the shared memory of a cluster of at most 8 SMs, with
      a kernel that accbpg_linreg_bpg_small covers (accbpg_linreg_abpg_small).  It reproduces the operator loop's
      default scheme (carried linear images), so it is taken only with config.linear_images on.
    Returns None when no fused solve applies, else (x, hist rows, k, T): the history rows F, G / Gain, Gdiv, theta,
    D(x,y), D(z,z-) truncated to the k entries written, and T from the device clock at the top of each iteration, offset
    by the host time of the launch.  `_abpg_small.last_info` keeps the kernel's info array."""
    from .objectives import DOptimalObj, PoissonRegression, KLdivRegression
    from .bregman import BurgEntropySimplex
    if not config.fused_small or maxitrs < 1:
        return None
    dopt = type(f) is DOptimalObj and type(h) is BurgEntropySimplex
    if not dopt and (not config.linear_images or type(f) not in (PoissonRegression, KLdivRegression) or
                     _small_hkind(h) is None):
        return None
    if f.shard is not None or h.shard is not None:
        return None
    if not all(np.isfinite(v) and v > 0 for v in (L, gamma, G0, ls_inc, ls_dec)):
        return None
    if dopt and (not (np.isfinite(h.eps) and h.eps > 0) or lib.accbpg_dopt_abpg_small_smem_bytes(f.m, f.n) == 0):
        return None
    if not dopt and lib.accbpg_linreg_abpg_small_smem_bytes(f.m, f.n) == 0:
        return None
    t0 = time.time()
    rt = f.rt
    x = rt.to_device(x0).clone()
    hist = torch.empty(7 * maxitrs + 16, dtype=torch.float64, device=rt.device)
    base = hist.data_ptr()
    rule = nat.MACROS["ACCBPG_SMALL_RESTART_" + {'f': "F", 'g': "G"}.get(restart_rule, "NONE")]
    drv = nat.MACROS["ACCBPG_SMALL_DRV_" + ("ABPG_GAIN" if gain else "ABPG")]
    with rt.on_device():
        t_launch = time.time() - t0
        if dopt:
            H = f._Hd
            nat.check(lib.accbpg_dopt_abpg_small(
                rt.ctx, rt.stream, drv, H.data_ptr(), f.m, f.n, H.stride(0), x.data_ptr(), float(L), float(gamma),
                int(maxitrs), float(epsilon), float(h.eps), 1 if theta_eq else 0, 1 if restart else 0, rule, float(G0),
                float(ls_inc), float(ls_dec), 1 if checkdiv else 0, base, base + 8 * 7 * maxitrs))
        else:
            A = f._Ad
            nat.check(lib.accbpg_linreg_abpg_small(
                rt.ctx, rt.stream, drv, f._kind, A.data_ptr(), f.m, f.n, A.stride(0), f._bd.data_ptr(),
                _small_hkind(h), float(h.lamda), float(getattr(h, "delta", 0.0)), x.data_ptr(), float(L), float(gamma),
                int(maxitrs), float(epsilon), 1 if theta_eq else 0, 1 if restart else 0, rule, float(G0),
                float(ls_inc), float(ls_dec), 1 if checkdiv else 0, max(int(config.reanchor_every), 1), base,
                base + 8 * 7 * maxitrs))
    rt.read(rt.S_F, 1)                                   # synchronises and raises on a status bit
    hh = hist.cpu().numpy()
    info = hh[7 * maxitrs:7 * maxitrs + 16].copy()
    _abpg_small.last_info = info
    if info[3]:
        raise UnboundLocalError("cannot access local variable 'Gdr' where it is not associated with a value")
    k = int(info[0])
    rows = [hh[r * maxitrs:r * maxitrs + k].copy() for r in range(6)]
    T = t_launch + hh[6 * maxitrs:6 * maxitrs + k] * 1e-9
    return like_input(x, is_host(x0)), rows, k, T


def BPG(f, h, L, x0, maxitrs, epsilon=1e-14, linesearch=True, ls_ratio=1.2,
        verbose=True, verbskip=1):
    """Bregman proximal gradient.   accbpg/algorithms.py:11-72.   Returns (x, F, Ls, T)."""
    if verbose:
        print("\nBPG_LS method for min_{x in C} F(x) = f(x) + Psi(x)")
        print("     k      F(x)         Lk       time")
    fused = _bpg_small(f, h, L, x0, maxitrs, epsilon, linesearch, ls_ratio, verbose, verbskip)
    if fused is not None:
        return fused
    lp = _Loop(f, h, x0)
    rt = lp.rt
    F = np.zeros(maxitrs)
    Ls = np.ones(maxitrs) * L
    T = np.zeros(maxitrs)
    x = lp.x0
    if not linesearch and lp.pipeline_depth(verbose):
        # no decision inside an iteration: iteration k+1 is enqueued before F[k] has come back
        pend = None                      # (k, ticket)
        stop = None
        for k in range(maxitrs):
            g = lp.enq_fg(x, rt.S_F)
            lp.enq_psi(x)
            ticket = lp.fetch_async()
            x_next = lp.div_prox(x, g, L)
            if pend is not None:
                pk = pend[0]
                vals = lp.fetch_wait(pend[1])
                F[pk] = vals[rt.S_F] + lp.psi(vals)
                T[pk] = lp.now()
                if pk > 0 and abs(F[pk] - F[pk - 1]) < epsilon:
                    stop = pk            # x currently holds the iterate produced by iteration pk
                    break
            pend = (k, ticket)
            x = x_next
        if stop is None:
            pk = pend[0]
            vals = lp.fetch_wait(pend[1])
            F[pk] = vals[rt.S_F] + lp.psi(vals)
            T[pk] = lp.now()
            stop = pk
        return lp.result(x), F[0:stop + 1], Ls[0:stop + 1], T[0:stop + 1]
    # Line search: f(x_{k+1}) is what the accepted trial already evaluated, and so is the objective's linear image
    # (M(x) / A x) of the accepted point, so from the second iteration on the gradient comes from the carried image
    # (no second pass over H / A) and there is no host round trip before the first trial.
    Ix = lp.img(x)
    fx_known = None
    for k in range(maxitrs):
        g = lp.enq_start(None, None, None, x, Ix, 2, rt.S_F)
        lp.enq_psi(x)
        T[k] = lp.now()
        if fx_known is None or not linesearch:
            vals = lp.fetch()
            fx = vals[rt.S_F]
            F[k] = fx + lp.psi(vals)
        else:
            fx = fx_known
            F[k] = np.nan                                 # completed by the first trial's fetch (Psi rides along)
        if linesearch:
            L = L / ls_ratio
            while True:
                x1 = lp.div_prox(x, g, L)
                Ix1 = lp.img(x1)
                lp.enq_f_img(x1, Ix1, rt.S_F2)
                lp.enq_dot_diff(g, x1, x)
                lp.enq_div(x1, x, rt.S_DXY)
                vals = lp.fetch()
                if np.isnan(F[k]):
                    F[k] = fx + lp.psi(vals)
                if vals[rt.S_F2] > fx + vals[rt.S_DOT] + L * vals[rt.S_DXY]:      # algorithms.py:53
                    L = L * ls_ratio
                else:
                    break
            x = x1
            Ix = Ix1
            fx_known = vals[rt.S_F2]
        else:
            x = lp.div_prox(x, g, L)
            Ix = lp.img(x)
        Ls[k] = L
        if verbose and k % verbskip == 0:
            print("{0:6d}  {1:10.3e}  {2:10.3e}  {3:6.1f}".format(k, F[k], L, T[k]))
        if k > 0 and abs(F[k] - F[k - 1]) < epsilon:
            break
    return lp.result(x), F[0:k + 1], Ls[0:k + 1], T[0:k + 1]


def _restart_now(lp, rule, F, k, g, x, x_1):
    """Restart predicate of algorithms.py:168, :279, :406."""
    if rule == 'f':
        return F[k] > F[k - 1]
    if rule == 'g':
        lp.enq_dot_diff(g, x, x_1)
        return lp.fetch()[lp.rt.S_DOT] > 0
    return False


def ABPG(f, h, L, x0, gamma, maxitrs, epsilon=1e-14, theta_eq=False,
         restart=False, restart_rule='g', verbose=True, verbskip=1):
    """Accelerated BPG.   accbpg/algorithms.py:94-180.   Returns (x, F, G, T)."""
    if verbose:
        print("\nABPG method for minimize_{x in C} F(x) = f(x) + Psi(x)")
        print("     k      F(x)       theta        TSG       D(x+,y)     D(z+,z)     time")
    fused = _abpg_small(False, f, h, L, x0, gamma, maxitrs, epsilon, theta_eq, restart, restart_rule)
    if fused is not None:
        x, (F, G, _, Th, Dxy, Dzz), k, T = fused
        if verbose:
            for i in range(0, k, max(int(verbskip), 1)):
                print("{0:6d}  {1:10.3e}  {2:10.3e}  {3:10.3e}  {4:10.3e}  {5:10.3e}  {6:6.1f}".format(
                    i, F[i], Th[i], G[i], Dxy[i], Dzz[i], T[i]))
        return x, F, G, T
    lp = _Loop(f, h, x0)
    rt = lp.rt
    F = np.zeros(maxitrs)
    G = np.zeros(maxitrs)
    T = np.zeros(maxitrs)
    x = lp.x0
    z = lp.x0.clone()
    Ix = lp.img(x)           # linear image of x (None when config.linear_images is off); z starts at x
    Iz = Ix
    theta = 1.0
    kk = 0
    depth = lp.pipeline_depth(verbose, restart)
    pend = None                  # (k, ticket, theta_k) of the iteration whose scalars are still in flight
    for k in range(maxitrs):
        # F[k] = f(x_k) is only recorded (and used by restart rule 'f' at the end of the iteration), so it is
        # evaluated together with the gradient at y_k and fetched with the divergences: one host sync per iteration.
        if not depth or k == 0:
            T[k] = lp.now()          # pipelined: T[k] is stamped when iteration k-1's scalars arrive
        z_1, x_1 = z, x
        Iz_1, Ix_1 = Iz, Ix
        if theta_eq and kk > 0:
            theta = solve_theta(theta, gamma)
        else:
            theta = gamma / (kk + gamma)
        y = lp.combo(1 - theta, x, theta, z_1)
        Iy = lp.img_combo(1 - theta, Ix_1, theta, Iz_1)
        g = lp.enq_start(x, Ix_1, rt.S_F, y, Iy, 1, rt.S_F2)
        lp.enq_psi(x)
        z = lp.div_prox(z_1, g, theta ** (gamma - 1) * L)
        Iz = lp.img(z)
        x = lp.combo(1 - theta, x, theta, z)
        Ix = lp.img_refresh(k, x, lp.img_combo(1 - theta, Ix_1, theta, Iz))
        lp.enq_div(x, y, rt.S_DXY)
        lp.enq_div(z, z_1, rt.S_DZZ)
        if depth:
            # deferred read: iteration k+1 is enqueued before these scalars are looked at; when the stopping test of
            # iteration k-1 fires, the iteration just enqueued is dropped and the iterate it started from is returned
            ticket = lp.fetch_async()
            if pend is not None:
                pk, ptheta = pend[0], pend[2]
                vals = lp.fetch_wait(pend[1])
                T[pk + 1] = lp.now()
                F[pk] = vals[rt.S_F] + lp.psi(vals)
                G[pk] = vals[rt.S_DXY] / vals[rt.S_DZZ] / ptheta ** gamma
                if vals[rt.S_DZZ] < epsilon:
                    return lp.result(x_1), F[0:pk + 1], G[0:pk + 1], T[0:pk + 1]
            pend = (k, ticket, theta)
            kk += 1
            continue
        vals = lp.fetch()
        F[k] = vals[rt.S_F] + lp.psi(vals)
        dxy, dzz = vals[rt.S_DXY], vals[rt.S_DZZ]
        Gdr = dxy / dzz / theta ** gamma
        G[k] = Gdr
        if verbose and k % verbskip == 0:
            print("{0:6d}  {1:10.3e}  {2:10.3e}  {3:10.3e}  {4:10.3e}  {5:10.3e}  {6:6.1f}".format(
                k, F[k], theta, Gdr, dxy, dzz, T[k]))
        kk += 1
        if restart and k > 0:
            if _restart_now(lp, restart_rule, F, k, g, x, x_1):
                theta = 1.0
                kk = 0
                z = x
                Iz = Ix
        if dzz < epsilon:
            break
    if depth and pend is not None:
        pk, ptheta = pend[0], pend[2]
        vals = lp.fetch_wait(pend[1])
        F[pk] = vals[rt.S_F] + lp.psi(vals)
        G[pk] = vals[rt.S_DXY] / vals[rt.S_DZZ] / ptheta ** gamma
    return lp.result(x), F[0:k + 1], G[0:k + 1], T[0:k + 1]


def ABPG_expo(f, h, L, x0, gamma0, maxitrs, epsilon=1e-14, delta=0.2,
              theta_eq=True, checkdiv=False, Gmargin=10, restart=False,
              restart_rule='g', verbose=True, verbskip=1):
    """ABPG with exponent adaption.   accbpg/algorithms.py:183-292.   Returns (x, F, Gamma, G, T)."""
    if verbose:
        print("\nABPG_expo method for min_{x in C} F(x) = f(x) + Psi(x)")
        print("     k      F(x)       theta       gamma        TSG       D(x+,y)     D(z+,z)     time")
    lp = _Loop(f, h, x0)
    rt = lp.rt
    F = np.zeros(maxitrs)
    G = np.zeros(maxitrs)
    Gamma = np.ones(maxitrs) * gamma0
    T = np.zeros(maxitrs)
    gamma = gamma0
    x = lp.x0
    z = lp.x0.clone()
    Ix = lp.img(x)           # linear image of x (None when config.linear_images is off); z starts at x
    Iz = Ix
    theta = 1.0
    kk = 0
    fx_known = None      # f(x_k) when the previous iteration's line search already evaluated it at this very vector
    for k in range(maxitrs):
        T[k] = lp.now()
        lp.enq_psi(x)
        z_1, x_1 = z, x
        if theta_eq and kk > 0:
            theta = solve_theta(theta, gamma)
        else:
            theta = gamma / (kk + gamma)
        Iz_1, Ix_1 = Iz, Ix
        y = lp.combo(1 - theta, x_1, theta, z_1)
        Iy = lp.img_combo(1 - theta, Ix_1, theta, Iz_1)
        # F[k] = f(x_k) rides along with func_grad(y_k) unless the last line search already produced it
        g = lp.enq_start(x_1 if fx_known is None else None, Ix_1, rt.S_AUX0, y, Iy, 2, rt.S_F2)
        fy = None
        again = True
        while again:
            z = lp.div_prox(z_1, g, theta ** (gamma - 1) * L)
            Iz = lp.img(z)
            x = lp.combo(1 - theta, x_1, theta, z)
            Ix = lp.img_combo(1 - theta, Ix_1, theta, Iz)
            lp.enq_div(x, y, rt.S_DXY)
            lp.enq_div(z, z_1, rt.S_DZZ)
            if not checkdiv:
                lp.enq_f_img(x, Ix, rt.S_F)
                lp.enq_dot_diff(g, x, y)
            vals = lp.fetch()
            if fy is None:
                fy = vals[rt.S_F2]
                F[k] = (vals[rt.S_AUX0] if fx_known is None else fx_known) + lp.psi(vals)
            dxy, dzz = vals[rt.S_DXY], vals[rt.S_DZZ]
            Gdr = dxy / dzz / theta ** gamma
            if checkdiv:
                again = (dxy > Gmargin * (theta ** gamma) * dzz)
            else:
                again = (vals[rt.S_F] > fy + vals[rt.S_DOT] + theta ** gamma * L * dzz)     # algorithms.py:260
            if again and gamma > 1:
                gamma = max(gamma - delta, 1)
            else:
                again = False
        fx_known = None if checkdiv else vals[rt.S_F]       # f at the accepted x: next iteration's F[k+1]
        Ix_new = lp.img_refresh(k, x, Ix)
        if Ix_new is not Ix:
            fx_known = None                                 # re-anchored: F[k+1] is evaluated from the fresh image
        Ix = Ix_new
        G[k] = Gdr
        Gamma[k] = gamma
        if verbose and k % verbskip == 0:
            print("{0:6d}  {1:10.3e}  {2:10.3e}  {3:10.3e}  {4:10.3e}  {5:10.3e}  {6:10.3e}  {7:6.1f}".format(
                k, F[k], theta, gamma, Gdr, dxy, dzz, T[k]))
        kk += 1
        if restart:
            if _restart_now(lp, restart_rule, F, k, g, x, x_1):
                theta = 1.0
                kk = 0
                z = x
                Iz = Ix
        if dzz < epsilon:
            break
    return lp.result(x), F[0:k + 1], Gamma[0:k + 1], G[0:k + 1], T[0:k + 1]


def ABPG_gain(f, h, L, x0, gamma, maxitrs, epsilon=1e-14, G0=1,
              ls_inc=1.2, ls_dec=1.2, theta_eq=True, checkdiv=False,
              restart=False, restart_rule='g', verbose=True, verbskip=1):
    """ABPG with gain adaption.   accbpg/algorithms.py:295-420.   Returns (x, F, Gain, Gdiv, Gavg, T)."""
    if verbose:
        print("\nABPG_gain method for min_{x in C} F(x) = f(x) + Psi(x)")
        print("     k      F(x)       theta         Gk         TSG       D(x+,y)     D(z+,z)      Gavg       time")
    fused = _abpg_small(True, f, h, L, x0, gamma, maxitrs, epsilon, theta_eq, restart, restart_rule, G0, ls_inc, ls_dec,
                        checkdiv)
    if fused is not None:
        x, (F, Gain, Gdiv, Th, Dxy, Dzz), k, T = fused
        Gavg = np.zeros(k)
        sumlogG = gamma * np.log(G0)
        for i in range(k):
            sumlogG += np.log(Gain[i])
            Gavg[i] = np.exp(sumlogG / (gamma + i))
        if verbose:
            for i in range(0, k, max(int(verbskip), 1)):
                print("{0:6d}  {1:10.3e}  {2:10.3e}  {3:10.3e}  {4:10.3e}  {5:10.3e}  {6:10.3e}  {7:10.3e}  {8:6.1f}".format(
                    i, F[i], Th[i], Gain[i], Gdiv[i], Dxy[i], Dzz[i], Gavg[i], T[i]))
        return x, F, Gain, Gdiv, Gavg, T
    lp = _Loop(f, h, x0)
    rt = lp.rt
    F = np.zeros(maxitrs)
    Gain = np.ones(maxitrs) * G0
    Gdiv = np.zeros(maxitrs)
    Gavg = np.zeros(maxitrs)
    T = np.zeros(maxitrs)
    x = lp.x0
    z = lp.x0.clone()
    Ix = lp.img(x)           # linear image of x (None when config.linear_images is off); z starts at x
    Iz = Ix
    G = G0
    sumlogG = gamma * np.log(G)
    theta = 1.0
    kk = 0
    fx_known = None      # f(x_k) when the previous iteration's line search already evaluated it at this very vector
    for k in range(maxitrs):
        T[k] = lp.now()
        lp.enq_psi(x)
        z_1, x_1 = z, x
        Iz_1, Ix_1 = Iz, Ix
        G_1 = G
        theta_1 = theta
        G = G / ls_dec
        again = True
        first = True
        while again:
            if kk > 0:
                if theta_eq:
                    theta = solve_theta(theta_1, gamma, G / G_1)
                else:
                    alpha = G / G_1
                    theta = theta_1 * ((1 + alpha * (gamma - 1)) / (gamma * alpha + theta_1))
            y = lp.combo(1 - theta, x_1, theta, z_1)
            Iy = lp.img_combo(1 - theta, Ix_1, theta, Iz_1)
            # F[k] = f(x_k) rides along with the first func_grad(y) unless the last line search already produced it
            g = lp.enq_start(x_1 if (first and fx_known is None) else None, Ix_1, rt.S_AUX0, y, Iy, 2, rt.S_F2)
            z = lp.div_prox(z_1, g, theta ** (gamma - 1) * G * L)
            Iz = lp.img(z)
            x = lp.combo(1 - theta, x_1, theta, z)
            Ix = lp.img_combo(1 - theta, Ix_1, theta, Iz)
            lp.enq_div(x, y, rt.S_DXY)
            lp.enq_div(z, z_1, rt.S_DZZ)
            if not checkdiv:
                # the reference evaluates f(x) only when dzz >= epsilon; doing it unconditionally here saves a
                # second round trip per trip and does not change any recorded value
                lp.enq_f_img(x, Ix, rt.S_F)
                lp.enq_dot_diff(g, x, y)
            vals = lp.fetch()
            if first:
                F[k] = (vals[rt.S_AUX0] if fx_known is None else fx_known) + lp.psi(vals)
                first = False
            fy = vals[rt.S_F2]
            dxy, dzz = vals[rt.S_DXY], vals[rt.S_DZZ]
            if dzz < epsilon:
                break
            Gdr = dxy / dzz / theta ** gamma
            if checkdiv:
                again = (Gdr > G)
            else:
                again = (vals[rt.S_F] > fy + vals[rt.S_DOT] + theta ** gamma * G * L * dzz)   # algorithms.py:387
            if again:
                G = G * ls_inc
        fx_known = None if checkdiv else vals[rt.S_F]       # f at the accepted x: next iteration's F[k+1]
        Ix_new = lp.img_refresh(k, x, Ix)
        if Ix_new is not Ix:
            fx_known = None                                 # re-anchored: F[k+1] is evaluated from the fresh image
        Ix = Ix_new
        Gain[k] = G
        Gdiv[k] = Gdr       # stale (or unbound on the very first trip) after the break above, as in the reference
        sumlogG += np.log(G)
        Gavg[k] = np.exp(sumlogG / (gamma + k))
        if verbose and k % verbskip == 0:
            print("{0:6d}  {1:10.3e}  {2:10.3e}  {3:10.3e}  {4:10.3e}  {5:10.3e}  {6:10.3e}  {7:10.3e}  {8:6.1f}".format(
                k, F[k], theta, G, Gdr, dxy, dzz, Gavg[k], T[k]))
        kk += 1
        if restart:
            if _restart_now(lp, restart_rule, F, k, g, x, x_1):
                theta = 1.0
                kk = 0
                z = x
                Iz = Ix
        if dzz < epsilon:
            break
    return lp.result(x), F[0:k + 1], Gain[0:k + 1], Gdiv[0:k + 1], Gavg[0:k + 1], T[0:k + 1]


def ABDA(f, h, L, x0, gamma, maxitrs, epsilon=1e-14, theta_eq=True,
         verbose=True, verbskip=1):
    """Accelerated Bregman dual averaging.   accbpg/algorithms.py:423-514.   Returns (x, F, G, T)."""
    if verbose:
        print("\nABDA method for min_{x in C} F(x) = f(x) + Psi(x)")
        print("     k      F(x)       theta        TSG       D(x+,y)     D(z+,z)     time")
    lp = _Loop(f, h, x0)
    rt = lp.rt
    F = np.zeros(maxitrs)
    G = np.zeros(maxitrs)
    T = np.zeros(maxitrs)
    x = lp.x0
    z = lp.x0.clone()
    Ix = lp.img(x)           # linear image of x (None when config.linear_images is off); z starts at x
    Iz = Ix
    theta = 1.0
    kk = 0
    gavg = rt.empty(lp.n).zero_()
    csum = 0
    depth = lp.pipeline_depth(verbose)
    pend = None
    for k in range(maxitrs):
        if not depth or k == 0:
            T[k] = lp.now()
        z_1, x_1 = z, x
        if theta_eq and kk > 0:
            theta = solve_theta(theta, gamma)
        else:
            theta = gamma / (kk + gamma)
        Iz_1, Ix_1 = Iz, Ix
        y = lp.combo(1 - theta, x_1, theta, z_1)
        Iy = lp.img_combo(1 - theta, Ix_1, theta, Iz_1)
        g = lp.enq_start(x_1, Ix_1, rt.S_F, y, Iy, 1, rt.S_F2)      # F[k] = f(x_k) rides along with the gradient at y_k
        lp.enq_psi(x_1)
        wgt = theta ** (1 - gamma)
        gavg = lp.combo(1.0, gavg, wgt, g)            # gavg + theta^(1-gamma) * g   (1.0*gavg is exact)
        csum = csum + wgt
        # gavg / csum: a true division, not a multiplication by the reciprocal (algorithms.py:482)
        gq = rt.empty(lp.n)
        nat.check(lib.accbpg_vec_divide(rt.ctx, rt.stream, lp.n, gavg.data_ptr(), float(csum), gq.data_ptr()))
        z = lp.prox(gq, L / csum)
        Iz = lp.img(z)
        x = lp.combo(1 - theta, x_1, theta, z)
        Ix = lp.img_refresh(k, x, lp.img_combo(1 - theta, Ix_1, theta, Iz))
        lp.enq_div(x, y, rt.S_DXY)
        lp.enq_div(z, z_1, rt.S_DZZ)
        if depth:
            ticket = lp.fetch_async()
            if pend is not None:
                pk, ptheta = pend[0], pend[2]
                vals = lp.fetch_wait(pend[1])
                T[pk + 1] = lp.now()
                F[pk] = vals[rt.S_F] + lp.psi(vals)
                G[pk] = vals[rt.S_DXY] / vals[rt.S_DZZ] / ptheta ** gamma
                if vals[rt.S_DZZ] < epsilon:
                    return lp.result(x_1), F[0:pk + 1], G[0:pk + 1], T[0:pk + 1]
            pend = (k, ticket, theta)
            kk += 1
            continue
        vals = lp.fetch()
        F[k] = vals[rt.S_F] + lp.psi(vals)
        dxy, dzz = vals[rt.S_DXY], vals[rt.S_DZZ]
        Gdr = dxy / dzz / theta ** gamma
        G[k] = Gdr
        if verbose and k % verbskip == 0:
            print("{0:6d}  {1:10.3e}  {2:10.3e}  {3:10.3e}  {4:10.3e}  {5:10.3e}  {6:6.1f}".format(
                k, F[k], theta, Gdr, dxy, dzz, T[k]))
        kk += 1
        if dzz < epsilon:
            break
    if depth and pend is not None:
        pk, ptheta = pend[0], pend[2]
        vals = lp.fetch_wait(pend[1])
        F[pk] = vals[rt.S_F] + lp.psi(vals)
        G[pk] = vals[rt.S_DXY] / vals[rt.S_DZZ] / ptheta ** gamma
    return lp.result(x), F[0:k + 1], G[0:k + 1], T[0:k + 1]
