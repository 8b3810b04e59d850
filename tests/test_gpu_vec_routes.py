"""Vector, Bregman, LMO and Poisson/KL product kernels (vecops.cu, linreg.cu) through the C ABI, route by route, against
an extended-precision reference.

Every driver iteration calls these kernels, and their host code picks a launch form from n and the SM count: the
Burg-simplex root-find keeps EPT = 1, 2, 3, 4, 6 or 8 elements per thread in registers (EPT 0 re-reads `out`), gathers
its block partials in one hop up to 128 blocks and through a leader block above; reductions and maps stop growing their
grid at 4 and 8 blocks per SM; the products take 16-byte or scalar loads, one or several column segments and up to 256
row chunks.  The sizes below are derived from the SM count so that each of those forms runs, and one profiler run shows
that it did.  Checks are bit for bit where the kernel and a NumPy restatement round the same operations (the files are
built with -fmad=false, and division and sqrt are correctly rounded), <= 2 ulp per element where exp or log is involved,
and, for sums, the worst-case bound of the kernel's summation tree: (passes + 2 log2(threads) + k) 2^-53 sum|t_i|.
Every output buffer is followed by GUARD sentinel entries that must stay untouched.
"""
import json
import math
import os
import re
import tempfile

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

F64 = torch.float64
LD = np.longdouble
GUARD = 8                    # guard entries after every output buffer
SENTINEL = 7.25e17           # what the guards hold; no result of these tests can equal it
EPS = 2.0 ** -53
EXTENDED = np.finfo(np.longdouble).nmant >= 63
SLACK = 1.0 if EXTENDED else 2.0     # without an extended long double the reference carries rounding of its own
ULPS = 2 if EXTENDED else 3
DELTA = 1e-20                # ShannonEntropy's clamp
BURG_THREADS = 512
BURG_EPT = (1, 2, 3, 4, 6, 8)        # register forms of burg_simplex_x_kernel; 0 is the generic one
BURG_EPS = 1e-8


@pytest.fixture(scope="module")
def acc():
    import accbpg_and_fw_b200 as a
    return a


@pytest.fixture(scope="module")
def rt(acc):
    return acc.Runtime.get()


# ------------------------------------------------------------------------------------------------------- harness
def _lib():
    from accbpg_and_fw_b200 import _native
    return _native


def call(rt, name, *args):
    """One C ABI call on the runtime's context and stream; returns the status word (the read synchronises)."""
    nat = _lib()
    nat.check(getattr(nat.lib, name)(rt.ctx, rt.stream, *args))
    return rt.read_raw(0, 0)[1]


def dev(a, off=0):
    """a on the device at offset `off` doubles of a NaN-filled buffer (a read outside the vector shows as NaN)."""
    a = np.ascontiguousarray(a, dtype=np.float64)
    buf = torch.full((off + a.size + GUARD,), float("nan"), dtype=F64, device="cuda")
    buf[off:off + a.size] = torch.from_numpy(a).cuda()
    return buf[off:off + a.size]


class Out:
    """An output of n doubles (preset to NaN, so an element the kernel skips shows) followed by GUARD sentinels."""

    def __init__(self, n, fill=float("nan")):
        self.n = n
        self.buf = torch.full((n + GUARD,), SENTINEL, dtype=F64, device="cuda")
        self.buf[:n] = fill

    @property
    def ptr(self):
        return self.buf.data_ptr()

    def get(self, what=""):
        h = self.buf.cpu().numpy()
        assert np.all(h[self.n:] == SENTINEL), ("written past the output", what)
        return h[:self.n].copy()


def same_bits(a, b):
    a, b = np.ascontiguousarray(a, dtype=np.float64), np.ascontiguousarray(b, dtype=np.float64)
    return a.shape == b.shape and np.array_equal(a.view(np.int64), b.view(np.int64))


def ulp_diff(a, b):
    """Per-element distance in units in the last place (both arrays finite)."""
    ka = np.ascontiguousarray(a, dtype=np.float64).view(np.int64)
    kb = np.ascontiguousarray(b, dtype=np.float64).view(np.int64)
    ka = np.where(ka < 0, np.int64(-2 ** 63) - ka, ka)
    kb = np.where(kb < 0, np.int64(-2 ** 63) - kb, kb)
    return np.abs(ka - kb)


def cdiv(a, b):
    return -(-a // b)


def tree(n, width, k):
    """Worst-case relative rounding of a sum of n terms over `width` threads: ceil(n/width) sequential adds per thread,
    two fixed trees of depth log2(width) (block and grid), k for forming a term; in units of sum|t_i|."""
    return (cdiv(n, width) + 2 * math.ceil(math.log2(width)) + k) * EPS * SLACK


# ------------------------------------------------------------------------------------------------------- host plans
def grid_for(sms, n, threads, items, per_sm):
    """common.cuh grid_for."""
    return int(max(1, min(cdiv(n, threads * items), min(sms * per_sm, 1184))))


def red_grid(sms, n):
    return grid_for(sms, n, 256, 4, 4)


def burg_route(n, sms):
    """burgx_launch: (grid, EPT, one-hop exchange).  ptxas gives every variant 128 registers at 512 threads, so one
    block per SM; the profiler test below fails if the grid the kernel really got differs."""
    grid = max(1, min(cdiv(n, BURG_THREADS), min(sms, 296)))
    if n <= 8 * BURG_THREADS:
        grid = 1
    per = cdiv(n, grid * BURG_THREADS)
    ept = next((e for e in BURG_EPT if per <= e), 0)
    return grid, ept, grid <= 128


def burg_sizes(sms):
    """One size per route the suite did not run before: one block with EPT 2..8, the leader exchange with EPT 1, the
    multi-block EPT 3..8 (each one past the previous form's limit, and 8 S at the EPT 8 limit), EPT 0 one past it."""
    S = BURG_THREADS * sms
    sizes = [513, 1100, 1800, 2900, 4096]
    if sms > 128:
        sizes.append((128 * BURG_THREADS + S) // 2 + 1)
    return sizes + [2 * S + 1, 3 * S + 1, 4 * S + 1, 6 * S + 1, 8 * S, 8 * S + 1]


def linreg_plan(m, n, sms):
    """linreg.cu linreg_plan: (column segments of A x, row chunks of A^T r, rows per chunk)."""
    nseg = max(1, cdiv(n, 1 << 16))
    colblocks = cdiv(n, 512)
    want = min(cdiv(sms * 16, colblocks), cdiv(m, 64))
    nchunk = int(min(max(want, 1), 256))
    return nseg, nchunk, cdiv(m, nchunk)


# ------------------------------------------------------------------------------------------------------- 1. Burg simplex
def burg_gg(g, y, L):
    """gg as the kernel forms it: (g - L*(-1/y))/L, or g/L."""
    return g / L if y is None else (g - L * (-1.0 / y)) / L


_BURG_IN = {}


def burg_inputs(n, sms):
    """g Gaussian, y log-uniform over 1e-9 .. 1, and at least 8 exact ties at the minimum of gg (same g and y): one at
    n - 1 and one in the last register slot its thread fills, first + (passes - 1) * stride (EPT 0: the last pass)."""
    if n not in _BURG_IN:
        grid = burg_route(n, sms)[0]
        rng = np.random.RandomState(n % 100003 + 5)
        g = rng.randn(n)
        y = 10.0 ** rng.uniform(-9.0, 0.0, n)
        stride = grid * BURG_THREADS
        base = (n - 1) // stride * stride
        ties = {n - 1, base + (n - 1 - base) // 2}
        while len(ties) < 8:
            ties.add(int(rng.randint(n)))
        idx = np.array(sorted(ties))
        g[idx] = g.min() - 1.0
        y[idx] = 1.0
        _BURG_IN[n] = (g, y, idx)
    return _BURG_IN[n]


def burg_replay(gg, eps=BURG_EPS):
    """The recurrence of BurgEntropySimplex in FP64 NumPy: (bisection steps, Newton steps).  The same vectorised
    restatement as test_gpu_operators.py::test_burg_simplex_newton_replay, with the kernel's two iteration guards
    (2000 bisections, 200 Newton steps) added.  The bisection count is always 0 here: at c = -min(gg) + 1 the minimum
    term alone is 1, so the sum is never below 1 and the halving loop never runs; only the Newton count is informative."""
    cmin = -gg.min()
    c = cmin + 1
    nbis = 0
    while np.sum(1 / (gg + c)) - 1 < 0 and nbis < 2000:
        c = (cmin + c) / 2.0
        nbis += 1
    fc = np.sum(1 / (gg + c)) - 1
    nnewt = 0
    while abs(fc) > eps:
        fpc = np.sum(-1.0 / (gg + c) ** 2)
        if (c - (c - fc / fpc)) == 0:
            break
        c = c - fc / fpc
        fc = np.sum(1 / (gg + c)) - 1
        nnewt += 1
        if nnewt >= 200:
            break
    return nbis, nnewt


_REPLAY = {}


def check_burg_result(x, info, gg, grid, key, what):
    """(a) x = 1/(gg + c) bit for bit; (b) the step counts of the FP64 replay; (c) sum x = 1 to eps plus the rounding
    of the kernel's sum, in long double."""
    nbis, nnewt, c = info
    assert np.isfinite(c), what
    fin = np.isfinite(gg)
    assert same_bits(x, 1.0 / (gg[fin] + c)), (what, "x != 1/(gg + c)")
    if key not in _REPLAY:
        _REPLAY[key] = burg_replay(gg)
    assert (int(nbis), int(nnewt)) == _REPLAY[key], (what, (nbis, nnewt), _REPLAY[key])
    t = 1.0 / (gg.astype(LD) + LD(c))
    s = np.sum(t)
    bar = BURG_EPS + (cdiv(gg.size, BURG_THREADS * grid) + 2 * math.ceil(math.log2(BURG_THREADS * grid)) + 4) \
        * EPS * SLACK * float(s)
    assert abs(float(s - 1)) <= bar, (what, float(s - 1), bar)


def burg_prox_call(rt, g_d, y_d, n, L):
    out, info = Out(n), Out(3)
    st = call(rt, "accbpg_burg_simplex_prox", n, None if y_d is None else y_d.data_ptr(), g_d.data_ptr(), L, BURG_EPS,
              out.ptr, info.ptr)
    assert st == 0, (n, st)
    return out.get(("burg prox", n)), info.get(("burg info", n))


def test_burg_simplex_prox_routes(acc, rt):
    """accbpg_burg_simplex_prox with y = NULL and with y at every route: checks (a)-(c) above, guards, inputs only read,
    the same bits on a repeat call and after a history that alternates the sizes from large to small and back (the
    token base and the parity of the slot table move with every call)."""
    L = 0.37
    sizes = burg_sizes(rt.sm_count)
    first = {}
    for n in sizes:
        grid, ept, _ = burg_route(n, rt.sm_count)
        g, y, _ = burg_inputs(n, rt.sm_count)
        g_d, y_d = dev(g), dev(y)
        for wy in (False, True):
            x, info = burg_prox_call(rt, g_d, y_d if wy else None, n, L)
            check_burg_result(x, info, burg_gg(g, y if wy else None, L), grid, (n, wy), (n, ept, grid, wy))
            first[(n, wy)] = (x, info)
            x2, info2 = burg_prox_call(rt, g_d, y_d if wy else None, n, L)
            assert same_bits(x2, x) and same_bits(info2, info), ("repeat call", n, wy)
        assert same_bits(g_d.cpu().numpy(), g) and same_bits(y_d.cpu().numpy(), y), ("inputs written", n)
    order = sorted(sizes)
    zigzag = [v for pair in zip(order[::-1], order) for v in pair][:len(order)]
    for n in zigzag + zigzag[::-1]:
        g, y, _ = burg_inputs(n, rt.sm_count)
        for wy in (True, False):
            x, info = burg_prox_call(rt, dev(g), dev(y) if wy else None, n, L)
            assert same_bits(x, first[(n, wy)][0]) and same_bits(info, first[(n, wy)][1]), ("after history", n, wy)
    # the Python operator the drivers call runs the same kernel
    h = acc.BurgEntropySimplex()
    for n in (sizes[2], sizes[-2]):
        g, y, _ = burg_inputs(n, rt.sm_count)
        assert same_bits(h.div_prox_map(y, g, L), first[(n, True)][0])
        assert same_bits(h.prox_map(g, L), first[(n, False)][0])


@pytest.mark.parametrize("world", [2, 4])
def test_burg_simplex_root_only_routes(acc, rt, world):
    """accbpg_burg_simplex_prepare -> _root -> _finish_dev, the column-sharded form on one GPU, at the EPT 3, 4, 6, 8
    and 0 sizes: every rank's slice of gg written into a +inf-padded gathered vector, the root-find on that vector
    (root-only entry, gg_in), then x = 1/(gg + c) per slice from the c left on the device."""
    L = 0.41
    S = BURG_THREADS * rt.sm_count
    seen = set()
    for n in (2 * S + 1, 3 * S + 1, 4 * S + 1, 6 * S + 1, 8 * S + 1):
        g, y, _ = burg_inputs(n, rt.sm_count)
        offs = acc.ColumnShard.partition(n, world)
        width = max(offs[r + 1] - offs[r] for r in range(world))
        total = world * width
        grid, ept, _ = burg_route(total, rt.sm_count)
        seen.add(ept)
        g_d, y_d = dev(g), dev(y)
        full = Out(total, fill=float("inf"))
        mins = Out(world)
        for r in range(world):
            lo, hi = offs[r], offs[r + 1]
            st = call(rt, "accbpg_burg_simplex_prepare", hi - lo, y_d[lo:].data_ptr(), g_d[lo:].data_ptr(), L,
                      full.ptr + 8 * r * width, mins.ptr + 8 * r)
            assert st == 0
        gg = burg_gg(g, y, L)
        gfull = np.full(total, np.inf)
        for r in range(world):
            gfull[r * width:r * width + offs[r + 1] - offs[r]] = gg[offs[r]:offs[r + 1]]
        assert same_bits(full.get("gathered gg"), gfull), (n, world, "prepared gg")
        assert same_bits(mins.get("prepare min"), [gg[offs[r]:offs[r + 1]].min() for r in range(world)])
        info = Out(3)
        assert call(rt, "accbpg_burg_simplex_root", total, full.ptr, BURG_EPS, info.ptr) == 0
        out = Out(n)
        for r in range(world):
            lo, hi = offs[r], offs[r + 1]
            assert call(rt, "accbpg_burg_simplex_finish_dev", hi - lo, full.ptr + 8 * r * width, info.ptr + 16,
                        out.ptr + 8 * lo) == 0
        inf_ = info.get("root info")
        assert same_bits(full.get("gathered gg after the root-find"), gfull), "root-only entry wrote its input"
        check_burg_result(out.get("finish"), inf_, gfull, grid, ("gathered", n, world), (n, world, ept, grid))
    assert seen == {3, 4, 6, 8, 0}, seen


# ------------------------------------------------------------------------------------------------------- route evidence
def _kernels_of(prof):
    """(name, grid) of every kernel in the profiler's trace, in launch order."""
    with tempfile.TemporaryDirectory(prefix="accbpg_trace_") as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            ev = json.load(f)["traceEvents"]
    ks = sorted((e for e in ev if e.get("cat") == "kernel"), key=lambda e: e["ts"])
    return [(e["name"], tuple(e["args"]["grid"])) for e in ks]


LINREG_LAYOUTS = [           # id, m, n, lda (None: n), A offset, x offset (doubles)
    ("1x1", 1, 1, None, 0, 0),                     # scalar path
    ("3x2", 3, 2, None, 0, 0),                     # vector path, rows clamped inside the one 4-row block
    ("4099x1024", 4099, 1024, None, 0, 0),         # A^T r in 65 chunks of 64 rows
    ("40001x300", 40001, 300, None, 0, 0),         # A^T r at the 256-chunk cap, 157 rows per chunk (unroll tail)
    ("50x65537", 50, 65537, None, 0, 0),           # odd lda: scalar path over two column segments (65536 + 1)
    ("50x65537 lda=65538", 50, 65537, 65538, 0, 0),   # vector path, odd tail column
    ("9x200001 lda=200002", 9, 200001, 200002, 0, 0),  # four column segments, one row chunk
    ("257x2050 A+1", 257, 2050, None, 1, 0),       # A base 8 but not 16-byte aligned: both products scalar
    ("257x2050 x+1", 257, 2050, None, 0, 1),       # x base likewise: A x scalar, A^T r stays on 16-byte loads
]


def linreg_routes(m, n, lda, a_off, x_off, sms):
    """(matvec VEC2, its grid), (rmatvec VEC2, its grid) as accbpg_linreg_matvec / _rmatvec choose them."""
    lda = lda or n
    nseg, nchunk, _ = linreg_plan(m, n, sms)
    vec_a = a_off % 2 == 0 and lda % 2 == 0
    return (vec_a and x_off % 2 == 0, (cdiv(m, 4), nseg, 1)), (vec_a, (cdiv(n, 512), nchunk, 1))


def test_route_evidence_in_the_trace(acc, rt):
    """One torch.profiler run: burg_simplex_x_kernel<EPT> ran with the expected EPT and grid at every Burg size (the
    leader exchange exactly where grid > 128), and the products took the expected template and grid per layout.  If
    occupancy ever allowed two root-find blocks per SM, the grids differ and this fails instead of covering less."""
    sms = rt.sm_count
    sizes = burg_sizes(sms)
    g_ds = {n: dev(burg_inputs(n, sms)[0]) for n in sizes}
    mats = []
    for _, m, n, lda, a_off, x_off in LINREG_LAYOUTS:
        mats.append((Mat(linreg_data(m, n)[0], lda, a_off), dev(np.ones(n), x_off), dev(np.ones(m))))
    torch.cuda.synchronize()
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for n in sizes:
            burg_prox_call(rt, g_ds[n], None, n, 0.37)
        for A, xd, rd in mats:
            A.matvec(rt, xd, Out(A.m))
            A.rmatvec(rt, rd, Out(A.n))
        torch.cuda.synchronize()
    ks = _kernels_of(prof)
    burg = [(int(m.group(1) or m.group(2)), gr) for k, gr in ks      # demangled or mangled names
            for m in [re.search(r"burg_simplex_x_kernel(?:<(\d+)>|ILi(\d+)E)", k)] if m]
    want = [(burg_route(n, sms)[1], (burg_route(n, sms)[0], 1, 1)) for n in sizes]
    assert burg == want, (burg, want)
    assert {e for e, _ in burg} == {0, 1, 2, 3, 4, 6, 8}
    assert any(gr[0] > 128 and e == 1 for e, gr in burg), "the leader exchange with EPT 1 did not run"
    prods = [(m.group(1), m.group(2) == "true" or m.group(3) == "1", gr) for k, gr in ks
             for m in [re.search(r"(r?matvec)_kernel(?:<(true|false)>|ILb([01])E)", k)] if m]
    want = []
    for _, m, n, lda, a_off, x_off in LINREG_LAYOUTS:
        (vm, gm), (vr, gr) = linreg_routes(m, n, lda, a_off, x_off, sms)
        want += [("matvec", vm, gm), ("rmatvec", vr, gr)]
    assert prods == want, (prods, want)
    segs = [gr for k, gr in ks if "seg_reduce_kernel" in k]
    assert len(segs) == sum(1 for _, m, n, *_ in LINREG_LAYOUTS if n > 65536) + len(LINREG_LAYOUTS)


# ------------------------------------------------------------------------------------------------------- 2. vectors
RED_N = [1, 1024, 1025, 606208, 606209, 1000003]


def _red(rt, name, n, *args):
    o = Out(1)
    assert call(rt, name, n, *[a.data_ptr() if isinstance(a, torch.Tensor) else a for a in args], o.ptr) == 0, name
    return float(o.get(name)[0])


def _close(val, ref, bar, what):
    assert abs(val - float(ref)) <= bar, (what, val, float(ref), abs(val - float(ref)), bar)


def _signed(rng, n, lo=0.5, hi=2.0):
    return rng.choice([-1.0, 1.0], n) * rng.uniform(lo, hi, n)


@pytest.mark.parametrize("n", RED_N)
def test_reductions_vs_extended_reference(rt, n):
    """Sums of products (k = 2) and of log terms (k = 4) against np.longdouble; every |t_i| >= 1e-3 of the mean (apart
    from the exact zeros that exercise the delta clamp), so one dropped or doubled element is far past the bar.  For a
    term made of several parts, sum|t_i| adds up the magnitudes of its parts."""
    rng = np.random.RandomState(n % 9973 + 17)
    G = red_grid(rt.sm_count, n)
    W = 256 * G
    a, b, g = _signed(rng, n), _signed(rng, n), _signed(rng, n)
    pa, nb = rng.uniform(0.5, 2.0, n), -rng.uniform(0.5, 2.0, n)
    ad, bd, gd, pad, nbd = (dev(v) for v in (a, b, g, pa, nb))
    al, bl, gl, pal, nbl = (v.astype(LD) for v in (a, b, g, pa, nb))

    t = al * bl
    _close(_red(rt, "accbpg_vec_dot", n, ad, bd), np.sum(t), tree(n, W, 2) * float(np.sum(abs(t))), "dot")
    t = gl * (pal - nbl)
    _close(_red(rt, "accbpg_vec_dot_diff", n, gd, pad, nbd), np.sum(t), tree(n, W, 2) * float(np.sum(abs(t))),
           "dot_diff")
    t = (pal - nbl) ** 2
    _close(_red(rt, "accbpg_vec_sqdist", n, pad, nbd), np.sum(t), tree(n, W, 2) * float(np.sum(t)), "sqdist")
    _close(_red(rt, "accbpg_vec_sum", n, ad), np.sum(al), tree(n, W, 2) * float(np.sum(abs(al))), "sum")

    # Burg: x = e^(+-[0.5, 5]), so |log x| >= 0.5; x/y = e^(+-[1, 6])
    xb = np.exp(rng.choice([-1.0, 1.0], n) * rng.uniform(0.5, 5.0, n))
    yb = xb * np.exp(-rng.choice([-1.0, 1.0], n) * rng.uniform(1.0, 6.0, n))
    xbd, ybd = dev(xb), dev(yb)
    t = -np.log(xb.astype(LD))
    _close(_red(rt, "accbpg_burg_value", n, xbd), np.sum(t), tree(n, W, 4) * float(np.sum(abs(t))), "burg value")
    r = xb.astype(LD) / yb.astype(LD)
    t = (r - np.log(r)) - 1
    _close(_red(rt, "accbpg_burg_divergence", n, xbd, ybd), np.sum(t),
           tree(n, W, 4) * float(np.sum(r + abs(np.log(r)) + 1)), "burg divergence")

    # Shannon: x log x with x in [1.5, 4] and exact zeros (the delta clamp); x log((x+d)/(y+d)) with x/y = e^(+-[0.5, 2])
    xs = rng.uniform(1.5, 4.0, n)
    xs[rng.rand(n) < 0.05] = 0.0
    xsl = np.maximum(xs, DELTA).astype(LD)
    t = xsl * np.log(xsl)
    _close(_red(rt, "accbpg_shannon_value", n, dev(xs), DELTA), np.sum(t), tree(n, W, 4) * float(np.sum(abs(t))),
           "shannon value")
    x2 = rng.uniform(0.5, 2.0, n)
    y2 = x2 * np.exp(rng.choice([-1.0, 1.0], n) * rng.uniform(0.5, 2.0, n))
    x2[rng.rand(n) < 0.05] = 0.0
    y2[rng.rand(n) < 0.05] = 0.0
    x2l, y2l = x2.astype(LD), y2.astype(LD)
    t0 = x2l * np.log((x2l + LD(DELTA)) / (y2l + LD(DELTA)))
    T0, T1, T2 = np.sum(t0), np.sum(y2l), np.sum(x2l)
    bar = tree(n, W, 4) * float(np.sum(abs(t0))) + tree(n, W, 2) * float(T1 + T2) \
        + 2 * EPS * SLACK * float(abs(T0) + T1 + T2)
    _close(_red(rt, "accbpg_shannon_divergence", n, dev(x2), dev(y2), DELTA), T0 + (T1 - T2), bar, "shannon div")

    # Shannon simplex: the un-normalised point and its sum (normalize = 2), then the normalisation given that sum
    ysp = rng.uniform(0.1, 1.0, n)
    gsp = rng.randn(n)
    ysd, gsd = dev(ysp), dev(gsp)
    for lam, yd in ((0.0, ysd), (0.3, ysd), (0.0, None)):
        yp = None if yd is None else yd.data_ptr()
        v, s = Out(n), Out(1)
        assert call(rt, "accbpg_shannon_prox", n, lam, yp, gsd.data_ptr(), 0.7, 2, v.ptr, s.ptr) == 0
        v, s = v.get("shannon prox sum: point"), float(s.get("shannon prox sum")[0])
        check_shannon_point(v, ysp if yd is not None else None, gsp, lam, 0.7, ("simplex sum point", lam))
        _close(s, np.sum(v.astype(LD)), tree(n, W, 2) * float(np.sum(v.astype(LD))), ("simplex sum", lam))
        x, s1 = Out(n), Out(1)
        assert call(rt, "accbpg_shannon_prox", n, lam, yp, gsd.data_ptr(), 0.7, 1, x.ptr, s1.ptr) == 0
        assert float(s1.get()[0]) == s
        assert same_bits(x.get("shannon normalised"), v / s), ("normalisation", lam)


def check_shannon_point(v, y, g, lam, L, what):
    """y exp(-(lam + g)/L) or exp(-(lam + g)/L - 1) to <= 2 ulp: the argument rounds as the kernel rounds it, the
    exponential and the product are taken in long double."""
    gi = g if lam == 0.0 else lam + g
    if y is None:
        ref = np.exp((-gi / L - 1.0).astype(LD)).astype(np.float64)
    else:
        ref = (y.astype(LD) * np.exp((-gi / L).astype(LD))).astype(np.float64)
    d = ulp_diff(v, ref)
    assert np.all(np.isfinite(v)) and int(d.max(initial=0)) <= ULPS, (what, int(d.max(initial=0)))


def _map(rt, name, n, *args):
    o = Out(n)
    assert call(rt, name, n, *[a.data_ptr() if isinstance(a, torch.Tensor) else a for a in args], o.ptr) == 0, name
    return o.get(name)


@pytest.mark.parametrize("n", RED_N)
def test_maps_vs_numpy_restatement(rt, n):
    """Element-wise kernels against NumPy stating the same expression in the same order: bit for bit, except the maps
    through exp or log (<= 2 ulp against long double)."""
    rng = np.random.RandomState(n % 7919 + 3)
    x, s, g = rng.randn(n), rng.randn(n), rng.randn(n)
    gp = rng.uniform(0.5, 2.0, n)
    y = rng.uniform(0.05, 1.0, n)
    xd, sd, gd, gpd, yd = (dev(v) for v in (x, s, g, gp, y))
    assert same_bits(_map(rt, "accbpg_vec_axpby", n, 0.3, xd, -1.7, sd), 0.3 * x + -1.7 * s)
    assert same_bits(_map(rt, "accbpg_vec_step_toward", n, xd, sd, 0.37), x + 0.37 * (s - x))
    assert same_bits(_map(rt, "accbpg_vec_divide", n, xd, 3.1), x / 3.1)
    assert same_bits(_map(rt, "accbpg_burg_gradient", n, gpd), -1.0 / gp)

    # Burg prox: plain, L1, L2 (four_lamL / two_lamL formed as the host forms them), without and with y
    L, lam = 0.7, 0.3
    lamL = lam / L
    for kind, gv, gvd in ((0, gp, gpd), (1, gp, gpd), (2, g, gd)):
        for yy, yyd in ((None, None), (y, yd)):
            sh = gv if yy is None else gv - L * (-1.0 / yy)
            if kind == 0:
                ref = L / sh
            elif kind == 1:
                ref = L / (lam + sh)
            else:
                gg = sh / L
                ref = (np.sqrt(gg * gg + 4 * lamL) - gg) / (2 * lamL)
            got = _map(rt, "accbpg_burg_prox", n, kind, lam, None if yyd is None else yyd.data_ptr(), gvd, L)
            assert same_bits(got, ref), ("burg prox", kind, yy is None)

    # Shannon gradient 1 + log(max(x, delta)): x in [2, 7.3], [e^-3.9, e^-3] and exact zeros, away from 1/e where the
    # sum cancels
    xs = np.where(rng.rand(n) < 0.5, rng.uniform(2.0, 7.3, n), np.exp(rng.uniform(-3.9, -3.0, n)))
    xs[rng.rand(n) < 0.05] = 0.0
    got = _map(rt, "accbpg_shannon_gradient", n, dev(xs), DELTA)
    ref = (1 + np.log(np.maximum(xs, DELTA).astype(LD))).astype(np.float64)
    assert int(ulp_diff(got, ref).max()) <= ULPS
    for lamv in (0.0, 0.3):
        for yy, yyd in ((None, None), (y, yd)):
            o = Out(n)
            assert call(rt, "accbpg_shannon_prox", n, lamv, None if yyd is None else yyd.data_ptr(), gd.data_ptr(), L, 0,
                        o.ptr, None) == 0
            check_shannon_point(o.get("shannon prox"), yy, g, lamv, L, ("shannon prox", lamv, yy is None))

    # LMOs: sign(g) with exact zeros, the l2 step, the box, a vertex at 0, n - 1, the middle and none (-1)
    gz = g.copy()
    gz[rng.rand(n) < 0.1] = 0.0
    gzd = dev(gz)
    for c, cd in ((None, None), (x, xd)):
        cc = 0.0 if c is None else c
        assert same_bits(_map(rt, "accbpg_lmo_linf", n, gzd, 0.5, None if cd is None else cd.data_ptr()),
                         cc - 0.5 * np.sign(gz))
        gnorm = float(np.sqrt(np.dot(g, g)))
        assert same_bits(_map(rt, "accbpg_lmo_l2", n, gd, 1.5, gnorm, None if cd is None else cd.data_ptr()),
                         cc - 1.5 * g / gnorm)
    assert same_bits(_map(rt, "accbpg_lmo_box", n, gzd, sd, yd), np.where(gz < 0.0, y, s))
    for idx in sorted({0, n - 1, n // 2, -1}):
        ref = np.full(n, 1e-15)
        if idx >= 0:
            ref[idx] = 2.5
        assert same_bits(_map(rt, "accbpg_lmo_fill_vertex", n, 1e-15, idx, 2.5), ref), idx


ARG_N = [1, 1024, 1025, 300001, 606208, 606209, 1000003]


def _arg_vectors(n, G):
    """(label, x): a tie between j < k with j in the last block's first grid-stride pass and k in block 0's second
    (two blocks and more), the extremum at n - 1, all equal, +-inf entries, all +inf, all -inf."""
    rng = np.random.RandomState(n % 4099 + 1)
    out = []
    x = rng.randn(n)
    if n >= 4:
        stride = 256 * G
        j, k = (G - 1) * 256 + 3, stride + 5
        if k + 1 >= n:                               # one block and one pass: a tie inside the block
            j, k = 1, n - 2
        x[[j, k]] = x.min() - 1.0
        x[[j + 1, k + 1]] = x.max() + 1.0
    out.append(("ties", x))
    for sgn in (-1.0, 1.0):
        x = rng.randn(n)
        x[n - 1] = sgn * 10.0
        out.append((f"extremum at n-1 ({sgn:+.0f})", x))
    out.append(("all equal", np.full(n, 0.25)))
    x = rng.randn(n)
    x[rng.choice(n, size=min(n, 6), replace=False)[:3]] = np.inf
    x[rng.choice(n, size=min(n, 6), replace=False)[3:]] = -np.inf
    out.append(("+-inf entries", x))
    out.append(("all +inf", np.full(n, np.inf)))
    out.append(("all -inf", np.full(n, -np.inf)))
    return out


@pytest.mark.parametrize("n", ARG_N)
def test_arg_extrema_and_simplex_lmo(rt, n):
    """vec_argext (argmin and argmax), vec_minmax and lmo_simplex equal np.argmin / np.argmax / np.min / np.max on
    every input of _arg_vectors, all-infinite ones included; the LMO's vertex vector bit for bit."""
    G = red_grid(rt.sm_count, n)
    for label, x in _arg_vectors(n, G):
        xd = dev(x)
        for want_max, arg, ext in ((0, np.argmin, np.min), (1, np.argmax, np.max)):
            o = Out(2)
            assert call(rt, "accbpg_vec_argext", n, xd.data_ptr(), want_max, o.ptr) == 0
            v = o.get(("argext", label))
            assert v[0] == ext(x) and int(v[1]) == int(arg(x)), (label, want_max, v, ext(x), int(arg(x)))
        o = Out(2)
        assert call(rt, "accbpg_vec_minmax", n, xd.data_ptr(), o.ptr) == 0
        assert list(o.get(("minmax", label))) == [x.min(), x.max()], label
        sv, o = Out(n), Out(2)
        assert call(rt, "accbpg_lmo_simplex", n, xd.data_ptr(), 2.0, sv.ptr, o.ptr) == 0
        v = o.get(("lmo", label))
        i = int(np.argmin(x))
        ref = np.full(n, 1e-15)
        ref[i] = 2.0
        assert v[0] == x.min() and int(v[1]) == i, (label, v, i)
        assert same_bits(sv.get(("lmo vertex", label)), ref), label
        assert same_bits(xd.cpu().numpy(), x)


@pytest.mark.parametrize("n", [1, 1025, 606209])
def test_simplex_lmo_on_an_all_infinite_gradient(acc, n):
    """np.argmin of an all-+inf vector is 0, so the reference's lmo_simplex puts the vertex at 0; so must the LMO, the
    matrix LMO and the arg-extremum the Kumar-Yildirim initialisation takes (argmax of an all--inf vector)."""
    from oracle import accbpg_oracle as orc
    g = np.full(n, np.inf)
    lmo = acc.lmo_simplex(2.0)
    s = lmo(g)
    assert lmo.last_index() == 0
    assert same_bits(s, orc.lmo_simplex_eval(g, 2.0))
    if n % 5 == 0:
        S = acc.lmo_matrix_simplex(3.0)(g.reshape(5, n // 5))
        assert S[0, 0] == 3.0 and np.sum(S == 3.0) == 1
    rt = acc.Runtime.get()
    o = Out(2)
    assert call(rt, "accbpg_vec_argext", n, dev(-g).data_ptr(), 1, o.ptr) == 0
    assert list(o.get()) == [-np.inf, 0.0]


# ------------------------------------------------------------------------------------------------------- 3. products
class Mat:
    """A as an m x n window of a device buffer: leading dimension lda, base offset `off` doubles; the padding columns
    and the space around hold NaN, so a read outside the matrix shows."""

    def __init__(self, A, lda=None, off=0, base=None):
        self.m, self.n = A.shape
        self.lda = lda or self.n
        if base is None:
            self.buf = torch.full((off + self.m * self.lda + GUARD,), float("nan"), dtype=F64, device="cuda")
            self.buf[off:off + self.m * self.lda].view(self.m, self.lda)[:, :self.n] = torch.from_numpy(A).cuda()
            self.ptr = self.buf.data_ptr() + 8 * off
        else:
            self.buf, self.ptr = base               # a window of someone else's buffer
        self.ws = torch.full((_lib().lib.accbpg_linreg_workspace_bytes(self.m, self.n),), 255, dtype=torch.uint8,
                             device="cuda")          # NaN everywhere: a partial read before it is written shows

    def matvec(self, rt, xd, out):
        return call(rt, "accbpg_linreg_matvec", self.ptr, self.m, self.n, self.lda, xd.data_ptr(), self.ws.data_ptr(),
                    out.ptr)

    def rmatvec(self, rt, rd, out):
        return call(rt, "accbpg_linreg_rmatvec", self.ptr, self.m, self.n, self.lda, rd.data_ptr(), self.ws.data_ptr(),
                    out.ptr)


_LIN = {}


def linreg_data(m, n):
    """Signed Gaussian A, x, r of shape (m, n) and their long-double products with sum|A_ij x_j| (rows) and
    sum|A_ij r_i| (columns)."""
    if (m, n) not in _LIN:
        rng = np.random.RandomState(m * 7 + n)
        A, x, r = rng.randn(m, n), rng.randn(n), rng.randn(m)
        Al, xl, rl = A.astype(LD), x.astype(LD), r.astype(LD)
        aA = np.abs(Al)
        _LIN[(m, n)] = (A, x, r, Al @ xl, aA @ np.abs(xl), rl @ Al, np.abs(rl) @ aA)
    return _LIN[(m, n)]


def check_products(Ax, g, m, n, sms, what, ref=None):
    A, x, r, Ax_l, sx, g_l, sr = ref or linreg_data(m, n)
    _, nchunk, rpc = linreg_plan(m, n, sms)
    bar_r = (cdiv(n, 256) + 24) * EPS * SLACK * sx
    err = np.abs(Ax.astype(LD) - Ax_l)
    assert np.all(err <= bar_r), (what, "A x", int(np.argmax(err - bar_r)), float(np.max(err / sx)))
    # a column's sum: rows_per_chunk sequential adds in its chunk, then the nchunk partials in chunk order
    bar_c = (rpc + nchunk + 2) * EPS * SLACK * sr
    err = np.abs(g.astype(LD) - g_l)
    assert np.all(err <= bar_c), (what, "A^T r", int(np.argmax(err - bar_c)), float(np.max(err / sr)))


@pytest.mark.parametrize("layout", LINREG_LAYOUTS, ids=[v[0] for v in LINREG_LAYOUTS])
def test_linreg_products_vs_extended_reference(rt, layout):
    """accbpg_linreg_matvec / _rmatvec on every layout of LINREG_LAYOUTS against the long-double products, per row
    and per column; guards, NaN padding, bit-identical repeat calls."""
    name, m, n, lda, a_off, x_off = layout
    A, x, r = linreg_data(m, n)[:3]
    M = Mat(A, lda, a_off)
    xd, rd = dev(x, x_off), dev(r)
    ax, gg = Out(m), Out(n)
    assert M.matvec(rt, xd, ax) == 0 and M.rmatvec(rt, rd, gg) == 0
    Ax, g = ax.get((name, "A x")), gg.get((name, "A^T r"))
    check_products(Ax, g, m, n, rt.sm_count, name)
    ax2, gg2 = Out(m), Out(n)
    assert M.matvec(rt, xd, ax2) == 0 and M.rmatvec(rt, rd, gg2) == 0
    assert same_bits(ax2.get(), Ax) and same_bits(gg2.get(), g), (name, "repeat")
    if rt.sm_count == 148:                       # the plans the layouts were chosen for
        plan = {"4099x1024": (1, 65, 64), "40001x300": (1, 256, 157), "50x65537": (2, 1, 50),
                "9x200001 lda=200002": (4, 1, 9)}.get(name)
        assert plan is None or linreg_plan(m, n, 148) == plan


def test_linreg_column_slices_add_up(rt):
    """A_full[:, lo:hi] windows with lda = n_full (even) and odd lo (8-byte aligned bases: scalar path) next to even
    lo (16-byte loads): the slices' partial A x, summed on the host, and their A^T r, side by side, match the
    long-double products of the full matrix; the full matrix itself too."""
    m, nf = 300, 4100
    A, x, r, Ax_l, sx, g_l, sr = linreg_data(m, nf)
    full = Mat(A)
    xd, rd = dev(x), dev(r)
    bounds = [0, 1, 1237, 3001, 3002, 4100]
    parts, gs, bar = [], [], np.zeros(m, dtype=LD)
    for lo, hi in zip(bounds[:-1], bounds[1:]):
        n = hi - lo
        M = Mat(A[:, lo:hi], lda=nf, base=(full.buf, full.ptr + 8 * lo))
        ax, gg = Out(m), Out(n)
        assert M.matvec(rt, dev(x[lo:hi]), ax) == 0 and M.rmatvec(rt, rd, gg) == 0
        parts.append(ax.get(("slice", lo)).astype(LD))
        gs.append(gg.get(("slice", lo)))
        Al = A[:, lo:hi].astype(LD)
        bar += (cdiv(n, 256) + 24) * EPS * SLACK * (np.abs(Al) @ np.abs(x[lo:hi].astype(LD)))
        _, nchunk, rpc = linreg_plan(m, n, rt.sm_count)
        err = np.abs(gs[-1].astype(LD) - g_l[lo:hi])
        assert np.all(err <= (rpc + nchunk + 2) * EPS * SLACK * sr[lo:hi]), ("slice A^T r", lo, hi)
    assert np.all(np.abs(np.sum(parts, axis=0) - Ax_l) <= bar), "slices of A x do not add up"
    ax, gg = Out(m), Out(nf)
    assert full.matvec(rt, xd, ax) == 0 and full.rmatvec(rt, rd, gg) == 0
    check_products(ax.get(), gg.get(), m, nf, rt.sm_count, "full")


def _ab(m, seed):
    rng = np.random.RandomState(seed)
    a = rng.uniform(0.5, 2.0, m)
    return a, a * np.exp(rng.uniform(-1.0, 1.0, m))


@pytest.mark.parametrize("kind", ["poisson", "kl"])
@pytest.mark.parametrize("m", [1, 1025, 700001])
def test_linreg_value_resid(acc, rt, kind, m):
    """accbpg_linreg_value_resid with r and with r = NULL (f the same bits, nothing written past f): f against long
    double with the tree bar over the value's parts, r to <= 2 ulp (Poisson's 1 - b/a bit for bit)."""
    K = _lib().MACROS["ACCBPG_LINREG_POISSON" if kind == "poisson" else "ACCBPG_LINREG_KL"]
    a, b = _ab(m, m + len(kind))
    ad, bd = dev(a), dev(b)
    al, bl = a.astype(LD), b.astype(LD)
    if kind == "poisson":
        q = bl / al
        t, scale = (bl * np.log(q) + al) - bl, np.abs(bl * np.log(q)) + al + bl
    else:
        lg = np.log(al / bl)
        t, scale = (al * lg - al) + bl, np.abs(al * lg) + al + bl
    G = red_grid(rt.sm_count, m)
    f, rr = Out(1), Out(m)
    assert call(rt, "accbpg_linreg_value_resid", K, m, ad.data_ptr(), bd.data_ptr(), f.ptr, rr.ptr) == 0
    fv, r = float(f.get()[0]), rr.get((kind, "r"))
    _close(fv, np.sum(t), tree(m, 256 * G, 4) * float(np.sum(scale)), (kind, m, "f"))
    if kind == "poisson":
        assert same_bits(r, 1.0 - b / a)
    else:
        ref = np.log((a / b).astype(LD)).astype(np.float64)
        assert int(ulp_diff(r, ref).max()) <= ULPS
    f2 = Out(1)
    assert call(rt, "accbpg_linreg_value_resid", K, m, ad.data_ptr(), bd.data_ptr(), f2.ptr, None) == 0
    assert float(f2.get()[0]) == fv


@pytest.mark.parametrize("kind", ["poisson", "kl"])
@pytest.mark.parametrize("m,n", [(4099, 1024), (50, 65537)])
def test_linreg_func_grad_tight(acc, kind, m, n):
    """PoissonRegression / KLdivRegression.func_grad: the project bar (1e-10) against the FP64 oracle and a tight bar
    against long double: the product bars carried through f and r to first order, plus the value's own tree bar."""
    from oracle import accbpg_oracle as orc
    rt = acc.Runtime.get()
    rng = np.random.RandomState(3 * m + n)
    A = rng.rand(m, n)
    A /= A.sum(axis=0)
    xs = rng.rand(n) + 0.05
    b = A @ xs * (1 + 0.1 * (rng.rand(m) - 0.5))
    x = rng.rand(n) + 0.05
    f = (acc.PoissonRegression if kind == "poisson" else acc.KLdivRegression)(A, b)
    fo = (orc.make_poisson if kind == "poisson" else orc.make_kl)(A, b)
    fx, g = f.func_grad(x)
    fxo, go = fo.func_grad(x)
    assert abs(fx - fxo) <= 1e-10 * max(abs(fxo), 1e-3), (fx, fxo)
    assert np.max(np.abs(g - go)) <= 1e-10 * np.max(np.abs(go))
    Al, xl, bl = A.astype(LD), x.astype(LD), b.astype(LD)
    a = Al @ xl                                       # A >= 0, x > 0: sum|A_ij x_j| = (A x)_i
    da = (cdiv(n, 256) + 24) * EPS * SLACK * a
    if kind == "poisson":
        q = bl / a
        fl, r = np.sum((bl * np.log(q) + a) - bl), 1 - q
        scale = np.abs(bl * np.log(q)) + a + bl
        dr = q / a * da + 2 * EPS * (q + np.abs(r))   # d(1 - b/a)/da = b/a^2; b/a and 1 - q rounded
    else:
        lg = np.log(a / bl)
        fl, r = np.sum((a * lg - a) + bl), lg
        scale = np.abs(a * lg) + a + bl
        dr = da / a + 2 * EPS * (1 + np.abs(r))       # d log(a/b)/da = 1/a; a/b rounded, log within 1 ulp
    bar_f = float(np.sum(np.abs(r) * da)) + tree(m, 256 * red_grid(rt.sm_count, m), 4) * float(np.sum(scale))
    assert abs(fx - float(fl)) <= bar_f, (kind, fx, float(fl), bar_f)
    gl = r @ Al
    _, nchunk, rpc = linreg_plan(m, n, rt.sm_count)
    bar_g = dr @ Al + (rpc + nchunk + 2) * EPS * SLACK * (np.abs(r) @ Al)
    assert np.all(np.abs(g.astype(LD) - gl) <= bar_g), (kind, float(np.max(np.abs(g - gl) / bar_g)))
