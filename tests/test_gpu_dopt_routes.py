"""D-optimal oracle (f(x) = -log det(H diag(x) H^T), g_j = -h_j^T M^{-1} h_j) through the C ABI, route by route, against
an extended-precision reference.

The host code of accbpg_dopt_func_grad / _pair / _pair_from_gram chooses between the per-step and the data-flow Cholesky
chain, with or without the gated triangular GEMM started under the chain, TMA or cp.async mainloops, and a number of
early row blocks, held-back panels and SM reserves that depend on m and n.  The shapes below run every one of those
branches.  Each numerical check asserts two bars: the project's (f 1e-10 relative, g 1e-9 relative per entry) and,
where the extended reference exists, a conditioning-aware 64 m kappa_2(M) 2^-53 (relative to max|g| for g).  Inputs are
built so that the two silent failure modes of a scheduled kernel show up: stale state (successive calls with very
different x, including x and 1000 x) and dropped edge work (x concentrated on the ragged last columns, H's last row -
the padding edge of the 128-row tiles - scaled up).
"""
import os
import subprocess
import sys

import numpy as np
import pytest
import scipy.linalg
import scipy.sparse as sp
import torch

from conftest import relerr

pytestmark = pytest.mark.gpu

F64 = torch.float64
GUARD = 8                    # guard entries after every output buffer
SENTINEL = 7.25e17           # what the guards hold; no result of these tests can equal it
EPS = 2.0 ** -53
EXTENDED = np.finfo(np.longdouble).nmant >= 63
SLOT_X, SLOT_Y = 50, 51      # result slots of the context used here (the operator methods use 32..)
NOT_PD = 0x002               # ACCBPG_ST_NOT_PD


@pytest.fixture(scope="module")
def acc():
    import accbpg_and_fw_b200 as a
    return a


# ------------------------------------------------------------------------------------------------------- reference
def _chol(M):
    """Column-by-column Cholesky of a symmetric positive definite M (any float dtype), written out in NumPy."""
    m = M.shape[0]
    L = np.zeros_like(M)
    for j in range(m):
        d = M[j, j] - L[j, :j] @ L[j, :j]
        assert d > 0, "reference: M is not positive definite"
        L[j, j] = np.sqrt(d)
        if j + 1 < m:
            L[j + 1:, j] = (M[j + 1:, j] - L[j + 1:, :j] @ L[j, :j]) / L[j, j]
    return L


class Ref:
    """f, g, kappa_2(M) and whether they were computed in extended precision."""

    def __init__(self, m, f, g, kappa, extended):
        self.m, self.f, self.g, self.kappa, self.extended = m, f, g, kappa, extended


_REF = {}


def ref_dopt(H, x, key=None):
    """Reference f(x) = -log det(H diag(x) H^T) and g_j = -||L^{-1} h_j||^2.

    m <= 300 and n <= 10^4: in np.longdouble (64-bit mantissa): M = (H x) H^T, the Cholesky factor written out above,
    L^{-1} H by forward substitution over all columns at once.  Larger shapes, or a platform without an extended long
    double: FP64 LAPACK with one step of iterative refinement of M^{-1} H (then only the project bars apply).
    `key` caches the result for inputs that several tests share."""
    if key is not None and key in _REF:
        return _REF[key]
    m, n = H.shape
    x = np.asarray(x, dtype=np.float64)
    if m <= 300 and n <= 10000 and EXTENDED:
        Hl = H.astype(np.longdouble)
        M = (Hl * x.astype(np.longdouble)) @ Hl.T
        L = _chol(M)
        f = -2.0 * np.sum(np.log(np.diag(L)))
        Y = np.empty_like(Hl)
        for i in range(m):
            Y[i] = (Hl[i] - L[i, :i] @ Y[:i]) / L[i, i]
        r = Ref(m, float(f), np.asarray(-np.sum(Y * Y, axis=0), dtype=np.float64),
                float(np.linalg.cond(np.asarray(M, dtype=np.float64))), True)
    else:
        M = (H * x) @ H.T
        cf = scipy.linalg.cho_factor(M, lower=True)
        Z = scipy.linalg.cho_solve(cf, H)
        Z += scipy.linalg.cho_solve(cf, H - M @ Z)
        r = Ref(m, -2.0 * float(np.sum(np.log(np.diag(cf[0])))), -np.sum(H * Z, axis=0), float("nan"), False)
    if key is not None:
        _REF[key] = r
    return r


def check_f(f, ref, what=""):
    assert np.isfinite(f), (what, f)
    assert abs(f - ref.f) <= 1e-10 * max(1.0, abs(ref.f)), (what, f, ref.f)
    if ref.extended:
        assert abs(f - ref.f) <= 64 * ref.m * ref.kappa * EPS * max(1.0, abs(ref.f)), (what, f, ref.f, ref.kappa)


def check_g(g, ref, what=""):
    g = np.asarray(g)
    assert g.shape == ref.g.shape and np.all(np.isfinite(g)), what
    err = relerr(g, ref.g)
    assert err <= 1e-9, (what, err)
    if ref.extended:
        dev, tight = float(np.max(np.abs(g - ref.g))), 64 * ref.m * ref.kappa * EPS * float(np.max(np.abs(ref.g)))
        assert dev <= tight, (what, dev, tight, ref.kappa)


# ------------------------------------------------------------------------------------------------------- inputs
def make_H(m, n, seed):
    """Gaussian H whose last row (the padding edge of the last 128-row tile) carries 8x the scale."""
    H = np.random.RandomState(seed).randn(m, n)
    H[m - 1] *= 8.0
    return H


def draw_x(n, kind, seed):
    """(a) uniform; (b) most of the weight on the ragged edge: the last n mod 16 and n mod 128 columns (the last 16 when
    n is a multiple of 128); (c) a dynamic range of 1e-12 .. 1 with exact zeros (half the columns keep O(1) weight, so
    M stays well conditioned)."""
    rng = np.random.RandomState(seed)
    if kind == "a":
        return rng.rand(n) + 0.05
    if kind == "b":
        x = 1e-3 * (rng.rand(n) + 0.5)
        edge = max(n % 16, n % 128) or 16
        x[n - edge:] = 1.0 + rng.rand(edge)
        return x
    x = 10.0 ** rng.uniform(-12.0, 0.0, n)
    sel = rng.rand(n)
    x[sel < 0.15] = 0.0
    x[sel > 0.5] = 0.5 + 0.5 * rng.rand(int(np.sum(sel > 0.5)))
    return x


_PROBLEMS = {}


def problem(m, n):
    """The shared instance of shape (m, n): H and the three draws of x (with cached references)."""
    if (m, n) not in _PROBLEMS:
        seed = 1000 * m + n % 1000
        _PROBLEMS[(m, n)] = (make_H(m, n, seed), {k: draw_x(n, k, seed + i) for i, k in enumerate("abc")})
    return _PROBLEMS[(m, n)]


def problem_ref(m, n, kind, scale=1.0):
    H, xs = problem(m, n)
    return ref_dopt(H, scale * xs[kind], key=(m, n, kind, scale))


# ------------------------------------------------------------------------------------------------------- C ABI harness
class Op:
    """One D-optimal operator driven through the C ABI: H (optionally a window of a wider device buffer: leading
    dimension ldh, base offset h_off doubles; the padding holds NaN, so a read outside the matrix shows), its own
    zero-filled workspace, output buffers with guards, result slots preset to NaN before every call."""

    def __init__(self, acc, H, ldh=None, h_off=0, x_off=0):
        from accbpg_and_fw_b200 import _native
        self.nat, self.lib = _native, _native.lib
        self.rt = acc.Runtime.get()
        self.m, self.n = H.shape
        self.ldh = ldh or self.n
        self.x_off = x_off
        self.Hbuf = torch.full((h_off + self.m * self.ldh,), float("nan"), dtype=F64, device="cuda")
        win = self.Hbuf[h_off:].view(self.m, self.ldh)
        win[:, :self.n] = torch.from_numpy(H).cuda()
        self.Hp = win.data_ptr()
        self.ws = torch.zeros(self.lib.accbpg_dopt_workspace_bytes(self.m, self.n), dtype=torch.uint8, device="cuda")
        self.g = torch.empty(self.n + GUARD, dtype=F64, device="cuda")

    # ---- plumbing
    def xdev(self, x):
        """x on the device at offset x_off doubles of its buffer (NaN around it); returns the view."""
        buf = torch.full((self.x_off + self.n + GUARD,), float("nan"), dtype=F64, device="cuda")
        buf[self.x_off:self.x_off + self.n] = torch.from_numpy(np.asarray(x, dtype=np.float64)).cuda()
        return buf[self.x_off:self.x_off + self.n]

    def mbuf(self):
        return torch.full((self.m * self.m + GUARD,), SENTINEL, dtype=F64, device="cuda")

    def _pre(self):
        self.rt.scal[SLOT_X:SLOT_Y + 1].fill_(float("nan"))
        self.g[:self.n].fill_(float("nan"))
        self.g[self.n:].fill_(SENTINEL)

    def _post(self, with_g):
        vals, st = self.rt.read_raw(SLOT_X, 2)
        gh = self.g.cpu().numpy()
        assert np.all(gh[self.n:] == SENTINEL), "gradient written past n"
        if not with_g:
            assert np.all(np.isnan(gh[:self.n])), "value-only call wrote the gradient buffer"
        return vals[0], vals[1], (gh[:self.n].copy() if with_g else None), st

    # ---- entry points
    def gram(self, x):
        xd = self.xdev(x)
        M = self.mbuf()
        self.nat.check(self.lib.accbpg_dopt_gram(self.rt.ctx, self.rt.stream, self.Hp, self.m, self.n, self.ldh,
                                                 xd.data_ptr(), self.ws.data_ptr(), M.data_ptr()))
        _, st = self.rt.read_raw(SLOT_X, 0)
        assert st == 0 and torch.all(M[self.m * self.m:] == SENTINEL), "Gram matrix written past m*m"
        return M

    def func_grad(self, x, flag):
        xd = self.xdev(x)
        self._pre()
        self.nat.check(self.lib.accbpg_dopt_func_grad(self.rt.ctx, self.rt.stream, self.Hp, self.m, self.n, self.ldh,
                                                      xd.data_ptr(), flag, self.ws.data_ptr(), self.rt.slot(SLOT_Y),
                                                      self.g.data_ptr() if flag else None))
        _, f, g, st = self._post(flag >= 1)
        return f, g, st

    def pair(self, xf, yg, flag_y=2):
        xfd, ygd = self.xdev(xf), self.xdev(yg)
        self._pre()
        self.nat.check(self.lib.accbpg_dopt_pair(self.rt.ctx, self.rt.stream, self.Hp, self.m, self.n, self.ldh,
                                                 xfd.data_ptr(), ygd.data_ptr(), flag_y, self.ws.data_ptr(),
                                                 self.rt.slot(SLOT_X), self.rt.slot(SLOT_Y), self.g.data_ptr()))
        return self._post(True)

    def pair_from_gram(self, Mx, My, flag_y):
        keep = [None if Mx is None else Mx.clone(), My.clone()]
        self._pre()
        self.nat.check(self.lib.accbpg_dopt_pair_from_gram(
            self.rt.ctx, self.rt.stream, self.Hp, self.m, self.n, self.ldh, None if Mx is None else Mx.data_ptr(),
            My.data_ptr(), flag_y, self.ws.data_ptr(), None if Mx is None else self.rt.slot(SLOT_X),
            self.rt.slot(SLOT_Y), self.g.data_ptr() if flag_y else None))
        fx, fy, g, st = self._post(flag_y >= 1)
        assert torch.equal(My, keep[1]), "pair_from_gram wrote into My"
        if Mx is not None:
            assert torch.equal(Mx, keep[0]), "pair_from_gram wrote into Mx"
        else:
            assert np.isnan(fx)
        return (None if Mx is None else fx), fy, g, st

    def factor(self, M, want_inverse, L=None):
        keep = M.clone()
        self._pre()
        self.nat.check(self.lib.accbpg_dopt_factor(self.rt.ctx, self.rt.stream, self.m, M.data_ptr(),
                                                   None if L is None else L.data_ptr(), want_inverse,
                                                   self.ws.data_ptr(), self.rt.slot(SLOT_Y)))
        _, f, _, st = self._post(False)
        assert torch.equal(M, keep), "factor wrote into M"
        return f, st

    def grad(self):
        self._pre()
        self.nat.check(self.lib.accbpg_dopt_grad(self.rt.ctx, self.rt.stream, self.Hp, self.m, self.n, self.ldh,
                                                 self.ws.data_ptr(), self.g.data_ptr()))
        _, _, g, st = self._post(True)
        return g, st


def check_gram(M, H, x):
    m = H.shape[0]
    Mh = M[:m * m].cpu().numpy().reshape(m, m)
    R = (H * x) @ H.T
    assert np.array_equal(Mh, Mh.T)
    assert float(np.max(np.abs(Mh - R))) <= 1e-12 * float(np.max(np.abs(R)))


# ------------------------------------------------------------------------------------------------------- 2. routes
# m, n: which branch of dopt_factor_grad / chol_factor_inv the shape takes (even n first; odd n makes ldh odd, so the
# overlap is refused and the cp.async kernels run)
ROUTES = [
    (64, 700), (64, 701),          # per-step chain, one row block
    (65, 1030), (65, 1031),        # data-flow chain, nib = 1, no early row block: plain factor + gradient
    (128, 1030), (128, 1031),
    (129, 2050), (129, 2051),      # nib = 2, n_early = 1: the gated overlap
    (256, 2050), (256, 2051),
    (300, 4098), (300, 4099),      # nib = 3
    (500, 20002), (500, 20001),    # 8 block columns: DF_SMALL_WORKERS, 20-SM reserve, n_early = 2, hold0 > 0
    (513, 6002), (513, 6001),      # 9 block columns: the wide-worker rule and the 52-SM reserve
    (1100, 9000), (1100, 9001),    # nib = 9, n_early = 4
]


@pytest.mark.parametrize("m,n", ROUTES)
def test_dopt_routes_vs_extended_reference(acc, monkeypatch, m, n):
    """pair / func_grad (flags 0, 1, 2) / pair_from_gram against the reference, and the contracts between them bit for
    bit: pair = func_grad(xf, 0) + func_grad(yg, 2); pair_from_gram(M(xf), M(yg)) = pair; the overlapped gradient =
    ACCBPG_OVERLAP=0; three repeated calls agree; inputs only read; nothing written past the outputs."""
    monkeypatch.delenv("ACCBPG_OVERLAP", raising=False)
    H, xs = problem(m, n)
    op = Op(acc, H)
    for kf, ky in (("a", "b"), ("b", "c"), ("c", "a")):
        rx, ry = problem_ref(m, n, kf), problem_ref(m, n, ky)
        fx, fy, g, st = op.pair(xs[kf], xs[ky])
        assert st == 0
        check_f(fx, rx, ("pair fx", kf))
        check_f(fy, ry, ("pair fy", ky))
        check_g(g, ry, ("pair g", ky))
        # the header's contract: the same bits as two separate calls
        f0, g0, st0 = op.func_grad(xs[kf], 0)
        f2, g2, st2 = op.func_grad(xs[ky], 2)
        assert st0 == st2 == 0 and g0 is None
        assert f0 == fx and f2 == fy and np.array_equal(g2, g)
        _, g1, _ = op.func_grad(xs[ky], 1)
        assert np.array_equal(g1, g)
        # from Gram matrices: the same bits again, M(xf) / M(yg) only read
        Mx, My = op.gram(xs[kf]), op.gram(xs[ky])
        check_gram(Mx, H, xs[kf])
        fx2, fy2, g3, st3 = op.pair_from_gram(Mx, My, 2)
        assert st3 == 0 and fx2 == fx and fy2 == fy and np.array_equal(g3, g)
        for flag_y in (0, 1, 2):
            _, fy3, g4, st4 = op.pair_from_gram(None, My, flag_y)
            assert st4 == 0 and fy3 == fy
            if flag_y:
                assert np.array_equal(g4, g)
        # the gated triangular GEMM under the chain against the plain factor + gradient (read on every call)
        monkeypatch.setenv("ACCBPG_OVERLAP", "0")
        f5, g5, _ = op.func_grad(xs[ky], 2)
        fx5, fy5, g6, _ = op.pair(xs[kf], xs[ky])
        monkeypatch.delenv("ACCBPG_OVERLAP")
        assert f5 == fy and np.array_equal(g5, g)
        assert fx5 == fx and fy5 == fy and np.array_equal(g6, g)
    # run to run
    outs = [op.pair(xs["c"], xs["b"]) for _ in range(3)]
    assert all(o[0] == outs[0][0] and o[1] == outs[0][1] and np.array_equal(o[2], outs[0][2]) for o in outs)


# ------------------------------------------------------------------------------------------------------- 3. switches
_SWITCH_SCRIPT = r"""
import hashlib, sys
sys.path.insert(0, {root!r})
import numpy as np, torch
import accbpg_and_fw_b200 as acc
from accbpg_and_fw_b200 import _native as nat
lib, rt = nat.lib, acc.Runtime.get()
h = hashlib.sha256()
for m, n in ((500, 20002), (1100, 9000)):
    gen = torch.Generator(device="cuda").manual_seed(m)
    H = torch.randn(m, n, dtype=torch.float64, device="cuda", generator=gen)
    H[m - 1] *= 8.0
    xf = torch.rand(n, dtype=torch.float64, device="cuda", generator=gen) + 0.05
    yg = 1000.0 * (torch.rand(n, dtype=torch.float64, device="cuda", generator=gen) + 0.05)
    ws = torch.zeros(lib.accbpg_dopt_workspace_bytes(m, n), dtype=torch.uint8, device="cuda")
    g = torch.empty(n, dtype=torch.float64, device="cuda")
    for rep in range(2):
        nat.check(lib.accbpg_dopt_pair(rt.ctx, rt.stream, H.data_ptr(), m, n, n, xf.data_ptr(), yg.data_ptr(), 2,
                                       ws.data_ptr(), rt.slot(50), rt.slot(51), g.data_ptr()))
        v = rt.read(50, 2)
        assert abs(float(torch.dot(yg, g)) + m) <= 1e-9 * m
        h.update(np.array(v).tobytes()); h.update(g.cpu().numpy().tobytes())
        nat.check(lib.accbpg_dopt_func_grad(rt.ctx, rt.stream, H.data_ptr(), m, n, n, xf.data_ptr(), 2, ws.data_ptr(),
                                            rt.slot(51), g.data_ptr()))
        v = rt.read(51, 1)
        h.update(np.array(v).tobytes()); h.update(g.cpu().numpy().tobytes())
print("DOPTHASH", h.hexdigest())
"""

_SWITCHES = ("ACCBPG_EARLY_BLOCKS", "ACCBPG_TRMM_HOLD", "ACCBPG_CHOL_WORKERS", "ACCBPG_CHAIN_SMS", "ACCBPG_OVERLAP")


def test_dopt_scheduling_switches_bit_identical():
    """Switches that only change the scheduling of the chain and the triangular GEMM (read once per process, hence the
    subprocesses) give the default's bits at m = 500 (8 block columns) and m = 1100 (18).  ACCBPG_EARLY_BLOCKS=99 is
    clamped to nib - 1 for each m.  The chain reserve stays at or above its default: below it, the gated GEMM could take
    the SMs the chain it waits for needs."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    res = {}
    for name, env in (("default", {}),
                      ("early 1", {"ACCBPG_EARLY_BLOCKS": "1"}), ("early nib-1", {"ACCBPG_EARLY_BLOCKS": "99"}),
                      ("hold 0", {"ACCBPG_TRMM_HOLD": "0"}), ("hold 90", {"ACCBPG_TRMM_HOLD": "90"}),
                      ("workers 1", {"ACCBPG_CHOL_WORKERS": "1"}), ("workers 3", {"ACCBPG_CHOL_WORKERS": "3"}),
                      ("reserve 100", {"ACCBPG_CHAIN_SMS": "100"})):
        e = {k: v for k, v in os.environ.items() if k not in _SWITCHES}
        e.update(env)
        r = subprocess.run([sys.executable, "-c", _SWITCH_SCRIPT.format(root=root)], env=e, capture_output=True,
                           text=True, timeout=600)
        assert r.returncode == 0, (name, r.stderr[-2000:])
        line = [ln for ln in r.stdout.splitlines() if ln.startswith("DOPTHASH ")]
        assert line, (name, r.stdout[-500:])
        res[name] = line[-1]
    assert len(set(res.values())) == 1, res


# ------------------------------------------------------------------------------------------------------- 4. history
@pytest.mark.parametrize("m,n", [(129, 2050), (500, 6002)])
def test_dopt_call_history_on_one_workspace(acc, m, n):
    """A scripted sequence of calls on one workspace, fresh x every time (alternately x and 1000 x), checked against
    the reference after every call; accbpg_dopt_grad after value-only calls uses the L^-1 of the last
    want_inverse = 1 call.  Two operators (two workspaces, different H) run the sequence interleaved on the one
    context, which shares its side streams, events and ticket words between them."""
    ops = []
    for k in range(2):
        H = make_H(m, n, 77 + k)
        ops.append({"op": Op(acc, H), "H": H, "seed": 500 + 100 * k, "i": 0, "g_inv": None})

    def nextx(s):
        s["i"] += 1
        x = draw_x(n, "abc"[s["i"] % 3], s["seed"] + s["i"])
        x = x * (1000.0 if s["i"] % 2 else 1.0)
        return x, ref_dopt(s["H"], x)

    def grad_is_last_inverse(s, what):
        g, st = s["op"].grad()
        assert st == 0 and np.array_equal(g, s["g_inv"]), what

    def s_fg2(s):
        x, r = nextx(s)
        f, g, st = s["op"].func_grad(x, 2)
        assert st == 0
        check_f(f, r, "fg2")
        check_g(g, r, "fg2")
        s["g_inv"] = g

    def s_fg0(s):
        x, r = nextx(s)
        f, _, st = s["op"].func_grad(x, 0)
        assert st == 0
        check_f(f, r, "fg0")
        grad_is_last_inverse(s, "grad after func_grad flag 0")

    def s_pair(s):
        (x, rx), (y, ry) = nextx(s), nextx(s)
        fx, fy, g, st = s["op"].pair(x, y)
        assert st == 0
        check_f(fx, rx, "pair fx")
        check_f(fy, ry, "pair fy")
        check_g(g, ry, "pair g")
        s["g_inv"] = g
        grad_is_last_inverse(s, "grad after pair")

    def s_pfg(s):
        (x, rx), (y, ry) = nextx(s), nextx(s)
        fx, fy, g, st = s["op"].pair_from_gram(s["op"].gram(x), s["op"].gram(y), 1)
        assert st == 0
        check_f(fx, rx, "pfg fx")
        check_f(fy, ry, "pfg fy")
        check_g(g, ry, "pfg g")
        s["g_inv"] = g

    def s_pfg_value(s):
        y, ry = nextx(s)
        _, fy, _, st = s["op"].pair_from_gram(None, s["op"].gram(y), 0)
        assert st == 0
        check_f(fy, ry, "pfg value")
        grad_is_last_inverse(s, "grad after pair_from_gram flag 0")

    def s_factor_L(s):
        x, r = nextx(s)
        M = s["op"].gram(x)
        L = torch.full((m, m), SENTINEL, dtype=F64, device="cuda")
        f, st = s["op"].factor(M, 0, L)
        assert st == 0
        check_f(f, r, "factor")
        Lh, Mh = L.cpu().numpy(), M[:m * m].cpu().numpy().reshape(m, m)
        assert np.array_equal(Lh, np.tril(Lh))
        assert float(np.max(np.abs(Lh @ Lh.T - Mh))) <= 1e-12 * float(np.max(np.abs(Mh)))
        grad_is_last_inverse(s, "grad after factor want_inverse = 0")

    def s_factor_inv(s):
        x, r = nextx(s)
        f, st = s["op"].factor(s["op"].gram(x), 1)
        assert st == 0
        check_f(f, r, "factor inv")
        g, st = s["op"].grad()
        assert st == 0
        check_g(g, r, "grad after factor want_inverse = 1")
        s["g_inv"] = g

    script = [s_fg2, s_fg0, s_pair, s_factor_L, s_pfg, s_pfg_value, s_fg0, s_factor_inv, s_pair, s_pfg_value,
              s_factor_L, s_fg2, s_fg0]
    for step in script:
        for s in ops:
            step(s)


# ------------------------------------------------------------------------------------------------------- 5. strided
@pytest.mark.parametrize("case", ["ldh=n+2", "ldh=n+3", "H+1", "x+1"])
@pytest.mark.parametrize("m,n", [(65, 1030), (300, 4098), (513, 6002)])
def test_dopt_strided_and_misaligned_operands(acc, m, n, case):
    """H as a column window of a wider device matrix (ldh = n + 2 keeps the TMA paths, ldh = n + 3 is odd), an H base
    8-byte but not 16-byte aligned, an x base likewise: gram, func_grad, pair and grad against the reference."""
    H, xs = problem(m, n)
    kw = {"ldh=n+2": dict(ldh=n + 2), "ldh=n+3": dict(ldh=n + 3), "H+1": dict(h_off=1), "x+1": dict(x_off=1)}[case]
    op = Op(acc, H, **kw)
    ra, rb = problem_ref(m, n, "a"), problem_ref(m, n, "b")
    check_gram(op.gram(xs["b"]), H, xs["b"])
    f, g, st = op.func_grad(xs["a"], 2)
    assert st == 0
    check_f(f, ra, case)
    check_g(g, ra, case)
    fx, fy, g2, st = op.pair(xs["a"], xs["b"])
    assert st == 0
    check_f(fx, ra, case)
    check_f(fy, rb, case)
    check_g(g2, rb, case)
    f0, _, st = op.func_grad(xs["a"], 0)
    assert st == 0 and f0 == fx
    g3, st = op.grad()
    assert st == 0 and np.array_equal(g3, g2)


# ------------------------------------------------------------------------------------------------------- 6. not PD
@pytest.mark.parametrize("m", [65, 200, 500])
@pytest.mark.parametrize("where", ["last", "mid"])
def test_dopt_exactly_singular_on_the_data_flow_chain(acc, m, where):
    """Row r of H is nonzero only on columns where x = 0: row and column r of M are exact zeros and the pivot is exactly
    0 (a support smaller than m would leave a Schur complement of rounding noise).  The chain replaces the pivot by 1
    and flags it: ValueError from the dense operator, the same status bits from pair as from two separate calls, and
    the next good call is correct."""
    n = 4 * m + 6
    r = m - 1 if where == "last" else 64 * ((m - 1) // 128) + 30
    rng = np.random.RandomState(m + (r << 3))
    H = make_H(m, n, 9 * m + r)
    zero = rng.rand(n) < 0.25
    H[r, ~zero] = 0.0
    bad = rng.rand(n) + 0.05
    bad[zero] = 0.0
    good = rng.rand(n) + 0.05
    rg = ref_dopt(H, good)
    op = Op(acc, H)
    _, _, st_bad0 = op.func_grad(bad, 0)
    _, _, st_bad2 = op.func_grad(bad, 2)
    f, g, st_good = op.func_grad(good, 2)
    assert st_bad0 & NOT_PD and st_bad2 & NOT_PD and st_good == 0
    check_f(f, rg, "good after bad")
    check_g(g, rg, "good after bad")
    for xf, yg in ((bad, good), (good, bad), (bad, bad)):
        _, _, st_f = op.func_grad(xf, 0)
        _, _, st_y = op.func_grad(yg, 2)
        _, _, _, st_p = op.pair(xf, yg)
        assert st_p == (st_f | st_y)
        Mx, My = op.gram(xf), op.gram(yg)
        _, _, _, st_q = op.pair_from_gram(Mx, My, 2)
        assert st_q == (st_f | st_y)
    fx, fy, g, st = op.pair(good, good)
    assert st == 0
    check_f(fx, rg, "pair after bad")
    check_f(fy, rg, "pair after bad")
    check_g(g, rg, "pair after bad")
    f_dense = acc.DOptimalObj(H)
    with pytest.raises(ValueError):
        f_dense(bad)
    with pytest.raises(ValueError):
        f_dense.func_grad(bad)
    assert abs(f_dense(good) - rg.f) <= 1e-10 * max(1.0, abs(rg.f))


# ------------------------------------------------------------------------------------------------------- 7. sparse
SPARSE_N = [1, 63, 64, 65, 1000, 296 * 64 + 17]   # 1 stands for m + 1; the last: more 64-column tiles than SP_GRID
SPARSE_CASES = [(m, n) for m in (2, 33, 64, 65, 127, 128)
                for n in sorted({m + 1 if k == 1 else k for k in SPARSE_N}) if n > m]


def sparse_H(m, n, seed):
    """CSC H with: a structural diagonal (row j in column j < m, so M is positive definite), column 0 fully dense, an
    empty last column, a skewed nnz distribution (most columns 0-2 entries, some near-dense) and explicit stored zeros."""
    rng = np.random.RandomState(seed)
    rows, cols, vals = [], [], []
    for j in range(n - 1):
        if j == 0:
            rr = np.arange(m)
        else:
            k = min(m, rng.geometric(0.5) - 1 if rng.rand() > 0.05 else rng.randint(m // 2, m + 1))
            rr = rng.choice(m, size=k, replace=False)
            if j < m and j not in rr:
                rr = np.append(rr, j)
        v = rng.randn(rr.size)
        if j < m:
            v[rr == j] = 1.0 + rng.rand()
        if rr.size > 1 and rng.rand() < 0.2:
            v[np.flatnonzero(rr != j)[0]] = 0.0     # explicit stored zero
        rows.append(rr)
        cols.append(np.full(rr.size, j))
        vals.append(v)
    rows, cols, vals = np.concatenate(rows), np.concatenate(cols), np.concatenate(vals)
    vals[rows == m - 1] *= 4.0                      # the last row carries a larger scale
    return sp.csc_matrix((vals, (rows, cols)), shape=(m, n))


def _check_sparse(acc, fs, Hd, x):
    ref = ref_dopt(Hd, x)
    fd = acc.DOptimalObj(Hd)
    v, g = fs.func_grad(x)
    vd, gd = fd.func_grad(x)
    check_f(v, ref, "sparse f")
    check_g(g, ref, "sparse g")
    assert abs(v - vd) <= 1e-10 * max(1.0, abs(vd)) and relerr(g, gd) <= 1e-9
    assert fs(x) == v and np.array_equal(fs.gradient(x), g)


@pytest.mark.parametrize("m,n", SPARSE_CASES)
def test_sparse_dopt_kernels(acc, m, n):
    """accbpg_dopt_sparse_gram / _grad (SparseDOptimalObj) against the reference and the dense operator on toarray():
    empty and fully dense columns, skewed nnz, explicit zeros, rows unsorted within a column (raw arrays)."""
    Hs = sparse_H(m, n, 31 * m + n)
    Hd = Hs.toarray()
    rng = np.random.RandomState(n)
    x = rng.rand(n) + 0.05
    x[-1] = 5.0                                        # weight on the empty column: contributes nothing
    fs = acc.SparseDOptimalObj(Hs)
    assert np.array_equal(fs.toarray(), Hd)
    _check_sparse(acc, fs, Hd, x)
    _check_sparse(acc, fs, Hd, 1000.0 * draw_x(n, "b", n))
    # raw arrays with the rows of every column in reverse order
    perm = np.concatenate([np.arange(Hs.indptr[j], Hs.indptr[j + 1])[::-1] for j in range(n)]).astype(np.int64)
    fr = acc.SparseDOptimalObj(Hs.indptr.copy(), Hs.indices[perm], Hs.data[perm], m)
    v, g = fr.func_grad(x)
    assert v == fs(x) and np.array_equal(g, fs.gradient(x))


@pytest.mark.parametrize("m,n", [(33, 1000), (128, 296 * 64 + 17)])
def test_sparse_dopt_duplicate_entries_are_summed(acc, m, n):
    """A duplicated (row, column) entry means the sum of the two values, as in scipy's toarray(): the Gram matrix, the
    gradient and the dense operator must all see the same H, from a scipy matrix and from raw arrays."""
    Hs = sparse_H(m, n, 7 * m + n)
    rng = np.random.RandomState(m)
    dup = rng.choice(Hs.nnz, size=max(8, Hs.nnz // 10), replace=False)
    col_of = np.repeat(np.arange(n), np.diff(Hs.indptr))
    rows = np.concatenate([Hs.indices, Hs.indices[dup]])
    cols = np.concatenate([col_of, col_of[dup]])
    vals = np.concatenate([Hs.data, 0.5 + rng.rand(dup.size)])
    order = np.argsort(cols, kind="stable")
    indptr = np.concatenate([[0], np.cumsum(np.bincount(cols, minlength=n))]).astype(np.int64)
    indices, values = rows[order], vals[order]
    Hd = sp.csc_matrix((values, indices, indptr), shape=(m, n)).toarray()   # sums the duplicates
    x = rng.rand(n) + 0.05
    raw = acc.SparseDOptimalObj(indptr, indices.copy(), values.copy(), m)
    _check_sparse(acc, raw, Hd, x)
    Hdup = sp.csc_matrix((values.copy(), indices.copy(), indptr.copy()), shape=(m, n))
    nnz0 = Hdup.nnz
    fs = acc.SparseDOptimalObj(Hdup)
    assert Hdup.nnz == nnz0                            # the caller's matrix is left as it was
    _check_sparse(acc, fs, Hd, x)


def test_sparse_dopt_errors(acc):
    """An empty row makes M singular (ValueError), x < 0 is an AssertionError, and row indices outside [0, m) are
    refused on construction instead of being dropped by the kernels."""
    m, n = 65, 1000
    Hs = sparse_H(m, n, 5).tolil()
    Hs[40, :] = 0.0
    Hs = Hs.tocsc()
    Hs.eliminate_zeros()
    fs = acc.SparseDOptimalObj(Hs)
    x = np.random.RandomState(1).rand(n) + 0.05
    with pytest.raises(ValueError):
        fs(x)
    with pytest.raises(ValueError):
        fs.func_grad(x)
    good = acc.SparseDOptimalObj(sparse_H(m, n, 5))
    xb = x.copy()
    xb[17] = -1e-3
    with pytest.raises(AssertionError):
        good(xb)
    assert np.isfinite(good(x))
    H2 = sparse_H(m, n, 6)
    for bad in (m, -1):
        idx = H2.indices.copy()
        idx[3] = bad
        with pytest.raises(AssertionError):
            acc.SparseDOptimalObj(H2.indptr, idx, H2.data, m)
