"""GPU parity: every operator of the hot path, called through the C ABI, against the CPU oracle
(oracle/accbpg_oracle.py) and the golden fixtures generated from the real reference.
Tolerances: objective values 1e-10 relative, gradients 1e-9 relative (FP64 throughout;
only summation order, Cholesky-vs-LU and 1-ulp libm differences separate the two paths);
index results (LMO vertices) bit-exact."""
import numpy as np
import pytest
import torch

from conftest import relerr
from oracle import accbpg_oracle as orc

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def acc():
    import accbpg_and_fw_b200 as a
    return a


def rel(a, b):
    return relerr(a, b)


# ------------------------------------------------------------------ D-optimal design objective
@pytest.mark.parametrize("m,n,seed", [(80, 200, 10), (30, 1000, 3), (129, 517, 7), (5, 6, 1), (64, 4096, 2),
                                      (200, 3001, 4), (300, 20000, 5),
                                      # TMA mainloops with ragged tiles: m just past a 128 / 64 boundary, n not a multiple of 16
                                      (129, 520, 8), (257, 1030, 9), (65, 130, 11), (384, 4098, 12), (1, 2, 13),
                                      # 65 block columns: one launch per block column, then the gradient after the chain
                                      (4160, 8322, 14)])
def test_dopt_func_grad_vs_oracle(acc, m, n, seed):
    rng = np.random.RandomState(seed)
    f, h, L, x0 = acc.D_opt_design(m, n, randseed=seed)
    fo = orc.make_dopt(f.H)
    x = rng.rand(n) + 1e-3
    x /= x.sum()
    for xx in (x0, x):
        fx, g = f.func_grad(xx)
        fxo, go = fo.func_grad(xx)
        assert abs(fx - fxo) <= 1e-10 * max(1.0, abs(fxo)), (fx, fxo)
        assert rel(g, go) <= 1e-9
        assert abs(f(xx) - fxo) <= 1e-10 * max(1.0, abs(fxo))
        assert rel(f.gradient(xx), go) <= 1e-9
        # size-independent identity: sum_j x_j g_j = -trace(M^-1 M) = -m
        assert abs(float(np.dot(xx, g)) + m) <= 1e-9 * m


@pytest.mark.parametrize("m", [1, 13, 63, 64, 65, 150, 257, 500, 777])
def test_dopt_factor_entry_point(acc, m):
    """accbpg_dopt_factor through the C ABI: L L^T = M, -log det, and the cached L^{-1} used by accbpg_dopt_grad."""
    from accbpg_and_fw_b200 import _native as nat
    lib = nat.lib
    rt = acc.Runtime.get()
    rng = np.random.RandomState(100 + m)
    n = 2 * m + 6
    H = rng.randn(m, n)
    x = rng.rand(n) + 0.05
    M = (H * x) @ H.T
    Md = torch.tensor(M, device="cuda")
    Hd = torch.tensor(H, device="cuda")
    Ld = torch.full((m, m), 7.0, dtype=torch.float64, device="cuda")
    gd = torch.empty(n, dtype=torch.float64, device="cuda")
    ws = torch.zeros(lib.accbpg_dopt_workspace_bytes(m, n), dtype=torch.uint8, device="cuda")
    for want_inv in (0, 1):
        nat.check(lib.accbpg_dopt_factor(rt.ctx, rt.stream, m, Md.data_ptr(), Ld.data_ptr(), want_inv, ws.data_ptr(),
                                         rt.slot(40)))
        val = rt.read(40, 1)[0]
        L = Ld.cpu().numpy()
        assert np.array_equal(L, np.tril(L))
        assert np.max(np.abs(L @ L.T - M)) <= 1e-12 * np.max(np.abs(M))
        sign, logdet = np.linalg.slogdet(M)
        assert abs(val + logdet) <= 1e-11 * max(1.0, abs(logdet))
    nat.check(lib.accbpg_dopt_grad(rt.ctx, rt.stream, Hd.data_ptr(), m, n, n, ws.data_ptr(), gd.data_ptr()))
    rt.read(40, 0)
    gref = -np.sum(H * np.linalg.solve(M, H), axis=0)
    assert rel(gd.cpu().numpy(), gref) <= 1e-9
    # value-only factorisation without an L output
    nat.check(lib.accbpg_dopt_factor(rt.ctx, rt.stream, m, Md.data_ptr(), None, 0, ws.data_ptr(), rt.slot(41)))
    assert rt.read(41, 1)[0] == val


def test_dopt_golden_fixtures(acc, golden_ops):
    for tag, (m, n, seed) in {"dopt_80x200": (80, 200, 10), "dopt_30x1000": (30, 1000, 3),
                              "dopt_129x517": (129, 517, 7)}.items():
        f, h, L, x0 = acc.D_opt_design(m, n, randseed=seed)
        fx, g = f.func_grad(golden_ops[tag + "_x"])
        assert abs(fx - golden_ops[tag + "_f"]) <= 1e-10 * abs(golden_ops[tag + "_f"])
        assert rel(g, golden_ops[tag + "_g"]) <= 1e-9
        assert abs(f(x0) - golden_ops[tag + "_f0"]) <= 1e-10 * abs(golden_ops[tag + "_f0"])
    f = acc.DOptimalObj(golden_ops["housing_H"])
    x0 = np.ones(506) / 506
    assert abs(f(x0) - golden_ops["housing_f0"]) <= 1e-10 * abs(golden_ops["housing_f0"])
    assert rel(f.gradient(x0), golden_ops["housing_g0"]) <= 1e-9


def test_dopt_device_tensor_in_out_and_sparse_x(acc):
    f, h, L, x0 = acc.D_opt_design(40, 300, randseed=3)
    fo = orc.make_dopt(f.H)
    xd = torch.tensor(x0, device="cuda")
    fx, g = f.func_grad(xd)
    assert isinstance(g, torch.Tensor) and g.is_cuda and g.dtype == torch.float64
    assert rel(g.cpu().numpy(), fo.gradient(x0)) <= 1e-9
    # x with exact zeros (support of 2m columns): still positive definite
    xs = np.zeros(300)
    xs[:80] = 1.0 / 80
    fx, g = f.func_grad(xs)
    fxo, go = fo.func_grad(xs)
    assert abs(fx - fxo) <= 1e-10 * abs(fxo) and rel(g, go) <= 1e-8


def test_dopt_error_behaviour(acc):
    f, h, L, x0 = acc.D_opt_design(20, 60, randseed=2)
    bad = x0.copy()
    bad[7] = -1e-3
    with pytest.raises(AssertionError):
        f.func_grad(bad)
    with pytest.raises(AssertionError):
        f.func_grad(x0[:-1])
    rank_def = np.zeros(60)
    rank_def[:5] = 0.2                       # only 5 columns for m = 20 -> singular
    with pytest.raises(ValueError):
        f(rank_def)
    assert np.isfinite(f(x0))                # status word was cleared by the failed calls
    with pytest.raises(AssertionError):
        acc.DOptimalObj(np.random.randn(10, 10))


def test_dopt_properties_at_benchmark_shape(acc):
    """C2 shape (500 x 50000): too slow for the NumPy oracle inside the suite, so size-independent properties:
    <x, g> = -m, f(c x) = f(x) - m log c, run-to-run bit reproducibility."""
    m, n = 500, 50000
    g0 = torch.Generator(device="cuda").manual_seed(1)
    H = torch.randn(m, n, dtype=torch.float64, device="cuda", generator=g0)
    f = acc.DOptimalObj(H)
    x = torch.rand(n, dtype=torch.float64, device="cuda", generator=g0) + 0.1
    x /= x.sum()
    fx, g = f.func_grad(x)
    assert abs(float(torch.dot(x, g)) + m) <= 1e-9 * m
    f2 = f(3.0 * x)
    assert abs(f2 - (fx - m * np.log(3.0))) <= 1e-10 * abs(fx)
    fx_b, g_b = f.func_grad(x)
    assert fx_b == fx and torch.equal(g, g_b)
    # spot-check 64 gradient entries against a dense solve
    M = (H * x) @ H.T
    cols = torch.arange(0, n, n // 64, device="cuda")[:64]
    ref = -(H[:, cols] * torch.linalg.solve(M, H[:, cols])).sum(0)
    assert rel(g[cols].cpu().numpy(), ref.cpu().numpy()) <= 1e-9
    assert abs(fx + float(torch.linalg.slogdet(M)[1])) <= 1e-10 * abs(fx)


# ------------------------------------------------------------------ Poisson / KL objectives
@pytest.mark.parametrize("kind", ["poisson", "kl"])
@pytest.mark.parametrize("m,n", [(200, 100), (37, 1001), (300, 70000), (4, 3)])
def test_linreg_vs_oracle(acc, kind, m, n):
    rng = np.random.RandomState(m + n)
    A = rng.rand(m, n)
    A = A / A.sum(axis=0)
    xs = rng.rand(n) + 0.05
    b = A @ xs * (1 + 0.1 * (rng.rand(m) - 0.5))
    x = rng.rand(n) + 0.05
    f = (acc.PoissonRegression if kind == "poisson" else acc.KLdivRegression)(A, b)
    fo = (orc.make_poisson if kind == "poisson" else orc.make_kl)(A, b)
    fx, g = f.func_grad(x)
    fxo, go = fo.func_grad(x)
    assert abs(fx - fxo) <= 1e-10 * max(abs(fxo), 1e-3), (fx, fxo)
    assert np.max(np.abs(g - go)) <= 1e-10 * np.max(np.abs(go))
    assert abs(f(x) - fxo) <= 1e-10 * max(abs(fxo), 1e-3)
    assert np.max(np.abs(f.gradient(x) - go)) <= 1e-10 * np.max(np.abs(go))


def test_linreg_golden(acc, golden_ops):
    o = golden_ops
    f = acc.PoissonRegression(o["poisson_A"], o["poisson_b"])
    fx, g = f.func_grad(o["poisson_x"])
    assert abs(fx - o["poisson_f"]) <= 1e-10 * abs(o["poisson_f"]) and rel(g, o["poisson_g"]) <= 1e-9
    f = acc.KLdivRegression(o["kl_A"], o["kl_b"])
    fx, g = f.func_grad(o["kl_x"])
    assert abs(fx - o["kl_f"]) <= 1e-10 * abs(o["kl_f"]) and rel(g, o["kl_g"]) <= 1e-8
    f, h, L, x0 = acc.Poisson_regrL1(200, 100, noise=1e-4, lamda=0, randseed=1)
    assert np.array_equal(f.A, o["poisson_A"]) and L == o["poisson_L"]
    assert abs(f(x0) - o["poisson_f0"]) <= 1e-10 * abs(o["poisson_f0"])
    f, h, L, x0 = acc.KL_nonneg_regr(1000, 100, noise=0.01, lamdaL1=0.001, randseed=1)
    assert abs(f(x0) + h.extra_Psi(x0) - o["kl1000_F0"]) <= 1e-10 * abs(o["kl1000_F0"])


# ------------------------------------------------------------------ Bregman kernels
def test_bregman_kernels_golden(acc, golden_ops):
    o = golden_ops
    x, y, g, gp, ys = o["vec_x"], o["vec_y"], o["vec_g"], o["vec_gpos"], o["vec_ysimplex"]
    L = 0.7
    tol = 1e-12
    b = acc.BurgEntropy()
    assert abs(b(x) - o["burg_h"]) <= tol * abs(o["burg_h"])
    assert rel(b.gradient(x), o["burg_grad"]) <= tol
    assert abs(b.divergence(x, y) - o["burg_div"]) <= tol * abs(o["burg_div"])
    assert rel(b.prox_map(gp, L), o["burg_prox"]) <= tol
    assert rel(b.div_prox_map(y, gp, L), o["burg_divprox"]) <= tol
    b1 = acc.BurgEntropyL1(lamda=0.3)
    assert rel(b1.prox_map(gp, L), o["burgl1_prox"]) <= tol
    assert rel(b1.div_prox_map(y, g * 0.1, L), o["burgl1_divprox"]) <= tol
    assert abs(b1.extra_Psi(x) - o["burgl1_psi"]) <= tol * abs(o["burgl1_psi"])
    b2 = acc.BurgEntropyL2(lamda=0.3)
    assert rel(b2.prox_map(g, L), o["burgl2_prox"]) <= 1e-10        # (sqrt(gg^2+4l)-gg) cancels for large gg
    assert rel(b2.div_prox_map(y, g, L), o["burgl2_divprox"]) <= 1e-10
    assert abs(b2.extra_Psi(x) - o["burgl2_psi"]) <= tol * abs(o["burgl2_psi"])
    bs = acc.BurgEntropySimplex()
    assert rel(bs.prox_map(g, L), o["burgs_prox"]) <= 1e-11
    assert rel(bs.div_prox_map(ys, g, L), o["burgs_divprox"]) <= 1e-11
    s = acc.ShannonEntropy()
    assert abs(s(x) - o["sh_h"]) <= tol * abs(o["sh_h"])
    assert rel(s.gradient(x), o["sh_grad"]) <= 1e-11
    assert abs(s.divergence(x, y) - o["sh_div"]) <= 1e-11 * abs(o["sh_div"])
    assert rel(s.prox_map(g, L), o["sh_prox"]) <= tol
    assert rel(s.div_prox_map(y, g, L), o["sh_divprox"]) <= tol
    s1 = acc.ShannonEntropyL1(lamda=0.3)
    assert rel(s1.prox_map(g, L), o["shl1_prox"]) <= tol
    assert rel(s1.div_prox_map(y, g, L), o["shl1_divprox"]) <= tol
    ss = acc.ShannonEntropySimplex()
    assert rel(ss.prox_map(g, L), o["shs_prox"]) <= tol
    assert rel(ss.div_prox_map(ys, g, L), o["shs_divprox"]) <= tol


@pytest.mark.parametrize("n", [1, 2, 33, 200, 4097, 100003, 1000000])
def test_burg_simplex_newton_replay(acc, n):
    """Same Newton iteration count and root as the reference recurrence, at every size incl. n = 10^6."""
    rng = np.random.RandomState(n % 1000 + 1)
    g = rng.randn(n)
    y = rng.rand(n) + 1e-3
    y /= y.sum()
    L = 0.37
    h = acc.BurgEntropySimplex()
    rt = h.rt
    for yy in (None, y):
        if n <= 5000:
            ho = orc.make_burg("simplex")
            xo = ho.prox_map(g, L) if yy is None else ho.div_prox_map(yy, g, L)
            nbis_o, nnewt_o, c_o = ho.newton_trace[-1]
        else:   # vectorised restatement of the same recurrence (the builtin-sum oracle takes minutes at 10^6)
            gg = (g if yy is None else g - L * (-1 / yy)) / L
            cmin = -gg.min(); c = cmin + 1; nbis_o = 0
            while np.sum(1 / (gg + c)) - 1 < 0:
                c = (cmin + c) / 2.0; nbis_o += 1
            fc = np.sum(1 / (gg + c)) - 1; nnewt_o = 0
            while abs(fc) > 1e-8:
                fpc = np.sum(-1.0 / (gg + c) ** 2)
                if (c - (c - fc / fpc)) == 0:
                    break
                c = c - fc / fpc; fc = np.sum(1 / (gg + c)) - 1; nnewt_o += 1
            xo, c_o = 1.0 / (gg + c), c
        x = h.prox_map(g, L) if yy is None else h.div_prox_map(yy, g, L)
        info = rt.scal[rt.S_AUX1:rt.S_AUX1 + 3].cpu().numpy()
        assert (int(info[0]), int(info[1])) == (nbis_o, nnewt_o)
        # the multiplier c is conditioned like n*eps (f'(c) = -sum 1/(gg+c)^2 ~ 1/n): compare on that scale
        assert abs(info[2] - c_o) <= 1e-13 * n * max(1.0, abs(c_o))
        assert rel(x, xo) <= 1e-10
        assert abs(x.sum() - 1.0) <= 1e-7       # normalised only to eps, like the reference


@pytest.mark.parametrize("n,world", [(200, 2), (4097, 4), (100003, 8)])
def test_burg_simplex_gathered_root_find(acc, n, world):
    """The column-sharded form of the Burg-simplex prox on one GPU: every rank's padded slice of gg gathered into
    one vector (padding = +inf), accbpg_burg_simplex_root on it, accbpg_burg_simplex_finish_dev per slice.  The result
    must equal the single-kernel prox (same recurrence, same stopping rule) independently of the sharding."""
    from accbpg_and_fw_b200 import _native as nat
    lib = nat.lib
    rng = np.random.RandomState(n)
    g = rng.randn(n)
    y = rng.rand(n) + 1e-3
    y /= y.sum()
    L = 0.41
    h = acc.BurgEntropySimplex()
    rt = h.rt
    ref = h.div_prox_map(y, g, L)
    info_ref = rt.read(rt.S_AUX1, 3)
    offs = acc.ColumnShard.partition(n, world)
    width = max(offs[r + 1] - offs[r] for r in range(world))
    full = torch.full((world * width,), float("inf"), dtype=torch.float64, device="cuda")
    yd, gd = torch.tensor(y, device="cuda"), torch.tensor(g, device="cuda")
    for r in range(world):
        lo, hi = offs[r], offs[r + 1]
        if hi > lo:
            ys, gs = yd[lo:hi].contiguous(), gd[lo:hi].contiguous()
            nat.check(lib.accbpg_burg_simplex_prepare(rt.ctx, rt.stream, hi - lo, ys.data_ptr(), gs.data_ptr(), L,
                                                      full[r * width:].data_ptr(), rt.slot(44)))
    nat.check(lib.accbpg_burg_simplex_root(rt.ctx, rt.stream, world * width, full.data_ptr(), 1e-8, rt.slot(45)))
    out = torch.empty(n, dtype=torch.float64, device="cuda")
    for r in range(world):
        lo, hi = offs[r], offs[r + 1]
        if hi > lo:
            nat.check(lib.accbpg_burg_simplex_finish_dev(rt.ctx, rt.stream, hi - lo, full[r * width:].data_ptr(),
                                                         rt.slot(47), out[lo:].data_ptr()))
    info = rt.read(45, 3)
    assert info[0] == info_ref[0] and info[1] == info_ref[1]          # same bisection and Newton step counts
    # c = cmin + (a small positive shift) with |cmin| ~ max|gg|: the padded layout changes the summation order, and the
    # rounding of the two sums is amplified by that cancellation; the prox point itself is the meaningful comparison
    assert abs(info[2] - info_ref[2]) <= 1e-9 * abs(info_ref[2])
    assert rel(out.cpu().numpy(), ref) <= 1e-10


def test_bregman_error_behaviour(acc):
    b = acc.BurgEntropy()
    x = np.array([0.5, 0.0, 1.0])
    with pytest.raises(AssertionError):
        b(x)
    with pytest.raises(AssertionError):
        b.divergence(np.ones(3), x)
    with pytest.raises(AssertionError):
        b.prox_map(np.array([1.0, -1.0, 2.0]), 1.0)
    with pytest.raises(AssertionError):
        acc.BurgEntropyL1(lamda=0.1).prox_map(np.array([1.0, -0.2, 2.0]), 1.0)
    with pytest.raises(AssertionError):
        b.prox_map(np.ones(3), -1.0)
    with pytest.raises(AssertionError):
        acc.ShannonEntropy()(np.array([0.1, -0.1]))
    with pytest.raises(AssertionError):
        acc.ShannonEntropySimplex().div_prox_map(np.array([0.5, 0.0, 0.5]), np.ones(3), 1.0)
    assert np.isfinite(b(np.ones(3)))
    # Shannon at exact zeros: h(0) = 0 through the delta clamp
    s = acc.ShannonEntropy()
    so = orc.make_shannon()
    z = np.array([0.0, 0.3, 0.0, 0.7])
    assert abs(s(z) - so(z)) <= 1e-15 and abs(s.divergence(z, np.array([0.25] * 4)) - so.divergence(z, np.array([0.25] * 4))) <= 1e-15


def test_vector_primitives(acc):
    from accbpg_and_fw_b200 import _native as nat
    rt = acc.Runtime.get()
    lib = nat.lib
    for n in (1, 5, 1000, 123457):
        rng = np.random.RandomState(n % 97)
        a, b, g = rng.randn(n), rng.randn(n), rng.randn(n)
        ad, bd, gd = (rt.to_device(v) for v in (a, b, g))
        out = rt.empty(n)
        nat.check(lib.accbpg_vec_axpby(rt.ctx, rt.stream, n, 0.3, ad.data_ptr(), 0.7, bd.data_ptr(), out.data_ptr()))
        assert np.array_equal(out.cpu().numpy(), 0.3 * a + 0.7 * b)          # bit-exact: same two roundings
        nat.check(lib.accbpg_vec_step_toward(rt.ctx, rt.stream, n, ad.data_ptr(), bd.data_ptr(), 0.25, out.data_ptr()))
        assert np.array_equal(out.cpu().numpy(), a + 0.25 * (b - a))
        nat.check(lib.accbpg_vec_dot_diff(rt.ctx, rt.stream, n, gd.data_ptr(), ad.data_ptr(), bd.data_ptr(), rt.slot(40)))
        nat.check(lib.accbpg_vec_dot(rt.ctx, rt.stream, n, ad.data_ptr(), bd.data_ptr(), rt.slot(41)))
        nat.check(lib.accbpg_vec_sum(rt.ctx, rt.stream, n, ad.data_ptr(), rt.slot(42)))
        nat.check(lib.accbpg_vec_minmax(rt.ctx, rt.stream, n, ad.data_ptr(), rt.slot(43)))
        nat.check(lib.accbpg_vec_argext(rt.ctx, rt.stream, n, ad.data_ptr(), 1, rt.slot(45)))
        v = rt.read(40, 7)
        scale = np.sum(np.abs(g * (a - b))) + 1e-300
        assert abs(v[0] - np.dot(g, a - b)) <= 1e-14 * scale
        assert abs(v[1] - np.dot(a, b)) <= 1e-14 * np.sum(np.abs(a * b))
        assert abs(v[2] - a.sum()) <= 1e-14 * np.sum(np.abs(a))
        assert v[3] == a.min() and v[4] == a.max()
        assert v[5] == a.max() and int(v[6]) == int(np.argmax(a))


# ------------------------------------------------------------------ LMOs
def test_lmos_golden(acc, golden_ops):
    o = golden_ops
    g, x, gt = o["vec_g"], o["vec_x"], o["lmo_gties"]
    lmo = acc.lmo_simplex(2.0)
    s = lmo(gt)
    assert np.array_equal(s, o["lmo_simplex"])                      # bit-exact, first index among 3 exact ties
    assert lmo.last_index() == 137
    assert rel(acc.lmo_l2_ball(1.5)(g), o["lmo_l2"]) <= 1e-14
    assert rel(acc.lmo_l2_ball(1.5, center=x)(g), o["lmo_l2_center"]) <= 1e-13
    assert np.max(np.abs(acc.lmo_l2_ball_positive_orthant(1.5, center=x, epsilon=1e-3)(g) - o["lmo_l2pos"])) <= 1e-14
    assert np.array_equal(acc.lmo_linf_ball(0.5, center=x)(g), o["lmo_linf"])
    assert np.array_equal(acc.lmo_matrix_simplex(3.0)(g.reshape(25, 40)), o["lmo_msimplex"])
    assert np.array_equal(acc.lmo_matrix_box(-np.ones((25, 40)), 2 * np.ones((25, 40)))(g.reshape(25, 40)), o["lmo_mbox"])


def test_lmo_simplex_large_ties(acc):
    n = 1000003
    g = np.ones(n)
    g[[999999, 5, 777777]] = -2.0
    lmo = acc.lmo_simplex()
    s = lmo(g)
    assert lmo.last_index() == 5 and s[5] == 1.0 and s[4] == 1e-15 and s.sum() == orc.lmo_simplex_eval(g).sum()


def test_squared_l2_norm_kernel(acc):
    """SquaredL2Norm (functions.py:738-759) against its NumPy definition."""
    rng = np.random.RandomState(3)
    x, y, g = rng.randn(1001), rng.randn(1001), rng.randn(1001)
    h = acc.SquaredL2Norm()
    assert abs(h(x) - 0.5 * np.vdot(x, x)) <= 1e-12 * np.vdot(x, x)
    assert np.array_equal(h.gradient(x), x)
    assert abs(h.divergence(x, y) - 0.5 * np.vdot(x - y, x - y)) <= 1e-12 * np.vdot(x - y, x - y)
    assert np.array_equal(h.prox_map(g, 0.7), -(1 / 0.7) * g)
    assert np.array_equal(h.div_prox_map(y, g, 0.7), y - (1 / 0.7) * g)
    assert h.extra_Psi(x) == 0


def test_lmo_nuclear_norm_ball(acc):
    """Leading singular pair by power iteration on the device against np.linalg.svd (functions_lmo.py:4-13)."""
    rng = np.random.RandomState(11)
    for p, q in [(60, 40), (33, 120), (7, 7)]:
        G = rng.randn(p, q) + 3.0 * np.outer(rng.randn(p), rng.randn(q)) / np.sqrt(p * q) * 4
        U, S, Vh = np.linalg.svd(G, full_matrices=False)
        ref = np.outer(U[:, 0], Vh[0])
        out = acc.lmo_nuclear_norm_ball()(G)
        assert out.shape == (p, q)
        assert np.max(np.abs(out - ref)) <= 1e-9
        outd = acc.lmo_nuclear_norm_ball()(torch.tensor(G, device="cuda"))
        assert outd.is_cuda and np.max(np.abs(outd.cpu().numpy() - ref)) <= 1e-9


def test_vertex_gram_matches_the_syrk_of_the_vertex(acc):
    """accbpg_dopt_vertex_gram: fill*HH^T + (radius - fill) h_i h_i^T against the SYRK of the LMO's vertex vector."""
    from accbpg_and_fw_b200 import _native as nat
    lib = nat.lib
    rt = acc.Runtime.get()
    for m, n in [(30, 1000), (129, 520)]:
        f, h, L, x0 = acc.D_opt_design(m, n, randseed=4)
        rng = np.random.RandomState(m)
        g = rng.randn(n)
        g[[7, 311]] = g.min() - 1.0                      # exact tie: the first index wins
        lmo = acc.lmo_simplex(radius=2.0)
        s = lmo(g)
        assert lmo.last_index() == 7
        gd = torch.tensor(g, device="cuda")
        sd = torch.empty(n, dtype=torch.float64, device="cuda")
        lmo._enq(gd, sd, rt.S_AUX0)
        Mv = f._img_vertex(rt.S_AUX0 + 1, 1e-15, 2.0).cpu().numpy()
        Ms = f._img_compute(sd).cpu().numpy()
        ref = (f.H * s) @ f.H.T
        assert np.max(np.abs(Mv - ref)) <= 1e-12 * np.max(np.abs(ref))
        assert np.max(np.abs(Ms - ref)) <= 1e-12 * np.max(np.abs(ref))


def test_host_results_are_fresh_arrays_and_can_be_passed_back(acc):
    """Ownership rule of the reference protocol (SURVEY 8b): operators return fresh, writable arrays and never mutate
    their inputs.  Host results live in page-locked memory and are uploaded in place when passed back; the values must
    equal those obtained from an ordinary copy of the same vector."""
    fo, ho, Lo, x0 = orc.D_opt_design(60, 3000, randseed=4)
    f = acc.DOptimalObj(fo.H)
    h = acc.BurgEntropySimplex()
    g1 = f.gradient(x0)
    g2 = f.gradient(x0)
    assert isinstance(g1, np.ndarray) and g1.flags.writeable and g1.dtype == np.float64
    assert not np.shares_memory(g1, g2) and np.array_equal(g1, g2)
    keep = g1.copy()
    z_direct = h.div_prox_map(x0, g1, 0.9)                 # g1: page-locked result passed back
    z_copy = h.div_prox_map(x0, np.array(keep), 0.9)       # ordinary pageable copy
    assert np.array_equal(z_direct, z_copy) and np.array_equal(g1, keep)
    z_view = h.div_prox_map(x0[5:], g1[5:], 0.9)           # a view into a page-locked result
    assert np.array_equal(z_view, h.div_prox_map(x0[5:].copy(), keep[5:].copy(), 0.9))
    g1 *= 2.0                                              # the caller owns the result
    assert np.array_equal(f.gradient(x0), g2)
    for _ in range(20):                                    # the host allocator recycles blocks of dropped results only
        a = f.gradient(x0)
        b = h.div_prox_map(x0, a, 0.9)
        assert np.array_equal(a, g2) and np.array_equal(b, z_copy)


# ---- sparse design matrix (D_opt_libsvm without densifying): the four LIBSVM regression sets the reference ships ------
_LIBSVM = {"housing": "-4.137e+01", "abalone": "3.978e+01", "bodyfat": "-3.475e+01", "mpg": "-3.416e+01"}     # F(x0), SURVEY 8c


@pytest.mark.parametrize("name", sorted(_LIBSVM))
def test_sparse_dopt_libsvm_matches_dense_and_oracle(acc, name):
    """SparseDOptimalObj (compressed columns on the device, accbpg_dopt_sparse_gram / _grad) against the dense operator,
    the NumPy oracle on the densified matrix (accbpg/applications.py:17-33, functions.py:43-59) and the reference's
    4-digit F(x0); then 60 BPG iterations with line search: F to 1e-9, identical L_k."""
    import os
    from conftest import GOLDEN
    path = os.path.join(GOLDEN, name + "_libsvm.txt")
    fs, hs, Ls, x0 = acc.D_opt_libsvm(path, sparse=True)
    fd, hd, Ld, x0d = acc.D_opt_libsvm(path)
    assert type(fs).__name__ == "SparseDOptimalObj" and (fs.m, fs.n) == (fd.m, fd.n)
    H = fd.H
    assert np.array_equal(fs.toarray(), H)
    fo = orc.make_dopt(H)
    ho = orc.make_burg("simplex")
    assert f"{fs(x0):.3e}" == _LIBSVM[name]
    rng = np.random.RandomState(7)
    for x in (x0, rng.rand(fs.n) / fs.n + 1e-4):
        v, g = fs.func_grad(x)
        vo, go = fo.func_grad(x)
        vd, gd = fd.func_grad(x)
        assert abs(v - vo) <= 1e-10 * abs(vo) and abs(v - vd) <= 1e-10 * abs(vd)
        assert relerr(g, go) <= 1e-9 and relerr(g, gd) <= 1e-9
        assert abs(fs(x) - vo) <= 1e-10 * abs(vo) and relerr(fs.gradient(x), go) <= 1e-9
    xs, Fs, Lss, Ts = acc.BPG(fs, hs, 1.0, x0, maxitrs=60, linesearch=True, ls_ratio=1.2, verbose=False)
    xo, Fo, Lso, To = orc.BPG(fo, ho, 1.0, x0, maxitrs=60, linesearch=True, ls_ratio=1.2)
    assert np.array_equal(Lss, Lso)
    assert float(np.max(np.abs(Fs - Fo) / np.abs(Fo))) <= 1e-9
    with pytest.raises(AssertionError):
        fs(-x0)
