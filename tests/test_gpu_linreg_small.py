"""BPG on small Poisson / KL regression instances as one launch (config.fused_small, csrc/linreg_small.cu) against the
operator-by-operator loop, the reference's golden runs and the NumPy oracle."""
import time

import numpy as np
import pytest

from conftest import relerr, first_fork
from oracle import accbpg_oracle as orc

FTOL = 1e-9
KERNELS = [("BurgEntropy", 0.0), ("BurgEntropyL1", 1e-2), ("BurgEntropyL2", 1e-2),
           ("ShannonEntropy", 0.0), ("ShannonEntropyL1", 1e-2), ("ShannonEntropySimplex", 0.0)]
MODES = {"ls1.2": dict(linesearch=True, ls_ratio=1.2), "ls2.0": dict(linesearch=True, ls_ratio=2.0),
         "nols": dict(linesearch=False)}
# (m, n) -> cluster size: tiny, m > n and m < n, odd and ragged column splits
SHAPES = [((3, 2), 1), ((4, 6), 1), ((7, 5), 1), ((200, 100), 1), ((301, 97), 2), ((120, 400), 2), ((777, 101), 4),
          ((600, 120), 4), ((1000, 100), 8), ((1500, 61), 8)]
# Line search on these instances is chaotic: the NumPy oracle itself, started from x0 perturbed by one ulp, takes another
# L_k within 20-60 iterations (KL with the unconstrained Shannon kernels) or moves F by more than 1e-10 (Poisson with the
# Shannon kernel at ratio 2), as the reference does on KL_nonneg_regr (tests/test_noise_floor.py).  There the two paths
# are compared on the first 15 iterations, the bar test_kl_poisson_golden sets for that instance, to 1e-10 or - where
# the instance's own rounding noise is larger - to ten times what one-ulp perturbations of A move the oracle's F
# (KL 4 x 6 with the plain Shannon kernel: 1e-10 to 7e-10 by iteration 15).
CHAOTIC = {("kl", "ShannonEntropy", "ls1.2"), ("kl", "ShannonEntropy", "ls2.0"), ("kl", "ShannonEntropyL1", "ls1.2"),
           ("kl", "ShannonEntropyL1", "ls2.0"), ("poisson", "ShannonEntropy", "ls2.0")}


@pytest.fixture(scope="module")
def acc():
    import accbpg_and_fw_b200 as a
    return a


def ferr(F, Fref):
    assert F.shape == Fref.shape, (F.shape, Fref.shape)
    return float(np.max(np.abs(F - Fref) / np.maximum(np.abs(Fref), 1e-3)))


def data(m, n, seed, simplex):
    """A with unit column sums, b = A x_true with 20% multiplicative noise (x_true on the simplex for the simplex
    kernel): a residual that stays away from zero keeps the line search off rounding-level ties."""
    rs = np.random.RandomState(seed)
    A = rs.rand(m, n)
    A = A / A.sum(axis=0)
    xt = rs.rand(n)
    if simplex:
        xt = xt / xt.sum()
    b = (A @ xt) * (1 + 0.2 * (rs.rand(m) - 0.5))
    return A, b


def instance(acc, obj, hname, lam, m, n, seed):
    """(f, h, L, x0) on the GPU and the same instance for the oracle."""
    simplex = hname == "ShannonEntropySimplex"
    A, b = data(m, n, seed, simplex)
    f = (acc.PoissonRegression if obj == "poisson" else acc.KLdivRegression)(A, b)
    fo = (orc.make_poisson if obj == "poisson" else orc.make_kl)(A, b)
    h = getattr(acc, hname)(lam) if lam else getattr(acc, hname)()
    burg = hname.startswith("Burg")
    kind = {"BurgEntropy": "plain", "BurgEntropyL1": "l1", "BurgEntropyL2": "l2", "ShannonEntropy": "plain",
            "ShannonEntropyL1": "l1", "ShannonEntropySimplex": "simplex"}[hname]
    ho = orc.make_burg(kind, lam) if burg else orc.make_shannon(kind, lam)
    L = b.sum() if burg else max(A.sum(axis=0))
    x0 = np.ones(n) / n if simplex else np.ones(n)
    return f, h, fo, ho, L, x0


def run(acc, fused, *args, **kw):
    from accbpg_and_fw_b200 import config
    old = config.fused_small
    config.fused_small = fused
    try:
        return acc.BPG(*args, verbose=False, **kw)
    finally:
        config.fused_small = old


def cluster_used():
    from accbpg_and_fw_b200 import drivers
    return int(drivers._bpg_small.last_info[3])


def test_smem_bytes_picks_what_fits():
    """The shape query is host-only: the notebook instances fit, a 3000 x 200 A does not."""
    from accbpg_and_fw_b200 import _native as nat
    lib = nat.lib
    for m, n in [(200, 100), (1000, 100), (300, 120), (1, 1)]:
        assert 0 < lib.accbpg_linreg_bpg_small_smem_bytes(m, n) <= 227 * 1024
    for m, n in [(3000, 200), (0, 5), (5, 0)]:
        assert lib.accbpg_linreg_bpg_small_smem_bytes(m, n) == 0


@pytest.mark.gpu
@pytest.mark.parametrize("fused", [True, False])
def test_kl_poisson_golden_both_paths(acc, golden_traj, fused):
    """The BPG cases of the reference's golden runs, through the fused kernel and through the operator loop."""
    t = golden_traj
    f, h, L, x0 = acc.KL_nonneg_regr(300, 120, noise=0.01, lamdaL1=0.001, randseed=1)
    x, F, Ls, T = run(acc, fused, f, h, L, x0, maxitrs=300, linesearch=True)
    if fused:
        assert cluster_used() == 2
    # chaotic under 1-ulp noise from k ~ 20 (tests/test_noise_floor.py): 1e-9 parity on [0, 15)
    assert first_fork(Ls, t["kl_bpg_Ls"]) >= 15 and ferr(F[:15], t["kl_bpg_F"][:15]) <= FTOL
    assert F[-1] <= F[0] and abs(F[-1] - t["kl_bpg_F"][-1]) <= 0.1 * abs(t["kl_bpg_F"][-1])
    x, F, Ls, T = run(acc, fused, f, h, L, x0, maxitrs=300, linesearch=False)
    fo, ho, Lo, x0o = orc.KL_nonneg_regr(300, 120, noise=0.01, lamdaL1=0.001, randseed=1)
    xo, Fo, Lso, To = orc.BPG(fo, ho, Lo, x0o, maxitrs=300, linesearch=False)
    assert ferr(F, Fo) <= FTOL and relerr(x, xo) <= 1e-6
    f, h, L, x0 = acc.Poisson_regrL1(200, 100, noise=1e-4, lamda=0, randseed=1)
    x, F, Ls, T = run(acc, fused, f, h, L, x0, maxitrs=300, linesearch=True)
    if fused:
        assert cluster_used() == 1
    assert ferr(F, t["poi_bpg_F"]) <= FTOL and np.array_equal(Ls, t["poi_bpg_Ls"])


def oracle_noise_floor(fo_make, A, b, ho, L, x0, its, kw):
    """Largest relative move of the oracle's F over `its` iterations when A is perturbed by one ulp (four draws)."""
    F0 = orc.BPG(fo_make(A, b), ho, L, x0, maxitrs=its, **kw)[1]
    worst = 0.0
    for seed in range(4):
        Ap = A * (1 + 2.2e-16 * np.sign(np.random.RandomState(seed).randn(*A.shape)))
        Fp = orc.BPG(fo_make(Ap, b), ho, L, x0, maxitrs=its, **kw)[1]
        k = min(len(F0), len(Fp))
        worst = max(worst, ferr(Fp[:k], F0[:k]))
    return worst


def check_against_operator_path(r1, r2, what):
    x1, F1, L1, T1 = r1
    x2, F2, L2, T2 = r2
    assert T1.shape == F1.shape
    # the stopping test |F_k - F_k-1| < 1e-14 fires at rounding level: the runs may stop at different iterations there
    k = min(len(F1), len(F2))
    assert k >= 10 or len(F1) == len(F2), (what, len(F1), len(F2))
    if len(F1) != len(F2):
        assert abs(F1[k - 1] - F1[k - 2]) <= 1e-12 * abs(F1[k - 1]), (what, len(F1), len(F2))
    assert ferr(F1[:k], F2[:k]) <= 1e-10, (what, ferr(F1[:k], F2[:k]))
    # once F moves by less than 1e-10 |F| per iteration the line-search test compares rounding noise
    small = np.nonzero(np.abs(np.diff(F2[:k])) < 1e-10 * np.abs(F2[1:k]))[0]
    kl = int(small[0]) if len(small) else k
    assert np.array_equal(L1[:kl], L2[:kl]), (what, first_fork(L1, L2), kl)
    assert relerr(x1, x2) <= 1e-6, (what, relerr(x1, x2))


@pytest.mark.gpu
@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("hname,lam", KERNELS)
@pytest.mark.parametrize("obj", ["poisson", "kl"])
def test_fused_matches_operator_path(acc, obj, hname, lam, mode):
    kw = MODES[mode]
    for (m, n), C in SHAPES:
        f, h, fo, ho, L, x0 = instance(acc, obj, hname, lam, m, n, seed=m + n)
        r1 = run(acc, True, f, h, L, x0, maxitrs=200, **kw)
        assert cluster_used() == C, ((m, n), cluster_used())
        r2 = run(acc, False, f, h, L, x0, maxitrs=200, **kw)
        if (obj, hname, mode) in CHAOTIC:
            A, b = data(m, n, m + n, hname == "ShannonEntropySimplex")
            fmake = orc.make_poisson if obj == "poisson" else orc.make_kl
            bar = max(1e-10, 10 * oracle_noise_floor(fmake, A, b, ho, L, x0, 15, kw))
            assert first_fork(r1[2], r2[2]) >= 15, (m, n, first_fork(r1[2], r2[2]))
            assert ferr(r1[1][:15], r2[1][:15]) <= bar, (m, n, ferr(r1[1][:15], r2[1][:15]), bar)
            assert r1[1][-1] <= r1[1][0]
            continue
        check_against_operator_path(r1, r2, (m, n))
        # the stopping test (algorithms.py:66) fires at the same iteration
        s1 = run(acc, True, f, h, L, x0, maxitrs=400, epsilon=1e-3, **kw)
        s2 = run(acc, False, f, h, L, x0, maxitrs=400, epsilon=1e-3, **kw)
        assert len(s1[1]) == len(s2[1]) and np.array_equal(s1[2], s2[2]), ((m, n), len(s1[1]), len(s2[1]))


@pytest.mark.gpu
@pytest.mark.parametrize("hname,lam", KERNELS)
@pytest.mark.parametrize("obj", ["poisson", "kl"])
def test_fused_against_numpy_oracle(acc, obj, hname, lam):
    for (m, n) in [(200, 100), (1000, 100)]:
        f, h, fo, ho, L, x0 = instance(acc, obj, hname, lam, m, n, seed=m + n)
        x, F, Ls, T = run(acc, True, f, h, L, x0, maxitrs=200, linesearch=False)
        xo, Fo, Lso, To = orc.BPG(fo, ho, L, x0, maxitrs=200, linesearch=False)
        assert len(F) == len(Fo) and ferr(F, Fo) <= FTOL, ((m, n), ferr(F, Fo))
        assert relerr(x, xo) <= 1e-6
        if (obj, hname, "ls1.2") in CHAOTIC:
            continue
        x, F, Ls, T = run(acc, True, f, h, L, x0, maxitrs=200, linesearch=True)
        xo, Fo, Lso, To = orc.BPG(fo, ho, L, x0, maxitrs=200, linesearch=True)
        assert len(F) == len(Fo) and ferr(F, Fo) <= FTOL, ((m, n), ferr(F, Fo))
        assert np.array_equal(Ls, Lso), ((m, n), first_fork(Ls, Lso))


@pytest.mark.gpu
def test_one_launch_and_fallback(acc):
    from accbpg_and_fw_b200 import _native as nat
    f, h, fo, ho, L, x0 = instance(acc, "kl", "ShannonEntropyL1", 1e-3, 1000, 100, seed=3)
    for kw in MODES.values():
        c0 = nat.launch_count()
        run(acc, True, f, h, L, x0, maxitrs=50, **kw)
        assert nat.launch_count() - c0 == 1
        c0 = nat.launch_count()
        run(acc, False, f, h, L, x0, maxitrs=50, **kw)
        assert nat.launch_count() - c0 > 1
    # too large for a cluster of 8: the operator loop runs, and still matches the oracle
    assert nat.lib.accbpg_linreg_bpg_small_smem_bytes(3000, 200) == 0
    f, h, fo, ho, L, x0 = instance(acc, "poisson", "BurgEntropyL1", 1e-3, 3000, 200, seed=4)
    c0 = nat.launch_count()
    x, F, Ls, T = run(acc, True, f, h, L, x0, maxitrs=50, linesearch=False)
    assert nat.launch_count() - c0 > 1
    xo, Fo, Lso, To = orc.BPG(fo, ho, L, x0, maxitrs=50, linesearch=False)
    assert ferr(F, Fo) <= FTOL


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(200, 100), (1000, 100)])
def test_fused_is_deterministic(acc, shape):
    """Fixed-order sums, rank-ordered cluster sums, no floating-point atomics: two solves are bit-identical."""
    f, h, fo, ho, L, x0 = instance(acc, "kl", "ShannonEntropyL1", 1e-3, *shape, seed=5)
    a = run(acc, True, f, h, L, x0, maxitrs=300)
    b = run(acc, True, f, h, L, x0, maxitrs=300)
    assert np.array_equal(a[1], b[1]) and np.array_equal(a[2], b[2])
    assert np.array_equal(np.asarray(a[0]), np.asarray(b[0]))


@pytest.mark.gpu
@pytest.mark.parametrize("fused", [True, False])
def test_fused_raises_like_the_operator_path(acc, fused):
    # a negative entry in x0
    for hname, lam in [("BurgEntropyL1", 1e-3), ("ShannonEntropyL1", 1e-3)]:
        f, h, fo, ho, L, x0 = instance(acc, "poisson", hname, lam, 200, 100, seed=6)
        bad = x0.copy()
        bad[17] = -0.5
        with pytest.raises(AssertionError):
            run(acc, fused, f, h, L, bad, maxitrs=20)
    # plain Burg on Poisson: from a tiny x0 with a tiny L the shifted gradient g + L/x is negative
    f, h, fo, ho, L, x0 = instance(acc, "poisson", "BurgEntropy", 0.0, 200, 100, seed=6)
    with pytest.raises(AssertionError):
        run(acc, fused, f, h, 1e-6, 1e-3 * x0, maxitrs=20, linesearch=False)
    with pytest.raises(AssertionError):
        orc.BPG(fo, ho, 1e-6, 1e-3 * x0, maxitrs=20, linesearch=False)
    # Shannon on the simplex from a start with a zero entry
    f, h, fo, ho, L, x0 = instance(acc, "kl", "ShannonEntropySimplex", 0.0, 1000, 100, seed=6)
    bad = x0.copy()
    bad[40] = 0.0
    bad = bad / bad.sum()
    with pytest.raises(AssertionError):
        run(acc, fused, f, h, L, bad, maxitrs=20)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(200, 100), (1000, 100)])
def test_fused_time_stamps(acc, shape):
    """T[k]: the device clock at the top of iteration k, offset by the host time at which the solve was launched."""
    f, h, fo, ho, L, x0 = instance(acc, "poisson", "BurgEntropyL2", 1e-3, *shape, seed=8)
    t0 = time.time()
    x, F, Ls, T = run(acc, True, f, h, L, x0, maxitrs=500)
    wall = time.time() - t0
    assert T.shape == F.shape
    assert np.all(T >= 0) and np.all(np.diff(T) >= 0)
    assert T[-1] <= wall
