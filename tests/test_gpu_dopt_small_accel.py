"""ABPG and ABPG_gain on small D-optimal designs as one launch (config.fused_small, dopt_abpg_small_kernel in
csrc/small.cu) against the reference's golden runs, the operator-by-operator loop and the NumPy oracle."""
import os
import time

import numpy as np
import pytest

from conftest import GOLDEN, relerr, first_fork
from oracle import accbpg_oracle as orc

FTOL = 1e-9
# (m, n, seed): the shapes of test_gpu_drivers.py's BPG comparison - tiny, ragged column splits, m close to n, n > 1024
SHAPES = [(80, 200, 10), (5, 6, 1), (30, 600, 3), (96, 120, 4), (16, 41, 5), (13, 506, 6), (2, 3, 7), (7, 9, 8),
          (64, 300, 9), (33, 400, 11), (8, 1100, 12), (70, 197, 13)]
ABPG_CONFIGS = {"eqF": dict(theta_eq=False), "eqT": dict(theta_eq=True),
                "rs_g": dict(restart=True, restart_rule='g'), "rs_f": dict(restart=True, restart_rule='f')}
GAIN_CONFIGS = {"default": dict(), "G0": dict(G0=0.1), "eqF": dict(theta_eq=False), "checkdiv": dict(checkdiv=True),
                "rs_g": dict(restart=True, restart_rule='g'), "rs_f": dict(restart=True, restart_rule='f'),
                "ls": dict(ls_inc=2.0, ls_dec=1.5)}
ITS = 100


@pytest.fixture(scope="module")
def acc():
    import accbpg_and_fw_b200 as a
    return a


@pytest.fixture(scope="module")
def dopt(acc):
    return acc.D_opt_design(80, 200, randseed=10)


def ferr(F, Fref):
    assert F.shape == Fref.shape, (F.shape, Fref.shape)
    return float(np.max(np.abs(F - Fref) / np.maximum(np.abs(Fref), 1e-3)))


def run(acc, fused, gain, *args, linear_images=True, pipeline=True, **kw):
    from accbpg_and_fw_b200 import config
    old = config.fused_small, config.linear_images, config.pipeline
    config.fused_small, config.linear_images, config.pipeline = fused, linear_images, pipeline
    try:
        return (acc.ABPG_gain if gain else acc.ABPG)(*args, verbose=kw.pop("verbose", False), **kw)
    finally:
        config.fused_small, config.linear_images, config.pipeline = old


def outcome(fn, *args, **kw):
    """The solve's result, or the type of the exception it raised (the reference's assertions, the operator loop's
    division by an exactly zero D(z+, z))."""
    try:
        return fn(*args, **kw)
    except (AssertionError, ZeroDivisionError, ValueError) as e:
        return type(e)


def last_info():
    from accbpg_and_fw_b200 import drivers
    return drivers._abpg_small.last_info


def oracle(H, L, x0, gamma, its, gain, kw):
    ho = orc.make_burg("simplex")
    return outcome(orc.ABPG_gain if gain else orc.ABPG, orc.make_dopt(H), ho, L, x0, gamma, its, **kw)


def oracle_noise(H, L, x0, its, gain, kw, gamma=2):
    """(largest relative move of the oracle's F, whether its discrete sequence or its length forks) when H is perturbed
    by one ulp, four draws: the instance's own sensitivity to rounding."""
    r0 = oracle(H, L, x0, gamma, its, gain, kw)
    if isinstance(r0, type):
        return np.inf, True
    worst, fork = 0.0, False
    for seed in range(4):
        Hp = H * (1 + 2.2e-16 * np.sign(np.random.RandomState(seed).randn(*H.shape)))
        rp = oracle(Hp, L, x0, gamma, its, gain, kw)
        if isinstance(rp, type):
            return np.inf, True
        k = min(len(r0[1]), len(rp[1]))
        worst = max(worst, ferr(rp[1][:k], r0[1][:k]))
        fork = fork or len(r0[1]) != len(rp[1]) or (gain and first_fork(rp[2], r0[2]) < k)
    return worst, fork


def check_against_operator_path(r1, r2, gain, what):
    """F to 1e-10, the gain sequence identical until F moves by less than 1e-10 |F| per iteration (then the line-search
    test compares rounding noise), x to 1e-6."""
    F1, F2 = r1[1], r2[1]
    assert r1[-1].shape == F1.shape
    k = min(len(F1), len(F2))
    assert len(F1) == len(F2) or abs(F1[k - 1] - F1[k - 2]) <= 1e-12 * abs(F1[k - 1]), (what, len(F1), len(F2))
    assert ferr(F1[:k], F2[:k]) <= 1e-10, (what, ferr(F1[:k], F2[:k]))
    if gain:
        small = np.nonzero(np.abs(np.diff(F2[:k])) < 1e-10 * np.abs(F2[1:k]))[0]
        kl = int(small[0]) if len(small) else k
        assert np.array_equal(r1[2][:kl], r2[2][:kl]), (what, first_fork(r1[2], r2[2]), kl)
    assert relerr(r1[0], r2[0]) <= 1e-6, (what, relerr(r1[0], r2[0]))


def check_golden(acc, dopt, t, fused, linear_images=True):
    """The 80 x 200 golden runs with the bars of test_gpu_drivers.py."""
    f, h, L, x0 = dopt
    kw = dict(linear_images=linear_images)
    x, F, G, T = run(acc, fused, False, f, h, L, x0, gamma=2, maxitrs=1000, theta_eq=False, **kw)
    assert ferr(F, t["abpg_F"]) <= FTOL
    assert relerr(G[:200], t["abpg_G"][:200]) <= 1e-6
    x, F, G, T = run(acc, fused, False, f, h, L, x0, gamma=2, maxitrs=1000, theta_eq=True, **kw)
    assert ferr(F, t["abpg_eq_F"]) <= FTOL
    x, F, G, T = run(acc, fused, False, f, h, L, x0, gamma=2, maxitrs=400, theta_eq=True, restart=True, **kw)
    assert ferr(F, t["abpg_rs_F"]) <= FTOL
    x, F, Gain, Gdiv, Gavg, T = run(acc, fused, True, f, h, L, x0, gamma=2, maxitrs=1000, G0=0.1, theta_eq=True, **kw)
    assert ferr(F, t["gain_F"]) <= FTOL
    k = first_fork(Gain, t["gain_Gain"])
    assert k >= 500 and np.mean(Gain != t["gain_Gain"]) <= 0.02, k
    assert relerr(Gavg[:k], t["gain_Gavg"][:k]) <= 1e-12
    assert relerr(Gdiv[:200], t["gain_Gdiv"][:200]) <= 1e-6
    assert relerr(x, t["gain_x"]) <= 1e-6
    x, F, Gain, Gdiv, Gavg, T = run(acc, fused, True, f, h, L, x0, gamma=2, maxitrs=400, G0=1, theta_eq=False,
                                    restart=True, **kw)
    assert ferr(F, t["gain_rs_F"]) <= FTOL and np.mean(Gain != t["gain_rs_Gain"]) <= 0.02


def test_smem_bytes_picks_what_fits():
    """The shape query is host-only: the notebook and test shapes fit one SM's plan, shapes outside the m <= 128,
    n > m domain or too large for a cluster of 4 do not."""
    from accbpg_and_fw_b200 import _native as nat
    lib = nat.lib
    for m, n in [(80, 200), (13, 506), (30, 600), (2, 3), (8, 1100)]:
        assert 0 < lib.accbpg_dopt_abpg_small_smem_bytes(m, n) <= 227 * 1024, (m, n)
    for m, n in [(128, 4096), (129, 500), (50, 50), (0, 5)]:
        assert lib.accbpg_dopt_abpg_small_smem_bytes(m, n) == 0, (m, n)


@pytest.mark.gpu
@pytest.mark.parametrize("fused", [True, False])
def test_golden_runs_both_paths(acc, dopt, golden_traj, fused):
    check_golden(acc, dopt, golden_traj, fused)
    if fused:
        assert int(last_info()[2]) == 4


@pytest.mark.gpu
def test_operator_loop_kept_at_this_shape(acc, dopt, golden_traj):
    """With fused_small off the 80 x 200 instance takes the operator loop: its pipelined and synchronous forms agree bit
    for bit (early stop included), and its direct-evaluation mode matches the golden runs."""
    f, h, L, x0 = dopt
    res = {}
    for mode in (False, True):
        res[mode] = (run(acc, False, False, f, h, L, x0, gamma=2, maxitrs=200, theta_eq=False, pipeline=mode),
                     run(acc, False, False, f, h, L, x0, gamma=2, maxitrs=200, epsilon=1e-3, theta_eq=False,
                         pipeline=mode))
    for a, b in zip(res[False], res[True]):
        assert len(a[1]) == len(b[1])
        assert np.array_equal(a[1], b[1]) and np.array_equal(a[2], b[2]) and np.array_equal(a[0], b[0])
    assert len(res[True][1][1]) < 200
    assert ferr(res[True][0][1], golden_traj["abpg_F"][:200]) <= FTOL
    check_golden(acc, dopt, golden_traj, False, linear_images=False)


@pytest.mark.gpu
def test_fused_golden_without_linear_images(acc, dopt, golden_traj):
    """The fused solve evaluates from scratch: it is the path with linear_images off too, and gives the same runs."""
    from accbpg_and_fw_b200 import _native as nat
    f, h, L, x0 = dopt
    c0 = nat.launch_count()
    run(acc, True, False, f, h, L, x0, gamma=2, maxitrs=50, linear_images=False)
    assert nat.launch_count() - c0 == 1
    check_golden(acc, dopt, golden_traj, True, linear_images=False)


@pytest.mark.gpu
@pytest.mark.parametrize("gain,cfg", [(False, c) for c in ABPG_CONFIGS] + [(True, c) for c in GAIN_CONFIGS])
def test_fused_matches_operator_path(acc, gain, cfg):
    kw = (GAIN_CONFIGS if gain else ABPG_CONFIGS)[cfg]
    for m, n, seed in SHAPES:
        f, h, L, x0 = acc.D_opt_design(m, n, randseed=seed)
        r1 = outcome(run, acc, True, gain, f, h, L, x0, gamma=2, maxitrs=ITS, **kw)
        r2 = outcome(run, acc, False, gain, f, h, L, x0, gamma=2, maxitrs=ITS, **kw)
        if isinstance(r2, type) or isinstance(r1, type):
            # the reference's own assertion fires on this instance: both paths raise it
            assert r1 is r2 or (r2 is ZeroDivisionError and not isinstance(r1, type)), ((m, n), r1, r2)
            continue
        try:
            check_against_operator_path(r1, r2, gain, (m, n))
        except AssertionError:
            # Where the instance itself is chaotic - one-ulp perturbations of H move the oracle's F past the bar or fork
            # its discrete sequence - the two paths are compared on the first 15 iterations only
            noise, fork = oracle_noise(f.H, L, x0, ITS, gain, kw)
            if not (fork or noise > 1e-10):
                raise
            bar = max(1e-10, 10 * oracle_noise(f.H, L, x0, 15, gain, kw)[0])
            k = min(15, len(r1[1]), len(r2[1]))
            assert ferr(r1[1][:k], r2[1][:k]) <= bar, ((m, n), ferr(r1[1][:k], r2[1][:k]), bar)
            assert r1[1][-1] <= r1[1][0]
            continue
        # a larger epsilon: the stop D(z+, z) < epsilon fires at the same iteration
        s1 = outcome(run, acc, True, gain, f, h, L, x0, gamma=2, maxitrs=2 * ITS, epsilon=1e-8, **kw)
        s2 = outcome(run, acc, False, gain, f, h, L, x0, gamma=2, maxitrs=2 * ITS, epsilon=1e-8, **kw)
        if isinstance(s1, type) or isinstance(s2, type):
            assert s1 is s2, ((m, n), s1, s2)
            continue
        assert len(s1[1]) == len(s2[1]), ((m, n), len(s1[1]), len(s2[1]))


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["design", "housing"])
def test_fused_against_numpy_oracle(acc, which):
    if which == "design":
        f, h, L, x0 = acc.D_opt_design(80, 200, randseed=10)
    else:
        f, h, L, x0 = acc.D_opt_libsvm(os.path.join(GOLDEN, "housing_libsvm.txt"))
        assert (f.m, f.n) == (13, 506)
    H = np.asarray(f.H)
    x, F, G, T = run(acc, True, False, f, h, L, x0, gamma=2, maxitrs=300)
    xo, Fo, Go, To = oracle(H, L, x0, 2, 300, False, {})
    assert len(F) == len(Fo) and ferr(F, Fo) <= FTOL, ferr(F, Fo)
    x, F, Gain, Gdiv, Gavg, T = run(acc, True, True, f, h, L, x0, gamma=2, maxitrs=300)
    xo, Fo, Gaino, Gdivo, Gavgo, To = oracle(H, L, x0, 2, 300, True, {})
    k = min(len(F), len(Fo))
    assert ferr(F[:k], Fo[:k]) <= FTOL, ferr(F[:k], Fo[:k])
    if not oracle_noise(H, L, x0, 300, True, {})[1]:
        assert len(F) == len(Fo) and np.array_equal(Gain, Gaino), first_fork(Gain, Gaino)


@pytest.mark.gpu
@pytest.mark.parametrize("gamma", [1.5, 3.0])
def test_non_integer_gamma(acc, gamma):
    """Exponents other than 1 and 2 go through pow on the device.  ABPG with gamma = 3 diverges on this instance, where
    one-ulp perturbations of H move the oracle's F far past the bar: there the first 15 iterations are compared, to ten
    times that noise."""
    f, h, L, x0 = acc.D_opt_design(80, 200, randseed=10)
    H = np.asarray(f.H)
    for gain in (False, True):
        r1 = run(acc, True, gain, f, h, L, x0, gamma=gamma, maxitrs=ITS)
        r2 = run(acc, False, gain, f, h, L, x0, gamma=gamma, maxitrs=ITS)
        k = min(len(r1[1]), len(r2[1]))
        if ferr(r1[1][:k], r2[1][:k]) > FTOL:
            noise, fork = oracle_noise(H, L, x0, ITS, gain, {}, gamma=gamma)
            assert fork or noise > 1e-10, (gain, ferr(r1[1][:k], r2[1][:k]), noise)
            bar = max(1e-10, 10 * oracle_noise(H, L, x0, 15, gain, {}, gamma=gamma)[0])
            k = min(15, k)
            assert ferr(r1[1][:k], r2[1][:k]) <= bar, (gain, ferr(r1[1][:k], r2[1][:k]), bar)


@pytest.mark.gpu
def test_one_launch_and_fallback(acc, dopt):
    from accbpg_and_fw_b200 import _native as nat
    f, h, L, x0 = dopt
    for gain in (False, True):
        for li in (True, False):
            c0 = nat.launch_count()
            run(acc, True, gain, f, h, L, x0, gamma=2, maxitrs=50, linear_images=li)
            assert nat.launch_count() - c0 == 1
        c0 = nat.launch_count()
        run(acc, False, gain, f, h, L, x0, gamma=2, maxitrs=50)
        assert nat.launch_count() - c0 > 1
    # too large for a cluster of 4: the operator loop runs, and still matches the oracle
    assert nat.lib.accbpg_dopt_abpg_small_smem_bytes(128, 4096) == 0
    f, h, L, x0 = acc.D_opt_design(128, 4096, randseed=3)
    for gain in (False, True):
        c0 = nat.launch_count()
        r = run(acc, True, gain, f, h, L, x0, gamma=2, maxitrs=20)
        assert nat.launch_count() - c0 > 1
        ro = oracle(np.asarray(f.H), L, x0, 2, 20, gain, {})
        assert ferr(r[1], ro[1]) <= FTOL


@pytest.mark.gpu
@pytest.mark.parametrize("cluster", [1, 2])
def test_other_cluster_sizes(cluster, golden_traj):
    """The default splits the columns of H over a 4-CTA cluster; the 1- and 2-CTA forms (ACCBPG_SMALL_CLUSTER, read once
    per process) run the golden 80 x 200 ABPG and ABPG_gain trajectories in a subprocess."""
    import subprocess
    import sys
    import tempfile
    from conftest import ROOT
    code = ("import sys, numpy as np; sys.path.insert(0, %r); import accbpg_and_fw_b200 as acc; "
            "from accbpg_and_fw_b200 import drivers; "
            "f, h, L, x0 = acc.D_opt_design(80, 200, randseed=10); "
            "a = acc.ABPG(f, h, L, x0, gamma=2, maxitrs=1000, theta_eq=False, verbose=False); "
            "ca = drivers._abpg_small.last_info[2]; "
            "g = acc.ABPG_gain(f, h, L, x0, gamma=2, maxitrs=1000, G0=0.1, theta_eq=True, verbose=False); "
            "cg = drivers._abpg_small.last_info[2]; "
            "np.savez(sys.argv[1], F=a[1], G=a[2], gF=g[1], Gain=g[2], C=[ca, cg])" % ROOT)
    with tempfile.TemporaryDirectory() as d:
        out = os.path.join(d, "r.npz")
        env = dict(os.environ, ACCBPG_SMALL_CLUSTER=str(cluster))
        subprocess.run([sys.executable, "-c", code, out], check=True, env=env, timeout=600)
        r = np.load(out)
        assert list(r["C"]) == [cluster, cluster]
        assert ferr(r["F"], golden_traj["abpg_F"]) <= FTOL
        assert relerr(r["G"][:200], golden_traj["abpg_G"][:200]) <= 1e-6
        assert ferr(r["gF"], golden_traj["gain_F"]) <= FTOL
        k = first_fork(r["Gain"], golden_traj["gain_Gain"])
        assert k >= 500 and np.mean(r["Gain"] != golden_traj["gain_Gain"]) <= 0.02, k


@pytest.mark.gpu
def test_fused_is_deterministic(acc, dopt):
    """Fixed-order sums, rank-ordered cluster sums, no floating-point atomics: two solves are bit-identical."""
    f, h, L, x0 = dopt
    for gain in (False, True):
        a = run(acc, True, gain, f, h, L, x0, gamma=2, maxitrs=300)
        c = run(acc, True, gain, f, h, L, x0, gamma=2, maxitrs=300)
        assert np.array_equal(a[1], c[1]) and np.array_equal(a[2], c[2])
        assert np.array_equal(np.asarray(a[0]), np.asarray(c[0]))


@pytest.mark.gpu
@pytest.mark.parametrize("fused", [True, False])
def test_fused_raises_like_the_operator_path(acc, dopt, fused):
    f, h, L, x0 = dopt
    for gain in (False, True):
        for bad_value in (-0.5, 0.0):
            bad = np.array(x0, dtype=float)
            bad[17] = bad_value
            with pytest.raises(AssertionError):
                run(acc, fused, gain, f, h, L, bad, gamma=2, maxitrs=20)
    # the first trip stops on D(z+, z) < epsilon: the reference's Gdr is unbound
    with pytest.raises(UnboundLocalError):
        run(acc, fused, True, f, h, L, x0, gamma=2, maxitrs=20, epsilon=1e300)


@pytest.mark.gpu
def test_fused_time_stamps(acc, dopt):
    """T[k]: the device clock at the top of iteration k, offset by the host time at which the solve was launched."""
    f, h, L, x0 = dopt
    for gain in (False, True):
        t0 = time.time()
        out = run(acc, True, gain, f, h, L, x0, gamma=2, maxitrs=300)
        wall = time.time() - t0
        F, T = out[1], out[-1]
        assert T.shape == F.shape
        assert np.all(T >= 0) and np.all(np.diff(T) >= 0)
        assert T[-1] <= wall


@pytest.mark.gpu
def test_verbose_lines_match(acc, dopt, capsys):
    """Same lines, same columns except the time, fused and operator loop."""
    f, h, L, x0 = dopt
    for gain in (False, True):
        outs = []
        for fused in (True, False):
            run(acc, fused, gain, f, h, L, x0, gamma=2, maxitrs=40, verbose=True, verbskip=3)
            outs.append(capsys.readouterr().out.strip().splitlines())
        a, c = outs
        assert len(a) == len(c) and len(a) > 10
        for la, lc in zip(a, c):
            assert la.split()[:-1] == lc.split()[:-1], (la, lc)


@pytest.mark.gpu
def test_entry_point_rejects_bad_arguments(acc, dopt):
    """NULL pointers, a shape that does not fit, ldh < n, non-finite or non-positive L, gamma, G0, ls_inc, ls_dec or
    eps_prox, maxitrs < 1, an unknown driver or restart rule: ACCBPG_E_ARG."""
    import torch
    from accbpg_and_fw_b200 import _native as nat
    f, h, L, x0 = dopt
    rt = f.rt
    x = rt.to_device(x0).clone()
    hist = torch.empty(7 * 10 + 16, dtype=torch.float64, device=rt.device)
    E_ARG = nat.MACROS["ACCBPG_E_ARG"]
    H = f._Hd

    def call(driver=nat.MACROS["ACCBPG_SMALL_DRV_ABPG_GAIN"], Hp=H.data_ptr(), m=f.m, n=f.n, ldh=H.stride(0),
             xp=x.data_ptr(), L=L, gamma=2.0, maxitrs=10, eps_prox=1e-8, rule=nat.MACROS["ACCBPG_SMALL_RESTART_NONE"],
             G0=1.0, ls_inc=1.2, ls_dec=1.2, histp=hist.data_ptr(), infop=hist.data_ptr() + 8 * 70):
        with rt.on_device():
            return nat.lib.accbpg_dopt_abpg_small(rt.ctx, rt.stream, driver, Hp, m, n, ldh, xp, L, gamma, maxitrs,
                                                  1e-14, eps_prox, 1, 0, rule, G0, ls_inc, ls_dec, 0, histp, infop)
    for bad in (dict(Hp=None), dict(xp=None), dict(histp=None), dict(infop=None), dict(m=128, n=4096),
                dict(m=129, n=500), dict(ldh=f.n - 1), dict(L=float("nan")), dict(L=0.0), dict(gamma=float("inf")),
                dict(gamma=-1.0), dict(G0=0.0), dict(ls_inc=float("nan")), dict(ls_dec=-2.0), dict(eps_prox=0.0),
                dict(eps_prox=float("inf")), dict(maxitrs=0), dict(driver=7), dict(rule=9)):
        assert call(**bad) == E_ARG, bad
    assert call() == nat.MACROS["ACCBPG_OK"]
    rt.read(rt.S_F, 1)
