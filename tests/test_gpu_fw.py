"""GPU parity: D_opt_FW / D_opt_FW_away (device-resident loop) against the oracle and the golden runs.
F_k, the slacks SP/SN and the selected vertex indices; the FW vertex index must be bit-exact."""
import hashlib

import numpy as np
import torch
import pytest

from conftest import relerr
from oracle import accbpg_oracle as orc

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def acc():
    import accbpg_and_fw_b200 as a
    return a


def close(a, b, tol, floor=1e-3):
    assert a.shape == b.shape, (a.shape, b.shape)
    err = float(np.max(np.abs(a - b) / np.maximum(np.abs(b), floor)))
    assert err <= tol, err


def test_fw_golden(acc, golden_traj):
    t = golden_traj
    f, h, L, x0 = acc.D_opt_design(80, 200, randseed=10)
    x, F, SP, SN, T = acc.D_opt_FW(f.H, x0, 1e-8, 2000, verbose=False)
    close(F, t["dfw_F"], 1e-9); close(SP, t["dfw_SP"], 1e-7); close(SN, t["dfw_SN"], 1e-7)
    close(x, t["dfw_x"], 1e-6, floor=1e-6)
    assert T.shape == F.shape and np.all(np.diff(T) >= 0)


def test_fw_away_golden(acc, golden_traj):
    t = golden_traj
    f, h, L, x0 = acc.D_opt_design(80, 200, randseed=10)
    x, F, SP, SN, T = acc.D_opt_FW_away(f.H, x0, 1e-8, 2000, verbose=False)
    close(F, t["dfwa_F"], 1e-9); close(SP, t["dfwa_SP"], 1e-7); close(SN, t["dfwa_SN"], 1e-7)
    close(x, t["dfwa_x"], 1e-6, floor=1e-6)
    x, F, SP, SN, T = acc.D_opt_FW_away(f.H, t["ky_x0"], 1e-8, 1000, verbose=False)
    close(F, t["dfwa_ky_F"], 1e-9); close(SP, t["dfwa_ky_SP"], 1e-7)


@pytest.mark.parametrize("away", [0, 1])
@pytest.mark.parametrize("m,n,seed,its", [(80, 200, 10, 400), (30, 1000, 3, 500), (13, 506, 0, 300), (24, 1001, 6, 300)])
def test_fw_vertex_indices_bit_exact(acc, golden_ops, away, m, n, seed, its):
    if seed == 0:
        V = golden_ops["housing_H"]
    else:
        np.random.seed(seed)
        V = np.random.randn(m, n)
    x0 = np.ones(n) / n
    log_o, log_g = [], []
    fo = orc.D_opt_FW_away if away else orc.D_opt_FW
    fg = acc.D_opt_FW_away if away else acc.D_opt_FW
    xo, Fo, SPo, SNo, To = fo(V, x0, 1e-9, its, index_log=log_o)
    xg, Fg, SPg, SNg, Tg = fg(V, x0, 1e-9, its, verbose=False, index_log=log_g)
    assert len(log_g) == len(log_o)
    assert [p[0] for p in log_g] == [p[0] for p in log_o]          # argmax vertex i
    assert [p[1] for p in log_g] == [p[1] for p in log_o]          # (masked) argmin vertex j
    if away:
        assert [p[2] for p in log_g[:-1]] == [int(p[2]) for p in log_o[:-1]]   # toward / away decisions
    close(Fg, Fo, 1e-9)
    close(xg, xo, 1e-6, floor=1e-6)


def test_fw_stops_like_reference(acc):
    np.random.seed(4)
    V = np.random.randn(10, 40)
    x0 = np.ones(40) / 40
    a = acc.D_opt_FW_away(V, x0, 1e-3, 5000, verbose=False, batch=16)
    b = orc.D_opt_FW_away(V, x0, 1e-3, 5000)
    assert a[1].shape == b[1].shape and a[1].shape[0] < 5000
    close(a[1], b[1], 1e-9)
    a = acc.D_opt_FW(V, x0, 1e-3, 5000, verbose=False, batch=7)
    b = orc.D_opt_FW(V, x0, 1e-3, 5000)
    assert a[1].shape == b[1].shape
    close(a[1], b[1], 1e-9)


def test_fw_midsize_vs_oracle(acc):
    np.random.seed(2)
    V = np.random.randn(200, 5000)
    x0 = np.ones(5000) / 5000
    a = acc.D_opt_FW_away(V, x0, 1e-8, 300, verbose=False)
    b = orc.D_opt_FW_away(V, x0, 1e-8, 300)
    close(a[1], b[1], 1e-9); close(a[2], b[2], 1e-7); close(a[3], b[3], 1e-7)


def test_ky_init_golden(acc, golden_traj):
    """D_opt_KYinit (applications.py:59-95) with the q^T V passes and the arg-extrema on the device: same support as
    the reference (x0 is a function of the chosen indices only), from a host matrix and from a CUDA tensor."""
    np.random.seed(10)
    H = np.random.randn(80, 200)
    np.random.seed(77)
    assert np.array_equal(acc.D_opt_KYinit(H), golden_traj["ky_x0"])
    np.random.seed(77)
    assert np.array_equal(acc.D_opt_KYinit(torch.tensor(H, device="cuda")), golden_traj["ky_x0"])
    assert np.array_equal(acc.D_opt_KYinit(H[:, :150]), np.ones(150) / 150)       # n <= 2m: uniform
    xa, Fa, SPa, SNa, Ta = acc.D_opt_FW_away(H, golden_traj["ky_x0"], 1e-8, 1000, verbose=False)
    n = min(len(Fa), len(golden_traj["dfwa_ky_F"]))
    assert np.max(np.abs(Fa[:n] - golden_traj["dfwa_ky_F"][:n]) / np.abs(golden_traj["dfwa_ky_F"][:n])) <= 1e-9


@pytest.mark.parametrize("away,world", [(1, 2), (0, 3), (1, 4)])
def test_sharded_fw_building_blocks_on_one_gpu(acc, away, world):
    """The column-sharded Frank-Wolfe loop emulated on one GPU: `world` slabs processed one after the other, records
    and the chosen column exchanged by hand exactly as the collectives would.  F, slacks and the vertex sequence must
    be those of the single-slab device loop (and of the oracle): the decision does not depend on the sharding."""
    from accbpg_and_fw_b200 import _native as nat
    from accbpg_and_fw_b200.dopt_fw import NCTRL, C_IMAX, C_JMIN, C_STOP, C_NITER
    lib = nat.lib
    rt = acc.Runtime.get()
    m, n, its = 12, 203, 60
    rng = np.random.RandomState(5)
    V = rng.randn(m, n)
    x0 = np.ones(n) / n
    offs = acc.ColumnShard.partition(n, world)
    dev = "cuda"
    Vs = [torch.tensor(np.ascontiguousarray(V[:, offs[r]:offs[r + 1]]), device=dev) for r in range(world)]
    xs = [torch.tensor(x0[offs[r]:offs[r + 1]].copy(), device=dev) for r in range(world)]
    nl = [offs[r + 1] - offs[r] for r in range(world)]
    wss = [torch.zeros(lib.accbpg_fw_workspace_bytes(m, nl[r]), dtype=torch.uint8, device=dev) for r in range(world)]
    M = torch.zeros(m, m, dtype=torch.float64, device=dev)
    Mr = torch.empty(m, m, dtype=torch.float64, device=dev)
    for r in range(world):
        nat.check(lib.accbpg_dopt_gram(rt.ctx, rt.stream, Vs[r].data_ptr(), m, nl[r], nl[r], xs[r].data_ptr(),
                                       wss[r].data_ptr(), Mr.data_ptr()))
        M += Mr
    Hinv = [torch.empty(m, m, dtype=torch.float64, device=dev) for _ in range(world)]
    ws_ = [torch.empty(nl[r], dtype=torch.float64, device=dev) for r in range(world)]
    ctrl = [torch.zeros(NCTRL, dtype=torch.float64, device=dev) for _ in range(world)]
    hist = [torch.zeros(4, its, dtype=torch.float64, device=dev) for _ in range(world)]
    rd = lib.accbpg_fw_record_bytes() // 8
    recs = torch.zeros(world * rd, dtype=torch.float64, device=dev)
    vcols = [torch.zeros(m, dtype=torch.float64, device=dev) for _ in range(world)]
    for r in range(world):
        nat.check(lib.accbpg_fw_setup_from_gram(rt.ctx, rt.stream, Vs[r].data_ptr(), m, nl[r], nl[r], M.data_ptr(),
                                                wss[r].data_ptr(), Hinv[r].data_ptr(), ws_[r].data_ptr(), ctrl[r].data_ptr()))
        nat.check(lib.accbpg_fw_select_local(rt.ctx, rt.stream, nl[r], offs[r], away, xs[r].data_ptr(), ws_[r].data_ptr(),
                                             wss[r].data_ptr(), m, recs[r * rd:].data_ptr()))
    log = []
    for k in range(its):
        for r in range(world):
            h = hist[r]
            nat.check(lib.accbpg_fw_decide(rt.ctx, rt.stream, Vs[r].data_ptr(), m, nl[r], nl[r], offs[r], away, 1e-9, k,
                                           recs.data_ptr(), world, wss[r].data_ptr(), ctrl[r].data_ptr(), h[0].data_ptr(),
                                           h[1].data_ptr(), h[2].data_ptr(), h[3].data_ptr(), vcols[r].data_ptr()))
        vsum = sum(vcols)                                   # the all-reduce
        c0 = ctrl[0].cpu().numpy()
        if c0[C_STOP] != 0:
            break
        log.append((int(c0[C_IMAX]), int(c0[C_JMIN])))
        new = torch.zeros_like(recs)
        for r in range(world):
            vr = vsum.clone()
            nat.check(lib.accbpg_fw_step(rt.ctx, rt.stream, Vs[r].data_ptr(), m, nl[r], nl[r], offs[r], away, k,
                                         wss[r].data_ptr(), Hinv[r].data_ptr(), vr.data_ptr(), xs[r].data_ptr(),
                                         ws_[r].data_ptr(), ctrl[r].data_ptr(), new[r * rd:].data_ptr()))
        torch.cuda.synchronize()
        recs = new                                          # the all-gather
    done = int(ctrl[0].cpu().numpy()[C_NITER])
    F = hist[0][0, :done].cpu().numpy()
    fn = orc.D_opt_FW_away if away else orc.D_opt_FW
    olog = []
    xo, Fo, SPo, SNo, To = fn(V, x0, 1e-9, its, index_log=olog)
    nn = min(len(F), len(Fo))
    assert nn >= its - 1
    assert np.max(np.abs(F[:nn] - Fo[:nn]) / np.maximum(np.abs(Fo[:nn]), 1e-3)) <= 1e-9
    assert [(a, b) for a, b in log[:nn - 1]] == [(a, b) for a, b, *_ in olog[:nn - 1]]
    xfull = np.concatenate([t.cpu().numpy() for t in xs])
    assert np.max(np.abs(xfull - xo)) <= 1e-9
    for r in range(1, world):                               # replicated state stays identical
        assert torch.equal(ctrl[r][:15], ctrl[0][:15]) and torch.equal(Hinv[r], Hinv[0])


def _fw_loop(acc, V, start, away, eps, its, batch):
    """The batches of D_opt_FW (away = 0) / D_opt_FW_away (away = 1) as dopt_fw drives them, on V as given, from a copy
    of the set-up state `start` = (workspace, x, Hinv, w, ctrl).  Returns ((history length, sha256 of x, F, SP, SN),
    kernels the loop launched)."""
    from accbpg_and_fw_b200 import _native as nat
    from accbpg_and_fw_b200.dopt_fw import C_NITER, C_STOP
    lib, rt = nat.lib, acc.Runtime.get()
    m, n = V.shape
    ws = start[0]
    x, Hinv, w, ctrl = (t.clone() for t in start[1:])
    hist = torch.zeros(4, its, dtype=torch.float64, device="cuda")
    before = nat.launch_count()
    k = 0
    while k < its:
        cnt = min(batch, its - k)
        nat.check(lib.accbpg_fw_run(rt.ctx, rt.stream, V.data_ptr(), m, n, n, away, eps, k, cnt, ws.data_ptr(),
                                    Hinv.data_ptr(), x.data_ptr(), w.data_ptr(), ctrl.data_ptr(), hist[0].data_ptr(),
                                    hist[1].data_ptr(), hist[2].data_ptr(), hist[3].data_ptr()))
        k += cnt
        if ctrl.cpu().numpy()[C_STOP] != 0:
            break
    launches = nat.launch_count() - before
    done = int(ctrl.cpu().numpy()[C_NITER])
    h = hashlib.sha256()
    for a in (x, hist[0, :done], hist[1, :done], hist[2, :done]):
        h.update(a.cpu().numpy().tobytes())
    return (done, h.hexdigest()), launches


def test_fw_paths_bit_identical(acc):
    """The two forms of the loop, each reached by its input, give the same bits (iterates, histories, stopping
    iteration) from the same set-up state.  m <= 4096: V contiguous runs the ring-fed persistent launch (one 3-D tensor
    copy per stage when 4 | m, four 2-D copies otherwise), the same values 8 bytes into a buffer (not 16-byte aligned)
    run the launch chain with the scalar-load pass.  m > 4096: V contiguous runs the launch chain with the vector-load
    pass and its early fetch, the offset copy the chain with the scalar-load pass."""
    from accbpg_and_fw_b200 import _native as nat
    from accbpg_and_fw_b200.dopt_fw import NCTRL
    lib, rt = nat.lib, acc.Runtime.get()
    for (m, n, seed, eps, its, batch) in [(200, 5000, 2, 1e-8, 200, 64), (64, 3000, 5, 1e-2, 4000, 32),
                                          (10, 40, 4, 1e-3, 5000, 16), (4100, 4200, 7, 1e-12, 40, 16)]:
        np.random.seed(seed)
        V = np.random.randn(m, n)
        Va = torch.tensor(V, device="cuda")
        buf = torch.empty(m * n + 1, dtype=torch.float64, device="cuda")
        Vo = buf[1:].view(m, n)
        Vo.copy_(Va)
        assert Va.data_ptr() % 16 == 0 and Vo.data_ptr() % 16 == 8 and Vo.is_contiguous()
        ws = torch.zeros(lib.accbpg_fw_workspace_bytes(m, n), dtype=torch.uint8, device="cuda")
        x = torch.full((n,), 1.0 / n, dtype=torch.float64, device="cuda")
        Hinv = torch.empty(m, m, dtype=torch.float64, device="cuda")
        w = torch.empty(n, dtype=torch.float64, device="cuda")
        ctrl = torch.zeros(NCTRL, dtype=torch.float64, device="cuda")
        nat.check(lib.accbpg_fw_setup(rt.ctx, rt.stream, Va.data_ptr(), m, n, n, x.data_ptr(), ws.data_ptr(),
                                      Hinv.data_ptr(), w.data_ptr(), ctrl.data_ptr()))
        rt.read(0, 0)
        start = (ws, x, Hinv, w, ctrl)
        for away in (1, 0):
            aligned, launches_aligned = _fw_loop(acc, Va, start, away, eps, its, batch)
            offset, launches_offset = _fw_loop(acc, Vo, start, away, eps, its, batch)
            assert aligned == offset, (m, n, away, aligned, offset)
            done = aligned[0]
            assert launches_offset >= 2 * done                          # the launch chain: two launches per iteration
            if m <= 4096:
                assert launches_offset - launches_aligned >= 2 * done   # the persistent loop: one launch per batch
            else:
                assert launches_aligned == launches_offset
