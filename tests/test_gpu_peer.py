"""GPU (one device): the NVLink peer-memory exchanges of the column-sharded path, driven through the C ABI with TWO
ranks emulated on one GPU - each "rank" has its own context, stream, workspace and receive buffers; the pointer tables
a real run fills from symmetric memory simply point at both sets.  Small m keeps the waiting kernels to a few CTAs so the
other rank's kernels always find room (on separate GPUs there is no such constraint).  The multi-process version of the
same checks is tests/multigpu_check.py (needs >= 2 GPUs)."""
import ctypes

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
F64 = torch.float64


@pytest.fixture(scope="module")
def acc():
    import accbpg_and_fw_b200 as a
    return a


class _Rank:
    def __init__(self, nat):
        self.nat = nat
        h = ctypes.c_void_p()
        nat.check(nat.lib.accbpg_ctx_create(ctypes.byref(h)))
        self.ctx = h
        self.stream = torch.cuda.Stream()

    def close(self):
        self.nat.check(self.nat.lib.accbpg_ctx_destroy(self.ctx))


def _table(tensors):
    return (ctypes.c_void_p * len(tensors))(*[t.data_ptr() for t in tensors])


@pytest.mark.parametrize("m,widths", [(96, (700, 500)), (33, (64, 130)), (128, (1024, 1024))])
def test_gram_allreduce_over_peer_buffers_two_emulated_ranks(acc, m, widths):
    from accbpg_and_fw_b200 import _native as nat
    lib = nat.lib
    dev = torch.device("cuda")
    world = 2
    gen = torch.Generator(device=dev)
    gen.manual_seed(7 + m)
    H = [torch.randn(m, w, dtype=F64, device=dev, generator=gen) for w in widths]
    ranks = [_Rank(nat) for _ in range(world)]
    try:
        recv = [torch.zeros(2 * world * m * m, dtype=F64, device=dev) for _ in range(world)]
        flags = [torch.zeros(world, dtype=torch.int64, device=dev) for _ in range(world)]
        ws = [torch.zeros(lib.accbpg_dopt_workspace_bytes(m, w), dtype=torch.uint8, device=dev) for w in widths]
        M = [torch.empty(m, m, dtype=F64, device=dev) for _ in range(world)]
        t_recv, t_flags = _table(recv), _table(flags)
        torch.cuda.synchronize()
        for epoch in range(1, 6):                           # several calls: flag epochs and the parity double buffer
            x = [torch.rand(w, dtype=F64, device=dev, generator=gen) + 0.01 * epoch for w in widths]
            torch.cuda.synchronize()
            for r in range(world):
                nat.check(lib.accbpg_dopt_gram_allreduce(
                    ranks[r].ctx, ranks[r].stream.cuda_stream, H[r].data_ptr(), m, widths[r], H[r].stride(0),
                    x[r].data_ptr(), ws[r].data_ptr(), r, world, t_recv, t_flags, epoch, M[r].data_ptr()))
            torch.cuda.synchronize()
            assert torch.equal(M[0], M[1])                  # every rank sums the same numbers in the same order
            ref = sum((H[r] * x[r]) @ H[r].T for r in range(world))
            err = float(((M[0] - ref).abs().max() / ref.abs().max()).item())
            assert err <= 1e-13, (epoch, err)
            assert torch.equal(M[0], M[0].T)
        assert [int(v) for v in flags[0].tolist()] == [5, 5] and [int(v) for v in flags[1].tolist()] == [5, 5]
    finally:
        torch.cuda.synchronize()
        for rk in ranks:
            rk.close()


@pytest.mark.parametrize("away", [1, 0])
def test_fw_loop_over_peer_buffers_two_emulated_ranks(acc, away):
    """accbpg_fw_run_peer on two emulated ranks against the single-device loop on the same instance: identical decisions
    (history entries equal on both ranks), F / slacks equal to rounding, the gathered iterate equal."""
    from accbpg_and_fw_b200 import _native as nat
    lib = nat.lib
    dev = torch.device("cuda")
    m, n, its, world = 40, 3000, 150, 2
    np.random.seed(5)
    V = np.random.randn(m, n)
    x0 = np.ones(n) / n
    fn = acc.D_opt_FW_away if away else acc.D_opt_FW
    xs, Fs, SPs, SNs, Ts = fn(V, x0, 1e-9, its, verbose=False, batch=50)
    bounds = [0, 1300, n]
    rec_d = lib.accbpg_fw_record_bytes() // 8
    ranks = [_Rank(nat) for _ in range(world)]
    try:
        Vd = [torch.tensor(np.ascontiguousarray(V[:, bounds[r]:bounds[r + 1]]), device=dev) for r in range(world)]
        xd = [torch.tensor(x0[bounds[r]:bounds[r + 1]], device=dev) for r in range(world)]
        Mtot = torch.tensor((V * x0) @ V.T, device=dev)
        rec = [torch.zeros(2 * world * rec_d, dtype=F64, device=dev) for _ in range(world)]
        col = [torch.zeros(2 * m, dtype=F64, device=dev) for _ in range(world)]
        flags = [torch.zeros(world + 1, dtype=torch.int64, device=dev) for _ in range(world)]
        t_rec, t_col, t_flags = _table(rec), _table(col), _table(flags)
        st = []
        for r in range(world):
            nl = bounds[r + 1] - bounds[r]
            d = {"ws": torch.zeros(lib.accbpg_fw_workspace_bytes(m, nl), dtype=torch.uint8, device=dev),
                 "Hinv": torch.empty(m, m, dtype=F64, device=dev), "w": torch.empty(nl, dtype=F64, device=dev),
                 "ctrl": torch.zeros(nat.MACROS["ACCBPG_FW_CTRL_DOUBLES"], dtype=F64, device=dev), "hist": torch.zeros(4, its, dtype=F64, device=dev)}
            nat.check(lib.accbpg_fw_setup_from_gram(ranks[r].ctx, ranks[r].stream.cuda_stream, Vd[r].data_ptr(), m, nl,
                                                    Vd[r].stride(0), Mtot.data_ptr(), d["ws"].data_ptr(),
                                                    d["Hinv"].data_ptr(), d["w"].data_ptr(), d["ctrl"].data_ptr()))
            st.append(d)
        torch.cuda.synchronize()
        for k0 in range(0, its, 50):                        # three batches: the records carry over between calls
            for r in range(world):
                nl = bounds[r + 1] - bounds[r]
                d = st[r]
                nat.check(lib.accbpg_fw_run_peer(
                    ranks[r].ctx, ranks[r].stream.cuda_stream, Vd[r].data_ptr(), m, nl, Vd[r].stride(0), bounds[r], away,
                    1e-9, k0, 50, r, world, t_rec, t_col, t_flags, d["ws"].data_ptr(), d["Hinv"].data_ptr(),
                    xd[r].data_ptr(), d["w"].data_ptr(), d["ctrl"].data_ptr(), d["hist"][0].data_ptr(),
                    d["hist"][1].data_ptr(), d["hist"][2].data_ptr(), d["hist"][3].data_ptr()))
            torch.cuda.synchronize()
        h0, h1 = st[0]["hist"].cpu().numpy(), st[1]["hist"].cpu().numpy()
        assert np.array_equal(h0[:3], h1[:3])               # replicated decisions: bit-identical histories
        assert torch.equal(st[0]["Hinv"], st[1]["Hinv"])
        nF = len(Fs)
        assert nF == its
        assert float(np.max(np.abs(h0[0, :nF] - Fs) / np.maximum(np.abs(Fs), 1e-3))) <= 1e-10
        assert float(np.max(np.abs(h0[1, :nF] - SPs))) <= 1e-9 and float(np.max(np.abs(h0[2, :nF] - SNs))) <= 1e-9
        xg = np.concatenate([t.cpu().numpy() for t in xd])
        assert float(np.max(np.abs(xg - xs))) <= 1e-12
    finally:
        torch.cuda.synchronize()
        for rk in ranks:
            rk.close()


@pytest.mark.parametrize("world", [2, 4, 8])
def test_scalar_sums_over_peer_buffers_emulated_ranks(acc, world):
    from accbpg_and_fw_b200 import _native as nat
    lib = nat.lib
    dev = torch.device("cuda")
    count = 4
    gen = torch.Generator(device=dev)
    gen.manual_seed(11)
    ranks = [_Rank(nat) for _ in range(world)]
    try:
        tab = [torch.zeros(2 * world * 16, dtype=F64, device=dev) for _ in range(world)]
        flags = [torch.zeros(world, dtype=torch.int64, device=dev) for _ in range(world)]
        t_tab, t_flags = _table(tab), _table(flags)
        for epoch in range(1, 8):
            parts = [torch.randn(count, dtype=F64, device=dev, generator=gen) * 10.0 ** (r % 3) for r in range(world)]
            vals = [torch.zeros(count, dtype=F64, device=dev) for _ in parts]
            torch.cuda.synchronize()
            if epoch == 3:
                # a precondition fails on the LAST rank's slice only (Burg divergence of a non-positive vector):
                # the exchange must hand its status bit to every rank
                bad = torch.tensor([-1.0, 1.0], dtype=F64, device=dev)
                with torch.cuda.stream(ranks[-1].stream):
                    nat.check(lib.accbpg_burg_divergence(ranks[-1].ctx, ranks[-1].stream.cuda_stream, 2, bad.data_ptr(),
                                                         bad.data_ptr(), parts[-1].data_ptr()))
                parts[-1].fill_(1.0)
                torch.cuda.synchronize()
            for r in range(world):
                nat.check(lib.accbpg_peer_sum_scalars(ranks[r].ctx, ranks[r].stream.cuda_stream, parts[r].data_ptr(),
                                                      vals[r].data_ptr(), count, r, world, t_tab, t_flags, epoch))
            torch.cuda.synchronize()
            ref = np.zeros(count)
            for r in range(world):                           # rank order, as the kernel adds them
                ref = ref + parts[r].cpu().numpy()
            hb = (ctypes.c_double * 4)()
            for r in range(world):
                assert np.array_equal(vals[r].cpu().numpy(), ref), (epoch, r)
                st = ctypes.c_uint32(0)
                nat.check(lib.accbpg_ctx_read(ranks[r].ctx, ranks[r].stream.cuda_stream, None, 0, None, ctypes.byref(st)))
                assert st.value == (nat.ST["ARG_NOT_POS"] if epoch == 3 else 0), (epoch, r, st.value)
    finally:
        torch.cuda.synchronize()
        for rk in ranks:
            rk.close()


@pytest.mark.parametrize("world,n", [(2, 1000), (3, 1499), (8, 4001)])
def test_burg_simplex_prox_gather_over_peer_buffers_emulated_ranks(acc, world, n):
    """prepare + push, root-find on the gathered vector, finishing map: the multiplier is bit-identical on every rank
    and the assembled prox equals the oracle's BurgEntropySimplex.div_prox_map on the whole vector."""
    from accbpg_and_fw_b200 import _native as nat
    from oracle import accbpg_oracle as orc
    lib = nat.lib
    dev = torch.device("cuda")
    rng = np.random.RandomState(3 + world)
    sh = acc.ColumnShard(n, rank=0, world=world)
    width, off = sh.width, sh.offsets
    ho = orc.make_burg("simplex")
    ranks = [_Rank(nat) for _ in range(world)]
    try:
        ggbuf = [torch.zeros(2 * world * width, dtype=F64, device=dev) for _ in range(world)]
        flags = [torch.zeros(world, dtype=torch.int64, device=dev) for _ in range(world)]
        t_gg, t_flags = _table(ggbuf), _table(flags)
        for epoch in range(1, 5):
            y = rng.rand(n) + 0.05
            y /= y.sum()
            g = rng.randn(n)
            L = 0.5 + epoch
            yd = [torch.tensor(y[off[r]:off[r + 1]], device=dev) for r in range(world)]
            gd = [torch.tensor(g[off[r]:off[r + 1]], device=dev) for r in range(world)]
            loc = [torch.full((width,), float("inf"), dtype=F64, device=dev) for _ in range(world)]
            info = [torch.zeros(8, dtype=F64, device=dev) for _ in range(world)]
            out = [torch.empty(off[r + 1] - off[r], dtype=F64, device=dev) for r in range(world)]
            torch.cuda.synchronize()
            # all pushes first: cooperative launches of different streams are serialised against each other on ONE
            # device, so a root-find queued behind a waiting kernel would hold back the other "ranks"' pushes here
            # (on separate GPUs the two calls simply follow each other)
            for r in range(world):
                nl = off[r + 1] - off[r]
                nat.check(lib.accbpg_burg_simplex_push_peer(ranks[r].ctx, ranks[r].stream.cuda_stream, nl, width,
                                                            yd[r].data_ptr(), gd[r].data_ptr(), L, r, world, t_gg,
                                                            t_flags, epoch, loc[r].data_ptr()))
            for r in range(world):
                nl = off[r + 1] - off[r]
                st = ranks[r].stream.cuda_stream
                nat.check(lib.accbpg_burg_simplex_root_peer(ranks[r].ctx, st, width, 1e-8, r, world, t_gg, t_flags, epoch,
                                                            info[r].data_ptr()))
                nat.check(lib.accbpg_burg_simplex_finish_dev(ranks[r].ctx, st, nl, loc[r].data_ptr(),
                                                             info[r].data_ptr() + 16, out[r].data_ptr()))
            torch.cuda.synchronize()
            cs = [float(i[2].item()) for i in info]
            assert len(set(cs)) == 1, cs
            x = np.concatenate([o.cpu().numpy() for o in out])
            xo = ho.div_prox_map(y, g, L)
            assert float(np.max(np.abs(x - xo) / np.abs(xo))) <= 1e-10
            assert abs(x.sum() - 1.0) <= 2e-8
    finally:
        torch.cuda.synchronize()
        for rk in ranks:
            rk.close()


@pytest.mark.parametrize("world,n", [(2, 17), (4, 1000), (8, 100000)])
def test_vector_sum_over_peer_buffers_emulated_ranks(acc, world, n):
    from accbpg_and_fw_b200 import _native as nat
    lib = nat.lib
    dev = torch.device("cuda")
    cap = 1 << (n - 1).bit_length()
    gen = torch.Generator(device=dev)
    gen.manual_seed(13)
    ranks = [_Rank(nat) for _ in range(world)]
    try:
        buf = [torch.zeros(2 * world * cap, dtype=F64, device=dev) for _ in range(world)]
        flags = [torch.zeros(world, dtype=torch.int64, device=dev) for _ in range(world)]
        t_buf, t_flags = _table(buf), _table(flags)
        for epoch in range(1, 5):
            parts = [torch.randn(n, dtype=F64, device=dev, generator=gen) for _ in range(world)]
            vals = [p.clone() for p in parts]
            torch.cuda.synchronize()
            for r in range(world):
                nat.check(lib.accbpg_peer_sum_vector(ranks[r].ctx, ranks[r].stream.cuda_stream, vals[r].data_ptr(), n, cap,
                                                     r, world, t_buf, t_flags, epoch))
            torch.cuda.synchronize()
            ref = torch.zeros(n, dtype=F64, device=dev)
            for r in range(world):                           # rank order, as the kernel adds them
                ref = ref + parts[r]
            for r in range(world):
                assert torch.equal(vals[r], ref), (epoch, r)
    finally:
        torch.cuda.synchronize()
        for rk in ranks:
            rk.close()


def test_argmin_pair_over_peer_buffers_lowest_index_wins(acc):
    from accbpg_and_fw_b200 import _native as nat
    lib = nat.lib
    dev = torch.device("cuda")
    world = 4
    ranks = [_Rank(nat) for _ in range(world)]
    try:
        tab = [torch.zeros(2 * world * 16, dtype=F64, device=dev) for _ in range(world)]
        flags = [torch.zeros(world, dtype=torch.int64, device=dev) for _ in range(world)]
        t_tab, t_flags = _table(tab), _table(flags)
        cases = [([(0.5, 3.0), (0.25, 40.0), (0.25, 17.0), (0.9, 2.0)], (0.25, 17.0)),      # tie in the value
                 ([(-1.0, 9.0), (2.0, 1.0), (3.0, 0.0), (-1.0, 8.0)], (-1.0, 8.0)),
                 ([(7.0, 5.0), (7.0, 6.0), (7.0, 4.0), (7.0, 11.0)], (7.0, 4.0))]
        for epoch, (pairs, want) in enumerate(cases, start=1):
            vals = [torch.tensor(p, dtype=F64, device=dev) for p in pairs]
            torch.cuda.synchronize()
            for r in range(world):
                nat.check(lib.accbpg_peer_argmin_pair(ranks[r].ctx, ranks[r].stream.cuda_stream, vals[r].data_ptr(), r,
                                                      world, t_tab, t_flags, epoch))
            torch.cuda.synchronize()
            for r in range(world):
                assert tuple(vals[r].tolist()) == want, (epoch, r, vals[r].tolist())
    finally:
        torch.cuda.synchronize()
        for rk in ranks:
            rk.close()
