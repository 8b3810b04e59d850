"""GPU-resident drop-ins for the Legendre kernels of accbpg/functions.py:199-490.

Burg entropy (plain, L1, L2, simplex) and Shannon entropy (plain, L1, simplex): value, gradient,
Bregman divergence, prox_map and div_prox_map, with the reference's names, arguments, defaults
and assertion behaviour.  NumPy in -> NumPy / float out, CUDA tensor in -> CUDA tensor out.
The `_enq_*` methods are the asynchronous device-level forms the drivers use.
"""
import torch

from . import _native as nat
from .runtime import Runtime, is_host, like_input

lib = nat.lib
_BURG_PLAIN = nat.MACROS["ACCBPG_BURG_PLAIN"]
_BURG_L1 = nat.MACROS["ACCBPG_BURG_L1"]
_BURG_L2 = nat.MACROS["ACCBPG_BURG_L2"]


class LegendreFunction:
    """Protocol of accbpg/functions.py:199-235 plus the shared host<->device plumbing."""
    has_psi = False

    def _setup(self, shard=None, device=None):
        self._device = device
        self._rt = None
        self.shard = shard

    @property
    def rt(self):
        if self._rt is None:
            self._rt = Runtime.get(self._device)
        return self._rt

    _defer_reduce = False      # set by the drivers: partial scalars are summed over the ranks once per fetch

    def _reduce(self, slot, count=1):
        if self._defer_reduce and slot < self.rt.S_TMP:
            return
        if self.shard is not None and self.shard.world > 1:
            self.shard.sum_(self.rt.scal[slot:slot + count])

    # ---- synchronous, reference-shaped API -------------------------------------------------
    def __call__(self, x):
        rt = self.rt
        self._enq_value(rt.to_device(x), rt.S_TMP)
        return rt.read(rt.S_TMP, 1)[0]

    def extra_Psi(self, x):
        if not self.has_psi:
            return 0
        rt = self.rt
        self._enq_extra_psi(rt.to_device(x), rt.S_TMP)
        return rt.read(rt.S_TMP, 1)[0]

    def gradient(self, x):
        rt = self.rt
        host = is_host(x)
        xd = rt.to_device(x)
        out = rt.empty(xd.numel())
        self._enq_gradient(xd, out)
        rt.read(rt.S_TMP, 0)                       # surface the positivity assertion
        return like_input(out, host)

    def divergence(self, x, y):
        rt = self.rt
        xd, yd = rt.to_device(x), rt.to_device(y)
        assert xd.shape == yd.shape, "Vectors x and y are of different sizes."
        self._enq_divergence(xd, yd, rt.S_TMP)
        return rt.read(rt.S_TMP, 1)[0]

    def prox_map(self, g, L):
        rt = self.rt
        host = is_host(g)
        gd = rt.to_device(g)
        out = rt.empty(gd.numel())
        self._enq_prox(gd, float(L), out)
        rt.read(rt.S_TMP, 0)
        return like_input(out, host)

    def div_prox_map(self, y, g, L):
        rt = self.rt
        host = is_host(g)
        yd, gd = rt.to_device(y), rt.to_device(g)
        assert yd.shape == gd.shape, "Vectors y and g are of different sizes."
        assert L > 0, "Relative smoothness constant L should be positive."
        out = rt.empty(gd.numel())
        self._enq_div_prox(yd, gd, float(L), out)
        rt.read(rt.S_TMP, 0)
        return like_input(out, host)

    # ---- default Bregman step: prox_map(g - L*grad h(y), L)     functions.py:228-235 ----------
    def _enq_div_prox(self, yd, gd, L, out):
        rt = self.rt
        tmp = rt.empty(yd.numel())
        self._enq_gradient(yd, tmp)
        nat.check(lib.accbpg_vec_axpby(rt.ctx, rt.stream, yd.numel(), 1.0, gd.data_ptr(), -L, tmp.data_ptr(),
                                       tmp.data_ptr()))
        self._enq_prox(tmp, L, out)


# ------------------------------------------------------------------------------------------------
class BurgEntropy(LegendreFunction):
    """h(x) = -sum log x, x > 0.   accbpg/functions.py:238-271."""
    _kind = _BURG_PLAIN
    lamda = 0.0

    def __init__(self, shard=None, device=None):
        self._setup(shard, device)

    def _enq_value(self, xd, slot):
        rt = self.rt
        nat.check(lib.accbpg_burg_value(rt.ctx, rt.stream, xd.numel(), xd.data_ptr(), rt.slot(slot)))
        self._reduce(slot)

    def _enq_gradient(self, xd, out):
        rt = self.rt
        nat.check(lib.accbpg_burg_gradient(rt.ctx, rt.stream, xd.numel(), xd.data_ptr(), out.data_ptr()))

    def _enq_divergence(self, xd, yd, slot):
        rt = self.rt
        nat.check(lib.accbpg_burg_divergence(rt.ctx, rt.stream, xd.numel(), xd.data_ptr(), yd.data_ptr(),
                                             rt.slot(slot)))
        self._reduce(slot)

    def _enq_prox(self, gd, L, out):
        assert L > 0, "BurgEntropy prox_map only takes positive L value."
        rt = self.rt
        nat.check(lib.accbpg_burg_prox(rt.ctx, rt.stream, gd.numel(), self._kind, float(self.lamda), None,
                                       gd.data_ptr(), L, out.data_ptr()))

    def _enq_div_prox(self, yd, gd, L, out):
        """prox_map(g - L*(-1/y), L) fused in one pass.   functions.py:264-271."""
        assert L > 0, "Either y or L is not positive."
        rt = self.rt
        nat.check(lib.accbpg_burg_prox(rt.ctx, rt.stream, gd.numel(), self._kind, float(self.lamda), yd.data_ptr(),
                                       gd.data_ptr(), L, out.data_ptr()))


class BurgEntropyL1(BurgEntropy):
    """Burg kernel for min f(x) + lamda*||x||_1.   accbpg/functions.py:274-298."""
    _kind = _BURG_L1
    has_psi = True

    def __init__(self, lamda=0, x_max=1e4, shard=None, device=None):
        assert lamda >= 0, "BurgEntropyL1: lambda should be nonnegative."
        self._setup(shard, device)
        self.lamda = lamda
        self.x_max = x_max

    def _enq_extra_psi(self, xd, slot):       # lamda * x.sum()
        rt = self.rt
        nat.check(lib.accbpg_vec_sum(rt.ctx, rt.stream, xd.numel(), xd.data_ptr(), rt.slot(slot)))
        self._reduce(slot)
        rt.scal[slot:slot + 1].mul_(float(self.lamda))


class BurgEntropyL2(BurgEntropy):
    """Burg kernel for min f(x) + (lamda/2)*||x||_2^2.   accbpg/functions.py:301-323."""
    _kind = _BURG_L2
    has_psi = True

    def __init__(self, lamda=0, shard=None, device=None):
        assert lamda >= 0, "BurgEntropyL2: lamda should be nonnegative."
        self._setup(shard, device)
        self.lamda = lamda

    def _enq_extra_psi(self, xd, slot):       # (lamda/2) * dot(x, x)
        rt = self.rt
        nat.check(lib.accbpg_vec_dot(rt.ctx, rt.stream, xd.numel(), xd.data_ptr(), xd.data_ptr(), rt.slot(slot)))
        self._reduce(slot)
        rt.scal[slot:slot + 1].mul_(float(self.lamda) / 2)


class BurgEntropySimplex(BurgEntropy):
    """Burg kernel on the unit simplex; prox by a Newton root-find.   accbpg/functions.py:326-356."""

    def __init__(self, eps=1e-8, shard=None, device=None):
        assert eps > 0, "BurgEntropySimplex: eps should be positive."
        self._setup(shard, device)
        self.eps = eps
        self.last_info = None          # device tensor [bisections, newton steps, c] of the last call

    def _enq_prox(self, gd, L, out):
        self._simplex(None, gd, L, out)

    def _enq_div_prox(self, yd, gd, L, out):
        self._simplex(yd, gd, L, out)

    def _simplex(self, yd, gd, L, out):
        assert L > 0, "BergEntropySimplex prox_map only takes positive L."
        rt = self.rt
        n = gd.numel()
        yp = yd.data_ptr() if yd is not None else None
        if self.shard is None or self.shard.world == 1:
            info = rt.slot(rt.S_AUX1)
            nat.check(lib.accbpg_burg_simplex_prox(rt.ctx, rt.stream, n, yp, gd.data_ptr(), L, float(self.eps),
                                                   out.data_ptr(), info))
            return
        # column-sharded: every rank gathers all slices of gg = (g [+ L/y]) / L (padding +inf) - pushed straight into every
        # rank's gathered vector over NVLink peer memory, else an NCCL all-gather - and replays the whole recurrence on
        # the gathered vector, so there is ONE exchange per prox call, no host round trip, and the multiplier c is
        # bit-identical on every rank (and independent of the sharding).
        sh = self.shard
        key = (n, sh.width, sh.world)
        if getattr(self, "_gg_key", None) != key:
            from .dist import peer_buffers
            self._gg_key = key
            self._gg_loc = torch.full((sh.width,), float("inf"), dtype=torch.float64, device=rt.device)
            self._gg_all = torch.empty(sh.width * sh.world, dtype=torch.float64, device=rt.device)
            # gathered vector in NVLink peer memory (double-buffered) + one flag word per rank; None -> NCCL all-gather
            self._gg_peer = peer_buffers(sh, rt.device, [(2 * sh.world * sh.width, torch.float64),
                                                         (sh.world, torch.int64)],
                                         cache_key=("burg_gg", sh.width), reset=False)
        info = rt.slot(rt.S_AUX1)
        gg = self._gg_loc
        if self._gg_peer is not None:
            pb = self._gg_peer
            ep = pb.next_epoch()
            nat.check(lib.accbpg_burg_simplex_push_peer(rt.ctx, rt.stream, n, sh.width, yp, gd.data_ptr(), L, sh.rank,
                                                        sh.world, pb.tables[0], pb.tables[1], ep, gg.data_ptr()))
            nat.check(lib.accbpg_burg_simplex_root_peer(rt.ctx, rt.stream, sh.width, float(self.eps), sh.rank, sh.world,
                                                        pb.tables[0], pb.tables[1], ep, info))
            nat.check(lib.accbpg_burg_simplex_finish_dev(rt.ctx, rt.stream, n, gg.data_ptr(), info + 16,
                                                         out.data_ptr()))
            return
        s0 = rt.S_TMP + 8
        nat.check(lib.accbpg_burg_simplex_prepare(rt.ctx, rt.stream, n, yp, gd.data_ptr(), L, gg.data_ptr(),
                                                  rt.slot(s0)))
        sh.all_gather_equal(self._gg_all, gg)
        nat.check(lib.accbpg_burg_simplex_root(rt.ctx, rt.stream, sh.width * sh.world, self._gg_all.data_ptr(),
                                               float(self.eps), info))
        nat.check(lib.accbpg_burg_simplex_finish_dev(rt.ctx, rt.stream, n, gg.data_ptr(), info + 16, out.data_ptr()))


# ------------------------------------------------------------------------------------------------
class ShannonEntropy(LegendreFunction):
    """h(x) = sum x log x, x >= 0.   accbpg/functions.py:398-438."""
    lamda = 0.0
    _normalize = 0

    def __init__(self, delta=1e-20, shard=None, device=None):
        self._setup(shard, device)
        self.delta = delta

    def _enq_value(self, xd, slot):
        rt = self.rt
        nat.check(lib.accbpg_shannon_value(rt.ctx, rt.stream, xd.numel(), xd.data_ptr(), float(self.delta),
                                           rt.slot(slot)))
        self._reduce(slot)

    def _enq_gradient(self, xd, out):
        rt = self.rt
        nat.check(lib.accbpg_shannon_gradient(rt.ctx, rt.stream, xd.numel(), xd.data_ptr(), float(self.delta),
                                              out.data_ptr()))

    def _enq_divergence(self, xd, yd, slot):
        rt = self.rt
        if self.shard is None or self.shard.world == 1:
            nat.check(lib.accbpg_shannon_divergence(rt.ctx, rt.stream, xd.numel(), xd.data_ptr(), yd.data_ptr(),
                                                    float(self.delta), rt.slot(slot)))
            return
        # sum x log(..) + (sum y - sum x) is linear in the per-rank partial triples: reduce the local value
        nat.check(lib.accbpg_shannon_divergence(rt.ctx, rt.stream, xd.numel(), xd.data_ptr(), yd.data_ptr(),
                                                float(self.delta), rt.slot(slot)))
        self._reduce(slot)

    def _point(self, yd, gd, L, out):
        assert L > 0, "ShannonEntropy prox_map require L > 0."
        rt = self.rt
        n = gd.numel()
        yp = yd.data_ptr() if yd is not None else None
        sharded = self.shard is not None and self.shard.world > 1
        if not self._normalize or not sharded:
            nat.check(lib.accbpg_shannon_prox(rt.ctx, rt.stream, n, float(self.lamda), yp, gd.data_ptr(), L,
                                              self._normalize, out.data_ptr(), rt.slot(rt.S_AUX2)))
            return
        s0 = rt.S_TMP + 8
        nat.check(lib.accbpg_shannon_prox(rt.ctx, rt.stream, n, float(self.lamda), yp, gd.data_ptr(), L, 2,
                                          out.data_ptr(), rt.slot(s0)))
        self.shard.sum_(rt.scal[s0:s0 + 1])
        total = rt.read(s0, 1)[0]
        nat.check(lib.accbpg_vec_divide(rt.ctx, rt.stream, n, out.data_ptr(), total, out.data_ptr()))

    def _enq_prox(self, gd, L, out):
        self._point(None, gd, L, out)

    def _enq_div_prox(self, yd, gd, L, out):
        self._point(yd, gd, L, out)


class ShannonEntropyL1(ShannonEntropy):
    """Shannon kernel for min f(x) + lamda*||x||_1.   accbpg/functions.py:441-466."""
    has_psi = True

    def __init__(self, lamda=0, delta=1e-20, shard=None, device=None):
        ShannonEntropy.__init__(self, delta, shard, device)
        self.lamda = lamda

    def _enq_extra_psi(self, xd, slot):
        rt = self.rt
        nat.check(lib.accbpg_vec_sum(rt.ctx, rt.stream, xd.numel(), xd.data_ptr(), rt.slot(slot)))
        self._reduce(slot)
        rt.scal[slot:slot + 1].mul_(float(self.lamda))


class ShannonEntropySimplex(ShannonEntropy):
    """Shannon kernel on the unit simplex (normalised multiplicative update).   functions.py:469-490."""
    _normalize = 1


# ------------------------------------------------------------------------------------------------
class SquaredL2Norm(LegendreFunction):
    """h(x) = (1/2)||x||_2^2.   accbpg/functions.py:738-759 (the kernel the Euclidean Frank-Wolfe examples pass)."""

    def __init__(self, shard=None, device=None):
        self._setup(shard, device)

    def _enq_value(self, xd, slot):
        rt = self.rt
        nat.check(lib.accbpg_vec_dot(rt.ctx, rt.stream, xd.numel(), xd.data_ptr(), xd.data_ptr(), rt.slot(slot)))
        self._reduce(slot)
        rt.scal[slot:slot + 1].mul_(0.5)

    def gradient(self, x):
        return x if is_host(x) else x.clone()

    def _enq_gradient(self, xd, out):
        out.copy_(xd)

    def _enq_divergence(self, xd, yd, slot):
        rt = self.rt
        nat.check(lib.accbpg_vec_sqdist(rt.ctx, rt.stream, xd.numel(), xd.data_ptr(), yd.data_ptr(), rt.slot(slot)))
        self._reduce(slot)
        rt.scal[slot:slot + 1].mul_(0.5)

    def _enq_prox(self, gd, L, out):                 # -(1/L) g
        assert L > 0, "SquaredL2Norm: L should be positive."
        rt = self.rt
        nat.check(lib.accbpg_vec_axpby(rt.ctx, rt.stream, gd.numel(), -(1 / L), gd.data_ptr(), 0.0, gd.data_ptr(),
                                       out.data_ptr()))

    def _enq_div_prox(self, yd, gd, L, out):         # y - (1/L) g
        assert L > 0, "Vectors y and g not same shape."
        rt = self.rt
        nat.check(lib.accbpg_vec_axpby(rt.ctx, rt.stream, gd.numel(), 1.0, yd.data_ptr(), -(1 / L), gd.data_ptr(),
                                       out.data_ptr()))
