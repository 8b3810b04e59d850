"""GPU-resident drop-ins for the relatively-smooth objectives of accbpg/functions.py.

Same duck-typed protocol as the reference (`f(x)`, `f.gradient(x)`, `f.func_grad(x, flag)`,
attributes H / A / b / m / n); NumPy in -> NumPy / float out, CUDA tensor in -> CUDA tensor
out.  The `_enqueue*` methods are the asynchronous form the drivers in this package use:
they write scalars to runtime slots and never synchronise.

With `shard=ColumnShard(...)` the matrix passed in is this rank's column slab and vectors are
local slices; the m x m Gram matrix (D-opt) or the m-vector Ax (Poisson / KL) is all-reduced.
"""
import numpy as np
import torch

from . import _native as nat
from .runtime import Runtime, is_host, like_input

lib = nat.lib


class RSmoothFunction:
    """Protocol of accbpg/functions.py:10-24."""

    def __call__(self, x):
        return self.func_grad(x, flag=0)

    def gradient(self, x):
        return self.func_grad(x, flag=1)

    def func_grad(self, x, flag=2):
        assert flag in (0, 1, 2), "flag must be 0, 1 or 2"
        rt = self.rt
        host = is_host(x)
        xd = rt.to_device(x)
        assert xd.numel() == self.n_local, f"{type(self).__name__}: x.size not equal to n"
        g = rt.empty(self.n_local) if flag >= 1 else None
        self._enqueue(xd, flag, rt.S_TMP, g)
        fval = rt.read(rt.S_TMP, 1)[0]            # also surfaces x<0 / not-PD like the reference's checks
        if flag == 0:
            return fval
        gout = like_input(g, host)
        return gout if flag == 1 else (fval, gout)


class DOptimalObj(RSmoothFunction):
    """f(x) = -log det(H diag(x) H^T), H m x n with m < n.   accbpg/functions.py:27-59.

    K1 gram (DMMA SYRK) -> [all-reduce M] -> K2 Cholesky / log det -> K3 L^{-1} -> K4 gradient.
    """

    def __init__(self, H, shard=None, device=None):
        self.rt = Runtime.get(device)
        self.shard = shard
        self.H = H                                     # kept as given: notebooks pass f.H to D_opt_FW*
        self._Hd = self.rt.to_device(H)
        self.m, self.n_local = int(self._Hd.shape[0]), int(self._Hd.shape[1])
        self.n = shard.n if shard is not None else self.n_local
        assert self.m < self.n, "DOptimalObj: need m < n"
        with self.rt.on_device():                      # the plan depends on the device's SM count
            self._ws = self.rt.workspace(("dopt", self.m, self.n_local),
                                         lib.accbpg_dopt_workspace_bytes(self.m, self.n_local))
        self._peer = None
        if shard is not None and shard.world > 1:
            self._M = torch.empty(self.m, self.m, dtype=torch.float64, device=self.rt.device)
            self._setup_peer_memory()

    # ---- peer-memory all-reduce of the Gram matrix (config.peer_allreduce) ------------------------------------
    def _setup_peer_memory(self):
        """Symmetric buffers for accbpg_dopt_gram_allreduce: the receive slots for every rank's Gram matrix and the flag
        words, mapped into every peer (collective call: every rank constructs the objective)."""
        from .dist import peer_buffers
        mm = self.m * self.m
        self._peer = peer_buffers(self.shard, self.rt.device, [(2 * self.shard.world * mm, torch.float64),
                                                               (self.shard.world, torch.int64)])

    def _gram_sharded(self, xd, M):
        """M <- sum over ranks of H_r diag(x_r) H_r^T."""
        rt = self.rt
        H = self._Hd
        if self._peer is not None:
            pr = self._peer
            nat.check(lib.accbpg_dopt_gram_allreduce(rt.ctx, rt.stream, H.data_ptr(), self.m, self.n_local, H.stride(0),
                                                     xd.data_ptr(), self._ws.data_ptr(), self.shard.rank, self.shard.world,
                                                     pr.tables[0], pr.tables[1], pr.next_epoch(), M.data_ptr()))
            return
        nat.check(lib.accbpg_dopt_gram(rt.ctx, rt.stream, H.data_ptr(), self.m, self.n_local, H.stride(0),
                                       xd.data_ptr(), self._ws.data_ptr(), M.data_ptr()))
        self.shard.sum_(M)

    # ---- linear image M(x) = H diag(x) H^T (config.linear_images) ------------------------------------------
    _lin_capable = True

    def _img_compute(self, xd):
        """M(x) as a new m x m device tensor (K1 SYRK; all-reduced when H is column-sharded)."""
        rt = self.rt
        H = self._Hd
        M = torch.empty(self.m, self.m, dtype=torch.float64, device=rt.device)
        if self.shard is not None and self.shard.world > 1:
            self._gram_sharded(xd, M)
            return M
        nat.check(lib.accbpg_dopt_gram(rt.ctx, rt.stream, H.data_ptr(), self.m, self.n_local, H.stride(0),
                                       xd.data_ptr(), self._ws.data_ptr(), M.data_ptr()))
        return M

    def _img_axpby(self, a, Ia, b, Ib):
        rt = self.rt
        out = torch.empty_like(Ia)
        nat.check(lib.accbpg_vec_axpby(rt.ctx, rt.stream, Ia.numel(), float(a), Ia.data_ptr(), float(b),
                                       Ib.data_ptr(), out.data_ptr()))
        return out

    def _img_vertex(self, idx_slot, fill, radius):
        """M(s) for the simplex vertex s (fill everywhere, radius at the column whose global index sits in the device
        slot idx_slot) from H H^T of the local columns: no pass over H (accbpg_dopt_vertex_gram)."""
        rt = self.rt
        H = self._Hd
        if getattr(self, "_G1", None) is None:
            ones = torch.ones(self.n_local, dtype=torch.float64, device=rt.device)
            self._G1 = torch.empty(self.m, self.m, dtype=torch.float64, device=rt.device)
            nat.check(lib.accbpg_dopt_gram(rt.ctx, rt.stream, H.data_ptr(), self.m, self.n_local, H.stride(0),
                                           ones.data_ptr(), self._ws.data_ptr(), self._G1.data_ptr()))
        M = torch.empty(self.m, self.m, dtype=torch.float64, device=rt.device)
        off = self.shard.lo if self.shard is not None else 0
        nat.check(lib.accbpg_dopt_vertex_gram(rt.ctx, rt.stream, H.data_ptr(), self.m, self.n_local, H.stride(0),
                                              self._G1.data_ptr(), float(fill), rt.slot(idx_slot), off, float(radius),
                                              M.data_ptr()))
        if self.shard is not None and self.shard.world > 1:
            self.shard.sum_(M)
        return M

    def _enqueue_img_pair(self, Ix, slot_x, Iy, flag_y, slot_y, g):
        """f from M(x) -> slot_x (skipped when Ix is None) and (f, grad f) from M(y) -> (slot_y, g): K2-K4 only."""
        rt = self.rt
        H = self._Hd
        nat.check(lib.accbpg_dopt_pair_from_gram(
            rt.ctx, rt.stream, H.data_ptr(), self.m, self.n_local, H.stride(0),
            Ix.data_ptr() if Ix is not None else None, Iy.data_ptr(), flag_y, self._ws.data_ptr(),
            rt.slot(slot_x) if Ix is not None else None, rt.slot(slot_y), g.data_ptr() if g is not None else None))

    def _enqueue_pair(self, xd, slot_x, yd, flag_y, slot_y, g):
        """f(x) -> slot_x and (f(y), grad f(y)) -> (slot_y, g): what an accelerated iteration starts with.
        On one GPU the value-only Cholesky chain overlaps the gradient chain (accbpg_dopt_pair)."""
        rt = self.rt
        if self.shard is not None and self.shard.world > 1:
            self._enqueue(xd, 0, slot_x, None)
            self._enqueue(yd, flag_y, slot_y, g)
            return
        H = self._Hd
        nat.check(lib.accbpg_dopt_pair(rt.ctx, rt.stream, H.data_ptr(), self.m, self.n_local, H.stride(0),
                                       xd.data_ptr(), yd.data_ptr(), flag_y, self._ws.data_ptr(), rt.slot(slot_x),
                                       rt.slot(slot_y), g.data_ptr()))

    def _enqueue(self, xd, flag, slot, g):
        rt = self.rt
        H = self._Hd
        gp = g.data_ptr() if g is not None else None
        if self.shard is None or self.shard.world == 1:
            nat.check(lib.accbpg_dopt_func_grad(rt.ctx, rt.stream, H.data_ptr(), self.m, self.n_local, H.stride(0),
                                                xd.data_ptr(), flag, self._ws.data_ptr(), rt.slot(slot), gp))
            return
        ws = self._ws.data_ptr()
        self._gram_sharded(xd, self._M)
        nat.check(lib.accbpg_dopt_factor(rt.ctx, rt.stream, self.m, self._M.data_ptr(), None, int(flag >= 1), ws,
                                         rt.slot(slot)))
        if flag >= 1:
            nat.check(lib.accbpg_dopt_grad(rt.ctx, rt.stream, H.data_ptr(), self.m, self.n_local, H.stride(0), ws, gp))


class SparseDOptimalObj(RSmoothFunction):
    """f(x) = -log det(H diag(x) H^T) with H (m x n) SPARSE, held in compressed-column form on the device: column j of
    H is the j-th sample of a LIBSVM file (accbpg/applications.py:17-33 densifies the same data with .toarray('C');
    accbpg/functions.py:43-59 is the oracle).  The Gram matrix and the gradient read only the stored entries
    (accbpg_dopt_sparse_gram / accbpg_dopt_sparse_grad); the m x m factorisation is the dense chain.  m <= 128, one GPU.

    indptr / indices / values: the CSC arrays of H (= the CSR arrays of the samples-by-features matrix X), or pass a
    scipy.sparse matrix H as the first argument.  `f.H` is the scipy CSC matrix (host); `f.toarray()` the dense H.
    Either form is brought to canonical CSC on the host (rows sorted within a column, duplicate (row, column) entries
    summed, as scipy's toarray() does); the caller's arrays are not modified."""

    _lin_capable = True

    def __init__(self, indptr, indices=None, values=None, m=None, device=None):
        import scipy.sparse as sp
        self.rt = Runtime.get(device)
        self.shard = None
        if indices is None:                                   # a scipy.sparse matrix
            Hs = sp.csc_matrix(indptr, dtype=np.float64, copy=True)
        else:
            indptr = np.asarray(indptr, dtype=np.int64)
            indices = np.asarray(indices)
            values = np.asarray(values, dtype=np.float64)
            assert indptr.ndim == 1 and indptr.size >= 1 and indptr[0] == 0 and np.all(np.diff(indptr) >= 0), \
                "SparseDOptimalObj: indptr must start at 0 and be non-decreasing"
            assert indices.size == values.size == int(indptr[-1]), "SparseDOptimalObj: indices / values / indptr sizes"
            assert indices.size == 0 or (indices.min() >= 0 and indices.max() < int(m)), \
                "SparseDOptimalObj: row index outside [0, m)"
            Hs = sp.csc_matrix((values.copy(), indices.copy(), indptr.copy()), shape=(int(m), indptr.size - 1))
        assert Hs.indices.size == 0 or (Hs.indices.min() >= 0 and Hs.indices.max() < Hs.shape[0]), \
            "SparseDOptimalObj: row index outside [0, m)"
        # The Gram kernel scatters a column's entries into a dense tile (one write per (row, column)) while the gradient
        # kernel sums over every stored entry: duplicates must be merged here for the two to describe the same H.
        Hs.sum_duplicates()
        indptr, indices, values, m = Hs.indptr, Hs.indices, Hs.data, Hs.shape[0]
        self._indptr_h = np.ascontiguousarray(indptr, dtype=np.int64)
        self._indices_h = np.ascontiguousarray(indices, dtype=np.int32)
        self._values_h = np.ascontiguousarray(values, dtype=np.float64)
        self.m = int(m)
        self.n = self.n_local = int(self._indptr_h.size - 1)
        assert self.m < self.n, "DOptimalObj: need m < n"
        assert self.m <= 128, "SparseDOptimalObj: m <= 128 (use DOptimalObj on the dense matrix beyond)"
        assert self._indices_h.size == self._values_h.size == int(self._indptr_h[-1])
        dev = self.rt.device
        self._colptr = torch.from_numpy(self._indptr_h).to(dev)
        self._rowidx = torch.from_numpy(self._indices_h).to(dev)
        self._vals = torch.from_numpy(self._values_h).to(dev)
        with self.rt.on_device():
            self._ws = self.rt.workspace(("dopt_sparse", self.m, id(self)), lib.accbpg_dopt_sparse_workspace_bytes(self.m))
        self._M = torch.empty(self.m, self.m, dtype=torch.float64, device=dev)

    @property
    def H(self):
        import scipy.sparse as sp
        return sp.csc_matrix((self._values_h, self._indices_h, self._indptr_h), shape=(self.m, self.n))

    def toarray(self):
        return np.ascontiguousarray(self.H.toarray())

    def _gram(self, xd, M):
        rt = self.rt
        nat.check(lib.accbpg_dopt_sparse_gram(rt.ctx, rt.stream, self._colptr.data_ptr(), self._rowidx.data_ptr(),
                                              self._vals.data_ptr(), self.m, self.n, xd.data_ptr(), self._ws.data_ptr(),
                                              M.data_ptr()))

    def _factor_grad(self, M, flag, slot, g):
        rt = self.rt
        nat.check(lib.accbpg_dopt_factor(rt.ctx, rt.stream, self.m, M.data_ptr(), None, int(flag >= 1),
                                         self._ws.data_ptr(), rt.slot(slot)))
        if flag >= 1:
            nat.check(lib.accbpg_dopt_sparse_grad(rt.ctx, rt.stream, self._colptr.data_ptr(), self._rowidx.data_ptr(),
                                                  self._vals.data_ptr(), self.m, self.n, self._ws.data_ptr(),
                                                  g.data_ptr()))

    def _enqueue(self, xd, flag, slot, g):
        self._gram(xd, self._M)
        self._factor_grad(self._M, flag, slot, g)

    # ---- linear image M(x) (config.linear_images), as DOptimalObj
    def _img_compute(self, xd):
        M = torch.empty(self.m, self.m, dtype=torch.float64, device=self.rt.device)
        self._gram(xd, M)
        return M

    def _img_axpby(self, a, Ia, b, Ib):
        rt = self.rt
        out = torch.empty_like(Ia)
        nat.check(lib.accbpg_vec_axpby(rt.ctx, rt.stream, Ia.numel(), float(a), Ia.data_ptr(), float(b),
                                       Ib.data_ptr(), out.data_ptr()))
        return out

    def _enqueue_img_pair(self, Ix, slot_x, Iy, flag_y, slot_y, g):
        if Ix is not None:
            self._factor_grad(Ix, 0, slot_x, None)
        self._factor_grad(Iy, flag_y, slot_y, g)


class _LinearInverse(RSmoothFunction):
    """Shared body of PoissonRegression / KLdivRegression: Ax, value + residual, A^T r."""
    _kind = None

    def __init__(self, A, b, shard=None, device=None):
        assert A.shape[0] == b.shape[0], "A and b sizes not matching"
        self.rt = Runtime.get(device)
        self.shard = shard
        self.A, self.b = A, b
        self._Ad = self.rt.to_device(A)
        self._bd = self.rt.to_device(b)
        self.m, self.n_local = int(self._Ad.shape[0]), int(self._Ad.shape[1])
        self.n = shard.n if shard is not None else self.n_local
        with self.rt.on_device():
            self._ws = self.rt.workspace(("linreg", self.m, self.n_local),
                                         lib.accbpg_linreg_workspace_bytes(self.m, self.n_local))
        self._Ax = self.rt.empty(self.m)
        self._r = self.rt.empty(self.m)

    # ---- linear image A x (config.linear_images) -------------------------------------------------------------
    _lin_capable = True

    def _img_compute(self, xd):
        """A x as a new m-vector (K5; all-reduced when A is column-sharded)."""
        rt = self.rt
        A = self._Ad
        Ax = rt.empty(self.m)
        nat.check(lib.accbpg_linreg_matvec(rt.ctx, rt.stream, A.data_ptr(), self.m, self.n_local, A.stride(0),
                                           xd.data_ptr(), self._ws.data_ptr(), Ax.data_ptr()))
        if self.shard is not None and self.shard.world > 1:
            self.shard.sum_(Ax)
        return Ax

    def _img_axpby(self, a, Ia, b, Ib):
        rt = self.rt
        out = torch.empty_like(Ia)
        nat.check(lib.accbpg_vec_axpby(rt.ctx, rt.stream, Ia.numel(), float(a), Ia.data_ptr(), float(b),
                                       Ib.data_ptr(), out.data_ptr()))
        return out

    def _enqueue_img_pair(self, Ix, slot_x, Iy, flag_y, slot_y, g):
        """f from A x -> slot_x (skipped when Ix is None); (f, grad f) from A y -> (slot_y, g): K7 (+ K6) only."""
        rt = self.rt
        A = self._Ad
        if Ix is not None:
            nat.check(lib.accbpg_linreg_value_resid(rt.ctx, rt.stream, self._kind, self.m, Ix.data_ptr(),
                                                    self._bd.data_ptr(), rt.slot(slot_x), None))
        nat.check(lib.accbpg_linreg_value_resid(rt.ctx, rt.stream, self._kind, self.m, Iy.data_ptr(),
                                                self._bd.data_ptr(), rt.slot(slot_y),
                                                self._r.data_ptr() if flag_y >= 1 else None))
        if flag_y >= 1:
            nat.check(lib.accbpg_linreg_rmatvec(rt.ctx, rt.stream, A.data_ptr(), self.m, self.n_local, A.stride(0),
                                                self._r.data_ptr(), self._ws.data_ptr(), g.data_ptr()))

    def _enqueue(self, xd, flag, slot, g):
        rt = self.rt
        A = self._Ad
        nat.check(lib.accbpg_linreg_matvec(rt.ctx, rt.stream, A.data_ptr(), self.m, self.n_local, A.stride(0),
                                           xd.data_ptr(), self._ws.data_ptr(), self._Ax.data_ptr()))
        if self.shard is not None and self.shard.world > 1:
            self.shard.sum_(self._Ax)
        # the value costs nothing extra next to the residual (one pass over m), so it is always produced
        nat.check(lib.accbpg_linreg_value_resid(rt.ctx, rt.stream, self._kind, self.m, self._Ax.data_ptr(),
                                                self._bd.data_ptr(), rt.slot(slot),
                                                self._r.data_ptr() if flag >= 1 else None))
        if flag >= 1:
            nat.check(lib.accbpg_linreg_rmatvec(rt.ctx, rt.stream, A.data_ptr(), self.m, self.n_local, A.stride(0),
                                                self._r.data_ptr(), self._ws.data_ptr(), g.data_ptr()))


class PoissonRegression(_LinearInverse):
    """f(x) = D_KL(b, Ax).   accbpg/functions.py:85-120."""
    _kind = nat.MACROS["ACCBPG_LINREG_POISSON"]


class KLdivRegression(_LinearInverse):
    """f(x) = D_KL(Ax, b).   accbpg/functions.py:123-158."""
    _kind = nat.MACROS["ACCBPG_LINREG_KL"]
