"""Device pipeline of the reference's 2D NN transfer-operator builder (NeuralMG_2D.define_hierarchy,
learn_multigrid/solvers/Multigrid.py:741-765 and helpers :401-739) on top of csrc/nn_kernels.cu.

Per level:  coarsening (lexicographically first independent set)  ->  patches (n_C x 43) + fill indices (n_C x 31)
->  (patches - mean) / std  ->  model.predict  ->  fill_B (ordered running mean)  ->  Q = B / rowsum(B)
->  M <- Q^T M Q  ->  pre_process (cut the coarse rows to the predicted neighbours).
Everything stays in device memory (CSR, fp64 / int32); the reference needs a dense copy of M and ~14 ms of Python per
coarse node.  The predictor is any object with `predict(ndarray) -> ndarray` (the reference's Keras interface; host
round trip) or `predict_device(tensor) -> tensor`.  The trained weights of the reference are not shipped
(data/models is empty), so two stand-ins live here: MassSurrogate (predicts the mass-matrix entries the patch already
contains: B[f, C(c)] = M[f, c], a mass-weighted direct interpolation) and TorchMLP (a randomly initialised MLP of the
reference's architecture family, to exercise the inference path).
"""
import ctypes

import numpy as np
import scipy.sparse as sp

from . import _lib
from . import formats as F
from . import setup_device as SD


class MassSurrogate:
    """pred[0] = M[c,c], pred[1:7] = M[c, neighbour_k] (what B_h = M_h P has on a nested mesh for the coarse node's own
    column, SURVEY 7.1), everything else 0 (treated as 'no entry' by fill_B)."""

    def __init__(self, mean=None, std=None):
        self.mean = np.zeros(43) if mean is None else np.asarray(mean, dtype=np.float64)
        self.std = np.ones(43) if std is None else np.asarray(std, dtype=np.float64)

    def predict(self, X):
        P = np.asarray(X, dtype=np.float64) * self.std + self.mean
        out = np.zeros((P.shape[0], 31))
        out[:, 0:7] = P[:, 0:7]
        return out

    def predict_device(self, X):
        import torch
        P = X * torch.from_numpy(self.std).to(X.device) + torch.from_numpy(self.mean).to(X.device)
        out = torch.zeros((P.shape[0], 31), dtype=torch.float64, device=X.device)
        out[:, 0:7] = P[:, 0:7]
        return out


class TorchMLP:
    """dense ReLU MLP 43 -> hidden... -> 31 (test/test_comparison_NNs.py:50-66 builds this family), random weights"""

    def __init__(self, hidden=(200, 200, 200), seed=0, device="cuda"):
        import torch
        g = torch.Generator().manual_seed(seed)
        sizes = (43,) + tuple(hidden) + (31,)
        self.layers = []
        for a, b in zip(sizes[:-1], sizes[1:]):
            W = (torch.randn(a, b, generator=g, dtype=torch.float64) / np.sqrt(a)).to(device)
            bias = torch.zeros(b, dtype=torch.float64, device=device)
            self.layers.append((W, bias))

    def predict_device(self, X):
        import torch
        h = X
        for i, (W, b) in enumerate(self.layers):
            h = h @ W + b
            if i + 1 < len(self.layers):
                h = torch.relu(h)
        return torch.nn.functional.softplus(h)      # keep B positive so that row sums cannot vanish

    def predict(self, X):
        import torch
        return self.predict_device(torch.from_numpy(np.asarray(X, dtype=np.float64)).to(self.layers[0][0].device)).cpu().numpy()


class NeuralBuilder:
    """device kernels of the builder, one method per reference function"""

    def __init__(self, torch=None, device=None):
        self.torch = torch = _lib.require_cuda() if torch is None else torch
        self.dev = torch.device("cuda", torch.cuda.current_device()) if device is None else device
        self.lib = _lib.load()
        self.S = SD.DeviceSetup(torch, self.dev)

    def st(self):
        return _lib.stream_handle(self.torch)

    def upload(self, M):
        return self.S.upload(M)

    def download(self, M):
        return self.S.download(M)

    # coarsening + map_coarse (Multigrid.py:401-426, 679-684)
    def coarsen(self, M):
        t, S = self.torch, self.S
        n = M.shape[0]
        MT = S.transpose(M)
        state = S.empty(n, t.int32)
        work = S.empty(n + 1, t.int32)
        rounds = self.lib.mg_nn_coarsen(n, *MT.ptrs(), state.data_ptr(), work.data_ptr(), self.st())
        if rounds < 0:
            _lib.check(rounds, "mg_nn_coarsen")
        flags = (state == 1).to(t.int32)
        scan, nc = S.scan(flags, n)
        cmap = S.empty(n, t.int32)
        clist = S.empty(nc, t.int32)
        _lib.check(self.lib.mg_nn_compact(n, state.data_ptr(), scan.data_ptr(), cmap.data_ptr(), clist.data_ptr(),
                                          self.st()), "mg_nn_compact")
        self.last_rounds = int(rounds)
        return cmap, clist, nc

    # extract_patches (:591-677); rows nc.. hold the extra patch variants of nodes with more than 6 neighbours (:631-663)
    def extract(self, M, cmap, clist):
        t, S = self.torch, self.S
        nc = clist.numel()
        extra = S.empty(nc, t.int32)
        _lib.check(self.lib.mg_nn_count_variants(nc, *M.ptrs(), clist.data_ptr(), extra.data_ptr(), self.st()),
                   "mg_nn_count_variants")
        extra_ptr, total = S.scan(extra, nc)
        rows = nc + total
        patches = S.empty(rows * 43, t.float64)
        fill = S.empty(rows * 31, t.int32)
        _lib.check(self.lib.mg_nn_extract_patches(nc, *M.ptrs(), cmap.data_ptr(), clist.data_ptr(), patches.data_ptr(),
                                                  fill.data_ptr(), S._flag.data_ptr(), self.st()),
                   "mg_nn_extract_patches")
        self.not_last = None
        if total:
            self.not_last = t.zeros(rows, dtype=t.int32, device=self.dev)
            _lib.check(self.lib.mg_nn_extract_variants(nc, *M.ptrs(), cmap.data_ptr(), clist.data_ptr(),
                                                       extra_ptr.data_ptr(), patches.data_ptr(), fill.data_ptr(),
                                                       self.not_last.data_ptr(), S._flag.data_ptr(), self.st()),
                       "mg_nn_extract_variants")
        return patches.view(rows, 43), fill.view(rows, 31)

    # (patches - mean) / std ; model.predict (:755-756)
    def predict(self, model, patches, mean, std):
        t = self.torch
        mean_t = t.from_numpy(np.broadcast_to(np.asarray(mean, dtype=np.float64), (43,)).copy()).to(self.dev)
        std_t = t.from_numpy(np.broadcast_to(np.asarray(std, dtype=np.float64), (43,)).copy()).to(self.dev)
        pn = (patches - mean_t) / std_t
        if hasattr(model, "predict_device"):
            res = model.predict_device(pn)
        else:
            res = t.from_numpy(np.ascontiguousarray(np.asarray(model.predict(pn.cpu().numpy()), dtype=np.float64))).to(self.dev)
        if tuple(res.shape) != (patches.shape[0], 31):
            raise ValueError("the predictor must return (n_patches, 31) values, got %r" % (tuple(res.shape),))
        return res.to(t.float64).contiguous()

    # fill_B (:687-732) -> (B as device CSR n x nc, d_neighs table nc x 6)
    def fill_B(self, pred, fill, cmap, n, nc, not_last=None):
        """not_last: int32 flag per patch, set for all but the last patch of a node that has several (`extract` leaves it
        in self.not_last); None = derive it here from the fill indices (any patch followed by one of the same node)"""
        t, S = self.torch, self.S
        np_ = fill.shape[0]
        if not_last is None and np_ > nc:
            node = fill[:, 0].to(t.int64)
            last = t.full((int(cmap.numel()),), -1, dtype=t.int64, device=self.dev)
            last.scatter_reduce_(0, node, t.arange(np_, device=self.dev), reduce="amax")
            not_last = (last[node] != t.arange(np_, device=self.dev)).to(t.int32).contiguous()
        m = np_ * 31
        rows, cols = S.empty(m, t.int32), S.empty(m, t.int32)
        vals = S.empty(m, t.float64)
        dneigh = t.full((nc * 6,), -1, dtype=t.int32, device=self.dev)
        _lib.check(self.lib.mg_nn_contributions(np_, fill.data_ptr(), pred.data_ptr(), cmap.data_ptr(),
                                                not_last.data_ptr() if not_last is not None else None, n,
                                                rows.data_ptr(), cols.data_ptr(), vals.data_ptr(), dneigh.data_ptr(),
                                                self.st()), "mg_nn_contributions")
        order = S.row_col_order(rows, cols, n + 1, nc)        # stable by column, then stably by row (unused: row n)
        head = S.empty(m, t.int32)
        folded = S.empty(m, t.float64)
        _lib.check(self.lib.mg_nn_fold(m, n, rows.data_ptr(), cols.data_ptr(), vals.data_ptr(), order.data_ptr(),
                                       head.data_ptr(), folded.data_ptr(), self.st()), "mg_nn_fold")
        slot, nnz = S.scan(head, m)
        orow, ocol = S.empty(nnz, t.int32), S.empty(nnz, t.int32)
        oval = S.empty(nnz, t.float64)
        _lib.check(self.lib.mg_nn_emit(m, rows.data_ptr(), cols.data_ptr(), order.data_ptr(), head.data_ptr(),
                                       slot.data_ptr(), folded.data_ptr(), orow.data_ptr(), ocol.data_ptr(),
                                       oval.data_ptr(), self.st()), "mg_nn_emit")
        indptr = t.searchsorted(orow, t.arange(n + 1, dtype=t.int32, device=self.dev)).to(t.int32)
        return SD.DevCSR((n, nc), indptr, ocol, oval), dneigh.view(nc, 6)

    # Q = B / rowsum(B) (:758-759); in place
    def normalise(self, B):
        _lib.check(self.lib.mg_nn_row_normalise(B.shape[0], B.indptr.data_ptr(), B.values.data_ptr(), self.st()),
                   "mg_nn_row_normalise")
        return B

    # pre_process (:735-739)
    def cut(self, M, dneigh):
        t, S = self.torch, self.S
        n = M.shape[0]
        keep = S.empty(M.nnz, t.int32)
        count = S.empty(n, t.int32)
        dn = dneigh.contiguous()
        _lib.check(self.lib.mg_nn_cut_count(n, *M.ptrs(), dn.data_ptr(), keep.data_ptr(), count.data_ptr(), self.st()),
                   "mg_nn_cut_count")
        optr, total = S.scan(count, n)
        oidx, oval = S.empty(total, t.int32), S.empty(total, t.float64)
        _lib.check(self.lib.mg_nn_cut_fill(n, *M.ptrs(), keep.data_ptr(), optr.data_ptr(), oidx.data_ptr(),
                                           oval.data_ptr(), self.st()), "mg_nn_cut_fill")
        return SD.DevCSR(M.shape, optr, oidx, oval)

    # define_hierarchy (:741-765)
    def define_hierarchy(self, M, model, mean, std, levels, keep_intermediates=False):
        """M: SciPy matrix or DevCSR.  Returns the list of device CSR transfer operators [Q_0, ...]."""
        mass = M if isinstance(M, SD.DevCSR) else self.upload(M)
        Qs, trace = [], []
        dneigh = None
        for i in range(levels - 1):
            if dneigh is not None:
                mass = self.cut(mass, dneigh)
            cmap, clist, nc = self.coarsen(mass)
            patches, fill = self.extract(mass, cmap, clist)
            pred = self.predict(model, patches, mean, std)
            B, dneigh = self.fill_B(pred, fill, cmap, mass.shape[0], nc, not_last=self.not_last)
            if keep_intermediates:
                trace.append({"M": mass, "cmap": cmap, "clist": clist, "patches": patches, "fill": fill,
                              "not_last": self.not_last, "pred": pred,
                              "B": SD.DevCSR(B.shape, B.indptr, B.indices, B.values.clone()), "dneigh": dneigh,
                              "rounds": self.last_rounds})
            Q = self.normalise(B)
            Qs.append(Q)
            if i + 1 < levels - 1:
                QT = self.S.transpose(Q)
                mass = self.S.galerkin(mass, Q, QT)
        self.trace = trace
        return Qs
