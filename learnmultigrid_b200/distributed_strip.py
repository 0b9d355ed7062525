"""Row-partitioned hierarchy built from THIS RANK'S ROW BLOCKS ONLY (DESIGN 7, weak scaling): no process ever holds
a global operator of a partitioned level, so the problem is bounded by the memory of all GPUs together instead of one.

    StripHierarchy(A_blk, Q_blks, offsets, fabric, n_dist, ...)

    A_blk   : rows [offsets[0][rank], offsets[0][rank+1]) of A_0, global column ids (SciPy CSR)
    Q_blks  : the same rows of every Q_l (blocks of the levels below n_dist are gathered: those levels are replicated)
    offsets : partition.block_offsets per level

The host side is partition_setup.strip_local_setup (remote-row fetch, transpose exchange, Galerkin row blocks, first-fit
colours coloured in rank order, halo plans, gathered replicated tail -- verified on the CPU against the replicated
setup, tests/test_partition_setup.py); the three local sparse products of every level run on the device SpGEMM
(`DeviceOps`, the contract of partition_setup.ScipyOps).  From the plans on, the construction is the one of
distributed.DistributedHierarchy._setup_dist with the row blocks uploaded instead of cut out of global device
matrices; the result -- SELL operators, layouts, exchange descriptors -- is the same, so the cycle's iterates are
bit-identical to DistributedHierarchy's and to the single-GPU hierarchy's.

STATUS: verified on B200 in round 2 -- bit-identical to DistributedHierarchy on virtual ranks and on 2-8 real ranks
(tests/test_gpu_strip.py, profiles/r02_pytest_gpu_unverified_first_run.log, profiles/r02_weak_*: 537 M unknowns on 8
GPUs).  _setup_dist below still repeats the second half of DistributedHierarchy._setup_dist (row blocks uploaded
instead of cut out of global device matrices); merging the two is housekeeping that has not been done.
"""
import ctypes

import numpy as np
import scipy.sparse as sp

from . import _lib
from . import formats as F
from . import partition_setup as PS
from . import setup_device as SD
from .distributed import DistributedHierarchy, _Layout
from .engine import DENSE_COARSE_MAX, Level


class DeviceOps:
    """local sparse kernels of partition_setup on the device (setup_device.DeviceSetup): CSR in, CSR out, sorted
    columns, csr_matmat accumulation order, exact zeros pruned -- the contract of partition_setup.ScipyOps"""

    def __init__(self, S):
        self.S = S

    def spgemm(self, A, B):
        A, B = sp.csr_matrix(A), sp.csr_matrix(B)
        if A.shape[0] == 0 or B.shape[1] == 0 or A.nnz == 0 or B.nnz == 0:
            return sp.csr_matrix((A.shape[0], B.shape[1]))          # nothing to launch
        S = self.S
        return S.download(S.spgemm(S.upload(A), S.upload(B)))

    def transpose(self, A):
        A = sp.csr_matrix(A)
        if A.shape[0] == 0 or A.shape[1] == 0 or A.nnz == 0:
            return sp.csr_matrix((A.shape[1], A.shape[0]))
        S = self.S
        return S.download(S.transpose(S.upload(A)))


class StripHierarchy(DistributedHierarchy):
    """DistributedHierarchy from row blocks.  `colors`: optional list with, per partitioned level, the colours of the
    OWN rows and, per replicated level, the global colour array (None entries = first-fit).  `device_products=False`
    runs the local products with SciPy (cross-check)."""

    def __init__(self, A_blk, Q_blks, offsets, fabric, n_dist, smoother="jacobi", colors=None, device=None,
                 dense_coarse_max=DENSE_COARSE_MAX, region_bytes=16 << 20, max_sites=512, timeout_s=10.0,
                 split_coarse_solve=True, bcr_split_min_blocks=32, device_products=True):
        if smoother == "chebyshev":
            raise ValueError("StripHierarchy supports 'jacobi' and 'mcgs'; the Chebyshev smoother needs the global "
                             "operators for its bounds (use DistributedHierarchy)")
        self._strip_inputs = (A_blk, list(Q_blks), [np.asarray(o, dtype=np.int64) for o in offsets])
        self._device_products = bool(device_products)
        super().__init__(None, [None] * len(Q_blks), fabric, smoother=smoother, colors=colors, device=device,
                         n_dist=n_dist, dense_coarse_max=dense_coarse_max, keep_host=False,
                         region_bytes=region_bytes, max_sites=max_sites, timeout_s=timeout_s,
                         split_coarse_solve=split_coarse_solve, bcr_split_min_blocks=bcr_split_min_blocks)

    def _setup_dist(self, A, Q_list, colors, dense_coarse_max, min_rows, n_dist):
        torch, dev = self.torch, self.device
        W, rank = self.world, self.rank
        S = SD.DeviceSetup(torch, dev)
        self._setup = S
        L = self.nlevels
        A_blk, Q_blks, offs = self._strip_inputs
        self._strip_inputs = None
        if len(offs) != L:
            raise ValueError("one offsets array per level expected")
        if n_dist is None or not 1 <= int(n_dist) <= L - 1:
            raise ValueError("n_dist must be between 1 and levels-1")
        self.n_dist = Lp = int(n_dist)
        ns = [int(o[-1]) for o in offs]
        self._global_n = ns
        self.offsets = offs

        # ---- host side: blocks of every partitioned level, colours, plans, the gathered replicated tail
        ops = DeviceOps(S) if self._device_products else PS.ScipyOps
        own_colors = None if colors is None else [colors[l] for l in range(Lp)]
        strip, A_rep, Q_rep = PS.strip_local_setup(self.fabric, A_blk, Q_blks, offs, Lp, self.smoother, own_colors, ops)
        del A_blk, Q_blks
        plans = [s.plan for s in strip]
        self.plans = plans
        self.own_colors = [s.colors for s in strip]
        nnz = self.fabric.allgather([(s.A.nnz, s.Q.nnz) for s in strip])
        self._global_nnzA = [sum(int(part[l][0]) for part in nnz) for l in range(Lp)]
        self._global_nnzQ = [sum(int(part[l][1]) for part in nnz) for l in range(Lp)]

        # ---- replicated tail in natural ordering on the device (small: formed redundantly on every rank as before)
        A_nat, Q_nat, QT_nat = [None] * Lp, [None] * Lp, [None] * Lp
        A_nat.append(S.upload(A_rep))
        for l in range(Lp, L - 1):
            Q = S.upload(Q_rep[l - Lp])
            QT = S.transpose(Q)
            Q_nat.append(Q)
            QT_nat.append(QT)
            A_nat.append(S.galerkin(A_nat[l], Q, QT))
        self._global_nnzA += [A_nat[l].nnz for l in range(Lp, L)]
        self._global_nnzQ += [Q_nat[l].nnz for l in range(Lp, L - 1)]
        self.colors = [None] * L                       # global colour arrays exist for the replicated levels only
        for l in range(Lp, L - 1):
            if self.smoother != "mcgs":
                break
            if colors is not None and colors[l] is not None:
                self.colors[l] = np.ascontiguousarray(colors[l], dtype=np.int32)
            else:
                pat = A_rep if l == Lp else S.download(A_nat[l])
                self.colors[l] = F.greedy_colors(pat)[0]
        del A_rep, Q_rep

        # who needs what from whom: every rank tells the others which of their rows it reads, in its halo order
        mine = []
        for l in range(Lp):
            p = plans[l]
            nc = max(p.ncolors, 1)
            d = {}
            for q in p.neighbours:
                s, e = p.seg[q]
                ptr = [p.seg_color[(q, c)][0] - s for c in range(nc)] + [e - s]
                d[q] = (p.halo_gid[s:e], ptr)
            mine.append(d)
        everyone = self.fabric.allgather(mine)

        # ---- layouts (global id -> position in my level vector)
        lays = []
        for l in range(L):
            if l < Lp:
                p = plans[l]
                slot = torch.full((ns[l],), -1, dtype=torch.int32, device=dev)
                if p.n_halo:
                    slot[torch.from_numpy(p.halo_gid).to(dev)] = torch.arange(p.n_halo, dtype=torch.int32, device=dev)
                ip = None if p.iperm is None else torch.from_numpy(p.iperm).to(dev)
                lays.append(_Layout(p.o0, p.o1, ip, p.n_own, slot, p.n_own + p.n_halo))
            else:
                lays.append(None)
        perms, iperms, cptrs = [None] * L, [None] * L, [None] * L
        for l in range(Lp, L):
            if self.colors[l] is not None:
                perms[l], iperms[l], cptrs[l] = S.color_perm(self.colors[l])
        dummy = torch.zeros(1, dtype=torch.int32, device=dev)
        lays[Lp] = _Layout(0, ns[Lp], iperms[Lp], ns[Lp], dummy, ns[Lp])

        # ---- partitioned levels: the row blocks are uploaded as they are (global column ids) and remapped
        self.levels = []
        for l in range(Lp):
            p = plans[l]
            lev = Level()
            lev.n = p.n_own
            lev.n_halo = p.n_halo
            lev.n_vec = p.n_own + p.n_halo
            lev.plan = p
            lev.perm = None if p.perm is None else torch.from_numpy(p.perm).to(dev)
            lev.color_ptr = p.color_ptr
            lev.nnz_A, lev.nnz_Q = self._global_nnzA[l], self._global_nnzQ[l]
            blk = S.upload(strip[l].A)
            loc = SD.DevCSR((p.n_own, lev.n_vec), blk.indptr, self._remap(S, blk.indices, lays[l]), blk.values)
            Ap = S.permute(loc, lev.perm, None)
            lev.A = S.to_sell(Ap)
            lev.dinv = S.dinv(Ap, None)
            lev.local_nnz_A = Ap.nnz
            if p.color_ptr is not None:
                # mg_level.flags must hold for the GLOBAL operator and be the same on every rank (they decide the
                # launch sequence, hence the exchange sites): this block's rows against the colours of everything they
                # read -- own rows by colour block, halo slots by (owner, colour) segment -- then AND over the ranks
                vcol = np.full(lev.n_vec, -1, dtype=np.int32)
                for c in range(len(p.color_ptr) - 1):
                    vcol[int(p.color_ptr[c]):int(p.color_ptr[c + 1])] = c
                for (q, c), (a, b) in p.seg_color.items():
                    vcol[p.n_own + a:p.n_own + b] = c
                mine_flags = S.coloring_flags(Ap, vcol)
                lev.flags = int(np.bitwise_and.reduce([int(f) for f in self.fabric.allgather(mine_flags)]))
            del blk, loc, Ap
            blk = S.upload(strip[l].Q)
            loc = SD.DevCSR((p.n_own, lays[l + 1].length), blk.indptr, self._remap(S, blk.indices, lays[l + 1]),
                            blk.values)
            lev.Q = S.to_sell(S.permute(loc, lev.perm, None))
            del blk, loc
            c0, c1 = int(offs[l + 1][rank]), int(offs[l + 1][rank + 1])
            blk = S.upload(strip[l].QT)
            loc = SD.DevCSR((c1 - c0, lev.n_vec), blk.indptr, self._remap(S, blk.indices, lays[l]), blk.values)
            cperm = None
            if l + 1 < Lp and plans[l + 1].perm is not None:
                cperm = torch.from_numpy(plans[l + 1].perm).to(dev)
            lev.QT = S.to_sell(S.permute(loc, cperm, None))
            del blk, loc
            strip[l] = None
            self._build_xfers(lev, l, everyone, offs, iperms, Lp)
            lev.masks = []
            for Msell, first_halo in ((lev.A, p.n_own), (lev.Q, lays[l + 1].n_own), (lev.QT, p.n_own)):
                mk = torch.zeros(max(int(Msell.struct.nslices), 1), dtype=torch.uint8, device=dev)
                _lib.check(self.lib.mg_sell_halo_mask(ctypes.byref(Msell.struct), int(first_halo), mk.data_ptr(),
                                                      S.st()), "mg_sell_halo_mask")
                lev.masks.append(mk)
            d = lev.dist_struct
            d.d_mask_A, d.d_mask_Q, d.d_mask_QT = (m.data_ptr() for m in lev.masks)
            self.levels.append(lev)
        del lays
        # ---- replicated levels
        for l in range(Lp, L):
            self.levels.append(SD.build_replicated_level(self, S, l, L, None, A_nat, Q_nat, QT_nat, perms, iperms,
                                                         cptrs, dense_coarse_max))
        last = self.levels[-1]
        if last.coarse_kind == _lib.MG_COARSE_BCR and self.split_coarse_solve:
            last.coarse_bcr_dist = last.coarse.make_dist(rank, W, self.bcr_split_min_blocks)
        self.host_A = None
        self.host_Q = None
        S._temp = None
        torch.cuda.current_stream().synchronize()
