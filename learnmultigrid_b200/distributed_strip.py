"""Row-partitioned hierarchy built from THIS RANK'S ROW BLOCKS ONLY (DESIGN 7, weak scaling): no process ever holds
a global operator of a partitioned level, so the problem is bounded by the memory of all GPUs together instead of one.

    StripHierarchy(A_blk, Q_blks, offsets, fabric, n_dist, ...)

    A_blk   : rows [offsets[0][rank], offsets[0][rank+1]) of A_0, global column ids (SciPy CSR)
    Q_blks  : the same rows of every Q_l (blocks of the levels below n_dist are gathered: those levels are replicated)
    offsets : partition.block_offsets per level

The host side is partition_setup.strip_local_setup (remote-row fetch, transpose exchange, Galerkin row blocks, first-fit
colours coloured in rank order, halo plans, gathered replicated tail -- verified on the CPU against the replicated
setup, tests/test_partition_setup.py); the three local sparse products of every level run on the device SpGEMM
(`DeviceOps`, the contract of partition_setup.ScipyOps).  From the plans on, the levels are built by
distributed.DistributedHierarchy._build_levels, the code DistributedHierarchy uses, with the row blocks uploaded
instead of cut out of global device matrices; the result -- SELL operators, layouts, exchange descriptors, mg_level.flags
-- is the same, so the cycle's iterates are bit-identical to DistributedHierarchy's and to the single-GPU hierarchy's.

STATUS: verified on B200 -- bit-identical to DistributedHierarchy on virtual ranks and on 2-8 real ranks
(tests/test_gpu_strip.py, profiles/r02_pytest_gpu_unverified_first_run.log, profiles/r02_weak_*: 537 M unknowns on 8
GPUs); both classes build the same level structs, field for field (tests/test_gpu_partitioned_levels.py).
"""
import numpy as np
import scipy.sparse as sp

from . import formats as F
from . import partition_setup as PS
from . import setup_device as SD
from .distributed import DistributedHierarchy
from .engine import DENSE_COARSE_MAX


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
        self._init_rank(fabric, smoother, len(Q_blks) + 1, device, split_coarse_solve, bcr_split_min_blocks)
        self._setup_strip(A_blk, list(Q_blks), [np.asarray(o, dtype=np.int64) for o in offsets], colors, n_dist,
                          dense_coarse_max, device_products)
        self._start(region_bytes, max_sites, timeout_s)

    def _setup_strip(self, A_blk, Q_blks, offs, colors, n_dist, dense_coarse_max, device_products):
        """The levels from this rank's row blocks: strip-local Galerkin products, colours and plans on the host side,
        the replicated tail gathered and formed on every rank."""
        S = SD.DeviceSetup(self.torch, self.device)
        L = self.nlevels
        if len(offs) != L:
            raise ValueError("one offsets array per level expected")
        if n_dist is None or not 1 <= int(n_dist) <= L - 1:
            raise ValueError("n_dist must be between 1 and levels-1")
        Lp = int(n_dist)
        self._global_n = [int(o[-1]) for o in offs]

        # ---- host side: blocks of every partitioned level, colours, plans, the gathered replicated tail
        ops = DeviceOps(S) if device_products else PS.ScipyOps
        own_colors = None if colors is None else [colors[l] for l in range(Lp)]
        strip, A_rep, Q_rep = PS.strip_local_setup(self.fabric, A_blk, Q_blks, offs, Lp, self.smoother, own_colors, ops)
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

        def row_block(l, m):
            blk = S.upload(getattr(strip[l], m))
            if m == "QT":
                strip[l] = None                        # the last block of level l: its host copy is not needed again
            return blk

        self._build_levels(S, offs, [s.plan for s in strip], row_block, A_nat, Q_nat, QT_nat, dense_coarse_max)
