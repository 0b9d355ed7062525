"""Row-partitioned multigrid hierarchy over the GPUs of one box (SURVEY.md 8e; no reference counterpart -- the
reference is single-process, the contract comes from BASELINE.json's north star).

Layout.  Every level l < n_dist is split into `world` contiguous row blocks (partition.block_offsets); rank r holds
the rows of A_l and Q_l that it owns and the rows of Q_l^T for the coarse rows it owns, as SELL-32 matrices whose
columns index the rank's level vector  [owned entries, colour-blocked | halo entries]  (partition.RankPlan).  Levels
below `n_dist` are small and latency-bound: they are replicated (every rank runs them redundantly on the full
vector), the hand-off being an all-gather of the restricted right-hand side; no broadcast is needed on the way up.

Exchanges go through libmgb200's peer-memory protocol (csrc/comm.cu): one fused kernel per exchange site writes the
boundary values straight into the neighbours' arenas over NVLink and unpacks what they wrote, inside the same CUDA
graph as the V-cycle kernels.  torch.distributed is used for plumbing only (IPC handles, send lists, barriers).

With the same global colouring the partitioned cycle performs the single-GPU cycle's arithmetic in the same order, so
iterates are bit-identical to DeviceHierarchy's; only the residual norm is summed per block (ranks in order).

The hierarchy SETUP is replicated: every rank forms the global Galerkin hierarchy on its own GPU (setup_device's
SpGEMM path) and cuts out its blocks.  That bounds the global problem by one GPU's memory (fine for the 67 M-DOF
configuration: ~9 GB) and keeps the partitioned operators bit-identical to the single-GPU ones.
"""
import ctypes
import os
import threading

import numpy as np

from . import _lib
from . import partition as PT
from . import setup_device as SD
from .engine import DeviceHierarchy, Level, DENSE_COARSE_MAX, algorithmic_bytes_csr


# ------------------------------------------------------------------------------------------------------------
# fabrics: the host-side "who are my peers" plumbing
class ThreadFabric:
    """`world` virtual ranks inside ONE process, one thread each (all on the current device unless told otherwise).
    Used by the single-GPU parity tests of the partitioned cycle: the peers' arenas are plain device pointers."""

    def __init__(self, world):
        self.world = int(world)
        self._barrier = threading.Barrier(self.world)
        self._slots = [None] * self.world

    def view(self, rank):
        return _ThreadView(self, rank)

    def abort(self):
        self._barrier.abort()


class _ThreadView:
    in_process = True

    def __init__(self, fabric, rank):
        self.fabric, self.rank, self.world = fabric, int(rank), fabric.world

    def allgather(self, obj):
        f = self.fabric
        f._slots[self.rank] = obj
        f._barrier.wait()
        out = list(f._slots)
        f._barrier.wait()
        return out

    def barrier(self):
        self.fabric._barrier.wait()


class TorchFabric:
    """One process per GPU; torch.distributed (NCCL or gloo) carries the setup-time host messages."""
    in_process = False

    def __init__(self, group=None):
        import torch.distributed as dist
        self.dist, self.group = dist, group
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)

    def allgather(self, obj):
        out = [None] * self.world
        self.dist.all_gather_object(out, obj, group=self.group)
        return out

    def barrier(self):
        self.dist.barrier(group=self.group)


def run_virtual_ranks(world, fn, device=None):
    """Run fn(fabric_view) on `world` threads, each with its own CUDA stream; returns the list of results."""
    import torch
    fab = ThreadFabric(world)
    out, err = [None] * world, [None] * world
    dev = torch.cuda.current_device() if device is None else device

    def work(r):
        try:
            torch.cuda.set_device(dev)
            with torch.cuda.stream(torch.cuda.Stream(device=dev)):
                out[r] = fn(fab.view(r))
                torch.cuda.current_stream().synchronize()
        except BaseException as e:       # noqa: BLE001 -- re-raised below
            err[r] = e
            fab.abort()

    ts = [threading.Thread(target=work, args=(r,)) for r in range(world)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    for e in err:
        if e is not None and not isinstance(e, threading.BrokenBarrierError):
            raise e
    for e in err:
        if e is not None:
            raise e
    return out


# ------------------------------------------------------------------------------------------------------------
class PeerComm:
    """This rank's arena + the peers' arenas mapped into this process (mg_comm of include/mgb200.h)."""

    def __init__(self, fabric, torch, region_bytes=16 << 20, max_sites=512, timeout_s=10.0):
        lib = _lib.load()
        self.lib, self.fabric, self.torch = lib, fabric, torch
        W, rank = fabric.world, fabric.rank
        if W > _lib.MG_MAX_RANKS:
            raise _lib.MgError("at most %d ranks per box" % _lib.MG_MAX_RANKS)
        region_bytes = (int(region_bytes) + 127) // 128 * 128
        nbytes = int(lib.mg_comm_arena_bytes(W, max_sites, region_bytes))
        if nbytes <= 0:
            raise _lib.MgError("bad communicator geometry")
        arena = ctypes.c_void_p()
        _lib.check(lib.mg_comm_alloc(nbytes, ctypes.byref(arena)), "mg_comm_alloc")
        self.arena = arena
        self.arena_bytes = nbytes
        self._imported = []
        c = _lib.mg_comm()
        c.rank, c.world, c.max_sites, c.region_bytes, c.timeout_s = rank, W, max_sites, region_bytes, float(timeout_s)
        if fabric.in_process:
            ptrs = fabric.allgather(arena.value)
            for q in range(W):
                c.d_arena[q] = ptrs[q]
        else:
            h = ctypes.create_string_buffer(64)
            _lib.check(lib.mg_comm_export(arena, h), "mg_comm_export")
            handles = fabric.allgather(bytes(h.raw))
            for q in range(W):
                if q == rank:
                    c.d_arena[q] = arena.value
                else:
                    p = ctypes.c_void_p()
                    _lib.check(lib.mg_comm_import(handles[q], ctypes.byref(p)), "mg_comm_import")
                    self._imported.append(p)
                    c.d_arena[q] = p.value
        self.struct = c
        _lib.check(lib.mg_comm_init(ctypes.byref(c), _lib.stream_handle(torch)), "mg_comm_init")
        torch.cuda.current_stream().synchronize()
        fabric.barrier()

    def check(self):
        e = ctypes.c_int32(0)
        _lib.check(self.lib.mg_comm_error(ctypes.byref(self.struct), ctypes.byref(e),
                                          _lib.stream_handle(self.torch)), "mg_comm_error")
        if e.value:
            raise _lib.MgError("rank %d: exchange site %d timed out waiting for a peer" % (self.struct.rank, e.value - 1))

    def close(self):
        if self.arena is None:
            return
        self.torch.cuda.current_stream().synchronize()
        self.fabric.barrier()
        for p in self._imported:
            self.lib.mg_comm_unmap(p)
        self._imported = []
        self.fabric.barrier()
        self.lib.mg_comm_free(self.arena)
        self.arena = None


class _Layout:
    """How the global ids of one level map to positions of THIS rank's level vector."""

    def __init__(self, c0, c1, own_iperm, n_own, slot_of, length):
        self.c0, self.c1, self.own_iperm, self.n_own, self.slot_of, self.length = c0, c1, own_iperm, n_own, slot_of, length


class DistributedHierarchy(DeviceHierarchy):
    """Multigrid hierarchy whose first `n_dist` levels are row-partitioned over the ranks of `fabric`.

    A, Q_list, smoother, colors : as DeviceHierarchy (GLOBAL operators, identical on every rank)
    fabric                      : TorchFabric() (one process per GPU) or a ThreadFabric view (virtual ranks)
    min_rows_per_rank           : levels with fewer rows per rank are replicated (latency-bound anyway)
    n_dist                      : force the number of partitioned levels (1 <= n_dist <= levels-1)
    split_coarse_solve          : split the large steps of a block-cyclic-reduction coarsest solve over the ranks
    """

    def __init__(self, A, Q_list, fabric, smoother="jacobi", colors=None, device=None, min_rows_per_rank=65536,
                 n_dist=None, dense_coarse_max=DENSE_COARSE_MAX, keep_host=False, region_bytes=16 << 20,
                 max_sites=512, timeout_s=10.0, split_coarse_solve=True, bcr_split_min_blocks=32, cheby_degree=2,
                 cheby_bounds=None):
        self._init_rank(fabric, smoother, len(Q_list) + 1, device, split_coarse_solve, bcr_split_min_blocks,
                        cheby_degree, cheby_bounds)
        self.keep_host = keep_host
        self._setup_dist(A, Q_list, colors, dense_coarse_max, min_rows_per_rank, n_dist)
        self._start(region_bytes, max_sites, timeout_s)

    def _init_rank(self, fabric, smoother, nlevels, device, split_coarse_solve, bcr_split_min_blocks, cheby_degree=2,
                   cheby_bounds=None):
        """This rank's state before any level exists: device, smoother, fabric."""
        torch = _lib.require_cuda()
        self.split_coarse_solve = bool(split_coarse_solve)
        self.bcr_split_min_blocks = int(bcr_split_min_blocks)
        self.torch = torch
        self.lib = _lib.load()
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        if smoother not in ("jacobi", "mcgs", "chebyshev"):
            raise ValueError("partitioned levels support 'jacobi', 'mcgs' and 'chebyshev' (index-order Gauss-Seidel is "
                             "serial across row blocks)")
        self.smoother = smoother
        self.nlevels = nlevels
        if self.nlevels < 2:
            raise ValueError("need at least one transfer operator (levels >= 2)")
        self._chebyshev_args(cheby_degree, cheby_bounds)
        self.fabric = fabric
        self.rank, self.world = fabric.rank, fabric.world
        self._graphs = {}
        self._keep = []
        self.setup_kind = "device"

    def _start(self, region_bytes, max_sites, timeout_s):
        """Communicator, level structs and warm-up once the levels are built; returns when every rank is ready."""
        torch = self.torch
        self.comm = PeerComm(self.fabric, torch, region_bytes, max_sites, timeout_s)
        self._finish_structs()
        self._norm_local = torch.zeros(1, dtype=torch.float64, device=self.device)
        self._norm_slots = torch.zeros(_lib.MG_MAX_RANKS, dtype=torch.float64, device=self.device)
        self._norm_struct = _lib.mg_dist_norm(self._norm_ws.data_ptr(), self._norm_local.data_ptr(),
                                              self._norm_slots.data_ptr(), self._norm_out.data_ptr())
        self._warm_up()
        torch.cuda.current_stream().synchronize()
        self.fabric.barrier()

    def _warm_up(self):
        """Launch every kernel of the cycle once with the exchanges disabled (mg_comm.dry_run), so that CUDA's lazy
        kernel loading happens now and not while a peer's exchange kernel is spinning (mgb200.h, mg_comm)."""
        torch = self.torch
        st = _lib.stream_handle(torch)
        c = self.comm.struct
        c.dry_run = 1
        try:
            for nu, after in ((1, 0), (2, 0), (1, 1)):          # norm before / after the cycle: different kernels
                params = self.make_params(nu_pre=nu, nu_post=nu, omega=2.0 / 3.0)
                self._norm_struct.after = after
                _lib.check(self.lib.mg_vcycle_dist(ctypes.byref(c), self._level_structs, self.nlevels,
                                                   ctypes.byref(params), ctypes.byref(self._norm_struct), st),
                           "mg_vcycle_dist (warm-up)")
            self._norm_struct.after = 0
            lev = self.levels[0]
            if lev.perm is not None:
                _lib.check(self.lib.mg_gather(self.n, lev.perm.data_ptr(), self._stage.data_ptr(), lev.tmp.data_ptr(),
                                              st), "mg_gather")
                _lib.check(self.lib.mg_scatter(self.n, lev.perm.data_ptr(), lev.tmp.data_ptr(), self._stage.data_ptr(),
                                               st), "mg_scatter")
            _lib.check(self.lib.mg_sell_residual(ctypes.byref(lev.A.struct), lev.x.data_ptr(), lev.b.data_ptr(),
                                                 lev.r.data_ptr(), st), "mg_sell_residual")
            self._norm_host.copy_(self._norm_out, non_blocking=True)
            self._pinned.copy_(lev.x[:self.n], non_blocking=True)
            torch.cuda.current_stream().synchronize()
        finally:
            c.dry_run = 0
        for lv in self.levels:
            for v in (lv.x, lv.b, lv.r, lv.tmp):
                v.zero_()
        self._stage.zero_()

    # ------------------------------------------------------------------------------------------------
    def _remap(self, S, cols, lay):
        t = self.torch
        out = S.empty(cols.numel(), t.int32)
        S._flag.zero_()
        _lib.check(self.lib.mg_csr_remap_cols(cols.numel(), cols.data_ptr(), lay.c0, lay.c1, _lib.ptr(lay.own_iperm),
                                              lay.n_own, lay.slot_of.data_ptr(), out.data_ptr(), S._flag.data_ptr(),
                                              S.st()), "mg_csr_remap_cols")
        if int(S._flag.item()):
            raise _lib.MgError("a column outside the halo plan was referenced (plan/operator mismatch)")
        return out

    @staticmethod
    def _rowblock(M, r0, r1):
        a, b = int(M.indptr[r0].item()), int(M.indptr[r1].item())
        ip = (M.indptr[r0:r1 + 1] - a).contiguous()
        return SD.DevCSR((r1 - r0, M.shape[1]), ip, M.indices[a:b], M.values[a:b])

    def _ext(self, M, r0, r1, c0, c1):
        a, b = int(M.indptr[r0].item()), int(M.indptr[r1].item())
        cols = M.indices[a:b]
        return self.torch.unique(cols[(cols < c0) | (cols >= c1)])

    def _setup_dist(self, A, Q_list, colors, dense_coarse_max, min_rows, n_dist):
        """The levels from the GLOBAL operators, formed on every rank; this rank's row blocks are cut out of them."""
        torch, dev = self.torch, self.device
        W, rank = self.world, self.rank
        S = SD.DeviceSetup(torch, dev)
        L = self.nlevels
        A_host0, A_nat, Q_nat, QT_nat = SD.build_natural(S, A, Q_list)
        if self.smoother == "chebyshev":
            self._chebyshev_setup(S, A_nat)      # from the GLOBAL operators: the same bounds on every rank
        ns = [a.shape[0] for a in A_nat]
        self._global_n = ns
        self._global_nnzA = [a.nnz for a in A_nat]
        self._global_nnzQ = [q.nnz for q in Q_nat]
        if n_dist is None:
            n_dist = 0
            for l in range(L - 1):
                if ns[l] // W >= min_rows:
                    n_dist = l + 1
                else:
                    break
            n_dist = max(n_dist, 1)
        if not 1 <= n_dist <= L - 1:
            raise ValueError("n_dist must be between 1 and levels-1")
        self.colors = SD.level_colors(S, self.smoother, colors, A_host0, A_nat)
        offs = [PT.block_offsets(n, W) for n in ns]

        # ---- halo plans of the partitioned levels
        plans = []
        for l in range(int(n_dist)):
            o0, o1 = int(offs[l][rank]), int(offs[l][rank + 1])
            parts = [self._ext(A_nat[l], o0, o1, o0, o1)]
            c0, c1 = int(offs[l + 1][rank]), int(offs[l + 1][rank + 1])
            parts.append(self._ext(QT_nat[l], c0, c1, o0, o1))
            if l >= 1:
                f0, f1 = int(offs[l - 1][rank]), int(offs[l - 1][rank + 1])
                parts.append(self._ext(Q_nat[l - 1], f0, f1, o0, o1))
            ext = torch.unique(torch.cat(parts)).cpu().numpy()
            plans.append(PT.RankPlan(offs[l], rank, ext, self.colors[l]))

        def row_block(l, m):
            M, o = {"A": (A_nat, offs[l]), "Q": (Q_nat, offs[l]), "QT": (QT_nat, offs[l + 1])}[m]
            return self._rowblock(M[l], int(o[rank]), int(o[rank + 1]))

        self._build_levels(S, offs, plans, row_block, A_nat, Q_nat, QT_nat, dense_coarse_max)
        if self.keep_host:
            self._dev_A_nat = A_nat
            self._dev_Q_nat = Q_nat

    def _build_levels(self, S, offs, plans, row_block, A_nat, Q_nat, QT_nat, dense_coarse_max):
        """This rank's levels, from
          offs                   : partition.block_offsets of every level
          plans                  : the RankPlans of the partitioned levels 0 .. n_dist-1 (n_dist = len(plans))
          row_block(l, m)        : this rank's row block of A_l (m = "A"), of Q_l (m = "Q", the fine rows it owns) or of
                                   Q_l^T (m = "QT", the coarse rows it owns) as a DevCSR with global column ids; called
                                   once per block, level by level, and the block is dropped once it is packed, so a
                                   source that forms blocks on demand holds one at a time
          A_nat, Q_nat, QT_nat   : the replicated levels' operators in natural order (entries below n_dist not read)
        self.colors[l] (l >= n_dist) and self._global_n / _global_nnzA / _global_nnzQ must be set."""
        torch, dev = self.torch, self.device
        W, rank = self.world, self.rank
        L, Lp = self.nlevels, len(plans)
        ns = self._global_n
        self._setup = S
        self.n_dist, self.offsets, self.plans = Lp, offs, plans
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
        # global colour permutations of the replicated levels
        perms, iperms, cptrs = [None] * L, [None] * L, [None] * L
        for l in range(Lp, L):
            if self.colors[l] is not None:
                perms[l], iperms[l], cptrs[l] = S.color_perm(self.colors[l])
        dummy = torch.zeros(1, dtype=torch.int32, device=dev)
        lays[Lp] = _Layout(0, ns[Lp], iperms[Lp], ns[Lp], dummy, ns[Lp])

        # ---- partitioned levels: the row blocks (global column ids) are remapped to my level vector and packed
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
            blk = row_block(l, "A")
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
            blk = row_block(l, "Q")
            loc = SD.DevCSR((p.n_own, lays[l + 1].length), blk.indptr, self._remap(S, blk.indices, lays[l + 1]),
                            blk.values)
            lev.Q = S.to_sell(S.permute(loc, lev.perm, None))
            del blk, loc
            c0, c1 = int(offs[l + 1][rank]), int(offs[l + 1][rank + 1])
            blk = row_block(l, "QT")
            loc = SD.DevCSR((c1 - c0, lev.n_vec), blk.indptr, self._remap(S, blk.indices, lays[l]), blk.values)
            cperm = None
            if l + 1 < Lp and plans[l + 1].perm is not None:
                cperm = torch.from_numpy(plans[l + 1].perm).to(dev)
            lev.QT = S.to_sell(S.permute(loc, cperm, None))
            del blk, loc
            self._build_xfers(lev, l, everyone, offs, iperms, Lp)
            # which slices of A / Q / Q^T read halo columns (lets an exchange ride on the kernel that needs it)
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

    def _build_xfers(self, lev, l, everyone, offs, iperms, Lp):
        """mg_xfer descriptors of level l: one per colour, one for the whole halo, and the coarse hand-off."""
        torch, dev = self.torch, self.device
        p, rank, W = lev.plan, self.rank, self.world
        sends = {}
        for q in range(W):
            if q != rank and l < len(everyone[q]) and rank in everyone[q][l]:
                gids, ptr = everyone[q][l][rank]
                sends[q] = (torch.from_numpy(p.local_of_owned(gids)).to(dev), [int(v) for v in ptr])
        peers = sorted(set(p.neighbours) | set(sends))
        nc = p.ncolors
        lev.send_idx = sends
        lev.peers = peers

        def make(color):
            x = _lib.mg_xfer()
            x.npeers = len(peers)
            for k, q in enumerate(peers):
                x.peer[k] = q
                if q in sends:
                    idx, ptr = sends[q]
                    a, b = (0, ptr[-1]) if color is None else (ptr[color], ptr[color + 1])
                    x.d_send_idx[k] = idx.data_ptr() + 4 * a if b > a else None
                    x.send_cnt[k] = b - a
                if q in p.seg:
                    a, b = p.seg[q] if color is None else p.seg_color[(q, color)]
                    x.recv_off[k] = p.n_own + a
                    x.recv_cnt[k] = b - a
            return x

        d = _lib.mg_dist_level()
        d.n_halo = p.n_halo
        d.ncolors = nc
        if nc:
            arr = (_lib.mg_xfer * nc)(*[make(c) for c in range(nc)])
            self._keep.append(arr)
            d.xfer_color = ctypes.cast(arr, ctypes.POINTER(_lib.mg_xfer))
        xa = make(None)
        self._keep.append(xa)
        d.xfer_all = ctypes.pointer(xa)
        if l == Lp - 1:
            # all-gather of the restricted right-hand side into every rank's full coarse vector
            oc = offs[l + 1]
            ip = iperms[l + 1]
            n_own_c = int(oc[rank + 1] - oc[rank])
            lev.gather_tmp = torch.zeros(max(n_own_c, 1), dtype=torch.float64, device=dev)
            if ip is None:
                ip = torch.arange(int(oc[-1]), dtype=torch.int32, device=dev)
            lev.gather_iperm = ip
            xg = _lib.mg_xfer()
            for q in range(W):
                if q == rank:
                    continue
                k = xg.npeers
                xg.npeers += 1
                xg.peer[k] = q
                xg.send_cnt[k] = n_own_c
                cnt = int(oc[q + 1] - oc[q])
                xg.d_recv_idx[k] = ip.data_ptr() + 4 * int(oc[q]) if cnt else None
                xg.recv_cnt[k] = cnt
            self._keep.append(xg)
            d.xfer_gather = ctypes.pointer(xg)
            d.d_gather_tmp = lev.gather_tmp.data_ptr()
            d.d_gather_self_idx = ip.data_ptr() + 4 * int(oc[rank])
            d.n_gather_own = n_own_c
        lev.dist_struct = d

    def _host_block(self, host_vec):
        torch = self.torch
        p = self.levels[0].plan
        n0 = self._global_n[0]
        if isinstance(host_vec, torch.Tensor):
            v = host_vec.reshape(-1)
            if v.numel() == n0:
                v = v[p.o0:p.o1]
            return v
        v = np.asarray(host_vec, dtype=np.float64).reshape(-1)
        if v.size == n0:
            v = v[p.o0:p.o1]
        return np.ascontiguousarray(v)

    def _to_level0(self, host_vec, dst):
        blk = self._host_block(host_vec)
        if (blk.numel() if hasattr(blk, "numel") else blk.size) != self.n:
            raise ValueError("vector must have %d (global) or %d (owned block) entries" % (self._global_n[0], self.n))
        super()._to_level0(blk, dst)

    def set_x(self, x):
        """x must be the GLOBAL vector here: the halo entries are taken from it directly."""
        torch = self.torch
        lev = self.levels[0]
        v = x.numpy() if isinstance(x, torch.Tensor) else np.asarray(x, dtype=np.float64)
        v = v.reshape(-1)
        if v.size != self._global_n[0]:
            raise ValueError("set_x needs the global vector (%d entries)" % self._global_n[0])
        self._to_level0(v, lev.x)
        if lev.n_halo:
            lev.x[lev.n:].copy_(torch.from_numpy(np.ascontiguousarray(v[lev.plan.halo_gid])))

    def get_x_local(self, view=False):
        """owned block of the iterate, natural order, (n_own,1)"""
        return self._from_level0(self.levels[0].x, view)

    def get_x(self, view=False):
        """the GLOBAL iterate on every rank (blocks exchanged through the fabric: an API convenience, not a hot path)"""
        parts = self.fabric.allgather(self.get_x_local().reshape(-1))
        return np.concatenate(parts).reshape(-1, 1)

    # ------------------------------------------------------------------------------------------------
    def residual_norm(self):
        """||b - A x||_2 over all row blocks (Multigrid.py:62-63): fused residual + norm on the owned rows, summed
        over the ranks in rank order by the peer-memory all-reduce; one D2H of 8 bytes."""
        torch = self.torch
        _lib.check(self.lib.mg_vcycle_dist(ctypes.byref(self.comm.struct), self._level_structs, self.nlevels, None,
                                           ctypes.byref(self._norm_struct), _lib.stream_handle(torch)),
                   "mg_vcycle_dist (norm)")
        self._norm_host.copy_(self._norm_out, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return float(np.sqrt(self._norm_host.item()))

    def residual_vector(self):
        lev = self.levels[0]
        _lib.check(self.lib.mg_sell_residual(ctypes.byref(lev.A.struct), lev.x.data_ptr(), lev.b.data_ptr(),
                                             lev.r.data_ptr(), _lib.stream_handle(self.torch)), "mg_sell_residual")
        parts = self.fabric.allgather(self._from_level0(lev.r).reshape(-1))
        return np.concatenate(parts).reshape(-1, 1)

    def vcycle(self, params, nlevels=None, use_graph=True, with_norm=False, dry=False, norm_after=False):
        """One V-cycle as one program, optionally with the residual norm of the outer loop: with_norm -- of the iterate
        the program starts from, evaluated first; norm_after -- of the iterate the cycle leaves, its last colour's share
        summed by the last sweep (mg_dist_norm.after); read it with last_norm().  Every rank must make the same call.
        Captured into a CUDA graph per parameter set.  dry=True captures the program with its exchanges disabled
        (results are meaningless; bench.py times it to separate kernel time from exchange time)."""
        torch = self.torch
        with_norm = bool(with_norm or norm_after)
        self._norm_struct.after = 1 if norm_after else 0
        if nlevels is not None and int(nlevels) != self.nlevels:
            raise ValueError("a partitioned hierarchy runs all of its levels")
        L = self.nlevels
        st = _lib.stream_handle(torch)
        norm = ctypes.byref(self._norm_struct) if with_norm else None
        comm = ctypes.byref(self.comm.struct)
        if not use_graph:
            _lib.check(self.lib.mg_vcycle_dist(comm, self._level_structs, L, ctypes.byref(params), norm, st),
                       "mg_vcycle_dist")
            self.last_launches = int(self.lib.mg_last_launch_count())
            return
        key = (L, params.smoother, params.nu_pre, params.nu_post, params.omega, params.zero_guess_skip,
               params.reverse_post, params.x0_zero, bool(with_norm), bool(norm_after), bool(dry), self._cheby_key)
        g = self._graphs.get(key)
        if g is None:
            cap = torch.cuda.Stream(device=self.device)
            cap.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(cap):
                h = cap.cuda_stream
                _lib.check(self.lib.mg_graph_begin(h), "mg_graph_begin")
                self.comm.struct.dry_run = 1 if dry else 0
                try:
                    rc = self.lib.mg_vcycle_dist(comm, self._level_structs, L, ctypes.byref(params), norm, h)
                finally:
                    self.comm.struct.dry_run = 0
                launches = int(self.lib.mg_last_launch_count())
                out = ctypes.c_void_p()
                rc2 = self.lib.mg_graph_end(h, ctypes.byref(out))
                _lib.check(rc, "mg_vcycle_dist (capture)")
                _lib.check(rc2, "mg_graph_end")
            torch.cuda.current_stream().wait_stream(cap)
            g = (out, launches)
            self._graphs[key] = g
        _lib.check(self.lib.mg_graph_launch(g[0], st), "mg_graph_launch")
        self.last_launches = g[1]

    def _comm_ptr(self):
        return ctypes.byref(self.comm.struct)

    def last_norm(self):
        """sqrt of the squared residual norm the last with_norm program computed (synchronises)"""
        self._norm_host.copy_(self._norm_out, non_blocking=True)
        self.torch.cuda.current_stream().synchronize()
        return float(np.sqrt(self._norm_host.item()))

    def check(self):
        self.comm.check()

    def close(self):
        try:
            for g, _ in self._graphs.values():
                self.lib.mg_graph_destroy(g)
            self._graphs = {}
        finally:
            self.comm.close()

    # ------------------------------------------------------------------------------------------------
    def cycle_bytes(self, nu_pre, nu_post):
        """Algorithmic bytes of one outer iteration of the GLOBAL problem (SURVEY.md 8d formula, actual nnz)."""
        S = algorithmic_bytes_csr
        n, a, q = self._global_n, self._global_nnzA, self._global_nnzQ
        outer = S(a[0], n[0]) + 16 * n[0]
        total = outer
        per_level = []
        for l in range(self.nlevels - 1):
            b = (nu_pre + nu_post + 1) * (S(a[l], n[l]) + 24 * n[l])
            b += S(q[l], n[l + 1]) + 8 * n[l] + 8 * n[l + 1]
            b += S(q[l], n[l]) + 8 * n[l + 1] + 16 * n[l]
            per_level.append(b)
            total += b
        coarse = self.levels[-1].coarse_bytes + 16 * n[-1]
        total += coarse
        return {"total": total, "outer": outer, "levels": per_level, "coarse": coarse}

    def level_matrix(self, l):
        return SD.download_level_matrix(self, l)
