"""The device NN transfer-operator builder (learnmultigrid_b200/neural2d.py, csrc/nn_kernels.cu) at the sizes the
irregular-mesh benchmark runs it at, stage by stage against the float64 host reference of tests/nn_oracle.py.

The golden vectors of test_gpu_neural2d.py stop at 289 nodes: there the independent set is found within one batch of
rounds, every extraction and contribution launch is one or two CTAs, the radix sorts of fill_B need a handful of bits,
and the coarser levels have a few dozen nodes.  Here, on a few hundred thousand nodes, all of that scales up, and every
stage must still agree exactly: coarse sets and maps, patches, fill indices, not_last flags, predictions, d_neighs, B
and Q bit for bit, and the next-level mass matrix before and after pre_process's cut.

Sizes: irregular_p1_2d(512), 263,169 nodes, with both predictors, and irregular_p1_2d(1024), 1,050,625 nodes, with the
mass surrogate; 4 levels each (263k / 66k / 17k / 4k and 1.05 M / 263k / 66k / 17k rows).  The host side (mesh and
serial reference) takes a few seconds per case at N = 1024.  On these meshes pre_process keeps the coarse patterns
symmetric; the patch-variant mesh is where its cut leaves unsymmetric ones (checked there).
"""
import numpy as np
import pytest
import scipy.sparse as sp

import nn_oracle as O
from test_assembly_golden import GoldenMesh

pytestmark = pytest.mark.gpu


class DensePredictor:
    """A deterministic stand-in for a trained network that fills all 31 outputs: values in [1, 2), and one in 32 each
    exactly 0, +0.5 and -0.5, so that runs of contributions to one B entry cancel to exactly 0 (then start again from
    the next contribution, or leave no entry) and some entries of B end negative.  A hash of the patch's own features
    picks the values, so a patch gets the same prediction on the host and through the device pipeline.
    signed: the outputs that may take +-0.5 (the others take 1.5 instead)."""

    def __init__(self, signed=slice(None)):
        self.signed = signed

    def predict(self, X):
        X = np.ascontiguousarray(X, dtype=np.float64)
        key = X[:, :7].view(np.uint64).sum(axis=1, dtype=np.uint64)
        h = key[:, None] * np.uint64(0x9E3779B97F4A7C15) + np.arange(31, dtype=np.uint64) * np.uint64(0xBF58476D1CE4E5B9)
        h ^= h >> np.uint64(29)
        h *= np.uint64(0x94D049BB133111EB)
        u = ((h >> np.uint64(40)) % np.uint64(32)).astype(np.int64)
        out = 1.0 + u / 32.0
        out[u == 0] = 0.0
        neg, pos = np.full(u.shape, 1.5), np.full(u.shape, 1.5)
        neg[:, self.signed] = -0.5
        pos[:, self.signed] = 0.5
        out[u == 1] = neg[u == 1]
        out[u == 2] = pos[u == 2]
        return out


# ---- comparisons ---------------------------------------------------------------------------------------------------
def same(got, want, what):
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape, "%s: shape %s, reference %s" % (what, got.shape, want.shape)
    bad = np.flatnonzero(got.ravel() != want.ravel())
    assert bad.size == 0, "%s: %d of %d entries differ, first at flat index %d: %r, reference %r" % (
        what, bad.size, got.size, bad[0], got.ravel()[bad[0]], want.ravel()[bad[0]])


def same_csr(got, want, what):
    assert got.shape == want.shape, "%s: shape %s, reference %s" % (what, got.shape, want.shape)
    same(got.indptr, want.indptr, what + " row pointer")
    same(got.indices, want.indices, what + " columns")
    same(got.data, want.data, what + " values")


def host(t):
    return t.cpu().numpy()


def compare_hierarchy(nb, Qs, ref):
    """every stage of every level of nb.define_hierarchy(..., keep_intermediates=True) against the oracle's"""
    assert len(Qs) == len(ref) == len(nb.trace)
    for l, (Q, r, tr) in enumerate(zip(Qs, ref, nb.trace)):
        lv = "level %d: " % l
        same_csr(nb.download(tr["M"]), r["M"], lv + "M (cut)" if l else lv + "M")
        same(host(tr["cmap"]), r["cmap"], lv + "cmap")
        same(host(tr["clist"]), r["clist"], lv + "clist")
        same(host(tr["fill"]), r["fill"], lv + "fill")
        same(host(tr["patches"]), r["patches"], lv + "patches")
        nl = tr["not_last"]
        same(host(nl) if nl is not None else np.zeros(len(r["not_last"]), dtype=np.int32), r["not_last"],
             lv + "not_last")
        same(host(tr["pred"]), r["pred"], lv + "predictions")
        same(host(tr["dneigh"]), r["dneigh"], lv + "d_neighs")
        same_csr(nb.download(tr["B"]), r["B"], lv + "B")
        same_csr(nb.download(Q), r["Q"], lv + "Q")
        if l + 1 < len(ref):
            # the product define_hierarchy formed from these operands, before the next level's cut
            full = nb.S.galerkin(tr["M"], Q, nb.S.transpose(Q))
            same_csr(nb.download(full), ref[l + 1]["M_full"], lv + "Q^T M Q")


def key_bits(largest):
    """bits an LSD radix sort needs for keys 0 .. largest"""
    return max(1, int(largest).bit_length())


# ---- meshes --------------------------------------------------------------------------------------------------------
def split_triangles(p, conn, tris):
    """insert the centroid of each listed triangle (new nodes numbered after all others, in list order) and replace the
    triangle by the three it spans with the centroid"""
    tris = np.asarray(tris)
    assert len(np.unique(tris)) == len(tris)
    t = conn[tris]
    g = len(p) + np.arange(len(tris))
    new_p = p[t].mean(axis=1)
    keep = np.ones(len(conn), dtype=bool)
    keep[tris] = False
    sub = np.concatenate([np.stack([t[:, 0], t[:, 1], g], axis=1), np.stack([t[:, 1], t[:, 2], g], axis=1),
                          np.stack([t[:, 2], t[:, 0], g], axis=1)])
    return np.vstack([p, new_p]), np.vstack([conn[keep], sub])


def triangles_of(conn, v):
    return np.flatnonzero((conn == v).any(axis=1))


def mass_matrix(p, conn):
    from learnmultigrid_b200.assembly.MassMatrix import MassMatrix
    from learnmultigrid_b200.assembly.Quadrature import Quadrature2D
    from learnmultigrid_b200.assembly.ShapeFunction import FunctionTriangle
    from learnmultigrid_b200 import formats as F
    M = MassMatrix(GoldenMesh(p, conn)).compute_mass_2d(FunctionTriangle(1), Quadrature2D(3), format="csr")
    return F.canonical_csr(M)


H = 320                             # Mesh2D(H * H): (H + 1)^2 = 103,041 vertices


def grid_mesh():
    from learnmultigrid_b200.mesh.Mesh2D import Mesh2D
    m = Mesh2D(H * H)
    return np.asarray(m.get_points(), dtype=np.float64), np.asarray(m.get_connections(), dtype=np.int64)


def coarse_vertex(q):
    """the vertex of coarse index q: the independent set of Mesh2D is every second vertex of every second grid line,
    and centroids (numbered last, each next to a coarse vertex) never join it"""
    per_row = H // 2 + 1
    return (2 * (q // per_row)) * (H + 1) + 2 * (q % per_row)


def variant_mesh():
    """Mesh2D(320^2) with centroids inserted into k of the triangles around chosen coarse vertices, so that these
    have 6 + k neighbours (interior: k = 1..6, valence 7..12) or 4 + 3 (boundary vertices of the last coarse rows and
    the first, valence 7).  The chosen coarse indices are spread over the 128-node blocks of the extraction launches,
    the last partial block included.  Returns (p, conn, {coarse index: extra patch variants})."""
    p, conn = grid_mesh()
    nc = (H // 2 + 1) ** 2
    per_row = H // 2 + 1
    chosen, extra = {}, {}                                        # triangles split, extra variants
    for q in range(nc):
        r, c = 2 * (q // per_row), 2 * (q % per_row)
        interior = 0 < r < H and 0 < c < H
        if interior and q % 7 == 3:
            chosen[q] = extra[q] = 1 + (q // 7) % 6
        elif not interior and 0 < c < H and (q < 128 or q >= nc - 65) and q % 5 == 0:
            chosen[q], extra[q] = 3, 1                             # all three triangles of a boundary vertex
    chosen[nc - 2], extra[nc - 2] = 3, 1                           # next to the last coarse node
    ne = len(conn)
    around = sp.csr_matrix((np.ones(3 * ne), (conn.ravel(), np.repeat(np.arange(ne), 3))), shape=(len(p), ne))
    tris = []
    for q, k in sorted(chosen.items()):
        v = coarse_vertex(q)
        t = around.indices[around.indptr[v]:around.indptr[v + 1]]
        assert len(t) in (3, 6) and len(t) >= k
        tris.extend(t[:k])
    p, conn = split_triangles(p, conn, tris)
    return p, conn, extra


# ---- fixtures ------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def nb():
    import torch
    assert torch.cuda.is_available()
    from learnmultigrid_b200.neural2d import NeuralBuilder
    return NeuralBuilder()


_meshes = {}


def irregular(N):
    """irregular_p1_2d(N); the last one generated is kept (the cases run grouped by N)"""
    from learnmultigrid_b200 import problems as P
    if N not in _meshes:
        _meshes.clear()
        _meshes[N] = P.irregular_p1_2d(N, seed=7)
    return _meshes[N]


def predictor_of(name, M):
    from learnmultigrid_b200.neural2d import MassSurrogate
    if name == "mass":
        return MassSurrogate(), np.zeros(43), np.ones(43)
    scale = float(M.data.max())
    # on meshes with patch variants only the coarse node's own entry (output 0, which only the node's patches feed)
    # changes sign: fine rows with two entries of +-0.5 would sum to 0
    model = DensePredictor() if name == "dense" else DensePredictor(signed=slice(0, 1))
    return model, np.full(43, 0.25 * scale), np.full(43, scale)


# ---- tests ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N,predictor", [(512, "mass"), (512, "dense"), (1024, "mass")])
def test_irregular_mesh_hierarchy_matches_oracle_at_scale(nb, N, predictor):
    """4 levels: level 0 on the refined mesh, levels 1-3 through the cut.  The parents, numbered first, are independent
    on the refined mesh, so level 0's set takes two rounds; the coarser levels inherit the grid-line numbering of the
    parent mesh, whose dependency chains need several batches of rounds"""
    M = irregular(N)["M"]
    model, mean, std = predictor_of(predictor, M)
    ref = O.define_hierarchy(M, model, mean, std, 4)
    Qs = nb.define_hierarchy(M, model, mean, std, 4, keep_intermediates=True)
    # the sizes land where the kernels care
    assert max(tr["rounds"] for tr in nb.trace) > 16               # more than one batch of rounds ran
    for r in ref:
        n, nc = r["M"].shape[0], len(r["clist"])
        assert nc % 128 != 0                                       # the last extraction CTA is partial
        assert key_bits(n) != key_bits(nc - 1)                     # row (incl. the unused row n) and column keys
    if predictor == "dense":
        assert all(r["stats"]["cancelled"] > 0 and r["stats"]["dropped"] > 0 for r in ref)
        assert all(r["B"].data.min() < 0 for r in ref)
    compare_hierarchy(nb, Qs, ref)


@pytest.mark.parametrize("predictor", ["mass", "dense-diagonal"])
def test_patch_variants_at_scale(nb, predictor):
    """~3,700 coarse vertices with 7..12 neighbours in a 116k-node mesh: extra patch variants in every extraction CTA,
    the last partial one included; with the dense predictor the variants of a node feed its own entry of B several
    times, so that runs cancel to 0 and start again"""
    p, conn, chosen = variant_mesh()
    M = mass_matrix(p, conn)
    assert M.shape[0] > 100_000
    model, mean, std = predictor_of(predictor, M)
    ref = O.define_hierarchy(M, model, mean, std, 3)
    Qs = nb.define_hierarchy(M, model, mean, std, 3, keep_intermediates=True)
    r0 = ref[0]
    nc = len(r0["clist"])
    assert np.array_equal(r0["clist"][sorted(chosen)], [coarse_vertex(q) for q in sorted(chosen)])
    # the variant layout the device must reproduce: variants 1.. of each node behind the nc regular patches, in node
    # order, each node's patches flagged not_last except its last one
    extra = np.zeros(nc, dtype=np.int64)
    for q, k in chosen.items():
        extra[q] = k
    degree = np.diff(M.indptr)[r0["clist"]] - 1
    assert np.array_equal(np.maximum(degree - 6, 0), extra)           # valence 6 + k exactly where chosen
    assert set(extra[extra > 0]) == set(range(1, 7)) and len(chosen) > 3000
    assert np.array_equal(r0["fill"][nc:, 0], np.repeat(r0["clist"], extra))
    blocks = np.unique(np.flatnonzero(extra) // 128)
    assert blocks[-1] == (nc - 1) // 128 and nc % 128 != 0 and len(blocks) == (nc + 127) // 128
    last = nc + np.cumsum(extra) - 1                               # row of each variant node's last patch
    want_nl = np.zeros(len(r0["fill"]), dtype=np.int32)
    want_nl[np.flatnonzero(extra)] = 1
    want_nl[nc:] = 1
    want_nl[last[extra > 0]] = 0
    assert np.array_equal(r0["not_last"], want_nl)
    # the surviving d_neighs are those of the last variant, and they differ from the first variant's for many nodes
    def dn_of(rows):
        f = r0["fill"][rows, 7:13]
        c = np.where(f >= 0, r0["cmap"][np.maximum(f, 0)], -1)
        return np.array([np.concatenate([x[x >= 0], -np.ones(6 - (x >= 0).sum(), dtype=np.int32)]) for x in c])
    vn = np.flatnonzero(extra)
    assert np.array_equal(r0["dneigh"][vn], dn_of(last[vn]))
    assert (dn_of(vn) != dn_of(last[vn])).any(axis=1).sum() > 100
    pattern = (ref[1]["M"] != 0).astype(np.int8)
    assert (pattern - pattern.T).nnz > 0                           # the cut left an unsymmetric pattern
    if predictor != "mass":
        assert r0["stats"]["restarts"] > 0
    compare_hierarchy(nb, Qs, ref)
    # not_last derived from the fill indices instead of taken from the variant kernel
    tr = nb.trace[0]
    B2, dn2 = nb.fill_B(tr["pred"], tr["fill"], tr["cmap"], M.shape[0], nc)
    same(host(dn2), r0["dneigh"], "d_neighs (derived not_last)")
    same_csr(nb.download(B2), r0["B"], "B (derived not_last)")


def test_device_assembled_mass_matrix_at_scale(nb):
    """the path of bench.py: M assembled on the device and handed over as a DevCSR (nothing uploaded); the oracle gets
    the same matrix downloaded"""
    from learnmultigrid_b200.assembly_device import DeviceAssembler
    from learnmultigrid_b200.assembly.Quadrature import Quadrature2D
    from learnmultigrid_b200.assembly.ShapeFunction import FunctionTriangle
    from learnmultigrid_b200.neural2d import MassSurrogate
    asm = DeviceAssembler()
    Md = asm.mass(*asm.mesh_to_device(irregular(512)["mesh"]), FunctionTriangle(1), Quadrature2D(3))
    Mh = asm.S.download(Md)
    assert Mh.shape[0] == 513 ** 2 and Mh.has_sorted_indices
    ref = O.define_hierarchy(Mh, MassSurrogate(), np.zeros(43), np.ones(43), 4)
    Qs = nb.define_hierarchy(Md, MassSurrogate(), np.zeros(43), np.ones(43), 4, keep_intermediates=True)
    assert nb.trace[0]["M"] is Md
    compare_hierarchy(nb, Qs, ref)


def test_thirteen_neighbours_are_reported_at_scale(nb):
    """one coarse vertex with 13 neighbours among 100k valid nodes: extraction raises MgError naming the limit and
    define_hierarchy returns nothing"""
    from learnmultigrid_b200 import _lib
    from learnmultigrid_b200.neural2d import MassSurrogate
    p, conn = grid_mesh()
    per_row = H // 2 + 1
    v = coarse_vertex((per_row // 2) * per_row + per_row // 2)          # a coarse vertex in the middle
    p, conn = split_triangles(p, conn, triangles_of(conn, v))           # 12 neighbours
    p, conn = split_triangles(p, conn, triangles_of(conn, v)[:1])       # 13
    M = mass_matrix(p, conn)
    assert (M[v] > 0).sum() - 1 == 13 and M.shape[0] > 100_000
    Md = nb.upload(M)
    cmap, clist, nc = nb.coarsen(Md)
    assert int(cmap[v]) >= 0
    with pytest.raises(_lib.MgError, match="more than 12 neighbours"):
        nb.extract(Md, cmap, clist)
    with pytest.raises(_lib.MgError, match="more than 12 neighbours"):
        nb.define_hierarchy(Md, MassSurrogate(), np.zeros(43), np.ones(43), 3)
