"""The device hierarchy setup at the sizes the benchmark runs it, stage by stage, against the host reference
(tests/setup_oracle.py): generators, Galerkin products (bit for bit against SciPy), first-fit colours (entry for entry
against the serial helper), colour permutations, the SELL-32 arrays of A, Q and Q^T, dinv, the level flags, and the
value dictionary, slice records, slice patterns and spec blocks DeviceSell attaches, compared by meaning.

Built the way bench.py builds: device generators (or host ones for quasi-L2 transfers), DeviceHierarchy with
multicolour Gauss-Seidel and the default first-fit colours, the default row floors (no MGB_*_MIN_ROWS overrides), so
that the production routes run.  Host memory stays bounded: every level is downloaded, compared and dropped before the
next one.  The per-level facts (rows, where the colouring ran, rounds, colours, which extras were attached) and the
peak host RSS are printed; with MGB_SETUP_SCALE_REPORT=<path> they are also appended there as JSON lines."""
import json
import os
import resource
import time

import numpy as np
import pytest

import setup_oracle as O

pytestmark = pytest.mark.gpu

DEVICE_COLOR_MIN_ROWS = 50000       # setup_device.level_colors: smaller levels take the serial helper
COLOR_BATCH = 128                   # mg_color_first_fit: rounds between two looks at the progress counter

CONFIGS = [
    pytest.param(dict(N=8192, levels=6, generate="device", coef="constant", transfer="linear", boundary="dirichlet"),
                 id="8193-constant-linear"),
    pytest.param(dict(N=8192, levels=6, generate="device", coef="variable", transfer="linear", boundary="dirichlet"),
                 id="8193-variable-linear"),
    pytest.param(dict(N=4096, levels=5, generate="host", coef="constant", transfer="quasi", boundary="dirichlet"),
                 id="4097-constant-quasi"),
    pytest.param(dict(N=4096, levels=6, generate="device", coef="constant", transfer="linear", boundary="neumann"),
                 id="4097-neumann-linear"),
]


def peak_rss_gb():
    return resource.getrusage(resource.RUSAGE_SELF).ru_maxrss / 2 ** 20


def report(rec):
    print(json.dumps(rec))
    path = os.environ.get("MGB_SETUP_SCALE_REPORT")
    if path:
        with open(path, "a") as f:
            f.write(json.dumps(rec) + "\n")


def host(t):
    return None if t is None else t.cpu().numpy()


@pytest.fixture
def recorders(monkeypatch):
    """Rounds of every device colouring (by level rows) and the pattern_records calls of every DeviceSell (the sample
    call first when there is one), recorded by wrapping the product functions for the test only."""
    from learnmultigrid_b200 import _lib, engine, formats as F, setup_device as SD
    rounds, patterns, stack = {}, {}, []
    ff = SD.DeviceSetup.first_fit_colors

    def first_fit(self, A, *a, **k):
        try:
            out = ff(self, A, *a, **k)
        except _lib.MgError:
            rounds[A.shape[0]] = None
            raise
        rounds[A.shape[0]] = self.last_color_rounds
        return out
    attach = engine.DeviceSell._attach_patterns

    def attach_patterns(self):
        stack.append([])
        try:
            attach(self)
        finally:
            patterns[id(self)] = stack.pop()
    pr = F.pattern_records

    def pattern_records(torch, cols, vals, nrows, length, *a, **k):
        out = pr(torch, cols, vals, nrows, length, *a, **k)
        if stack:
            stack[-1].append((int(nrows), int(out[-1])))
        return out
    monkeypatch.setattr(SD.DeviceSetup, "first_fit_colors", first_fit)
    monkeypatch.setattr(engine.DeviceSell, "_attach_patterns", attach_patterns)
    monkeypatch.setattr(F, "pattern_records", pattern_records)
    return rounds, patterns


def same_csr(got, want, what, rtol=None):
    assert got.shape == want.shape, "%s: shape %s, reference %s" % (what, got.shape, want.shape)
    assert np.array_equal(got.indptr, want.indptr), "%s: row pointers differ" % what
    assert np.array_equal(got.indices, want.indices), "%s: sparsity pattern differs" % what
    if rtol is None:
        assert np.array_equal(got.data.view(np.int64), np.asarray(want.data, np.float64).view(np.int64)), \
            "%s: values differ (max %.3e)" % (what, np.abs(got.data - want.data).max())
    else:
        np.testing.assert_allclose(got.data, want.data, rtol=rtol, atol=0, err_msg=what)


def spec(st, nb):
    rows = [st.h_spec_row[k] for k in range(nb + 1)]
    rec = [st.h_spec_rec[k] for k in range(9 * nb)]
    vals = None if not st.h_spec_vals else np.array([st.h_spec_vals[k] for k in range(8 * nb)])
    return rows, rec, vals


def check_matrix(what, dev, ref, blocks, patterns):
    """SELL arrays exactly, then the value dictionary, slice records, slice patterns and spec blocks by meaning;
    returns the report entry of the matrix.  blocks: the colour blocks of the level the rows belong to.  A level
    operator's offset records are spec'd per colour block (its launches run over them); a transfer operator's offset
    records keep the one block of the whole matrix, its slice patterns get the colour blocks."""
    from learnmultigrid_b200.engine import DeviceSell
    assert np.array_equal(host(dev.slice_ptr), ref["slice_ptr"]), "%s: SELL slice_ptr" % what
    assert np.array_equal(host(dev.cols), ref["cols"]), "%s: SELL cols" % what
    assert np.array_equal(host(dev.vals).view(np.int64), ref["vals"].view(np.int64)), "%s: SELL vals" % what
    assert (dev.max_len, dev.uniform_len) == (ref["max_len"], ref["uniform_len"]), "%s: max_len / uniform_len" % what
    vd = O.value_dict(ref)
    O.check_value_dict(vd, ref, host(dev.val_idx), host(dev.val_table), dev.distinct_values)
    sr = O.slice_records(ref, vd["attached"])
    O.check_slice_records(sr, ref, host(dev.slice_rec), host(dev.rec_table), host(dev.rec_vals))
    if sr["attached"]:
        square = ref["shape"][0] == ref["shape"][1]
        O.check_offset_spec_blocks(blocks if square else [0, ref["nrows"]], *spec(dev.struct, dev.struct.n_spec), host(dev.slice_rec),
                                   host(dev.rec_table), host(dev.rec_vals))
    pr = O.pattern_records(ref, sr["attached"])
    log = patterns.get(id(dev), [])
    nsl = len(ref["slice_ptr"]) - 1
    sampled = bool(log) and nsl > 2 * DeviceSell.PATTERN_SAMPLE and log[0][0] == DeviceSell.PATTERN_SAMPLE * 32
    assert sampled == pr["sampled"], "%s: sampled pattern pre-check ran: %s, reference %s" % (what, sampled, pr["sampled"])
    if sampled:
        assert (2 * log[0][1] >= DeviceSell.PATTERN_SAMPLE) == (2 * pr["sample_slices"] >= DeviceSell.PATTERN_SAMPLE), \
            "%s: the sample's decision differs (%d vs %d slices)" % (what, log[0][1], pr["sample_slices"])
    ids = host(dev.pat_rec)
    delta = pvals = base = None
    if ids is not None:
        L = dev.uniform_len
        nrec = -int(dev.struct.nrec)
        tab = host(dev.pat_table)
        delta, base, pvals = tab[:nrec * L * 32].reshape(nrec, L, 32), tab[nrec * L * 32:], host(dev.pat_vals)
    O.check_pattern_records(pr, ref, ids, delta, pvals, base)
    if pr["attached"]:
        O.check_pattern_spec_blocks(blocks, *spec(dev.struct, dev.struct.n_spec)[:2], ids, pr["group"])
    return {"rows": ref["nrows"], "max_len": ref["max_len"], "uniform_len": ref["uniform_len"], "value_dict": vd["attached"],
            "distinct_values": vd["count"] if vd["count"] <= 256 else ">256",
            "slice_records": sr["attached"], "implied_values": bool(sr.get("with_values")),
            "pattern_records": pr["attached"], "pattern_sample": pr["sampled"]}


def generate(cfg):
    """the operators as bench.py generates them; the host generators' (reference) level-0 operator, and Q_l one at a
    time"""
    from learnmultigrid_b200 import formats as F, problems as P, problems_device as PD
    N, L = cfg["N"], cfg["levels"]
    hcoef = None if cfg["coef"] == "constant" else P.variable_coefficient
    if cfg["generate"] == "device":
        dcoef = None if cfg["coef"] == "constant" else PD.variable_coefficient
        return (PD.structured_laplacian_2d(N, dcoef, boundary=cfg["boundary"]), PD.structured_hierarchy_2d(N, L),
                lambda: P.structured_laplacian_2d(N, hcoef, boundary=cfg["boundary"]),
                lambda l: P.linear_P_2d(N >> l))
    A = P.structured_laplacian_2d(N, hcoef, boundary=cfg["boundary"])
    Qs = P.structured_hierarchy_2d(N, L, transfer=cfg["transfer"])
    return A, Qs, lambda: F.solver_csr(A), lambda l: F.canonical_csr(Qs[l])


@pytest.mark.parametrize("cfg", CONFIGS)
def test_device_setup_matches_host_reference(cfg, recorders, request):
    import torch
    import scipy.sparse as sp
    from learnmultigrid_b200 import _lib, formats as F
    from learnmultigrid_b200.engine import DeviceHierarchy
    t0 = time.perf_counter()
    rounds, patterns = recorders
    L = cfg["levels"]
    A, Qs, host_A, host_Q = generate(cfg)
    null = {"null_space": "constant"} if cfg["boundary"] == "neumann" else {}
    h = DeviceHierarchy(A, Qs, smoother="mcgs", keep_host=True, **null)
    del A, Qs
    torch.cuda.synchronize()
    t_build = time.perf_counter() - t0
    S = h._setup
    name = request.node.callspec.id

    # 1. generators: patterns exactly, values exactly (rtol 1e-14 where the device's sin() differs in the last bits);
    # Q_l is compared when its level is checked
    rtol = 1e-14 if cfg["coef"] == "variable" and cfg["generate"] == "device" else None
    Aref = S.download(h._dev_A_nat[0])
    same_csr(Aref, host_A(), "%s: level-0 operator against the host generator" % name, rtol)
    Aref = F.canonical_csr(Aref)

    rows = []
    prev = None                      # level l-1: perm, iperm, colour offsets
    Q = None                         # Q_{l-1}, downloaded
    for l in range(L):
        lev = h.levels[l]
        if l > 0:
            Q = S.download(h._dev_Q_nat[l - 1])
            same_csr(Q, host_Q(l - 1), "%s: Q_%d against the host generator" % (name, l - 1))
            # 2. Galerkin: bit for bit against SciPy, the chain started from the device's own level-0 operator, which
            # the reference stores CSC (Solver.py:18)
            chain = sp.csc_matrix(Aref) if l == 1 else Aref
            Aref = None
            Aref = O.galerkin(chain, Q)
            del chain
            same_csr(S.download(h._dev_A_nat[l]), Aref, "%s: Galerkin level %d" % (name, l))
        n = Aref.shape[0]
        row = {"config": name, "level": l, "rows": n}
        cur = None
        if l < L - 1:
            # 3. colours, entry for entry; the device path for every level of at least 50 000 rows
            col, nc = O.colors(Aref)
            on_device = n >= DEVICE_COLOR_MIN_ROWS
            assert (n in rounds and rounds[n] is not None) == on_device, \
                "%s: level %d (%d rows) coloured on the %s" % (name, l, n, "device" if n in rounds else "host")
            assert np.array_equal(h.colors[l], col), "%s: level %d colours differ from the serial helper" % (name, l)
            assert len(lev.color_ptr) - 1 == nc, "%s: level %d: %d colours, reference %d" % (
                name, l, len(lev.color_ptr) - 1, nc)
            row.update(coloring="device" if on_device else "host", rounds=rounds.get(n), colors=nc)
            # 4. permutation
            perm, iperm, cptr = O.permutation(col)
            assert np.array_equal(host(lev.perm), perm), "%s: level %d permutation" % (name, l)
            assert np.array_equal(np.asarray(lev.color_ptr, np.int64), cptr), "%s: level %d colour offsets" % (name, l)
            dperm, diperm, dcptr = S.color_perm(h.colors[l])
            assert np.array_equal(host(dperm), perm) and np.array_equal(host(diperm), iperm), \
                "%s: level %d inverse permutation" % (name, l)
            del dperm, diperm
            # 6. dinv and level flags
            assert np.array_equal(host(lev.dinv).view(np.int64), O.dinv(Aref, perm).view(np.int64)), \
                "%s: level %d dinv" % (name, l)
            proper, diag = O.level_flags(Aref, col)
            want = (_lib.MG_LEVEL_PROPER_COLORING if proper else 0) | (_lib.MG_LEVEL_NONZERO_DIAG if diag else 0)
            assert lev.flags == want, "%s: level %d flags %d, reference %d" % (name, l, lev.flags, want)
            # 5 + 7. SELL of A and its extras
            ref = O.sell(Aref, perm, iperm)
            row["A"] = check_matrix("%s: A_%d" % (name, l), lev.A, ref, cptr, patterns)
            del ref
            cur = (perm, iperm, cptr)
        if l > 0:
            # 5 + 7. SELL of Q_{l-1} (rows of level l-1) and Q_{l-1}^T (rows of level l), extras, pattern blocks
            pl = h.levels[l - 1]
            perm_c, iperm_c = (None, None) if cur is None else cur[:2]
            ref = O.sell(Q, prev[0], iperm_c)
            row["Q"] = check_matrix("%s: Q_%d" % (name, l - 1), pl.Q, ref, prev[2], patterns)
            del ref
            ref = O.sell(F.transpose_csr(Q), perm_c, prev[1])
            row["QT"] = check_matrix("%s: Q_%d^T" % (name, l - 1), pl.QT, ref, [0, n] if cur is None else cur[2],
                                     patterns)
            del ref, Q
            Q = None
        prev = cur
        rows.append(row)
    del Aref
    lv0 = rows[0]
    assert lv0["coloring"] == "device" and lv0["rounds"] > COLOR_BATCH, \
        "%s: level 0 took %s rounds, not more than one batch of %d" % (name, lv0["rounds"], COLOR_BATCH)
    if cfg["coef"] == "constant" and cfg["transfer"] == "linear" and cfg["N"] == 8192:
        # the headline: dictionary on A and the transfers, implied values, sampled pattern records on the transfers
        assert rows[0]["A"]["value_dict"] and rows[0]["A"]["implied_values"]
        assert rows[1]["Q"]["value_dict"] and rows[1]["Q"]["pattern_records"] and rows[1]["Q"]["pattern_sample"]
        assert rows[1]["QT"]["pattern_records"] and rows[1]["QT"]["pattern_sample"]
    if cfg["coef"] == "variable":
        assert not rows[0]["A"]["value_dict"]
    if cfg["transfer"] == "quasi":
        assert rows[1]["A"]["max_len"] > 8 and not rows[1]["A"]["slice_records"]
    for r in rows:
        report(r)
    del h
    torch.cuda.empty_cache()
    report({"config": name, "build_s": round(t_build, 1), "test_s": round(time.perf_counter() - t0, 1),
            "peak_rss_gb": round(peak_rss_gb(), 2)})


@pytest.mark.parametrize("distinct", [256, 257])
def test_value_dict_256_and_257_distinct_values_on_the_device(distinct):
    """mg_value_dict_build at the dictionary floor: +0.0 and -0.0 are two entries; 256 distinct values take a
    dictionary that decodes to the same bits, 257 take none"""
    import torch
    from learnmultigrid_b200 import formats as F
    from learnmultigrid_b200.engine import DeviceSell
    n = DeviceSell.VALUE_DICT_MIN_ROWS
    v = np.concatenate([[0.0, -0.0], 1.0 + np.arange(distinct - 2) / 7.0])
    vals = np.resize(np.random.default_rng(2).permutation(v), 2 * n)
    cols = np.stack([np.arange(n), (np.arange(n) + 5) % n], axis=1).ravel()
    A = F.raw_csr(np.arange(n + 1) * 2, cols, vals, (n, n))
    dev = DeviceSell(torch, A, torch.device("cuda", 0))
    ref = O.sell(A)
    assert np.array_equal(host(dev.vals).view(np.int64), ref["vals"].view(np.int64))
    vd = O.value_dict(ref)
    assert vd["count"] == distinct and vd["attached"] == (distinct == 256)
    O.check_value_dict(vd, ref, host(dev.val_idx), host(dev.val_table), dev.distinct_values)
