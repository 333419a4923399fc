"""CPU suite (-m "not gpu"): the oracle against the reference's golden vectors, the C ABI
surface, the host-side MPS reader and the multi-rank host logic (gloo)."""
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, load_golden

from clp_b200 import generators as G
from oracle import oracle as O

MANIFEST = json.load(open(os.path.join(ROOT, "tests", "golden", "manifest.json")))
SMALL = [k for k, v in MANIFEST.items() if v["m"] * v["n"] < 4_000_000 and k != "NQueens-100"]


def test_unit_test_3x5_factorize_ftran():
    """src/unitTest.cpp:1415-1482: basis {c0,c1,c4} -> colsol = {20/7, 3, 0, 0, 23/7}."""
    lp = load_golden("unitTest-3x5")
    o = O.OracleSimplex(lp)
    rc, pv = o.factorize([0, 1, 4])
    assert rc == 0
    # rows are equalities 14,3,3 and are nonbasic at that value: B x_B = +rowvalue (slack col -e_i)
    x = o.ftran(lp.row_lower.copy())
    col = np.zeros(5)
    for p, seq in enumerate(pv):
        col[seq] = x[p]
    np.testing.assert_allclose(col, [20.0 / 7.0, 3.0, 0.0, 0.0, 23.0 / 7.0], rtol=1e-12, atol=1e-12)


@pytest.mark.parametrize("name", SMALL)
def test_oracle_matches_reference_values(name):
    lp = load_golden(name)
    o = O.OracleSimplex(lp)
    st = o.dual()
    assert st == lp.expect_status
    if st == 0:
        tol = 1e-4 if MANIFEST[name]["objective_source"] == "reference" else 1e-8
        assert abs(o.objective_value - lp.known_objective) <= tol * (1 + abs(lp.known_objective))
        assert O.kkt_violations(lp, o.column_solution(), o.row_activity(), o.reduced_cost()) == 0


def test_oracle_planted_random_lp():
    lp = G.random_sparse_lp(300, 3000, 0.02, 7)
    o = O.OracleSimplex(lp)
    assert o.dual() == 0
    assert abs(o.objective_value - lp.known_objective) <= 1e-8 * (1 + abs(lp.known_objective))


def test_oracle_ft_update_consistency():
    """FTRAN/BTRAN after Forrest-Tomlin updates == FTRAN/BTRAN after refactorizing the same basis."""
    lp = G.random_sparse_lp(120, 600, 0.05, 3)
    rng = np.random.default_rng(0)
    o = O.OracleSimplex(lp)
    basis = list(range(lp.n, lp.n + lp.m))
    rc, pv = o.factorize(basis)
    assert rc == 0
    entering = rng.choice(lp.n, size=40, replace=False)
    for q in entering:
        col = np.zeros(lp.m)
        col[lp.row_index[lp.col_start[q]:lp.col_start[q + 1]]] = lp.element[lp.col_start[q]:lp.col_start[q + 1]]
        a = o.ftran(col)
        r = int(np.argmax(np.abs(a)))
        assert o.replace_column(int(q), r) in (0, 1)
        pv[r] = q
    b = rng.standard_normal(lp.m)
    x1, y1 = o.ftran(b), o.btran(b)
    o2 = O.OracleSimplex(lp)
    rc, pv2 = o2.factorize(pv)
    assert rc == 0
    x2, y2 = o2.ftran(b), o2.btran(b)
    # same basis, possibly different pivot-row labels: compare per variable
    xv1 = {int(s): x1[p] for p, s in enumerate(pv)}
    xv2 = {int(s): x2[p] for p, s in enumerate(pv2)}
    for s in xv1:
        assert abs(xv1[s] - xv2[s]) <= 1e-8 * (1 + abs(xv2[s]))
    cb = rng.standard_normal(lp.n + lp.m)
    y1 = o.btran(np.array([cb[s] for s in pv]))
    y2 = o2.btran(np.array([cb[s] for s in pv2]))
    np.testing.assert_allclose(y1, y2, rtol=1e-8, atol=1e-8)


def test_generators_are_frozen():
    """the libc-rand generators reproduce the committed fixtures bit for bit"""
    for lp in (G.tsp_mtz(20, 42), G.ufl(10, 30, 99), G.set_cover(30, 100, 0.15, 11)):
        ref = load_golden(lp.name)
        assert np.array_equal(ref.col_start, lp.col_start)
        assert np.array_equal(ref.row_index, lp.row_index)
        assert np.array_equal(ref.element, lp.element)
        assert np.array_equal(ref.objective, lp.objective)


@pytest.mark.parametrize("mode", [1, 2, 3])
def test_scale_factors_match_restatement(mode):
    """Engine::computeScaling (host C++) against the numpy restatement of ClpPackedMatrix::scale
    (src/ClpPackedMatrix.cpp:4120) on every golden LP and a planted random LP."""
    import clp_b200
    from oracle.scaling import scale_factors

    names = sorted(json.load(open(os.path.join(ROOT, "tests", "golden", "manifest.json"))))
    cases = [load_golden(nm) for nm in names] + [G.random_sparse_lp(300, 3000, 0.02, 7)]
    scaled = 0
    for lp in cases:
        s = clp_b200.ClpSimplex()
        s.loadLP(lp)
        s.scaling(mode)
        rc, r, c = s.scaleFactors()
        rc2, r2, c2 = scale_factors(lp, mode)
        assert rc == rc2, lp.name
        np.testing.assert_allclose(r, r2, rtol=1e-12, err_msg=lp.name)
        np.testing.assert_allclose(c, c2, rtol=1e-12, err_msg=lp.name)
        if rc == 0:
            scaled += 1
            # the defining property of the final column pass: the largest scaled entry of every
            # non-fixed, non-empty column is the same value (overallLargest <= 100)
            A = lp.to_scipy().tocsc()
            big = np.array([np.abs(A.data[A.indptr[j]:A.indptr[j + 1]] * r[A.indices[A.indptr[j]:A.indptr[j + 1]]]).max() * c[j]
                            for j in range(lp.n) if A.indptr[j + 1] > A.indptr[j] and lp.col_upper[j] - lp.col_lower[j] > 1e-5 * c[j]])
            assert big.max() <= 100.0 * (1 + 1e-12) and big.max() - big.min() <= 1e-9 * big.max(), lp.name
    assert scaled >= 6


def test_perturbation_rule_properties():
    """Engine::perturbCosts (ClpSimplexDual::perturb :6533, default setting 50) on the host: only
    non-fixed nonbasic columns move, towards the dual feasible side of their bound (up at lower
    bound), by at most max(1e3*dualTolerance, maximumFraction*average cost); deterministic; and the automatic
    setting (100) leaves LPs with many distinct cost values alone (:6575)."""
    import clp_b200

    for name in ("transport-20x500", "NQueens-20", "UFL-20x60", "staircase-480"):
        lp = load_golden(name)
        s = clp_b200.ClpSimplex(); s.loadLP(lp); s.setPerturbation(50)
        rc, pc = s.perturbedCosts()
        rc2, pc2 = s.perturbedCosts()
        assert rc == rc2 == 0 and np.array_equal(pc, pc2), name
        delta = pc - lp.objective
        moved = delta != 0.0
        assert moved.any(), name
        fixed = lp.col_upper <= lp.col_lower
        assert not (moved & fixed).any(), name
        assert (delta[moved] > 0).all(), name  # all-slack start: every column sits at its lower bound
        nz = np.abs(lp.objective[lp.objective != 0])
        avg = nz.mean() if nz.size else 1.0
        # largestAllowed = max(1e3*dualTolerance, maximumFraction*averageCost) with maximumFraction <= 1e-3 (:6709, :6803)
        assert np.abs(delta).max() <= max(1e-4, 1e-3 * avg) * 1.0001, name
    lp = G.random_sparse_lp(200, 2000, 0.03, 5)  # 2000 distinct costs: automatic mode does nothing
    s = clp_b200.ClpSimplex(); s.loadLP(lp); s.setPerturbation(100)
    rc, pc = s.perturbedCosts()
    assert rc == 1 and np.array_equal(pc, lp.objective)


def test_basis_file_round_trip(tmp_path):
    """ClpSimplex::writeBasis / readBasis (ClpSimplexOther.cpp:1018): the optimal basis of the CPU
    oracle written in the reference's no-names format and read back into a fresh model."""
    import clp_b200
    from oracle.oracle import OracleSimplex

    lp = load_golden("UFL-10x30")
    o = OracleSimplex(lp)
    assert o.dual() == 0
    st = np.asarray(o.status(), dtype=np.uint8)
    st[(st != 1) & (st != 2)] = 3  # the file distinguishes basic / at upper / everything else
    s = clp_b200.ClpSimplex(); s.loadLP(lp); s.copyinStatus(st)
    f = tmp_path / "opt.bas"
    assert s.writeBasis(f) == 0
    text = f.read_text().splitlines()
    assert text[0].startswith("NAME") and text[-1] == "ENDATA"
    nb_cols = int((st[: lp.n] == 1).sum())
    assert sum(l.startswith((" XU", " XL")) for l in text) == nb_cols
    assert all(len(l.split()) == 3 and l.split()[1][0] == "C" and l.split()[2][0] == "R" for l in text if l.startswith(" X"))
    t = clp_b200.ClpSimplex(); t.loadLP(lp)
    assert t.readBasis(f) == 0
    back = t.statusArray()
    assert np.array_equal(back == 1, st == 1)                      # same basic set
    assert np.array_equal(back[: lp.n] == 2, st[: lp.n] == 2)     # same columns at upper bound
    nonbasic_rows = st[lp.n:] != 1
    assert np.array_equal(back[lp.n:][nonbasic_rows] == 2, st[lp.n:][nonbasic_rows] == 2)
    assert t.readBasis(tmp_path / "missing.bas") == -1
    g = tmp_path / "bad.bas"
    g.write_text("NAME x\n XU C0000001 R9999999\n ZZ C0000001\nENDATA\n")
    assert t.readBasis(g) == 2


def test_cabi_exports_every_declared_symbol():
    from clp_b200 import _capi

    header = open(os.path.join(ROOT, "include", "clp_b200.h")).read()
    declared = set(re.findall(r"\b(Clpb_[A-Za-z0-9]+)\s*\(", header))
    assert declared, "no declarations parsed"
    L = _capi.lib()
    for name in sorted(declared):
        assert hasattr(L, name), f"{name} declared in include/clp_b200.h but not exported"
    assert declared == set(_capi.SIGNATURES), declared ^ set(_capi.SIGNATURES)


def test_product_does_not_reference_oracle():
    """the product path must not include, link or call anything under oracle/"""
    for dirpath, _, files in os.walk(os.path.join(ROOT, "clp_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".hpp", ".cpp", ".h")) or f == "Makefile":
                txt = open(os.path.join(dirpath, f), errors="ignore").read()
                assert "oracle" not in txt.lower() or f == "generators.py", os.path.join(dirpath, f)
    out = subprocess.run(["ldd", os.path.join(ROOT, "clp_b200", "_lib", "libclp_b200.so")],
                         capture_output=True, text=True).stdout
    assert "oracle" not in out


def _write_mps(lp, path):
    """tiny MPS writer (test side) for the reader round trip"""
    inf = 1e29
    with open(path, "w") as f:
        f.write("NAME          RT\nROWS\n N  COST\n")
        kinds = []
        for i in range(lp.m):
            lo, up = lp.row_lower[i], lp.row_upper[i]
            k = "E" if lo == up else ("G" if up >= inf else ("L" if lo <= -inf else "R"))
            kinds.append(k)
            f.write(f" {'L' if k == 'R' else k}  R{i}\n")
        f.write("COLUMNS\n")
        for j in range(lp.n):
            if lp.objective[j] != 0.0:
                f.write(f"    C{j}  COST  {float(lp.objective[j])!r}\n")
            for e in range(lp.col_start[j], lp.col_start[j + 1]):
                f.write(f"    C{j}  R{lp.row_index[e]}  {float(lp.element[e])!r}\n")
        f.write("RHS\n")
        for i in range(lp.m):
            v = lp.row_lower[i] if kinds[i] in "EG" else lp.row_upper[i]
            if v != 0.0:
                f.write(f"    RHS  R{i}  {float(v)!r}\n")
        f.write("RANGES\n")
        for i in range(lp.m):
            if kinds[i] == "R":
                f.write(f"    RNG  R{i}  {float(lp.row_upper[i] - lp.row_lower[i])!r}\n")
        f.write("BOUNDS\n")
        for j in range(lp.n):
            lo, up = lp.col_lower[j], lp.col_upper[j]
            if lo <= -inf and up >= inf:
                f.write(f" FR BND  C{j}\n")
                continue
            if lo <= -inf:
                f.write(f" MI BND  C{j}\n")
            elif lo != 0.0:
                f.write(f" LO BND  C{j}  {float(lo)!r}\n")
            if up < inf:
                f.write(f" UP BND  C{j}  {float(up)!r}\n")
        f.write("ENDATA\n")


@pytest.mark.parametrize("name", ["TSP-MTZ-20", "hello", "modified_afiro", "SetPack-40x120"])
def test_mps_reader_round_trip(tmp_path, name):
    import clp_b200

    lp = load_golden(name)
    path = tmp_path / "rt.mps"
    _write_mps(lp, path)
    s = clp_b200.ClpSimplex()
    assert s.readMps(path) == 0
    got = s.getProblem()
    assert (got.m, got.n) == (lp.m, lp.n)
    A0, A1 = lp.to_scipy(), got.to_scipy()
    assert abs(A0 - A1).max() == 0
    for a, b in ((lp.col_lower, got.col_lower), (lp.col_upper, got.col_upper),
                 (lp.row_lower, got.row_lower), (lp.row_upper, got.row_upper),
                 (lp.objective, got.objective)):
        np.testing.assert_allclose(np.clip(a, -1e30, 1e30), np.clip(b, -1e30, 1e30), rtol=1e-15)


@pytest.mark.parametrize("name", ["TSP-MTZ-20", "hello", "modified_afiro", "UFL-10x30", "transport-10x200",
                                  "staircase-480", "Unbounded-10"])
def test_write_mps_round_trip(tmp_path, name):
    """ClpModel::writeMps -> ClpModel::readMps through the library's own writer and reader: the
    model comes back bit for bit (17 significant digits)."""
    import clp_b200

    lp = load_golden(name)
    s = clp_b200.ClpSimplex(); s.loadLP(lp)
    path = tmp_path / "w.mps"
    assert s.writeMps(path) == 0
    t = clp_b200.ClpSimplex()
    assert t.readMps(path) == 0
    got = t.getProblem()
    assert (got.m, got.n) == (lp.m, lp.n)
    assert abs(lp.to_scipy() - got.to_scipy()).max() == 0
    for a, b in ((lp.col_lower, got.col_lower), (lp.col_upper, got.col_upper),
                 (lp.row_lower, got.row_lower), (lp.row_upper, got.row_upper),
                 (lp.objective, got.objective)):
        assert np.array_equal(np.clip(a, -1e30, 1e30), np.clip(b, -1e30, 1e30))


MPS_EDGE = """* comment line
NAME          EDGE   a second token is ignored
OBJSENSE
    MAX
ROWS
 N  COST
 N  FREEROW
 E  EQ1
 E  EQ2
 L  LE1
 G  GE1
 L  LE2
COLUMNS
    X1        COST      1.5        EQ1       1.0
    X1        LE1       2.0        FREEROW   9.0
    MARKER    'MARKER'  'INTORG'
    X2        COST      -2.0       EQ2       1.0
    X2        GE1       1.0
    MARKER    'MARKER'  'INTEND'
    X3        EQ1       1.0        LE2       4.0
    X3        EQ1       0.5
    X4        GE1       1.0
    X5        LE1       1.0
    X6        LE2       1.0
    X7        COST      0.25
RHS
    RHS       COST      -7.0       EQ1       3.0
    RHS       EQ2       4.0        LE1       10.0
    RHS       GE1       1.0        LE2       8.0
RANGES
    RNG       EQ1       2.0        EQ2       -1.5
    RNG       LE1       4.0        GE1       3.0
BOUNDS
 UP BND       X1        4.0
 UP BND       X2        -1.0
 LO BND       X3        -2.0
 UP BND       X3        -0.5
 MI BND       X4
 BV BND       X5
 FX BND       X6        2.5
 FR BND       X7
ENDATA
"""


def test_mps_reader_conventions(tmp_path):
    """The fixed conventions of the MPS format the reference inherits from CoinMpsIO (CoinUtils;
    ClpModel::readMps src/ClpModel.cpp:2884): first N row is the objective, further N rows are
    dropped, RHS on the objective row is minus the constant, OBJSENSE MAX negates the objective,
    RANGES on E rows extend up (R>0) or down (R<0), on L rows down, on G rows up, an UP bound < 0
    without a lower bound makes the lower bound -infinity, MI / BV / FX / FR, repeated entries of a
    column add up, MARKER lines are skipped."""
    import clp_b200

    f = tmp_path / "edge.mps"
    f.write_text(MPS_EDGE)
    s = clp_b200.ClpSimplex()
    assert s.readMps(f) == 0
    lp = s.getProblem()
    assert (lp.m, lp.n) == (5, 7)                       # FREEROW dropped
    inf = 1e30
    np.testing.assert_array_equal(lp.objective, -np.array([1.5, -2.0, 0, 0, 0, 0, 0.25]))   # MAX -> negated
    rl, ru = np.clip(lp.row_lower, -inf, inf), np.clip(lp.row_upper, -inf, inf)
    np.testing.assert_array_equal(rl, [3.0, 2.5, 6.0, 1.0, -inf])   # EQ1 [3,5], EQ2 [2.5,4], LE1 [6,10], GE1 [1,4], LE2 <= 8
    np.testing.assert_array_equal(ru, [5.0, 4.0, 10.0, 4.0, 8.0])
    cl, cu = np.clip(lp.col_lower, -inf, inf), np.clip(lp.col_upper, -inf, inf)
    np.testing.assert_array_equal(cl, [0.0, -inf, -2.0, -inf, 0.0, 2.5, -inf])
    np.testing.assert_array_equal(cu, [4.0, -1.0, -0.5, inf, 1.0, 2.5, inf])
    A = lp.to_scipy().toarray()
    assert A[0, 2] == 1.5 and A[0, 0] == 1.0 and A[2, 0] == 2.0 and A[4, 2] == 4.0   # 1.0 + 0.5 merged
    assert lp.nnz == 9
    # the constant: objective row RHS -7 means +7 on the objective, negated again by MAX
    st_all = clp_b200.ClpSimplex(); st_all.readMps(f)
    out = tmp_path / "edge_out.mps"
    assert st_all.writeMps(out) == 0
    assert "OBJROW" in out.read_text()
    t = clp_b200.ClpSimplex(); assert t.readMps(out) == 0
    lp2 = t.getProblem()
    assert abs(lp.to_scipy() - lp2.to_scipy()).max() == 0
    for a, b in ((lp.col_lower, lp2.col_lower), (lp.col_upper, lp2.col_upper), (lp.row_lower, lp2.row_lower),
                 (lp.row_upper, lp2.row_upper), (lp.objective, lp2.objective)):
        assert np.array_equal(np.clip(a, -inf, inf), np.clip(b, -inf, inf))


def test_mps_reader_rejects_unknown_names(tmp_path):
    import clp_b200

    f = tmp_path / "bad.mps"
    f.write_text("NAME B\nROWS\n N C\n L R1\nCOLUMNS\n    X1 NOPE 1.0\nENDATA\n")
    assert clp_b200.ClpSimplex().readMps(f) == -2
    g = tmp_path / "bad2.mps"
    g.write_text("NAME B\nROWS\n N C\n L R1\nCOLUMNS\n    X1 R1 1.0\nBOUNDS\n UP B X9 1.0\nENDATA\n")
    assert clp_b200.ClpSimplex().readMps(g) == -3
    assert clp_b200.ClpSimplex().readMps(tmp_path / "missing.mps") == -1


def test_mps_reader_on_reference_files():
    """the reference's own example files (examples/modified_afiro.mps, examples/hello.mps), kept
    verbatim in tests/golden/"""
    import clp_b200

    for fn, name in (("modified_afiro.mps", "modified_afiro"), ("hello.mps", "hello")):
        s = clp_b200.ClpSimplex()
        assert s.readMps(os.path.join(ROOT, "tests", "golden", fn)) == 0
        got, ref = s.getProblem(), load_golden(name)
        assert abs(got.to_scipy() - ref.to_scipy()).max() == 0
        np.testing.assert_array_equal(got.row_lower, ref.row_lower)


def test_no_device_fails_loudly():
    """no visible CUDA device: dual() raises instead of falling back to a CPU path.  Run in a child
    process with the devices hidden, so that machines with a GPU check it as well."""
    code = r"""
import sys
sys.path[:0] = [%r, %r]
import clp_b200
from conftest import load_golden
s = clp_b200.ClpSimplex()
s.loadLP(load_golden("NQueens-8"))
try:
    s.dual()
except clp_b200.NoDeviceError:
    print("raised NoDeviceError")
""" % (ROOT, os.path.join(ROOT, "tests"))
    out = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                         capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stderr
    assert "raised NoDeviceError" in out.stdout


def test_two_rank_sharding_host_logic():
    """world_size=2 over gloo: unique-id broadcast and column shard ranges (the host logic of
    the column-sharded pricing pass; the NCCL exchange itself is exercised on the GPU box)."""
    code = r"""
import os, sys
sys.path.insert(0, %r)
import numpy as np, torch, torch.distributed as dist
from clp_b200.sharding import shard_range, broadcast_unique_id
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%%s" %% os.environ["PORT"],
                        rank=int(os.environ["RANK"]), world_size=2)
rank = dist.get_rank()
uid = np.arange(128, dtype=np.uint8) if rank == 0 else np.zeros(128, dtype=np.uint8)
uid = broadcast_unique_id(uid, src=0)
assert np.array_equal(uid, np.arange(128, dtype=np.uint8))
n = 1001
lo, hi = shard_range(n, rank, 2)
t = torch.tensor([lo, hi])
out = [torch.zeros(2, dtype=torch.long) for _ in range(2)]
dist.all_gather(out, t)
assert out[0][0] == 0 and out[0][1] == out[1][0] and out[1][1] == n
# the exchange of Engine::enqueueIteration: every rank prices its block, then ONE in-place
# all-gather of shards padded to per = ceil(n/world) entries; the padding of the last shard lands
# on the slack part of the row (entries n..n+m), which the row kernel recomputes from rho
rng = np.random.default_rng(7)
m = 40
A = rng.standard_normal((m, n)) * (rng.uniform(size=(m, n)) < 0.1)
rho = rng.standard_normal(m)
per = (n + 2 - 1) // 2
row = np.full(n + m, np.nan)
row[lo:hi] = rho @ A[:, lo:hi]                      # this rank's raw dot products
send = torch.from_numpy(row[rank * per: rank * per + per].copy())
parts = [torch.zeros(per, dtype=torch.float64) for _ in range(2)]
dist.all_gather(parts, send)
for r in range(2):
    row[r * per: r * per + per] = parts[r].numpy()
row[n:] = -rho                                       # slack part rewritten after the gather
assert np.array_equal(row[:n], np.concatenate([rho @ A[:, :per], rho @ A[:, per:]]))
assert 2 * per <= n + m
dist.destroy_process_group()
print("ok", rank)
""" % ROOT
    import socket

    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), PORT=str(port))
        procs.append(subprocess.Popen([sys.executable, "-c", code], env=env, stdout=subprocess.PIPE,
                                      stderr=subprocess.PIPE, text=True))
    for p in procs:
        out, err = p.communicate(timeout=120)
        assert p.returncode == 0, err
        assert "ok" in out


def test_two_rank_row_sharded_gemv_protocol():
    """world_size=2 over gloo: the row-sharded FTRAN GEMV of the multi-GPU path -- every rank computes its
    block of rows of y = Ninv b for three right-hand sides into its chunk of the [rank][rhs][perMax] buffer,
    ONE all-gather of fixed-size chunks completes it, and gather_slot() finds every entry (the index math
    of gemv_rows_kernel / gemv_result in solve.cu restated in clp_b200/sharding.py), for nucleus sizes that
    are not multiples of anything."""
    code = r"""
import os, sys
sys.path.insert(0, %r)
import numpy as np, torch, torch.distributed as dist
from clp_b200.sharding import factor_row_range, gather_slot, round_up8
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%%s" %% os.environ["PORT"],
                        rank=int(os.environ["RANK"]), world_size=2)
rank, world = dist.get_rank(), 2
m, nrhs = 203, 3
per_max = round_up8((m + world - 1) // world)
rng = np.random.default_rng(11)
for k in (1, 7, 8, 9, 100, 101, 203):
    Ninv = rng.standard_normal((k, k)); b = rng.standard_normal((nrhs, k))
    lo, hi, per_k = factor_row_range(k, rank, world)
    assert per_k <= per_max
    chunk = np.zeros(nrhs * per_max)
    for c in range(nrhs):
        chunk[c * per_max: c * per_max + (hi - lo)] = Ninv[lo:hi] @ b[c]
    parts = [torch.zeros(nrhs * per_max, dtype=torch.float64) for _ in range(world)]
    dist.all_gather(parts, torch.from_numpy(chunk))
    gathered = np.concatenate([p.numpy() for p in parts])
    for c in range(nrhs):
        y = np.array([gathered[gather_slot(i, c, k, world, nrhs, per_max)] for i in range(k)])
        assert np.array_equal(y, np.concatenate([Ninv[:min(k, per_k)] @ b[c], Ninv[min(k, per_k):] @ b[c]]))
dist.destroy_process_group()
print("ok", rank)
""" % ROOT
    import socket

    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), PORT=str(port))
        procs.append(subprocess.Popen([sys.executable, "-c", code], env=env, stdout=subprocess.PIPE,
                                      stderr=subprocess.PIPE, text=True))
    for p in procs:
        out, err = p.communicate(timeout=120)
        assert p.returncode == 0, err
        assert "ok" in out


def test_netlib_afiro_reference_objective():
    """BASELINE.json configs[0]: Netlib afiro through this repo's MPS reader and the oracle; the value is
    the reference's own (src/unitTest.cpp:480-486: 28 rows incl. the objective, 32 columns,
    -4.6475314286e+02 to objValueTol 1e-8)"""
    import clp_b200

    s = clp_b200.ClpSimplex()
    assert s.readMps(os.path.join(ROOT, "tests", "golden", "afiro.mps")) == 0
    assert (s.numberRows() + 1, s.numberColumns(), s.getNumElements()) == (28, 32, 83)
    lp = s.getProblem()
    o = O.OracleSimplex(lp)
    assert o.dual() == 0
    assert abs(o.objective_value - (-4.6475314286e+02)) <= 1e-8 * (1 + 464.75314286)
    fx = load_golden("afiro")
    assert (fx.m, fx.n, fx.nnz) == (lp.m, lp.n, lp.nnz)
    assert np.array_equal(fx.element, lp.element) and np.array_equal(fx.row_index, lp.row_index)


def test_default_refactorization_interval_policy():
    """host-only: the default interval is twice ClpSimplex::defaultFactorizationFrequency
    (src/ClpSimplex.cpp:11401-11431) and is stretched only where the dense refactorization of a large
    nucleus would dominate a cycle (staircase-like bases); an explicit factorizationFrequency wins"""
    import clp_b200
    from bench import clp_default_frequency, default_cycle

    for m, n, dens in ((1000, 10000, 0.01), (10000, 100000, 0.01)):
        lp = G.random_sparse_lp(m, n, dens, 1) if m < 5000 else None
        if lp is None:   # sizes only: an LP with the right dimensions and nnz is enough for the model
            lp = G.LP("dims", m, n, np.arange(0, 100 * n + 1, 100, dtype=np.int32), np.zeros(100 * n, dtype=np.int32),
                      np.ones(100 * n), np.zeros(n), np.ones(n), np.zeros(n), np.zeros(m), np.ones(m))
        s = clp_b200.ClpSimplex(); s.loadLP(lp)
        base = 2 * clp_default_frequency(m)
        assert default_cycle(m) == base
        assert s.refactorizationInterval(0) == base
        assert s.refactorizationInterval(m // 2) == base          # C2's nucleus: the base interval
        assert base <= s.refactorizationInterval(m) <= 2048
        s.setFactorizationFrequency(123)
        assert s.refactorizationInterval(m) == 123
    # staircase shape (m = n = 20 000, 4e5 nonzeros): the interval grows with the nucleus
    m = n = 20000
    lp = G.LP("dims", m, n, np.arange(0, 20 * n + 1, 20, dtype=np.int32), np.zeros(20 * n, dtype=np.int32),
              np.ones(20 * n), np.zeros(n), np.ones(n), np.zeros(n), np.zeros(m), np.ones(m))
    s = clp_b200.ClpSimplex(); s.loadLP(lp)
    vals = [s.refactorizationInterval(k) for k in (2000, 8000, 12000, 17000, 20000)]
    assert vals[0] == 2 * clp_default_frequency(m) and vals == sorted(vals) and vals[-1] > 2 * vals[0]
