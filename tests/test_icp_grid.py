"""The re-association grid (`model->update(x)` for point2point, csrc/mopt_icp.cu, DESIGN.md §3.5) against brute force.

Contract under test: the nearest target point within max_dist, the radius inclusive, ties to the lowest original
index; an fp32 index forms the query and the distances in fp32 from fp32-rounded data and writes fp32-rounded target
coordinates; a target point with a non-finite coordinate never matches.

The CPU part restates build_index's grid arithmetic (bounding box of the finite points, cell growth, dims,
floor((v - origin) / cell)) and shows that each named cloud reaches the case it names: exactly 2^24 cells, one
coarsening step, a coarse grid, a single cell, a flat axis, midpoint queries on cell boundaries.  It also checks the
expectations of the exact data sets (2-, 4- and 8-way ties, distances of exactly max_dist) with a numpy brute force
and the C++ oracle.  The GPU part holds the device to them in every store x index dtype pair and both host dtypes of
the index build (a memcpy when the dtypes agree, a host conversion loop when they do not)."""
import os
import subprocess
import sys
import tempfile
from contextlib import ExitStack
from types import SimpleNamespace

import numpy as np
import pytest

from oracle import oracle_py as orc
from tests.common import fachada
from tests.test_icp import MAX_DIST as FACHADA_MAX_DIST
from tests.test_icp import X_TRUE, clouds

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# ---- build_index (csrc/mopt_icp.cu), mirrored ----------------------------------------------------------------------
CELL_CAP = 1 << 24     # at most 2^24 cells
GROWTH = 1.26          # cell *= 1.26 until the grid fits
SCAN_TILE = 256 * 8    # kScanThreads * kScanItems
F32, F64 = 0, 1        # capi / oracle dtype codes
NP = {F32: np.float32, F64: np.float64}
UNIT = {F32: 2.0 ** -24, F64: 2.0 ** -53}   # unit roundoff


def grid_of(tgt, max_dist):
    """(origin, cell, inv_cell, dims, ncells, growth steps, scan tiles) of the grid build_index makes for `tgt` (the
    values the index holds)."""
    t = np.asarray(tgt, dtype=np.float64).reshape(-1, 3)
    fin = np.all(np.isfinite(t), axis=1)
    lo = t[fin].min(axis=0) if fin.any() else np.zeros(3)
    hi = t[fin].max(axis=0) if fin.any() else np.zeros(3)
    with np.errstate(over="ignore", invalid="ignore"):
        ext = hi - lo
        cell, steps = float(max_dist), 0
        while True:
            dims = [float(np.floor(e / cell)) + 1.0 if np.isfinite(e) else 1.0 for e in ext]
            if dims[0] * dims[1] * dims[2] <= CELL_CAP:
                break
            cell *= GROWTH
            steps += 1
    dims = np.array([int(d) for d in dims], dtype=np.int64)
    ncells = int(np.prod(dims))
    return SimpleNamespace(origin=lo, cell=cell, inv=1.0 / cell, dims=dims, ncells=ncells, steps=steps,
                           tiles=-(-(ncells + 2) // SCAN_TILE))


def cell_coords(v, g):
    """cell_coord per axis: floor((v - origin) * inv_cell), -1 below the grid (and for NaN), dims above it."""
    with np.errstate(over="ignore", invalid="ignore"):
        c = np.floor((np.asarray(v, dtype=np.float64) - g.origin) * g.inv)
        return np.where(c >= 0, np.where(c < g.dims, c, g.dims), -1).astype(np.int64)


def brute(q, tgt, max_dist, dtype=np.float64):
    """Nearest target within max_dist (inclusive) in `dtype` arithmetic, ties to the first index (argmin).
    -> (matched, index, squared distance, members of the tie)."""
    q = np.asarray(q, dtype=dtype)
    t = np.asarray(tgt, dtype=dtype)
    r2 = dtype(max_dist * max_dist)
    ok, arg, best, ties = [], [], [], []
    for s in range(0, len(q), 2048):
        qq = q[s:s + 2048]
        with np.errstate(over="ignore", invalid="ignore"):
            d = [t[None, :, k] - qq[:, None, k] for k in range(3)]
            dd = d[0] * d[0] + d[1] * d[1] + d[2] * d[2]
        dd = np.where(np.isnan(dd), np.inf, dd)
        j = np.argmin(dd, axis=1) if t.shape[0] else np.zeros(len(qq), dtype=np.int64)
        b = dd[np.arange(len(qq)), j] if t.shape[0] else np.full(len(qq), np.inf)
        ok.append(b <= r2)
        arg.append(j)
        best.append(b)
        ties.append((dd == b[:, None]).sum(axis=1) if t.shape[0] else np.zeros(len(qq), dtype=np.int64))
    return np.concatenate(ok), np.concatenate(arg), np.concatenate(best), np.concatenate(ties)


# ---- exact data: the integer lattice {-4..4}^3 in a fixed shuffled order, R = I, a dyadic translation ----------------
LATTICE = np.stack(np.meshgrid(*[np.arange(-4.0, 5.0)] * 3, indexing="ij"), axis=-1).reshape(-1, 3)
TARGETS = LATTICE[np.random.default_rng(11).permutation(len(LATTICE))]
X_EXACT = np.array([0.5, -0.25, 0.75, 0.0, 0.0, 0.0])   # R = I exactly, so the query is src + t without rounding
EXACT_RADII = [0.5, 0.75, 1.0]
STEP = 2.0 ** -10
TIE_OFFSETS = {2: [(0.5, 0, 0), (0, 0.5, 0), (0, 0, 0.5)], 4: [(0.5, 0.5, 0), (0.5, 0, 0.5), (0, 0.5, 0.5)],
               8: [(0.5, 0.5, 0.5)]}


def tie_queries():
    """Lattice points of {-4..3}^3 plus a half step on 1, 2 or 3 axes: 2-, 4- and 8-way ties -> (q, ways)."""
    base = LATTICE[np.all(LATTICE < 4, axis=1)]
    q, ways = [], []
    for w, offs in TIE_OFFSETS.items():
        for o in offs:
            q.append(base + np.array(o))
            ways.append(np.full(len(base), w))
    return np.concatenate(q), np.concatenate(ways)


def boundary_queries(md):
    """Queries outside the lattice's box on each of the 6 faces, 12 edges and 8 corners -> (q, inside, nearest point).
    Faces: at distance exactly md and md + 2^-10 along the normal.  Edges and corners: no dyadic offset puts a query at
    exactly md from a lattice point off one axis (a^2 + b^2 = md^2 has no dyadic solution for md in {0.5, 0.75, 1}), so
    they are displaced by the same multiple of 2^-10 on each outer axis, the largest inside md and the smallest beyond
    md + 2^-10."""
    q, inside, near = [], [], []
    other = np.array([1.0, -2.0, 3.0])
    for axes in ([0], [1], [2], [0, 1], [0, 2], [1, 2], [0, 1, 2]):
        k = len(axes)
        for signs in np.array(np.meshgrid(*[[-1.0, 1.0]] * k, indexing="ij")).reshape(k, -1).T:
            p = other.copy()
            p[axes] = 4.0 * signs
            if k == 1:
                offs = [(md, True), (md + STEP, False)]
            else:
                offs = [(np.floor(md / np.sqrt(k) / STEP) * STEP, True),
                        (np.ceil((md + STEP) / np.sqrt(k) / STEP) * STEP, False)]
            for o, ins in offs:
                qq = p.copy()
                qq[axes] += o * signs
                q.append(qq)
                inside.append(ins)
                near.append(p)
    return np.array(q), np.array(inside), np.array(near)


def exact_queries(md):
    tq, ways = tie_queries()
    bq, _, _ = boundary_queries(md)
    return np.concatenate([tq, bq])


# ---- the named grids ---------------------------------------------------------------------------------------------
def cap_lattice(nx):
    """The lattice nx x 256 x 256 with spacing 1 (max_dist = 1): 2^24 cells at nx = 256, one coarsening step at 257."""
    return np.stack(np.meshgrid(np.arange(nx, dtype=np.float32), *[np.arange(256, dtype=np.float32)] * 2,
                                indexing="ij"), axis=-1).reshape(-1, 3)


CAP_OFFSET = np.array([0.25, -0.125, 0.375], dtype=np.float32)


def shape_case(name):
    """name -> (targets, queries in the target frame, max_dist)."""
    rng = np.random.default_rng(sum(map(ord, name)))
    if name == "coarse":          # a 1000 m cube with a 1 cm radius: the cell grows far beyond the radius
        t = rng.uniform(0, 1000, (20_000, 3))
        q = np.concatenate([t[:4000] + rng.uniform(-0.004, 0.004, (4000, 3)), rng.uniform(-1, 1001, (2000, 3))])
        return t, q, 0.01
    if name == "one_cell":        # 50 k targets in one cell
        return rng.uniform(0, 1, (50_000, 3)), rng.uniform(-1, 2, (3000, 3)), 1.5
    if name == "single":
        return np.array([[0.3, -0.7, 2.1]]), np.array([0.3, -0.7, 2.1]) + rng.uniform(-1, 1, (3000, 3)), 0.8
    if name == "identical":       # 1 000 copies of one point: whichever wins, the coordinates are the same
        return np.tile([[0.5, 0.25, -1.5]], (1000, 1)), np.array([0.5, 0.25, -1.5]) + rng.uniform(-0.5, 0.5, (3000, 3)), 0.4
    if name == "plane":           # z = 0 (dims[2] == 1), queries at z = +-(md - 2^-10) and +-(md + 2^-10)
        xy = np.stack(np.meshgrid(np.arange(-10.0, 11.0), np.arange(-10.0, 11.0), indexing="ij"), -1).reshape(-1, 2)
        t = np.column_stack([xy, np.zeros(len(xy))])
        q = np.concatenate([t + [0, 0, z] for z in (0.5 - STEP, -(0.5 - STEP), 0.5 + STEP, -(0.5 + STEP))])
        return t, q, 0.5
    if name == "line":            # along x (dims[1] == dims[2] == 1)
        t = np.column_stack([np.arange(-50, 50) * 0.25, np.zeros(100), np.zeros(100)])
        return t, rng.uniform([-13, -0.3, -0.3], [13, 0.3, 0.3], (3000, 3)), 0.2
    raise KeyError(name)


SHAPES = ["coarse", "one_cell", "single", "identical", "plane", "line"]


def uniform_cloud():
    rng = np.random.default_rng(21)
    return rng.uniform(-6, 6, (20_000, 3)), rng.uniform(-5, 5, (20_000, 3))


X_UNIFORM = np.array([0.3, -0.2, 0.1, 0.2, -0.1, 0.3])
RANDOM_CASES = {"fachada": ([[0.0] * 6, X_TRUE, [0.3, 0.1, -0.2, 0.05, 0.05, -0.05]], FACHADA_MAX_DIST),
                "uniform": ([X_UNIFORM], 0.3)}


def random_case(name):
    return clouds() if name == "fachada" else uniform_cloud()


def query_error(idx_dt, src, x):
    """Per-query bound on |q_device - q_ref|, q_ref = R p + t in fp64 from the stored source p and the reference's
    rotation.  In the index dtype (unit roundoff u) coordinate k of the query is formed from p, R and t rounded to it
    (u each) by 3 products and 3 sums, each rounded relative to at most M_k = sum_j |R_kj p_j| + |t_k|: to first order
    |dq_k| <= 6 u M_k.  The device's fp64 rotation comes from its own so3 evaluation, which may differ from the
    reference's by a few fp64 ulps.  The bound used is (8 u + 16 u64) |M|_2, u64 = 2^-53."""
    T = orc.so3_convert6dof(x)
    M = np.abs(np.asarray(src, dtype=np.float64)) @ np.abs(T[:3, :3]).T + np.abs(T[:3, 3])
    return (8.0 * UNIT[idx_dt] + 16.0 * UNIT[F64]) * np.linalg.norm(M, axis=1)


def kd_reference(q, tgt, md, qerr, idx_dt):
    """fp64 cKDTree with k = 2 -> (d1, d2, idx1, err, decidable), err(d) = qerr + 4 u d the per-query bound on a
    distance the device computes (the query's error plus the differences, squares and sums of the squared distance,
    under 5 u relative, i.e. 2.5 u in the distance).  Decidable: d2 - d1 > err(d1) + err(d2) (or no second target) and
    |d1 - md| > err(d1) + u md (the radius is compared squared, md^2 rounded to the index dtype)."""
    from scipy.spatial import cKDTree
    u = UNIT[idx_dt]
    d, idx = cKDTree(tgt).query(q, k=2)
    d1, d2, i1 = d[:, 0], d[:, 1], idx[:, 0]

    def err(dist):
        return qerr + 4.0 * u * dist

    with np.errstate(invalid="ignore"):
        sep = np.where(np.isfinite(d2), d2 - d1 > err(d1) + err(d2), True)
    return d1, d2, i1, err, sep & (np.abs(d1 - md) > err(d1) + u * md)


def query_of(src, x):
    T = orc.so3_convert6dof(x)
    return src @ T[:3, :3].T + T[:3, 3]


def src_of(q, x):
    T = orc.so3_convert6dof(x)
    return (q - T[:3, 3]) @ T[:3, :3]


def rounded(a, *dts):
    a = np.asarray(a, dtype=np.float64)
    with np.errstate(over="ignore"):   # 1e308 -> inf in fp32
        for dt in dts:
            a = a.astype(NP[dt]).astype(np.float64)
    return a


# ---- CPU: the data mean what the tests say ------------------------------------------------------------------------
def corners(nx):
    """The 8 corners of cap_lattice(nx): the same bounding box, so the same grid."""
    return np.array(np.meshgrid([0.0, nx - 1.0], [0.0, 255.0], [0.0, 255.0], indexing="ij")).reshape(3, -1).T


def test_grid_mirror_reaches_each_named_case():
    g = grid_of(corners(256), 1.0)
    assert g.ncells == CELL_CAP and g.steps == 0 and g.tiles == 8193 and list(g.dims) == [256, 256, 256]
    g = grid_of(corners(257), 1.0)
    assert g.steps == 1 and g.ncells <= CELL_CAP and 257 * 256 * 256 > CELL_CAP and g.cell == GROWTH
    t, _, md = shape_case("coarse")
    g = grid_of(t, md)
    assert g.steps > 10 and g.cell > 10 * md and g.ncells <= CELL_CAP
    for name in ("one_cell", "single", "identical"):
        t, _, md = shape_case(name)
        assert grid_of(t, md).ncells == 1, name
    t, _, md = shape_case("plane")
    g = grid_of(t, md)
    assert g.dims[2] == 1 and g.dims[0] == g.dims[1] == 41
    t, _, md = shape_case("line")
    assert list(grid_of(t, md).dims[1:]) == [1, 1]
    assert grid_of(np.zeros((0, 3)), 0.5).ncells == 1
    # the lattice at the three radii: the cell is the radius (no growth), the origin its lowest corner
    for md in EXACT_RADII:
        g = grid_of(TARGETS, md)
        assert g.steps == 0 and g.cell == md and np.array_equal(g.origin, [-4.0] * 3)
    # at md = 0.5 every coordinate of the tie queries, half steps included, lies exactly on a cell boundary
    tq, _ = tie_queries()
    g = grid_of(TARGETS, 0.5)
    scaled = (tq - g.origin) * g.inv
    assert np.array_equal(scaled, np.floor(scaled))


def test_non_finite_clouds_give_finite_grids():
    """The sizing loop ends and every cell is in range for the non-finite clouds (it used to spin on an infinite extent
    and give dims = INT_MIN on an axis without a finite value)."""
    for name in NONFINITE_CASES:
        tgt, _, md = nonfinite_case(name)
        for dt in (F32, F64):
            g = grid_of(rounded(tgt, dt), md)
            assert 1 <= g.ncells <= CELL_CAP and np.all(g.dims >= 1) and np.all(np.isfinite(g.origin)), (name, dt)


@pytest.mark.parametrize("md", EXACT_RADII)
def test_exact_data_expectations(md):
    tq, ways = tie_queries()
    ok, arg, best, ties = brute(tq, TARGETS, md)
    assert np.array_equal(ties, ways)                     # 2, 4 or 8 members
    assert np.array_equal(best, np.log2(ways) / 4)         # squared distances 0.25, 0.5, 0.75
    assert np.array_equal(ok, best <= md * md)
    # the tie goes to the lowest original index, and that is not the spatially first member
    for i in np.flatnonzero(ok)[:400]:
        members = np.flatnonzero(np.sum((TARGETS - tq[i]) ** 2, axis=1) == best[i])
        assert arg[i] == members.min()
    spatial_first = [np.lexsort(TARGETS[np.sum((TARGETS - q) ** 2, axis=1) == b].T[::-1])[0] for q, b in
                     zip(tq[ok][:200], best[ok][:200])]
    assert np.mean(np.array(spatial_first) != 0) > 0.3
    if md == 0.5:
        assert ok[ways == 2].all() and not ok[ways > 2].any()  # the 2-way ties sit at exactly the radius
    bq, inside, near = boundary_queries(md)
    ok, arg, best, ties = brute(bq, TARGETS, md)
    assert np.array_equal(ok, inside) and np.array_equal(TARGETS[arg[ok]], near[ok])
    assert np.all(ties[ok] == 1)
    faces = np.sum(np.abs(bq) > 4, axis=1) == 1
    assert np.all(best[faces & inside] == md * md)        # faces: exactly the radius
    # single precision arrives at the same answers: every value is exact in fp32
    q = exact_queries(md)
    assert all(np.array_equal(u, v) for u, v in zip(brute(q, TARGETS, md), brute(q, TARGETS, md, np.float32)))
    # the grid search finds them: each expected target's cell is within one of the query's cell on every axis
    g = grid_of(TARGETS, md)
    ok, arg, _, _ = brute(q, TARGETS, md)
    cq = cell_coords(q[ok], g)
    ct = np.clip(cell_coords(TARGETS[arg[ok]], g), 0, g.dims - 1)
    assert np.all(np.abs(cq - ct) <= 1)


@pytest.mark.parametrize("md", EXACT_RADII)
def test_exact_data_oracle_chooses_the_same_targets(md):
    q = exact_queries(md)
    src = src_of(q, X_EXACT)
    assert np.array_equal(query_of(src, X_EXACT), q)       # R = I: the queries are formed without rounding
    ok, arg, _, _ = brute(q, TARGETS, md)
    icp = orc.Cost(orc.P2P_ICP, 6, 3, len(q), a=src, jac_mode=orc.JAC_ANALYTICAL, target=TARGETS, max_dist=md)
    ref = orc.Cost(orc.P2P, 6, 3, int(ok.sum()), a=src[ok], b=TARGETS[arg[ok]], jac_mode=orc.JAC_ANALYTICAL)
    for u, v in zip(orc.linearize(icp, X_EXACT), orc.linearize(ref, X_EXACT)):
        assert np.array_equal(u, v)


@pytest.mark.parametrize("name", list(RANDOM_CASES))
def test_random_clouds_are_decidable(name):
    """The share of queries the rounding bound leaves undecided is below 1 % even for an fp32 index."""
    src, tgt = random_case(name)
    xs, md = RANDOM_CASES[name]
    for x in xs:
        src32 = rounded(src, F32)
        *_, dec = kd_reference(query_of(src32, x), rounded(tgt, F32), md, query_error(F32, src32, x), F32)
        assert 1.0 - dec.mean() < 0.01, (name, x, 1.0 - dec.mean())


# ---- non-finite target clouds ---------------------------------------------------------------------------------------
NONFINITE_CASES = ["inf", "nan_some", "all_nan", "z_nan", "huge"]


def nonfinite_case(name):
    """name -> (targets, queries in the target frame, max_dist)."""
    rng = np.random.default_rng(31)
    t = rng.uniform(0, 10, (3000, 3))
    q = np.concatenate([t[:1500] + rng.normal(0, 0.05, (1500, 3)), rng.uniform(-1, 11, (1500, 3))])
    if name == "inf":
        t[5] = [np.inf, 1.0, 1.0]
        t[17] = [2.0, -np.inf, 3.0]
    elif name == "nan_some":
        rows = rng.choice(3000, 90, replace=False)
        t[rows, rng.integers(0, 3, 90)] = np.nan
    elif name == "all_nan":
        t[:] = np.nan
    elif name == "z_nan":
        t[:, 2] = np.nan
    elif name == "huge":            # finite, but the extent overflows (and an fp32 index rounds them to inf)
        t[7] = [1e308, 0.0, 0.0]
        t[8] = [-1e308, 5.0, 5.0]
        t[9] = [3.0, 1e308, -1e308]
    return t, q, 0.3


def nonfinite_worker_results(tmp):
    """Builds every non-finite case in a fresh process with a timeout: a build that spins fails the test instead of
    hanging the suite.  -> {(case, index dtype, host dtype): (matched, targets downloaded)}"""
    p = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "icp_grid_worker.py"), tmp], capture_output=True,
                       text=True, timeout=300)
    assert p.returncode == 0, p.stderr[-3000:]
    out = {}
    for name in NONFINITE_CASES:
        for it in (F32, F64):
            for ht in (F32, F64):
                d = np.load(os.path.join(tmp, f"{name}_{it}_{ht}.npy"))
                out[(name, it, ht)] = (int(d[0, 0]), d[1:])
    return out


def run_nonfinite_case(capi, ctx, name, it, ht):
    """The worker's body: the case through an fp64 store and an index of dtype `it` from a host array of dtype `ht`."""
    tgt, q, md = nonfinite_case(name)
    src = src_of(q, X_EXACT)
    with Reassoc(capi, ctx, src, tgt.astype(NP[ht]), md, F64, it, X_EXACT) as r:
        return r.matched, r.got


# ---- device ---------------------------------------------------------------------------------------------------------
capi = None


@pytest.fixture(scope="module")
def env():
    global capi
    from moptimizer_0_b200 import capi as _capi
    capi = _capi
    c = capi.Context(0)
    yield c
    c.close()


class Reassoc:
    """A point2point store of `src` with an index of `tgt` attached, re-associated at x."""

    def __init__(self, capi, ctx, src, tgt, md, store_dt, index_dt, x):
        self.st = capi.Store(ctx, capi.MODEL_POINT2POINT, src.shape[0], store_dt)
        self.st.upload(0, np.asarray(src, dtype=NP[store_dt]))
        self.ix = capi.NNIndex(ctx, tgt, md, dtype=index_dt)
        capi.store_set_target(self.st, self.ix)
        self.matched = capi.store_reassociate(self.st, x)
        self.got = self.st.download(1)

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.ix.close()
        self.st.close()


DTYPES = [(s, i, h) for s in (F32, F64) for i in (F32, F64) for h in (F32, F64)]
DTYPE_IDS = [f"store{'32' if s == F32 else '64'}-index{'32' if i == F32 else '64'}-host{'32' if h == F32 else '64'}"
             for s, i, h in DTYPES]


def expected_targets(tgt_index, ok, arg, store_dt):
    """What the store holds after re-association: the index's target rounded to the store dtype, NaN unmatched."""
    out = np.full((len(ok), 3), np.nan)
    out[ok] = rounded(tgt_index[arg[ok]], store_dt)
    return out


def same(a, b):
    return np.array_equal(a, b, equal_nan=True)


@pytest.mark.gpu
@pytest.mark.parametrize("store_dt,index_dt,host_dt", DTYPES, ids=DTYPE_IDS)
def test_exact_lattice_bit_for_bit(env, store_dt, index_dt, host_dt):
    """Ties, the inclusive radius and the faces, edges and corners of the grid: the downloaded targets and the NaN mask
    equal the brute force, H, b and the sum equal the oracle's, a second build gives the same bits, and a permuted
    target order moves exactly the ties the lowest-index rule says it moves."""
    ctx = env
    perm = np.random.default_rng(12).permutation(len(TARGETS))
    for md in EXACT_RADII:
        q = exact_queries(md)
        src = src_of(q, X_EXACT)
        ok, arg, _, ties = brute(q, TARGETS, md)
        want = expected_targets(TARGETS, ok, arg, store_dt)
        with Reassoc(capi, ctx, src, TARGETS.astype(NP[host_dt]), md, store_dt, index_dt, X_EXACT) as r:
            assert r.matched == int(ok.sum()), (md, r.matched, int(ok.sum()))
            assert same(r.got, want), (md, np.flatnonzero(~np.all((r.got == want) | np.isnan(want), axis=1))[:10])
            prob = capi.make_problem(capi.MODEL_POINT2POINT, capi.JAC_ANALYTICAL, capi.F64)
            H, b, s = ctx.linearize(r.st, prob, X_EXACT)
            icp = orc.Cost(orc.P2P_ICP, 6, 3, len(q), a=src, jac_mode=orc.JAC_ANALYTICAL, target=TARGETS, max_dist=md)
            Ho, bo, so = orc.linearize(icp, X_EXACT)
            assert np.array_equal(H, Ho) and np.array_equal(b, bo) and s == so, (md, s, so)
            assert ctx.compute_cost(r.st, prob, X_EXACT) == so
        with Reassoc(capi, ctx, src, TARGETS.astype(NP[host_dt]), md, store_dt, index_dt, X_EXACT) as r2:
            assert r2.matched == int(ok.sum()) and same(r2.got, want)
        P = TARGETS[perm]
        pok, parg, _, _ = brute(q, P, md)
        pwant = expected_targets(P, pok, parg, store_dt)
        assert np.array_equal(pok, ok)
        moved = np.flatnonzero(np.any(pwant != want, axis=1) & ok)
        assert len(moved) > 0 and np.all(ties[moved] > 1)   # only ties change, and some do
        with Reassoc(capi, ctx, src, P.astype(NP[host_dt]), md, store_dt, index_dt, X_EXACT) as r3:
            assert same(r3.got, pwant), md


def check_against_kdtree(got, matched, q, tgt_index, md, qerr, index_dt, store_dt):
    """Decidable queries exactly (the index's nearest target, rounded to the store dtype, or NaN).  The others: a target
    whose distance the device could have found no larger than d1's and within the radius (d <= d1 + err(d1) + err(md)
    and d <= md + err(md) + u md), NaN only if d1 >= md - err(d1) - u md.  The store's rounding of the written target
    adds 2 u_store |target|.  -> (undecidable share, per-query bound err(d1) of the queries)."""
    u = UNIT[index_dt]
    d1, _, i1, err, dec = kd_reference(q, tgt_index, md, qerr, index_dt)
    nan = np.isnan(got[:, 0])
    assert matched == int((~nan).sum())
    assert np.array_equal(np.isnan(got).any(axis=1), nan)
    hit = dec & (d1 <= md)
    assert np.array_equal(got[hit], rounded(tgt_index[i1[hit]], store_dt))
    assert nan[dec & (d1 > md)].all()
    und = ~dec
    m = und & ~nan
    slack = 2.0 * UNIT[store_dt] * np.linalg.norm(got[m], axis=1)
    dist = np.linalg.norm(got[m] - q[m], axis=1)
    assert np.all(dist <= d1[m] + err(d1)[m] + err(md)[m] + slack)
    assert np.all(dist <= md + err(md)[m] + u * md + slack)
    assert np.all(d1[und & nan] >= md - err(d1)[und & nan] - u * md)
    return float(und.mean()), err(d1)


@pytest.mark.gpu
@pytest.mark.parametrize("store_dt,index_dt,host_dt", DTYPES, ids=DTYPE_IDS)
@pytest.mark.parametrize("name", list(RANDOM_CASES))
def test_random_clouds_against_kdtree(env, name, store_dt, index_dt, host_dt):
    ctx = env
    src, tgt = random_case(name)
    xs, md = RANDOM_CASES[name]
    src_s = rounded(src, store_dt)
    tgt_i = rounded(tgt, host_dt, index_dt)
    with Reassoc(capi, ctx, src_s, tgt.astype(NP[host_dt]), md, store_dt, index_dt, xs[0]) as r:
        for x in xs:
            matched = capi.store_reassociate(r.st, x)
            share, dl = check_against_kdtree(r.st.download(1), matched, query_of(src_s, x), tgt_i, md,
                                             query_error(index_dt, src_s, x), index_dt, store_dt)
            print(f"{name} x={np.round(x, 3).tolist()}: delta median {np.median(dl):.2e} max {dl.max():.2e}, "
                  f"undecidable {100 * share:.3f} %")
            assert share < 0.01


@pytest.mark.gpu
@pytest.mark.parametrize("index_dt", [F32, F64])
@pytest.mark.parametrize("name", SHAPES)
def test_grid_shapes(env, name, index_dt):
    ctx = env
    tgt, q, md = shape_case(name)
    for store_dt, host_dt in ((F64, F64), (F32, F32), (F64, 1 - index_dt)):
        src = src_of(q, X_EXACT)
        tgt_i = rounded(tgt, host_dt, index_dt)
        src_s = rounded(src, store_dt)
        with Reassoc(capi, ctx, src_s, tgt.astype(NP[host_dt]), md, store_dt, index_dt, X_EXACT) as r:
            qs = query_of(src_s, X_EXACT)
            share, _ = check_against_kdtree(r.got, r.matched, qs, tgt_i, md, query_error(index_dt, src_s, X_EXACT),
                                            index_dt, store_dt)
            if name != "identical":              # 1 000 copies of one point: every query is a tie
                assert share < 0.01, (name, store_dt, share)
            if name in ("plane", "identical"):   # exact data: every answer is known
                ok, arg, _, _ = brute(qs, tgt_i, md)
                assert same(r.got, expected_targets(tgt_i, ok, arg, store_dt)), name
            if name == "plane":
                assert r.matched == len(q) // 2
            assert r.matched > 0


@pytest.mark.gpu
@pytest.mark.parametrize("index_dt", [F32, F64])
def test_empty_index(env, index_dt):
    ctx = env
    src = np.random.default_rng(2).uniform(-1, 1, (1000, 3))
    with Reassoc(capi, ctx, src, np.zeros((0, 3)), 0.5, F64, index_dt, X_EXACT) as r:
        assert r.matched == 0 and np.isnan(r.got).all()
        H, b, s = ctx.linearize(r.st, capi.make_problem(capi.MODEL_POINT2POINT), X_EXACT)
        assert not H.any() and not b.any() and s == 0.0


@pytest.mark.gpu
@pytest.mark.parametrize("nx", [256, 257])
def test_cap_lattice_known_answer(env, nx):
    """nx x 256 x 256 unit lattice at max_dist = 1: 2^24 cells and 8 193 scan tiles at nx = 256, one coarsening step at
    nx = 257.  Each query is its own lattice point + (0.25, -0.125, 0.375) and must match it."""
    ctx = env
    lat = cap_lattice(nx)
    src = lat + (CAP_OFFSET - np.array(X_EXACT[:3], dtype=np.float32))    # exact in fp32
    for index_dt, host_dt in ((F32, F32), (F64, F32)):
        with Reassoc(capi, ctx, src, lat if host_dt == F32 else lat.astype(np.float64), 1.0, F32, index_dt,
                     X_EXACT) as r:
            assert r.matched == len(lat)
            assert np.array_equal(r.got.astype(np.float32), lat)


@pytest.mark.gpu
def test_non_finite_targets_never_match():
    """One +inf and one -inf point, NaN in some points, every point NaN, every z NaN, finite points at +-1e308: each
    build returns (in a subprocess with a timeout) and matches as the same cloud without its non-finite points."""
    with tempfile.TemporaryDirectory() as tmp:
        res = nonfinite_worker_results(tmp)
    for (name, it, ht), (matched, got) in res.items():
        tgt, q, md = nonfinite_case(name)
        tgt_i = rounded(tgt, ht, it)
        keep = np.flatnonzero(np.all(np.isfinite(tgt_i), axis=1))
        src = src_of(q, X_EXACT)
        qs = query_of(src, X_EXACT)
        ok, arg, _, _ = brute(qs, tgt_i[keep], md)
        want = expected_targets(tgt_i[keep], ok, arg, F64)
        if name in ("all_nan", "z_nan"):
            assert not ok.any()
        if it == F64:
            assert matched == int(ok.sum()) and same(got, want), (name, it, ht)
        elif len(keep):   # fp32 distances: the decidable queries exactly, the rest within the rounding bound
            check_against_kdtree(got, matched, qs, tgt_i[keep], md, query_error(F32, src, X_EXACT), F32, F64)
        else:
            assert matched == 0 and np.isnan(got).all(), (name, it, ht)


# ---- inside lm_minimize ---------------------------------------------------------------------------------------------
def icp_orc(src, tgt, md, jac=orc.JAC_ANALYTICAL):
    return orc.Cost(orc.P2P_ICP, 6, 3, src.shape[0], a=src, jac_mode=jac, target=tgt, max_dist=md, cost_threads=4)


def decisive_prefix(r, ro, floor):
    k = min(len(r.sequence), len(ro.sequence))
    decisive = [i for i in range(k) if abs(ro.trace[i, 2] - ro.trace[i, 3]) > floor * ro.trace[i, 2]]
    return (decisive[-1] + 1) if decisive else 0


def lm_case(name):
    """name -> (device terms [(src, tgt or None, md, b or None)], jacobian)."""
    src, tgt = clouds()
    h = src.shape[0] // 2
    if name == "central":
        return [(src, tgt, FACHADA_MAX_DIST, None)], capi.JAC_CENTRAL
    if name == "icp+p2p":
        full, _, _, _ = fachada()
        pick = full[np.random.default_rng(3).choice(full.shape[0], 2000, replace=False)]
        T = orc.so3_convert6dof(X_TRUE)
        return [(src, tgt, FACHADA_MAX_DIST, None), (pick, None, None, pick @ T[:3, :3].T + T[:3, 3])], 0
    if name == "two_icp":
        return [(src[:h], tgt, FACHADA_MAX_DIST, None), (src[h:], tgt, 0.35, None)], 0
    raise KeyError(name)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["central", "icp+p2p", "two_icp", "shared_index"])
def test_lm_matches_oracle(env, name):
    """The device LM with re-association against the oracle's: the same trial sequence while the decisions are decisive,
    y0 of each of those trials, x to 1e-6.  Central differences move the intermediate iterates by the finite-difference
    noise (4e-5 of y0 measured on B200 in the middle of the solve), as forward ones do in test_icp.py."""
    ctx = env
    stores, probs, costs = [], [], []
    with ExitStack() as stack:      # closed in reverse order of creation, on failure too
        def store(src):
            st = capi.Store(ctx, capi.MODEL_POINT2POINT, src.shape[0], capi.F64)
            stack.callback(st.close)
            st.upload(0, src)
            stores.append(st)
            return st

        def index(tgt, md):
            ix = capi.NNIndex(ctx, tgt, md, dtype=capi.F64)
            stack.callback(ix.close)
            return ix

        def attach(st, ix):
            capi.store_set_target(st, ix)
            stack.callback(capi.store_set_target, st, None)

        if name == "shared_index":
            src, tgt = clouds()
            h = src.shape[0] // 2
            ix = index(tgt, FACHADA_MAX_DIST)
            for part in (src[:h], src[h:]):
                attach(store(part), ix)
                probs.append(capi.make_problem(capi.MODEL_POINT2POINT, capi.JAC_ANALYTICAL, capi.F64))
                costs.append(icp_orc(part, tgt, FACHADA_MAX_DIST))
        else:
            terms, jac = lm_case(name)
            for s, t, md, b in terms:
                st = store(s)
                if t is not None:
                    attach(st, index(t, md))
                    costs.append(icp_orc(s, t, md, jac))
                else:
                    st.upload(1, b)
                    costs.append(orc.Cost(orc.P2P, 6, 3, s.shape[0], a=s, b=b, jac_mode=jac))
                probs.append(capi.make_problem(capi.MODEL_POINT2POINT, jac, capi.F64))
        r = ctx.lm_minimize(stores, probs, [0.0] * 6, max_iterations=30)
    ro = orc.lm_minimize(costs, [0.0] * 6, max_iterations=30)
    cut = decisive_prefix(r, ro, 1e-9)
    print(f"{name}: {r.sequence} / oracle {ro.sequence}, |dx| {np.max(np.abs(r.x - ro.x)):.2e}")
    assert cut >= 3 and r.sequence[:cut] == ro.sequence[:cut]
    assert np.allclose(r.trace[:cut, 2], ro.trace[:cut, 2], rtol=1e-9 if name != "central" else 1e-4)
    assert np.max(np.abs(r.x - ro.x)) < 1e-6
    assert np.allclose(r.x, X_TRUE, atol=2e-3)


@pytest.mark.gpu
def test_lm_fp32_store_index_and_compute(env):
    """fp32 store, fp32 index, fp32 compute against the float oracle on the same fp32 data.  y0 is a sum of ~2 800
    fp32-evaluated squared residuals, so decisions are compared while the relative decrease is above 1e-5 of y0, as
    for the plain fp32 point2point solve (test_p2p_lm_fp32_store_reaches_ground_truth).  Near the solution each
    residual is a ~2e-3 m difference of ~20 m fp32 coordinates (6e-4 relative rounding), and the float oracle adds the
    ~2 800 squares serially in fp32 (up to n u = 1.7e-4 relative): y0 is held to 2e-4 (5.7e-5 measured on B200).
    x: 1e-5 (2.2e-6 measured, on a translation of 0.12)."""
    ctx = env
    src, tgt = clouds()
    src32, tgt32 = src.astype(np.float32), tgt.astype(np.float32)
    st = capi.Store(ctx, capi.MODEL_POINT2POINT, src.shape[0], capi.F32)
    try:
        st.upload(0, src32)
        ix = capi.NNIndex(ctx, tgt32, FACHADA_MAX_DIST, dtype=capi.F32)
        try:
            capi.store_set_target(st, ix)
            r = ctx.lm_minimize([st], [capi.make_problem(capi.MODEL_POINT2POINT, capi.JAC_ANALYTICAL, capi.F32)],
                                [0.0] * 6, max_iterations=30)
            capi.store_set_target(st, None)
        finally:
            ix.close()
    finally:
        st.close()
    ro = orc.lm_minimize([icp_orc(src32, tgt32, FACHADA_MAX_DIST)], [0.0] * 6, max_iterations=30, scalar=orc.F32)
    cut = decisive_prefix(r, ro, 1e-5)
    print(f"fp32 ICP LM: {r.sequence} / float oracle {ro.sequence}, |dx| {np.abs(r.x - ro.x)}")
    assert cut >= 3 and r.sequence[:cut] == ro.sequence[:cut]
    assert np.allclose(r.trace[:cut, 2], ro.trace[:cut, 2], rtol=2e-4)
    assert np.max(np.abs(r.x - ro.x)) < 1e-5
    assert np.allclose(r.x, X_TRUE, atol=2e-3)


# ---- error paths ----------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_error_paths(env):
    ctx = env
    tgt = np.random.default_rng(1).uniform(0, 1, (100, 3))
    for md in (0.0, -0.5, float("nan"), float("inf")):
        with pytest.raises(capi.MoptError):
            capi.NNIndex(ctx, tgt, md)
    ix = capi.NNIndex(ctx, tgt, 0.1)
    curve = capi.Store(ctx, capi.MODEL_EXP_CURVE, 10, capi.F64)
    with pytest.raises(capi.MoptError):
        capi.store_set_target(curve, ix)
    st = capi.Store(ctx, capi.MODEL_POINT2POINT, 10, capi.F64)
    with pytest.raises(capi.MoptError):
        capi.store_reassociate(st, [0.0] * 6)
    other = capi.Context(0)
    try:
        ix2 = capi.NNIndex(other, tgt, 0.1)
        with pytest.raises(capi.MoptError):
            capi.store_set_target(st, ix2)
        ix2.close()
    finally:
        other.close()
    capi.store_set_target(st, ix)
    capi.store_reassociate(st, [0.0] * 6)
    capi.store_set_target(st, None)
    with pytest.raises(capi.MoptError):
        capi.store_reassociate(st, [0.0] * 6)
    ix.close()
    curve.close()
    st.close()
