"""The map pipeline against exact references: occupancy grid -> distance transform (k_edt) -> map storage (k_brick: f32
reciprocal clearance or u8 quantisation, bricked layout) -> what the cost kernel reads.

References are independent of the library: the FP64 oracle's EDT, the closed form of a single obstacle, and numpy
statements of the storage rules in include/lmcma_b200.h.  Bars as in test_gpu_parity.py: distances and stored values
bit-exact, collision and sample counts bit-exact, costs within COST_RTOL of po.CostProblem on the row-major map."""
import numpy as np
import pytest

import lmcma_path_planner_b200 as L
from lmcma_path_planner_b200 import _capi as K
from lmcma_path_planner_b200 import maps

pytestmark = pytest.mark.gpu

COST_RTOL = 1e-5
FLT_MAX = np.finfo(np.float32).max
F32 = np.float32


def rel_err(a, b, floor=1e-30):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), floor))) if a.size else 0.0


def bits_equal(a, b):
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


def mismatch(got, want):
    """Where two distance fields differ: count, and the smallest / largest wanted distance among those cells."""
    bad = got.view(np.uint32) != want.view(np.uint32)
    if not bad.any():
        return "equal"
    return "%d cells differ, wanted distances %.3f .. %.3f there, got e.g. %r" % (
        int(bad.sum()), float(want[bad].min()), float(want[bad].max()), float(got[bad][0]))


# ---- independent statements of the header's rules (include/lmcma_b200.h) ----
def clamped(d, clamp):
    return np.minimum(d, F32(clamp)) if clamp > 0 else d


def one_obstacle_field(shape_xyz, at_xyz, clamp=0.0):
    """Exact distance to a single obstacle cell: float32(sqrt(float64(dx^2 + dy^2 [+ dz^2]))), array order [z][y][x]."""
    dims = len(shape_xyz)
    d2 = np.zeros(shape_xyz[::-1], np.float64)
    for c in range(dims):
        a = (np.arange(shape_xyz[c], dtype=np.float64) - at_xyz[c]) ** 2
        d2 += a.reshape([-1 if dims - 1 - k == c else 1 for k in range(dims)])
    return clamped(np.sqrt(d2).astype(np.float32), clamp)


def u8_rule(E, scale):
    """q = E > 0 ? clamp(floor(E / u8_scale), 1, 255) : 0 in FP32 (IEEE division), read back as float32(q) * scale."""
    E, s = np.asarray(E, np.float32), F32(scale)
    with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
        q = np.where(E > 0, np.clip(np.floor(E / s), 1, 255), 0).astype(np.float32)
    return (q * s).astype(np.float32)


def f32_rule(E, c_min):
    """Stored g = E > 0 ? 1 / max(E, c_min) : -1 / c_min, read back as g < 0 ? 0 : 1 / g (FP32, IEEE)."""
    E, c = np.asarray(E, np.float32), F32(c_min)
    with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
        g = np.where(E > 0, F32(1) / np.maximum(E, c), -F32(1) / c).astype(np.float32)
        return np.where(g < 0, F32(0), F32(1) / g).astype(np.float32)


def stored_rule(E, storage, u8_scale, c_min):
    return u8_rule(E, u8_scale) if storage == "u8" else f32_rule(E, c_min)


# ------------------------------------------------------------------------------------------------
# a. exact distance transform at its edges
# ------------------------------------------------------------------------------------------------
# (shape xyz, obstacle xyz).  Squared distances here go past 2^29 (distance 23 170.475), up to the longest axis accepted.
PAST_SENTINEL = {
    "x_pass_24000x3": ((24000, 3), (0, 1)),
    "y_pass_3x30000": ((3, 30000), (1, 0)),
    "z_pass_1x1x30000": ((1, 1, 30000), (0, 0, 29999)),
    # the x pass stays below 2^29; only the second pass crosses it
    "second_pass_23170x600": ((23170, 600), (0, 0)),
    "second_pass_23170x1x600": ((23170, 1, 600), (23169, 0, 599)),
    # the longest axis the ABI accepts
    "x_axis_32767": ((32767, 2), (32766, 0)),
    "y_axis_32767": ((2, 32767), (0, 0)),
    "z_axis_32767": ((1, 1, 32767), (0, 0, 32766)),
}


def occupancy_with(shape_xyz, at_xyz):
    occ = np.zeros(shape_xyz[::-1], np.uint8)
    occ[tuple(at_xyz[::-1])] = 1
    return occ


@pytest.mark.parametrize("case", sorted(PAST_SENTINEL))
def test_edt_exact_past_the_squared_distance_sentinel(case):
    """Distances of more than 23 170 cells are real distances, with the clamp off, above them (30 000) and just below
    the old sentinel's distance (23 170.3)."""
    shape, at = PAST_SENTINEL[case]
    occ = occupancy_with(shape, at)
    exact = one_obstacle_field(shape, at)
    assert exact.max() > 23170.5                      # the case does reach past the old sentinel
    bad = {}
    for clamp in (0.0, 30000.0, 23170.3):
        got = maps.edt_device(occ, clamp=clamp)
        want = clamped(exact, clamp)
        if not bits_equal(got, want):
            bad[clamp] = mismatch(got, want)
    assert not bad, (case, bad)


@pytest.mark.parametrize("case", ["x_pass_24000x3", "z_pass_1x1x30000", "second_pass_23170x600"])
@pytest.mark.parametrize("storage", ["f32", "u8"])
def test_map_from_occupancy_past_the_squared_distance_sentinel(case, storage):
    """The same distances through from_occupancy, unclamped: the stored map reads back as the header's rule applied to
    the exact distance (u8_scale 128 keeps distances up to 32 767 cells on distinct levels)."""
    shape, at = PAST_SENTINEL[case]
    cm = L.CostMap.from_occupancy(occupancy_with(shape, at), 0.0, storage, u8_scale=128.0, c_min=0.5)
    want = stored_rule(one_obstacle_field(shape, at), storage, 128.0, 0.5)
    got = cm.dequantized()
    assert bits_equal(got, want), (case, storage, mismatch(got, want))


@pytest.mark.parametrize("shape", [(32768, 1), (1, 32768), (1, 1, 32768), (32768, 2, 1)])
def test_axis_longer_than_32767_cells_is_refused(shape):
    occ = np.zeros(shape[::-1], np.uint8)
    occ.flat[0] = 1
    with pytest.raises(K.LmcmaError) as e:
        maps.edt_device(occ)
    assert e.value.code == K.ERR_ARG
    for storage in ("f32", "u8"):
        with pytest.raises(K.LmcmaError) as e:
            L.CostMap.from_occupancy(occ, 0.0, storage)
        assert e.value.code == K.ERR_ARG


def _random_occupancy(rng, shape, p):
    occ = (rng.random(shape) < p).astype(np.uint8)
    occ.flat[int(rng.integers(occ.size))] = 1         # never empty: the oracle has no "no obstacle" sentinel
    return occ


# array order [z][y][x] / [y][x]
DEGENERATE = [(1, 1), (1, 777), (777, 1), (1, 1, 1), (1, 1, 90), (1, 90, 1), (90, 1, 1), (1, 19, 37), (19, 1, 37), (19, 37, 1)] + \
             [(5, n) for n in (31, 32, 33, 63, 64, 65)] + [(3, 2, n) for n in (31, 32, 33, 63, 64, 65)]


@pytest.mark.parametrize("shape", DEGENERATE, ids=lambda s: "x".join(map(str, s[::-1])))
def test_edt_degenerate_shapes_and_scan_chunk_edges(po, shape):
    """Axes of length 1, and x lines of 31 .. 65 cells (the chunk carry of pass x's warp scans): random sparse and dense
    obstacles, an obstacle only at the first or only at the last cell of a line, with and without the clamp."""
    rng = np.random.default_rng(sum(shape) * 7 + len(shape))
    cases = [_random_occupancy(rng, shape, p) for p in (0.02, 0.3)]
    for first in (True, False):
        occ = np.zeros(shape, np.uint8)
        occ[..., 0 if first else -1] = 1
        cases.append(occ)
    for occ in cases:
        want = po.edt_exact(occ)
        got = maps.edt_device(occ)
        assert bits_equal(got, want), (shape, mismatch(got, want))
        assert bits_equal(maps.edt_device(occ, clamp=2.5), np.minimum(want, F32(2.5))), shape


EMPTY_FULL = [(1, 1), (7, 33), (1, 1, 1), (3, 5, 65), (2, 9, 17)]


@pytest.mark.parametrize("shape", EMPTY_FULL, ids=lambda s: "x".join(map(str, s[::-1])))
def test_edt_grid_without_obstacles_and_grid_of_obstacles_only(shape):
    """Only obstacles: all zeros.  No obstacle: the clamp when one is set, FLT_MAX when not (include/lmcma_b200.h); the
    map built from it reads back as the header's rule applied to that value."""
    full, empty = np.ones(shape, np.uint8), np.zeros(shape, np.uint8)
    for clamp in (0.0, 9.25):
        assert bits_equal(maps.edt_device(full, clamp=clamp), np.zeros(shape, np.float32)), clamp
        want = np.full(shape, F32(clamp) if clamp > 0 else FLT_MAX, np.float32)
        got = maps.edt_device(empty, clamp=clamp)
        assert bits_equal(got, want), (clamp, got.ravel()[:4])
        for storage in ("f32", "u8"):
            for occ, field in ((full, np.zeros(shape, np.float32)), (empty, want)):
                cm = L.CostMap.from_occupancy(occ, clamp, storage, u8_scale=0.25, c_min=0.5)
                assert bits_equal(cm.dequantized(), stored_rule(field, storage, 0.25, 0.5)), (clamp, storage, occ.max())


# ------------------------------------------------------------------------------------------------
# b. map storage against numpy statements of the header's rules, on both sides of every brick size
# ------------------------------------------------------------------------------------------------
# xyz; bricks: 2-D f32 8 x 4, u8 16 x 8; 3-D f32 4 x 4 x 2, u8 8 x 4 x 4
STORAGE_SHAPES = [(1, 1), (8, 4), (9, 5), (16, 8), (17, 9), (1, 1, 1), (4, 4, 2), (5, 5, 3), (8, 4, 4), (33, 17, 9)]
SHAPE_IDS = ["x".join(map(str, s)) for s in STORAGE_SHAPES]


def _special_u8_values(scale):
    s = F32(scale)
    mult = np.array([1, 2, 3, 7, 100, 254, 255, 256], np.float32) * s               # exact multiples (FP32 products)
    vals = [F32(1e-45), F32(1e-38), s * F32(0.5), np.nextafter(s, F32(0))]         # 0 < E < scale
    vals += list(mult) + list(np.nextafter(mult, F32(0))) + list(np.nextafter(mult, F32(np.inf)))
    vals += [F32(256) * s, F32(300) * s, F32(1e30), FLT_MAX]                       # saturation
    vals += [F32(np.inf), F32(np.nan), F32(-0.0), F32(0.0), F32(-1.0), F32(-np.inf), F32(-1e-45)]
    return np.array(vals, np.float32)


def _special_f32_values(c_min):
    c = F32(c_min)
    vals = [F32(1e-45), F32(1e-38), c, np.nextafter(c, F32(0)), np.nextafter(c, F32(np.inf)), c * F32(0.5), c * F32(3),
            F32(1.0), F32(1 / 3), F32(1e30), FLT_MAX, F32(np.inf), F32(np.nan), F32(-0.0), F32(0.0), F32(-1.0), F32(-np.inf)]
    return np.array(vals, np.float32)


def _fill(rng, shape_xyz, special, hi):
    """Every cell from a seeded mix: the special values (each at least once when there are enough cells) and uniform
    values in [0, hi)."""
    n = int(np.prod(shape_xyz))
    pool = np.concatenate([special, rng.uniform(0, hi, size=max(0, n - len(special))).astype(np.float32)])
    pool = pool[rng.permutation(len(pool))][:n] if n < len(pool) else rng.permutation(pool)
    return pool.reshape(shape_xyz[::-1]).astype(np.float32)


@pytest.mark.parametrize("scale", [0.25, 1 / 3, 0.1, 2.0])
@pytest.mark.parametrize("shape", STORAGE_SHAPES, ids=SHAPE_IDS)
def test_u8_storage_equals_the_quantisation_rule(shape, scale):
    rng = np.random.default_rng(len(shape) * 1000 + int(np.prod(shape)) + int(scale * 100))
    E = _fill(rng, shape, _special_u8_values(scale), 300 * scale)
    got = L.CostMap(E, "u8", u8_scale=scale, c_min=0.5).dequantized()
    want = u8_rule(E, scale)
    bad = got.view(np.uint32) != want.view(np.uint32)
    assert not bad.any(), (shape, scale, E[bad][:6], got[bad][:6], want[bad][:6])


@pytest.mark.parametrize("c_min", [0.1, 0.5, 7.5])
@pytest.mark.parametrize("shape", STORAGE_SHAPES, ids=SHAPE_IDS)
def test_f32_storage_reads_back_as_the_floored_clearance(shape, c_min):
    rng = np.random.default_rng(len(shape) * 1000 + int(np.prod(shape)) + int(c_min * 10))
    E = _fill(rng, shape, _special_f32_values(c_min), 20.0)
    got = L.CostMap(E, "f32", u8_scale=0.25, c_min=c_min).dequantized()
    want = f32_rule(E, c_min)
    bad = got.view(np.uint32) != want.view(np.uint32)
    assert not bad.any(), (shape, c_min, E[bad][:6], got[bad][:6], want[bad][:6])


# ------------------------------------------------------------------------------------------------
# c. layout-sensitive costs: i.i.d. random maps, trajectories into the last row / column / plane
# ------------------------------------------------------------------------------------------------
# sizes that are multiples of no brick extent; the last index is even along x (n - 0.5 rounds to the last cell) and odd
# along y (n - 0.5 rounds to n: outside)
LAYOUT_SHAPES = {2: (37, 22), 3: (21, 14, 11)}
LAYOUT_CASES = [(2, "f32", 0.25, 0.5), (2, "f32", 0.25, 3.0), (2, "u8", 0.25, 0.5), (2, "u8", 0.23, 3.0),
                (3, "f32", 0.25, 0.5), (3, "f32", 0.25, 3.0), (3, "u8", 0.25, 0.5), (3, "u8", 0.23, 3.0)]
LAYOUT_IDS = ["%dd-%s-scale%g-cmin%g" % c for c in LAYOUT_CASES]


def random_field(rng, shape_xyz, storage, scale):
    """i.i.d. values in [0.6, 60), about 10 % obstacles; for u8, mid-level values of distinct quantisation levels."""
    shp = shape_xyz[::-1]
    if storage == "u8":
        q = rng.integers(int(np.ceil(0.6 / scale)), min(256, int(60 / scale)), size=shp)
        E = ((q + 0.5) * scale).astype(np.float32)
    else:
        E = rng.uniform(0.6, 60.0, size=shp).astype(np.float32)
    E[rng.random(shp) < 0.1] = 0.0
    return E


def endpoint_pairs(shape_xyz):
    n = np.asarray(shape_xyz, np.float64)
    last, half = n - 1.0, n - 0.5
    return [(np.full(len(n), 1.0), last),                               # goal on the last cell
            (half, np.full(len(n), 0.3)),                               # start at n - 0.5 on every axis
            (np.concatenate([[-3.0], last[1:] * 0.5]), n + 2.0),        # both outside the map
            (np.concatenate([[half[0]], np.zeros(len(n) - 1)]), np.concatenate([last[:-1], [half[-1]]]))]


def trajectories(rng, shape_xyz, count, W):
    """Dimension-major waypoints; each coordinate from [-1.5, n + 0.5) or from the last few cells, [n - 3, n + 0.25)."""
    n = np.asarray(shape_xyz, np.float64)[:, None, None]
    wide = rng.uniform(-1.5, n + 0.5, size=(len(shape_xyz), count, W))
    edge = rng.uniform(n - 3.0, n + 0.25, size=(len(shape_xyz), count, W))
    X = np.where(rng.random((len(shape_xyz), count, W)) < 0.5, wide, edge)
    return np.ascontiguousarray(X.transpose(1, 0, 2).reshape(count, -1)).astype(np.float32)


@pytest.mark.parametrize("dims,storage,scale,c_min", LAYOUT_CASES, ids=LAYOUT_IDS)
def test_cost_on_a_random_map_reads_every_cell_from_its_place(po, dims, storage, scale, c_min):
    shape = LAYOUT_SHAPES[dims]
    rng = np.random.default_rng(dims * 10 + len(storage) + int(c_min))
    E = random_field(rng, shape, storage, scale)
    ref_map = stored_rule(E, storage, scale, c_min) if storage == "u8" else E
    cm = L.CostMap(E, storage, u8_scale=scale, c_min=c_min)
    assert bits_equal(cm.dequantized(), stored_rule(E, storage, scale, c_min))
    W = 6
    X = trajectories(rng, shape, 300, W)
    seen = set()
    for start, goal in endpoint_pairs(shape):
        prob = po.CostProblem(ref_map, start, goal, W, c_min=c_min)
        ref = prob.evaluate(X)
        got = cm.evaluate(X, start, goal, W)
        assert np.array_equal(got["ncoll"], ref["ncoll"]), (start, goal)
        assert np.array_equal(got["nsamp"], ref["nsamp"]), (start, goal)
        assert rel_err(got["f"], ref["f"]) < COST_RTOL, (start, goal, rel_err(got["f"], ref["f"]))
        for x in X[:40]:
            cells = prob.trace(x, max_cells=1 << 14)
            seen.update(int(c) for c in cells[cells >= 0])
    # the trajectories do read the last column, row and plane
    idx = np.unravel_index(np.array(sorted(seen)), shape[::-1])
    for axis in range(dims):
        assert (idx[dims - 1 - axis] == shape[axis] - 1).any(), axis


# ------------------------------------------------------------------------------------------------
# d. from_occupancy == map_create(exact EDT)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("clamp", [0.0, 6.5])
@pytest.mark.parametrize("dims,storage,scale,c_min", [(2, "f32", 0.25, 0.5), (2, "f32", 0.25, 1.7), (2, "u8", 0.25, 0.5),
                                                      (2, "u8", 0.09, 1.7), (3, "f32", 0.25, 0.5), (3, "f32", 0.25, 1.7),
                                                      (3, "u8", 0.25, 0.5), (3, "u8", 0.09, 1.7)],
                         ids=lambda v: str(v))
def test_map_from_occupancy_equals_map_from_the_exact_field(po, dims, storage, scale, c_min, clamp):
    shape = LAYOUT_SHAPES[dims]
    rng = np.random.default_rng(dims * 100 + int(clamp) + int(c_min * 10))
    occ = maps.random_boxes_occupancy(shape[::-1], 6, 1, 4, seed=dims + int(clamp), border=0)
    occ[rng.random(occ.shape) < 0.02] = 1
    a = L.CostMap.from_occupancy(occ, clamp, storage, u8_scale=scale, c_min=c_min)
    b = L.CostMap(po.edt_exact(occ, clamp), storage, u8_scale=scale, c_min=c_min)
    assert bits_equal(a.dequantized(), b.dequantized())
    W = 6
    X = trajectories(rng, shape, 200, W)
    for start, goal in endpoint_pairs(shape)[:2]:
        ra, rb = a.evaluate(X, start, goal, W), b.evaluate(X, start, goal, W)
        assert np.array_equal(ra["f"], rb["f"]) and np.array_equal(ra["ncoll"], rb["ncoll"]) and \
            np.array_equal(ra["nsamp"], rb["nsamp"]), (start, goal)
