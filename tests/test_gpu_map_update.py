"""In-place occupancy updates of a cost map (lmcma_b200_map_update_occupancy) and re-scoring the best-so-far candidates on
the updated map (lmcma_b200_rescore_best).

The oracle of an update is a fresh build: after CostMap.update_occupancy the map must hold, bit for bit, what
CostMap.from_occupancy of the edited grid holds, and evaluate the same costs, collision counts and sample counts.  Optimiser
handles attached to the map must follow the update without re-attaching: a twin re-attached to the fresh map at the same
point computes the same bits."""
import ctypes as C

import numpy as np
import pytest

import lmcma_path_planner_b200 as L
from lmcma_path_planner_b200 import _capi as K
from lmcma_path_planner_b200 import maps

pytestmark = pytest.mark.gpu

F32 = np.float32
FLT_MAX = np.finfo(np.float32).max
HUGE_CLAMP = 1e4                    # past the diagonal of every grid here


def bits_equal(a, b):
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


def box_slices(lo_xyz, size_xyz):
    """Array-order slices ([z][y][x]) of the box [lo, lo + size) given in x y [z]."""
    return tuple(slice(lo_xyz[c], lo_xyz[c] + size_xyz[c]) for c in reversed(range(len(lo_xyz))))


def edited(occ, lo_xyz, box):
    out = (np.asarray(occ) != 0).astype(np.uint8)
    out[box_slices(lo_xyz, box.shape[::-1])] = np.asarray(box) != 0
    return out


def random_paths(shape_xyz, count, waypoints, seed):
    """count trajectories of `waypoints` interior points drawn uniformly over the grid, dimension-major rows."""
    rng = np.random.default_rng(seed)
    cols = [rng.uniform(0.0, s - 1.0, (count, waypoints)) for s in shape_xyz]
    return np.concatenate(cols, axis=1).astype(np.float32)


def assert_same_map(got, want, shape_xyz, seed=0, what=""):
    """Bit-equal stored values, and bit-equal f / ncoll / nsamp of seeded random trajectories."""
    assert bits_equal(got.dequantized(), want.dequantized()), what
    W = 6
    X = random_paths(shape_xyz, 64, W, seed)
    start, goal = [0.0] * len(shape_xyz), [s - 1.0 for s in shape_xyz]
    a = got.evaluate(X, start, goal, W, L.LONGSAFE, 1e4)
    b = want.evaluate(X, start, goal, W, L.LONGSAFE, 1e4)
    for k in ("f", "ncoll", "nsamp"):
        assert np.array_equal(a[k].view(np.uint32) if k == "f" else a[k], b[k].view(np.uint32) if k == "f" else b[k]), (what, k)


EDITS = ("add", "clear", "mix", "cell", "lo0", "hi", "whole")


def make_edit(shape_xyz, kind, clamp, seed):
    """(grid, lo_xyz, box) of one edit kind on a sparse random grid of shape_xyz (x y [z]).
    clear: the box holds the only obstacles near it, plus one obstacle floor(clamp) cells beyond its +x face (exactly the
    clamp for an integer clamp); clearing it changes the distances up to the clamp beyond the box."""
    rng = np.random.default_rng(seed)
    dims = len(shape_xyz)
    occ = (rng.random(shape_xyz[::-1]) < 0.03).astype(np.uint8)
    if kind == "whole":
        lo, size = (0,) * dims, tuple(shape_xyz)
    elif kind == "cell":
        lo, size = tuple(s // 2 for s in shape_xyz), (1,) * dims
    elif kind == "lo0":
        lo, size = (0,) * dims, tuple(max(1, s // 4) for s in shape_xyz)
    elif kind == "hi":
        size = tuple(max(1, s // 4) for s in shape_xyz)
        lo = tuple(s - z for s, z in zip(shape_xyz, size))
    else:
        size = tuple(max(1, min(4, s // 4)) for s in shape_xyz)
        lo = tuple((s - z) // 2 for s, z in zip(shape_xyz, size))
    bshape = size[::-1]
    if kind == "add":
        box = np.ones(bshape, np.uint8)
    elif kind == "clear":
        r = int(np.ceil(clamp)) if 0 < clamp < HUGE_CLAMP else 4
        hood_lo = tuple(max(0, l - 2 * r) for l in lo)
        hood_sz = tuple(min(s, l + z + 2 * r) - h for s, l, z, h in zip(shape_xyz, lo, size, hood_lo))
        occ[box_slices(hood_lo, hood_sz)] = 0
        occ[box_slices(lo, size)] = 1
        far = [lo[0] + size[0] - 1 + (int(np.floor(clamp)) if 0 < clamp < HUGE_CLAMP else r)] + list(lo[1:])
        if far[0] < shape_xyz[0]:
            occ[tuple(far[::-1])] = 1
        box = np.zeros(bshape, np.uint8)
    elif kind == "cell":
        box = 1 - occ[box_slices(lo, size)]
    else:
        box = (rng.random(bshape) < 0.3).astype(np.uint8)
    return occ, lo, box


SHAPES = {"2d-37x22": (37, 22), "2d-301x203": (301, 203), "3d-21x14x11": (21, 14, 11), "3d-61x45x37": (61, 45, 37)}


@pytest.mark.parametrize("storage", ["f32", "u8"])
@pytest.mark.parametrize("clamp", [0.0, 6.0, 6.5, HUGE_CLAMP])
@pytest.mark.parametrize("shape", list(SHAPES))
def test_update_equals_rebuild(shape, clamp, storage):
    """Every edit kind, on grids whose extents are not multiples of the bricks: clamp 0 (whole-grid recompute), clamps
    small enough that the windows are a strict part of the larger grids, and a clamp past the diagonal."""
    shape_xyz = SHAPES[shape]
    for i, kind in enumerate(EDITS):
        occ, lo, box = make_edit(shape_xyz, kind, clamp, seed=100 + i)
        cm = L.CostMap.from_occupancy(occ, clamp, storage)
        cm.update_occupancy(lo, box)
        fresh = L.CostMap.from_occupancy(edited(occ, lo, box), clamp, storage)
        assert_same_map(cm, fresh, shape_xyz, seed=i, what=(shape, clamp, storage, kind))
        cm.close()
        fresh.close()


@pytest.mark.parametrize("storage", ["f32", "u8"])
@pytest.mark.parametrize("clamp", [0.0, 6.5])
@pytest.mark.parametrize("shape", ["2d-301x203", "3d-61x45x37"])
def test_twenty_updates_in_sequence(shape, clamp, storage):
    """Each of twenty seeded random edits, applied one after the other, leaves what a build of the running grid holds."""
    shape_xyz = SHAPES[shape]
    rng = np.random.default_rng(7)
    grid = (rng.random(shape_xyz[::-1]) < 0.02).astype(np.uint8)
    cm = L.CostMap.from_occupancy(grid, clamp, storage)
    for step in range(20):
        size = tuple(int(rng.integers(1, min(s, 24) + 1)) for s in shape_xyz)
        lo = tuple(int(rng.integers(0, s - z + 1)) for s, z in zip(shape_xyz, size))
        box = (rng.random(size[::-1]) < rng.uniform(0.0, 0.6)).astype(np.uint8)
        cm.update_occupancy(lo, box)
        grid = edited(grid, lo, box)
        fresh = L.CostMap.from_occupancy(grid, clamp, storage)
        assert_same_map(cm, fresh, shape_xyz, seed=step, what=(shape, clamp, storage, step))
        fresh.close()
    cm.close()


def f32_rule(E, c_min):
    E, c = np.asarray(E, np.float32), F32(c_min)
    with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
        g = np.where(E > 0, F32(1) / np.maximum(E, c), -F32(1) / c).astype(np.float32)
        return np.where(g < 0, F32(0), F32(1) / g).astype(np.float32)


def u8_rule(E, scale):
    E, s = np.asarray(E, np.float32), F32(scale)
    with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
        q = np.where(E > 0, np.clip(np.floor(E / s), 1, 255), 0).astype(np.float32)
    return (q * s).astype(np.float32)


@pytest.mark.parametrize("storage", ["f32", "u8"])
@pytest.mark.parametrize("clamp", [0.0, 6.5])
@pytest.mark.parametrize("shape", ["2d-37x22", "3d-21x14x11"])
def test_clearing_every_obstacle_gives_the_empty_grid_rule(shape, clamp, storage):
    """No obstacle left: the clamp everywhere, or FLT_MAX unclamped (include/lmcma_b200.h), through the storage rule.
    Once by a box over the whole grid, once by a box that holds every obstacle."""
    shape_xyz = SHAPES[shape]
    E = np.full(shape_xyz[::-1], F32(clamp) if clamp > 0 else FLT_MAX, np.float32)
    want = u8_rule(E, 0.25) if storage == "u8" else f32_rule(E, 0.5)
    lo = tuple(s // 3 for s in shape_xyz)
    size = tuple(max(1, s // 3) for s in shape_xyz)
    occ = np.zeros(shape_xyz[::-1], np.uint8)
    occ[box_slices(lo, size)] = np.random.default_rng(3).random(size[::-1]) < 0.5
    occ[box_slices(lo, (1,) * len(lo))] = 1
    for box_lo, box_size in (((0,) * len(shape_xyz), shape_xyz), (lo, size)):
        cm = L.CostMap.from_occupancy(occ, clamp, storage)
        cm.update_occupancy(box_lo, np.zeros(box_size[::-1], np.uint8))
        assert bits_equal(cm.dequantized(), want), (box_lo, box_size)
        cm.close()


def _raw_update(cm, lo, size, occ):
    lo_a, size_a = np.array(lo, np.int32), np.array(size, np.int32)
    return K.lib().lmcma_b200_map_update_occupancy(cm._h, K.iptr(lo_a), K.iptr(size_a),
                                                   None if occ is None else occ.ctypes.data_as(C.POINTER(C.c_uint8)))


@pytest.mark.parametrize("storage", ["f32", "u8"])
def test_refused_updates_leave_the_map_unchanged(storage):
    shape_xyz = (37, 22)
    occ = (np.random.default_rng(5).random(shape_xyz[::-1]) < 0.05).astype(np.uint8)
    cm = L.CostMap.from_occupancy(occ, 6.0, storage)
    before = cm.dequantized()
    ones = np.ones(64 * 64, np.uint8)
    for lo, size, buf in (((0, 0), (4, 4), None),              # null box
                          ((0, 0), (0, 4), ones),              # size below 1
                          ((3, 3), (4, -1), ones),
                          ((-1, 0), (4, 4), ones),             # box not inside the grid
                          ((34, 0), (4, 4), ones),
                          ((0, 19), (4, 4), ones),
                          ((0, 0), (38, 22), ones),
                          ((2**31 - 2, 0), (4, 4), ones)):
        assert _raw_update(cm, lo, size, buf) == K.ERR_ARG, (lo, size)
        assert bits_equal(cm.dequantized(), before), (lo, size)
    # a map built from a caller's distance field has no occupancy behind it
    dm = L.CostMap(maps.distance_field(occ), storage)
    dbefore = dm.dequantized()
    assert _raw_update(dm, (0, 0), (4, 4), ones) == K.ERR_STATE
    assert bits_equal(dm.dequantized(), dbefore)
    cm.close()
    dm.close()


# ------------------------------------------------------------------------------------------------
# attached optimisers: the C2-shaped problem of test_gpu_launch_graphs.py on a map built from its occupancy
# ------------------------------------------------------------------------------------------------
W, LAM, M, SIZE, CLAMP = 200, 1024, 40, 1024, 64.0
KEYS = ("X", "xmean", "sigma", "V", "P", "pc", "fit", "t", "vec", "Nj", "Lj")


def launches():
    return K.lib().lmcma_b200_launch_count()


@pytest.fixture(scope="module")
def c2():
    """The occupancy behind maps.config2_map(size=1024, n_rects=128, seed=42), an edit that crosses the straight path
    from start to goal, and the grid with it applied."""
    start, goal = (64.0, 64.0), (SIZE - 64.0, SIZE - 64.0)
    occ = maps.random_boxes_occupancy((SIZE, SIZE), 128, 8, 128, 42, border=2, clear=[(start, 64.0), (goal, 64.0)])
    lo, box = (488, 488), np.ones((48, 48), np.uint8)
    return dict(occ=occ, start=start, goal=goal, lo=lo, box=box, edited=edited(occ, lo, box),
                x0=maps.straight_line(start, goal, W), bounds=maps.box_bounds((SIZE, SIZE), W))


def _handle(p, cmap, monkeypatch, env=None, batch=1, seed=3):
    for k, v in (env or {}).items():
        monkeypatch.setenv(k, v)
    lo, hi = p["bounds"]
    x0 = np.repeat(p["x0"][None], batch, 0)
    dev = L.Optimizer(2 * W, x0=x0, lam=LAM, m=M, batch=batch, lo=lo, hi=hi, sigma0=16.0, seed=seed)
    for k in env or {}:
        monkeypatch.delenv(k)
    dev.attach_cost(cmap, [p["start"]], [p["goal"]], W, L.LONGSAFE, 1e4)
    return dev


FOLLOW_CASES = {"c2": dict(), "c2-linear": dict(env={"LMCMA_B200_OVERLAP": "0"}), "batch8": dict(batch=8)}


@pytest.mark.parametrize("case", list(FOLLOW_CASES))
def test_attached_handles_follow_an_update_without_reattaching(c2, monkeypatch, case):
    p, c = c2, FOLLOW_CASES[case]
    old = L.CostMap.from_occupancy(p["occ"], CLAMP, "f32")
    cmap = L.CostMap.from_occupancy(p["occ"], CLAMP, "f32")
    fresh = L.CostMap.from_occupancy(p["edited"], CLAMP, "f32")
    dev = _handle(p, cmap, monkeypatch, **c)
    twin = _handle(p, old, monkeypatch, **c)
    dev.run(3)
    twin.run(3)
    cmap.update_occupancy(p["lo"], p["box"])
    twin.attach_cost(fresh, [p["start"]], [p["goal"]], W, L.LONGSAFE, 1e4)
    X = dev.get("X")
    dev.run(1)
    twin.run(1)
    n = 2 * W
    fit = dev.get("fit")
    want = fresh.evaluate(X.reshape(-1, n), p["start"], p["goal"], W, L.LONGSAFE, 1e4)["f"].reshape(fit.shape)
    on_old = old.evaluate(X.reshape(-1, n), p["start"], p["goal"], W, L.LONGSAFE, 1e4)["f"].reshape(fit.shape)
    assert bits_equal(fit, want)
    assert not np.array_equal(fit, on_old), "the edit does not reach the population"
    l = dev.launch()
    per_generation = 1 + l["overlap"] + 3 + l["rank_tile_sorted"] + (3 if l["upd_gram"] else 0)
    before = launches()
    dev.run(16)
    assert launches() - before == 16 * per_generation, l
    twin.run(16)
    for k in KEYS:
        assert np.array_equal(dev.get(k), twin.get(k)), (case, k)
    xb, fb = dev.best()
    xt, ft = twin.best()
    assert np.array_equal(xb, xt) and np.array_equal(fb, ft)
    for h in (dev, twin, old, cmap, fresh):
        h.close()


def test_rescore_best_takes_the_cost_on_the_updated_map(c2, monkeypatch):
    """After an edit onto the best path, best_f is the cost of best_x on the new map, bit for bit; best_x and counteval do
    not change."""
    p = c2
    cmap = L.CostMap.from_occupancy(p["occ"], CLAMP, "f32")
    dev = _handle(p, cmap, monkeypatch)
    dev.run(8)
    xb, fb = dev.best()
    ce = dev.get("counteval")
    cells = cmap.trace(xb[0], p["start"], p["goal"], W)
    cells = cells[cells >= 0]
    y, x = divmod(int(cells[len(cells) // 2]), SIZE)
    lo = (max(0, x - 4), max(0, y - 4))
    box = np.ones((9, 9), np.uint8)
    cmap.update_occupancy(lo, box)
    fresh = L.CostMap.from_occupancy(edited(p["occ"], lo, box), CLAMP, "f32")
    dev.rescore_best()
    xb2, fb2 = dev.best()
    want = fresh.evaluate(xb, p["start"], p["goal"], W, L.LONGSAFE, 1e4)
    assert bits_equal(fb2, want["f"])
    assert dev.get("best_f")[0] == np.float64(want["f"][0])
    assert want["ncoll"][0] > 0 and fb2[0] > fb[0]
    assert np.array_equal(xb2, xb) and np.array_equal(dev.get("counteval"), ce)
    for h in (dev, cmap, fresh):
        h.close()


def test_rescore_best_of_a_batch(monkeypatch):
    """Instances with queries of their own: each best_f becomes the cost of its best_x for its own end points; an
    instance with no evaluation (counteval 0) keeps its best_f.  One k_cost width for every launch, so that the handle's
    launch shape (picked from the first query) and evaluate's (picked per query) sum in the same order."""
    monkeypatch.setenv("LMCMA_B200_COST_TPT", "64")
    rng = np.random.default_rng(11)
    occ = (rng.random((160, 200)) < 0.01).astype(np.uint8)
    occ[:2, :] = occ[-2:, :] = 1
    cmap = L.CostMap.from_occupancy(occ, 12.0, "f32")
    dist = cmap.dequantized()
    Wb, B = 16, 5
    starts, goals = maps.random_queries(dist, B, seed=4, min_sep=80)
    x0 = np.stack([maps.straight_line(s, g, Wb) for s, g in zip(starts, goals)])
    lo, hi = maps.box_bounds((200, 160), Wb)
    dev = L.Optimizer(2 * Wb, x0=x0, lam=32, m=8, batch=B, lo=lo, hi=hi, sigma0=6.0, seed=5)
    dev.attach_cost(cmap, starts, goals, Wb)
    dev.run(10)
    xb, fb = dev.best()
    ce = dev.get("counteval")
    ce_zero = ce.copy()
    ce_zero[1] = 0
    dev.set("counteval", ce_zero)
    bf_before = dev.get("best_f")
    box = np.ones((60, 80), np.uint8)
    lo_box = (60, 50)
    cmap.update_occupancy(lo_box, box)
    fresh = L.CostMap.from_occupancy(edited(occ, lo_box, box), 12.0, "f32")
    dev.rescore_best()
    xb2, fb2 = dev.best()
    bf = dev.get("best_f")
    assert np.array_equal(xb2, xb)
    assert bf[1] == bf_before[1]
    changed = 0
    for b in (0, 2, 3, 4):
        want = fresh.evaluate(xb[b], starts[b], goals[b], Wb)["f"][0]
        assert bf[b] == np.float64(want) and bits_equal(fb2[b], want), b
        changed += int(bf[b] != bf_before[b])
    assert changed > 0, "the edit reaches no best path"
    for h in (dev, cmap, fresh):
        h.close()


def test_rescore_best_leaves_unevaluated_instances_and_refuses_without_a_map_or_with_a_split_population(c2, monkeypatch):
    p = c2
    lo, hi = p["bounds"]
    n = 2 * W
    bare = L.Optimizer(n, x0=p["x0"], lam=64, lo=lo, hi=hi, sigma0=16.0, seed=2)
    with pytest.raises(K.LmcmaError) as e:
        bare.rescore_best()
    assert e.value.code == K.ERR_STATE
    cmap = L.CostMap.from_occupancy(p["occ"], CLAMP, "f32")
    bare.attach_cost(cmap, [p["start"]], [p["goal"]], W, L.LONGSAFE, 1e4)
    before = bare.get("best_f")
    bare.rescore_best()                                  # nothing evaluated yet
    assert np.array_equal(bare.get("best_f"), before)
    split = L.Optimizer(n, x0=p["x0"], lam=64, lo=lo, hi=hi, sigma0=16.0, seed=2, pop_offset=0, pop_count=32)
    split.attach_cost(cmap, [p["start"]], [p["goal"]], W, L.LONGSAFE, 1e4)
    with pytest.raises(K.LmcmaError) as e:
        split.rescore_best()
    assert e.value.code == K.ERR_STATE
    for h in (bare, split, cmap):
        h.close()
