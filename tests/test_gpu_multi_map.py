"""One handle on several maps (attach_cost_maps): instance b is evaluated on maps[map_of[b]].  Every comparison is bitwise:
an instance of a multi-map handle against the same instance of a single-map twin attached to its map (same batch, seed
and end points; Philox keys on the instance index, so every instance can be compared), a switched instance's fitness
against CostMap.evaluate on its new map, instances on untouched maps against a run without the change.

The cost's launch shape is chosen from instance 0's end points (attach) or from the query's (CostMap.evaluate) and the
block reduction depends on the CTA width: it is pinned for every map and handle this module creates."""
from ctypes import byref, c_void_p

import numpy as np
import pytest

import lmcma_path_planner_b200 as L
from lmcma_path_planner_b200 import _capi as K
from lmcma_path_planner_b200 import maps
from test_gpu_launch_graphs import _tail_kernels, launches
from test_gpu_reset import PINNED_COST, STATE

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

W, M_PAIRS, SIGMA0 = 30, 20, 12.0
MAP_OF_STATE = STATE + ("ncoll", "nsamp")


@pytest.fixture(scope="module", autouse=True)
def pinned_cost_shape():
    with pytest.MonkeyPatch.context() as mp:
        for k, v in PINNED_COST.items():
            mp.setenv(k, v)
        yield


def _occ(shape, seed):
    return maps.random_boxes_occupancy(shape, 12 if len(shape) == 2 else 10, 6, 24 if len(shape) == 2 else 10, seed, border=1)


def _maps(kind, seed=0):
    """(CostMaps, the box shape x y [z] every handle uses: the largest extent per axis)"""
    if kind == "2d_f32":
        shapes = [(160, 192), (208, 150), (180, 180)]                            # [ny, nx]
        cm = [L.CostMap.from_occupancy(_occ(s, 10 + seed + i), 32.0, "f32", c_min=0.5) for i, s in enumerate(shapes)]
    elif kind == "2d_u8":
        shapes = [(160, 192), (208, 150)]
        cm = [L.CostMap.from_occupancy(_occ(shapes[0], 20 + seed), 32.0, "u8", u8_scale=0.25, c_min=0.5),
              L.CostMap.from_occupancy(_occ(shapes[1], 21 + seed), 40.0, "u8", u8_scale=0.5, c_min=1.0)]
    else:
        shapes = [(40, 48, 56), (48, 40, 50)]                                    # [nz, ny, nx]
        cm = [L.CostMap.from_occupancy(_occ(s, 30 + seed + i), 16.0, "u8", u8_scale=0.25, c_min=0.5) for i, s in enumerate(shapes)]
    box = tuple(int(v) for v in np.max([s[::-1] for s in shapes], axis=0))
    return cm, box


def _queries(dims, B, seed):
    """per-instance start / goal inside the smallest map of every kind (every axis >= 40 cells)"""
    rng = np.random.default_rng(seed)
    top = 36.0 if dims == 3 else 140.0
    starts = rng.uniform(3.0, top, (B, dims)).astype(np.float32)
    goals = rng.uniform(3.0, top, (B, dims)).astype(np.float32)
    return starts, goals


def _problem(kind, B, seed=0):
    cm, box = _maps(kind, seed)
    dims = len(box)
    starts, goals = _queries(dims, B, 100 + seed)
    x0 = np.stack([maps.straight_line(starts[b], goals[b], W) for b in range(B)])
    lo, hi = maps.box_bounds(box, W)
    return dict(cm=cm, dims=dims, starts=starts, goals=goals, x0=x0, lo=lo, hi=hi, B=B)


def _handle(p, cmaps, lam, seed, map_of=None, x0=None, starts=None, goals=None):
    o = L.Optimizer(p["dims"] * W, x0=p["x0"] if x0 is None else x0, lam=lam, m=M_PAIRS, batch=p["B"], lo=p["lo"], hi=p["hi"],
                    sigma0=SIGMA0, seed=seed)
    o.attach_cost(cmaps, p["starts"] if starts is None else starts, p["goals"] if goals is None else goals, W, L.LONGSAFE, 1e4,
                  map_of=map_of)
    return o


def _same_rows(a, b, rows, tag="", names=STATE):
    rows = np.atleast_1d(rows)
    for k in names:
        assert np.array_equal(a.get(k)[rows], b.get(k)[rows], equal_nan=True), (tag, k)
    xa, fa = a.best()
    xb, fb = b.best()
    assert np.array_equal(xa[rows], xb[rows]), (tag, "best_x")
    assert np.array_equal(fa[rows], fb[rows]), (tag, "best_f")


def _evaluate(cmap, X, start, goal):
    return cmap.evaluate(X, start, goal, W, L.LONGSAFE, 1e4)


TWIN_CASES = {
    "2d_f32": dict(kind="2d_f32", B=8, lam=64, map_of=[0, 1, 2, 2, 1, 0, 1, 2]),
    "2d_u8": dict(kind="2d_u8", B=8, lam=64, map_of=[1, 0, 0, 1, 1, 1, 0, 1]),
    "3d_u8": dict(kind="3d_u8", B=4, lam=64, map_of=[1, 0, 1, 0]),
    "2d_f32_lambda1024": dict(kind="2d_f32", B=2, lam=1024, map_of=[2, 0]),
}


@pytest.mark.parametrize("case", list(TWIN_CASES))
def test_each_instance_equals_its_single_map_twin(case):
    """After 1 and 60 fused generations, instance b of the multi-map handle equals instance b of a single-map handle of the
    same batch, seed and end points attached to map map_of[b]."""
    c = TWIN_CASES[case]
    p = _problem(c["kind"], c["B"])
    map_of = np.asarray(c["map_of"], np.int32)
    dev = _handle(p, p["cm"], c["lam"], 3, map_of=map_of)
    twins = [_handle(p, cm, c["lam"], 3) for cm in p["cm"]]
    assert np.array_equal(dev.get("map_of"), map_of)
    for gens in (1, 59):
        dev.run(gens)
        for t in twins:
            t.run(gens)
        for b in range(p["B"]):
            _same_rows(dev, twins[map_of[b]], b, (case, gens, b), MAP_OF_STATE)
    dev.close()
    for t in twins:
        t.close()


def test_switching_maps_from_the_host():
    """set("map_of") between runs: the next generation's fitness of every instance is CostMap.evaluate of its previous
    population on its new map, and run(1) after the switch replays the graphs it has (one generation's launches)."""
    p = _problem("2d_f32", 8)
    dev = _handle(p, p["cm"], 64, 5, map_of=np.zeros(8, np.int32))
    dev.run(6)
    X = dev.get("X")
    new = np.array([2, 1, 0, 1, 2, 2, 0, 1], np.int32)
    dev.set("map_of", new)
    assert np.array_equal(dev.get("map_of"), new)
    l = dev.launch()
    per_generation = 1 + l["overlap"] + _tail_kernels(l, False)
    before = launches()
    dev.run(1)
    assert launches() - before == per_generation, l
    fit = dev.get("fit")
    for b in range(8):
        ref = _evaluate(p["cm"][new[b]], X[b], p["starts"][b], p["goals"][b])
        assert np.array_equal(fit[b], ref["f"]), b
        assert np.array_equal(dev.get("ncoll")[b], ref["ncoll"]), b
    dev.close()


def test_switch_and_reset_inside_a_torch_graph():
    """device_map_index() written by torch inside a torch.cuda.graph capture next to reset_instances_dev: the reset
    instance, now on another map with new end points, equals a fresh twin attached to that map (epoch 1), right after the
    replay and 60 generations later; the instances whose map changed without a reset score their population on the new
    map."""
    p = _problem("2d_f32", 8)
    B, n, row = 8, 2 * W, 3
    map_of = np.array([0, 1, 2, 0, 1, 2, 0, 1], np.int32)
    new = map_of.copy()
    new[row], new[6] = 2, 1
    rng = np.random.default_rng(9)
    new_start, new_goal = rng.uniform(3.0, 140.0, 2).astype(np.float32), rng.uniform(3.0, 140.0, 2).astype(np.float32)
    new_x0 = maps.straight_line(new_start, new_goal, W)
    sigma_new = 6.0

    dev = _handle(p, p["cm"], 64, 7, map_of=map_of)
    dev.run(20)
    s = torch.cuda.Stream()
    dev.set_stream(s.cuda_stream)
    idx = dev.device_map_index()
    assert idx.dtype == torch.int32 and tuple(idx.shape) == (B,)
    assert np.array_equal(idx.cpu().numpy(), map_of)
    flags = torch.zeros(B, dtype=torch.int32, device="cuda")
    flags[row] = 1
    x0_t = torch.zeros((B, n), dtype=torch.float64, device="cuda")
    x0_t[row] = torch.from_numpy(new_x0)
    sig_t = torch.full((B,), sigma_new, dtype=torch.float64, device="cuda")
    ends_t = torch.zeros((B, 6), dtype=torch.float32, device="cuda")
    ends_t[row, :2] = torch.from_numpy(new_start)
    ends_t[row, 3:5] = torch.from_numpy(new_goal)
    new_t = torch.from_numpy(new).cuda()
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=s):
        idx.copy_(new_t)
        dev.reset_instances_dev(flags, x0_t, sig_t, ends_t)
    torch.cuda.synchronize()
    assert np.array_equal(dev.get("map_of"), map_of)            # capturing ran nothing
    X = dev.get("X")
    graph.replay()
    torch.cuda.synchronize()
    assert np.array_equal(dev.get("map_of"), new)

    x0 = p["x0"].copy()
    x0[row] = new_x0
    starts, goals = p["starts"].copy(), p["goals"].copy()
    starts[row], goals[row] = new_start, new_goal
    twin = _handle(p, p["cm"][2], 64, 7, x0=x0, starts=starts, goals=goals)
    sigma = twin.get("sigma")
    sigma[row] = sigma_new
    twin.set("sigma", sigma)
    twin.set("epoch", 1)
    twin.resample()
    _same_rows(dev, twin, row, "after the reset")

    dev.run(1)
    fit = dev.get("fit")
    ref = _evaluate(p["cm"][1], X[6], p["starts"][6], p["goals"][6])
    assert np.array_equal(fit[6], ref["f"])                      # switched without a reset
    twin.run(1)
    dev.run(59)
    twin.run(59)
    _same_rows(dev, twin, row, "60 generations later")
    del graph
    dev.close()
    twin.close()


def test_an_occupancy_update_reaches_the_instances_on_that_map():
    """update_occupancy on one map: its instances score their population on the new map; instances on the other maps
    stay bit-equal to a handle on untouched copies of the maps; rescore_best gives every instance the cost of its best_x
    on its own map."""
    map_of = np.array([0, 1, 2, 1, 0, 1, 2, 1], np.int32)
    p = _problem("2d_f32", 8)
    q = _problem("2d_f32", 8)                                    # the same maps, built again: never updated
    dev = _handle(p, p["cm"], 64, 11, map_of=map_of)
    ref = _handle(q, q["cm"], 64, 11, map_of=map_of)
    dev.run(25)
    ref.run(25)
    X = dev.get("X")
    box = np.ones((30, 40), np.uint8)
    lo = (70, 60)
    p["cm"][1].update_occupancy(lo, box)
    dev.run(1)
    ref.run(1)
    fit = dev.get("fit")
    on1 = np.nonzero(map_of == 1)[0]
    others = np.nonzero(map_of != 1)[0]
    for b in on1:
        want = _evaluate(p["cm"][1], X[b], p["starts"][b], p["goals"][b])
        assert np.array_equal(fit[b], want["f"]), b
    assert not np.array_equal(fit[on1], ref.get("fit")[on1])    # the box crosses their straight lines' region
    dev.run(30)
    ref.run(30)
    _same_rows(dev, ref, others, "other maps", MAP_OF_STATE)

    dev.rescore_best()
    bx, bf = dev.best()
    for b in range(8):
        want = _evaluate(p["cm"][map_of[b]], bx[b], p["starts"][b], p["goals"][b])["f"][0]
        assert np.float32(dev.get("best_f")[b]) == want, b
        assert bf[b] == want, b
    dev.close()
    ref.close()


def test_an_index_outside_the_table_gives_inf():
    """A map_of entry set to map_count through the device view: that instance's trajectories get f = +inf and
    ncoll = nsamp = 0; every other instance computes what a handle without the bad entry computes."""
    p = _problem("2d_u8", 8)
    map_of = np.array([0, 1, 0, 1, 0, 1, 0, 1], np.int32)
    dev = _handle(p, p["cm"], 64, 13, map_of=map_of)
    ref = _handle(p, p["cm"], 64, 13, map_of=map_of)
    dev.run(10)
    ref.run(10)
    idx = dev.device_map_index()
    idx[2] = len(p["cm"])
    torch.cuda.synchronize()
    dev.run(1)
    ref.run(1)
    assert np.all(np.isposinf(dev.get("fit")[2]))
    assert np.all(dev.get("ncoll")[2] == 0) and np.all(dev.get("nsamp")[2] == 0)
    rows = [b for b in range(8) if b != 2]
    _same_rows(dev, ref, rows, "other instances", MAP_OF_STATE)
    dev.close()
    ref.close()


def _snapshot(h):
    out = {k: h.get(k) for k in STATE + ("fit_sorted", "prev_fit", "arindex", "rank", "ncoll", "nsamp", "map_of")}
    out["best() x"], out["best() f"] = h.best()
    return out


def _attach_raw(h, count, hs, map_of, waypoints=W, obj=True, ends=True):
    lib = K.lib()
    o = L.optimizer._objective(waypoints, L.LONGSAFE, 1e4)
    e = (K.Endpoints * h.batch)()
    arr = None if hs is None else (c_void_p * len(hs))(*hs)
    mo = None if map_of is None else K.iptr(np.ascontiguousarray(map_of, np.int32))
    return lib.lmcma_b200_attach_cost_maps(h._h, count, arr, mo, byref(o) if obj else None, e if ends else None)


def test_refusals_change_nothing():
    """Every ERR_ARG / ERR_STATE case of attach_cost_maps, set("map_of") and instance_maps_dev is refused and leaves the
    state, map_of and the attachment as they were: the handle then runs on as a twin that saw no refusal."""
    p = _problem("2d_f32", 8)
    map_of = np.array([0, 1, 2, 0, 1, 2, 0, 1], np.int32)
    dev = _handle(p, p["cm"], 64, 17, map_of=map_of)
    twin = _handle(p, p["cm"], 64, 17, map_of=map_of)
    dev.run(3)
    twin.run(3)
    before = _snapshot(dev)
    hs = [m._h.value for m in p["cm"]]
    q3, _ = _maps("3d_u8")
    u8, _ = _maps("2d_u8")
    arg_cases = {
        "null maps": (3, None, map_of, {}),
        "null map_of": (3, hs, None, {}),
        "null objective": (3, hs, map_of, dict(obj=False)),
        "null ends": (3, hs, map_of, dict(ends=False)),
        "map_count 0": (0, hs, map_of, {}),
        "map_count negative": (-1, hs, map_of, {}),
        "null map entry": (3, [hs[0], None, hs[2]], map_of, {}),
        "dims differ": (2, [hs[0], q3[0]._h.value], np.zeros(8, np.int32), {}),
        "storage differs": (2, [hs[0], u8[0]._h.value], np.zeros(8, np.int32), {}),
        "dims * waypoints != n": (3, hs, map_of, dict(waypoints=W + 1)),
        "map_of == map_count": (3, hs, np.where(np.arange(8) == 4, 3, map_of), {}),
        "map_of negative": (3, hs, np.where(np.arange(8) == 4, -1, map_of), {}),
        "map_of past a shorter list": (2, hs[:2], map_of, {}),
    }
    for name, (count, h_list, mo, kw) in arg_cases.items():
        assert _attach_raw(dev, count, h_list, mo, **kw) == K.ERR_ARG, name
    for bad in (np.where(np.arange(8) == 1, 3, map_of), np.where(np.arange(8) == 1, -1, map_of)):
        with pytest.raises(K.LmcmaError) as e:
            dev.set("map_of", bad)
        assert e.value.code == K.ERR_ARG
    lib = K.lib()
    assert lib.lmcma_b200_set_i32(dev._h, K.I32["map_of"], K.iptr(map_of), 7) == K.ERR_ARG
    assert lib.lmcma_b200_instance_maps_dev(dev._h, None) == K.ERR_ARG
    after = _snapshot(dev)
    for k, v in before.items():
        assert np.array_equal(after[k], v, equal_nan=True), k
    dev.run(5)
    twin.run(5)
    _same_rows(dev, twin, np.arange(8), "after the refusals", MAP_OF_STATE)
    for m in q3 + u8:
        m.close()
    dev.close()
    twin.close()

    split = L.Optimizer(2 * W, x0=p["x0"][0], lam=64, lo=p["lo"], hi=p["hi"], pop_offset=0, pop_count=32, seed=2)
    assert _attach_raw(split, 3, hs, np.zeros(1, np.int32)) == K.ERR_STATE
    assert _attach_raw(split, 1, hs[:1], np.zeros(1, np.int32)) == K.ERR_STATE
    split.close()
    single = _handle(p, p["cm"][0], 64, 19)
    ptr = c_void_p()
    assert lib.lmcma_b200_instance_maps_dev(single._h, byref(ptr)) == K.ERR_STATE
    assert np.array_equal(single.get("map_of"), np.zeros(8, np.int32))
    with pytest.raises(K.LmcmaError) as e:
        single.set("map_of", np.ones(8, np.int32))
    assert e.value.code == K.ERR_ARG
    single.close()


def test_one_map_through_attach_cost_maps_is_attach_cost():
    """attach_cost_maps with map_count == 1 equals attach_cost bit for bit over 60 generations and launches the same
    kernels; the handle is a single-map one (map_of all zeros, no device view)."""
    p = _problem("2d_f32", 8)
    a = _handle(p, p["cm"][1], 64, 23)
    b = _handle(p, [p["cm"][1]], 64, 23, map_of=np.zeros(8, np.int32))
    a.run(1)
    b.run(1)
    c0 = launches()
    a.run(59)
    c1 = launches()
    b.run(59)
    assert launches() - c1 == c1 - c0
    _same_rows(a, b, np.arange(8), "one map", MAP_OF_STATE + ("map_of",))
    with pytest.raises(K.LmcmaError) as e:
        b.device_map_index()
    assert e.value.code == K.ERR_STATE
    a.close()
    b.close()
