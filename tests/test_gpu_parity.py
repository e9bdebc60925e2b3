"""GPU parity tests proper: the CUDA path (through the C ABI) against the CPU oracle on the same seeded
inputs.  Bars: integer / index work bit-exact; costs 1e-5 relative; optimiser state after a
teacher-forced generation 1e-5 relative (FP32 device vs FP64 oracle); sigma 1e-12."""
import numpy as np
import pytest

import lmcma_path_planner_b200 as L
from lmcma_path_planner_b200 import maps
from conftest import weighted_sphere

pytestmark = pytest.mark.gpu

COST_RTOL = 1e-5


def rel_err(a, b, floor=1e-30):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), floor))) if a.size else 0.0


# ------------------------------------------------------------------------------------------------
# cost kernel
# ------------------------------------------------------------------------------------------------
def _candidates(rng, x0, count, sigma, lo, hi):
    X = x0[None, :] + sigma * rng.standard_normal((count, len(x0)))
    return np.clip(X, lo, hi).astype(np.float32)


@pytest.mark.parametrize("name", ["problem1", "problem2", "two_bars"])
@pytest.mark.parametrize("weights", [L.LONGSAFE, L.SHORTRISKY])
def test_cost_2d_bundled_maps(po, golden_maps, name, weights):
    """C1 shape: the reference's 100x100 maps, query (99,0)->(0,99) (planner.cpp:701-706), 20 waypoints."""
    dist = po.edt_exact(golden_maps[name])
    W, start, goal = 20, (99.0, 0.0), (0.0, 99.0)
    rng = np.random.default_rng(3)
    lo, hi = maps.box_bounds((100, 100), W)
    X = _candidates(rng, maps.straight_line(start, goal, W), 257, 6.0, lo, hi)
    ref = po.CostProblem(dist, start, goal, W, *weights, w_col=1e4).evaluate(X)
    cm = L.CostMap(dist, "f32")
    got = cm.evaluate(X, start, goal, W, weights, 1e4)
    assert np.array_equal(got["ncoll"], ref["ncoll"])          # collision flags: bit-exact
    assert np.array_equal(got["nsamp"], ref["nsamp"])
    assert rel_err(got["f"], ref["f"]) < COST_RTOL
    assert ref["ncoll"].max() > 0                              # the population does hit obstacles


def test_cost_cell_indices_bit_exact(po, golden_maps):
    dist = po.edt_exact(golden_maps["problem1"])
    W, start, goal = 20, (99.0, 0.0), (0.0, 99.0)
    rng = np.random.default_rng(11)
    lo, hi = maps.box_bounds((100, 100), W)
    cm = L.CostMap(dist, "f32")
    prob = po.CostProblem(dist, start, goal, W)
    x0 = maps.straight_line(start, goal, W)
    for i in range(8):
        x = _candidates(rng, x0, 1, 8.0, lo - 3, hi + 3)[0]   # some samples leave the map
        if i == 0:
            x = (np.round(x * 2) / 2).astype(np.float32)      # half-integer coordinates: rint ties
        assert np.array_equal(cm.trace(x, start, goal, W), prob.trace(x))


def test_cost_edge_cases(po, golden_maps):
    dist = po.edt_exact(golden_maps["two_bars"])
    W, start, goal = 5, (99.0, 0.0), (0.0, 99.0)
    x0 = maps.straight_line(start, goal, W).astype(np.float32)
    X = np.stack([x0, x0, x0, x0, x0])
    X[1, 2] = np.nan                     # NaN waypoint
    X[2, :] = 50.0                       # degenerate: all waypoints coincide (zero-length segments)
    X[3, 0] = -40.0; X[3, 7] = 400.0     # far outside the map
    X[4, :] = 0.25                       # sub-cell segments
    ref = po.CostProblem(dist, start, goal, W).evaluate(X)
    got = L.CostMap(dist, "f32").evaluate(X, start, goal, W)
    assert np.array_equal(got["ncoll"], ref["ncoll"])
    assert np.array_equal(got["nsamp"], ref["nsamp"])
    assert np.isnan(got["f"][1]) and np.isnan(ref["f"][1])
    ok = [0, 2, 3, 4]
    assert rel_err(got["f"][ok], ref["f"][ok]) < COST_RTOL
    # empty batch
    e = L.CostMap(dist, "f32").evaluate(np.zeros((0, 2 * W), np.float32), start, goal, W)
    assert e["f"].shape == (0,)


def test_cost_u8_storage_matches_oracle_on_dequantized_map(po):
    dist, start, goal = maps.config2_map(size=512, n_rects=64, seed=5, clamp=60.0)
    W = 60
    cm = L.CostMap(dist, "u8", u8_scale=0.25)
    dq = cm.dequantized()
    assert np.array_equal(dq == 0, dist == 0)            # obstacles preserved exactly
    assert np.all(dq <= dist + 1e-6) and np.all((dist - dq)[dist < 63] < 0.25 + 1e-6)
    rng = np.random.default_rng(2)
    lo, hi = maps.box_bounds((512, 512), W)
    X = _candidates(rng, maps.straight_line(start, goal, W), 300, 12.0, lo, hi)
    ref = po.CostProblem(dq, start, goal, W).evaluate(X)
    got = cm.evaluate(X, start, goal, W)
    assert np.array_equal(got["ncoll"], ref["ncoll"])
    assert rel_err(got["f"], ref["f"]) < COST_RTOL


def test_cost_3d(po):
    dist, start, goal = maps.config4_map(size=64, n_boxes=4096, seed=9, clamp=16.0)
    W = 40
    rng = np.random.default_rng(4)
    lo, hi = maps.box_bounds((64, 64, 64), W)
    X = _candidates(rng, maps.straight_line(start, goal, W), 200, 3.0, lo, hi)
    for storage, d in (("f32", dist), ("u8", None)):
        cm = L.CostMap(dist, storage, u8_scale=0.125)
        dd = dist if d is not None else cm.dequantized()
        prob = po.CostProblem(dd, start, goal, W)
        ref = prob.evaluate(X)
        got = cm.evaluate(X, start, goal, W)
        assert np.array_equal(got["ncoll"], ref["ncoll"])
        assert np.array_equal(got["nsamp"], ref["nsamp"])
        assert rel_err(got["f"], ref["f"]) < COST_RTOL
        assert np.array_equal(cm.trace(X[0], start, goal, W), prob.trace(X[0]))


def test_cost_full_size_properties(po):
    """C2 size (4096^2, n = 400, lambda = 1024): a seeded sample is checked against the oracle, the whole
    population through size-independent properties (reversal symmetry, sample count, monotone penalty)."""
    dist, start, goal = maps.config2_map()
    W = 200
    rng = np.random.default_rng(42)
    lo, hi = maps.box_bounds((4096, 4096), W)
    X = _candidates(rng, maps.straight_line(start, goal, W), 1024, 32.0, lo, hi)
    cm = L.CostMap(dist, "f32")
    got = cm.evaluate(X, start, goal, W)
    idx = rng.choice(1024, 48, replace=False)
    ref = po.CostProblem(dist, start, goal, W, threads=8).evaluate(X[idx])
    assert np.array_equal(got["ncoll"][idx], ref["ncoll"])
    assert np.array_equal(got["nsamp"][idx], ref["nsamp"])
    assert rel_err(got["f"][idx], ref["f"]) < COST_RTOL
    # the same poly-line walked goal->start has the same length / sample count (cells may differ by rounding)
    Xr = X.reshape(1024, 2, W)[:, :, ::-1].reshape(1024, -1).copy()
    rev = cm.evaluate(Xr, goal, start, W)
    assert np.array_equal(rev["nsamp"], got["nsamp"])
    # raising the collision weight can only raise the cost, and by exactly w_col * ncoll
    hi_pen = cm.evaluate(X, start, goal, W, L.LONGSAFE, 2e4)
    assert np.all(hi_pen["f"] >= got["f"] - 1e-3)
    assert rel_err(hi_pen["f"] - got["f"], 1e4 * got["ncoll"], floor=1.0) < 1e-3


# ------------------------------------------------------------------------------------------------
# optimiser: teacher-forced generations against the FP64 oracle (SURVEY 7.2 #3)
# ------------------------------------------------------------------------------------------------
def _teacher_forced(po, n, lam, m, gens, seed, lo=None, hi=None, sigma=1.0, fobj=weighted_sphere, x0=None,
                    tol=2e-5, tol_v=None, warm=None):
    """`gens` teacher-forced generations.  warm: an oracle state of the same (n, m) (OracleLMCMA.state(), e.g. from a cheap
    small-population run) to start from instead of the empty state, so that a few generations have every slot live and
    being recycled; the previous fitness is then the sorted fitness of the first population."""
    rng = np.random.default_rng(seed)
    x0 = np.full(n, 0.5) if x0 is None else x0
    dev = L.Optimizer(n, x0=x0, lam=lam, m=m, lo=lo, hi=hi, sigma0=sigma, rng="inject")
    lam = dev.lam
    zs = rng.standard_normal((gens + 1, lam, n)).astype(np.float32)
    ora = po.OracleLMCMA(n, x0=x0, lam=lam, m=m, lo=lo, hi=hi, sigma=sigma, seed=1, Z0=zs[0].astype(np.float64))
    dev.inject_z(zs[0])
    if warm is not None:
        ora.load_state(warm, np.zeros(lam), zs[0].astype(np.float64))
        prev = np.sort(fobj(ora.array("X")).astype(np.float32))
        ora.load_state(warm, prev.astype(np.float64), zs[0].astype(np.float64))
        dev.load_state(dict(warm, prev_fit=prev))
        dev.resample()
    worst = {}
    for g in range(gens):
        Xo = ora.array("X")
        Xd = dev.ask_all()[0]
        xs = max(1e-3, float(np.abs(Xo).max()))               # waypoint-coordinate scale
        worst["X"] = max(worst.get("X", 0), float(np.abs(Xd - Xo).max()) / xs)
        f = fobj(Xo).astype(np.float32)            # both sides are told the same FP32 fitness
        ora.tell_all(f.astype(np.float64), zs[g + 1].astype(np.float64))
        dev.inject_z(zs[g + 1])
        dev.tell_all(f)
        so = ora.state()
        # integer state: bit-exact
        assert np.array_equal(dev.get("t")[0][:so["live"]], so["t"][:so["live"]]), g
        live_slots = so["t"][:so["live"]]
        assert np.array_equal(dev.get("vec")[0][live_slots], so["vec"][live_slots]), g
        assert int(dev.get("itr")[0]) == so["itr"] and int(dev.get("live")[0]) == so["live"]
        assert np.array_equal(dev.get("arindex")[0], ora.int_array("arindex")), g
        assert int(dev.get("counteval")[0]) == so["counteval"]
        # floating state
        scale = max(1e-3, float(np.abs(so["xmean"]).max()))
        worst["xmean"] = max(worst.get("xmean", 0), float(np.abs(dev.get("xmean")[0] - so["xmean"]).max()) / scale)
        worst["sigma"] = max(worst.get("sigma", 0), abs(dev.get("sigma")[0] - so["sigma"]) / so["sigma"])
        pcs = max(1e-6, float(np.abs(so["pc"]).max()))
        worst["pc"] = max(worst.get("pc", 0), float(np.abs(dev.get("pc")[0] - so["pc"]).max()) / pcs)
        Vd, Pd = dev.get("V")[0], dev.get("P")[0]
        for slot in live_slots:
            vs = max(1e-6, float(np.abs(so["V"][slot]).max()))
            worst["V"] = max(worst.get("V", 0), float(np.abs(Vd[slot] - so["V"][slot]).max()) / vs)
            worst["P"] = max(worst.get("P", 0), float(np.abs(Pd[slot] - so["P"][slot]).max()) / vs)
        worst["Nj"] = max(worst.get("Nj", 0), rel_err(dev.get("Nj")[0][live_slots], so["Nj"][live_slots]))
        worst["Lj"] = max(worst.get("Lj", 0), rel_err(dev.get("Lj")[0][live_slots], so["Lj"][live_slots]))
        assert abs(dev.get("best_f")[0] - so["best_f"]) <= 1e-6 * max(1.0, abs(so["best_f"]))
        # teacher forcing: the device continues from the oracle's exact state
        dev.load_state(so)
        dev.resample()            # X of the next generation comes from the oracle's exact state + the same z
    assert worst["sigma"] < 1e-12, worst
    for k in ("X", "xmean", "pc", "V", "P"):
        assert worst[k] < (tol_v if (k == "V" and tol_v) else tol), (k, worst)
    assert worst["Nj"] < 1e-4 and worst["Lj"] < 1e-4, worst
    return worst


def test_lmcma_teacher_forced_small(po):
    """n = 10, lambda = m = 6 (the golden trace's shape): covers the slot-recycling logic (itr >= m)."""
    _teacher_forced(po, 10, 6, 0, 30, seed=1)


def test_lmcma_teacher_forced_default_lambda(po):
    """C1 shape: n = 40, default lambda = 15, m = lambda."""
    _teacher_forced(po, 40, 0, 0, 40, seed=2)


def test_lmcma_teacher_forced_bounds(po):
    _teacher_forced(po, 10, 8, 0, 20, seed=5, lo=np.full(10, 0.2), hi=np.full(10, 1.0))


def test_lmcma_teacher_forced_m_not_lambda(po):
    """C2-like shape scaled down: n = 400, lambda = 128, m = 2*sqrt(n) = 40."""
    _teacher_forced(po, 400, 128, 40, 50, seed=3, sigma=0.5)


def test_lmcma_teacher_forced_five_rows_per_warp(po):
    """48 < m <= 80 with rows that fit shared memory: the register sweep with five pending rows per warp (k_update<4, 5>) and
    the newest row's four-warp chain over eight blocks of factors, past the point where slots are recycled."""
    _teacher_forced(po, 100, 64, 60, 70, seed=6, sigma=0.5)


def test_lmcma_teacher_forced_eight_warp_update(po, monkeypatch):
    """k_update as a CTA of 8 warps with five rows per warp (two CTAs per SM: what large batches of instances take) on the
    C2 / C3 per-instance shape n = 400, m = 40, against the FP64 oracle past the point where slots are recycled."""
    monkeypatch.setenv("LMCMA_B200_UPDATE_WARPS", "8")
    _teacher_forced(po, 400, 128, 40, 50, seed=3, sigma=0.5)


def test_lmcma_teacher_forced_large_n(po):
    """C4-like row length: n = 1500, m = 77 (narrow sampler k_sample<12>; the 77 rows of 1500 fit neither registers nor
    shared memory, so the update is the Gram-matrix recompute with k_coef<10>).  The streaming update that keeps the rows
    in global memory is tested in tests/test_gpu_dispatch_variants.py."""
    _teacher_forced(po, 1500, 32, 77, 6, seed=4, sigma=0.3)


def test_rank_ties_and_nan(po, golden):
    """Ties keep the lower id (stable), -0 == +0 (golden vector from the reference's myqsort); NaN ranks last."""
    ties = np.array(golden["qsort_ties"]["in"], np.float32)
    lam = len(ties)
    dev = L.Optimizer(4, x0=np.zeros(4), lam=lam, rng="inject")
    dev.inject_z(np.zeros((lam, 4), np.float32))
    dev.inject_z(np.zeros((lam, 4), np.float32))
    dev.tell_all(ties)
    assert dev.get("arindex")[0].tolist() == golden["qsort_ties"]["ids"]
    assert np.array_equal(dev.get("fit_sorted")[0], np.array(golden["qsort_ties"]["sorted"], np.float32))
    f = ties.copy(); f[3] = np.nan
    dev.inject_z(np.zeros((lam, 4), np.float32))
    dev.tell_all(f)
    assert dev.get("arindex")[0][-1] == 3


def test_free_running_matches_oracle_short_window(po):
    """Free-running (no teacher forcing) for a few generations on a well-conditioned problem: the FP32
    device trajectory stays within 1e-4 of the FP64 oracle fed the device's own recorded deviates."""
    n, lam = 40, 16
    dev = L.Optimizer(n, x0=np.full(n, 0.5), lam=lam, sigma0=0.3, seed=7, rng="philox", record_z=True)
    z0 = dev.get("Z")[0].astype(np.float64)
    ora = po.OracleLMCMA(n, x0=np.full(n, 0.5), lam=lam, sigma=0.3, seed=1, Z0=z0)
    for g in range(6):
        Xd = dev.ask_all()[0]
        assert rel_err(Xd, ora.array("X"), floor=1e-2) < 1e-4, g
        f = weighted_sphere(Xd).astype(np.float32)
        dev.tell_all(f)
        ora.tell_all(f.astype(np.float64), dev.get("Z")[0].astype(np.float64))
    assert abs(dev.get("sigma")[0] - ora.doubles()["sigma"]) / ora.doubles()["sigma"] < 1e-9


def test_reference_class_protocol_hansen_stream(po, golden):
    """The reference-shaped class with inseed = 1 draws the reference's own deviates: the first candidate
    is x0 + sigma * z with the golden normals (lmcma.cpp:296, 435) and a short run tracks the golden sigmas."""
    g = golden["run_n10"]
    opt = L.LMCMA(np.array(g["x0"]), lambda_=g["lambda"], sigma=g["sigma0"], inseed=1)
    opt.init(10)
    x = opt.getNextParameterVector()
    want = np.array(g["x0"]) + g["sigma0"] * np.array(golden["rng"]["1"]["gauss"][:10])
    assert np.allclose(x, want, rtol=1e-6, atol=1e-6)
    x2 = opt.getNextParameterVector()          # does not advance (lmcma.cpp:172-182)
    assert np.array_equal(x, x2)
    sig = [g["sigma0"]]
    for gen in range(6):
        for i in range(g["lambda"]):
            xi = opt.getNextParameterVector()
            assert np.allclose(xi, np.array(g["gens"][gen]["X"][i]), rtol=2e-4, atol=2e-4), (gen, i)
            opt.setEvaluationFeedback([float(weighted_sphere(xi)[0])], 1)
        sig.append(float(opt._opt.get("sigma")[0]))
    assert opt.counteval == 6 * g["lambda"]
    assert not opt.isBehaviorLearningDone()
    assert np.allclose(sig, g["sigma"][:7], rtol=1e-3)


# ------------------------------------------------------------------------------------------------
# fused on-device planning
# ------------------------------------------------------------------------------------------------
def test_fused_generation_equals_ask_evaluate_tell(po, golden_maps):
    """One graph-replayed generation == ask_all -> cost_evaluate -> tell_all through host buffers."""
    dist = po.edt_exact(golden_maps["problem1"])
    W, start, goal = 20, (99.0, 0.0), (0.0, 99.0)
    lo, hi = maps.box_bounds((100, 100), W)
    x0 = maps.straight_line(start, goal, W)
    cm = L.CostMap(dist, "f32")
    a = L.Optimizer(2 * W, x0=x0, lo=lo, hi=hi, sigma0=5.0, seed=3, rng="philox")
    b = L.Optimizer(2 * W, x0=x0, lo=lo, hi=hi, sigma0=5.0, seed=3, rng="philox")
    a.attach_cost(cm, [start], [goal], W)
    for g in range(25):
        a.run(1)
        X = b.ask_all()[0]
        r = cm.evaluate(X, start, goal, W)
        b.tell_all(r["f"])
        assert np.array_equal(a.get("fit")[0], r["f"])
        assert np.array_equal(a.get("ncoll")[0], r["ncoll"])
    assert np.array_equal(a.get("xmean"), b.get("xmean"))
    assert np.array_equal(a.get("sigma"), b.get("sigma"))
    assert np.array_equal(a.ask_all(), b.ask_all())
    xa, fa = a.best(); xb, fb = b.best()
    assert np.array_equal(xa, xb) and fa == fb


def test_planning_c1_improves_and_best_cost_matches_oracle(po, golden_maps):
    """C1: 100x100 bundled maps, 20 waypoints: the fused planner lowers the cost, its reported best cost is the
    oracle's cost of its reported best path, and on problem1 that path is collision-free."""
    W, start, goal = 20, (99.0, 0.0), (0.0, 99.0)
    lo, hi = maps.box_bounds((100, 100), W)
    for name in ("problem1", "two_bars"):
        dist = po.edt_exact(golden_maps[name])
        cm = L.CostMap(dist, "f32")
        x0 = maps.straight_line(start, goal, W)
        opt = L.Optimizer(2 * W, x0=x0, lam=64, lo=lo, hi=hi, sigma0=8.0, seed=5)
        opt.attach_cost(cm, [start], [goal], W, L.LONGSAFE, 1e4)
        f0 = po.CostProblem(dist, start, goal, W).evaluate(x0.astype(np.float32))
        opt.run(400)
        xb, fb = opt.best()
        ref = po.CostProblem(dist, start, goal, W).evaluate(xb[0])
        assert rel_err(fb[0], ref["f"][0]) < COST_RTOL
        assert fb[0] < f0["f"][0]
        assert ref["ncoll"][0] <= f0["ncoll"][0]
        if name == "problem1":
            assert ref["ncoll"][0] == 0


@pytest.mark.parametrize("update_warps", ["0", "8"])
def test_batched_instances_are_independent(po, golden_maps, monkeypatch, update_warps):
    """C3 mechanics: B instances in one launch == the same instances run one at a time.  update_warps = 8: the batch's k_update
    as CTAs of 8 warps, two per SM (what large batches take by themselves) against single instances on 16 warps."""
    monkeypatch.setenv("LMCMA_B200_COST_TPT", "64")   # same reduction tree whatever the query length
    monkeypatch.setenv("LMCMA_B200_UPDATE_WARPS", update_warps)
    dist = po.edt_exact(golden_maps["problem2"])
    W = 12
    lo, hi = maps.box_bounds((100, 100), W)
    cm = L.CostMap(dist, "f32")
    starts, goals = maps.random_queries(dist, 5, seed=7, min_sep=40)
    x0 = np.stack([maps.straight_line(s, g, W) for s, g in zip(starts, goals)])
    batched = L.Optimizer(2 * W, x0=x0, lam=16, m=8, batch=5, lo=lo, hi=hi, sigma0=4.0, seed=11, record_z=True)
    batched.attach_cost(cm, starts, goals, W)
    z0 = batched.get("Z")
    batched.run(12)
    for b in (0, 3, 4):
        monkeypatch.setenv("LMCMA_B200_UPDATE_WARPS", "16")
        one = L.Optimizer(2 * W, x0=x0[b], lam=16, m=8, lo=lo, hi=hi, sigma0=4.0, rng="inject")
        one.attach_cost(cm, [starts[b]], [goals[b]], W)
        monkeypatch.setenv("LMCMA_B200_UPDATE_WARPS", update_warps)
        # replay instance b's deviates: regenerate them with a batch whose instance index matches
        ref = L.Optimizer(2 * W, x0=x0, lam=16, m=8, batch=5, lo=lo, hi=hi, sigma0=4.0, seed=11, record_z=True)
        ref.attach_cost(cm, starts, goals, W)
        one.inject_z(ref.get("Z")[b])
        for g in range(12):
            ref.run(1)
            one.inject_z(ref.get("Z")[b])
            one.run(1)
        assert np.array_equal(one.get("xmean")[0], batched.get("xmean")[b])
        assert one.get("sigma")[0] == batched.get("sigma")[b]


def test_split_population_single_process(po, golden_maps):
    """C4 mechanics on one GPU: two handles owning lambda/2 rows each, 'all-gather' done by hand, must
    reproduce the unsplit optimiser bit for bit (same Philox rows, same deterministic reductions)."""
    import torch
    dist = po.edt_exact(golden_maps["problem1"])
    W, start, goal = 20, (99.0, 0.0), (0.0, 99.0)
    lo, hi = maps.box_bounds((100, 100), W)
    x0 = maps.straight_line(start, goal, W)
    cm = L.CostMap(dist, "f32")
    lam, G = 64, 2
    whole = L.Optimizer(2 * W, x0=x0, lam=lam, m=12, lo=lo, hi=hi, sigma0=5.0, seed=9)
    whole.attach_cost(cm, [start], [goal], W)
    parts = []
    for r in range(G):
        p = L.Optimizer(2 * W, x0=x0, lam=lam, m=12, lo=lo, hi=hi, sigma0=5.0, seed=9, pop_offset=r * lam // G,
                        pop_count=lam // G)
        p.attach_cost(cm, [start], [goal], W)
        parts.append(p)
    pf = parts[0].mg_payload_floats()
    f_all = torch.zeros(lam, dtype=torch.float32, device="cuda")
    pay_all = torch.zeros(G * pf, dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    for g in range(8):
        whole.run(1)
        for r, p in enumerate(parts):
            p.mg_evaluate(f_all.data_ptr() + 4 * r * (lam // G))
            p.sync()
        for r, p in enumerate(parts):
            p.mg_rank(f_all.data_ptr(), pay_all.data_ptr() + 4 * r * pf)
            p.sync()
        for p in parts:
            p.mg_update(pay_all.data_ptr(), G)
            p.sync()
        if g == 0:   # identical Philox rows -> identical first population and fitness
            assert np.array_equal(f_all.cpu().numpy(), whole.get("fit")[0])
        # the split sums its partials in a different (fixed) association, so FP32 rounding differs slightly
        assert np.allclose(f_all.cpu().numpy(), whole.get("fit")[0], rtol=1e-3)
        for p in parts:
            assert np.allclose(p.get("xmean"), whole.get("xmean"), rtol=1e-5, atol=1e-2)
            assert abs(p.get("sigma")[0] - whole.get("sigma")[0]) <= 1e-9 * whole.get("sigma")[0]
        assert np.array_equal(parts[0].get("xmean"), parts[1].get("xmean"))   # replicas stay bit-identical
        assert parts[0].get("sigma")[0] == parts[1].get("sigma")[0]
    X = np.concatenate([p.ask_all()[0] for p in parts])
    assert np.allclose(X, whole.ask_all()[0], rtol=1e-4, atol=1e-2)


# ------------------------------------------------------------------------------------------------
# the C++ host side (the reference's language): facade header + demo / planner driver
# ------------------------------------------------------------------------------------------------
def _example(args, cwd):
    import os
    import subprocess
    exe = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "examples", "example_lmcma")
    return subprocess.run([exe] + args, cwd=cwd, capture_output=True, text=True, timeout=300)


def test_cpp_facade_demo_converges_like_the_reference(tmp_path):
    """example_lmcma.cpp:28-76 against lmcma_b200::LMCMA: 1000 evaluations of the two-Gaussian function with
    bounds [-2,15]^2 from (0,0); the reference converges to (3.99966, 3.99966), f = -4.00067 (SURVEY.md 8c)."""
    r = _example(["demo", "1"], tmp_path)
    assert r.returncode == 0, r.stderr
    tail = r.stdout.strip().split("is:")[1].split()
    x, y = (float(v) for v in tail[0].split(","))
    best = float(tail[2].split("=")[1])
    assert abs(x - 3.99966) < 2e-2 and abs(y - 3.99966) < 2e-2
    assert abs(best + 4.00067) < 1e-3
    assert "counteval=1000" in r.stdout
    rows = open(tmp_path / "path_to_min.csv").read().strip().splitlines()
    assert rows[0] == "x,y,z," and len(rows) == 1001


def test_cpp_planner_driver_improves_on_the_straight_line(tmp_path):
    """plan() mirrors optimal_palnning_without_setting_path (planner.cpp:694-775) on the two-bar map: the returned
    path is the one that achieved the returned cost (re-evaluated through the host-buffer entry point), it beats
    the straight line LM-CMA starts from, and it is written one state per line (printAsMatrix convention)."""
    r = _example(["plan", "path.txt", "300"], tmp_path)
    assert r.returncode == 0, r.stdout + r.stderr
    fields = r.stdout.split()
    assert float(fields[fields.index("best") + 2]) < float(fields[fields.index("initial") + 2])
    pts = np.loadtxt(tmp_path / "path.txt")
    assert pts.shape == (22, 2) and tuple(pts[0]) == (99.0, 0.0) and tuple(pts[-1]) == (0.0, 99.0)


def test_long_free_run_stays_finite_and_tracks_the_oracle(po):
    """Regression for two FP32 hazards found on the C2 workload once sigma has collapsed (evolution paths nearly
    collinear with the stored directions, steps below ulp(x)): the recombination works on offsets formed in FP64
    (OptDev::D), and |v|^2 is a real reduction over the finished row (a scalar recurrence cancels catastrophically).
    The device runs fused generations; the FP64 oracle is fed the device's deviates and fitness."""
    W, lam, m = 100, 256, 28
    dist, start, goal = maps.config2_map(size=1024, n_rects=128, seed=42, clamp=64.0)
    lo, hi = maps.box_bounds((1024, 1024), W)
    x0 = maps.straight_line(start, goal, W)
    cm = L.CostMap(dist, "f32")
    dev = L.Optimizer(2 * W, x0=x0, lam=lam, m=m, lo=lo, hi=hi, sigma0=8.0, seed=5, record_z=True)
    dev.attach_cost(cm, [start], [goal], W, L.LONGSAFE, 1e4)
    ora = po.OracleLMCMA(2 * W, x0=x0, lam=lam, m=m, lo=lo, hi=hi, sigma=8.0, seed=1, Z0=dev.get("Z")[0].astype(np.float64))
    worst = 0.0
    for g in range(260):
        Xd, Xo = dev.get("X")[0], ora.array("X")
        assert np.isfinite(Xd).all(), g
        if g < 40:
            worst = max(worst, float(np.abs(Xd - Xo).max()))
        dev.run(1)
        ora.tell_all(dev.get("fit")[0].astype(np.float64), dev.get("Z")[0].astype(np.float64))
    assert worst < 5e-2, worst                                   # cells; same ranks -> same sigma, FP32 drift only
    assert np.isfinite(dev.get("V")[0]).all() and np.isfinite(dev.get("xmean")[0]).all()
    sd, so = float(dev.get("sigma")[0]), ora.doubles()["sigma"]
    assert abs(sd - so) <= 1e-6 * so                             # sigma depends on the (shared) fitness ranks only


def test_smoothness_prior_sampling_matches_the_reference(golden):
    """The covariance-prior path (cholesky + applyCovL before computeAz, lmcma.cpp:165-169, 216-217, 844-864) against
    the compiled reference (Eigen stand-in: shim-pinned): same Hansen stream, prior = covariance(2, 10).  The first
    population is x0 + sigma L z exactly; later generations are compared free-running over a short window."""
    g = golden["run_prior_shim_pinned"]
    cov = np.array(golden["covariance_2_10_shim_pinned"]).reshape(20, 20)
    opt = L.LMCMA(np.array(g["x0"]), lambda_=g["lambda"], sigma=g["sigma0"], covariance=cov, inseed=1)
    opt.init(20)
    for gen in range(4):
        ref = g["gens"][gen]
        for i in range(g["lambda"]):
            xi = opt.getNextParameterVector()
            tol = 2e-5 if gen == 0 else 2e-3
            assert np.allclose(xi, np.array(ref["X"][i]), rtol=tol, atol=tol), (gen, i, np.abs(xi - np.array(ref["X"][i])).max())
            opt.setEvaluationFeedback(ref["f"][i])      # the reference's fitness: identical ranks on both sides
        assert abs(opt._opt.get("sigma")[0] - g["sigma"][gen + 1]) < 1e-9 * g["sigma"][gen + 1]
    # throughput mode: device Philox deviates through the same contraction, large population (tiled kernel, wide sampler)
    n, lam = 400, 512
    big = np.zeros(n * n)
    from lmcma_path_planner_b200 import _capi as K
    assert K.lib().lmcma_b200_covariance(2, 200, K.dptr(big)) == 0
    big = big.reshape(n, n)
    dev = L.Optimizer(n, x0=np.zeros(n), lam=lam, sigma0=1.0, seed=3, record_z=True, covariance=big)
    Z, X = dev.get("Z")[0].astype(np.float64), dev.get("X")[0].astype(np.float64)
    want = Z @ np.linalg.cholesky(big).T                          # no pairs yet: x = x0 + sigma * L z
    assert np.abs(X - want).max() < 1e-5 * max(1.0, np.abs(want).max())


# ------------------------------------------------------------------------------------------------
# distance transform on the device (SURVEY 8f.1)
# ------------------------------------------------------------------------------------------------
def test_edt_device_is_exact(po, golden_maps):
    """k_edt against scipy's exact EDT (bit-equal: integer squared distances, one FP64 sqrt rounded to FP32) on the
    reference's 100 x 100 maps, random 2-D / 3-D grids with odd sizes, and the clamp; the 8SSEDT the reference uses
    (planner.cpp:403-490) is only approximate, so it is compared with a tolerance of one cell."""
    rng = np.random.default_rng(2)
    cases = [golden_maps["problem1"], golden_maps["two_bars"], (rng.random((37, 53)) < 0.05), (rng.random((130, 257)) < 0.002),
             (rng.random((9, 21, 34)) < 0.03), (rng.random((40, 33, 65)) < 0.001)]
    for occ in cases:
        want = po.edt_exact(np.asarray(occ, np.uint8))
        got = maps.edt_device(occ)
        assert np.array_equal(got, want), (np.asarray(occ).shape, float(np.abs(got - want).max()))
    occ = cases[3]
    assert np.array_equal(maps.edt_device(occ, clamp=7.5), np.minimum(po.edt_exact(np.asarray(occ, np.uint8)), np.float32(7.5)))
    sd = po.ssedt8_signed(golden_maps["problem1"])                        # int(sqrt(d1)) - int(sqrt(d2)) of the reference
    ours = np.floor(maps.edt_device(golden_maps["problem1"])) - np.floor(maps.edt_device(1 - golden_maps["problem1"]))
    assert np.abs(ours - sd).max() <= 1


def test_map_from_occupancy_equals_map_from_distance_field(po):
    """distance transform + bricking on the device == host EDT + lmcma_b200_map_create: identical costs and collisions."""
    rng = np.random.default_rng(4)
    occ = maps.random_boxes_occupancy((200, 300), 12, 5, 30, seed=9, border=2, clear=[((20.0, 20.0), 12.0), ((280.0, 180.0), 12.0)])
    W, start, goal = 30, (20.0, 20.0), (280.0, 180.0)
    lo, hi = maps.box_bounds((300, 200), W)
    X = _candidates(rng, maps.straight_line(start, goal, W), 64, 9.0, lo, hi)
    for storage in ("f32", "u8"):
        a = L.CostMap(maps.distance_field(occ, 40.0), storage).evaluate(X, start, goal, W)
        b = L.CostMap.from_occupancy(occ, 40.0, storage).evaluate(X, start, goal, W)
        assert np.array_equal(a["ncoll"], b["ncoll"]) and np.array_equal(a["f"], b["f"])


def test_cpp_planner_driver_from_a_map_file(tmp_path):
    """File -> occupancy (g < 128) -> distance transform -> LM-CMA planning -> printAsMatrix-style path, in C++."""
    import struct
    occ = maps.two_bars_occupancy()
    rgb = np.where(occ[:, :, None] > 0, 0, 255).astype(np.uint8).repeat(3, axis=2)
    h, w, _ = rgb.shape
    stride = (w * 3 + 3) & ~3
    data = b"".join(rgb[y, :, ::-1].tobytes() + b"\0" * (stride - w * 3) for y in range(h - 1, -1, -1))
    hdr = b"BM" + struct.pack("<IHHI", 54 + len(data), 0, 0, 54) + struct.pack("<IiiHHIIiiII", 40, w, h, 1, 24, 0, len(data), 2835, 2835, 0, 0)
    (tmp_path / "bars.bmp").write_bytes(hdr + data)
    r = _example(["planfile", "bars.bmp", "99,0", "0,99", "p.txt", "200", "20", "128"], tmp_path)
    assert r.returncode == 0, r.stdout + r.stderr
    pts = np.loadtxt(tmp_path / "p.txt")
    assert pts.shape == (22, 2) and tuple(pts[0]) == (99.0, 0.0) and tuple(pts[-1]) == (0.0, 99.0)


def test_cpp_planner_driver_from_an_octomap_tree(tmp_path):
    """.bt (OcTree::writeBinary, what planner.cpp:152-163 reads) -> dense occupancy -> device EDT -> 3-D LM-CMA planning.
    A ball on the straight line: the planned path must go around it (the driver re-evaluates it: no collisions)."""
    from test_ingest_cpu import _write_bt
    base = 32768 - 10
    g = np.arange(40)
    ball = (g[:, None, None] - 19.5) ** 2 + (g[None, :, None] - 19.5) ** 2 + (g[None, None, :] - 19.5) ** 2 <= 7.0 ** 2
    occ = {(base + int(x), base + int(y), base + int(z)) for x, y, z in zip(*np.nonzero(ball))}
    occ.update((base + x, base + y, base + z) for x in (0, 39) for y in (0, 39) for z in (0, 39))   # bounding box = 40^3
    _write_bt(str(tmp_path / "ball.bt"), occ, set(), 0.1)
    r = _example(["planfile", "ball.bt", "5,5,5", "34,34,34", "p.txt", "300", "12", "256"], tmp_path)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "map 40x40x40" in r.stdout and "collisions 0" in r.stdout, r.stdout
    pts = np.loadtxt(tmp_path / "p.txt")
    assert pts.shape == (14, 3) and tuple(pts[0]) == (5.0, 5.0, 5.0) and tuple(pts[-1]) == (34.0, 34.0, 34.0)


def test_lmcma_teacher_forced_gram_path(po, monkeypatch):
    """The Gram-matrix recompute (k_gram / k_coef / k_combine): forced on the C2-like shape so that slot recycling
    (itr >= m, first_stale > 0) is exercised, then on the C4 row length where it is the default (m * n = 115 K floats
    fit neither registers nor shared memory), past the point where all 77 slots are live."""
    monkeypatch.setenv("LMCMA_B200_UPDATE_GRAM", "1")
    _teacher_forced(po, 400, 128, 40, 50, seed=3, sigma=0.5)
    monkeypatch.delenv("LMCMA_B200_UPDATE_GRAM")
    _teacher_forced(po, 1500, 32, 77, 84, seed=4, sigma=0.3)


def test_progressive_and_overlapped_generations_are_bit_identical_to_the_serial_order(po, monkeypatch):
    """k_sample consuming the direction pairs while k_update's sweep is still publishing them (release / acquire flags,
    k_update.cuh "progressive") must not change a single bit relative to running the two kernels back to back: same
    operations in the same order, only earlier.  Fused generations past the point where slots are recycled."""
    W, lam, m = 100, 512, 24
    dist, start, goal = maps.config2_map(size=1024, n_rects=128, seed=42, clamp=64.0)
    lo, hi = maps.box_bounds((1024, 1024), W)
    x0 = maps.straight_line(start, goal, W)
    cm = L.CostMap(dist, "f32")
    state = {}
    # serial order / progressive hand-over / overlapped generation (k_update on a side branch of the graph, concurrent with
    # k_cost and k_rank: everything that does not depend on this generation's fitness runs first)
    for mode, (prog, ovl) in {"serial": ("0", "0"), "progressive": ("1", "0"), "overlapped": ("1", "1")}.items():
        monkeypatch.setenv("LMCMA_B200_PROGRESSIVE", prog)
        monkeypatch.setenv("LMCMA_B200_OVERLAP", ovl)
        dev = L.Optimizer(2 * W, x0=x0, lam=lam, m=m, lo=lo, hi=hi, sigma0=8.0, seed=11)
        dev.attach_cost(cm, [start], [goal], W, L.LONGSAFE, 1e4)
        dev.run(70)
        state[mode] = {k: dev.get(k).copy() for k in ("X", "xmean", "V", "P", "sigma", "fit", "t", "vec", "Nj", "Lj")}
        state[mode]["best_f"] = dev.best()[1].copy()
    for mode in ("progressive", "overlapped"):
        for k in state["serial"]:
            assert np.array_equal(state[mode][k], state["serial"][k]), (mode, k)
    # the same through the host-buffer protocol: tell_all runs k_update's fitness-independent part on a side stream while
    # the fitness is copied and ranked (LMCMA_B200_TELL_OVERLAP, default on) — same bits as the fused generations above
    monkeypatch.setenv("LMCMA_B200_PROGRESSIVE", "1")
    monkeypatch.setenv("LMCMA_B200_OVERLAP", "1")
    for tell in ("1", "0"):
        monkeypatch.setenv("LMCMA_B200_TELL_OVERLAP", tell)
        dev = L.Optimizer(2 * W, x0=x0, lam=lam, m=m, lo=lo, hi=hi, sigma0=8.0, seed=11)
        for g in range(70):
            r = cm.evaluate(dev.ask_all()[0], start, goal, W, L.LONGSAFE, 1e4)
            dev.tell_all(r["f"])
        for k in ("X", "xmean", "V", "P", "sigma", "t", "vec", "Nj", "Lj"):
            assert np.array_equal(dev.get(k), state["serial"][k]), ("tell_all overlap " + tell, k)
        assert np.array_equal(dev.best()[1], state["serial"]["best_f"])


def test_speculative_update_of_tell_all_never_shows_and_never_goes_stale(po, monkeypatch):
    """Every tell_all graph ends with the fitness-independent part of the NEXT generation's update (k_update phase 1, into a
    scratch buffer) and the next tell_all resumes from it (phase 2).  The optimiser's state between two calls must be the
    state of the generation just told — getters never see the pass — and anything else that advances or overwrites the state
    (fused generations, a setter) must make the next tell_all recompute: bit-identical to the same calls with the pass off."""
    W, lam, m = 60, 256, 16
    dist, start, goal = maps.config2_map(size=512, n_rects=48, seed=4, clamp=64.0)
    lo, hi = maps.box_bounds((512, 512), W)
    x0 = maps.straight_line(start, goal, W)
    cm = L.CostMap(dist, "f32")
    keys = ("X", "xmean", "V", "P", "sigma", "t", "vec", "Nj", "Lj", "pc")
    trace = {}
    for spec in ("0", "1"):
        monkeypatch.setenv("LMCMA_B200_TELL_SPEC", spec)
        dev = L.Optimizer(2 * W, x0=x0, lam=lam, m=m, lo=lo, hi=hi, sigma0=6.0, seed=5)
        dev.attach_cost(cm, [start], [goal], W, L.LONGSAFE, 1e4)
        snaps = []
        for g in range(40):
            # ask_all_view: the pass is part of tell_all only with the host mirror on (the candidates' trip across PCIe hides it)
            r = cm.evaluate(np.array(dev.ask_all_view()[0]), start, goal, W, L.LONGSAFE, 1e4)
            dev.tell_all(r["f"])
            snaps.append({k: dev.get(k).copy() for k in keys})    # between two calls: the generation just told
            if g == 12:
                dev.run(3)                                        # fused generations: the rows left behind are stale
                snaps.append({k: dev.get(k).copy() for k in keys})
            if g == 25:
                dev.set("V", dev.get("V"))                        # a setter (same values): the next tell_all must not resume
            if g == 30:
                dev.set("sigma", dev.get("sigma") * 0.5)
        trace[spec] = snaps
    assert len(trace["0"]) == len(trace["1"])
    for i, (a, b) in enumerate(zip(trace["0"], trace["1"])):
        for k in keys:
            assert np.array_equal(a[k], b[k]), (i, k)


def test_cost_evaluate_page_locked_buffers_match_staged(po, golden_maps, monkeypatch):
    """lmcma_b200_cost_evaluate hands page-locked caller buffers to the kernel directly (candidates read across PCIe
    by the CTAs, results stored into the caller's arrays); pageable buffers are staged.  Same bits either way."""
    import ctypes as C
    import torch
    from lmcma_path_planner_b200 import _capi as K
    from lmcma_path_planner_b200.optimizer import _endpoints, _objective
    dist = po.edt_exact(golden_maps["problem1"])
    W, start, goal = 23, (99.0, 0.0), (0.0, 99.0)                # n = 46: rows are not 16-byte aligned
    lo, hi = maps.box_bounds((100, 100), W)
    rng = np.random.default_rng(5)
    X = _candidates(rng, maps.straight_line(start, goal, W), 300, 9.0, lo - 4.0, hi + 4.0)   # some samples leave the map
    cm = L.CostMap(dist, "f32")
    ref = cm.evaluate(X, start, goal, W)                          # pageable numpy buffers: staged
    Xp = torch.from_numpy(X.copy()).pin_memory().numpy()
    fp = torch.zeros(300, dtype=torch.float32).pin_memory().numpy()
    ncp = torch.zeros(300, dtype=torch.int32).pin_memory().numpy()
    nsp = torch.zeros(300, dtype=torch.int32).pin_memory().numpy()
    obj, ends = _objective(W, L.LONGSAFE, 1e4), _endpoints(start, goal)
    for zc in ("1", "0"):
        monkeypatch.setenv("LMCMA_B200_ZEROCOPY", zc)
        cm2 = L.CostMap(dist, "f32")                              # the knob is read when the map handle is created
        fp[:] = 0; ncp[:] = 0; nsp[:] = 0
        K.check(K.lib().lmcma_b200_cost_evaluate(cm2._h, C.byref(obj), C.byref(ends), K.fptr(Xp), 300, K.fptr(fp), K.iptr(ncp), K.iptr(nsp)))
        assert np.array_equal(fp, ref["f"]) and np.array_equal(ncp, ref["ncoll"]) and np.array_equal(nsp, ref["nsamp"]), zc
    orc = po.CostProblem(dist, start, goal, W).evaluate(X)
    assert np.array_equal(ref["ncoll"], orc["ncoll"]) and rel_err(ref["f"], orc["f"]) < COST_RTOL


def test_cost_long_trajectories_and_staged_rounds(po, monkeypatch):
    """More segments than threads (W = 600: three segments per thread), and the per-block record stage forced small so
    that every trajectory takes many rounds of block records (k_cost phase 2a / 2b); both storages, bit-exact counts."""
    dist, start, goal = maps.config2_map(size=512, n_rects=48, seed=3, clamp=64.0)
    W = 600
    rng = np.random.default_rng(8)
    lo, hi = maps.box_bounds((512, 512), W)
    X = _candidates(rng, maps.straight_line(start, goal, W), 64, 6.0, lo - 3.0, hi + 3.0)
    for cb in ("0", "8"):
        monkeypatch.setenv("LMCMA_B200_COST_CB", cb)
        for storage in ("f32", "u8"):
            cm = L.CostMap(dist, storage, u8_scale=0.25)
            dd = dist if storage == "f32" else cm.dequantized()
            ref = po.CostProblem(dd, start, goal, W).evaluate(X)
            got = cm.evaluate(X, start, goal, W)
            assert np.array_equal(got["ncoll"], ref["ncoll"]), (cb, storage)
            assert np.array_equal(got["nsamp"], ref["nsamp"]), (cb, storage)
            assert rel_err(got["f"], ref["f"]) < COST_RTOL, (cb, storage)


def test_cost_six_ctas_per_sm_build_meets_the_same_bar(po, monkeypatch):
    """LMCMA_B200_COST_MINB=6 selects k_cost compiled for six CTAs per SM (40 registers, no local-memory spill; kept
    for many-wave batched shapes, DESIGN.md section 8.7): same source, so the same parity bar against the oracle - cell
    indices bit-exact (collision and sample counts), cost within COST_RTOL - in 2-D and 3-D, f32 and u8 storage."""
    monkeypatch.setenv("LMCMA_B200_COST_MINB", "6")
    rng = np.random.default_rng(12)
    dist, start, goal = maps.config2_map(size=512, n_rects=48, seed=3, clamp=64.0)
    W = 60
    lo, hi = maps.box_bounds((512, 512), W)
    X = _candidates(rng, maps.straight_line(start, goal, W), 200, 6.0, lo - 3.0, hi + 3.0)
    for storage in ("f32", "u8"):
        cm = L.CostMap(dist, storage, u8_scale=0.25)
        dd = dist if storage == "f32" else cm.dequantized()
        ref = po.CostProblem(dd, start, goal, W).evaluate(X)
        got = cm.evaluate(X, start, goal, W)
        assert np.array_equal(got["ncoll"], ref["ncoll"]) and np.array_equal(got["nsamp"], ref["nsamp"]), storage
        assert rel_err(got["f"], ref["f"]) < COST_RTOL, storage
    d3, s3, g3 = maps.config4_map(size=64, n_boxes=4096, seed=9, clamp=16.0)
    W3 = 40
    lo3, hi3 = maps.box_bounds((64, 64, 64), W3)
    X3 = _candidates(rng, maps.straight_line(s3, g3, W3), 100, 3.0, lo3, hi3)
    ref = po.CostProblem(d3, s3, g3, W3).evaluate(X3)
    got = L.CostMap(d3, "f32").evaluate(X3, s3, g3, W3)
    assert np.array_equal(got["ncoll"], ref["ncoll"]) and np.array_equal(got["nsamp"], ref["nsamp"])
    assert rel_err(got["f"], ref["f"]) < COST_RTOL


def test_cpp_facade_demo_with_the_covariance_prior(tmp_path):
    """test_lmcma_using_cov (example_lmcma.cpp:78-127) against the facade: covariance(2, 1) through the reference's free
    function name is the identity, so the run draws the same stream as the plain demo and converges to the same basin."""
    r = _example(["democov", "1"], tmp_path)
    assert r.returncode == 0, r.stderr
    tail = r.stdout.strip().split("is:")[1].split()
    x, y = (float(v) for v in tail[0].split(","))
    assert abs(x - 3.99966) < 2e-2 and abs(y - 3.99966) < 2e-2
    assert "cov=[1 0; 0 1]" in r.stdout and "counteval=1000" in r.stdout
    assert len(open(tmp_path / "path_to_max_using_cov.csv").read().strip().splitlines()) == 1001


def test_the_reference_s_own_demo_binary_runs_on_the_b200_library(tmp_path):
    """oracle/_ref/ref_example_lmcma is the reference's example_lmcma.cpp compiled UNCHANGED against include/lmcma.hpp
    (oracle/Makefile ref_example; tests/test_capi_cpu.py repeats the compile where the reference tree exists): both of its
    demos (plain and with the covariance prior) must run on the device library and end in the global basin (4, 4)."""
    import os
    import subprocess
    exe = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "_ref", "ref_example_lmcma")
    if not os.path.exists(exe):
        pytest.skip("oracle/_ref/ref_example_lmcma was not built (no reference tree in the authoring container)")
    r = subprocess.run([exe], cwd=tmp_path, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    pts = [ln.split("is:")[1] for ln in r.stdout.splitlines() if "optimum point is:" in ln]
    assert len(pts) == 2, r.stdout
    for p in pts:
        x, y = (float(v) for v in p.split(","))
        assert abs(x - 4.0) < 5e-2 and abs(y - 4.0) < 5e-2, r.stdout
    assert (tmp_path / "path_to_min.csv").exists() and (tmp_path / "path_to_max_using_cov.csv").exists()


def test_ask_all_view_mirror_tracks_the_population(po, golden_maps):
    """lmcma_b200_ask_all_view: the page-locked mirror the sampler writes while it runs holds exactly what ask_all copies,
    generation after generation through tell_all (graph path and stream-ordered path), after fused on-device generations
    (which do not write it: one ordinary copy refreshes it) and after a state setter; lmcma_b200_cost_evaluate called with
    the view pointer evaluates the device copy and returns the same bits as with the caller's own buffer."""
    import ctypes as C
    import torch
    from lmcma_path_planner_b200 import _capi as K
    from lmcma_path_planner_b200.optimizer import _endpoints, _objective
    dist = po.edt_exact(golden_maps["problem2"])
    cm = L.CostMap(dist, "f32")
    W, start, goal = 100, (99.0, 0.0), (0.0, 99.0)
    lo, hi = maps.box_bounds((100, 100), W)
    x0 = maps.straight_line(start, goal, W)
    obj, ends = _objective(W, L.LONGSAFE, 1e4), _endpoints(start, goal)
    for lam, n_extra in ((512, 0), (24, 0)):                       # wide sampler + tell graph / narrow sampler, stream-ordered tell
        dev = L.Optimizer(2 * W, x0=x0, lam=lam, m=12, lo=lo, hi=hi, sigma0=4.0, seed=3)
        dev.attach_cost(cm, [start], [goal], W, L.LONGSAFE, 1e4)
        fp = torch.zeros(lam, dtype=torch.float32).pin_memory().numpy()
        for g in range(15):
            V = dev.ask_all_view()
            X = dev.ask_all()
            assert np.array_equal(V, X), (lam, g)
            ref = cm.evaluate(X[0], start, goal, W)
            xp, ld = C.POINTER(C.c_float)(), C.c_int64(0)
            K.check(K.lib().lmcma_b200_ask_all_view(dev._h, C.byref(xp), C.byref(ld)))
            K.check(K.lib().lmcma_b200_cost_evaluate(cm._h, C.byref(obj), C.byref(ends), xp, lam, K.fptr(fp), None, None))
            assert np.array_equal(fp, ref["f"]), (lam, g)
            dev.tell_all(fp)
            if g == 6:
                dev.run(3)                                         # fused generations do not write the mirror
                assert np.array_equal(dev.ask_all_view(), dev.ask_all())
            if g == 9:
                dev.set("X", dev.ask_all() + 1.0)                  # a setter invalidates it
                assert np.array_equal(dev.ask_all_view(), dev.ask_all())


def test_ipop_restarts_tool_runs_and_reports(tmp_path):
    """C5 mechanics (tools/c5_ipop_restarts.py): doubling populations on the cluttered map, every restart a fresh optimiser
    stopped by the reference's sigma rule or the generation cap, best path re-evaluated for its collision count.  Small
    sizes here (512^2 map, lambda 64..256); the 8-GPU run at lambda 1024..65536 is under profiles/."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "tools", "c5_ipop_restarts.py"), "256", "40", "64", "512"],
                       cwd=tmp_path, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("  rank") and "generations" in ln]
    assert len(lines) == 3 and "C5: 3 restarts (lambda 64..256)" in r.stdout, r.stdout
    assert all("colliding samples" in ln for ln in lines)


def test_split_population_over_nccl_two_ranks(tmp_path):
    """C4 mechanics over REAL NCCL (needs >= 2 visible GPUs; skipped on a single-GPU box): tools/c4_split_population.py under
    torchrun, two ranks, 64^3 u8 map, lambda = 512, 8 generations: the split run must equal the unsplit optimiser to 1e-9 on
    sigma and 1e-2 cells on the mean (only the association of the per-rank partial sums differs), and the replicas must be
    bit-identical on both ranks."""
    import os
    import subprocess
    import sys
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                        "--master-port", "29541", os.path.join(root, "tools", "c4_split_population.py"), "64", "40", "512", "5", "strict"],
                       cwd=tmp_path, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "strict check passed" in r.stdout and "replicas bit-identical on all 2 ranks" in r.stdout
