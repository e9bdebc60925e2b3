"""GPU parity at the EXACT shapes bench.py times (VERDICT r1, weak #1): the kernel variants the launcher picks for the
benchmarked populations — k_sample_wide<4,512>, k_rank with 32 slices / its multi-tile path (lambda > 4096),
k_update<4,3,smem>(+OVERLAP), the Gram-matrix update of the C4 row length, the split-population stages — against the
FP64 oracle on the same inputs.  Same bars as tests/test_gpu_parity.py: integer state bit-exact, floating state 2e-5
of its scale, sigma 1e-12, cost 1e-5."""
import numpy as np
import pytest

import lmcma_path_planner_b200 as L
from lmcma_path_planner_b200 import maps
from test_gpu_parity import _teacher_forced, rel_err, COST_RTOL

pytestmark = pytest.mark.gpu


def test_teacher_forced_at_the_c2_shape(po):
    """C2 exactly: n = 400, lambda = 1024, m = 40, 46 generations (slots recycle from generation 40 on).  lambda >= 1024
    selects k_sample_wide<4,512> (RBW = 4) and k_rank with 32 row slices; m = 40 the register sweep k_update<4,3,smem>."""
    _teacher_forced(po, 400, 1024, 40, 46, seed=21, sigma=0.5)


def test_teacher_forced_at_the_c2_shape_with_bounds(po):
    """The same launch shapes with the box bounds of the planning problem active on part of the population."""
    n = 400
    _teacher_forced(po, n, 1024, 40, 12, seed=22, sigma=0.8, lo=np.full(n, -0.2), hi=np.full(n, 1.1))


@pytest.fixture(scope="module")
def c2_problem():
    dist, start, goal = maps.config2_map()
    W = 200
    lo, hi = maps.box_bounds((4096, 4096), W)
    return dict(dist=dist, start=start, goal=goal, W=W, lo=lo, hi=hi, x0=maps.straight_line(start, goal, W),
                cmap=L.CostMap(dist, "f32"))


@pytest.mark.parametrize("overlap", ["1", "0"])
def test_fused_c2_generation_tracks_the_oracle(po, c2_problem, monkeypatch, overlap):
    """The graph-replayed generation bench.py times (4096^2 map, device Philox deviates, k_update on the side branch when
    LMCMA_B200_OVERLAP=1 / the serial PDL chain when 0), teacher-forced every generation: the oracle is fed the device's
    recorded deviates and fitness, the device then continues from the oracle's exact state.  46 generations, so the
    recycling branch of the slot logic runs inside the overlapped k_update too."""
    monkeypatch.setenv("LMCMA_B200_OVERLAP", overlap)
    p = c2_problem
    n, lam, m = 2 * p["W"], 1024, 40
    dev = L.Optimizer(n, x0=p["x0"], lam=lam, m=m, lo=p["lo"], hi=p["hi"], sigma0=32.0, seed=5, record_z=True)
    dev.attach_cost(p["cmap"], [p["start"]], [p["goal"]], p["W"], L.LONGSAFE, 1e4)
    ora = po.OracleLMCMA(n, x0=p["x0"], lam=lam, m=m, lo=p["lo"], hi=p["hi"], sigma=32.0, seed=1,
                         Z0=dev.get("Z")[0].astype(np.float64))
    prob = po.CostProblem(p["dist"], p["start"], p["goal"], p["W"], threads=8)
    rng = np.random.default_rng(1)
    worst = {}
    for g in range(46):
        Xd, Xo = dev.get("X")[0], ora.array("X")
        worst["X"] = max(worst.get("X", 0), float(np.abs(Xd - Xo).max()) / 4095.0)
        dev.run(1)                                                 # k_cost -> k_rank -> k_update -> k_sample, one graph
        f = dev.get("fit")[0]
        if g % 9 == 0:                                             # the fitness itself, on a row sample
            idx = rng.choice(lam, 16, replace=False)
            ref = prob.evaluate(Xd[idx])
            assert np.array_equal(dev.get("ncoll")[0][idx], ref["ncoll"]), g
            assert rel_err(f[idx], ref["f"]) < COST_RTOL, g
        ora.tell_all(f.astype(np.float64), dev.get("Z")[0].astype(np.float64))
        so = ora.state()
        live = so["live"]
        assert np.array_equal(dev.get("t")[0][:live], so["t"][:live]), g
        assert np.array_equal(dev.get("vec")[0][so["t"][:live]], so["vec"][so["t"][:live]]), g
        assert np.array_equal(dev.get("arindex")[0], ora.int_array("arindex")), g
        assert int(dev.get("itr")[0]) == so["itr"] and int(dev.get("live")[0]) == live
        worst["sigma"] = max(worst.get("sigma", 0), abs(dev.get("sigma")[0] - so["sigma"]) / so["sigma"])
        worst["xmean"] = max(worst.get("xmean", 0), float(np.abs(dev.get("xmean")[0] - so["xmean"]).max()) / 4095.0)
        pcs = max(1e-6, float(np.abs(so["pc"]).max()))
        worst["pc"] = max(worst.get("pc", 0), float(np.abs(dev.get("pc")[0] - so["pc"]).max()) / pcs)
        Vd = dev.get("V")[0]
        for slot in so["t"][:live]:
            vs = max(1e-6, float(np.abs(so["V"][slot]).max()))
            worst["V"] = max(worst.get("V", 0), float(np.abs(Vd[slot] - so["V"][slot]).max()) / vs)
        dev.load_state(so)
        dev.resample()                                             # same Philox rows (counter = itr), oracle's exact state
    assert worst["sigma"] < 1e-12, worst
    for k in ("X", "xmean", "pc", "V"):
        assert worst[k] < 2e-5, (k, worst)


@pytest.mark.parametrize("lam", [4097, 8192, 65536])
def test_rank_beyond_one_fitness_tile(po, lam):
    """k_rank for lambda > 4096 (fitness re-staged tile by tile, several passes per thread group) against the oracle's
    stable sort (= the reference's myqsort order, tests/test_oracle_golden.py): heavy ties, -0 / +0, NaN, +inf; and the
    pair count of the merged 2*lambda ranking through the step size of the following generation."""
    rng = np.random.default_rng(lam)
    n = 8
    def fitness():
        f = rng.integers(0, max(4, lam // 64), lam).astype(np.float32)      # ~64 candidates per distinct value
        f[rng.integers(0, lam, 9)] = -0.0
        f[rng.integers(0, lam, 9)] = 0.0
        f[rng.integers(0, lam, 5)] = np.inf
        return f
    dev = L.Optimizer(n, x0=np.zeros(n), lam=lam, m=4, rng="inject", sigma0=1.0)
    ora = po.OracleLMCMA(n, x0=np.zeros(n), lam=lam, m=4, sigma=1.0, Z0=np.zeros((lam, n)))
    z = np.zeros((lam, n), np.float32)
    dev.inject_z(z)
    for g in range(3):
        f = fitness()
        dev.inject_z(z)
        dev.tell_all(f)
        ora.tell_all(f.astype(np.float64), z.astype(np.float64))
        want_sorted, want_ids = po.rank(f.astype(np.float64))
        assert np.array_equal(dev.get("arindex")[0], want_ids), g
        assert np.array_equal(dev.get("arindex")[0], ora.int_array("arindex")), g
        assert np.array_equal(dev.get("fit_sorted")[0].view(np.uint32) & 0x7fffffff,
                              want_sorted.astype(np.float32).view(np.uint32) & 0x7fffffff), g   # -0 == +0
        inv = np.empty(lam, np.int32); inv[want_ids] = np.arange(lam, dtype=np.int32)
        assert np.array_equal(dev.get("rank")[0], inv), g
        so = ora.doubles()["sigma"]
        assert abs(dev.get("sigma")[0] - so) <= 1e-12 * so, g       # S = #{prev_j < cur_i} over 2*lambda values
    f = fitness(); f[7] = np.nan; f[lam - 3] = np.nan                # NaN ranks as +inf (DESIGN.md 5): last, ties by id
    dev.inject_z(z)
    dev.tell_all(f)
    _, want_ids = po.rank(np.where(np.isnan(f), np.inf, f).astype(np.float64))
    got = dev.get("arindex")[0]
    assert np.array_equal(got, want_ids)
    tail = got[-int(np.sum(np.isinf(f) | np.isnan(f))):].tolist()      # the +inf and the two NaN candidates, in id order
    assert 7 in tail and lam - 3 in tail and tail == sorted(tail)


def test_split_population_at_the_c4_shape(po):
    """C4 per-rank shapes: n = 1500, m = 77, lambda = 8192 in 8 slices of pop_count = 1024 (wide sampler, Gram-matrix
    update, split ranking with the payload fold), on a 256^3 u8 voxel map.  All 8 slice handles live on this one GPU and
    the two all-gathers are done by hand (same kernels and buffers as the NCCL run).  The oracle (lambda = 8192) is
    warm-started from a cheap small-population run of the same restatement so that all 77 slots are live and being
    recycled; every generation is teacher-forced from the oracle's exact state."""
    import torch
    size, W, lam, G = 256, 500, 8192, 8
    n, m, pc = 3 * W, 77, lam // G
    dist, start, goal = maps.config4_map(size=size, n_boxes=512, seed=43)
    cmap = L.CostMap(dist, "u8", u8_scale=0.25)
    prob = po.CostProblem(cmap.dequantized(), start, goal, W, threads=8)
    lo, hi = maps.box_bounds((size, size, size), W)
    x0 = maps.straight_line(start, goal, W)
    # warm state: 90 generations of a lambda = 32 oracle around the straight line (cheap quadratic bowl)
    small = po.OracleLMCMA(n, x0=x0, lam=32, m=m, lo=lo, hi=hi, sigma=4.0, seed=1)
    for g in range(90):
        X = small.array("X")
        small.tell_all(np.sum((X - x0) ** 2 * (1.0 + np.arange(n) % 7), axis=1))
    st = small.state()
    assert st["live"] == m and st["itr"] == 90
    st["sigma"] = 4.0                                               # a population that spreads over several cells again
    rng = np.random.default_rng(8)
    prev = np.sort(rng.random(lam) * 1e6).astype(np.float32)
    parts = []
    for r in range(G):
        p = L.Optimizer(n, x0=x0, lam=lam, m=m, lo=lo, hi=hi, sigma0=4.0, seed=43, pop_offset=r * pc, pop_count=pc, record_z=True)
        p.attach_cost(cmap, [start], [goal], W, L.LONGSAFE, 1e4)
        parts.append(p)
    ora = po.OracleLMCMA(n, x0=x0, lam=lam, m=m, lo=lo, hi=hi, sigma=4.0, seed=1)
    pf = parts[0].mg_payload_floats()
    f_all = torch.zeros(lam, dtype=torch.float32, device="cuda")
    pay_all = torch.zeros(G * pf, dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    worst = {}
    for g in range(3):
        for p in parts:
            p.load_state(dict(st, prev_fit=prev))
            p.resample()
        Z = np.concatenate([p.get("Z")[0] for p in parts]).astype(np.float64)
        ora.load_state(st, prev.astype(np.float64), Z)
        Xo = ora.array("X")
        Xd = np.concatenate([p.get("X")[0] for p in parts])
        worst["X"] = max(worst.get("X", 0), float(np.abs(Xd - Xo).max()) / (size - 1.0))
        for r, p in enumerate(parts):
            p.mg_evaluate(f_all.data_ptr() + 4 * r * pc)
            p.sync()
        f = f_all.cpu().numpy()
        idx = rng.choice(lam, 24, replace=False)                    # the 3-D u8 cost at this map size, on a row sample
        ref = prob.evaluate(Xd[idx])
        nc = np.concatenate([p.get("ncoll")[0] for p in parts])
        assert np.array_equal(nc[idx], ref["ncoll"]), g
        assert rel_err(f[idx], ref["f"]) < COST_RTOL, g
        for r, p in enumerate(parts):
            p.mg_rank(f_all.data_ptr(), pay_all.data_ptr() + 4 * r * pf)
            p.sync()
        for p in parts:
            p.mg_update(pay_all.data_ptr(), G)
            p.sync()
        # the oracle recombines ITS candidates (FP64) with the shared fitness
        ora.tell_all(f.astype(np.float64), None)
        so = ora.state()
        want_ids = ora.int_array("arindex")
        inv = np.empty(lam, np.int32); inv[want_ids] = np.arange(lam, dtype=np.int32)
        for r, p in enumerate(parts):
            assert np.array_equal(p.get("rank")[0][r * pc:(r + 1) * pc], inv[r * pc:(r + 1) * pc]), (g, r)
            assert np.array_equal(p.get("t")[0], so["t"]) and np.array_equal(p.get("vec")[0], so["vec"]), (g, r)
            assert int(p.get("itr")[0]) == so["itr"]
            worst["sigma"] = max(worst.get("sigma", 0), abs(p.get("sigma")[0] - so["sigma"]) / so["sigma"])
            worst["xmean"] = max(worst.get("xmean", 0), float(np.abs(p.get("xmean")[0] - so["xmean"]).max()) / (size - 1.0))
            pcs = max(1e-6, float(np.abs(so["pc"]).max()))
            worst["pc"] = max(worst.get("pc", 0), float(np.abs(p.get("pc")[0] - so["pc"]).max()) / pcs)
        for p in (parts[0], parts[G - 1]):
            Vd = p.get("V")[0]
            for slot in range(m):
                vs = max(1e-6, float(np.abs(so["V"][slot]).max()))
                worst["V"] = max(worst.get("V", 0), float(np.abs(Vd[slot] - so["V"][slot]).max()) / vs)
            worst["Nj"] = max(worst.get("Nj", 0), rel_err(p.get("Nj")[0], so["Nj"]))
        for k in ("xmean", "sigma", "V", "pc"):                     # replicas stay bit-identical
            assert np.array_equal(parts[0].get(k), parts[G - 1].get(k)), (g, k)
        st, prev = so, np.sort(f)
    assert worst["sigma"] < 1e-12, worst
    for k in ("X", "xmean", "pc", "V"):
        assert worst[k] < 2e-5, (k, worst)
    assert worst["Nj"] < 1e-4, worst


def test_is_done_and_constants(po, golden):
    """a14: sigma < 1e-20 ends the run (lmcma.cpp:426-429), per instance; a15: the constants the device derives at create
    (c1, cc, K, M, mueff, cs, target — lmcma.cpp:144-156, 238, 268-272) against the golden values read out of the compiled
    reference, and the recombination weights against the oracle's."""
    g = golden["run_n10"]
    dev = L.Optimizer(g["n"], x0=np.array(g["x0"]), lam=g["lambda"], sigma0=g["sigma0"], batch=3, rng="inject")
    c = dict(zip(("c1", "cc", "cs", "target", "K", "M", "mueff"), dev.get("consts")))
    for k, v in g["consts"].items():
        assert c[k] == v, k
    assert c["cs"] == 0.3 and c["target"] == 0.25
    ora = po.OracleLMCMA(g["n"], x0=np.array(g["x0"]), lam=g["lambda"], sigma=g["sigma0"])
    assert np.array_equal(dev.get("weights"), ora.array("weights"))
    assert dev.mu == g["mu"]
    assert not dev.is_done().any()
    dev.set("sigma", [1.0, 9.9e-21, 1e-20])                         # strict '<'
    assert dev.is_done().tolist() == [False, True, False]
    # and through the optimiser itself: a fitness that gets worse every generation makes every generation a failure (all of
    # the previous population ranks ahead: success = -1 < target), sigma shrinks geometrically and the run ends by the
    # reference's own rule
    one = L.LMCMA(np.zeros(6), lambda_=8, sigma=1e-18, inseed=1)
    one.init(6)
    gens = 0
    while not one.isBehaviorLearningDone() and gens < 400:
        for i in range(8):
            one.getNextParameterVector()
            one.setEvaluationFeedback([float(gens)], 1)
        gens += 1
    assert one.isBehaviorLearningDone() and 1 < gens < 400
    ref = po.OracleLMCMA(6, x0=np.zeros(6), lam=8, sigma=1e-18, seed=1)
    rg = 0
    while not ref.done():
        ref.tell_all(np.full(8, float(rg)))
        rg += 1
    assert rg == gens                                               # same stopping generation as the restated reference


def _device_state(dev, b):
    """The distribution state of instance b as the dict oracle.pyoracle.OracleLMCMA.load_state takes."""
    st = {k: dev.get(k)[b].astype(np.float64) for k in ("xmean", "pc", "V", "P", "Nj", "Lj")}
    st.update({k: dev.get(k)[b].copy() for k in ("t", "vec")})
    st.update(itr=int(dev.get("itr")[b]), live=int(dev.get("live")[b]), sigma=float(dev.get("sigma")[b]), s=float(dev.get("s")[b]))
    return st


def _sampler_matches_oracle(po, dev, n, lam, m, lo, hi, instances):
    """The population the device has just sampled == the oracle's sample() from the device's own state and deviates."""
    worst = 0.0
    Z, X = dev.get("Z"), dev.get("X")
    for b in instances:
        st = _device_state(dev, b)
        ora = po.OracleLMCMA(n, x0=np.zeros(n), lam=lam, m=m, lo=lo, hi=hi, sigma=1.0)
        ora.load_state(st, np.zeros(lam), Z[b].astype(np.float64))
        Xo = ora.array("X")
        scale = max(1.0, float(np.abs(Xo).max()))
        worst = max(worst, float(np.abs(X[b] - Xo).max()) / scale)
    return worst


def test_rows_sampler_batched_queries_at_the_c3_shape(po, c2_problem):
    """k_sample_rows (rows on lanes, column slices on warps, two passes; chosen for many rows) at the C3 per-query shape:
    320 queries x lambda 64, n = 400, m = 40 on the 4096^2 map — two rows per lane (RL = 2, QW = 7).  After 12 and after 47
    fused generations (pairs being filled / all 40 live and recycled) the sampled population of several instances is
    held against the FP64 oracle's sample() from the same state and the same recorded deviates; fitness on a row sample
    against the cost oracle."""
    p = c2_problem
    W, lam, m, B = p["W"], 64, 40, 320
    n = 2 * W
    starts, goals = maps.random_queries(p["dist"], B, seed=7, min_sep=1024)
    x0 = np.stack([maps.straight_line(starts[q], goals[q], W) for q in range(B)])
    dev = L.Optimizer(n, x0=x0, lam=lam, m=m, batch=B, lo=p["lo"], hi=p["hi"], sigma0=32.0, seed=7, record_z=True)
    dev.attach_cost(p["cmap"], starts, goals, W, L.LONGSAFE, 1e4)
    for gens in (12, 35):
        dev.run(gens)
        dev.sync()
        assert _sampler_matches_oracle(po, dev, n, lam, m, p["lo"], p["hi"], (0, 7, B - 1)) < 2e-5
    assert int(dev.get("live")[3]) == m
    dev.run(1)
    Xprev = None                                                   # fitness of the population evaluated by that generation: re-evaluate
    b = 5
    X = dev.get("X")[b]
    ref = po.CostProblem(p["dist"], starts[b], goals[b], W, threads=8).evaluate(X[:16])
    got = p["cmap"].evaluate(X[:16], starts[b], goals[b], W)
    assert np.array_equal(got["ncoll"], ref["ncoll"]) and rel_err(got["f"], ref["f"]) < COST_RTOL


@pytest.mark.parametrize("shape", [(400, 4096, 40, 46, 1), (100, 20480, 6, 14, 2), (48, 4096, 11, 30, 1)])
def test_rows_sampler_teacher_forced_single_population(po, monkeypatch, shape):
    """The same kernel forced on ONE large population (LMCMA_B200_SAMPLE_ROWS=1), teacher-forced against the oracle through
    slot recycling: (n, lambda, m, generations, rows per lane) = C2 row length at lambda 4096; a short row (QW = 4) with two
    rows per lane; an odd shape (n = 48: 12 float4 columns over 16 warps, four of them idle; m = 11: a partial chunk)."""
    n, lam, m, gens, rl = shape
    monkeypatch.setenv("LMCMA_B200_SAMPLE_ROWS", "1")
    # V (k_update's FP32 sweep, not this kernel) carries 4e-5 of its scale at lambda = 4096: with mueff ~ 2300 the evolution
    # paths are long and nearly collinear with the stored directions, so each factor removes most of a row (DESIGN.md 5);
    # the sampled candidates X, the state the sampler produces, stay at 1e-6
    _teacher_forced(po, n, lam, m, gens, seed=31, sigma=0.5, tol_v=1e-4)


def test_rows_sampler_streams_pairs_that_do_not_fit(po, monkeypatch):
    """m = 120 pairs of n = 400 (192 KB) do not fit next to the partial-sum and coefficient buffers: both passes stream the
    chunks through a ring of stages.  The state with all 120 slots live comes from a cheap small-population run of the
    oracle; the device samples lambda = 4096 offspring from it with injected deviates."""
    monkeypatch.setenv("LMCMA_B200_SAMPLE_ROWS", "1")
    n, lam, m = 400, 4096, 120
    small = po.OracleLMCMA(n, x0=np.full(n, 0.5), lam=16, m=m, sigma=0.4, seed=1)
    for g in range(m + 9):
        small.tell_all(weighted_sphere_np(small.array("X")))
    st = small.state()
    assert st["live"] == m
    rng = np.random.default_rng(4)
    Z = rng.standard_normal((lam, n)).astype(np.float32)
    dev = L.Optimizer(n, x0=np.full(n, 0.5), lam=lam, m=m, sigma0=0.4, rng="inject")
    dev.inject_z(Z)
    dev.load_state(dict(st, prev_fit=np.zeros(lam)))
    dev.resample()
    ora = po.OracleLMCMA(n, x0=np.full(n, 0.5), lam=lam, m=m, sigma=0.4)
    ora.load_state(st, np.zeros(lam), Z.astype(np.float64))
    Xo, Xd = ora.array("X"), dev.get("X")[0]
    assert float(np.abs(Xd - Xo).max()) / max(1.0, float(np.abs(Xo).max())) < 2e-5


def weighted_sphere_np(X):
    X = np.atleast_2d(X)
    return np.sum((1.0 + np.arange(X.shape[1])) * X * X, axis=1)


def test_bench_dumps_the_last_timed_generation(tmp_path):
    """bench.py --dump-outputs DIR: after the timed steps, the arrays of the last timed generation land in DIR as float32 /
    float64 .npy files, they are the state the JSON line of the same run reports after its timed region, and a second
    run with the same arguments writes the same bits (what makes the files comparable from build to build)."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

    def run(out):
        r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--gpus", "1", "--steps", "3", "--warmup", "1",
                            "--skip", "c3,c4,cpu", "--dump-outputs", str(out)], capture_output=True, text=True, timeout=900)
        assert r.returncode == 0, r.stderr[-2000:]
        j = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
        return j, {p[:-len(".npy")]: np.load(out / p) for p in os.listdir(out)}

    j, d = run(tmp_path / "a")
    assert j["steps"] == 3
    assert sorted(d) == ["X", "best_f", "best_x", "fit", "ncoll", "sigma", "xmean"]
    assert all(a.dtype in (np.float32, np.float64) for a in d.values())
    assert d["X"].shape == (1, 1024, 400) and d["fit"].shape == (1, 1024) and d["best_x"].shape == d["xmean"].shape == (1, 400)
    assert d["sigma"][0] == j["config"]["sigma_in_timed_region"][1]
    assert d["ncoll"].min() == j["config"]["min_collisions_in_last_population"]
    assert np.isfinite(d["fit"]).all() and np.isfinite(d["X"]).all()
    _, d2 = run(tmp_path / "b")
    assert sorted(d2) == sorted(d)
    for name in d:
        assert d2[name].dtype == d[name].dtype and np.array_equal(d2[name], d[name]), name
