"""The covariance-prior sampling path (lmcma_b200_create_with_prior, k_gauss + k_prior in front of every sampler) against
the FP64 oracle, at every sampler build a prior handle can get.

With a prior every deviate vector z becomes L z before computeAz (L: lower Cholesky factor of the prior).  The oracle has
no prior, so it is fed z L^T in FP64 wherever it takes deviates (test_gpu_parity.prior_deviates), with L the same FP64
factor the library rounds to FP32.  A prior also changes which builds plan_launch picks: never the rows sampler, never
the progressive or overlapped generation.  Each case first asserts, through Optimizer.launch(), the build it is there
for; the coverage test at the end requires the cases to reach every narrow and wide sampler build.

Bars are those of _teacher_forced: integer state and ranks bit-exact, sigma 1e-12, X / mean / pc / V / P 2e-5 of their
scale, Nj / Lj 1e-4.  The equivalences (batch against single handles, split population, fused graphs against the
host-buffer protocol) are bit for bit."""
import collections
import ctypes as C

import numpy as np
import pytest

import lmcma_path_planner_b200 as L
from lmcma_path_planner_b200 import _capi as K
from lmcma_path_planner_b200 import maps
from conftest import weighted_sphere
from test_gpu_bench_shapes import _sampler_matches_oracle
from test_gpu_dispatch_variants import _warm_state
from test_gpu_parity import _teacher_forced, prior_deviates, prior_factor

pytestmark = pytest.mark.gpu


def smoothness(dims, W):
    """covariance(dims, W) of the reference: block-diagonal, one W x W block per dimension."""
    n = dims * W
    c = np.zeros(n * n)
    K.check(K.lib().lmcma_b200_covariance(dims, W, K.dptr(c)))
    return c.reshape(n, n)


def dense(n, length=50.0):
    """A dense SPD prior over all n coordinates: exp(-|i - j| / length)."""
    i = np.arange(n)
    return np.exp(-np.abs(i[:, None] - i[None, :]) / length)


Case = collections.namedtuple("Case", "n lam m batch prior expect where")
Case.__new__.__defaults__ = (None,)

# id -> (n, lambda, m, batch, prior, expected launch fields, test elsewhere that holds this shape against a reference)
CASES = {
    "golden-n20": Case(20, 0, 0, 1, ("smooth", 2, 10), dict(sampler="narrow", smp_nv=1),
                       where="test_gpu_parity.py::test_smoothness_prior_sampling_matches_the_reference"),
    # the reference's defaults; n = 201 / 603 / 2046 are 3-D paths whose rows end in padded columns (ns = 204 / 604 / 2048)
    "defaults-n201": Case(201, 0, 0, 1, ("smooth", 3, 67), dict(sampler="narrow", smp_nv=2)),
    "dense-n400": Case(400, 128, 40, 1, ("dense", 400), dict(sampler="narrow", smp_nv=4)),
    "defaults-n603": Case(603, 0, 0, 1, ("smooth", 3, 201), dict(sampler="narrow", smp_nv=8)),
    "defaults-n2046": Case(2046, 0, 0, 1, ("smooth", 3, 682), dict(sampler="narrow", smp_nv=16)),
    "gram-n1500": Case(1500, 32, 77, 1, ("smooth", 3, 500), dict(sampler="narrow", smp_nv=12, upd_gram=1)),
    "wide2-n400": Case(400, 512, 24, 1, ("smooth", 2, 200), dict(sampler="wide", smp_RBW=2, progressive=0, overlap=0)),
    "fused-n200": Case(200, 512, 24, 1, ("smooth", 2, 100), dict(sampler="wide", smp_RBW=2, progressive=0, overlap=0)),
    "c2-fused": Case(400, 1024, 40, 1, ("smooth", 2, 200), dict(sampler="wide", smp_RBW=4, overlap=0)),
    # shapes where the rows sampler runs without a prior
    "lam65536": Case(400, 65536, 40, 1, ("smooth", 2, 200), dict(sampler="wide", smp_RBW=4)),
    "c3-batch": Case(400, 64, 40, 320, ("smooth", 2, 200), dict(sampler="narrow", smp_nv=4)),
    # more than 65 535 x 64 population rows in one launch
    "rows-inject": Case(8, 16384, 8, 257, ("smooth", 2, 4), dict(sampler="narrow", smp_nv=1)),
    "rows-philox": Case(8, 65536, 8, 64, ("smooth", 2, 4), dict(sampler="narrow", smp_nv=1)),
    "split-n40": Case(40, 64, 12, 1, ("smooth", 2, 20), dict(sampler="narrow", smp_nv=1)),
}


def _prior(case_id):
    p = CASES[case_id].prior
    return smoothness(p[1], p[2]) if p[0] == "smooth" else dense(p[1])


def _open(case_id, **kw):
    """The handle of a table case, with its prior, its launch fields checked."""
    c = CASES[case_id]
    x0 = kw.pop("x0", np.full(c.n, 0.5))
    dev = L.Optimizer(c.n, x0=x0, lam=c.lam, m=c.m, batch=c.batch, covariance=kw.pop("covariance", _prior(case_id)), **kw)
    got = dev.launch()
    for k, v in c.expect.items():
        assert got[k] == v, (case_id, k, got)
    return dev


def _sampler_without_prior(case_id):
    c = CASES[case_id]
    dev = L.Optimizer(c.n, x0=np.full(c.n, 0.5), lam=c.lam, m=c.m, batch=c.batch, rng="inject")
    kind = dev.launch()["sampler"]
    dev.close()
    return kind


@pytest.fixture(scope="module")
def map1024():
    dist, start, goal = maps.config2_map(size=1024, n_rects=128, seed=42, clamp=64.0)
    return dict(dist=dist, start=start, goal=goal, cmap=L.CostMap(dist, "f32"))


def _planning(p, W):
    lo, hi = maps.box_bounds((1024, 1024), W)
    return lo, hi, maps.straight_line(p["start"], p["goal"], W)


# ------------------------------------------------------------------------------------------------
# 1. teacher-forced past the point where slots are recycled, the oracle fed z L^T
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", ["defaults-n201", "defaults-n603", "defaults-n2046"])
def test_reference_defaults_with_prior_teacher_forced(po, case):
    cov = _prior(case)
    dev = _open(case, rng="inject", covariance=cov)
    n, m = CASES[case].n, dev.m
    dev.close()
    _teacher_forced(po, n, 0, 0, m + 6, seed=n, covariance=cov)


def test_dense_prior_teacher_forced(po):
    """A prior that is not block-diagonal: every coordinate of L z depends on all earlier ones (the full lower triangle
    of k_prior's tiles is non-zero).  X, the mean and pc stay at 5e-7 of their scale.  V (k_update's FP32 sweep, not the
    prior's kernels) carries 3e-5 (NVIDIA B200, 1000 W): the candidates of so correlated a prior are smooth, so successive
    evolution paths are nearly collinear with the stored directions and each factor removes most of a row (DESIGN.md 5).
    The FP64 oracle shows the same conditioning by itself: rounding only its state and deviates to FP32 between
    generations moves its V by 5e-6 of its scale here, against 2e-7 at the same shape without a prior."""
    cov = _prior("dense-n400")
    _open("dense-n400", rng="inject", covariance=cov).close()
    _teacher_forced(po, 400, 128, 40, 50, seed=3, sigma=0.5, covariance=cov, tol_v=1e-4)


def test_gram_update_with_prior_from_a_warm_state(po):
    cov = _prior("gram-n1500")
    _open("gram-n1500", rng="inject", covariance=cov).close()
    _teacher_forced(po, 1500, 32, 77, 8, seed=77, warm=_warm_state(po, 1500, 77), covariance=cov)


def test_wide_sampler_two_rows_per_warp_with_prior(po):
    """lambda = 512: the wide sampler with RBW = 2; with a prior the progressive hand-over and the overlapped generation are
    off (asserted by _open), so the sampler reads the Zc that k_prior wrote before it."""
    cov = _prior("wide2-n400")
    _open("wide2-n400", rng="inject", covariance=cov).close()
    _teacher_forced(po, 400, 512, 24, 30, seed=24, sigma=0.5, covariance=cov)


# ------------------------------------------------------------------------------------------------
# 2. the fused graph with k_gauss + k_prior at the C2 shape
# ------------------------------------------------------------------------------------------------
def test_fused_c2_generation_with_prior_tracks_the_oracle(po, map1024):
    """n = 400, lambda = 1024, m = 40, device Philox deviates, 46 graph-replayed generations on a 1024^2 map: the oracle is
    fed the device's recorded deviates times L^T and its fitness, the device then continues from the oracle's exact state."""
    W, p = 200, map1024
    lo, hi, x0 = _planning(p, W)
    cov = _prior("c2-fused")
    L64 = prior_factor(cov)
    dev = _open("c2-fused", x0=x0, lo=lo, hi=hi, sigma0=32.0, seed=5, record_z=True, covariance=cov)
    dev.attach_cost(p["cmap"], [p["start"]], [p["goal"]], W, L.LONGSAFE, 1e4)
    n, lam, m = dev.n, dev.lam, dev.m
    ora = po.OracleLMCMA(n, x0=x0, lam=lam, m=m, lo=lo, hi=hi, sigma=32.0, seed=1, Z0=prior_deviates(dev.get("Z")[0], L64))
    worst = {}
    for g in range(46):
        Xd, Xo = dev.get("X")[0], ora.array("X")
        worst["X"] = max(worst.get("X", 0), float(np.abs(Xd - Xo).max()) / 1023.0)
        dev.run(1)
        ora.tell_all(dev.get("fit")[0].astype(np.float64), prior_deviates(dev.get("Z")[0], L64))
        so = ora.state()
        live = so["t"][:so["live"]]
        assert np.array_equal(dev.get("t")[0][:so["live"]], live), g
        assert np.array_equal(dev.get("vec")[0][live], so["vec"][live]), g
        assert np.array_equal(dev.get("arindex")[0], ora.int_array("arindex")), g
        assert int(dev.get("itr")[0]) == so["itr"]
        worst["sigma"] = max(worst.get("sigma", 0), abs(dev.get("sigma")[0] - so["sigma"]) / so["sigma"])
        worst["xmean"] = max(worst.get("xmean", 0), float(np.abs(dev.get("xmean")[0] - so["xmean"]).max()) / 1023.0)
        pcs = max(1e-6, float(np.abs(so["pc"]).max()))
        worst["pc"] = max(worst.get("pc", 0), float(np.abs(dev.get("pc")[0] - so["pc"]).max()) / pcs)
        Vd = dev.get("V")[0]
        for slot in live:
            vs = max(1e-6, float(np.abs(so["V"][slot]).max()))
            worst["V"] = max(worst.get("V", 0), float(np.abs(Vd[slot] - so["V"][slot]).max()) / vs)
        dev.load_state(so)
        dev.resample()                                             # same Philox rows (counter = itr), oracle's exact state
    assert so["live"] == m and so["itr"] > m
    assert worst["sigma"] < 1e-12, worst
    for k in ("X", "xmean", "pc", "V"):
        assert worst[k] < 2e-5, (k, worst)


# ------------------------------------------------------------------------------------------------
# 3. population rows past the grid's y / z limit of 65 535
# ------------------------------------------------------------------------------------------------
def test_population_of_65536_with_prior_matches_the_oracle(po):
    """lambda = 65 536 (the largest population a handle takes, C5's last restart) with device Philox deviates: k_gauss has
    one block row per population row.  From a warm state with all 40 pairs live, the sampled population against the
    oracle's sample() from the device's own state, for three generations.  Without a prior this shape runs the rows
    sampler; with one it is the wide sampler with four rows per warp."""
    assert _sampler_without_prior("lam65536") == "rows"
    n, lam, m = 400, 65536, 40
    cov = _prior("lam65536")
    L64 = prior_factor(cov)
    dev = _open("lam65536", sigma0=0.4, seed=9, record_z=True, covariance=cov)
    warm = _warm_state(po, n, m)
    dev.load_state(dict(warm, prev_fit=np.zeros(lam)))
    dev.resample()
    dev.set("prev_fit", np.sort(weighted_sphere(dev.get("X")[0]).astype(np.float32)))
    for g in range(3):
        assert _sampler_matches_oracle(po, dev, n, lam, m, None, None, (0,), L64) < 2e-5, g
        dev.tell_all(weighted_sphere(dev.get("X")[0]).astype(np.float32))
    assert int(dev.get("live")[0]) == m and int(dev.get("itr")[0]) == warm["itr"] + 3
    assert _sampler_matches_oracle(po, dev, n, lam, m, None, None, (0,), L64) < 2e-5


@pytest.mark.parametrize("case", ["rows-inject", "rows-philox"])
def test_more_than_4194240_population_rows_with_prior(po, case):
    """B x lambda rows past 65 535 x 64, the most k_prior's row tiles could once cover: 257 x 16 384 injected deviates, and
    64 x 65 536 device Philox deviates.  The first population is x0 + sigma L z on the first, a middle and the last
    instance; after one tell_all their mean, step size and next population match the oracle fed the same fitness."""
    c = CASES[case]
    n, lam, m, B = c.n, c.lam, c.m, c.batch
    rng = np.random.default_rng(B)
    cov = _prior(case)
    L64 = prior_factor(cov)
    x0 = rng.standard_normal((B, n))
    sigma0 = 0.7
    inject = case == "rows-inject"
    dev = _open(case, x0=x0, sigma0=sigma0, seed=4, rng="inject" if inject else "philox", record_z=True, covariance=cov)
    if inject:
        dev.inject_z(rng.standard_normal((B, lam, n)).astype(np.float32))
    Z0, X = dev.get("Z"), dev.get("X")
    picks = (0, B // 2, B - 1)
    for b in picks:
        want = x0[b] + sigma0 * prior_deviates(Z0[b], L64)       # no pairs yet, no bounds
        assert np.abs(X[b] - want).max() < 2e-5 * max(1.0, np.abs(want).max()), b
    f = weighted_sphere(X.reshape(-1, n)).astype(np.float32).reshape(B, lam)
    if inject:
        dev.inject_z(rng.standard_normal((B, lam, n)).astype(np.float32))
    dev.tell_all(f)
    Z1, X1 = dev.get("Z"), dev.get("X")
    xmean, sigma, arindex = dev.get("xmean"), dev.get("sigma"), dev.get("arindex")
    for b in picks:
        ora = po.OracleLMCMA(n, x0=x0[b], lam=lam, m=m, sigma=sigma0, seed=1, Z0=prior_deviates(Z0[b], L64))
        ora.tell_all(f[b].astype(np.float64), prior_deviates(Z1[b], L64))
        so = ora.state()
        assert np.array_equal(arindex[b], ora.int_array("arindex")), b
        assert abs(sigma[b] - so["sigma"]) <= 1e-12 * so["sigma"], b
        assert np.abs(xmean[b] - so["xmean"]).max() < 2e-5 * max(1.0, np.abs(so["xmean"]).max()), b
        Xo = ora.array("X")
        assert np.abs(X1[b] - Xo).max() < 2e-5 * max(1.0, np.abs(Xo).max()), b


# ------------------------------------------------------------------------------------------------
# 4. bit-for-bit equivalences
# ------------------------------------------------------------------------------------------------
def test_batched_queries_with_prior_equal_single_handles(po, map1024, monkeypatch):
    """The C3 per-query shape (n = 400, lambda = 64, m = 40, 320 queries), where the prior turns the rows sampler into the
    narrow one: instance b of the batch equals a single handle fed instance b's deviates, 12 fused generations."""
    monkeypatch.setenv("LMCMA_B200_COST_TPT", "64")            # same reduction tree of k_cost whatever the launch
    assert _sampler_without_prior("c3-batch") == "rows"
    W, p, B = 200, map1024, 320
    lo, hi = maps.box_bounds((1024, 1024), W)
    starts, goals = maps.random_queries(p["dist"], B, seed=7, min_sep=256)
    x0 = np.stack([maps.straight_line(s, g, W) for s, g in zip(starts, goals)])
    cov = _prior("c3-batch")
    picks = (0, 161, B - 1)
    batched = _open("c3-batch", x0=x0, lo=lo, hi=hi, sigma0=16.0, seed=11, record_z=True, covariance=cov)
    batched.attach_cost(p["cmap"], starts, goals, W, L.LONGSAFE, 1e4)
    zs = [batched.get("Z")[list(picks)]]
    for g in range(12):
        batched.run(1)
        zs.append(batched.get("Z")[list(picks)])
    monkeypatch.setenv("LMCMA_B200_UPDATE_WARPS", "16")
    for i, b in enumerate(picks):
        one = L.Optimizer(2 * W, x0=x0[b], lam=64, m=40, lo=lo, hi=hi, sigma0=16.0, rng="inject", covariance=cov)
        one.attach_cost(p["cmap"], [starts[b]], [goals[b]], W, L.LONGSAFE, 1e4)
        one.inject_z(zs[0][i])
        for g in range(12):
            one.inject_z(zs[g + 1][i])
            one.run(1)
        for k in ("X", "xmean", "sigma", "V", "pc", "fit"):
            assert np.array_equal(one.get(k)[0], batched.get(k)[b]), (b, k)
        one.close()


def test_split_population_with_prior(po, golden_maps):
    """Two handles owning lambda / 2 rows each (G = 2) on the bundled 100^2 map: their first population is the whole
    optimiser's, bit for bit (k_gauss keys a row by its global index, k_prior computes each element alike whichever tile
    holds it), and after every mg_update each part's population is the oracle's sample() from that part's own state."""
    import torch
    dist = po.edt_exact(golden_maps["problem1"])
    W, start, goal = 20, (99.0, 0.0), (0.0, 99.0)
    lo, hi = maps.box_bounds((100, 100), W)
    x0 = maps.straight_line(start, goal, W)
    cm = L.CostMap(dist, "f32")
    n, lam, m, G = 2 * W, 64, 12, 2
    pc = lam // G
    cov = _prior("split-n40")
    L64 = prior_factor(cov)
    whole = _open("split-n40", x0=x0, lo=lo, hi=hi, sigma0=5.0, seed=9, covariance=cov)
    parts = [L.Optimizer(n, x0=x0, lam=lam, m=m, lo=lo, hi=hi, sigma0=5.0, seed=9, pop_offset=r * pc, pop_count=pc,
                         record_z=True, covariance=cov) for r in range(G)]
    for r, p in enumerate(parts):
        assert p.launch()["sampler"] == "narrow"
        assert np.array_equal(p.get("X")[0], whole.get("X")[0][r * pc:(r + 1) * pc]), r
        p.attach_cost(cm, [start], [goal], W)
    whole.close()
    pf = parts[0].mg_payload_floats()
    f_all = torch.zeros(lam, dtype=torch.float32, device="cuda")
    pay_all = torch.zeros(G * pf, dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    for g in range(8):
        for r, p in enumerate(parts):
            p.mg_evaluate(f_all.data_ptr() + 4 * r * pc)
            p.sync()
        for r, p in enumerate(parts):
            p.mg_rank(f_all.data_ptr(), pay_all.data_ptr() + 4 * r * pf)
            p.sync()
        for p in parts:
            p.mg_update(pay_all.data_ptr(), G)
            p.sync()
        Z = np.concatenate([p.get("Z")[0] for p in parts])       # the whole population's deviates, by global row
        for r, p in enumerate(parts):
            st = {k: p.get(k)[0].astype(np.float64) for k in ("xmean", "pc", "V", "P", "Nj", "Lj")}
            st.update({k: p.get(k)[0].copy() for k in ("t", "vec")})
            st.update(itr=int(p.get("itr")[0]), live=int(p.get("live")[0]), sigma=float(p.get("sigma")[0]), s=float(p.get("s")[0]))
            ora = po.OracleLMCMA(n, x0=np.zeros(n), lam=lam, m=m, lo=lo, hi=hi, sigma=1.0)
            ora.load_state(st, np.zeros(lam), prior_deviates(Z, L64))
            Xo = ora.array("X")[r * pc:(r + 1) * pc]
            assert np.abs(p.get("X")[0] - Xo).max() < 2e-5 * max(1.0, np.abs(Xo).max()), (g, r)
        for k in ("xmean", "sigma", "V", "pc"):                    # replicas stay bit-identical
            assert np.array_equal(parts[0].get(k), parts[1].get(k)), (g, k)
    assert int(parts[0].get("itr")[0]) == 8


def test_fused_graphs_with_prior_equal_the_host_buffer_protocol(map1024, monkeypatch):
    """n = 200, lambda = 512, m = 24: 30 fused generations give the same bits with eight generations per CUDA graph and
    with one per graph, and the same bits as 30 rounds of ask_all -> cost_evaluate -> tell_all through host buffers."""
    W, p = 100, map1024
    lo, hi, x0 = _planning(p, W)
    cov = _prior("fused-n200")
    keys = ("X", "xmean", "V", "P", "pc", "sigma", "t", "vec", "Nj", "Lj", "fit")
    out = {}
    for unroll in ("8", "1"):
        monkeypatch.setenv("LMCMA_B200_GRAPH_UNROLL", unroll)
        dev = _open("fused-n200", x0=x0, lo=lo, hi=hi, sigma0=6.0, seed=3, covariance=cov)
        dev.attach_cost(p["cmap"], [p["start"]], [p["goal"]], W, L.LONGSAFE, 1e4)
        dev.run(30)
        out[unroll] = {k: dev.get(k).copy() for k in keys}
        out[unroll]["best"] = dev.best()
        dev.close()
    monkeypatch.delenv("LMCMA_B200_GRAPH_UNROLL")
    host = _open("fused-n200", x0=x0, lo=lo, hi=hi, sigma0=6.0, seed=3, covariance=cov)
    for g in range(30):
        r = p["cmap"].evaluate(host.ask_all()[0], p["start"], p["goal"], W, L.LONGSAFE, 1e4)
        host.tell_all(r["f"])
    assert int(host.get("live")[0]) == 24 and int(host.get("itr")[0]) == 30
    for k in keys:
        assert np.array_equal(out["8"][k], out["1"][k]), ("graph unroll", k)
        assert np.array_equal(out["8"][k], host.get(k)), ("host protocol", k)
    xb, fb = host.best()
    assert np.array_equal(out["8"]["best"][0], xb) and np.array_equal(out["8"]["best"][1], fb)


# ------------------------------------------------------------------------------------------------
# 5. coverage and refusal
# ------------------------------------------------------------------------------------------------
def test_every_sampler_build_of_a_prior_handle_is_reached():
    """The cases reach narrow NV = 1, 2, 4, 8, 12, 16 and wide RBW = 2, 4, every sampler build a prior handle can get; no
    prior handle runs the rows sampler (its k_sample_rows draws its own deviates and would skip L z)."""
    import importlib
    reached = set()
    for cid, c in CASES.items():
        dev = _open(cid, rng="inject")                            # no sample before inject_z: nothing runs on the device
        got = dev.launch()
        assert got["sampler"] != "rows", cid
        reached.add(("narrow", got["smp_nv"]) if got["sampler"] == "narrow" else ("wide", got["smp_RBW"]))
        dev.close()
        if c.where:                                                # the older test holding this shape still exists
            mod, name = c.where.split("::")
            assert hasattr(importlib.import_module(mod[:-3]), name), c.where
    want = {("narrow", v) for v in (1, 2, 4, 8, 12, 16)} | {("wide", 2), ("wide", 4)}
    assert reached == want, sorted(reached ^ want)


@pytest.mark.parametrize("kind", ["indefinite", "singular", "nan"])
def test_covariance_that_is_not_positive_definite_is_refused(kind):
    n = 12
    cov = smoothness(2, 6)
    if kind == "indefinite":
        cov[3, 3] = -cov[3, 3]
    elif kind == "singular":
        v = np.arange(1.0, n + 1)
        cov = np.outer(v, v)                                       # rank one
    else:
        cov[5, 5] = np.nan
    cfg = K.Config()
    cfg.n, cfg.lambda_, cfg.m, cfg.batch, cfg.sigma0, cfg.seed, cfg.rng = n, 0, 0, 1, 1.0, 1, K.RNG_PHILOX
    x0 = np.zeros(n)
    h = C.c_void_p()
    rc = K.lib().lmcma_b200_create_with_prior(C.byref(cfg), K.dptr(x0), None, None, K.dptr(np.ascontiguousarray(cov)), C.byref(h))
    assert rc == K.ERR_ARG and h.value is None, (kind, rc)
    assert b"positive definite" in K.lib().lmcma_b200_last_error()
    with pytest.raises(K.LmcmaError) as e:
        L.Optimizer(n, x0=x0, covariance=cov)
    assert e.value.code == K.ERR_ARG
