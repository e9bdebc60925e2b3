"""Restarting chosen instances of a live batch in place (reset_instances, reset_instances_dev).  Every comparison is bitwise:
a reset instance against a twin handle created at the reset's start and end points (its deviate stream moved to epoch 1
by hand), the instances a reset leaves alone against a handle that was never reset, a captured device loop against an
uncaptured host loop.

Whether a handle got the overlapped generation depends on a co-scheduling probe that a busy card can fail, so it is read
from launch(), never assumed."""
import numpy as np
import pytest

import lmcma_path_planner_b200 as L
from lmcma_path_planner_b200 import _capi as K
from lmcma_path_planner_b200 import maps
from conftest import weighted_sphere
from test_gpu_launch_graphs import GENERATION_CASES, W, LAM, M, _smooth_covariance, _tail_kernels, launches

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

STATE = ("xmean", "sigma", "s", "best_f", "X", "V", "P", "pc", "fit", "t", "vec", "Nj", "Lj", "counteval", "itr", "live",
         "epoch")
ALL_STATE = STATE + ("fit_sorted", "prev_fit", "arindex", "rank", "ncoll", "nsamp")
GENERATION_AND_BATCH = dict(GENERATION_CASES, batch8=dict(batch=8))
# the cost's launch shape is chosen from instance 0's end points at attach_cost: pinned, so that a reset of instance 0 to
# other end points and a twin attached with those end points launch k_cost alike
PINNED_COST = {"LMCMA_B200_COST_TPT": "128", "LMCMA_B200_COST_CB": "256"}


@pytest.fixture(scope="module")
def problem():
    dist, start, goal = maps.config2_map(size=1024, n_rects=128, seed=42, clamp=64.0)
    lo, hi = maps.box_bounds((1024, 1024), W)
    new_start, new_goal = (start[0], goal[1]), (goal[0], start[1])           # the other diagonal
    return dict(dist=dist, start=start, goal=goal, lo=lo, hi=hi, x0=maps.straight_line(start, goal, W),
                new_start=new_start, new_goal=new_goal, new_x0=maps.straight_line(new_start, new_goal, W),
                cmap=L.CostMap(dist, "f32"))


def _handle(p, monkeypatch, lam=LAM, env=None, covariance=None, seed=1, batch=1, x0=None, starts=None, goals=None):
    for k, v in (env or {}).items():
        monkeypatch.setenv(k, v)
    dev = L.Optimizer(2 * W, x0=p["x0"] if x0 is None else x0, lam=lam, m=M, batch=batch, lo=p["lo"], hi=p["hi"],
                      sigma0=16.0, seed=seed, covariance=covariance)
    for k in env or {}:
        monkeypatch.delenv(k)
    dev.attach_cost(p["cmap"], [p["start"]] if starts is None else starts, [p["goal"]] if goals is None else goals, W,
                    L.LONGSAFE, 1e4)
    return dev


def _same_rows(a, b, rows, tag="", names=STATE):
    for k in names:
        assert np.array_equal(a.get(k)[rows], b.get(k)[rows]), (tag, k)
    xa, fa = a.best()
    xb, fb = b.best()
    assert np.array_equal(xa[rows], xb[rows]), (tag, "best_x")
    assert np.array_equal(fa[rows], fb[rows]), (tag, "best_f")


def _snapshot(h, names=ALL_STATE):
    out = {k: h.get(k) for k in names}
    out["best() x"], out["best() f"] = h.best()
    return out


def _unchanged(h, before, tag=""):
    after = _snapshot(h, [k for k in before if not k.startswith("best()")])
    for k, v in before.items():
        assert np.array_equal(after[k], v, equal_nan=True), (tag, k)


def _sphere(X):
    """conftest.weighted_sphere as a torch expression on the device"""
    w = 1.0 + torch.arange(X.shape[-1], device=X.device, dtype=torch.float32)
    return (w * X * X).sum(-1)


def _case(name):
    c = dict(GENERATION_AND_BATCH[name])
    cov = _smooth_covariance() if c.pop("covariance", False) else None
    return c, cov


@pytest.mark.parametrize("case", list(GENERATION_AND_BATCH))
def test_a_reset_instance_is_a_fresh_instance(problem, monkeypatch, case):
    """50 generations (past slot recycling at m = 40), a reset to a new start, step size and end points, 60 more: the reset
    instances equal a twin created there, right after the reset and 60 generations later.  In the batch (slots 2 and 5
    reset) the other instances equal a handle that was never reset."""
    p = problem
    c, cov = _case(case)
    B = c.get("batch", 1)
    rows = [2, 5] if B > 1 else [0]
    if B == 1:
        c["env"] = dict(c.get("env", {}), **PINNED_COST)
    sigma_new = 8.0
    dev = _handle(p, monkeypatch, covariance=cov, **c)
    dev.run(50)
    dev.reset_instances(rows, p["new_x0"], sigma_new, starts=[p["new_start"]], goals=[p["new_goal"]])

    x0 = np.repeat(p["x0"][None], B, 0)
    x0[rows] = p["new_x0"]
    starts = np.repeat(np.asarray(p["start"], np.float32)[None], B, 0)
    goals = np.repeat(np.asarray(p["goal"], np.float32)[None], B, 0)
    starts[rows], goals[rows] = p["new_start"], p["new_goal"]
    twin = _handle(p, monkeypatch, covariance=cov, x0=x0, starts=starts, goals=goals, **c)
    sigma = twin.get("sigma")
    sigma[rows] = sigma_new
    twin.set("sigma", sigma)
    twin.set("epoch", 1)
    twin.resample()
    _same_rows(dev, twin, rows, (case, "after the reset"))
    assert np.all(dev.get("epoch")[rows] == 1)

    dev.run(60)
    twin.run(60)
    _same_rows(dev, twin, rows, (case, "60 generations later"))
    if B > 1:
        kept = [b for b in range(B) if b not in rows]
        plain = _handle(p, monkeypatch, covariance=cov, **c)
        plain.run(110)
        _same_rows(dev, plain, kept, (case, "untouched instances"))
        assert np.all(dev.get("epoch")[kept] == 0)
        plain.close()
    dev.close()
    twin.close()


def test_each_reset_draws_a_fresh_stream(problem):
    """Two resets to the same start and step size draw different populations (epoch 1, then 2); epoch 0 and resample()
    after a reset to the creation start and step size give back the created handle's first population, bit for bit."""
    n, lam, B = 40, 32, 4
    x0 = np.linspace(0.0, 1.0, n)
    h = L.Optimizer(n, x0=x0, lam=lam, batch=B, sigma0=0.5, seed=2)
    first = h.get("X")
    for _ in range(5):
        h.tell_all(weighted_sphere(h.ask_all().reshape(-1, n)).reshape(B, lam))
    h.reset_instances(np.arange(B), x0, 0.5)
    one = h.get("X")
    assert np.all(h.get("epoch") == 1) and np.all(h.get("itr") == 0)
    h.reset_instances(np.arange(B), x0, 0.5)
    two = h.get("X")
    assert np.all(h.get("epoch") == 2)
    for b in range(B):
        assert not np.array_equal(one[b], two[b]), b
        assert not np.array_equal(one[b], first[b]), b
    h.set("epoch", 0)
    h.resample()
    assert np.array_equal(h.get("X"), first)
    h.close()


def _flags(F):
    """a device criterion with no meaning but a mix of flags: two low bits of each instance's best fitness this generation"""
    return ((F.min(dim=1).values.view(torch.int32) & 3) == 0).to(torch.int32)


def test_captured_reset_loop_equals_the_host_loop(problem, monkeypatch):
    """k = 4 generations of [torch cost -> tell_all_dev -> flags from F on the device -> reset_instances_dev] captured in
    torch.cuda.graph and replayed 3 times equal an uncaptured twin that copies the flags to the host every generation and
    calls reset_instances.  The harvested best_x / best_f of each reset equal the twin's best just before its reset, and
    rows not reset are not written."""
    p = problem
    B, k, replays = 8, 4, 3
    n = 2 * W
    x0_np = np.stack([p["x0"] + 3.0 * b for b in range(B)])
    sig_np = 4.0 + np.arange(B, dtype=np.float64)

    twin = _handle(p, monkeypatch, seed=11, batch=B)
    s2 = torch.cuda.Stream()
    twin.set_stream(s2.cuda_stream)
    X2, F2 = twin.device_tensors()
    records = []
    for _ in range(k * replays):
        with torch.cuda.stream(s2):
            F2.copy_(_sphere(X2))
        twin.tell_all_dev()
        with torch.cuda.stream(s2):
            fl = _flags(F2).cpu().numpy()
        bx, _ = twin.best()
        bf = twin.get("best_f")
        idx = np.nonzero(fl)[0]
        if len(idx):
            twin.reset_instances(idx, x0_np[idx], sig_np[idx])
        records.append((fl != 0, bx, bf))
    assert sum(int(r[0].sum()) for r in records) > 0

    dev = _handle(p, monkeypatch, seed=11, batch=B)
    s = torch.cuda.Stream()
    dev.set_stream(s.cuda_stream)
    X, F = dev.device_tensors()
    x0_t = torch.from_numpy(x0_np).cuda()
    sig_t = torch.from_numpy(sig_np).cuda()
    bx_out = [torch.empty((B, n), dtype=torch.float32, device="cuda") for _ in range(k)]
    bf_out = [torch.empty(B, dtype=torch.float64, device="cuda") for _ in range(k)]
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    before = launches()
    with torch.cuda.graph(graph, stream=s):
        for j in range(k):
            F.copy_(_sphere(X))
            dev.tell_all_dev()
            dev.reset_instances_dev(_flags(F), x0_t, sig_t, None, bx_out[j], bf_out[j])
    assert launches() == before
    torch.cuda.synchronize()
    for r in range(replays):
        for j in range(k):
            bx_out[j].fill_(float("nan"))
            bf_out[j].fill_(float("nan"))
        torch.cuda.synchronize()
        graph.replay()
        torch.cuda.synchronize()
        for j in range(k):
            rows, bx, bf = records[r * k + j]
            got_x, got_f = bx_out[j].cpu().numpy(), bf_out[j].cpu().numpy()
            assert np.array_equal(got_x[rows], bx[rows]), (r, j)
            assert np.array_equal(got_f[rows], bf[rows]), (r, j)
            assert np.isnan(got_x[~rows]).all() and np.isnan(got_f[~rows]).all(), (r, j)
    _same_rows(dev, twin, slice(None), "captured")
    del graph
    dev.close()
    twin.close()


@pytest.mark.parametrize("case", list(GENERATION_AND_BATCH))
def test_all_zero_flags_change_nothing(problem, monkeypatch, case):
    """reset_instances_dev with no instance flagged leaves every state array as it was, the population included, and
    launches k_reset and the sampler's kernels only."""
    p = problem
    c, cov = _case(case)
    dev = _handle(p, monkeypatch, covariance=cov, **c)
    dev.run(45)
    s = torch.cuda.Stream()
    dev.set_stream(s.cuda_stream)
    before = _snapshot(dev)
    flags = torch.zeros(dev.batch, dtype=torch.int32, device="cuda")
    x0 = torch.zeros((dev.batch, dev.n), dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    count = launches()
    dev.reset_instances_dev(flags, x0)
    assert launches() - count == 1 + 1 + (2 if cov is not None else 0)
    s.synchronize()
    _unchanged(dev, before, case)
    dev.close()


@pytest.mark.parametrize("case", list(GENERATION_CASES))
def test_a_reset_keeps_the_graphs(problem, monkeypatch, case):
    """After run(1) has built the graphs, a reset and run(1) add the reset's kernels and one generation's: nothing is
    captured again."""
    p = problem
    c, cov = _case(case)
    c["env"] = dict(c.get("env", {}), **PINNED_COST)
    dev = _handle(p, monkeypatch, covariance=cov, **c)
    dev.run(1)
    l = dev.launch()
    prior = cov is not None
    per_generation = 1 + l["overlap"] + _tail_kernels(l, prior)
    before = launches()
    dev.reset_instances([0], p["new_x0"], 4.0, starts=[p["new_start"]], goals=[p["new_goal"]])
    dev.run(1)
    assert launches() - before == 1 + 1 + (2 if prior else 0) + per_generation, (case, l)
    dev.close()


def _host_f(X):
    return weighted_sphere(X.reshape(-1, X.shape[-1])).astype(np.float32).reshape(X.shape[0], X.shape[1])


def test_tell_reset_tell_with_the_host_mirror(problem, monkeypatch):
    """With ask_all_view on, tell_all's graphs end with the speculative pass of the next update; a reset in between makes
    the next tell take the whole update.  Equal to a twin without the host mirror, and the mirror shows the new
    population."""
    p = problem
    dev = _handle(p, monkeypatch, seed=13)
    twin = _handle(p, monkeypatch, seed=13)
    for g in range(8):
        if g == 4:
            for h in (dev, twin):
                h.reset_instances([0], p["new_x0"], 6.0)
            assert np.array_equal(dev.ask_all_view(), twin.ask_all())
        dev.tell_all(_host_f(np.array(dev.ask_all_view())))
        twin.tell_all(_host_f(twin.ask_all()))
    _same_rows(dev, twin, slice(None), "host mirror")
    dev.close()
    twin.close()


def test_a_reset_drops_a_half_told_generation(problem):
    """Half a generation of ask_one / tell_one, a reset, then a whole generation of ask_one / tell_one computes what a twin
    that skipped the half generation computes."""
    Ws, lam, m = 20, 16, 8
    lo, hi = maps.box_bounds((1024, 1024), Ws)
    hs = []
    for _ in range(2):
        h = L.Optimizer(2 * Ws, x0=maps.straight_line(problem["start"], problem["goal"], Ws), lam=lam, m=m, lo=lo, hi=hi,
                        sigma0=16.0, seed=5)
        h.attach_cost(problem["cmap"], [problem["start"]], [problem["goal"]], Ws, L.LONGSAFE, 1e4)
        hs.append(h)
    dev, twin = hs
    x_new = maps.straight_line(problem["new_start"], problem["new_goal"], Ws)
    for _ in range(lam // 2):
        dev.tell_one(weighted_sphere(dev.ask_one())[0])
    for h in (dev, twin):
        h.reset_instances([0], x_new, 8.0)
        for _ in range(lam):
            h.tell_one(weighted_sphere(h.ask_one())[0])
    _same_rows(dev, twin, slice(None), "half told")
    dev.close()
    twin.close()


def _lib_reset(h, count, idx, x0, sigma0=None, ends=None):
    return K.lib().lmcma_b200_reset_instances(h._h, count, None if idx is None else K.iptr(idx),
                                              None if x0 is None else K.dptr(x0), None if sigma0 is None else K.dptr(sigma0),
                                              ends)


def test_refusals_change_nothing(problem):
    """Every refusal returns its code and leaves every getter's output as it was; count == 0 launches nothing."""
    n, lam, B = 40, 32, 4
    x0 = np.linspace(0.0, 1.0, n)
    h = L.Optimizer(n, x0=x0, lam=lam, batch=B, seed=2)
    h.tell_all(_host_f(h.ask_all()))
    s = torch.cuda.Stream()
    h.set_stream(s.cuda_stream)
    before = _snapshot(h)
    row = K.f64c(x0[None])
    two = K.f64c(np.stack([x0, x0]))
    arg_cases = {
        "out of range": (1, np.array([B], np.int32), row, None),
        "negative": (1, np.array([-1], np.int32), row, None),
        "repeated": (2, np.array([1, 1], np.int32), two, None),
        "null x0": (1, np.array([0], np.int32), None, None),
        "null idx": (1, None, row, None),
        "sigma0 zero": (1, np.array([0], np.int32), row, np.array([0.0])),
        "sigma0 negative": (1, np.array([0], np.int32), row, np.array([-1.0])),
        "sigma0 inf": (1, np.array([0], np.int32), row, np.array([np.inf])),
        "sigma0 nan": (1, np.array([0], np.int32), row, np.array([np.nan])),
        "x0 nan": (1, np.array([0], np.int32), K.f64c(np.where(np.arange(n) == 3, np.nan, x0)[None]), None),
        "x0 inf": (1, np.array([0], np.int32), K.f64c(np.where(np.arange(n) == 7, -np.inf, x0)[None]), None),
        "count negative": (-1, np.array([0], np.int32), row, None),
    }
    for name, (count, idx, xs, sg) in arg_cases.items():
        count0 = launches()
        assert _lib_reset(h, count, idx, xs, sg) == K.ERR_ARG, name
        assert launches() == count0, name
    ends = (K.Endpoints * 1)()
    assert _lib_reset(h, 1, np.array([0], np.int32), row, None, ends) == K.ERR_STATE   # no cost attached
    count0 = launches()
    assert _lib_reset(h, 0, None, None) == K.OK
    assert launches() == count0
    flags = torch.ones(B, dtype=torch.int32, device="cuda")
    xd = torch.zeros((B, n), dtype=torch.float64, device="cuda")
    ed = torch.zeros((B, 6), dtype=torch.float32, device="cuda")
    lib = K.lib()
    assert lib.lmcma_b200_reset_instances_dev(h._h, None, xd.data_ptr(), None, None, None, None) == K.ERR_ARG
    assert lib.lmcma_b200_reset_instances_dev(h._h, flags.data_ptr(), None, None, None, None, None) == K.ERR_ARG
    assert lib.lmcma_b200_reset_instances_dev(h._h, flags.data_ptr(), xd.data_ptr(), None, ed.data_ptr(), None, None) == K.ERR_STATE
    torch.cuda.synchronize()
    _unchanged(h, before, "philox")
    h.close()

    others = {
        "hansen": L.Optimizer(n, x0=x0, lam=lam, rng="hansen", seed=2),
        "inject": L.Optimizer(n, x0=x0, lam=lam, rng="inject", seed=2),
        "split": L.Optimizer(n, x0=x0, lam=lam, pop_offset=0, pop_count=lam // 2, seed=2),
    }
    others["inject"].inject_z(np.random.default_rng(0).standard_normal((1, lam, n)).astype(np.float32))
    for name, o in others.items():
        st = torch.cuda.Stream()
        o.set_stream(st.cuda_stream)
        snap = _snapshot(o)
        assert _lib_reset(o, 1, np.array([0], np.int32), row) == K.ERR_STATE, name
        f1 = torch.ones(1, dtype=torch.int32, device="cuda")
        x1 = torch.zeros((1, n), dtype=torch.float64, device="cuda")
        assert lib.lmcma_b200_reset_instances_dev(o._h, f1.data_ptr(), x1.data_ptr(), None, None, None, None) == K.ERR_STATE, name
        torch.cuda.synchronize()
        _unchanged(o, snap, name)
        o.close()


def test_python_checks_of_the_device_reset(problem):
    """Optimizer.reset_instances_dev refuses the handle's own stream (ERR_STATE) and tensors of the wrong dtype, shape or
    contiguity (ValueError) before anything reaches the library."""
    n, lam, B = 40, 32, 4
    h = L.Optimizer(n, x0=np.zeros(n), lam=lam, batch=B, seed=2)
    flags = torch.zeros(B, dtype=torch.int32, device="cuda")
    x0 = torch.zeros((B, n), dtype=torch.float64, device="cuda")
    with pytest.raises(K.LmcmaError) as e:
        h.reset_instances_dev(flags, x0)
    assert e.value.code == K.ERR_STATE
    s = torch.cuda.Stream()
    h.set_stream(s.cuda_stream)
    count = launches()
    for bad in (dict(flags=flags.to(torch.int64)), dict(x0=x0.float()), dict(x0=x0[:, :n - 1]),
                dict(x0=torch.zeros((n, B), dtype=torch.float64, device="cuda").t()), dict(flags=flags.cpu()),
                dict(sigma0=torch.ones(B + 1, dtype=torch.float64, device="cuda")),
                dict(ends=torch.zeros((B, 6), dtype=torch.float64, device="cuda"))):
        args = dict(flags=flags, x0=x0)
        args.update(bad)
        with pytest.raises(ValueError):
            h.reset_instances_dev(**args)
    assert launches() == count
    h.close()
