"""The device-resident batched protocol: device_buffers / device_tensors -> the caller's own cost on the GPU ->
tell_all_dev.  Every comparison is bitwise against a twin that takes another path to the same generations: the fused
run(G), host tell_all with the same fitness, an uncaptured loop for a loop captured in torch.cuda.graph, and a twin that
synchronised before each entry point called right after an unsynchronised tell_all_dev.

Whether a handle got the overlapped generation (and with it the forked tell graph) depends on a co-scheduling probe that
a busy card can fail, so it is read from launch(), never assumed."""
import numpy as np
import pytest

import lmcma_path_planner_b200 as L
from lmcma_path_planner_b200 import _capi as K
from lmcma_path_planner_b200 import maps
from test_gpu_launch_graphs import GENERATION_CASES, W, LAM, M, _smooth_covariance, _tail_kernels, launches

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

G = 60                               # past slot recycling at m = 40
STATE = ("xmean", "sigma", "X", "V", "P", "fit", "counteval", "pc", "t", "vec", "Nj", "Lj")


@pytest.fixture(scope="module")
def problem():
    dist, start, goal = maps.config2_map(size=1024, n_rects=128, seed=42, clamp=64.0)
    lo, hi = maps.box_bounds((1024, 1024), W)
    return dict(dist=dist, start=start, goal=goal, lo=lo, hi=hi, x0=maps.straight_line(start, goal, W),
                cmap=L.CostMap(dist, "f32"))


def _handle(p, monkeypatch, lam=LAM, env=None, covariance=None, seed=1, batch=1):
    for k, v in (env or {}).items():
        monkeypatch.setenv(k, v)
    dev = L.Optimizer(2 * W, x0=p["x0"], lam=lam, m=M, batch=batch, lo=p["lo"], hi=p["hi"], sigma0=16.0, seed=seed,
                      covariance=covariance)
    for k in env or {}:
        monkeypatch.delenv(k)
    dev.attach_cost(p["cmap"], [p["start"]], [p["goal"]], W, L.LONGSAFE, 1e4)
    return dev


def _same(a, b, tag=""):
    for k in STATE:
        assert np.array_equal(a.get(k), b.get(k)), (tag, k)
    xa, fa = a.best()
    xb, fb = b.best()
    assert np.array_equal(xa, xb), (tag, "best_x")
    assert np.array_equal(fa, fb), (tag, "best_f")


def _map_cost(p, dev, X, F, stream):
    """CostMap.evaluate_dev of every instance's rows of X into its row of F, on `stream`."""
    for b in range(dev.batch):
        p["cmap"].evaluate_dev(X[b].data_ptr(), dev.ld, dev.pop_count, F[b].data_ptr(), p["start"], p["goal"], W,
                               L.LONGSAFE, 1e4, stream=stream.cuda_stream)


def _sphere(X):
    """the weighted sphere of conftest.weighted_sphere, as a torch expression on the device"""
    w = 1.0 + torch.arange(X.shape[-1], device=X.device, dtype=torch.float32)
    return (w * X * X).sum(-1)


GENERATION_AND_BATCH = dict(GENERATION_CASES, batch8=dict(batch=8))


@pytest.mark.parametrize("case", list(GENERATION_AND_BATCH))
def test_device_loop_equals_the_fused_run(problem, monkeypatch, case):
    """G x (evaluate_dev from X_dev into f_dev on the handle's stream, tell_all_dev) computes what run(G) computes."""
    p = problem
    c = dict(GENERATION_AND_BATCH[case])
    cov = _smooth_covariance() if c.pop("covariance", False) else None
    twin = _handle(p, monkeypatch, covariance=cov, **c)
    twin.run(G)
    dev = _handle(p, monkeypatch, covariance=cov, **c)
    s = torch.cuda.Stream()
    dev.set_stream(s.cuda_stream)
    X, F = dev.device_tensors()
    assert X.shape == (dev.batch, dev.pop_count, dev.n) and F.shape == (dev.batch, dev.lam)
    assert X.stride() == (dev.pop_count * dev.ld, dev.ld, 1)
    for _ in range(G):
        _map_cost(p, dev, X, F, s)
        dev.tell_all_dev()
    s.synchronize()
    _same(dev, twin, case)
    assert torch.equal(X.cpu(), torch.from_numpy(twin.get("X")))
    dev.close()
    twin.close()


@pytest.mark.parametrize("env", [{}, {"LMCMA_B200_TELL_SPEC": "0"}, {"LMCMA_B200_TELL_OVERLAP": "0"}],
                         ids=["default", "tell_spec0", "tell_overlap0"])
def test_device_loop_equals_host_tell_all(problem, monkeypatch, env):
    """A torch cost on the device, fed to tell_all_dev, and the same values fed to a twin through host tell_all with the
    host mirror on (ask_all_view), so that by default its graphs end with the speculative pass and resume from it."""
    p = problem
    dev = _handle(p, monkeypatch, env=env, seed=3)
    twin = _handle(p, monkeypatch, env=env, seed=3)
    s = torch.cuda.Stream()
    dev.set_stream(s.cuda_stream)
    X, F = dev.device_tensors()
    twin.ask_all_view()                                          # the host mirror on: tell_all's graphs take the speculative pass
    for g in range(50):
        with torch.cuda.stream(s):
            F.copy_(_sphere(X))
            f = F.cpu().numpy()                                  # the values the device twin ranks (a synchronising copy)
        dev.tell_all_dev()
        twin.tell_all(f)
    s.synchronize()
    _same(dev, twin, env)
    dev.close()
    twin.close()


def test_captured_loop_equals_the_uncaptured_one(problem, monkeypatch):
    """k = 4 generations (torch cost + tell_all_dev) captured in torch.cuda.graph right after device_tensors() and replayed
    3 times equal 12 uncaptured generations: the Philox counter, like the rest of the state, advances across replays.
    Capture launches nothing and adds nothing to launch_count."""
    p = problem
    twin = _handle(p, monkeypatch, seed=5)
    s2 = torch.cuda.Stream()
    twin.set_stream(s2.cuda_stream)
    X2, F2 = twin.device_tensors()
    for _ in range(12):
        with torch.cuda.stream(s2):
            F2.copy_(_sphere(X2))
        twin.tell_all_dev()
    s2.synchronize()

    dev = _handle(p, monkeypatch, seed=5)
    s = torch.cuda.Stream()
    dev.set_stream(s.cuda_stream)
    X, F = dev.device_tensors()
    graph = torch.cuda.CUDAGraph()
    before = launches()
    with torch.cuda.graph(graph, stream=s):
        for _ in range(4):
            F.copy_(_sphere(X))
            dev.tell_all_dev()
    assert launches() == before
    torch.cuda.synchronize()
    for _ in range(3):
        graph.replay()
    torch.cuda.synchronize()
    _same(dev, twin)
    del graph
    dev.close()
    twin.close()


def test_tell_all_dev_returns_without_waiting(problem, monkeypatch):
    """Behind a long kernel on the handle's stream, tell_all_dev returns while the stream is still busy."""
    p = problem
    dev = _handle(p, monkeypatch)
    s = torch.cuda.Stream()
    dev.set_stream(s.cuda_stream)
    X, F = dev.device_tensors()
    _map_cost(p, dev, X, F, s)
    dev.tell_all_dev()                                           # builds the graphs the next call replays
    _map_cost(p, dev, X, F, s)
    with torch.cuda.stream(s):
        torch.cuda._sleep(int(2e9))
    dev.tell_all_dev()
    assert not s.query()
    s.synchronize()
    dev.close()


def _join_op(name, dev):
    if name == "get_V":
        return dev.get("V")
    if name == "set_sigma":
        dev.set("sigma", 3.0)
    elif name == "ask_all":
        return dev.ask_all()
    elif name == "best":
        return dev.best()
    elif name == "run":
        dev.run(1)
    return None


@pytest.mark.parametrize("op", ["get_V", "set_sigma", "ask_all", "best", "run"])
def test_entry_points_right_after_tell_all_dev(problem, monkeypatch, op):
    """Called right after tell_all_dev, before its generation has run, each entry point gives what it gives a twin that
    synchronised first, and the generations after it stay bit-identical."""
    p = problem
    dev = _handle(p, monkeypatch, seed=7)
    twin = _handle(p, monkeypatch, seed=7)
    streams = []
    for h in (dev, twin):
        streams.append(torch.cuda.Stream())
        h.set_stream(streams[-1].cuda_stream)
    views = [h.device_tensors() for h in (dev, twin)]
    for g in range(8):
        for h, (X, F), s in zip((dev, twin), views, streams):
            _map_cost(p, h, X, F, s)
            h.tell_all_dev()
        if g == 6:
            got = _join_op(op, dev)
            twin.sync()
            want = _join_op(op, twin)
            if isinstance(got, tuple):
                for a, b in zip(got, want):
                    assert np.array_equal(a, b), op
            elif got is not None:
                assert np.array_equal(got, want), op
    for s in streams:
        s.synchronize()
    _same(dev, twin, op)
    dev.close()
    twin.close()


def test_refusals_leave_the_state_alone(problem):
    """HANSEN, INJECT and a split-population handle: ERR_STATE; a null handle: ERR_ARG; a refused call changes nothing."""
    assert K.lib().lmcma_b200_tell_all_dev(None) == K.ERR_ARG
    n, lam = 40, 32
    x0 = np.linspace(0.0, 1.0, n)
    handles = {
        "hansen": L.Optimizer(n, x0=x0, lam=lam, rng="hansen", seed=2),
        "inject": L.Optimizer(n, x0=x0, lam=lam, rng="inject", seed=2),
        "split": L.Optimizer(n, x0=x0, lam=lam, pop_offset=0, pop_count=lam // 2, seed=2),
    }
    handles["inject"].inject_z(np.random.default_rng(0).standard_normal((1, lam, n)).astype(np.float32))
    streams = []
    for name, h in handles.items():
        streams.append(torch.cuda.Stream())
        h.set_stream(streams[-1].cuda_stream)                    # past the Python layer's own check: the library refuses
        before = {k: h.get(k) for k in ("xmean", "sigma", "X", "counteval", "itr")}
        with pytest.raises(K.LmcmaError) as e:
            h.tell_all_dev()
        assert e.value.code == K.ERR_STATE, name
        for k, v in before.items():
            assert np.array_equal(h.get(k), v), (name, k)
        h.close()


def test_a_tell_on_the_handles_own_stream_is_refused(problem, monkeypatch):
    """Optimizer.tell_all_dev refuses a handle on its own stream, including the one set_stream(0) selects when the cost
    runs on torch's default stream: that stream is not ordered with anything torch enqueues.  Nothing is launched."""
    p = problem
    dev = _handle(p, monkeypatch, seed=4)
    X, F = dev.device_tensors()
    assert torch.cuda.current_stream().cuda_stream == 0
    F.copy_(_sphere(X))
    torch.cuda.synchronize()
    before = {k: dev.get(k) for k in STATE}
    for stream in (None, torch.cuda.current_stream().cuda_stream):
        if stream is not None:
            dev.set_stream(stream)
        count = launches()
        with pytest.raises(K.LmcmaError) as e:
            dev.tell_all_dev()
        assert e.value.code == K.ERR_STATE
        assert launches() == count
    for k, v in before.items():
        assert np.array_equal(dev.get(k), v), k
    dev.close()


def test_calls_between_replays_of_a_captured_loop(problem, monkeypatch):
    """Replays of a caller's graph advance the state behind the library's back.  Between replays, ask_all_view and ask_one
    still return the current population, and a setter of V reaches the pair mirror the next replayed sampler reads: the
    same as an uncaptured twin that runs the same generations and the same calls."""
    p = problem
    twin = _handle(p, monkeypatch, seed=9)
    s2 = torch.cuda.Stream()
    twin.set_stream(s2.cuda_stream)
    X2, F2 = twin.device_tensors()

    def twin_generations(k):
        for _ in range(k):
            with torch.cuda.stream(s2):
                F2.copy_(_sphere(X2))
            twin.tell_all_dev()
        s2.synchronize()

    dev = _handle(p, monkeypatch, seed=9)
    s = torch.cuda.Stream()
    dev.set_stream(s.cuda_stream)
    X, F = dev.device_tensors()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=s):
        for _ in range(2):
            F.copy_(_sphere(X))
            dev.tell_all_dev()
    torch.cuda.synchronize()
    for r in range(3):
        graph.replay()
        torch.cuda.synchronize()
        twin_generations(2)
        assert np.array_equal(dev.ask_all_view(), twin.ask_all_view()), r
        assert np.array_equal(dev.ask_one(), twin.ask_one()), r
        if r == 1:
            V = (0.5 * twin.get("V")).astype(np.float32)
            dev.set("V", V)
            twin.set("V", V)
    _same(dev, twin)
    del graph
    dev.close()
    twin.close()


@pytest.mark.parametrize("env", [{}, {"LMCMA_B200_TELL_OVERLAP": "0"}], ids=["default", "tell_overlap0"])
def test_tell_all_dev_counts_the_kernels_it_runs(problem, monkeypatch, env):
    """Uncaptured: rank + update + sample, + k_gate through the forked graph; no speculative pass."""
    p = problem
    dev = _handle(p, monkeypatch, env=env)
    s = torch.cuda.Stream()
    dev.set_stream(s.cuda_stream)
    X, F = dev.device_tensors()
    l = dev.launch()
    graph = l["overlap"] == 1 and env.get("LMCMA_B200_TELL_OVERLAP") != "0"
    expected = _tail_kernels(l, False) + int(graph)
    for g in range(3):
        _map_cost(p, dev, X, F, s)
        before = launches()
        dev.tell_all_dev()
        assert launches() - before == expected, (g, graph, l)
    s.synchronize()
    dev.close()
