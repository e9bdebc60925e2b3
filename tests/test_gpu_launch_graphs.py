"""The CUDA graphs of the fused generation and of tell_all, seen from outside: what a replay adds to
lmcma_b200_launch_count(), that re-attaching a cost map rebuilds the fused graph, and that moving a handle to another
stream between runs changes no bit.

The expected launch counts are derived from each handle's launch() fields and the kernels a generation is made of:
k_cost, k_rank, k_update and a sampler, plus k_gate when the generation is overlapped, k_rank_tiles when the fitness
tiles are sorted first, k_gram + k_coef + k_combine with the Gram-matrix update, and k_gauss + k_prior with a covariance
prior.  Whether a handle got the overlapped generation depends on a co-scheduling probe that a busy card can fail, so it
is read from launch(), never assumed."""
import numpy as np
import pytest

import lmcma_path_planner_b200 as L
from lmcma_path_planner_b200 import _capi as K
from lmcma_path_planner_b200 import maps

pytestmark = pytest.mark.gpu

W, LAM, M = 200, 1024, 40           # the C2 shape: n = 2 W = 400


def launches():
    return K.lib().lmcma_b200_launch_count()


@pytest.fixture(scope="module")
def problem():
    dist, start, goal = maps.config2_map(size=1024, n_rects=128, seed=42, clamp=64.0)
    lo, hi = maps.box_bounds((1024, 1024), W)
    return dict(dist=dist, start=start, goal=goal, lo=lo, hi=hi, x0=maps.straight_line(start, goal, W),
                cmap=L.CostMap(dist, "f32"))


def _handle(p, monkeypatch, lam=LAM, env=None, covariance=None, seed=1):
    for k, v in (env or {}).items():
        monkeypatch.setenv(k, v)
    dev = L.Optimizer(2 * W, x0=p["x0"], lam=lam, m=M, lo=p["lo"], hi=p["hi"], sigma0=16.0, seed=seed, covariance=covariance)
    for k in env or {}:
        monkeypatch.delenv(k)
    dev.attach_cost(p["cmap"], [p["start"]], [p["goal"]], W, L.LONGSAFE, 1e4)
    return dev


def _tail_kernels(l, prior):
    """Kernels of rank + update + sample."""
    return (3 + l["rank_tile_sorted"] + (3 if l["upd_gram"] else 0) + (2 if prior else 0))


def _smooth_covariance():
    i = np.arange(W)
    block = np.exp(-np.abs(i[:, None] - i[None, :]) / 8.0)      # SPD (exponential kernel), one block per dimension
    return np.kron(np.eye(2), block)


GENERATION_CASES = {
    "c2": dict(),
    "c2-linear": dict(env={"LMCMA_B200_OVERLAP": "0"}),
    "lambda8192": dict(lam=8192),
    "gram": dict(env={"LMCMA_B200_UPDATE_GRAM": "1"}),
    "prior": dict(covariance=True),
}


@pytest.mark.parametrize("case", list(GENERATION_CASES))
def test_fused_run_counts_the_kernels_of_each_generation(problem, monkeypatch, case):
    """run(3) replays the one-generation graph three times, run(16) the eight-generation graph twice: either way each
    generation adds the kernels it is made of."""
    c = dict(GENERATION_CASES[case])
    prior = c.pop("covariance", False)
    dev = _handle(problem, monkeypatch, covariance=_smooth_covariance() if prior else None, **c)
    dev.run(1)                                                   # builds the graphs (the overlapped one may fall back)
    l = dev.launch()
    if case == "c2-linear":
        assert l["overlap"] == 0
    if case == "lambda8192":
        assert l["rank_tile_sorted"] == 1
    if case == "gram":
        assert l["upd_gram"] == 1
    per_generation = 1 + l["overlap"] + _tail_kernels(l, prior)   # k_cost, k_gate
    for gens in (3, 16):
        before = launches()
        dev.run(gens)
        assert launches() - before == gens * per_generation, (case, gens, l)
    dev.close()


@pytest.mark.parametrize("tell_overlap", ["1", "0"])
@pytest.mark.parametrize("view", [False, True])
def test_tell_all_counts_the_kernels_it_runs(problem, monkeypatch, tell_overlap, view):
    """tell_all of one query: through its graph (k_update, k_gate, k_rank, the sampler, and with the host mirror of
    ask_all_view the speculative k_update of the next generation) when the handle has the overlapped generation, else
    stream-ordered (k_rank, k_update, the sampler).  Three calls: the whole graph first, then the one that resumes from
    the speculative pass."""
    p = problem
    dev = _handle(p, monkeypatch, env={"LMCMA_B200_TELL_OVERLAP": tell_overlap})
    l = dev.launch()
    graph = l["overlap"] == 1 and tell_overlap == "1"
    expected = _tail_kernels(l, False) + (1 + int(view) if graph else 0)   # k_gate, speculative k_update
    for g in range(3):
        X = np.array(dev.ask_all_view()[0]) if view else dev.ask_all()[0]
        f = p["cmap"].evaluate(X, p["start"], p["goal"], W, L.LONGSAFE, 1e4)["f"]
        before = launches()
        dev.tell_all(f)
        assert launches() - before == expected, (g, graph, view, l)
    dev.close()


def test_reattaching_a_cost_rebuilds_the_fused_graph(problem, monkeypatch):
    """The fused graph holds the map it was captured with: after attach_cost with another map, the next generation's
    fitness is that of the new map, bit for bit what CostMap.evaluate gives on the same candidates."""
    p = problem
    dist_b, _, _ = maps.config2_map(size=1024, n_rects=128, seed=7, clamp=64.0)
    cmap_b = L.CostMap(dist_b, "f32")
    dev = _handle(p, monkeypatch)
    dev.run(2)
    dev.attach_cost(cmap_b, [p["start"]], [p["goal"]], W, L.LONGSAFE, 1e4)
    X = dev.get("X")[0]
    dev.run(1)
    fit = dev.get("fit")[0]
    want = cmap_b.evaluate(X, p["start"], p["goal"], W, L.LONGSAFE, 1e4)["f"]
    on_a = p["cmap"].evaluate(X, p["start"], p["goal"], W, L.LONGSAFE, 1e4)["f"]
    assert np.array_equal(fit, want)
    assert not np.array_equal(fit, on_a)
    dev.close()


def test_set_stream_between_runs_keeps_the_bits(problem, monkeypatch):
    """A handle moved to a torch stream between runs (its graphs are rebuilt for that stream) and back computes what a
    twin that stayed on its own stream computes."""
    import torch
    p = problem
    keys = ("X", "xmean", "sigma", "V", "P", "pc", "fit", "t", "vec", "Nj", "Lj")
    twin = _handle(p, monkeypatch, seed=9)
    twin.run(5)
    twin.run(12)
    twin.run(3)
    dev = _handle(p, monkeypatch, seed=9)
    dev.run(5)
    stream = torch.cuda.Stream()
    dev.set_stream(stream.cuda_stream)
    dev.run(12)
    dev.set_stream(None)
    dev.run(3)
    for k in keys:
        assert np.array_equal(dev.get(k), twin.get(k)), k
    assert np.array_equal(dev.best()[1], twin.best()[1])
    dev.close()
    twin.close()
