"""What a handle's host side keeps across entry points.  After anything that samples a new population (run, resample),
the one-at-a-time protocol (ask_one / tell_one) starts that population from its first row: a half-told generation is
dropped, never mixed with rows of the new one."""
import numpy as np
import pytest

import lmcma_path_planner_b200 as L
from lmcma_path_planner_b200 import maps
from conftest import weighted_sphere

pytestmark = pytest.mark.gpu

SHAPES = {"small": dict(W=20, lam=16, m=8), "c2": dict(W=200, lam=1024, m=40)}   # c2: the forked tell graph, if the card allows


@pytest.fixture(scope="module")
def problem():
    dist, start, goal = maps.config2_map(size=1024, n_rects=128, seed=42, clamp=64.0)
    return dict(start=start, goal=goal, cmap=L.CostMap(dist, "f32"))


def _handle(p, W, lam, m):
    lo, hi = maps.box_bounds((1024, 1024), W)
    dev = L.Optimizer(2 * W, x0=maps.straight_line(p["start"], p["goal"], W), lam=lam, m=m, lo=lo, hi=hi, sigma0=16.0, seed=5)
    dev.attach_cost(p["cmap"], [p["start"]], [p["goal"]], W, L.LONGSAFE, 1e4)
    return dev


def _ask_tell(dev, count):
    """count rounds of ask_one -> tell_one.  The weighted sphere: which objective does not matter, only that both
    handles are told the same."""
    for _ in range(count):
        dev.tell_one(weighted_sphere(dev.ask_one())[0])


def _run(dev):
    dev.run(1)


def _set_mean_and_resample(dev):
    dev.set("xmean", dev.get("xmean") + 0.5)
    dev.resample()


@pytest.mark.parametrize("new_population", [_run, _set_mean_and_resample], ids=["run", "set_resample"])
@pytest.mark.parametrize("shape", list(SHAPES))
def test_a_new_population_drops_a_half_told_generation(problem, shape, new_population):
    """Half a generation of ask_one / tell_one, a new population, then a whole generation of ask_one / tell_one computes
    what a twin that skipped the half generation computes."""
    s = SHAPES[shape]
    dev, twin = _handle(problem, **s), _handle(problem, **s)
    _ask_tell(dev, s["lam"] // 2)
    for h in (dev, twin):
        new_population(h)
        _ask_tell(h, s["lam"])
    for k in ("X", "xmean", "sigma", "V", "fit"):
        assert np.array_equal(dev.get(k), twin.get(k)), k
    xd, fd = dev.best()
    xt, ft = twin.best()
    assert np.array_equal(xd, xt) and np.array_equal(fd, ft)
    dev.close()
    twin.close()
