"""The device timeline of LMCMA_B200_DBG=1: globaltimer stamps of k_update, k_rank and the wide sampler in one buffer per
handle, printed and cleared by lmcma_b200_sync and profile_kernels.  The stamps must change no result and no launch
count, the printout must carry every section, and each stamp must land in a slot of its own."""
import re

import numpy as np
import pytest

import lmcma_path_planner_b200 as L
from lmcma_path_planner_b200 import _capi as K
from lmcma_path_planner_b200 import maps

pytestmark = pytest.mark.gpu

W, LAM, M = 200, 1024, 40           # the C2 shape: n = 2 W = 400
STATE = ("xmean", "sigma", "V", "P")


def launches():
    return K.lib().lmcma_b200_launch_count()


@pytest.fixture(scope="module")
def problem():
    dist, start, goal = maps.config2_map(size=1024, n_rects=128, seed=42, clamp=64.0)
    return dict(dist=dist, start=start, goal=goal, cmap=L.CostMap(dist, "f32"))


def _handle(p, monkeypatch, env, w=W, lam=LAM, m=M, seed=3):
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    lo, hi = maps.box_bounds((1024, 1024), w)
    dev = L.Optimizer(2 * w, x0=maps.straight_line(p["start"], p["goal"], w), lam=lam, m=m, lo=lo, hi=hi, sigma0=16.0,
                      seed=seed)
    for k in env:
        monkeypatch.delenv(k)
    dev.attach_cost(p["cmap"], [p["start"]], [p["goal"]], w, L.LONGSAFE, 1e4)
    return dev


def _timeline(text):
    """The last printed timeline: {section: {name: ns or None}}, and its series {name: [ns or None]}."""
    def value(v):
        return None if v == "-" else int(v)
    last = text[text.rindex("device timeline"):]
    sections, series, cur = {}, {}, {}
    for line in last.splitlines()[1:]:
        head, _, body = line.strip().partition(":")
        if not line.startswith("    "):                          # "  section: name=ns ..."
            sections[head] = cur = {k: value(v) for k, v in re.findall(r"(\w+)=(-|-?\d+)", body)}
        elif "=" in line:                                        # "    first_stale=.. live=..": values of the section above
            cur.update({k: value(v) for k, v in re.findall(r"(\w+)=(-|-?\d+)", line)})
        else:                                                    # "    series: ns ns - ..."
            series[head] = [value(v) for v in body.split()]
    return sections, series


def _same_state(a, b):
    for k in STATE:
        assert np.array_equal(a.get(k), b.get(k)), k
    for x, y in zip(a.best(), b.best()):
        assert np.array_equal(x, y)


def _tell_rounds(p, dev, rounds=10):
    for _ in range(rounds):
        X = np.array(dev.ask_all_view()[0])
        dev.tell_all(p["cmap"].evaluate(X, p["start"], p["goal"], W, L.LONGSAFE, 1e4)["f"])


@pytest.mark.parametrize("tell_overlap", ["1", "0"])
def test_the_timeline_changes_no_bit_and_no_launch_count(problem, monkeypatch, capfd, tell_overlap):
    """run(3) (the one-generation graph), run(16) (two replays of the eight-generation graph) and ten tell_all rounds with
    ask_all_view (the tell graph with its speculative pass, or stream-ordered with LMCMA_B200_TELL_OVERLAP=0): a handle
    with the timeline computes what its twin without it computes, with the same launches."""
    p = problem
    env = {"LMCMA_B200_TELL_OVERLAP": tell_overlap}
    dev = _handle(p, monkeypatch, dict(env, LMCMA_B200_DBG="1"))
    twin = _handle(p, monkeypatch, env)
    assert dev.launch() == twin.launch()
    steps = [("run3", lambda h: h.run(3)), ("run16", lambda h: h.run(16)),
             ("tell", lambda h: (_tell_rounds(p, h), h.sync()))]
    for name, step in steps:
        deltas = []
        for h in (dev, twin):
            before = launches()
            step(h)
            deltas.append(launches() - before)
        assert deltas[0] == deltas[1], (name, deltas)
        _same_state(dev, twin)
        out = capfd.readouterr().err
        sections, series = _timeline(out)
        assert {"k_update", "k_rank CTA 0", "k_sample_wide CTA 0"} <= set(sections), (name, out[-2000:])
        upd = sections["k_update"]
        assert upd["start"] is not None and upd["end"] is not None and upd["end"] > upd["start"], (name, upd)
        assert sections["k_rank CTA 0"]["start"] is not None, (name, sections)
        assert len(series["rows"]) == 40 and len(series["chain blocks"]) == 10, series
    dev.sync()                                                   # nothing ran since the last print: it was cleared
    sections, series = _timeline(capfd.readouterr().err)
    stamps = [v for s in sections.values() for k, v in s.items() if k not in ("first_stale", "live")]
    assert all(v is None for v in stamps + series["rows"] + series["chain blocks"] + series["chunks"]), (sections, series)
    dev.close()
    twin.close()


def test_profile_kernels_runs_the_generations_it_is_asked_for(problem, monkeypatch, capfd):
    """profile_kernels(g) with the timeline on advances the optimiser by exactly g generations and prints the timeline
    and the per-CTA timeline of k_cost.  LMCMA_B200_UPDATE_DBG, a retired name, is ignored: it used to add one more
    generation."""
    dev = _handle(problem, monkeypatch, {"LMCMA_B200_DBG": "1", "LMCMA_B200_UPDATE_DBG": "1"})
    dev.run(2)
    itr = int(dev.get("itr")[0])
    dev.profile_kernels(3)
    assert int(dev.get("itr")[0]) == itr + 3
    out = capfd.readouterr().err
    sections, _ = _timeline(out)
    assert sections["k_update"]["start"] is not None and sections["k_update"]["end"] is not None, sections
    assert "k_cost timeline" in out
    dev.close()


def test_chain_block_stamps_have_slots_of_their_own(problem, monkeypatch, capfd):
    """At m = 64 (the overlapped build with five rows per warp) the newest row's chain runs eight blocks of eight
    factors.  Each block's stamp lands in its own slot, none of them in the slot of "best-so-far copied", which the
    same thread stamps after the chain: the chain stamps rise block by block and end before that one."""
    dev = _handle(problem, monkeypatch, {"LMCMA_B200_DBG": "1"}, w=100, lam=512, m=64, seed=5)
    l = dev.launch()
    assert l["upd_rmax"] == 5, l
    if not l["overlap"]:
        pytest.skip("the co-scheduling probe ruled out the overlapped generation on this device")
    dev.run(70)                                                  # past m generations: every slot is live
    assert int(dev.get("live")[0]) == 64
    capfd.readouterr()
    dev.run(1)
    sections, series = _timeline(capfd.readouterr().err)
    upd = sections["k_update"]
    assert upd["live"] == 64, upd
    chain = series["chain blocks"]
    blocks = (64 - 1 + 7) // 8
    assert all(t is not None for t in chain[:blocks]) and all(t is None for t in chain[blocks:]), chain
    assert chain[:blocks] == sorted(chain[:blocks]), chain
    assert upd["best_copied"] is not None and upd["best_copied"] >= chain[blocks - 1], (upd, chain)
    dev.close()
