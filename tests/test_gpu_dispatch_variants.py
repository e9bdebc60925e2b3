"""Every sampler / update / k_coef build the launcher can pick by default, against the FP64 oracle.

The launcher picks a template instantiation from n, lambda, m and the batch size (plan_launch in lmcma_plan.cpp,
launch_sample / launch_update in lmcma_capi.cu), not from a workload name, so the shapes bench.py times leave builds
untested that users reach just by asking for more waypoints or a larger population.  Each case below first asserts,
through Optimizer.launch(), that it got the build it is there for, then runs the oracle comparison; the coverage test at
the end requires the cases (plus the shapes of older tests, named in the table) to reach every instantiation in
lmcma_capi.cu, so that a moved threshold or a new build without a case fails here.

Bars are those of _teacher_forced: integer state and ranks bit-exact, sigma 1e-12, X / mean / pc / V / P 2e-5 of their
scale, Nj / Lj 1e-4.  Shared-memory limits below are those of the B200 (227 KB opt-in per block)."""
import collections
import os
import re

import numpy as np
import pytest

import lmcma_path_planner_b200 as L
from lmcma_path_planner_b200 import _capi as K
from lmcma_path_planner_b200 import maps
from conftest import ROOT, weighted_sphere
from test_gpu_bench_shapes import _sampler_matches_oracle
from test_gpu_parity import _teacher_forced, rel_err

pytestmark = pytest.mark.gpu

Case = collections.namedtuple("Case", "n lam m batch env expect where")
Case.__new__.__defaults__ = (1, {}, {}, None)

# id -> (n, lambda, m, batch, env, expected launch fields, test elsewhere that holds this shape against the oracle)
CASES = {
    # the reference's defaults (lambda = 4 + int(3 ln n), m = lambda) past 512 columns; n = 201 / 603 / 2046 are 3-D paths
    # (n = 3W) whose rows end in padded columns
    "defaults-n201": Case(201, 0, 0, expect=dict(sampler="narrow", smp_nv=2, upd_nvb=4, upd_rmax=3, upd_rows_in_smem=1)),
    "defaults-n600": Case(600, 0, 0, expect=dict(sampler="narrow", smp_nv=8, upd_nvb=16, upd_rows_in_smem=1, upd_gram=0)),
    "defaults-n603": Case(603, 0, 0, expect=dict(sampler="narrow", smp_nv=8, upd_nvb=16, upd_rows_in_smem=1, upd_gram=0)),
    "defaults-n1026": Case(1026, 0, 0, expect=dict(sampler="narrow", smp_nv=12, upd_nvb=16, upd_rows_in_smem=1, upd_gram=0)),
    "defaults-n2046": Case(2046, 0, 0, expect=dict(sampler="narrow", smp_nv=16, smp_kc=4, upd_nvb=16, upd_rows_in_smem=1,
                                                   upd_gram=0)),
    "defaults-n2048": Case(2048, 0, 0, expect=dict(sampler="narrow", smp_nv=16, upd_nvb=16, upd_rows_in_smem=1, upd_gram=0)),
    # m = lambda beyond 80: rows in shared memory without the register sweep, rows in global memory, the Gram recompute
    # with 12 / 16 elements per lane.  k_coef's two m x m FP64 matrices fit 227 KB up to m = 119, so m = 119 is the
    # largest Gram shape and m = 120 the first that streams its rows from global memory at n = 1500
    "m100-n400": Case(400, 100, 100, expect=dict(sampler="narrow", smp_nv=4, smp_spec=1, upd_nvb=4, upd_rmax=0,
                                                 upd_rows_in_smem=1, upd_gram=0)),
    "m200-n400": Case(400, 200, 200, expect=dict(upd_nvb=4, upd_rmax=0, upd_rows_in_smem=0, upd_gram=0)),
    "m112-n512": Case(512, 112, 112, expect=dict(upd_nvb=4, upd_gram=1, coef_elems=16)),
    "m90-n1500": Case(1500, 90, 90, expect=dict(smp_nv=12, upd_nvb=16, upd_gram=1, coef_elems=12)),
    "m119-n1500": Case(1500, 119, 119, expect=dict(upd_nvb=16, upd_gram=1, coef_elems=16)),
    "m120-n1500": Case(1500, 120, 120, expect=dict(upd_nvb=16, upd_rows_in_smem=0, upd_gram=0)),
    "m160-n1500": Case(1500, 160, 160, expect=dict(upd_nvb=16, upd_rows_in_smem=0, upd_gram=0)),
    # the narrow -> wide sampler and 256 -> 1024-thread k_rank step
    "m255-n400": Case(400, 255, 255, expect=dict(sampler="narrow", rank_threads=256, rank_ftile=256, upd_rows_in_smem=0,
                                                 upd_gram=0)),
    "m257-n400": Case(400, 257, 257, expect=dict(sampler="wide", smp_RBW=2, rank_threads=1024, rank_ftile=4096,
                                                 upd_rows_in_smem=0, upd_gram=0)),
    # one query, wide sampler, five pending rows per warp: the overlapped generation, and the same shape in serial order
    "overlap-rmax5": Case(200, 512, 64, expect=dict(sampler="wide", smp_CW=2, upd_nvb=4, upd_rmax=5, progressive=1, overlap=1)),
    "serial-rmax5": Case(200, 512, 64, env={"LMCMA_B200_PROGRESSIVE": "0", "LMCMA_B200_OVERLAP": "0"},
                         expect=dict(upd_rmax=5, progressive=0, overlap=0)),
    # wide sampler with 10 / 16 column-warps together with the 16-block update
    "wide-cw10": Case(1200, 256, 24, expect=dict(sampler="wide", smp_CW=10, smp_RBW=2, upd_nvb=16, upd_rows_in_smem=1,
                                                 upd_gram=0)),
    "wide-cw16-gram": Case(2046, 1024, 30, expect=dict(sampler="wide", smp_CW=16, smp_RBW=4, upd_nvb=16, upd_gram=1,
                                                       coef_elems=5)),
    # rows sampler with 8 float4 columns per warp (n in 449..512), one / two rows per lane
    "rows-qw8-rl1": Case(480, 64, 40, 64, expect=dict(sampler="rows", smp_rows_qw=8, smp_rows_rl=1, upd_warps=16, upd_rmax=3)),
    "rows-qw8-rl2": Case(480, 64, 40, 300, expect=dict(sampler="rows", smp_rows_qw=8, smp_rows_rl=2, upd_warps=8, upd_rmax=5)),
    # shapes of older tests, kept here so that the coverage test sees every build
    "c1-default": Case(40, 0, 0, expect=dict(sampler="narrow", smp_nv=1),
                       where="test_gpu_parity.py::test_lmcma_teacher_forced_default_lambda"),
    "m40-n400": Case(400, 128, 40, expect=dict(sampler="narrow", smp_nv=4, upd_rmax=3),
                     where="test_gpu_parity.py::test_lmcma_teacher_forced_m_not_lambda"),
    "gram-n1500": Case(1500, 32, 77, expect=dict(smp_nv=12, upd_gram=1, coef_elems=10),
                       where="test_gpu_parity.py::test_lmcma_teacher_forced_large_n"),
    "gram-forced-n400": Case(400, 128, 40, env={"LMCMA_B200_UPDATE_GRAM": "1"}, expect=dict(upd_nvb=4, upd_gram=1, coef_elems=5),
                             where="test_gpu_parity.py::test_lmcma_teacher_forced_gram_path"),
    "eight-warps-rmax3": Case(24, 16, 8, 5, env={"LMCMA_B200_UPDATE_WARPS": "8"}, expect=dict(upd_warps=8, upd_rmax=3),
                              where="test_gpu_parity.py::test_batched_instances_are_independent"),
    "c2-fused": Case(400, 1024, 40, expect=dict(sampler="wide", smp_RBW=4, upd_rmax=3, overlap=1),
                     where="test_gpu_bench_shapes.py::test_fused_c2_generation_tracks_the_oracle"),
    "rows-qw7-rl2": Case(400, 64, 40, 320, expect=dict(sampler="rows", smp_rows_qw=7, smp_rows_rl=2),
                         where="test_gpu_bench_shapes.py::test_rows_sampler_batched_queries_at_the_c3_shape"),
    "rows-qw7-rl1": Case(400, 4096, 40, env={"LMCMA_B200_SAMPLE_ROWS": "1"}, expect=dict(sampler="rows", smp_rows_qw=7, smp_rows_rl=1),
                         where="test_gpu_bench_shapes.py::test_rows_sampler_teacher_forced_single_population"),
    "rows-qw4-rl2": Case(100, 20480, 6, expect=dict(sampler="rows", smp_rows_qw=4, smp_rows_rl=2),
                         where="test_gpu_bench_shapes.py::test_rows_sampler_teacher_forced_single_population"),
    "rows-qw4-rl1": Case(48, 4096, 11, env={"LMCMA_B200_SAMPLE_ROWS": "1"}, expect=dict(sampler="rows", smp_rows_qw=4, smp_rows_rl=1),
                         where="test_gpu_bench_shapes.py::test_rows_sampler_teacher_forced_single_population"),
}


def _instantiations(l):
    """The template instantiations (spelled as in lmcma_capi.cu, without spaces) a handle with launch() == l runs."""
    if l["sampler"] == "rows":
        smp = "launch_sample_rows_t<%d,%d>" % (l["smp_rows_qw"], l["smp_rows_rl"])
    elif l["sampler"] == "wide":
        smp = "launch_sample_wide_t<%d>" % l["smp_RBW"]
    else:
        smp = "launch_sample_t<%d>" % l["smp_nv"]
    nvb, rmax = l["upd_nvb"], l["upd_rmax"]
    if l["upd_gram"]:
        return {smp, "launch_update_t<%d,-1,false>" % nvb, "k_coef<%d>" % l["coef_elems"]}
    smem = "true" if l["upd_rows_in_smem"] else "false"
    if nvb == 4 and rmax in (3, 5):
        upd = "<4,%d,true,true>" % rmax if l["overlap"] else ("<4,%d,true,false,8>" % rmax if l["upd_warps"] == 8 else "<4,%d,true>" % rmax)
    else:
        upd = "<%d,0,%s>" % (nvb, smem)
    return {smp, "launch_update_t" + upd}


def _source_instantiations():
    src = open(os.path.join(ROOT, "lmcma_path_planner_b200", "csrc", "lmcma_capi.cu")).read()
    found = {"%s<%s>" % (name, args.replace(" ", "")) for name, args in
             re.findall(r"\b(launch_sample_t|launch_sample_wide_t|launch_sample_rows_t|launch_update_t)<([^<>]*)>\(", src)}
    return found | set(re.findall(r"\bk_coef<\d+>", src))


def _open(case_id, monkeypatch, **kw):
    """The handle of a table case (its environment knobs set while it is created) with its launch fields checked."""
    c = CASES[case_id]
    for k, v in c.env.items():
        monkeypatch.setenv(k, v)
    x0 = kw.pop("x0", np.full(c.n, 0.5))
    dev = L.Optimizer(c.n, x0=x0, lam=c.lam, m=c.m, batch=c.batch, **kw)
    got = dev.launch()
    for k, v in c.expect.items():
        assert got[k] == v, (case_id, k, got)
    for k in c.env:
        monkeypatch.delenv(k)
    return dev


def _warm_state(po, n, m, sigma=0.4):
    """An oracle state with all m slots live and recycled: a cheap lambda = 16 run of m + 9 generations."""
    small = po.OracleLMCMA(n, x0=np.full(n, 0.5), lam=16, m=m, sigma=sigma, seed=1)
    for _ in range(m + 9):
        small.tell_all(weighted_sphere(small.array("X")))
    st = small.state()
    assert st["live"] == m and st["itr"] == m + 9
    return st


@pytest.fixture(scope="module")
def map1024():
    dist, start, goal = maps.config2_map(size=1024, n_rects=128, seed=42, clamp=64.0)
    return dict(dist=dist, start=start, goal=goal, cmap=L.CostMap(dist, "f32"))


# ------------------------------------------------------------------------------------------------
# 1. the reference's defaults beyond 512 columns, teacher-forced past slot recycling
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", ["defaults-n201", "defaults-n600", "defaults-n603", "defaults-n1026", "defaults-n2046",
                                  "defaults-n2048"])
def test_reference_defaults_teacher_forced(po, monkeypatch, case):
    dev = _open(case, monkeypatch, rng="inject")
    n, m = CASES[case].n, dev.m
    dev.close()
    _teacher_forced(po, n, 0, 0, m + 6, seed=n)


@pytest.mark.parametrize("n", [2049, 2050])
def test_rows_beyond_2048_are_refused(n):
    with pytest.raises(K.LmcmaError) as e:
        L.Optimizer(n, x0=np.zeros(n), rng="inject")
    assert e.value.code == K.ERR_ARG and "max 2048" in str(e.value)


# ------------------------------------------------------------------------------------------------
# 2. m = lambda beyond 80, warm-started so that every slot is live and being recycled
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", ["m100-n400", "m200-n400", "m112-n512", "m90-n1500", "m119-n1500", "m120-n1500",
                                  "m160-n1500", "m255-n400", "m257-n400"])
def test_many_pairs_teacher_forced_from_a_warm_state(po, monkeypatch, case):
    c = CASES[case]
    _open(case, monkeypatch, rng="inject").close()
    _teacher_forced(po, c.n, c.lam, c.m, 8, seed=c.m, warm=_warm_state(po, c.n, c.m))


# ------------------------------------------------------------------------------------------------
# 3. odd n, device Philox deviates: padded columns must not leak into V z or the mean
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", ["defaults-n603", "defaults-n2046"])
def test_free_running_odd_n_matches_oracle_short_window(po, monkeypatch, case):
    n = CASES[case].n
    dev = _open(case, monkeypatch, sigma0=0.3, seed=7, record_z=True)
    lam, m = dev.lam, dev.m
    z0 = dev.get("Z")[0].astype(np.float64)
    ora = po.OracleLMCMA(n, x0=np.full(n, 0.5), lam=lam, m=m, sigma=0.3, seed=1, Z0=z0)
    for g in range(6):
        Xd = dev.ask_all()[0]
        assert rel_err(Xd, ora.array("X"), floor=1e-2) < 1e-4, g
        f = weighted_sphere(Xd).astype(np.float32)
        dev.tell_all(f)
        ora.tell_all(f.astype(np.float64), dev.get("Z")[0].astype(np.float64))
    assert rel_err(dev.get("xmean")[0], ora.array("xmean"), floor=1e-2) < 1e-4
    assert abs(dev.get("sigma")[0] - ora.doubles()["sigma"]) / ora.doubles()["sigma"] < 1e-9


# ------------------------------------------------------------------------------------------------
# 4. the overlapped generation with five pending rows per warp (k_update<4, 5, smem, OVERLAP>)
# ------------------------------------------------------------------------------------------------
def _planning(map1024, W):
    lo, hi = maps.box_bounds((1024, 1024), W)
    return lo, hi, maps.straight_line(map1024["start"], map1024["goal"], W)


def test_overlapped_five_rows_per_warp_tracks_the_oracle(po, map1024, monkeypatch):
    """Fused generations teacher-forced every generation: the oracle gets the device's deviates and fitness, the device
    continues from the oracle's exact state.  70 generations: all 64 slots live and being recycled."""
    W, p = 100, map1024
    lo, hi, x0 = _planning(p, W)
    dev = _open("overlap-rmax5", monkeypatch, x0=x0, lo=lo, hi=hi, sigma0=8.0, seed=5, record_z=True)
    dev.attach_cost(p["cmap"], [p["start"]], [p["goal"]], W, L.LONGSAFE, 1e4)
    n, lam, m = dev.n, dev.lam, dev.m
    ora = po.OracleLMCMA(n, x0=x0, lam=lam, m=m, lo=lo, hi=hi, sigma=8.0, seed=1, Z0=dev.get("Z")[0].astype(np.float64))
    worst = {}
    for g in range(70):
        Xd, Xo = dev.get("X")[0], ora.array("X")
        worst["X"] = max(worst.get("X", 0), float(np.abs(Xd - Xo).max()) / 1023.0)
        dev.run(1)
        ora.tell_all(dev.get("fit")[0].astype(np.float64), dev.get("Z")[0].astype(np.float64))
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
        worst["Nj"] = max(worst.get("Nj", 0), rel_err(dev.get("Nj")[0][live], so["Nj"][live]))
        dev.load_state(so)
        dev.resample()
    assert so["live"] == m and so["itr"] > m
    assert worst["sigma"] < 1e-12, worst
    for k in ("X", "xmean", "pc", "V"):
        assert worst[k] < 2e-5, (k, worst)
    assert worst["Nj"] < 1e-4, worst


def test_overlapped_five_rows_per_warp_bits_equal_the_serial_order(map1024, monkeypatch):
    """Serial, progressive and overlapped fused generations, and the host-buffer protocol (ask_all_view -> cost_evaluate
    -> tell_all, with tell_all's speculative update on and off) give the same bits, 70 generations from the same seed."""
    W, p = 100, map1024
    lo, hi, x0 = _planning(p, W)
    keys = ("X", "xmean", "V", "P", "pc", "sigma", "t", "vec", "Nj", "Lj")
    state = {}
    for mode, (prog, ovl) in {"serial": ("0", "0"), "progressive": ("1", "0"), "overlapped": ("1", "1")}.items():
        monkeypatch.setenv("LMCMA_B200_PROGRESSIVE", prog)
        monkeypatch.setenv("LMCMA_B200_OVERLAP", ovl)
        dev = L.Optimizer(2 * W, x0=x0, lam=512, m=64, lo=lo, hi=hi, sigma0=8.0, seed=11)
        got = dev.launch()
        assert got["upd_rmax"] == 5 and (got["progressive"], got["overlap"]) == (int(prog), int(prog) * int(ovl)), (mode, got)
        dev.attach_cost(p["cmap"], [p["start"]], [p["goal"]], W, L.LONGSAFE, 1e4)
        dev.run(70)
        state[mode] = {k: dev.get(k).copy() for k in keys}
        state[mode]["best_f"] = dev.best()[1].copy()
        dev.close()
    for mode in ("progressive", "overlapped"):
        for k in state["serial"]:
            assert np.array_equal(state[mode][k], state["serial"][k]), (mode, k)
    monkeypatch.setenv("LMCMA_B200_PROGRESSIVE", "1")
    monkeypatch.setenv("LMCMA_B200_OVERLAP", "1")
    for spec in ("0", "1"):
        monkeypatch.setenv("LMCMA_B200_TELL_SPEC", spec)
        dev = L.Optimizer(2 * W, x0=x0, lam=512, m=64, lo=lo, hi=hi, sigma0=8.0, seed=11)
        assert dev.launch()["overlap"] == 1
        for g in range(70):
            r = p["cmap"].evaluate(np.array(dev.ask_all_view()[0]), p["start"], p["goal"], W, L.LONGSAFE, 1e4)
            dev.tell_all(r["f"])
        for k in keys:
            assert np.array_equal(dev.get(k), state["serial"][k]), ("tell_all, speculative update " + spec, k)
        assert np.array_equal(dev.best()[1], state["serial"]["best_f"])
        dev.close()


# ------------------------------------------------------------------------------------------------
# 5. wide sampler together with the 16-block update
# ------------------------------------------------------------------------------------------------
def test_wide_sampler_ten_column_warps_with_the_long_row_update(po, monkeypatch):
    _open("wide-cw10", monkeypatch, rng="inject").close()
    _teacher_forced(po, 1200, 256, 24, 30, seed=12)


def test_wide_sampler_sixteen_column_warps_with_the_gram_update(po, monkeypatch):
    _open("wide-cw16-gram", monkeypatch, rng="inject").close()
    _teacher_forced(po, 2046, 1024, 30, 6, seed=13, warm=_warm_state(po, 2046, 30))


# ------------------------------------------------------------------------------------------------
# 6. rows sampler with eight float4 columns per warp (n in 449..512)
# ------------------------------------------------------------------------------------------------
def test_rows_sampler_eight_columns_per_warp(po, map1024, monkeypatch):
    """Batched queries at n = 480: 64 instances (one row per lane, 16-warp k_update) and 300 instances (two rows per lane,
    8-warp k_update, two CTAs per SM).  The sampled population of a few instances is held against the oracle's sample()
    from the device's own state and deviates while the pairs fill and once all 40 are live and recycled; and instance b of
    the 64-instance batch equals instance b of the 300-instance batch bit for bit (same deviates: Philox keyed by seed,
    instance and row; same per-row arithmetic whatever the rows per lane and the update's CTA size)."""
    monkeypatch.setenv("LMCMA_B200_COST_TPT", "64")            # same reduction tree of k_cost whatever the launch
    W, p = 240, map1024
    lo, hi = maps.box_bounds((1024, 1024), W)
    starts, goals = maps.random_queries(p["dist"], 300, seed=7, min_sep=256)
    x0 = np.stack([maps.straight_line(s, g, W) for s, g in zip(starts, goals)])
    devs = {}
    for case, B in (("rows-qw8-rl1", 64), ("rows-qw8-rl2", 300)):
        dev = _open(case, monkeypatch, x0=x0[:B], lo=lo, hi=hi, sigma0=16.0, seed=7, record_z=True)
        dev.attach_cost(p["cmap"], starts[:B], goals[:B], W, L.LONGSAFE, 1e4)
        for gens in (12, 35):
            dev.run(gens)
            assert _sampler_matches_oracle(po, dev, 2 * W, 64, 40, lo, hi, (0, B // 2, B - 1)) < 2e-5, (case, gens)
        assert int(dev.get("live")[B - 1]) == 40 and int(dev.get("itr")[0]) == 47
        devs[B] = dev
    for k in ("X", "xmean", "sigma", "V", "P", "pc", "Nj", "t", "vec", "fit"):
        assert np.array_equal(devs[300].get(k)[:64], devs[64].get(k)), k


# ------------------------------------------------------------------------------------------------
# 7. fused graphs at a shape past 512 columns
# ------------------------------------------------------------------------------------------------
def test_fused_graphs_beyond_512_columns(map1024, monkeypatch):
    """n = 600 (W = 300, the reference's default lambda and m): nine fused generations give the same bits with eight
    generations per CUDA graph (one graph of 8 + one of 1) and with one per graph, and the same bits as nine rounds of
    ask_all -> cost_evaluate -> tell_all through host buffers."""
    W, p = 300, map1024
    lo, hi, x0 = _planning(p, W)
    keys = ("X", "xmean", "V", "P", "pc", "sigma", "t", "vec", "Nj", "Lj", "fit")
    out = {}
    for unroll in ("8", "1"):
        monkeypatch.setenv("LMCMA_B200_GRAPH_UNROLL", unroll)
        dev = _open("defaults-n600", monkeypatch, x0=x0, lo=lo, hi=hi, sigma0=6.0, seed=3)
        dev.attach_cost(p["cmap"], [p["start"]], [p["goal"]], W, L.LONGSAFE, 1e4)
        dev.run(9)
        out[unroll] = {k: dev.get(k).copy() for k in keys}
        out[unroll]["best"] = dev.best()
        dev.close()
    monkeypatch.delenv("LMCMA_B200_GRAPH_UNROLL")
    host = _open("defaults-n600", monkeypatch, x0=x0, lo=lo, hi=hi, sigma0=6.0, seed=3)
    for g in range(9):
        r = p["cmap"].evaluate(host.ask_all()[0], p["start"], p["goal"], W, L.LONGSAFE, 1e4)
        host.tell_all(r["f"])
    for k in keys:
        assert np.array_equal(out["8"][k], out["1"][k]), ("graph unroll", k)
        assert np.array_equal(out["8"][k], host.get(k)), ("host protocol", k)
    xb, fb = host.best()
    assert np.array_equal(out["8"]["best"][0], xb) and np.array_equal(out["8"]["best"][1], fb)


# ------------------------------------------------------------------------------------------------
# 8. coverage: the table reaches every instantiation the launcher has
# ------------------------------------------------------------------------------------------------
def test_every_launcher_instantiation_is_reached_by_a_case(monkeypatch):
    import importlib
    reached = {}
    for cid, c in CASES.items():
        with monkeypatch.context() as mp:
            dev = _open(cid, mp)                                   # device deviates: the progressive / overlapped builds need them
            for inst in _instantiations(dev.launch()):
                reached.setdefault(inst, []).append(cid)
            dev.close()
        if c.where:                                                # the older test holding this shape still exists
            mod, name = c.where.split("::")
            assert hasattr(importlib.import_module(mod[:-3]), name), c.where
    in_source = _source_instantiations()
    assert len(in_source) >= 30, sorted(in_source)                 # the patterns still match the launcher's spelling
    assert set(reached) <= in_source, sorted(set(reached) - in_source)
    unreached = in_source - set(reached)
    assert not unreached, sorted(unreached)
