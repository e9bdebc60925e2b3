"""CPU: the C-ABI library loads without a GPU, exports every symbol include/lmcma_b200.h declares, its
host-side pieces match the golden vectors, and every compute entry point FAILS LOUDLY without a device
(no CPU fallback)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import lmcma_path_planner_b200 as L
from lmcma_path_planner_b200 import _capi as K

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _cuda_present():
    c = C.c_int(0)
    return K.lib().lmcma_b200_device_count(C.byref(c)) == 0 and c.value > 0


def test_every_declared_symbol_is_exported_and_bound():
    hdr = open(os.path.join(ROOT, "include", "lmcma_b200.h")).read()
    declared = set(re.findall(r"\b(lmcma_b200_[a-z0-9_]+)\s*\(", hdr))
    assert len(declared) >= 40
    lib = K.lib()
    for name in declared:
        assert hasattr(lib, name), name
    assert declared == set(K.SIGNATURES), declared ^ set(K.SIGNATURES)
    assert lib.lmcma_b200_abi_version() == 1


def test_launch_query_fields_follow_the_header():
    """Optimizer.launch() names the values of LMCMA_B200_I32_LAUNCH in the order of the header's LMCMA_B200_LAUNCH_* enum."""
    hdr = open(os.path.join(ROOT, "include", "lmcma_b200.h")).read()
    assert int(re.search(r"LMCMA_B200_I32_LAUNCH\s*=\s*(\d+)", hdr).group(1)) == K.I32_LAUNCH
    assert K.I32_LAUNCH not in K.I32.values()
    body = re.search(r"enum\s*\{\s*(LMCMA_B200_LAUNCH_SAMPLER\s*=\s*0[^}]*)\}", hdr).group(1)
    names = re.findall(r"LMCMA_B200_LAUNCH_([A-Z0-9_]+)", body)
    assert names[-1] == "FIELDS"
    assert [s.lower() for s in names[:-1]] == [f.lower() for f in K.LAUNCH_FIELDS]


def test_header_cites_the_reference_for_every_entry_point_group():
    hdr = open(os.path.join(ROOT, "include", "lmcma_b200.h")).read()
    for cite in ("lmcma.hpp:131", "lmcma.cpp:172-182", "lmcma.cpp:184-205", "lmcma.cpp:313-424", "lmcma.cpp:301-311",
                 "planner.cpp:591", "planner.cpp:677-690", "lmcma.cpp:426-429", "lmcma.cpp:14-82", "lmcma.cpp:769-810"):
        assert cite in hdr, cite


def test_hansen_stream_matches_reference_golden(golden):
    for seed, vec in golden["rng"].items():
        out = np.zeros(16)
        assert K.lib().lmcma_b200_hansen_gauss(int(seed), 0, 16, K.dptr(out)) == 0
        assert out.tolist() == vec["gauss"]
        u = np.zeros(8)
        assert K.lib().lmcma_b200_hansen_uniform(int(seed), 8, K.dptr(u)) == 0
        assert u.tolist() == vec["uniform"]
    a, b = np.zeros(5), np.zeros(8)
    K.lib().lmcma_b200_hansen_gauss(1, 3, 5, K.dptr(a))
    K.lib().lmcma_b200_hansen_gauss(1, 0, 8, K.dptr(b))
    assert np.array_equal(a, b[3:])


def test_covariance_known_answers(golden):
    """covariance(2,1) is the 2x2 identity (SURVEY section 4); covariance(2,4) matches the reference compiled
    against the Eigen stand-in (shim-pinned); the heap-based builder works where the reference's stack arrays
    overflow (n = 1500)."""
    c = np.zeros(4)
    assert K.lib().lmcma_b200_covariance(2, 1, K.dptr(c)) == 0
    assert np.allclose(c, golden["covariance_2_1"]) and np.allclose(c.reshape(2, 2), np.eye(2))
    c = np.zeros(64)
    assert K.lib().lmcma_b200_covariance(2, 4, K.dptr(c)) == 0
    assert np.allclose(c, golden["covariance_2_4_shim_pinned"], rtol=1e-9, atol=1e-12)
    n = 3 * 500
    big = np.zeros(n * n)
    assert K.lib().lmcma_b200_covariance(3, 500, K.dptr(big)) == 0
    big = big.reshape(n, n)
    assert np.allclose(big, big.T, atol=1e-9)
    assert np.all(big[:500, 500:] == 0)                       # block diagonal, dimension-major
    assert abs(big.diagonal().max() - 1.0 / 500) < 1e-12      # scaled by max variance * waypoints
    assert np.all(np.linalg.eigvalsh(big[:500, :500]) > 0)


def test_argument_errors_are_reported():
    h = C.c_void_p()
    cfg = K.Config()
    cfg.n, cfg.batch, cfg.sigma0 = 0, 1, 1.0
    assert K.lib().lmcma_b200_create(C.byref(cfg), None, None, None, C.byref(h)) == K.ERR_ARG
    assert b"n must be" in K.lib().lmcma_b200_last_error()
    assert K.lib().lmcma_b200_covariance(0, 3, None) == K.ERR_ARG
    assert K.lib().lmcma_b200_sync(None) == K.ERR_ARG


@pytest.mark.skipif(_cuda_present(), reason="this check is about machines WITHOUT a GPU")
def test_no_cpu_fallback_without_a_gpu():
    with pytest.raises(K.LmcmaError) as e:
        L.Optimizer(8, x0=np.zeros(8))
    assert e.value.code == K.ERR_CUDA
    with pytest.raises(K.LmcmaError):
        L.CostMap(np.ones((8, 8), np.float32))
    opt = L.LMCMA(np.zeros(4))
    with pytest.raises(K.LmcmaError):
        opt.init(4)


def test_library_is_in_tree_and_missing_library_is_fatal(tmp_path, monkeypatch):
    assert os.path.dirname(K.LIB_PATH) == os.path.join(ROOT, "lmcma_path_planner_b200")
    monkeypatch.setattr(K, "_lib", None)
    monkeypatch.setattr(K, "LIB_PATH", str(tmp_path / "nope.so"))
    with pytest.raises(ImportError):
        K.lib()


def test_workload_generators():
    from lmcma_path_planner_b200 import maps
    x0 = maps.straight_line((0, 0), (10, 20), 4)
    assert np.allclose(x0, [2, 4, 6, 8, 4, 8, 12, 16])         # dimension-major
    lo, hi = maps.box_bounds((100, 50), 3)
    assert lo.tolist() == [0] * 6 and hi.tolist() == [99] * 3 + [49] * 3
    d, s, g = maps.config2_map(size=256, n_rects=8, seed=3, clamp=20.0)
    assert d.shape == (256, 256) and d.max() <= 20.0 and d[int(s[1]), int(s[0])] > 0 and d[int(g[1]), int(g[0])] > 0
    assert np.all(d[:2] == 0) and np.all(d[:, -2:] == 0)       # solid border
    d2, _, _ = maps.config2_map(size=256, n_rects=8, seed=3, clamp=20.0)
    assert np.array_equal(d, d2)                               # seeded
    st, gl = maps.random_queries(d, 9, seed=1, min_sep=60)
    assert st.shape == (9, 2) and np.all(np.linalg.norm(st - gl, axis=1) >= 60)
    assert all(d[int(p[1]), int(p[0])] > 0 for p in st)


EXAMPLE = os.path.join(ROOT, "examples", "example_lmcma")


def test_cpp_facade_compiles_against_the_c_abi():
    """The C++ host side (include/lmcma_b200.hpp + examples/example_lmcma.cpp) is built by csrc/Makefile with
    plain g++ -std=c++11: the facade keeps the reference's constructor and method signatures."""
    assert os.path.exists(EXAMPLE), "run __graft_entry__.build()"
    hpp = open(os.path.join(ROOT, "include", "lmcma_b200.hpp")).read()
    for sig in ("LMCMA(double* initialParams, int lambda = 0, double* loBounds = 0, double* hiBounds = 0, double sigma = 1.0,",
                "void init(int N)", "void getNextParameterVector(double* params, int N)",
                "void setEvaluationFeedback(double* feedbacks, int numFeedbacks)", "bool isBehaviorLearningDone()",
                "int counteval;", "double BestF;"):
        assert sig in hpp, sig


@pytest.mark.skipif(_cuda_present(), reason="this check is about machines WITHOUT a GPU")
def test_cpp_example_fails_loudly_without_a_gpu(tmp_path):
    import subprocess
    r = subprocess.run([EXAMPLE, "demo"], cwd=tmp_path, capture_output=True, text=True, timeout=60)
    assert r.returncode == 3 and "lmcma_b200" in r.stderr


def test_cholesky_matches_numpy_and_rejects_indefinite(golden):
    """cholesky() of the reference (lmcma.cpp:844-855) restated on the host: L L^T = C for the smoothness prior."""
    cov = np.array(golden["covariance_2_10_shim_pinned"]).reshape(20, 20)
    Lm = np.zeros((20, 20))
    assert K.lib().lmcma_b200_cholesky(20, K.dptr(K.f64c(cov)), K.dptr(Lm)) == 0
    assert np.allclose(Lm, np.linalg.cholesky(cov), rtol=1e-12, atol=1e-15)
    assert np.all(np.triu(Lm, 1) == 0)
    bad = np.eye(3); bad[2, 2] = -1.0
    assert K.lib().lmcma_b200_cholesky(3, K.dptr(K.f64c(bad)), K.dptr(np.zeros((3, 3)))) == K.ERR_ARG
    ours = np.zeros(400)
    assert K.lib().lmcma_b200_covariance(2, 10, K.dptr(ours)) == 0
    assert np.allclose(ours, golden["covariance_2_10_shim_pinned"], rtol=1e-9, atol=1e-12)


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the reference's CPU implementation of the path: oracle/_ref when it was built here, else
    the restatement) runs without a GPU and prints ONE JSON line with the keys the driver reads."""
    import json
    import subprocess
    import sys
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    j = json.loads(lines[0])
    assert j["impl"] == "reference" and j["n_gpus"] == 1 and j["steps"] == 2 and j["warmup"] == 1
    assert j["unit"] == "evals/s" and j["higher_is_better"] is True and j["value"] > 0
    assert j["config"]["lambda"] == 1024 and j["config"]["n"] == 400 and "C2" in j["config"]["workload"]
    assert j["cpu_baseline"]["kind"] in ("reference", "port") and j["cpu_baseline"]["cores"] >= 1
    assert j["e2e"] == {"value": j["value"], "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert j["gpu_launches"] == 0


def test_reference_free_functions_match_the_compiled_reference():
    """differentiationMatrix / invert / cholesky / applyCovL / myqsort / random_* behind the reference's names
    (include/lmcma.hpp -> lmcma_b200_* host entry points) against golden outputs of the compiled reference
    (tests/golden/free_functions_reference.json; invert / cholesky / applyCovL there ran on the Eigen stand-in)."""
    import json
    g = json.load(open(os.path.join(ROOT, "tests", "golden", "free_functions_reference.json")))
    lib = K.lib()
    for case in g["diff"]:
        want = np.array(case["out"])
        got = np.full(want.shape, 7.0)
        assert lib.lmcma_b200_differentiation_matrix(case["steps"], case["order"], case["dt"], K.dptr(got), case["row_len"]) == 0
        assert np.array_equal(got, want), case["order"]                                   # bit-exact, untouched cells included
    A = np.array(g["invert"]["A"])
    Ai = np.zeros_like(A)
    assert lib.lmcma_b200_invert(K.dptr(A), K.dptr(Ai), 5) == 0
    assert np.allclose(Ai, np.array(g["invert"]["Ainv_shim_pinned"]), rtol=1e-12, atol=1e-14)
    assert np.allclose(Ai @ A, np.eye(5), atol=1e-12)
    assert lib.lmcma_b200_invert(K.dptr(np.zeros((3, 3))), K.dptr(np.zeros((3, 3))), 3) == K.ERR_ARG      # singular
    Cm = np.array(g["cholesky"]["C"])
    Lr = np.zeros_like(Cm)
    assert lib.lmcma_b200_cholesky(5, K.dptr(Cm), K.dptr(Lr)) == 0
    Lcol = np.ascontiguousarray(Lr.T)                                                      # the reference's layout: L[m*N+n] = L(n,m)
    assert np.allclose(Lcol, np.array(g["cholesky"]["L_shim_pinned"]), rtol=1e-12, atol=1e-14)
    z = np.array(g["cholesky"]["z"])
    assert lib.lmcma_b200_apply_cov_l(K.dptr(Lcol), K.dptr(z), 5) == 0
    assert np.allclose(z, np.array(g["cholesky"]["Lz_shim_pinned"]), rtol=1e-12, atol=1e-14)


def test_myqsort_and_rng_stream_objects(golden):
    ties = np.array(golden["qsort_ties"]["in"], np.float64)
    ids = np.zeros(len(ties), np.int32)
    assert K.lib().lmcma_b200_myqsort(len(ties), K.dptr(ties), K.iptr(ids)) == 0
    assert ids.tolist() == golden["qsort_ties"]["ids"] and ties.tolist() == golden["qsort_ties"]["sorted"]
    h = C.c_void_p()
    assert K.lib().lmcma_b200_rng_create(1, C.byref(h)) == 0
    u = [K.lib().lmcma_b200_rng_uniform(h) for _ in range(4)]
    assert u == golden["rng"]["1"]["uniform"][:4]
    K.lib().lmcma_b200_rng_destroy(h)
    assert K.lib().lmcma_b200_rng_create(1, C.byref(h)) == 0
    gs = [K.lib().lmcma_b200_rng_gauss(h) for _ in range(6)]
    assert gs == golden["rng"]["1"]["gauss"][:6]
    K.lib().lmcma_b200_rng_destroy(h)


def test_the_reference_s_own_demo_compiles_unchanged_against_the_drop_in_header(tmp_path):
    """INTEGRATION.md section 1.1: lmcma_path_planner/src/example_lmcma.cpp (test_lmcma + test_lmcma_using_cov: LMCMA,
    covariance(), the ask/tell loop) builds UNCHANGED with include/ on the include path instead of the reference's src/
    and links against liblmcma_b200.so.  The source is fed through stdin so that `#include "lmcma.hpp"` resolves to
    include/lmcma.hpp; <eigen3/Eigen/Dense>, which the demo includes but never uses, comes from the test stand-in."""
    import subprocess
    src = "/root/reference/lmcma_path_planner/src/example_lmcma.cpp"
    if not os.path.exists(src):
        pytest.skip("reference tree not present on this box (the prebuilt oracle/_ref/ref_example_lmcma is run by the GPU tests)")
    exe = tmp_path / "ref_example"
    with open(src) as fh:
        r = subprocess.run(["g++", "-std=c++11", "-O2", "-w", "-I" + os.path.join(ROOT, "include"),
                            "-I" + os.path.join(ROOT, "oracle", "eigen_shim"), "-x", "c++", "-", "-o", str(exe),
                            "-L" + os.path.join(ROOT, "lmcma_path_planner_b200"), "-llmcma_b200",
                            "-Wl,-rpath," + os.path.join(ROOT, "lmcma_path_planner_b200")], stdin=fh, capture_output=True, text=True, cwd=tmp_path)
    assert r.returncode == 0, r.stderr
    assert exe.exists()
