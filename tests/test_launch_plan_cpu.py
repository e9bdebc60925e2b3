"""CPU: the launch plan (csrc/lmcma_plan.cpp) of every shape in the dispatch table, without a GPU.

plan_launch is plain integer arithmetic over the shape, the LMCMA_B200_* knobs and two device limits; here it is compiled
with g++ and no CUDA include path, so the compile itself shows that it needs no CUDA.  With the B200's limits, every
case of test_gpu_dispatch_variants.py must get the launch fields it expects there, and the cases together must reach
every kernel build lmcma_capi.cu instantiates.  The GPU file checks the same fields on a live handle.  The knobs the plan
reads come from Tuning::from_env (lmcma_plan.hpp), whose variables INTEGRATION.md section 5 must list."""
import math
import os
import re
import subprocess

import pytest

from lmcma_path_planner_b200 import _capi as K
from test_gpu_dispatch_variants import CASES, _instantiations, _source_instantiations

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "lmcma_path_planner_b200", "csrc")
B200 = (148, 232448)   # SMs, shared memory one block may opt into (bytes)

DRIVER = r"""
#include <cstdio>
#include <cstdlib>
#include "lmcma_plan.hpp"
#include "lmcma_b200.h"
// argv: n lambda m batch pop_count rng has_prior sm_count smem_optin; the knobs come from the environment
int main(int argc, char** argv) {
    if (argc != 10) return 2;
    lmcma_capi::PlanInput in{atoi(argv[1]), atoi(argv[2]), atoi(argv[3]), atoi(argv[4]), atoi(argv[5]), atoi(argv[6]),
                             atoi(argv[7]) != 0};
    const lmcma_capi::DeviceLimits dev{atoi(argv[8]), (size_t)atoll(argv[9])};
    lmcma_capi::LaunchPlan plan;
    std::string err;
    if (!lmcma_capi::plan_launch(in, dev, lmcma_capi::Tuning::from_env(), &plan, &err)) {
        printf("refused: %s\n", err.c_str());
        return 1;
    }
    int32_t v[LMCMA_B200_LAUNCH_FIELDS];
    lmcma_capi::launch_fields(plan, v);
    for (int i = 0; i < LMCMA_B200_LAUNCH_FIELDS; ++i) printf("%d ", v[i]);
    printf("\n");
    return 0;
}
"""


@pytest.fixture(scope="module")
def planner(tmp_path_factory):
    d = tmp_path_factory.mktemp("plan")
    (d / "driver.cpp").write_text(DRIVER)
    exe = str(d / "plan")
    r = subprocess.run(["g++", "-std=c++17", "-O1", "-Wall", "-I" + CSRC, "-I" + os.path.join(ROOT, "include"),
                        str(d / "driver.cpp"), os.path.join(CSRC, "lmcma_plan.cpp"), "-o", exe], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr

    def plan(n, lam, m, batch=1, env=None, rng=K.RNG_PHILOX, prior=False):
        """launch() of a handle with these arguments (unsplit population) on a B200, or the refusal's message."""
        lam = lam if lam >= 1 else 4 + int(3 * math.log(n))       # create's defaults (lmcma.cpp:134-135, 266)
        m = m if m >= 1 else lam
        envs = {k: v for k, v in os.environ.items() if not k.startswith("LMCMA_B200_")}
        envs.update(env or {})
        r = subprocess.run([exe] + [str(a) for a in (n, lam, m, batch, lam, rng, int(prior)) + B200], env=envs,
                           capture_output=True, text=True, timeout=60)
        if r.returncode == 1:
            return r.stdout.strip()
        assert r.returncode == 0, (r.returncode, r.stderr)
        out = dict(zip(K.LAUNCH_FIELDS, (int(x) for x in r.stdout.split())))
        out["sampler"] = K.SAMPLERS[out["sampler"]]
        return out
    return plan


@pytest.mark.parametrize("case", sorted(CASES))
def test_every_dispatch_case_gets_its_build(planner, case):
    c = CASES[case]
    got = planner(c.n, c.lam, c.m, c.batch, c.env)
    assert isinstance(got, dict), got
    assert {k: got[k] for k in c.expect} == c.expect, (case, got)


def test_the_cases_reach_every_launcher_instantiation(planner):
    reached = set()
    for c in CASES.values():
        reached |= _instantiations(planner(c.n, c.lam, c.m, c.batch, c.env))
    in_source = _source_instantiations()
    assert len(in_source) >= 30, sorted(in_source)                 # the patterns still match the launcher's spelling
    assert reached == in_source, ("not in lmcma_capi.cu", sorted(reached - in_source), "no case", sorted(in_source - reached))


@pytest.mark.parametrize("n", [2049, 2050])
def test_rows_beyond_2048_are_refused(planner, n):
    got = planner(n, 0, 0, rng=K.RNG_INJECT)
    assert isinstance(got, str) and "max 2048" in got, got


def test_integration_guide_lists_every_environment_switch():
    """INTEGRATION.md section 5 names exactly the LMCMA_B200_* variables Tuning::from_env reads."""
    src = open(os.path.join(CSRC, "lmcma_plan.hpp")).read()
    body = re.search(r"static Tuning from_env\(\) \{(.*?)\n    \}", src, re.S).group(1)
    read = set(re.findall(r"\"LMCMA_B200_([A-Z0-9_]+)\"", body))
    doc = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    section = re.search(r"^## 5\.(.*?)(?=^## |\Z)", doc, re.S | re.M).group(1)
    listed = set(re.findall(r"\bLMCMA_B200_([A-Z0-9_]+)", section))
    assert len(read) >= 10, sorted(read)                       # the pattern still matches from_env's spelling
    assert read == listed, ("read, not listed", sorted(read - listed), "listed, not read", sorted(listed - read))
