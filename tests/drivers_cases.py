"""Shared body of tests/test_drivers_gpu.py and tests/test_drivers_host.py: the reference's UNMODIFIED drivers
``example/inverse/{macro,micro,hybrid}.py`` (``InverseProblem.initialize`` + ``solve_gd``, _inverse.py:66-88,185-242)
run on top of the drop-in ``road/ model/ dmath/`` packages and must reproduce the curves frozen from the same
drivers on the reference's own lanes (tests/golden/drivers_fp32.npz, oracle/gen_golden_drivers.py).

The driver files live in the git-ignored reference install ``baseline/_ref``, which baseline/install_ref.py copies
from the checkout of the reference named by $DHTS_REFERENCE; the tests skip when it is absent.  One subprocess per
problem: the drivers import ``road.*`` by name, and this pytest process may already hold other modules under those
names.

Two tiers, as everywhere in this suite (SURVEY 8c):
  * fp64 -- the drivers and the reference run in float64 (no-edit dtype rebinding, ``run_drivers.py --fp64``), the
    drop-in with precision="float64": error curves and states to 1e-8 (only re-association separates the two);
  * fp32 -- the reference as shipped (fp32 state between steps, fp64 step) against precision="mixed": target end
    state 2e-5, error curves 5e-4 when every ``RoadNetwork.forward`` is stepped immediately (per-step fp32 rounding
    as in the reference) and 3e-3 with DEFERRED stepping, where the queued steps run as one fp64 rollout and the
    state is rounded to fp32 once at the end: the curves are sums of squared differences of nearly equal states, so
    they amplify that rounding difference (the fp64 tier shows the deferred path itself is exact).
"""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, golden, relerr


def run_driver(problem, tmp_path, tier="fp32", defer=True, extra=()):
    ref = os.path.join(ROOT, "baseline", "_ref", "example", "inverse", problem + ".py")
    if not os.path.exists(ref):
        pytest.skip("baseline/_ref is absent (python baseline/install_ref.py populates it from $DHTS_REFERENCE)")
    g = golden("drivers_" + tier)
    out = str(tmp_path / (problem + ".npz"))
    env = dict(os.environ, DHTS_RUN_DIR=str(tmp_path))
    args = ["--fp64"] if tier == "fp64" else ["--precision", "mixed"]
    if not defer:
        args.append("--no-defer")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "baseline", "run_drivers.py"), "--impl", "dropin", "--problem",
                        problem, "--episodes", str(int(g["episodes"])), "--seed", str(int(g["seed"])), "--out", out] + args
                       + list(extra), capture_output=True, text=True, env=env, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    # the drivers are the reference's files, the lanes / network underneath are ours
    assert line["drivers_from"].endswith(os.path.join("baseline", "_ref", "example", "inverse")), line
    assert line["core_packages_from"].endswith("dropin"), line
    z = np.load(out)
    tol_s, tol_e = (1e-8, 1e-8) if tier == "fp64" else (2e-5, 3e-3 if defer else 5e-4)
    # same RNG consumption as the reference: identical true / estimated initial states
    assert relerr(z["beg_state"], g[problem + "_beg_state"]) < 1e-6
    assert relerr(z["est0"], g[problem + "_est0"]) < 1e-6
    assert relerr(z["end_state"], g[problem + "_end_state"]) < tol_s
    assert relerr(z["end_errors"], g[problem + "_end_errors"]) < tol_e
    assert relerr(z["beg_errors"], g[problem + "_beg_errors"]) < tol_e
    return line
