"""bench.py --dump-outputs: every array it writes -- losses, ARZ rT / yT / uT / g_r0 / g_u0 and IDM pT / vT / g_p0 /
g_v0 of the sampled lanes -- against the oracle on the same inputs.  The batch is larger than the dump budget, so
both samples are strict subsets of the lanes."""
import os
import subprocess
import sys
import types

import numpy as np
import pytest
import torch

from conftest import ROOT, relerr

pytestmark = pytest.mark.gpu


def test_dumped_outputs_match_the_oracle(tmp_path, dev):
    import bench
    from oracle import oracle as O
    a = types.SimpleNamespace(lanes=1100, cells=1024, micro_lanes=8200, lane_vehicles=64, sim_steps=20)
    out = str(tmp_path / "dump")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--lanes", str(a.lanes), "--cells", str(a.cells),
                        "--micro-lanes", str(a.micro_lanes), "--lane-vehicles", str(a.lane_vehicles),
                        "--sim-steps", str(a.sim_steps), "--steps", "2", "--warmup", "1", "--no-e2e", "--no-net",
                        "--no-cpu-baseline", "--no-drivers", "--dump-outputs", out],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    got = {f[:-4]: np.load(os.path.join(out, f)) for f in os.listdir(out)}
    assert sorted(got) == sorted(["losses"] + ["arz_" + k for k in ("rT", "yT", "uT", "g_r0", "g_u0")]
                                 + ["idm_" + k for k in ("pT", "vT", "g_p0", "g_v0")])
    assert all(v.dtype == np.float64 for v in got.values())
    assert sum(v.nbytes for v in got.values()) <= 64 << 20

    A = {k: (v.double().numpy() if hasattr(v, "numpy") else v) for k, v in bench.make_arz_inputs(a, 0, torch).items()}
    gh = np.stack([A["gr"], A["gu"]], -1)
    f = O.arz_rollout(A["r0"], A["u0"], gh, A["dx"], A["umax"], A["dt"], a.sim_steps)
    o = O.arz_rollout(A["r0"], A["u0"], gh, A["dx"], A["umax"], A["dt"], a.sim_steps,
                      g_rT=2.0 * (f["rT"] - A["tr"]), g_uT=2.0 * (f["uT"] - A["tu"]))
    lanes = bench.dump_sample(a.lanes, 5 * a.cells * 8, bench.DUMP_ARZ_BYTES)
    assert 0 < len(lanes) < a.lanes and got["arz_rT"].shape == (len(lanes), a.cells)
    for k in ("rT", "yT", "uT"):
        assert relerr(got["arz_" + k], o[k][lanes]) < 1e-9, k
    for k in ("g_r0", "g_u0"):
        assert relerr(got["arz_" + k], o[k][lanes]) < 1e-8, k

    M = {k: (v.double().numpy() if hasattr(v, "numpy") else v) for k, v in bench.make_idm_inputs(a, 0, torch).items()}
    fi = O.idm_rollout(M["p0"], M["v0"], M["params"], M["off"], M["head"], M["dt"], a.sim_steps)
    oi = O.idm_rollout(M["p0"], M["v0"], M["params"], M["off"], M["head"], M["dt"], a.sim_steps,
                       g_pT=2.0 * (fi["pT"] - M["tp"]), g_vT=2.0 * (fi["vT"] - M["tv"]))
    mlanes = bench.dump_sample(a.micro_lanes, 4 * a.lane_vehicles * 8, bench.DUMP_IDM_BYTES)
    assert 0 < len(mlanes) < a.micro_lanes
    veh = np.concatenate([np.arange(l * a.lane_vehicles, (l + 1) * a.lane_vehicles) for l in mlanes])
    for k in ("pT", "vT"):
        assert relerr(got["idm_" + k], oi[k][veh]) < 1e-9, k
    for k in ("g_p0", "g_v0"):
        assert relerr(got["idm_" + k], oi[k][veh]) < 1e-8, k

    want = [((o["rT"] - A["tr"]) ** 2).sum() + ((o["uT"] - A["tu"]) ** 2).sum(),
            ((oi["pT"] - M["tp"]) ** 2).sum() + ((oi["vT"] - M["tv"]) ** 2).sum()]
    assert relerr(got["losses"], np.array(want)) < 1e-9
