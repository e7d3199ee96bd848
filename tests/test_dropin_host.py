"""Host logic of the drop-in object API on a CPU-only box.

(1) The public surface SURVEY.md 8(b) lists exists under the reference's import paths and refuses to step without
    CUDA.  (2) The same end-to-end cases as tests/test_dropin_gpu.py, with the four kernel-backed calls swapped for
    the oracle-based stand-ins of tests/cpu_standin.py: everything ELSE -- marshalling between objects and vectors,
    boundary rules, spawn / absorb / hand-off bookkeeping, autograd wiring across lanes -- is the product code and is
    checked against the live-reference fixtures.  (3) Where $DHTS_REFERENCE names a checkout of the reference, the
    host-only rules are also compared with the live reference directly.
"""
import os
import sys

import numpy as np
import pytest
import torch as th

import cpu_standin
import dropin_cases as C


def test_surface_and_no_cpu_fallback():
    import dhts_b200.dropin as dropin
    dropin.install(precision="mixed")
    from dmath.operation import sigmoid
    from model.macro._arz import ARZ
    from road.lane._base_lane import BaseLane
    from road.lane._macro_lane import MacroLane
    from road.lane._micro_lane import DEFAULT_HEAD_POSITION_DELTA, DEFAULT_HEAD_SPEED_DELTA, MicroLane, MicroVehicle
    from road.lane.dmacro_lane import dMacroForwardLayer, dMacroLane
    from road.lane.dmicro_lane import dMicroForwardLayer, dMicroLane
    from road.network.conversion import Conversion
    from road.network.road_network import RoadNetwork
    from road.network.route import MacroRoute, MicroRoute
    from road.vehicle.vehicle import DEFAULT_VEHICLE_LENGTH, Vehicle
    here = os.path.dirname(os.path.abspath(dropin.__file__))
    for m in ("road.lane.dmacro_lane", "road.network.road_network", "model.macro._arz", "dmath.operation"):
        assert os.path.abspath(sys.modules[m].__file__).startswith(here), m
    lane = dMacroLane(0, 50.0, 30.0, 5.0)
    for name in ("forward update_state clear set_state_vector_u set_state_vector_y get_state_vector set_leftmost_cell "
                 "set_rightmost_cell get_leftmost_cell get_rightmost_cell curr_cell next_cell cell_length num_cell length "
                 "id speed_limit is_macro is_micro prev_lane next_lane has_prev_lane num_prev_lane flux_capacitor "
                 "add_flux_capacitor vectorize_input which d_lane").split():
        assert hasattr(lane, name), name
    assert lane.num_cell == 10 and lane.curr_cell[3].start == 15.0 and lane.curr_cell[3].end == 20.0
    assert lane.curr_cell[0].state.q.r == 0 and lane.curr_cell[0].state.u == 30.0
    ml = dMicroLane(1, 50.0, 30.0)
    for name in ("forward update_state clear set_state_vector get_state_vector curr_vehicle num_vehicle get_head_vehicle "
                 "get_tail_vehicle add_vehicle add_head_vehicle add_tail_vehicle entering_free_space on_this_lane "
                 "head_position_delta head_speed_delta vectorize_input clear_gradient").split():
        assert hasattr(ml, name), name
    assert (ml.head_position_delta, ml.head_speed_delta) == (DEFAULT_HEAD_POSITION_DELTA, DEFAULT_HEAD_SPEED_DELTA) == (1000, 0)
    net = RoadNetwork(30.0)
    for name in ("lane vehicle micro_route macro_route num_vehicle vehicle_length add_lane add_vehicle connect_lane "
                 "forward conversion setup_macro_boundary setup_micro_boundary get_macro_boundary "
                 "create_random_macro_route create_random_route create_default_vehicle_with_random_route "
                 "get_macro_state_of_micro_lane").split():
        assert hasattr(net, name), name
    v = MicroVehicle.default_micro_vehicle(30.0)
    assert (v.accel_max, v.accel_pref, v.target_speed, v.min_space, v.time_pref, v.length, v.a) == (30.0, 24.0, 27.0, 0.5, 0.1, 5.0, 5.0)
    assert abs(float(sigmoid(0.1, 16.0)) - 1 / (1 + np.exp(-1.6))) < 1e-6 and float(sigmoid(10.0, 16.0)) == float(th.sigmoid(th.tensor(16.0)))
    assert abs(ARZ.compute_u_eq(0.25, 30.0) - 30.0 * (1 - np.sqrt(0.25 + 1e-5))) < 1e-12
    if not th.cuda.is_available():
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            lane.set_state_vector_u(th.rand(10), th.rand(10))


@pytest.mark.parametrize("tier,precision,dtype,tol_s,tol_g", C.TIERS)
@pytest.mark.parametrize("mode", ["macro", "hybrid"])
def test_inverse_macro_and_hybrid_host_logic(tier, precision, dtype, tol_s, tol_g, mode):
    with cpu_standin.patched(precision):
        C.case_inverse_macro_and_hybrid_loss_curves(tier, precision, dtype, tol_s, tol_g, mode)


@pytest.mark.parametrize("tier,precision,dtype,tol_s,tol_g", C.TIERS)
def test_inverse_micro_host_logic(tier, precision, dtype, tol_s, tol_g):
    with cpu_standin.patched(precision):
        C.case_inverse_micro_loss_curve(tier, precision, dtype, tol_s, tol_g)


@pytest.mark.parametrize("tier,precision,dtype,tol_s,tol_g", C.TIERS)
def test_hybrid_chain_host_logic(tier, precision, dtype, tol_s, tol_g):
    with cpu_standin.patched(precision):
        C.case_hybrid_chain_spawn_absorb_and_gradients(tier, precision, dtype, tol_s, tol_g)


def test_macro_rollout_ghost_gradients_host_logic():
    with cpu_standin.patched("float64"):
        C.case_macro_lane_rollout_and_ghost_gradients(*C.TIERS[0])


def test_object_surface_host_logic():
    with cpu_standin.patched("float64"):
        C.case_object_surface_on_device()
        C.case_cfl_violation_raises_like_the_reference()


# ---------------------------------------------------------------------------------------------------------------
# (3) host-only rules against the LIVE reference (skipped unless $DHTS_REFERENCE names a checkout of it)

REF = os.environ.get("DHTS_REFERENCE", "")

_PROBE = r'''
import json, sys
import numpy as np
from road.lane.dmacro_lane import dMacroLane
from road.lane.dmicro_lane import dMicroLane
from road.network.road_network import RoadNetwork
from road.network.route import MicroRoute
from road.vehicle.micro_vehicle import MicroVehicle
out = {}
np.random.seed(11)
net = RoadNetwork(30.0)
kinds = "m M m m M m m m"          # m = micro, M = macro
for i, k in enumerate(kinds.split()):
    net.add_lane(dMicroLane(i, 40.0 + i, 30.0) if k == "m" else dMacroLane(i, 40.0, 30.0, 5.0))
for a, b in ((0, 2), (0, 1), (2, 3), (2, 5), (3, 4), (5, 6), (6, 7), (1, 7), (4, 7)):
    net.connect_lane(a, b)
out["macro_route"] = [sorted((int(k), int(v)) for k, v in net.create_random_macro_route().next_lane_dict.items()) for _ in range(3)]
out["routes"] = [[int(x) for x in net.create_random_route(s).route] for s in (0, 0, 0, 2, 2, 5, 1)]
rv = [MicroVehicle.random_micro_vehicle(30.0) for _ in range(2)]
out["random_vehicle"] = [[v.accel_max, v.accel_pref, v.target_speed, v.min_space, v.time_pref, v.length, v.a] for v in rv]
def put(lane, pos, speed, route):
    v = MicroVehicle.default_micro_vehicle(30.0); v.position = pos; v.speed = speed
    net.add_vehicle(v, MicroRoute(route, route.index(lane)))
    return v
put(0, 10.0, 7.0, [0, 2, 5, 6, 7]); put(0, 31.0, 9.0, [0, 2, 5, 6, 7]); put(0, 3.0, 5.0, [0, 2, 3, 4])
put(6, 12.5, 4.0, [0, 2, 5, 6, 7]); put(3, 39.0, 11.0, [0, 2, 3, 4]); put(5, 2.0, 3.0, [5, 6, 7]); put(7, 1.0, 2.0, [6, 7])
out["order0"] = [float(v.position) for v in net.lane[0].curr_vehicle]
try:
    put(0, 20.0, 1.0, [0, 2]); out["middle_insert"] = "accepted"
except AssertionError:
    out["middle_insert"] = "AssertionError"
try:
    put(0, 33.0, 1.0, [0, 2]); out["too_close"] = "accepted"
except AssertionError:
    out["too_close"] = "AssertionError"
heads = {}
for lid, lane in net.lane.items():
    if lane.is_micro():
        net.setup_micro_boundary(lid, True)
        heads[lid] = [float(lane.head_position_delta), float(lane.head_speed_delta)]
out["heads"] = heads
out["free"] = {lid: float(l.entering_free_space()) for lid, l in net.lane.items() if l.is_micro()}
out["macro_state"] = {lid: [float(x) for x in net.get_macro_state_of_micro_lane(lid, d)] for lid in (0, 2, 5, 6) for d in (False,)}
out["macro_state_soft"] = {lid: [float(x) for x in net.get_macro_state_of_micro_lane(lid, True)] for lid in (0, 2, 5, 6)}
m = net.lane[4]
m.set_leftmost_cell(0.25, 12.0); m.set_rightmost_cell(0.5, 3.0)
out["ghost"] = [float(m.leftmost_cell.state.q.r), float(m.leftmost_cell.state.q.y), float(m.leftmost_cell.state.u),
                float(m.leftmost_cell.state.u_eq), float(m.rightmost_cell.state.q.y)]
out["bdry"] = [[float(x) for x in net.get_macro_boundary(4, side, True)] for side in (True, False)]
print("PROBE" + json.dumps(out))
'''


@pytest.mark.skipif(not (REF and os.path.isdir(os.path.join(REF, "road"))), reason="$DHTS_REFERENCE: no checkout of the reference")
def test_host_rules_match_live_reference():
    import json
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

    def run(prefix, path):
        env = dict(os.environ, PYTHONPATH=path, PYTHONDONTWRITEBYTECODE="1")
        r = subprocess.run([sys.executable, "-c", prefix + _PROBE], capture_output=True, text=True, env=env, timeout=300)
        assert r.returncode == 0, r.stderr[-2000:]
        return json.loads(r.stdout[r.stdout.index("PROBE") + 5:])

    ref = run("", REF)
    ours = run("import dhts_b200.dropin as d; d.install()\n", root)
    assert ref["middle_insert"] == "AssertionError" and ref["too_close"] == "AssertionError"
    for k in ref:
        a, b = ref[k], ours[k]
        if k in ("heads", "free", "macro_state", "macro_state_soft", "ghost", "bdry", "random_vehicle", "order0"):
            fa = np.array([v for v in (a.values() if isinstance(a, dict) else a)], dtype=float)
            fb = np.array([v for v in (b.values() if isinstance(b, dict) else b)], dtype=float)
            assert fa.shape == fb.shape and np.abs(fa - fb).max() < 1e-6 * max(1.0, np.abs(fa).max()), (k, a, b)
            if isinstance(a, dict):
                assert list(a.keys()) == list(b.keys())
        else:
            assert a == b, (k, a, b)
