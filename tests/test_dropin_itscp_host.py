"""The reference's UNMODIFIED ``ItscpRoadNetwork`` (example/control/itscp/_simulator.py, loaded by path) on top of OUR
drop-in ``road.*`` / ``model.*`` / ``dmath.*`` packages: it subclasses ``RoadNetwork`` and overrides
``setup_macro_boundary`` / ``setup_micro_boundary`` (signal-blended ghost cells and head deltas), which is the part of the
ITSCP scripts that touches the hot path.  Host logic only (CPU box: kernel calls swapped for the oracle-backed stand-ins of
tests/cpu_standin.py); the frames must reproduce the live-reference fixture tests/golden/itscp_hybrid_h*_fp64.npz, which was
frozen from the same class over the reference's own lanes.  Skipped unless $DHTS_REFERENCE names a checkout of the
reference."""
import os
import sys

import numpy as np
import pytest
import torch as th

import cpu_standin
from hyb_cases import fixture_case

REF = os.environ.get("DHTS_REFERENCE", "")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def f(x):
    return float(x.detach()) if isinstance(x, th.Tensor) else float(x)


@pytest.mark.skipif(not (REF and os.path.isdir(os.path.join(REF, "example"))), reason="$DHTS_REFERENCE: no checkout of the reference")
def test_reference_itscp_simulator_runs_on_the_dropin_lanes():
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    G = fixture_case("h")
    T = 24
    with cpu_standin.patched("float64"):
        th.set_default_dtype(th.float64)
        try:
            from gen_golden_net import load_reference_simulator
            import road.network.road_network as ours_net
            assert os.path.abspath(ours_net.__file__).startswith(os.path.join(ROOT, "diff-hybrid-traffic-sim_b200"))
            ItscpRoadNetwork, _ = load_reference_simulator()

            class _NP64:                     # the fixture's RunningMean accumulated in float64 (oracle/gen_golden_hyb.py)
                float32 = np.float64

                def __getattr__(self, k):
                    return getattr(np, k)
            sys.modules["example.common.rms"].np = _NP64()
            assert ItscpRoadNetwork.__mro__[1] is ours_net.RoadNetwork                  # their subclass, our base class
            assert os.path.abspath(sys.modules[ItscpRoadNetwork.__module__].__file__).startswith(REF)
            from dhts_b200.itscp import ItscpGrid
            from dmath.operation import sigmoid
            from road.lane.dmacro_lane import dMacroLane
            from road.lane.dmicro_lane import dMicroLane
            grid = ItscpGrid(int(G["num_intersection"]), int(G["num_lane"]), float(G["lane_length"]), float(G["cell_length"]))
            umax, dt, fps, n = float(G["umax"]), float(G["dt"]), int(G["frames_per_signal"]), grid.num_intersection
            np.random.seed(21)                                                          # gen_golden_hyb.main: case h
            net = ItscpRoadNetwork(umax)
            kind = G["kind"].tolist()
            for info, k in zip(grid.lanes, kind):
                net.add_lane(dMicroLane(len(net.lane), info.length, umax) if k else dMacroLane(len(net.lane), info.length, umax, grid.cell_length))
            for a, b in grid.links:
                net.connect_lane(a, b)
            L = grid.L
            mic = [l for l in range(L) if kind[l]]
            off = np.concatenate([[0], np.cumsum([0 if kind[l] else net.lane[l].num_cell for l in range(L)])]).astype(int)
            bl = grid.boundary_lanes()
            routes = [net.create_random_macro_route() for _ in range(int(G["T"]))]      # same np.random consumption as the fixture run
            tab = np.array([[[r.get_prev_lane(l) for l in range(L)], [r.get_next_lane(l) for l in range(L)]] for r in routes[:T]])
            assert (tab == G["route"][:T]).all()
            action = th.tensor(G["action"])
            for l in range(L):
                if not kind[l]:
                    net.lane[l].set_state_vector_u(th.tensor(G["r0"][off[l]:off[l + 1]]), th.tensor(G["u0"][off[l]:off[l + 1]]))
            n2, n_phase = n * n, max(1, int(G["T"]) // fps)
            for t in range(T):
                phase, progress = min(t // fps, n_phase - 1), min((t % fps) / fps, 1.0)
                for l, info in enumerate(grid.lanes):
                    if info.loc == "mid" or not info.approaching:
                        s = 1.0
                    else:
                        a = action[phase * n2 + info.row * n + info.col]
                        s = sigmoid(a - progress, constant=32) if info.loc in ("west", "east") else sigmoid(progress - a, constant=32)
                    net.lane_signal[l] = s
                    net.lane_incoming[l] = th.tensor(G["incoming"][t, l]) if l in bl else -1
                net.macro_route = routes[t]
                net.forward(dt, True)
                # every frame against the fixture: cells, vehicle counts, vehicles head first, head deltas
                for l in range(L):
                    if kind[l]:
                        m = mic.index(l); lane = net.lane[l]
                        assert lane.num_vehicle() == G["vcnt"][t + 1, m], (t, l)
                        for j, mv in enumerate(reversed(lane.curr_vehicle)):
                            got = np.array([f(mv.position), f(mv.speed), f(mv.a)])
                            assert np.abs(got - G["veh"][t + 1, m, j]).max() < 1e-8, (t, l, j)
                        want = G["head"][t, m]
                        assert abs(f(lane.head_position_delta) - want[0]) < 1e-7 * max(1.0, abs(want[0])) and \
                            abs(f(lane.head_speed_delta) - want[1]) < 1e-7 * max(1.0, abs(want[1])), (t, l)
                    else:
                        got = np.array([[f(c.state.q.r), f(c.state.q.y), f(c.state.u)] for c in net.lane[l].curr_cell]).T
                        assert np.abs(got - G["hist"][t + 1][:, off[l]:off[l + 1]]).max() < 1e-8, (t, l)
            assert G["vcnt"][T].sum() >= 1, "the compared frames must include spawned vehicles"
        finally:
            th.set_default_dtype(th.float32)
            for k in [k for k in sys.modules if k.split(".")[0] == "example"]:
                del sys.modules[k]
