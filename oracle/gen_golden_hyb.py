"""TEST INFRASTRUCTURE: freeze outputs of the LIVE reference's ITSCP network in HYBRID mode into tests/golden/.

Run in THIS container only (needs /root/reference):

    python oracle/gen_golden_hyb.py            # fp64 tier (dtype-proxied reference, SURVEY 8c tier 2)

Same approach as oracle/gen_golden_net.py (the reference's ``ItscpRoadNetwork`` and lanes are imported unmodified,
the pieces of ``_env.py`` that drive them are restated here): lanes of interior intersections are ``dMicroLane``s,
all others ``dMacroLane``s (_env.py:490-500), so one frame exercises the signal-blended ghost cells, the IDM lanes
with the signal-blended head deltas (_simulator.py:144-276), the cross-lane leader lookup
(road_network.py:429-580) and every conversion (conversion.py:15-215) in lane-id order.

The routes ``create_random_route`` draws for spawned vehicles (road_network.py:604-646) are random INPUTS: they are
recorded per vehicle, in spawn order per entry lane, and handed to the kernels as such.

Fixture: tests/golden/itscp_hybrid_<case>_fp64.npz (+ _hist0 / _hist1, see save_case).
"""
import os
import sys

import numpy as np
import torch as th

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REF = os.environ.get("DHTS_REFERENCE", "/root/reference")
OUT = os.path.join(ROOT, "tests", "golden")
sys.path.insert(0, REF)
sys.path.insert(1, ROOT)
sys.path.insert(2, HERE)

from gen_golden import switch_fp64  # noqa: E402
from gen_golden_net import load_reference_simulator, f  # noqa: E402

CAP = 4          # vehicles recorded per micro lane (asserted below)
RLEN = 32        # MAX_ROUTE_LENGTH, road_network.py:15


def run_case(tag, grid, T, frames_per_signal, seed, umax=60.0, freq=30, static_speed=0.2, inflow=(0.2, 0.9), empty=False,
             schedule=None, action_range=(0.1, 0.9)):
    from dmath.operation import sigmoid
    from road.lane.dmacro_lane import dMacroLane
    from road.lane.dmicro_lane import dMicroLane
    ItscpRoadNetwork, RunningMean = load_reference_simulator()

    class _NP64:
        float32 = np.float64

        def __getattr__(self, k):
            return getattr(np, k)
    sys.modules["example.common.rms"].np = _NP64()      # RunningMean accumulates in the state dtype
    rng = np.random.default_rng(seed)
    np.random.seed(seed)
    dt = 1.0 / freq
    n = grid.num_intersection
    net = ItscpRoadNetwork(umax)
    kind = []
    for info in grid.lanes:
        interior = not (info.row == 0 or info.row == n - 1 or info.col == 0 or info.col == n - 1)
        if interior:
            net.add_lane(dMicroLane(len(net.lane), info.length, umax)); kind.append(1)
        else:
            net.add_lane(dMacroLane(len(net.lane), info.length, umax, grid.cell_length)); kind.append(0)
    for a, b in grid.links:
        net.connect_lane(a, b)
    L = grid.L
    kind = np.array(kind, dtype=np.int32)
    mic = [l for l in range(L) if kind[l]]
    mic_idx = {l: i for i, l in enumerate(mic)}
    ML = len(mic)
    ncell = [0 if kind[l] else net.lane[l].num_cell for l in range(L)]
    off = np.concatenate([[0], np.cumsum(ncell)]).astype(int)
    NC = int(off[-1])
    n2 = n * n
    n_phase = max(1, T // frames_per_signal)
    action = th.tensor(rng.uniform(action_range[0], action_range[1], n_phase * n2), requires_grad=True)
    bl = grid.boundary_lanes()
    assert all(kind[l] == 0 for l in bl)
    inc_np = np.zeros((T, L))
    if schedule is not None:      # an _env.py schedule callback restated by the caller (lane infos, T) -> [T, L]
        full = schedule(grid.lanes, T)
        for l in bl:
            inc_np[:, l] = full[:, l]
    else:
        for l in bl:
            for s0 in range(0, T, max(1, T // 5)):
                inc_np[s0:s0 + max(1, T // 5), l] = rng.uniform(*inflow)
    inc = {(t, l): th.tensor(inc_np[t, l], requires_grad=True) for t in range(T) for l in bl}
    routes = [net.create_random_macro_route() for _ in range(T)]       # macro_route_schedule, _env.py:194-200
    route_tab = np.array([[[r.get_prev_lane(l) for l in range(L)], [r.get_next_lane(l) for l in range(L)]] for r in routes],
                         dtype=np.int32)
    r0_np = rng.uniform(0.1, 0.8, NC); u0_np = rng.uniform(0.3, 1.0, NC) * umax * (1.0 - 0.7 * r0_np)
    if empty:                     # lanes as _make_lane leaves them: ARZ.FullQ(u_max), model/macro/_arz.py:59-63
        r0_np = np.zeros(NC); u0_np = np.full(NC, umax)
    r0 = th.tensor(r0_np, requires_grad=True); u0 = th.tensor(u0_np, requires_grad=True)
    for l in range(L):
        if not kind[l]:
            net.lane[l].set_state_vector_u(r0[off[l]:off[l + 1]], u0[off[l]:off[l + 1]])
    rms = RunningMean(100_000)
    sig_t = {}
    hist = np.zeros((T + 1, 3, NC)); sig_np = np.ones((T, L))
    kcell = np.zeros((T, NC)); kveh = np.zeros((T, ML, CAP))
    veh = np.zeros((T + 1, ML, CAP, 3)); vcnt = np.zeros((T + 1, ML), dtype=np.int32); vid = -np.ones((T + 1, ML, CAP), dtype=np.int32)
    head = np.zeros((T, ML, 2))
    reward = 0

    def snapshot(t):
        for l in range(L):
            if kind[l]:
                lane = net.lane[l]; m = mic_idx[l]
                assert lane.num_vehicle() <= CAP, "raise CAP"
                vcnt[t, m] = lane.num_vehicle()
                for j, mv in enumerate(reversed(lane.curr_vehicle)):      # front (head) first
                    veh[t, m, j] = (f(mv.position), f(mv.speed), f(mv.a)); vid[t, m, j] = mv.id
            else:
                for i, c in enumerate(net.lane[l].curr_cell):
                    hist[t, 0, off[l] + i] = f(c.state.q.r); hist[t, 1, off[l] + i] = f(c.state.q.y); hist[t, 2, off[l] + i] = f(c.state.u)

    snapshot(0)
    for t in range(T):
        phase = min(t // frames_per_signal, n_phase - 1)
        progress = min((t % frames_per_signal) / frames_per_signal, 1.0)
        for l, info in enumerate(grid.lanes):
            if info.loc == "mid" or not info.approaching:
                s = 1.0
            else:
                a = action[phase * n2 + info.row * n + info.col]
                s = sigmoid(a - progress, constant=32) if info.loc in ("west", "east") else sigmoid(progress - a, constant=32)
                s.retain_grad(); sig_t[(t, l)] = s
                sig_np[t, l] = f(s)
            net.lane_signal[l] = s
            net.lane_incoming[l] = inc[(t, l)] if l in bl else -1
        net.macro_route = routes[t]
        net.forward(dt, True)
        for l in mic:      # head deltas the IDM step just used (set by setup_micro_boundary)
            head[t, mic_idx[l]] = (f(net.lane[l].head_position_delta), f(net.lane[l].head_speed_delta))
        snapshot(t + 1)
        # queue length (_env.py:662-742): cells of macro lanes, vehicles of micro lanes, lanes in id order
        for l in range(L):
            lane = net.lane[l]
            q = 0
            if kind[l]:
                for j, mv in enumerate(lane.curr_vehicle):                # tail first, as the reference iterates
                    speed = mv.speed if isinstance(mv.speed, th.Tensor) else th.tensor(mv.speed)
                    with th.no_grad():
                        rms.update((static_speed - speed).cpu().numpy())
                        constant = 16.0 / np.abs(rms.mean())
                    kveh[t, mic_idx[l], lane.num_vehicle() - 1 - j] = constant
                    q = q + sigmoid(static_speed - speed, constant=constant)
            else:
                for i, c in enumerate(lane.curr_cell):
                    speed = c.state.u if isinstance(c.state.u, th.Tensor) else th.tensor(c.state.u)
                    with th.no_grad():
                        rms.update((static_speed - speed).cpu().numpy())
                        constant = 16.0 / np.abs(rms.mean())
                    kcell[t, off[l] + i] = constant
                    q = q + sigmoid(static_speed - speed, constant=constant) * (c.state.q.r * lane.cell_length / net.vehicle_length)
            reward = reward + (-1.0) * ((q ** 2.0) * dt)
    w_r = rng.normal(size=NC); w_u = rng.normal(size=NC) / umax
    w_veh = rng.normal(size=(ML, CAP, 3)) * np.array([0.02, 0.02, 0.2])
    term = 0
    for l in range(L):
        if kind[l]:
            for j, mv in enumerate(reversed(net.lane[l].curr_vehicle)):
                w = w_veh[mic_idx[l], j]
                term = term + w[0] * mv.position + w[1] * mv.speed + w[2] * mv.a
        else:
            for i, c in enumerate(net.lane[l].curr_cell):
                term = term + w_r[off[l] + i] * c.state.q.r + w_u[off[l] + i] * c.state.u
    loss = reward + term
    loss.backward()
    g_sig = np.zeros((T, L)); g_inc = np.zeros((T, L))
    for (t, l), s in sig_t.items():
        g_sig[t, l] = 0.0 if s.grad is None else f(s.grad)
    for (t, l), x in inc.items():
        g_inc[t, l] = 0.0 if x.grad is None else f(x.grad)
    nveh = net.num_vehicle
    vroute = -np.ones((max(nveh, 1), RLEN), dtype=np.int32)
    for v in range(nveh):
        rt = net.micro_route[v].route
        vroute[v, :len(rt)] = rt
    out = dict(T=T, frames_per_signal=frames_per_signal, umax=umax, dt=dt, veh_len=net.vehicle_length, static_speed=static_speed,
               num_intersection=n, num_lane=grid.num_lane, lane_length=grid.lane_length, cell_length=grid.cell_length,
               kind=kind, action=action.detach().numpy(), incoming=inc_np, route=route_tab, r0=r0_np, u0=u0_np, hist=hist,
               veh=veh, vcnt=vcnt, vid=vid, head=head, vroute=vroute, kcell=kcell, kveh=kveh, sig=sig_np, reward=f(reward),
               term=f(term), w_r=w_r, w_u=w_u, w_veh=w_veh, g_action=action.grad.numpy(), g_sig=g_sig, g_inc=g_inc,
               g_r0=r0.grad.numpy(), g_u0=u0.grad.numpy())
    moved = int(((vid[1:, :, 0] != vid[:-1, :, 0]) & (vid[:-1, :, 0] >= 0)).sum())
    print(tag, "L", L, "micro", ML, "NC", NC, "T", T, "vehicles spawned", nveh, "front changes", moved, "max on lane", vcnt.max(),
          "reward %.6g term %.6g |g_action| %.3g |g_r0| %.3g |g_inc| %.3g" %
          (out["reward"], out["term"], np.abs(out["g_action"]).max(), np.abs(out["g_r0"]).max(), np.abs(g_inc).max()))
    return {tag + "_" + k: v for k, v in out.items()}


def main():
    switch_fp64()
    from dhts_b200.itscp import ItscpGrid
    out = {}
    T = int(os.environ.get("HYB_T", "120"))
    out.update(run_case("h", ItscpGrid(3, 1, 5.0, 5.0), T=T, frames_per_signal=30, seed=21))          # C4's geometry
    out.update(run_case("g", ItscpGrid(3, 1, 20.0, 5.0), T=T, frames_per_signal=24, seed=22))         # longer access lanes
    os.makedirs(OUT, exist_ok=True)
    for tag in ("h", "g"):
        save_case(tag, {k[2:]: v for k, v in out.items() if k.startswith(tag + "_")})


def save_case(tag, case):
    """itscp_hybrid_<tag>_fp64.npz plus the state history in two halves along the frames, _hist0 / _hist1: every
    stored file stays under 1 MB (tests/hyb_cases.fixture_case joins them)."""
    hist = case.pop("hist")
    half = (len(hist) + 1) // 2
    for name, arrays in (("", case), ("_hist0", {"hist": hist[:half]}), ("_hist1", {"hist": hist[half:]})):
        path = os.path.join(OUT, "itscp_hybrid_%s%s_fp64.npz" % (tag, name))
        np.savez_compressed(path, **arrays)
        print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
