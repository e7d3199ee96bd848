"""Shared pieces of the hybrid-network tests: load the live-reference ITSCP hybrid fixtures
(oracle/gen_golden_hyb.py) and run the fused hybrid rollout on them."""
import numpy as np
import torch

from conftest import golden

F64 = torch.float64


def fixture_case(tag):
    g = golden("itscp_hybrid_%s_fp64" % tag)
    G = {k: g[k] for k in g.files}
    G["hist"] = np.concatenate([golden("itscp_hybrid_%s_hist%d_fp64" % (tag, i))["hist"] for i in (0, 1)])
    return G


def t64(a, dev, grad=False):
    t = torch.tensor(np.asarray(a, dtype=np.float64), dtype=F64, device=dev)
    return t.requires_grad_() if grad else t


def build(G, dev, veh_cap=4):
    from dhts_b200.hybrid_network import HybridNetTopology
    from dhts_b200.itscp import ItscpGrid
    from dhts_b200.network import MODE_ITSCP
    grid = ItscpGrid(int(G["num_intersection"]), int(G["num_lane"]), float(G["lane_length"]), float(G["cell_length"]))
    topo = HybridNetTopology(G["kind"].tolist(), grid.num_cell, grid.dx, [l.length for l in grid.lanes], grid.links, dev,
                             MODE_ITSCP, veh_cap=veh_cap, veh_len=float(G["veh_len"]))
    return grid, topo


def spawn_routes(G, topo, max_spawn=16):
    """Routes the reference drew, per entry lane in spawn order (vehicle ids are handed out in spawn order)."""
    tab = np.zeros((topo.ML, max_spawn), dtype=np.int32)
    nsp = [0] * topo.ML
    vroute = G["vroute"]
    nveh = int((G["vid"].max() + 1)) if G["vid"].size else 0
    for v in range(nveh):
        path = [int(x) for x in vroute[v] if x >= 0]
        m = topo.mic_of[path[0]]
        tab[m, nsp[m]] = topo.route_id(path)
        nsp[m] += 1
    return tab


def run_fixture(G, dev, soft=True):
    """action -> signals -> fused hybrid rollout -> queue reward (fixture constants) + terminal term -> gradients."""
    from dhts_b200 import Flags
    from dhts_b200.hybrid_network import hybrid_rollout
    grid, topo = build(G, dev)
    T, umax, dt = int(G["T"]), float(G["umax"]), float(G["dt"])
    action = t64(G["action"][None], dev, True)
    sig = grid.signals(action, T, int(G["frames_per_signal"]), soft=soft)
    sig.retain_grad()
    inc = t64(G["incoming"][None], dev, True)
    r0 = t64(G["r0"][None], dev, True); u0 = t64(G["u0"][None], dev, True)
    route = torch.tensor(G["route"], dtype=torch.int32, device=dev)
    sp = torch.tensor(spawn_routes(G, topo), dtype=torch.int32, device=dev)
    flags = Flags(dev)
    st = hybrid_rollout(topo, r0, u0, umax, dt, T, sig=sig, incoming=inc, route=route, spawn_route=sp, soft=soft, flags=flags)
    p, v, a, valid = st.by_rank()
    # queue reward (_env.py:662-742) with the fixture's running-mean constants
    static = float(G["static_speed"])
    cells = st.cells
    r = cells[1:, 0, 0]; u = cells[1:, 0, 2]                         # [T, NC]
    kc = t64(G["kcell"], dev); kv = t64(G["kveh"], dev)
    w = (topo.real("dx", F64)[topo.lane_of_cell()] / float(G["veh_len"]))
    per_cell = torch.sigmoid(torch.clamp((static - u) * kc, -16, 16)) * r * w
    q = torch.zeros((T, topo.L), dtype=F64, device=dev).index_add(1, topo.lane_of_cell(), per_cell)
    vv = v[1:, 0]                                                    # [T, ML, cap]
    per_veh = torch.sigmoid(torch.clamp((static - vv) * kv, -16, 16)) * valid[1:, 0].to(F64)
    mic = torch.tensor(topo.micro, device=dev)
    q = q.index_add(1, mic, per_veh.sum(-1))
    reward = -(q ** 2.0).sum() * dt
    wv = t64(G["w_veh"], dev)
    vm = valid[T, 0].to(F64)
    term = (cells[T, 0, 0] * t64(G["w_r"], dev)).sum() + (cells[T, 0, 2] * t64(G["w_u"], dev)).sum() + \
        ((p[T, 0] * wv[..., 0] + v[T, 0] * wv[..., 1] + a[T, 0] * wv[..., 2]) * vm).sum()
    return dict(grid=grid, topo=topo, st=st, action=action, sig=sig, inc=inc, r0=r0, u0=u0, reward=reward, term=term,
                flags=flags, p=p, v=v, a=a, valid=valid)
