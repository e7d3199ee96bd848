"""Random plain-mode hybrid networks and their CPU reference: the drop-in ``RoadNetwork`` stepped immediately, lane by lane,
with the lane kernels swapped for the oracle stand-ins of tests/cpu_standin.py.  What is left is per-lane Python -- boundary
rules, leader lookup along vehicle routes, the conversions in lane-id order (dropin/road/network/road_network.py) -- and it
shares no code with csrc/net_hybrid.cu, so it is an independent reference for the fused hybrid rollout
(``dhts_hyb_rollout_{fwd,bwd}``).

  build(seed, spec)                  one drop-in network from a spec (lane kinds and links) and a seed (sizes, states, vehicles)
  run_reference(case, T, every_step) step it T times, record every step, backpropagate a seeded positional loss
  pack(cases, topo, dev, dtype)      the INITIAL networks of R replicas as ``hybrid_rollout`` inputs
  kernel_loss(...)                   the same loss on the kernel's ``HybridStates``

The loss is positional: a seeded weight per (step, macro cell) and per (step, micro lane, rank from the head).  The kernel
carries no vehicle identity through micro -> micro hand-offs, so vehicles are compared by their rank on a lane, never by id.
fp64, plain mode only (ITSCP mode is pinned by the frozen fixtures of tests/test_hyb_gpu.py).
"""
import contextlib
import functools

import numpy as np
import torch as th

import cpu_standin

UMAX, DT, VLEN = 30.0, 0.02, 5.0
KMAX = 64                     # ranks the loss weights cover (more than any lane holds)
F64 = th.float64

# kinds: "M" = dMacroLane, "m" = dMicroLane; links in connect_lane order (a DAG: no micro cycle, so that
# HybridNetTopology's route enumeration is exact); ncell / dx / mlen override the seeded draws per lane; veh: initial
# vehicles per micro lane as (count, random parameters?); expect: events the reference run must show.
SPECS = {
    # a micro lane (1) with two micro successors (2, 5); micro -> micro hand-offs, spawns and absorptions in one conversion
    # group; macro lane 0 feeds two micro lanes (two flux capacitors); a macro merge (3, 4 -> 6) and a micro merge
    # (0, 1 -> 5); micro lane 8 has no successor (micro_to_none)
    "branch": dict(kinds="M m m M M m M M m", links=[(0, 1), (1, 2), (2, 3), (1, 5), (5, 4), (4, 6), (3, 6), (6, 7), (0, 5), (7, 8)],
                   dx={4: 2.5}, veh={1: (3, True), 8: (2, False), 5: (1, True)}, mlen={1: (40, 50), 8: (25, 35)},
                   expect={"spawn", "absorb", "handoff", "drop", "two_succ"}, T=300),
    # macro -> micro -> micro -> micro -> macro(dx 2.5) with heterogeneous initial vehicles handed from lane to lane
    "chain": dict(kinds="M m m m M", links=[(0, 1), (1, 2), (2, 3), (3, 4)], dx={4: 2.5}, ncell={4: (6, 10)},
                  veh={1: (3, True), 2: (2, True), 3: (1, True)}, mlen={1: (35, 45), 2: (25, 35), 3: (20, 30)},
                  expect={"spawn", "absorb", "handoff"}, T=300),
    # two macro lanes feed one micro lane (one capacitor each, the MacroRoute picks which one converts); the micro lane
    # splits into two micro lanes without successor
    "merge_drop": dict(kinds="M M m m m", links=[(0, 2), (1, 2), (2, 3), (2, 4)], veh={2: (3, True), 3: (1, False)},
                       mlen={2: (35, 45), 3: (15, 25), 4: (15, 25)}, expect={"spawn", "handoff", "drop", "two_succ"}, T=300),
    # the same with a new MacroRoute drawn before every step
    "merge_reroute": dict(kinds="M M m m m", links=[(0, 2), (1, 2), (2, 3), (2, 4)], veh={2: (3, True)},
                          mlen={2: (35, 45), 3: (15, 25), 4: (15, 25)}, expect={"spawn", "handoff", "drop"}, T=300,
                          every_step=True),
    # degenerate: no micro lane (ML = 0), a macro merge
    "macro_only": dict(kinds="M M M", links=[(0, 2), (1, 2)], expect=set(), T=200),
    # degenerate: no macro cell (NC = 0): initial vehicles only, hand-offs into two successors, drops
    "micro_only": dict(kinds="m m m m", links=[(0, 1), (1, 2), (1, 3)], veh={0: (3, True), 1: (2, True)},
                       mlen={0: (35, 45), 1: (25, 35), 2: (15, 20), 3: (15, 20)}, expect={"handoff", "drop", "two_succ"}, T=200),
    "single_micro": dict(kinds="m", links=[], veh={0: (4, True)}, mlen={0: (40, 50)}, expect={"drop"}, T=200),
    "single_macro": dict(kinds="M", links=[], expect=set(), T=200),
    # launch shapes of dhts_hyb_rollout_*: about 260 macro cells (more than 192 interfaces: the 512-thread adjoint)
    "wide": dict(kinds="M m M M m M", links=[(0, 1), (1, 2), (2, 3), (3, 4), (4, 5)], ncell={0: (60, 70), 2: (60, 70), 3: (60, 70), 5: (60, 70)},
                 veh={1: (2, True), 4: (2, True)}, mlen={1: (30, 40), 4: (30, 40)}, expect={"spawn", "absorb"}, T=150),
    # 24 short lanes: the (side, lane) pairs (2 L + ML = 60) outnumber the interfaces, so the thread count is set by sides
    "many_sides": dict(kinds=" ".join(["M m"] * 12), links=[(i, i + 1) for i in range(23)], ncell={2 * i: (1, 2) for i in range(12)},
                       veh={2 * i + 1: (1, True) for i in range(12)}, mlen={2 * i + 1: (20, 30) for i in range(12)},
                       expect={"spawn", "absorb"}, T=40),
    # about 1500 macro cells: the fp64 adjoint fits in shared memory only without prefetch
    "big": dict(kinds="M m M", links=[(0, 1), (1, 2)], ncell={0: (740, 750), 2: (740, 750)}, veh={1: (2, True)},
                mlen={1: (30, 40)}, expect=set(), T=20),
    # about 2000 macro cells: the forward fits, the adjoint does not even without prefetch
    "huge": dict(kinds="M m M", links=[(0, 1), (1, 2)], ncell={0: (1000, 1010), 2: (1000, 1010)}, veh={1: (2, True)},
                 mlen={1: (30, 40)}, expect=set(), T=20),
}

# the random networks and the degenerate ones the GPU tests compare: (spec, layout seed); replica b has seed layout + 100 b
RANDOM = [("branch", 1), ("branch", 7), ("chain", 3), ("merge_drop", 4), ("merge_reroute", 5), ("chain", 6)]
DEGENERATE = ["macro_only", "micro_only", "single_micro", "single_macro"]


def seeds_of(name, layout, R=3):
    return [layout + 100 * b for b in range(R)]


@contextlib.contextmanager
def standin():
    """The drop-in API on the CPU stand-ins, every step run at once (no deferral), fp64."""
    from dhts_b200.dropin import runtime as rt
    with cpu_standin.patched("float64"):
        saved = rt._cfg["defer"]
        rt.configure(defer=False)
        try:
            yield
        finally:
            rt.configure(defer=saved)


class Case:
    """A drop-in network plus a record of its initial state (the leaves the gradients are taken against)."""

    def __init__(self, net, spec, seed, macro, micro, leaves, own, caps, veh):
        self.net, self.spec, self.seed = net, spec, seed
        self.macro, self.micro = macro, micro            # lane ids
        self.leaves = leaves                             # macro lane id -> (r, u) leaves
        self.own = own                                   # (side, lane) -> (r, u) of its own ghost record
        self.caps = caps                                 # (macro lane, micro lane) -> initial capacitor
        self.veh = veh                                   # micro lane id -> [(p leaf, v leaf, a, params[6], route list)] head first


def _spec(spec):
    return SPECS[spec] if isinstance(spec, str) else spec


def build(seed, spec, layout=None):
    """One drop-in RoadNetwork (call inside ``standin()``).  ``layout`` (default: the seed) draws cell counts, dx in
    {2.5, 5, 7} and micro lane lengths, so replicas of one network share it; the seed draws initial macro states, own
    ghost records, initial capacitors and the initial vehicles, and seeds ``np.random``, which the reference draws
    routes, MacroRoutes and random vehicles from."""
    from road.lane.dmacro_lane import dMacroLane
    from road.lane.dmicro_lane import dMicroLane
    from road.network.road_network import RoadNetwork
    from road.vehicle.micro_vehicle import MicroVehicle
    sp = _spec(spec)
    rng = np.random.default_rng(seed)
    lay = np.random.default_rng(seed if layout is None else layout)
    np.random.seed(seed)
    kinds = sp["kinds"].split()
    net = RoadNetwork(UMAX)
    leaves, macro, micro = {}, [], []
    for i, k in enumerate(kinds):
        if k == "M":
            lo, hi = sp.get("ncell", {}).get(i, (3, 9))
            n = int(lay.integers(lo, hi + 1))
            dx = float(sp.get("dx", {}).get(i, lay.choice([2.5, 5.0, 7.0])))
            lane = dMacroLane(i, n * dx, UMAX, dx)
            r = th.tensor(rng.uniform(0.15, 0.7, n), dtype=F64, requires_grad=True)
            u = th.tensor(rng.uniform(8.0, 22.0, n), dtype=F64, requires_grad=True)
            lane.set_state_vector_u(r, u)
            leaves[i] = (r, u)
            macro.append(i)
        else:
            lo, hi = sp.get("mlen", {}).get(i, (30, 50))
            lane = dMicroLane(i, float(lay.uniform(lo, hi)), UMAX)
            micro.append(i)
        net.add_lane(lane)
    for a, b in sp["links"]:
        net.connect_lane(a, b)
    own = {}
    for i in macro:
        lane = net.lane[i]
        for side, adj in ((0, lane.prev_lane), (1, lane.next_lane)):
            if not adj or any(x.is_micro() for x in adj.values()):
                rg, ug = float(rng.uniform(0.1, 0.6)), float(rng.uniform(5.0, 25.0))
                (lane.set_leftmost_cell if side == 0 else lane.set_rightmost_cell)(rg, ug)
                own[(side, i)] = (rg, ug)
    caps = {}
    for i in macro:
        for j in net.lane[i].next_lane:
            if net.lane[j].is_micro():
                caps[(i, j)] = float(rng.uniform(0.0, 4.0))
                net.lane[i].flux_capacitor[j] = caps[(i, j)]
    veh = {}
    for i in micro:
        n, rnd = sp.get("veh", {}).get(i, (0, False))
        length = float(net.lane[i].length)
        pos, x = [], length - float(rng.uniform(1.0, 4.0))
        for _ in range(n):
            pos.append(x)
            x -= float(rng.uniform(11.0, 15.0))
        assert not pos or pos[-1] >= 0, "lane %d too short for its initial vehicles" % i
        rows = []
        for k, x in enumerate(pos):                                   # head first
            mv = MicroVehicle.random_micro_vehicle(UMAX) if rnd and k % 3 != 2 else MicroVehicle.default_micro_vehicle(UMAX)
            mv.position = th.tensor(x, dtype=F64, requires_grad=True)
            mv.speed = th.tensor(float(rng.uniform(6.0, 14.0)), dtype=F64, requires_grad=True)
            route = net.create_random_route(i)
            net.add_vehicle(mv, route)
            rows.append((mv.position, mv.speed, float(mv.a), mv.idm_params(), list(route.route)))
        veh[i] = rows
    return Case(net, sp, seed, macro, micro, leaves, own, caps, veh)


@functools.lru_cache(maxsize=None)
def loss_weights(seed, T, NC, ML):
    """Seeded weights of the positional loss, at steps T/3, 2T/3 and T."""
    rng = np.random.default_rng(1000 + seed)
    steps = sorted({max(1, T // 3), max(1, 2 * T // 3), T})
    return {s: (rng.normal(size=(2, NC)), rng.normal(size=(2, ML, KMAX))) for s in steps}


class Ref:
    """What the reference did, per step t = 0..T (the state after t steps)."""


def run_reference(case, T, every_step=False):
    """Step ``case.net`` T times (call inside ``standin()``), recording per step the macro cells (r, y, u), the vehicle
    count of every micro lane, the flux capacitors, the vehicles head first (p, v, a), the routes the reference drew
    for every spawned vehicle and the MacroRoute of every step; classify every vehicle event; then backpropagate the
    seeded positional loss into the initial macro states and vehicles."""
    from dhts_b200.dropin import runtime as rt
    net, macro, micro = case.net, case.macro, case.micro
    lanes = net.lane
    L = len(lanes)
    cap_pairs = [(a, b) for a in macro for b in lanes[a].next_lane if lanes[b].is_micro()]
    ref = Ref()
    ref.T = T
    ref.cells, ref.count, ref.capac, ref.veh, ref.macro_route = [], [], [], [], []
    ref.spawns = []                     # (step, lane, route) in spawn order (vehicle id order)
    ref.events = []                     # (step, kind, from lane, to lane)
    ref.bits, ref.ncol = 0, 0
    cells_t, veh_t = [], []

    def record():
        cs = [th.stack([lanes[l]._vec("curr", k) for k in ("r", "y", "u")]) for l in macro]
        cells = th.cat(cs, dim=1) if cs else th.zeros((3, 0), dtype=F64)
        cells_t.append(cells)
        ref.cells.append(cells.detach().numpy().copy())
        ref.count.append([lanes[l].num_vehicle() for l in micro])
        c = [lanes[a].flux_capacitor.get(b, 0.0) for a, b in cap_pairs]
        ref.capac.append([float(x.detach()) if th.is_tensor(x) else float(x) for x in c])
        vs = []
        for l in micro:
            vs.append([(mv.position, mv.speed, mv.a) for mv in reversed(lanes[l].curr_vehicle)])
        veh_t.append(vs)
        f = lambda x: float(x.detach()) if th.is_tensor(x) else float(x)
        ref.veh.append([[(f(p), f(v), f(a)) for p, v, a in lane] for lane in vs])

    def where():
        return {mv.id: l for l in micro for mv in lanes[l].curr_vehicle}

    orig_check = rt.check_flags

    def check_flags():                  # remember what the stand-ins flagged before the step clears it
        for fl in rt._flags.values():
            b, n = fl.read()
            ref.bits |= b
            ref.ncol += n
        orig_check()

    record()
    before = where()
    rt.check_flags = check_flags
    try:
        for t in range(1, T + 1):
            if every_step or t == 1:
                net.macro_route = net.create_random_macro_route()
            mr = net.macro_route
            ref.macro_route.append(([mr.get_prev_lane(l) for l in range(L)], [mr.get_next_lane(l) for l in range(L)]))
            n0 = net.num_vehicle
            net.forward(DT, True)
            for vid in range(n0, net.num_vehicle):
                route = list(net.micro_route[vid].route)
                ref.spawns.append((t, route[0], route))
                ref.events.append((t, "spawn", -1, route[0]))
            now = where()
            for vid, l in before.items():
                if vid in now:
                    if now[vid] != l:
                        ref.events.append((t, "handoff", l, now[vid]))
                else:
                    nxt = net.micro_route[vid].next_lane_id()
                    ref.events.append((t, "drop" if nxt == -1 else "absorb", l, nxt))
            before = now
            record()
    finally:
        rt.check_flags = orig_check
    ref.count, ref.capac = np.array(ref.count).reshape(T + 1, len(micro)), np.array(ref.capac).reshape(T + 1, len(cap_pairs))
    ref.cap_pairs = cap_pairs
    # ---- positional loss and its gradients
    W = loss_weights(case.seed, T, ref.cells[0].shape[1], len(micro))
    loss = th.zeros((), dtype=F64)
    for s, (wc, wv) in W.items():
        c = cells_t[s]
        loss = loss + (c[0] * th.tensor(wc[0])).sum() + (c[2] * th.tensor(wc[1]) / UMAX).sum()
        for m, lane in enumerate(veh_t[s]):
            for k, (p, v, a) in enumerate(lane):
                loss = loss + 0.01 * (float(wv[0, m, k]) * p + float(wv[1, m, k]) * v)
    ref.loss = float(loss.detach())
    leaves = [x for l in macro for x in case.leaves[l]] + [x for l in micro for row in case.veh[l] for x in row[:2]]
    loss.backward(inputs=leaves)
    g = lambda x: 0.0 if x.grad is None else x.grad.numpy().copy()
    ref.g_r0 = np.concatenate([np.broadcast_to(g(case.leaves[l][0]), case.leaves[l][0].shape) for l in macro]) if macro else np.zeros(0)
    ref.g_u0 = np.concatenate([np.broadcast_to(g(case.leaves[l][1]), case.leaves[l][1].shape) for l in macro]) if macro else np.zeros(0)
    ref.g_p0 = [[float(g(row[0])) for row in case.veh[l]] for l in micro]
    ref.g_v0 = [[float(g(row[1])) for row in case.veh[l]] for l in micro]
    return ref


@functools.lru_cache(maxsize=None)
def reference(spec_name, seed, layout=None, T=None):
    """(case, ref) of a named spec, cached per process."""
    sp = SPECS[spec_name]
    with standin():
        case = build(seed, spec_name, layout)
        ref = run_reference(case, T or sp["T"], sp.get("every_step", False))
    return case, ref


def veh_cap(case, extra=6):
    longest = max([float(case.net.lane[l].length) for l in case.micro] or [0.0])
    return int(longest / VLEN) + extra


def topology(case, dev, cap=None):
    from dhts_b200.hybrid_network import HybridNetTopology
    from dhts_b200.network import MODE_PLAIN
    return HybridNetTopology.from_network(case.net, dev, MODE_PLAIN, veh_cap=cap or veh_cap(case))


def pack(pairs, topo, dev, dtype=F64, KS=None):
    """``hybrid_rollout`` inputs of R replicas, one per (case, ref) pair, all of the same spec: every replica its own
    initial state, vehicles (counts, routes, parameter sets), MacroRoute per step ([R, T, 2, L]) and spawn routes
    ([R, ML, KS], the routes its reference drew, in spawn order).  p0 / v0 are leaves [R, ML, cap], head first."""
    from dhts_b200.hybrid_network import default_vehicle_params
    R, ML, cap, L = len(pairs), topo.ML, topo.veh_cap, topo.L
    T = pairs[0][1].T
    t = lambda a: th.tensor(np.asarray(a, dtype=np.float64), dtype=dtype, device=dev)
    r0 = t([np.concatenate([c.leaves[l][0].detach().numpy() for l in c.macro]) if c.macro else np.zeros(0) for c, _ in pairs])
    u0 = t([np.concatenate([c.leaves[l][1].detach().numpy() for l in c.macro]) if c.macro else np.zeros(0) for c, _ in pairs])
    r0 = r0.reshape(R, topo.NC).requires_grad_(); u0 = u0.reshape(R, topo.NC).requires_grad_()
    own = np.zeros((R, max(topo.n_own, 1), 2))
    for b, (c, _) in enumerate(pairs):
        for (side, l), ru in c.own.items():
            own[b, topo.own_slot[side * L + l]] = ru
    own0 = t(own[:, :topo.n_own]) if topo.n_own else None
    par = [default_vehicle_params(UMAX, VLEN)]
    p0, v0, a0 = np.zeros((R, ML, cap)), np.zeros((R, ML, cap)), np.zeros((R, ML, cap))
    rid, pid, cnt = np.zeros((R, ML, cap)), np.zeros((R, ML, cap)), np.zeros((R, ML))
    capac = np.zeros((R, topo.NCAP))
    pairs_cap = [(l, topo.cap_lane[j]) for l in range(L) for j in range(topo.cap_off[l], topo.cap_off[l + 1])]
    for b, (c, _) in enumerate(pairs):
        for m, l in enumerate(topo.micro):
            rows = c.veh.get(l, [])
            cnt[b, m] = len(rows)
            for k, (p, v, a, prm, route) in enumerate(rows):
                p0[b, m, k], v0[b, m, k], a0[b, m, k] = float(p), float(v), a
                rid[b, m, k] = topo.route_id(route)
                if prm == par[0]:
                    pid[b, m, k] = 0
                else:
                    pid[b, m, k] = len(par); par.append(prm)
        for j, key in enumerate(pairs_cap):
            capac[b, j] = c.caps[key]
    tp0, tv0 = t(p0).requires_grad_(), t(v0).requires_grad_()
    aux0 = th.cat([topo.make_aux0(1, dtype, tp0[b:b + 1], tv0[b:b + 1], t(a0[b:b + 1]), rid[b], cnt[b], t(capac[b:b + 1]),
                                  pid0=pid[b]) for b in range(R)])
    route = th.tensor(np.array([ref.macro_route for _, ref in pairs]), dtype=th.int32, device=dev)     # [R, T, 2, L]
    sp = None
    if ML:
        n_sp = [[sum(1 for s in ref.spawns if s[1] == l) for l in topo.micro] for _, ref in pairs]
        KS = KS or max(2, max(max(x) for x in n_sp) + 2)
        first = {l: min(i for i, r in enumerate(topo.routes) if r[0] == l) for l in topo.micro}
        sp = np.array([[[first[l]] * KS for l in topo.micro] for _ in pairs], dtype=np.int32)
        for b, (_, ref) in enumerate(pairs):
            k = {l: 0 for l in topo.micro}
            for _, l, r in ref.spawns:
                if k[l] < KS:
                    sp[b, topo.mic_of[l], k[l]] = topo.route_id(r)
                k[l] += 1
        sp = th.tensor(sp, device=dev)
    return dict(r0=r0, u0=u0, own0=own0, aux0=aux0, p0=tp0, v0=tv0, veh_params=np.array(par), route=route, spawn_route=sp,
                T=T, R=R)


def kernel_loss(st, pairs, T):
    """The reference's positional loss of every replica on the kernel's HybridStates (cells, and vehicles by rank)."""
    topo = st.topo
    dev, dtype, cap = st.hist.device, st.hist.dtype, topo.veh_cap
    Ws = [loss_weights(case.seed, T, topo.NC, topo.ML) for case, _ in pairs]
    loss = th.zeros((), dtype=dtype, device=dev)
    p, v, _, valid = st.by_rank() if topo.ML else (None,) * 4
    for s in Ws[0]:
        wc = th.tensor(np.stack([W[s][0] for W in Ws]), dtype=dtype, device=dev)                  # [R, 2, NC]
        loss = loss + (st.cells[s, :, 0] * wc[:, 0]).sum() + (st.cells[s, :, 2] * wc[:, 1] / UMAX).sum()
        if topo.ML:
            wv = th.tensor(np.stack([W[s][1][:, :, :cap] for W in Ws]), dtype=dtype, device=dev)   # [R, 2, ML, cap]
            vm = valid[s]
            loss = loss + 0.01 * (th.where(vm, p[s] * wv[:, 0], 0).sum() + th.where(vm, v[s] * wv[:, 1], 0).sum())
    return loss


def event_kinds(ref):
    return {e[1] for e in ref.events}


def two_successors_used(pairs):
    """True when, for every micro lane with two or more successors, vehicles left it into each of them in one of the
    replicas (case, ref) of a network."""
    case = pairs[0][0]
    lanes = case.net.lane
    for l in case.micro:
        succ = list(lanes[l].next_lane.keys())
        if len(succ) >= 2:
            used = {e[3] for _, ref in pairs for e in ref.events if e[2] == l and e[1] in ("handoff", "absorb")}
            if not set(succ) <= used:
                return False
    return True
