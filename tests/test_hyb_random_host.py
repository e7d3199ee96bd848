"""The random hybrid-network cases of tests/hyb_random_cases.py on the CPU: every case reaches the events it is meant to
cover (judged from the reference run alone), and ``pack`` turns the initial networks into consistent kernel inputs.
tests/test_hyb_random_gpu.py compares the fused hybrid rollout with the same reference runs."""
import numpy as np
import pytest

import hyb_random_cases as H
from hyb_random_cases import DEGENERATE, RANDOM, seeds_of


def _cases():
    out = [(name, layout) for name, layout in RANDOM] + [(name, 1) for name in DEGENERATE]
    return out + [("wide", 1), ("many_sides", 1)]


@pytest.mark.parametrize("name,layout", _cases())
def test_case_reaches_its_events(name, layout):
    """Spawns, absorptions, micro -> micro hand-offs and micro_to_none drops where the spec says so, in every replica;
    both successors of a two-successor micro lane used; no collision, no CFL or NaN flag, finite gradients."""
    spec = H.SPECS[name]
    pairs = [H.reference(name, s, layout) for s in seeds_of(name, layout)]
    for case, ref in pairs:
        kinds = H.event_kinds(ref)
        assert (spec["expect"] - {"two_succ"}) <= kinds, (name, case.seed, kinds)
        assert ref.bits == 0 and ref.ncol == 0
        assert np.isfinite(ref.g_r0).all() and np.isfinite(ref.g_u0).all()
        assert all(np.isfinite(g).all() for g in ref.g_p0 + ref.g_v0)
        if case.macro:
            assert np.abs(ref.g_r0).max() > 0
        if spec.get("every_step"):
            assert len({tuple(map(tuple, r)) for r in ref.macro_route}) > 1, "the MacroRoute must change"
    if "two_succ" in spec["expect"]:
        assert H.two_successors_used(pairs), name
    if "handoff" in spec["expect"] and any(v[1] for v in spec.get("veh", {}).values()):
        # a vehicle with its own parameter set is handed from micro lane to micro lane
        case, ref = pairs[0]
        assert any(e[1] == "handoff" for e in ref.events)


@pytest.mark.parametrize("name,layout", [("branch", 1), ("micro_only", 1), ("macro_only", 1)])
def test_pack_is_self_consistent(name, layout):
    """own0 rows sit at topo.own_slot, every recorded route has a route id, aux0 counts / fronts / vehicles / parameter
    sets match the initial vehicles, spawn routes start on their lane."""
    import torch
    pairs = [H.reference(name, s, layout) for s in seeds_of(name, layout)]
    case0 = pairs[0][0]
    topo = H.topology(case0, "cpu")
    inp = H.pack(pairs, topo, "cpu")
    R, L = len(pairs), topo.L
    assert inp["r0"].shape == (R, topo.NC) and inp["aux0"].shape == (R, topo.AUX)
    for b, (case, ref) in enumerate(pairs):
        if topo.n_own:
            for (side, l), ru in case.own.items():
                assert topo.own_slot[side * L + l] >= 0
                assert np.allclose(inp["own0"][b, topo.own_slot[side * L + l]].numpy(), ru)
            assert len(case.own) == topo.n_own
        for _, l, route in ref.spawns:
            rid = topo.route_id(route)
            assert topo.routes[rid][0] == l
        aux = inp["aux0"][b].detach()
        for m, l in enumerate(topo.micro):
            rows = case.veh.get(l, [])
            assert int(aux[topo.A_CNT + m]) == len(rows) and int(aux[topo.A_FRONT + m]) == 0
            for k, (p, v, a, prm, route) in enumerate(rows):
                o = m * topo.veh_cap + k
                assert float(aux[topo.A_P + o]) == float(p) and float(aux[topo.A_V + o]) == float(v)
                assert float(aux[topo.A_A + o]) == a
                assert topo.routes[int(aux[topo.A_RID + o])] == tuple(route[:len(topo.routes[int(aux[topo.A_RID + o])])])
                assert list(inp["veh_params"][int(aux[topo.A_PID + o])]) == prm
        if inp["spawn_route"] is not None:
            sp = inp["spawn_route"][b]
            for m, l in enumerate(topo.micro):
                assert all(topo.routes[int(x)][0] == l for x in sp[m])
        route = inp["route"][b]
        assert route.shape == (ref.T, 2, L) and route.dtype == torch.int32
