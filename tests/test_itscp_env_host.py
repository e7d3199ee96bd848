"""Host side of the headless ITSCP env, trainer and log formats (no GPU): construction as run.py configures it,
observation, schedules, MacroRoute draws against the reference's stored ones, the running-mean sigmoid constants
against a restatement of common/rms.py, and that stepping refuses to run without CUDA."""
import copy
import os

import numpy as np
import pytest
import torch

from hyb_cases import fixture_case
from itscp_env_cases import c4_env, c4_fixture, c4_spawn_routes


def test_env_surface_matches_run_py_configuration():
    G = c4_fixture()
    env = c4_env(G, "cpu")
    assert env.num_timestep == 600 == int(G["T"])
    assert env.action_size() == 45 and env.action_space.shape == (45,)
    assert np.allclose(env.action_space.low, 0.1) and np.allclose(env.action_space.high, 0.9)
    assert env.observation_space.shape == (10 * 144,)            # SURVEY 8e: obs 1440 -> 256 -> 256 -> 45
    assert env.kind == G["kind"].tolist() and env.topo.ML == 16 and env.topo.NC == 256
    obs = env.observe()
    assert obs.dtype == np.float32 and obs.shape == (1440,)
    # lanes with a predecessor observe 0, boundary lanes the mean of their schedule slice (_env.py:517-535)
    o = obs.reshape(144, 10)
    bl = env.boundary
    assert len(bl) == 12 and np.abs(o[[l for l in range(144) if l not in bl]]).max() == 0
    assert np.allclose(o[bl], G["incoming"][:, bl].reshape(10, 60, -1).mean(1).T, atol=1e-6)
    assert torch.equal(env.incoming().cpu()[:, bl], torch.tensor(G["incoming"][:, bl]))
    # deep copies (trainer.py:172) share the topology and reset the counters
    env.steps = 3
    c = copy.deepcopy(env)
    assert c.topo is env.topo and c.steps == 0 and c.config == env.config and c.config is not env.config
    # every route of the fixture's spawned vehicles is known to the topology
    tab = c4_spawn_routes(G, env.topo)
    assert tab.max() < len(env.topo.routes)
    # micro mode (run_itscp_micro.sh) builds an all-micro network whose boundary lanes are waiting-list sources
    e2 = c4_env(G, "cpu", mode="micro")
    assert e2.micro_mode and e2.topo.NC == 0 and e2.topo.ML == 144 and sum(e2.topo.src) == 12


def test_no_cpu_fallback():
    G = c4_fixture()
    env = c4_env(G, "cpu")
    with pytest.raises(Exception):
        env.step(torch.full((45,), 0.5), True)


def test_signal_info_matches_batched_signals():
    G = c4_fixture()
    env = c4_env(G, "cpu")
    act = torch.tensor(G["action"])
    sig = env.grid.signals(act[None], 600, 120, soft=True)[0]
    hard = env.grid.signals(act[None], 600, 120, soft=False)[0]
    for frame in (0, 37, 119, 120, 599):
        for info, l in list(env.lane.items())[::7]:
            prev, nxt = env.lane_signal_info(info, act, frame, True)
            assert abs(float(nxt) - float(sig[frame, l])) < 1e-12
            assert float(env.lane_signal_info(info, act, frame, False)[1]) == float(hard[frame, l])
            if info.loc == "mid":
                assert float(nxt) == 1.0 and 0.0 <= float(prev) <= 1.0


def test_schedule_callbacks():
    from dhts_b200.itscp import ItscpGrid
    from dhts_b200.itscp_env import itscp_random_schedule, problem_1, problem_3
    lanes = ItscpGrid(2, 1, 5.0, 5.0).lanes
    np.random.seed(3)
    s = problem_3(lanes, 100)
    assert set(s.keys()) == set(lanes) and all(len(v) == 99 for v in s.values())     # 3 sessions of 33 frames (problem.py:14,62)
    for info, v in s.items():
        a, b, c = v[0], v[33], v[66]
        if info.loc in ("north", "south", "west", "east"):
            assert (a >= 0.9) == (c >= 0.9) != (b >= 0.9)                               # directions alternate per session
        else:
            assert max(v) <= 0.01 + 1e-12                                               # 'mid' lanes are never hot
    np.random.seed(3)
    s1 = problem_1(lanes, 60)
    ns = [v[0] >= 0.9 for i, v in s1.items() if i.loc in ("north", "south")]
    we = [v[0] >= 0.9 for i, v in s1.items() if i.loc in ("west", "east")]
    assert all(ns) != all(we) and (all(ns) or not any(ns))
    r = itscp_random_schedule(lanes, 50)
    assert all(len(v) == 50 and len(set(v)) == 5 for v in r.values())


def test_running_mean_constants_match_rms_restatement():
    from dhts_b200.itscp_env import running_mean_constants
    rng = np.random.default_rng(0)
    x = rng.normal(size=500) - 3.0
    valid = rng.uniform(size=500) < 0.7
    for window in (100_000, 37):
        data, want = [], np.zeros(500)
        for i in range(500):                      # common/rms.py:11-18 + _env.py:566-569
            if valid[i]:
                data.append(x[i]); data = data[-window:]
                want[i] = 16.0 / abs(np.mean(data))
        got = running_mean_constants(torch.tensor(x), torch.tensor(valid), 16.0, window).numpy()
        assert np.abs(got[valid] - want[valid]).max() < 1e-9 * np.abs(want).max()


def test_macro_route_draws_follow_the_reference_rng_order():
    """_make_macro_route consumes np.random exactly as ItscpRoadNetwork.create_random_macro_route does: the hybrid
    fixture's case h holds the reference's own draws on the config-4 grid, 120 frames after np.random.seed(21)
    (oracle/gen_golden_hyb.py)."""
    H = fixture_case("h")
    env = c4_env(c4_fixture(), "cpu")
    assert env.kind == H["kind"].tolist()
    env.num_timestep = int(H["T"])
    np.random.seed(21); env._make_macro_route()
    assert (env.macro_route_schedule.numpy() == H["route"]).all()


def test_trainer_log_formats(tmp_path):
    """eval.txt / model.zip / best/model.zip / scalars as trainer.py writes them, with the rollout stubbed (host logic only)."""
    from dhts_b200.control import Controller, Trainer
    G = c4_fixture()
    env = c4_env(G, "cpu")
    calls = []

    def fake_rollout(action, differentiable, **kw):
        calls.append((tuple(action.shape), differentiable))
        env.flags = type("F", (), {"check": staticmethod(lambda **k: None)})()
        return -((action.double() - 0.3) ** 2).sum(1)
    env.rollout = fake_rollout
    torch.manual_seed(0)
    tr = Trainer(env, lr=1e-2, tensorboard=False)
    assert isinstance(tr.controller, Controller)
    assert [tuple(p.shape) for p in tr.controller.parameters()] == [(256, 1440), (256,), (256, 256), (256,), (45, 256), (45,)]
    log = str(tmp_path / "trial_0")
    losses = tr.train(2, 5, 2, 1, log)
    assert len(losses) == 5 and losses[-1] < losses[0]                    # Adam descends the stub objective
    ev = open(log + "/eval.txt").read().splitlines()
    assert len(ev) == 3 and all(len(x.split(".")[1]) == 6 for x in ev)    # "{:08f}"
    assert os.path.exists(log + "/model.zip") and os.path.exists(log + "/best/model.zip")
    ck = torch.load(log + "/model.zip")
    assert set(ck.keys()) == {"controller_state_dict", "optimizer_state_dict"}
    tr2 = Trainer(env, lr=1e-2, tensorboard=False); tr2.load(log + "/model.zip")
    assert all(torch.equal(a, b) for a, b in zip(tr.controller.state_dict().values(), tr2.controller.state_dict().values()))
    assert (2, 45) in [c[0] for c in calls if c[1]] and (1, 45) in [c[0] for c in calls if not c[1]]
    import json
    sc = [json.loads(x) for x in open(log + "/scalars.jsonl")]
    assert sum(s["tag"] == "loss/train" for s in sc) == 5 and sum(s["tag"] == "loss/eval" for s in sc) == 3
    r, a, info = tr.run_episode(True)
    assert r.dim() == 0 and a.shape == (45,) and float(a.min()) >= 0.1 and float(a.max()) <= 0.9 and len(info["img"]) == 600
