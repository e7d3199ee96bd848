#!/usr/bin/env python
"""Headline benchmark: fwd+bwd cell-updates/s (ARZ) and vehicle-updates/s (IDM) on the synthetic batch of
BASELINE.json configs[4]: 65536 independent ARZ lanes x 1024 cells + 4,194,304 IDM vehicles (65536 lanes x 64),
1000 simulation steps forward + adjoint.

One bench "step" = one full pass of the hot path over that batch: ARZ rollout fwd + loss + adjoint, IDM
rollout fwd + loss + adjoint (one update = one cell / vehicle advanced one simulation step forward AND its
adjoint propagated one step back, SURVEY 8d).  Lanes are independent, so ranks hold shards and the only
collective is one all-reduce of the scalar losses per pass.  Two splits are timed under torchrun:

  * weak   (`value`, `e2e`): every rank runs its OWN 65536-lane batch (seed = SEED + rank);
  * strong (`strong`): the ONE global batch of configs[4] (seed = SEED) is cut into N contiguous lane blocks, one
    per rank, so the whole job is the N = 1 job and the results are independent of N (checked bitwise on
    sampled lanes).

    python bench.py [--gpus N] [--steps K] [--warmup W]             # our CUDA path
    python bench.py --impl reference ...                            # CPU arm (oracle port + the live Python reference)

Prints ONE JSON line (rank 0).  DESIGN.md section 4 says how each field is derived.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# SURVEY 8(d): algorithmic bytes per update, single-pass streaming model, in scalars of the state dtype
ARZ_SCALARS_FWD, ARZ_SCALARS_BWD = 4, 6          # fwd: read (r,y) write (r,y); bwd: read (r,y), read adj, write adj
IDM_SCALARS_FWD, IDM_SCALARS_BWD = 10, 12        # fwd: read (p,v)+6 params, write (p,v); bwd: read 8 + adj 2 + write 2
SEED = 20221008
# --dump-outputs: bytes for the 5 ARZ arrays of [lanes, cells] and the 4 IDM arrays of [vehicles]; 56 MB in all
DUMP_ARZ_BYTES, DUMP_IDM_BYTES = 40 << 20, 16 << 20


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dtype", default="f64", choices=["f64", "f32"])
    ap.add_argument("--lanes", type=int, default=65536, help="ARZ lanes per GPU (weak) / in the global batch (strong)")
    ap.add_argument("--cells", type=int, default=1024)
    ap.add_argument("--micro-lanes", type=int, default=65536, help="IDM lanes per GPU (weak) / in the global batch (strong)")
    ap.add_argument("--lane-vehicles", type=int, default=64)
    ap.add_argument("--sim-steps", type=int, default=1000)
    ap.add_argument("--ckpt-every", type=int, default=0,
                    help="ARZ checkpoint interval; 0 = auto: store every state (no recompute in the adjoint) and walk "
                         "the lanes in chunks that fit the free HBM, else 32 with segment recompute")
    ap.add_argument("--idm-ckpt-every", type=int, default=16)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-net", action="store_true", help="skip the secondary connected-network (ITSCP) measurement")
    ap.add_argument("--no-strong", action="store_true", help="skip the strong-scaling split under torchrun")
    ap.add_argument("--no-parity", action="store_true", help="skip the oracle check of sampled lanes")
    ap.add_argument("--no-drivers", action="store_true", help="skip configs 1-3 under the reference's unchanged drivers")
    ap.add_argument("--net-replicas", type=int, default=2048)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy in the state dtype: "
                         "the losses, and final states and initial-state gradients of a fixed seeded sample of lanes. "
                         "The sample is gathered on the device in the last timed step, after each rollout's closing "
                         "event: the per-phase times and rates exclude it, ms_per_step includes those few small copies")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl ours)")
    return a


def workload_name(a):
    return ("synthetic batch per GPU: %d ARZ lanes x %d cells + %d IDM vehicles (%d lanes x %d), %d steps fwd+bwd"
            % (a.lanes, a.cells, a.micro_lanes * a.lane_vehicles, a.micro_lanes, a.lane_vehicles, a.sim_steps))


# ----------------------------------------------------------------------------------------- synthetic inputs

def make_arz_inputs(a, shard, torch, lo=0, hi=None):
    """SURVEY 8(d) 'Synthetic ARZ input' (C1's physics, example/inverse/macro.py:48-49,88-89,246-252).  The whole
    batch of `shard` is drawn from one generator and rows [lo, hi) are returned, so a lane's inputs depend on
    (shard, lane index) only -- not on how many ranks share the batch."""
    g = torch.Generator().manual_seed(SEED + shard)
    B, N, umax = a.lanes, a.cells, 30.0
    hi = B if hi is None else hi
    r0 = torch.rand((B, N), generator=g, dtype=torch.float32)[lo:hi].clone()
    u0 = (torch.rand((B, N), generator=g, dtype=torch.float32) * umax)[lo:hi].clone()
    gr = torch.rand((B, 2), generator=g, dtype=torch.float32)[lo:hi].clone()
    gu = (torch.rand((B, 2), generator=g, dtype=torch.float32) * umax)[lo:hi].clone()
    tr = torch.rand((B, N), generator=g, dtype=torch.float32)[lo:hi].clone()
    tu = (torch.rand((B, N), generator=g, dtype=torch.float32) * umax)[lo:hi].clone()
    return dict(r0=r0, u0=u0, gr=gr, gu=gu, tr=tr, tu=tu, dx=5.0, umax=umax, dt=0.01)


def make_idm_inputs(a, shard, torch, lo=0, hi=None):
    """SURVEY 8(d) 'Synthetic IDM input' (example/inverse/micro.py:77-81; road/vehicle/micro_vehicle.py:88-109);
    micro lanes [lo, hi) of the shard's batch."""
    g = torch.Generator().manual_seed(SEED + 7919 + shard)
    L, n, umax = a.micro_lanes, a.lane_vehicles, 30.0
    hi = L if hi is None else hi
    V = L * n
    rnd = lambda *s: torch.rand(s, generator=g, dtype=torch.float32)
    p0 = (torch.arange(n, dtype=torch.float32)[None, :] * 20.0 + rnd(L, n) * 10.0).reshape(V)
    v0 = 9.0 + 12.0 * rnd(V)
    params = torch.stack([(1.5 + 0.5 * rnd(V)) * umax, (1.0 + 0.5 * rnd(V)) * umax, (0.8 + 0.4 * rnd(V)) * umax,
                          1.0 + rnd(V), 0.2 + 0.4 * rnd(V), torch.full((V,), 5.0)])
    tp = p0 + 0.01 * 1000 * 15.0 + rnd(V)
    tv = 9.0 + 12.0 * rnd(V)
    s = slice(lo * n, hi * n)
    off = (torch.arange(hi - lo + 1, dtype=torch.int64) * n).to(torch.int32)
    head = torch.tensor([[1000.0, 0.0]], dtype=torch.float32).repeat(hi - lo, 1)
    return dict(p0=p0[s].clone(), v0=v0[s].clone(), params=params[:, s].clone(), tp=tp[s].clone(), tv=tv[s].clone(),
                off=off, head=head, dt=0.01, n=n)


# ----------------------------------------------------------------------------------------- clocks sampler

class Clocks:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for ts, line in self.rows:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 8 or not (t0 <= ts <= t1 + 0.3):
                continue
            try:
                sm.append(float(f[1])); mx = float(f[2])
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ----------------------------------------------------------------------------------------- CPU arms

CPU_SAMPLE = {"arz_lanes_per_core": 32, "arz_steps": 20, "idm_lanes_per_core": 512, "idm_steps": 100}


def cpu_port_rates(a):
    """Times the oracle port (oracle/dhts_oracle.c, OpenMP over lanes) on a FIXED bounded sample of the workload:
    lanes of the config's shape (N cells / n vehicles), 32 ARZ lanes and 512 IDM lanes per host core, 20 / 100 steps,
    repeated until ~6 s have passed (the best repetition counts).  Returns rates + sample text."""
    import numpy as np
    from oracle import oracle as O
    cores = O.set_threads(len(os.sched_getaffinity(0)))     # explicit: torchrun exports OMP_NUM_THREADS=1
    rng = np.random.default_rng(SEED)
    N, n, umax = a.cells, a.lane_vehicles, 30.0
    Ta, Ti = min(CPU_SAMPLE["arz_steps"], a.sim_steps), min(CPU_SAMPLE["idm_steps"], a.sim_steps)
    Ba, Li = CPU_SAMPLE["arz_lanes_per_core"] * cores, CPU_SAMPLE["idm_lanes_per_core"] * cores

    r0 = rng.uniform(0, 1, (Ba, N)); u0 = rng.uniform(0, 1, (Ba, N)) * umax
    gh = np.stack([rng.uniform(0, 1, (Ba, 2)), rng.uniform(0, 1, (Ba, 2)) * umax], -1)
    w = rng.normal(size=(Ba, N))
    V = Li * n
    p0 = (np.arange(n)[None] * 20.0 + rng.uniform(0, 10, (Li, n))).ravel(); v0 = rng.uniform(9, 21, V)
    par = np.stack([rng.uniform(1.5, 2, V) * umax, rng.uniform(1, 1.5, V) * umax, rng.uniform(0.8, 1.2, V) * umax,
                    rng.uniform(1, 2, V), rng.uniform(0.2, 0.6, V), np.full(V, 5.0)])
    off = np.arange(Li + 1) * n; head = np.tile([[1000.0, 0.0]], (Li, 1)); wv = rng.normal(size=V)

    def best(fn, units, budget):
        rate, t_end = 0.0, time.perf_counter() + budget
        while True:
            t = time.perf_counter(); fn(); dt = time.perf_counter() - t
            rate = max(rate, units / dt)
            if time.perf_counter() + dt > t_end:
                return rate

    rate_a = best(lambda: O.arz_rollout(r0, u0, gh, 5.0, umax, 0.01, Ta, g_rT=w, g_uT=w / umax), Ba * N * Ta, 4.0)
    rate_i = best(lambda: O.idm_rollout(p0, v0, par, off, head, 0.01, Ti, g_pT=wv, g_vT=wv), V * Ti, 2.0)
    sample = ("%d ARZ lanes x %d cells x %d steps fwd+bwd; %d IDM lanes x %d vehicles x %d steps fwd+bwd; "
              "OpenMP over lanes, best repetition" % (Ba, N, Ta, Li, n, Ti))
    return rate_a, rate_i, cores, sample


def reference_python_rates():
    """The reference's OWN Python lanes (baseline/_ref, unmodified), one process per host core (baseline/time_reference.py)."""
    try:
        from baseline import time_reference
        return time_reference.measure()
    except Exception as e:      # the reference install is optional on a box
        return {"unavailable": "%s: %s" % (type(e).__name__, str(e)[:200])}


def driver_episode_times(impls=("reference", "dropin")):
    """Configs 1-3 of BASELINE.json: seconds per gradient-descent episode of the reference's UNMODIFIED drivers
    example/inverse/{macro,micro,hybrid}.py, on the reference's own CPU lanes and on the drop-in (GPU) lanes
    (baseline/run_drivers.py, one process each; the reference ones run concurrently, one core each)."""
    from baseline import install_ref
    if not install_ref.available():
        return {"unavailable": "baseline/_ref is absent (python baseline/install_ref.py)"}
    script = os.path.join(ROOT, "baseline", "run_drivers.py")
    out = {}

    def launch(impl, prob, episodes):
        return subprocess.Popen([sys.executable, script, "--impl", impl, "--problem", prob, "--episodes", str(episodes)],
                                stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)

    def collect(p):
        o, e = p.communicate()
        if p.returncode != 0:
            return {"error": e.strip()[-300:]}
        j = json.loads(o.strip().splitlines()[-1])
        return {"s_per_episode": j["s_per_episode"], "episodes": j["episodes"], "end_errors": j["end_errors"]}

    probs = ("macro", "micro", "hybrid")
    if "reference" in impls:
        ps = {prob: launch("reference", prob, 2) for prob in probs}
        for prob, p in ps.items():
            out.setdefault(prob, {})["reference_cpu"] = collect(p)
    if "dropin" in impls:
        for prob in probs:
            out.setdefault(prob, {})["dropin_gpu"] = collect(launch("dropin", prob, 6))
    out["note"] = ("s per solve_gd episode (500 steps fwd + backward + Adam step), drivers = the reference's own files; "
                   "reference_cpu: its Python lanes on one host core each; dropin_gpu: dhts_b200.dropin lanes on cuda:0")
    return out


def run_reference(a):
    """CPU arm.  `value` is the oracle port (C, OpenMP, every host thread: the FASTEST CPU statement of the step we
    have, so the driver's ratio is conservative); `cpu_baseline.reference_python` is the reference's own Python path
    timed beside it (baseline/_ref, one process per core)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    t0 = time.time()
    for _ in range(min(a.warmup, 1)):
        cpu_port_rates(a)
    ra, ri, ms = [], [], []
    for _ in range(max(1, a.steps)):
        t = time.perf_counter()
        x, y, cores, sample = cpu_port_rates(a)
        ms.append((time.perf_counter() - t) * 1e3); ra.append(x); ri.append(y)
    va, vi = sum(ra) / len(ra), sum(ri) / len(ri)
    line = {"impl": "reference", "metric": "fwd+bwd cell-updates/s", "value": va, "unit": "cell-updates/s",
            "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": sum(ms) / len(ms),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_name(a), "sample_per_step": sample},
            "idm": {"value": vi, "unit": "vehicle-updates/s"},
            "cpu_baseline": {"value": va, "unit": "cell-updates/s", "cores": cores, "kind": "port", "sample": sample,
                             "idm_value": vi, "idm_unit": "vehicle-updates/s",
                             "note": "C port of the reference step (oracle/dhts_oracle.c); the reference's own Python "
                                     "path is in reference_python"},
            "e2e": {"value": va, "unit": "cell-updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    if not a.no_cpu_baseline:
        line["cpu_baseline"]["reference_python"] = reference_python_rates()
    line["wall_s"] = time.time() - t0
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------- connected network (secondary)

def network_bench(a, dev, dt_t, torch):
    """Secondary measurement (SURVEY 8f): BASELINE.json configs[3]'s lane graph in macro mode -- 3 x 3 intersections,
    1 lane per road, 5 m access lanes (144 lanes, 288 cells), u_max 60, 30 Hz, 600 frames, 4 s signals -- rolled out
    for `net_replicas` candidate signal plans at once, forward + adjoint (gradient of the fused queue reward wrt
    every action), through dhts_net_rollout_{fwd,bwd}."""
    import numpy as np
    from dhts_b200.itscp import ItscpBatch, ItscpGrid
    grid = ItscpGrid(3, 1, 5.0, 5.0)
    env = ItscpBatch(grid, dev, speed_limit=60.0, simulation_frequency=30, signal_length=4.0, dtype=dt_t)
    R, T, L, NC = a.net_replicas, 600, grid.L, env.topo.NC
    rng = np.random.default_rng(SEED)
    nxt, route = env.topo.next, -np.ones((T, 2, L), dtype=np.int32)
    for t in range(T):          # RoadNetwork.create_random_macro_route (road_network.py:389-423)
        for l in rng.permutation(L):
            for n in (rng.permutation(nxt[l]) if nxt[l] else []):
                if route[t, 0, n] < 0:
                    route[t, 1, l] = n; route[t, 0, n] = l
                    break
    g = torch.Generator().manual_seed(SEED + 31)
    n_act = (T // env.frames_per_signal) * 9
    action = (0.1 + 0.8 * torch.rand((R, n_act), generator=g, dtype=torch.float32)).to(dt_t).to(dev).requires_grad_()
    sess = torch.rand((R, 5, L), generator=g, dtype=torch.float32).to(dt_t)          # itscp_random_schedule: 5 sessions
    incoming = sess.repeat_interleave(T // 5, dim=1).contiguous().to(dev)
    route_t = torch.tensor(route, device=dev)
    qk = torch.full((T,), 16.0 / 30.0, dtype=dt_t, device=dev)
    ev = lambda: torch.cuda.Event(enable_timing=True)
    fwd_ms, bwd_ms = [], []
    for it in range(3):
        action.grad = None
        e = [ev() for _ in range(4)]
        sig = grid.signals(action, T, env.frames_per_signal, soft=True)
        e[0].record()
        reward, states = env.rollout(action, incoming, route_t, T, differentiable=True, exact_constants=False, qk=qk)
        e[1].record()
        loss = reward.sum()
        e[2].record()
        loss.backward()
        e[3].record()
        torch.cuda.synchronize()
        if it:
            fwd_ms.append(e[0].elapsed_time(e[1])); bwd_ms.append(e[2].elapsed_time(e[3]))
        del states, reward, loss, sig
    f, b = sum(fwd_ms) / len(fwd_ms), sum(bwd_ms) / len(bwd_ms)
    upd = R * NC * T
    esz = 8 if dt_t == torch.float64 else 4
    return {"workload": "ITSCP 3x3 grid, macro mode: %d lanes / %d cells per replica, %d replicas, %d frames fwd+bwd "
                        "(signals from %d actions per replica, fused queue reward)" % (L, NC, R, T, n_act),
            "value": upd / ((f + b) / 1e3), "unit": "cell-updates/s", "fwd_ms": f, "bwd_ms": b,
            "replica_rollouts_per_s": R / ((f + b) / 1e3),
            "stored_state_bytes": (T + 1) * R * 3 * NC * esz, "gpu_launches": 2,
            "mean_reward": float(env.rollout(action.detach(), incoming, route_t, T, exact_constants=False, qk=qk)[0].mean()),
            "grad_abs_mean": float(action.grad.abs().mean()),
            "reference_note": "the reference steps this network lane by lane in Python: ~2.5-4.3e3 cell-updates/s per "
                              "core (BASELINE.md sec. 2), i.e. ~40-70 s per 600-frame episode fwd+bwd"}


def config4_bench(a, dev, dt_t, torch):
    """Secondary measurement: BASELINE.json configs[3] itself -- one training episode of run_itscp_hybrid.sh (hybrid mode,
    3 x 3 intersections, centre intersection micro, 600 frames, 45 actions, problem_1 inflow) through the headless env:
    action -> signals -> fused hybrid rollout -> queue reward with running-mean constants -> gradient wrt the actions.
    R = 1 is what the reference's trainer does per epoch (trainer.py:140-162 with 1 episode); R = 256 batches episodes."""
    import numpy as np
    from dhts_b200.itscp_env import ItscpEnv, problem_1
    np.random.seed(SEED)
    env = ItscpEnv(device=dev, dtype=dt_t)
    env.schedule_callback = problem_1
    env.config.update(num_intersection=3, lane_length=5.0, num_lane=1, policy_length=20, signal_length=4, mode="hybrid",
                      speed_limit=60.0)
    env.reset()
    g = torch.Generator().manual_seed(SEED + 41)
    out = {"workload": "run_itscp_hybrid.sh episode: 144 lanes (128 macro / 16 micro), 600 frames fwd+bwd, exact running-mean "
                       "queue reward, gradient wrt 45 actions"}
    ev = lambda: torch.cuda.Event(enable_timing=True)
    for R in (1, 256):
        action = (0.3 + 0.4 * torch.rand((R, env.action_size()), generator=g, dtype=torch.float32)).to(dt_t).to(dev).requires_grad_()
        env.resample_spawn_routes(R, g)
        ms = []
        for it in range(3):
            action.grad = None
            e0, e1 = ev(), ev()
            e0.record()
            reward = env.rollout(action, True)
            reward.sum().backward()
            e1.record()
            torch.cuda.synchronize()
            if it:
                ms.append(e0.elapsed_time(e1))
        bits, ncol = env.flags.read()
        out["R%d" % R] = {"ms_per_batch": sum(ms) / len(ms), "episodes_per_s": R / (sum(ms) / len(ms) / 1e3),
                          "mean_reward": float(reward.mean()), "grad_abs_mean": float(action.grad.abs().mean()),
                          "flag_bits": bits, "collision_steps": ncol}
    out["reference_note"] = ("the live reference needs ~200 s for the same episode forward + backward on one host core "
                             "(oracle/gen_golden_c4.py in the build container; it is single-threaded Python)")
    return out


# ----------------------------------------------------------------------------------------- our arm

class Batch:
    """One rank's lanes of the synthetic workload: pinned host inputs, device copies, the ARZ chunk plan with its
    checkpoint arena, and the passes over them."""

    def __init__(self, a, A, M, dev, dt_t, flags, torch):
        import dhts_b200  # noqa: F401
        from dhts_b200 import dist as shards
        from dhts_b200 import functional as F
        self.a, self.A, self.M, self.dev, self.dt_t, self.flags, self.torch, self.F, self.shards = a, A, M, dev, dt_t, flags, torch, F, shards
        pin = lambda t: t.to(dt_t if t.is_floating_point() else t.dtype).pin_memory()
        self.hostA = {k: pin(v) for k, v in A.items() if hasattr(v, "shape")}
        self.hostM = {k: pin(v) for k, v in M.items() if hasattr(v, "shape")}
        self.devA = {k: v.to(dev) for k, v in self.hostA.items()}
        self.devM = {k: v.to(dev) for k, v in self.hostM.items()}
        self.B, self.N, self.T = self.hostA["r0"].shape[0], a.cells, a.sim_steps
        self.V = self.hostM["p0"].numel()
        self.esz = 8 if a.dtype == "f64" else 4
        B, N, T = self.B, self.N, self.T
        # ARZ plan: lanes per chunk and checkpoint interval (functional.arz_rollout_plan: every state stored when a
        # chunk of >= 296 lanes fits the free HBM, which removes the segment recompute from the adjoint)
        if a.ckpt_every > 0:
            self.K = a.ckpt_every
            self.chunk = F.arz_rollout_plan(B, N, T, dt_t, dev)[0] if self.K == 1 else B
        else:
            self.chunk, self.K = F.arz_rollout_plan(B, N, T, dt_t, dev)
        self.chunks = [(lo, min(B, lo + self.chunk)) for lo in range(0, B, self.chunk)]
        # one checkpoint arena for all chunks and passes (a chunk's checkpoints are dead once its adjoint has run)
        self.arena = torch.empty(F.arz_ckpt_elems(self.chunk, N, T, self.K, dt_t), dtype=dt_t, device=dev)   # states (+ interface outcomes)

    def ev(self):
        return self.torch.cuda.Event(enable_timing=True)

    def arz_pass(self, d, timers=None, before_chunk=None, after_chunk=None, capture=None):
        """fwd + loss + adjoint of all B lanes, chunk of lanes by chunk of lanes (lanes are independent).
        before_chunk(i) / after_chunk(i, g_r0, g_u0) let the end-to-end pass pipeline its copies with the compute;
        capture = self.lane_capture(lanes) collects the rT / yT / uT / g_r0 / g_u0 rows of those lanes with device-side
        gathers only, so that a timed pass can capture without a host synchronisation."""
        torch, F, A = self.torch, self.F, self.A
        g_r0 = torch.empty_like(d["r0"]); g_u0 = torch.empty_like(d["u0"])
        total = torch.zeros((), dtype=self.dt_t, device=self.dev)
        for ci, (lo, hi) in enumerate(self.chunks):
            if before_chunk: before_chunk(ci)
            r0 = d["r0"][lo:hi].detach().requires_grad_(); u0 = d["u0"][lo:hi].detach().requires_grad_()
            ev4 = [self.ev() for _ in range(4)] if timers is not None else None
            if ev4: ev4[0].record()
            rT, yT, uT = F.arz_rollout(r0, u0, d["gr"][lo:hi], d["gu"][lo:hi], A["dx"], A["umax"], A["dt"], self.T,
                                       ckpt_every=self.K, flags=self.flags, ckpt_buffer=self.arena)
            if ev4: ev4[1].record()
            loss = ((rT - d["tr"][lo:hi]) ** 2).sum() + ((uT - d["tu"][lo:hi]) ** 2).sum()   # example/inverse/macro.py:226-241
            if ev4: ev4[2].record()
            loss.backward()
            if ev4: ev4[3].record(); timers.append(ev4)
            g_r0[lo:hi] = r0.grad; g_u0[lo:hi] = u0.grad
            total += loss.detach()
            if capture is not None:
                for k, x in (("rT", rT), ("yT", yT), ("uT", uT)):
                    capture.setdefault(k, []).append(x.detach().index_select(0, capture["rows"][ci]))
            if after_chunk: after_chunk(ci, g_r0, g_u0)
            del rT, yT, uT, loss, r0, u0
        if capture is not None:
            for k in ("rT", "yT", "uT"):
                capture[k] = torch.cat(capture[k])
            capture["g_r0"], capture["g_u0"] = (g.index_select(0, capture["lanes"]) for g in (g_r0, g_u0))
        return total, g_r0, g_u0

    def lane_capture(self, lanes):
        """Capture spec of arz_pass for the sorted lane indices `lanes`: their device indices, and per lane chunk the
        row indices within the chunk."""
        torch = self.torch
        return {"lanes": torch.tensor(lanes, dtype=torch.int64, device=self.dev),
                "rows": [torch.tensor([i - lo for i in lanes if lo <= i < hi], dtype=torch.int64, device=self.dev)
                         for lo, hi in self.chunks]}

    def idm_pass(self, d, timers=None, capture=None):
        F, M = self.F, self.M
        p0 = d["p0"].detach().requires_grad_(); v0 = d["v0"].detach().requires_grad_()
        ev4 = [self.ev() for _ in range(4)] if timers is not None else None
        if ev4: ev4[0].record()
        pT, vT = F.idm_rollout(p0, v0, d["params"], d["off"], d["head"], M["dt"], self.T, ckpt_every=self.a.idm_ckpt_every,
                               flags=self.flags, max_lane=M["n"])
        if ev4: ev4[1].record()
        loss = ((pT - d["tp"]) ** 2).sum() + ((vT - d["tv"]) ** 2).sum()     # example/inverse/micro.py:221-236
        if ev4: ev4[2].record()
        loss.backward()
        if ev4: ev4[3].record(); timers.append(ev4)
        if capture is not None:
            capture["pT"], capture["vT"], capture["g_p0"], capture["g_v0"] = pT.detach(), vT.detach(), p0.grad, v0.grad
        return loss.detach(), p0.grad, v0.grad

    def reduce_loss(self, la, li):
        return self.shards.reduce_losses(la, li)     # the only collective: scalar losses over the lane shards

    def timed(self, steps, warmup, barrier, capture=None):
        """Device-resident passes: W warm-up, then K timed, CUDA events around the whole region and around every launch.
        `capture` (see arz_pass) receives the outputs of the last timed pass."""
        torch = self.torch
        for _ in range(warmup):
            la, _, _ = self.arz_pass(self.devA); li, _, _ = self.idm_pass(self.devM); self.reduce_loss(la, li)
        barrier()
        t_wall0 = time.time()
        tA, tM = [], []              # CUDA events (start, fwd done, loss done, bwd done) per launch pair
        e0, e1 = self.ev(), self.ev()
        e0.record()
        for i in range(steps):
            cap = capture if i == steps - 1 else None
            la, _, _ = self.arz_pass(self.devA, tA, capture=cap); li, _, _ = self.idm_pass(self.devM, tM, capture=cap)
            losses = self.reduce_loss(la, li)
        e1.record()
        barrier()
        t_wall1 = time.time()
        r = {"total_ms": e0.elapsed_time(e1),
             "arz_fwd": sum(t[0].elapsed_time(t[1]) for t in tA), "arz_bwd": sum(t[2].elapsed_time(t[3]) for t in tA),
             "arz_all": sum(t[0].elapsed_time(t[3]) for t in tA),
             "idm_fwd": sum(t[0].elapsed_time(t[1]) for t in tM), "idm_bwd": sum(t[2].elapsed_time(t[3]) for t in tM),
             "idm_all": sum(t[0].elapsed_time(t[3]) for t in tM)}
        return r, losses, (la, li), (t_wall0, t_wall1)

    def e2e(self, steps, barrier):
        """End-to-end passes: host (pinned) inputs -> H2D -> rollouts -> D2H of losses and gradients, every step.
        Copies are pipelined with the compute, lane chunk by lane chunk: inputs of chunk i+1.. travel on a copy-in
        stream while chunk i computes; its gradients leave on a copy-out stream.  Everything is inside the timed
        region; a pass ends with the host read of the reduced losses after both streams have drained."""
        torch, dev, dt_t = self.torch, self.dev, self.dt_t
        B, N, V = self.B, self.N, self.V
        outA = [torch.empty((B, N), dtype=dt_t).pin_memory() for _ in range(2)]
        outM = [torch.empty((V,), dtype=dt_t).pin_memory() for _ in range(2)]
        h2d = sum(v.numel() * v.element_size() for v in self.hostA.values()) + sum(v.numel() * v.element_size() for v in self.hostM.values())
        d2h = sum(t.numel() * t.element_size() for t in outA + outM) + 2 * self.esz
        s_in, s_out = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
        dA = {k: torch.empty_like(v, device=dev) for k, v in self.hostA.items()}
        dM = {k: torch.empty_like(v, device=dev) for k, v in self.hostM.items()}
        pass_done = self.ev()
        pass_done.record()

        def e2e_pass():
            cur = torch.cuda.current_stream(dev)
            in_ready = []
            s_in.wait_event(pass_done)                      # the previous pass no longer reads the staging buffers
            with torch.cuda.stream(s_in):
                for lo, hi in self.chunks:
                    for k, v in self.hostA.items():
                        dA[k][lo:hi].copy_(v[lo:hi], non_blocking=True)
                    e = self.ev(); e.record(s_in); in_ready.append(e)
                for k, v in self.hostM.items():
                    dM[k].copy_(v, non_blocking=True)
                idm_ready = self.ev(); idm_ready.record(s_in)

            def before(ci):
                cur.wait_event(in_ready[ci])

            def after(ci, g_r0, g_u0):
                lo, hi = self.chunks[ci]
                done = self.ev(); done.record(cur)
                s_out.wait_event(done)
                with torch.cuda.stream(s_out):
                    outA[0][lo:hi].copy_(g_r0[lo:hi], non_blocking=True); outA[1][lo:hi].copy_(g_u0[lo:hi], non_blocking=True)
                g_r0.record_stream(s_out); g_u0.record_stream(s_out)

            la, _, _ = self.arz_pass(dA, before_chunk=before, after_chunk=after)
            cur.wait_event(idm_ready)
            li, gp0, gv0 = self.idm_pass(dM)
            outM[0].copy_(gp0, non_blocking=True); outM[1].copy_(gv0, non_blocking=True)
            cur.wait_stream(s_out)
            pass_done.record(cur)
            return self.reduce_loss(la, li).cpu()

        e2e_pass()
        barrier()
        f0, f1 = self.ev(), self.ev()
        f0.record()
        for _ in range(steps):
            e2e_pass()
        f1.record()
        barrier()
        ms = f0.elapsed_time(f1)
        del dA, dM, outA, outM
        return ms, h2d, d2h

    def parity_check(self, timed_losses):
        """Oracle check of the TIMED configuration itself (same inputs, same K, same chunk plan and arena): one more
        pass, rows of sampled lanes -- first / last lane of every chunk, i.e. every arena reuse boundary, plus seeded
        extras -- against oracle/dhts_oracle.c run for the full T steps (example/inverse/_inverse.py:91-99 semantics:
        set_state_vector_u -> T x forward -> get_state_vector, squared-error loss, backward)."""
        import numpy as np
        from oracle import oracle as O
        torch, T = self.torch, self.T
        O.set_threads(len(os.sched_getaffinity(0)))
        rng = np.random.default_rng(SEED)
        idx = sorted(set([lo for lo, _ in self.chunks] + [hi - 1 for _, hi in self.chunks]
                         + [int(x) for x in rng.integers(0, self.B, 4)]))[:28]
        cap = self.lane_capture(idx)
        la, _, _ = self.arz_pass(self.devA, capture=cap)
        capM = {}
        li, g_p0, g_v0 = self.idm_pass(self.devM, capture=capM)
        rT, uT = cap["rT"].cpu().numpy().astype(np.float64), cap["uT"].cpu().numpy().astype(np.float64)
        h = lambda k, t=self.hostA: t[k][idx].numpy().astype(np.float64)
        gh = np.stack([h("gr"), h("gu")], -1)
        f = O.arz_rollout(h("r0"), h("u0"), gh, self.A["dx"], self.A["umax"], self.A["dt"], T)
        o = O.arz_rollout(h("r0"), h("u0"), gh, self.A["dx"], self.A["umax"], self.A["dt"], T,
                          g_rT=2.0 * (f["rT"] - h("tr")), g_uT=2.0 * (f["uT"] - h("tu")))
        rel = lambda x, y: float(np.abs(np.asarray(x, dtype=np.float64) - y).max() / (1e-300 + np.abs(y).max()))
        res = {"lanes": idx, "steps": T, "ckpt_every": self.K, "chunks": len(self.chunks),
               "arz": {"rT": rel(rT, o["rT"]), "uT": rel(uT, o["uT"]),
                       "g_r0": rel(cap["g_r0"].cpu().numpy(), o["g_r0"]), "g_u0": rel(cap["g_u0"].cpu().numpy(), o["g_u0"])}}
        # IDM: 32 sampled lanes (first, last, seeded)
        n, L = self.M["n"], self.hostM["head"].shape[0]
        lidx = sorted(set([0, L - 1] + [int(x) for x in rng.integers(0, L, 30)]))
        vsel = np.concatenate([np.arange(l * n, (l + 1) * n) for l in lidx])
        hm = lambda k: self.hostM[k].numpy().astype(np.float64)
        p0, v0, par = hm("p0")[vsel], hm("v0")[vsel], hm("params")[:, vsel]
        off = np.arange(len(lidx) + 1) * n; head = hm("head")[lidx]
        fi = O.idm_rollout(p0, v0, par, off, head, self.M["dt"], T)
        oi = O.idm_rollout(p0, v0, par, off, head, self.M["dt"], T, g_pT=2.0 * (fi["pT"] - hm("tp")[vsel]),
                           g_vT=2.0 * (fi["vT"] - hm("tv")[vsel]))
        res["idm"] = {"lanes": len(lidx), "pT": rel(capM["pT"].cpu().numpy()[vsel], oi["pT"]),
                      "vT": rel(capM["vT"].cpu().numpy()[vsel], oi["vT"]),
                      "g_p0": rel(g_p0.cpu().numpy()[vsel], oi["g_p0"]), "g_v0": rel(g_v0.cpu().numpy()[vsel], oi["g_v0"])}
        # the checked pass IS the timed pass: same kernels, same plan -> bitwise the same losses
        res["losses_equal_timed_pass"] = bool(float(la) == float(timed_losses[0]) and float(li) == float(timed_losses[1]))
        f64 = self.a.dtype == "f64"
        tol_s, tol_g = (1e-9, 1e-8) if f64 else (2e-3, 5e-2)     # fp32 build: 1000 steps of fp32 rounding vs the fp64 oracle
        res["tol"] = {"states": tol_s, "grads": tol_g, "norm": "max |a-b| / max |b| over the sampled lanes"}
        res["ok"] = bool(all(res[m][k] <= tol_s for m, ks in (("arz", ("rT", "uT")), ("idm", ("pT", "vT"))) for k in ks)
                         and all(res[m][k] <= tol_g for m, ks in (("arz", ("g_r0", "g_u0")), ("idm", ("g_p0", "g_v0"))) for k in ks)
                         and res["losses_equal_timed_pass"])
        return res

    def free(self):
        for k in ("arena", "devA", "devM", "hostA", "hostM"):
            setattr(self, k, None)
        self.torch.cuda.empty_cache()


def dump_sample(n, bytes_per_item, budget):
    """The sorted, seeded sample of items (lanes) of 0..n-1 whose outputs --dump-outputs writes: as many as fit the
    budget, so the same arguments always select the same lanes."""
    import numpy as np
    k = min(n, max(1, budget // bytes_per_item))
    return sorted(np.random.default_rng(SEED).choice(n, k, replace=False).tolist())


def write_outputs(path, cap, losses, idm_lanes, lane_vehicles):
    """--dump-outputs: the last timed pass's losses [arz, idm] and, for the sampled ARZ lanes and IDM lanes, the final
    states and the gradients of the loss wrt the initial states, in the state dtype."""
    import numpy as np
    import torch
    veh = torch.tensor([l * lane_vehicles + j for l in idm_lanes for j in range(lane_vehicles)], device=losses.device)
    out = {"losses": losses}
    out.update({"arz_" + k: cap[k] for k in ("rT", "yT", "uT", "g_r0", "g_u0")})
    out.update({"idm_" + k: cap[k].index_select(0, veh) for k in ("pT", "vT", "g_p0", "g_v0")})
    os.makedirs(path, exist_ok=True)
    for name, t in out.items():
        np.save(os.path.join(path, name + ".npy"), t.detach().cpu().numpy())


def fp64_peak(dev, torch, lib):
    """MEASURED fp64 issue peak (DFMA thread-instructions per second) of this GPU: dhts_fp64_probe timed with CUDA events."""
    blocks = 148 * 8
    out = torch.empty(blocks * 256, dtype=torch.float64, device=dev)
    st = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    best = 0.0
    for it in range(4):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        n = lib.dhts_fp64_probe(ctypes.c_void_p(out.data_ptr()), blocks, 1 << 16, st)
        e1.record()
        torch.cuda.synchronize()
        if it and n > 0:
            best = max(best, n / (e0.elapsed_time(e1) / 1e3))
    return best


def run_ours(a):
    import torch
    import torch.distributed as dist
    import dhts_b200
    from dhts_b200 import dist as shards

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU fallback of the product path)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = dhts_b200._lib.load()
    dt_t = torch.float64 if a.dtype == "f64" else torch.float32
    esz = 8 if a.dtype == "f64" else 4
    flags = dhts_b200.Flags(dev)
    T, N = a.sim_steps, a.cells

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def rank_max(vals):
        t = torch.tensor(vals, dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.tolist()

    # ================= weak split: this rank's own batch (value / e2e of the contract)
    bt = Batch(a, make_arz_inputs(a, rank, torch), make_idm_inputs(a, rank, torch), dev, dt_t, flags, torch)
    B, V = bt.B, bt.V
    clocks = Clocks(local) if rank == 0 else None
    cap = None
    if a.dump_outputs and rank == 0:
        arz_lanes = dump_sample(B, 5 * N * esz, DUMP_ARZ_BYTES)
        idm_lanes = dump_sample(V // a.lane_vehicles, 4 * a.lane_vehicles * esz, DUMP_IDM_BYTES)
        cap = bt.lane_capture(arz_lanes)
    tm, losses, last_losses, (tw0, tw1) = bt.timed(a.steps, a.warmup, barrier, cap)
    clk = clocks.stop(tw0, tw1) if clocks else None
    if cap is not None:
        write_outputs(a.dump_outputs, cap, losses, idm_lanes, a.lane_vehicles)
        del cap
    bits, ncol = flags.read()
    e2e_ms, h2d, d2h = (None, 0, 0)
    if not a.no_e2e:
        e2e_ms, h2d, d2h = bt.e2e(a.steps, barrier)
    keys = ["total_ms", "arz_all", "idm_all", "arz_fwd", "arz_bwd", "idm_fwd", "idm_bwd"]
    vals = rank_max([tm[k] for k in keys] + [e2e_ms or 0.0])
    tmx = dict(zip(keys, vals[:-1])); e2e_ms_max = vals[-1]
    parity = None
    if rank == 0 and not a.no_parity:
        parity = bt.parity_check(last_losses)
    arz_K, arz_chunk, arz_chunks = bt.K, bt.chunk, bt.chunks
    peak_dfma = fp64_peak(dev, torch, lib) if rank == 0 else 0.0

    # ================= strong split: the global batch (shard 0's inputs) cut into `world` lane blocks
    strong = None
    if world > 1 and not a.no_strong:
        bt.free(); del bt
        lo, hi = shards.shard_range(a.lanes, rank, world)
        mlo, mhi = shards.shard_range(a.micro_lanes, rank, world)
        bs = Batch(a, make_arz_inputs(a, 0, torch, lo, hi), make_idm_inputs(a, 0, torch, mlo, mhi), dev, dt_t, flags, torch)
        ts, s_losses, _, _ = bs.timed(a.steps, a.warmup, barrier)
        s_e2e = None
        if not a.no_e2e:
            s_e2e, _, _ = bs.e2e(a.steps, barrier)
        svals = rank_max([ts["total_ms"], ts["arz_all"], ts["idm_all"], s_e2e or 0.0])
        # results must not depend on the split: rank 0 re-runs the FIRST lane of every rank's block on its own and
        # compares bitwise with what that rank computed inside its block
        _, g_r0, _ = bs.arz_pass(bs.devA)
        mine = g_r0[0].contiguous()
        rows = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(rows, mine)
        same = None
        if rank == 0:
            firsts = [shards.shard_range(a.lanes, r, world)[0] for r in range(world)]
            A0 = make_arz_inputs(a, 0, torch)
            sub = {k: (v[firsts].to(dt_t).to(dev) if hasattr(v, "shape") else v) for k, v in A0.items()}
            r0 = sub["r0"].requires_grad_(); u0 = sub["u0"].requires_grad_()
            rT, yT, uT = bs.F.arz_rollout(r0, u0, sub["gr"], sub["gu"], sub["dx"], sub["umax"], sub["dt"], T,
                                          ckpt_every=bs.K, flags=flags)
            (((rT - sub["tr"]) ** 2).sum() + ((uT - sub["tu"]) ** 2).sum()).backward()
            same = bool(all(torch.equal(r0.grad[i], rows[i]) for i in range(world)))
        if rank == 0:
            strong = {"workload": "ONE global batch (%d ARZ lanes x %d cells + %d IDM vehicles, %d steps fwd+bwd) split into "
                                  "%d contiguous lane blocks" % (a.lanes, N, a.micro_lanes * a.lane_vehicles, T, world),
                      "value": a.lanes * N * T * a.steps / (svals[1] / 1e3), "unit": "cell-updates/s",
                      "idm_value": a.micro_lanes * a.lane_vehicles * T * a.steps / (svals[2] / 1e3),
                      "ms_per_step": svals[0] / a.steps, "lanes_per_gpu": hi - lo, "arz_chunks_per_pass": len(bs.chunks),
                      "arz_lanes_per_chunk": bs.chunk, "ckpt_every": bs.K,
                      "e2e": (a.lanes * N * T * a.steps / (svals[3] / 1e3)) if s_e2e else None,
                      "e2e_ms_per_step": (svals[3] / a.steps) if s_e2e else None,
                      "losses": [float(x) for x in s_losses.tolist()],
                      "shard_equals_unshard_bitwise": same,
                      "note": "value = global cell-updates / max-over-ranks time of the ARZ phase; efficiency vs the 1-GPU run of "
                              "the same job is value / (N x the N=1 `value`)"}
        bs.free(); del bs
    else:
        bt.free(); del bt

    if rank == 0:
        K = a.steps
        cell_updates = world * B * N * T * K
        veh_updates = world * V * T * K
        arz_fwd, arz_bwd, arz_all = tmx["arz_fwd"], tmx["arz_bwd"], tmx["arz_all"]
        idm_fwd, idm_bwd, idm_all = tmx["idm_fwd"], tmx["idm_bwd"], tmx["idm_all"]
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "6650 GB/s (of fallback)"
        # dominant kernel: arz_rollout_bwd (one launch per lane chunk)
        nl = len(arz_chunks)
        bwd_bytes = B * N * T * ARZ_SCALARS_BWD * esz / nl      # algorithmic bytes of ONE launch (average chunk)
        bwd_s = arz_bwd / K / nl / 1e3                         # average duration of one launch
        prof = {}
        try:
            prof = json.load(open(os.path.join(ROOT, "profiles", "kernel_mix.json")))
        except Exception:
            pass
        tag = lambda kern: "%s_%s_k%d" % (kern, a.dtype, arz_K if kern.startswith("arz") else a.idm_ckpt_every)
        pk = lambda kern: prof.get(tag(kern)) or prof.get("%s_%s" % (kern, a.dtype)) or {}
        traffic = None
        pb = pk("arz_rollout_bwd")
        if pb.get("dram_bytes_per_update") is not None:
            traffic = pb["dram_bytes_per_update"] * B * N * T / nl
        both_bytes = B * N * T * (ARZ_SCALARS_FWD + ARZ_SCALARS_BWD) * esz
        both_s = (arz_fwd + arz_bwd) / K / 1e3
        idm_bytes = V * T * (IDM_SCALARS_FWD + IDM_SCALARS_BWD) * esz
        idm_s = (idm_fwd + idm_bwd) / K / 1e3
        # fp64 issue roofline: fp64-pipe thread-instructions per update (ncu, profiles/kernel_mix.json) x updates/s of the
        # kernel, against the DFMA rate measured on this GPU just now (dhts_fp64_probe)
        sm_hz = (clk or {}).get("sm_mhz") or 1965.0
        issue_peak = 148 * 4 * 32 * sm_hz * 1e6                 # thread-instruction issue slots per second

        def fp64_block(kern, updates_per_s):
            p = pk(kern)
            if not p or not peak_dfma:
                return None
            return {"fp64_pipe_inst_per_update": p.get("fp64_pipe_inst_per_update"),
                    "fp64_arith_inst_per_update": p.get("fp64_arith_inst_per_update"),
                    "thread_inst_per_update": p.get("thread_inst_per_update"),
                    "achieved_fp64_inst_per_s": p["fp64_pipe_inst_per_update"] * updates_per_s,
                    "frac_of_fp64_peak": p["fp64_pipe_inst_per_update"] * updates_per_s / peak_dfma,
                    "frac_of_issue_slots": p["thread_inst_per_update"] * updates_per_s / issue_peak,
                    "profile": p.get("source")}

        per_gpu = lambda ms: 1.0 / (ms / K / 1e3)
        roof64 = {"peak_dfma_per_s": peak_dfma, "peak_tflops": 2 * peak_dfma / 1e12,
                  "peak_source": "dhts_fp64_probe (8 independent DFMA chains per thread, 148 x 8 CTAs), timed in this run",
                  "sm_mhz_for_issue_slots": sm_hz,
                  "arz_rollout_fwd": fp64_block("arz_rollout_fwd", B * N * T * per_gpu(arz_fwd)),
                  "arz_rollout_bwd": fp64_block("arz_rollout_bwd", B * N * T * per_gpu(arz_bwd)),
                  "idm_rollout_fwd": fp64_block("idm_rollout_fwd", V * T * per_gpu(idm_fwd)),
                  "idm_rollout_bwd": fp64_block("idm_rollout_bwd", V * T * per_gpu(idm_bwd)),
                  "note": "the rollout kernels are bound by fp64 issue + dependency latency, not by HBM: these fractions are the "
                          "honest roof; per-update instruction counts come from the committed ncu capture named in `profile`"}
        finite = all(x == x and abs(x) != float("inf") for x in losses.tolist())
        # a run whose rollouts violated CFL / produced NaN adjoints, or (fp64) disagrees with the oracle, is not a result
        valid = finite and not (bits & 3) and (parity is None or parity["ok"] or a.dtype != "f64")
        line = {
            "metric": "fwd+bwd cell-updates/s", "value": cell_updates / (arz_all / 1e3), "unit": "cell-updates/s",
            "n_gpus": world, "steps": K, "warmup": a.warmup, "ms_per_step": tmx["total_ms"] / K, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": a.dtype, "data": "synthetic",
            "config": {"workload": workload_name(a), "arz": {"lanes_per_gpu": B, "cells": N, "dx": 5.0, "dt": 0.01,
                                                             "u_max": 30.0},
                       "idm": {"vehicles_per_gpu": V, "lane_vehicles": a.lane_vehicles, "params": "per-vehicle"},
                       "sim_steps": T, "ckpt_every": arz_K, "arz_lanes_per_chunk": arz_chunk,
                       "arz_chunks_per_pass": len(arz_chunks), "idm_ckpt_every": a.idm_ckpt_every, "parallelism": "lane shards x%d, all-reduce(loss)" % world,
                       "l2": "inputs (%.1f GB per pass) are larger than the 126 MB L2" % ((2 * B * N + 8 * V) * esz / 1e9)},
            "idm": {"metric": "fwd+bwd vehicle-updates/s", "value": veh_updates / (idm_all / 1e3),
                    "unit": "vehicle-updates/s", "ms_per_step": idm_all / K},
            "phase_ms_per_step": {"arz_fwd": arz_fwd / K, "arz_bwd": arz_bwd / K, "arz_total": arz_all / K,
                                  "idm_fwd": idm_fwd / K, "idm_bwd": idm_bwd / K, "idm_total": idm_all / K},
            "gpu_launches": (2 * len(arz_chunks) + 2) * K,
            # template arguments: cells per thread, register budget, adjoint mode, per-step inputs, stored outcomes, uniform geometry
            "roofline": {"kernel": "arz_rollout_bwd_reg_kernel<%s, 4, 2, %d, false, %s>" % (
                             "double" if a.dtype == "f64" else "float", 0 if arz_K == 1 else 2,
                             "true, true" if dhts_b200.ops.arz_ckpt_elems(arz_chunk, N, T, arz_K, dt_t)[1] else "false, false"),
                         "bound": "hbm", "achieved": bwd_bytes / bwd_s / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": bwd_bytes / bwd_s / 1e9 / peak, "frac_is": "of_streaming_model",
                         "traffic": traffic, "traffic_source": pb.get("source"), "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": bwd_bytes,
                         "launches_per_pass": len(arz_chunks),
                         "note": "achieved = ALGORITHMIC bytes (6 scalars x cell-steps of one adjoint launch, SURVEY 8d) / its mean "
                                 "CUDA-event time: the fraction of the speed a perfectly streaming kernel would reach, NOT achieved "
                                 "DRAM bandwidth -- traffic = DRAM bytes of that launch from the ncu capture named in "
                                 "traffic_source (bench-shaped launch), and roofline_fp64 is the roof that actually binds"},
            "roofline_fp64": roof64,
            "roofline_fwd_bwd": {"arz": {"achieved": both_bytes / both_s / 1e9, "frac_of_streaming_model": both_bytes / both_s / 1e9 / peak,
                                         "bytes_per_update": (ARZ_SCALARS_FWD + ARZ_SCALARS_BWD) * esz},
                                 "idm": {"algorithmic_gb_per_s": idm_bytes / idm_s / 1e9,
                                         "bytes_per_update": (IDM_SCALARS_FWD + IDM_SCALARS_BWD) * esz,
                                         "note": "no HBM fraction is quoted for IDM: state and parameters stay in registers for the "
                                                 "whole rollout, so the 176 B/update streaming model does not describe the kernel "
                                                 "(measured DRAM traffic is a few bytes per vehicle-step); see roofline_fp64"},
                                 "unit": "GB/s", "peak": peak},
            "clocks": clk,
            "flags": {"bits": bits, "collisions": ncol},
            "losses": [float(x) for x in losses.tolist()],
            "parity_check": parity,
            "valid": bool(valid),
        }
        if e2e_ms is not None:
            line["e2e"] = {"value": cell_updates / (e2e_ms_max / 1e3), "unit": "cell-updates/s",
                           "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms_max / K,
                           "note": "whole pass (ARZ + IDM) from pinned host buffers, gradients and losses read back, copies "
                                   "pipelined with the compute per lane chunk; value counts ARZ cell-updates over the "
                                   "WHOLE pass time (IDM and copies included)"}
        if world == 1:
            line["strong"] = {"note": "N = 1: the strong split is the weak one (same batch, seed SEED + 0)",
                              "value": line["value"], "e2e": line.get("e2e", {}).get("value")}
        elif strong is not None:
            line["strong"] = strong
        if not a.no_net:
            torch.cuda.empty_cache()
            line["itscp_net"] = network_bench(a, dev, dt_t, torch)
            torch.cuda.empty_cache()
            line["itscp_c4"] = config4_bench(a, dev, dt_t, torch)
        if not a.no_cpu_baseline and world == 1:      # the CPU leg is reported at N = 1 only
            ra, ri, cores, sample = cpu_port_rates(a)
            line["cpu_baseline"] = {"value": ra, "unit": "cell-updates/s", "cores": cores, "kind": "port",
                                    "sample": sample, "idm_value": ri, "idm_unit": "vehicle-updates/s",
                                    "reference_python": reference_python_rates()}
        if not a.no_drivers and world == 1:
            torch.cuda.empty_cache()
            line["configs_1_3"] = driver_episode_times()
        print(json.dumps(line), flush=True)
        if not valid:
            print("bench: INVALID RESULT (flags %d, finite losses %s, parity %s)" % (bits, finite, parity and parity["ok"]),
                  file=sys.stderr, flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0 and not valid:
        sys.exit(3)


if __name__ == "__main__":
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)
