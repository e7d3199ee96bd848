"""Cost of the IDM parameter adjoint: dhts_idm_rollout_bwd_f64 (state adjoint) against
dhts_idm_rollout_bwd_params_f64 (state + parameter adjoint) at the bench's IDM shape -- 4,194,304 vehicles in 64-vehicle
lanes, 1000 steps, ckpt_every 16, fp64, bench.py's synthetic inputs.  One forward fills the checkpoints; the two
adjoints then run alternately after warm-up, each timed with CUDA events.  Prints the GPU's name and power limit
beside the times, and one JSON line."""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lanes", type=int, default=65536)
    ap.add_argument("--lane-vehicles", type=int, default=64)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--ckpt-every", type=int, default=16)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--reps", type=int, default=10)
    a = ap.parse_args()
    import torch
    import bench
    import dhts_b200
    from dhts_b200._lib import check, creal, ptr, stream_ptr
    assert torch.cuda.is_available(), "needs a GPU"
    dev = torch.device("cuda:0")
    gpu = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    print("GPU:", gpu)
    d = bench.make_idm_inputs(types.SimpleNamespace(micro_lanes=a.lanes, lane_vehicles=a.lane_vehicles), 0, torch)
    f64 = lambda x: x.to(device=dev, dtype=torch.float64).contiguous()
    p0, v0, par, head, tp, tv = (f64(d[k]) for k in ("p0", "v0", "params", "head", "tp", "tv"))
    off = d["off"].to(dev)
    V, L, n, T, K = p0.numel(), a.lanes, a.lane_vehicles, a.steps, a.ckpt_every
    lib = dhts_b200._lib.load()
    flags = dhts_b200.Flags(dev)
    S = (T + K - 1) // K
    ckpt = torch.empty((S, 2, V), dtype=torch.float64, device=dev)
    pT, vT = torch.empty_like(p0), torch.empty_like(p0)
    dt = creal(torch.float64, d["dt"])
    check(lib.dhts_idm_rollout_fwd_f64(ptr(p0), ptr(v0), ptr(par), ptr(off), ptr(head), ptr(None), dt, V, L, n, T, K,
                                       ptr(ckpt), ptr(pT), ptr(vT), ptr(flags.t), stream_ptr(dev)), "fwd")
    g_pT, g_vT = 2.0 * (pT - tp), 2.0 * (vT - tv)                # the bench's loss
    g_p0, g_v0, g_head = torch.empty_like(p0), torch.empty_like(p0), torch.empty_like(head)
    g_par = torch.empty_like(par)
    base = lambda: (ptr(ckpt), ptr(par), ptr(off), ptr(head), ptr(None), dt, V, L, n, T, K, ptr(g_pT), ptr(g_vT),
                    ptr(None), ptr(g_p0), ptr(g_v0), ptr(g_head), ptr(None))
    calls = {
        "plain": lambda: check(lib.dhts_idm_rollout_bwd_f64(*base(), ptr(flags.t), stream_ptr(dev)), "bwd"),
        "params": lambda: check(lib.dhts_idm_rollout_bwd_params_f64(*base(), ptr(g_par), ptr(flags.t), stream_ptr(dev)),
                                "bwd_params"),
    }
    ms = {k: [] for k in calls}
    for rep in range(a.warmup + a.reps):
        for k, fn in calls.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); fn(); e1.record()
            torch.cuda.synchronize()
            if rep >= a.warmup:
                ms[k].append(e0.elapsed_time(e1))
    bits, _ = flags.read()
    med = {k: sorted(v)[len(v) // 2] for k, v in ms.items()}
    for k, v in ms.items():
        print("%-6s adjoint: median %.2f ms, min %.2f, max %.2f (%d runs)" % (k, med[k], min(v), max(v), len(v)))
    print("parameter adjoint / state adjoint: %.3f" % (med["params"] / med["plain"]))
    print(json.dumps({"gpu": gpu, "vehicles": V, "lane_vehicles": n, "steps": T, "ckpt_every": K, "dtype": "f64",
                      "plain_ms": med["plain"], "params_ms": med["params"], "ratio": med["params"] / med["plain"],
                      "flags": bits, "finite": bool(torch.isfinite(g_par).all())}))


if __name__ == "__main__":
    main()
