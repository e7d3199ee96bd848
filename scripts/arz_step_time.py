"""Single-step ARZ kernels of two builds of the library, alternated in one process: dhts_arz_step_{fwd,bwd}_{f64,f32}
called through ctypes from two shared libraries given by path (e.g. this tree's and a parent commit's, built
separately).  Shapes: B = 1, N = 1024 (latency of the drop-in object API), B = 8192, N = 1024 (throughput; the inputs do
not fit in L2) and B = 64, N = 3000 (lanes too long for the fused rollouts).  After warm-up, each timing is one CUDA-event
pair around --inner back-to-back calls; the median of --reps timings per call is printed beside the GPU's name and power
limit, and as one JSON line.  Both builds also get the same inputs once and must agree within --tol."""
import argparse
import ctypes
import json
import subprocess

import numpy as np
import torch

SHAPES = ((1, 1024), (8192, 1024), (64, 3000))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--new", required=True, help="path of the library under test")
    ap.add_argument("--old", required=True, help="path of the library to compare with")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--reps", type=int, default=15)
    ap.add_argument("--inner", type=int, default=20)
    ap.add_argument("--tol", type=float, default=1e-9, help="largest relative difference of the two builds' outputs (fp64)")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a GPU"
    dev = torch.device("cuda:0")
    gpu = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    print("GPU:", gpu)
    libs = {"new": ctypes.CDLL(a.new), "old": ctypes.CDLL(a.old)}
    p = lambda t: ctypes.c_void_p(0 if t is None else t.data_ptr())
    stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    rng = np.random.default_rng(0)
    results = []
    for dtype, suf, real in ((torch.float64, "f64", ctypes.c_double), (torch.float32, "f32", ctypes.c_float)):
        for B, N in SHAPES:
            t = lambda x: torch.tensor(x, dtype=dtype, device=dev)
            dx, umax, dt = 5.0, 30.0, 0.01
            r = t(rng.uniform(0, 1, (B, N + 2))); u = t(rng.uniform(0, umax, (B, N + 2)))
            y = r * (u - umax * (1 - torch.sqrt(r + 1e-5)))
            dxs, ums = t(np.full(B, dx)), t(np.full(B, umax))
            g = [t(rng.normal(size=(B, N))) for _ in range(3)]
            flags = torch.zeros(4, dtype=torch.int32, device=dev)
            outs = {}
            calls = {}
            for name, lib in libs.items():
                nr, ny, nu = (torch.empty((B, N), dtype=dtype, device=dev) for _ in range(3))
                gr, gy = torch.empty_like(r), torch.empty_like(r)
                fwd, bwd = getattr(lib, f"dhts_arz_step_fwd_{suf}"), getattr(lib, f"dhts_arz_step_bwd_{suf}")

                def f(fwd=fwd, nr=nr, ny=ny, nu=nu):
                    rc = fwd(p(r), p(y), p(u), p(None), p(dxs), p(ums), real(dt), B, N, p(nr), p(ny), p(nu), p(None), p(flags),
                             stream)
                    assert rc == 0, rc

                def b(bwd=bwd, nr=nr, ny=ny, gr=gr, gy=gy):
                    rc = bwd(p(r), p(y), p(u), p(None), p(dxs), p(ums), real(dt), B, N, p(nr), p(ny), p(g[0]), p(g[1]),
                             p(g[2]), p(gr), p(gy), p(flags), stream)
                    assert rc == 0, rc

                f(); b()
                outs[name] = [x.clone() for x in (nr, ny, nu, gr, gy)]
                calls[name] = {"fwd": f, "bwd": b}
            torch.cuda.synchronize()
            assert int(flags[0]) == 0, "flags raised: %d" % int(flags[0])
            diff = max(((x - z).abs().max() / z.abs().max().clamp_min(1e-30)).item()
                       for x, z in zip(outs["new"], outs["old"]))
            assert diff < (a.tol if dtype == torch.float64 else 1e-4), ("builds disagree", suf, B, N, diff)
            for d in ("fwd", "bwd"):
                ms = {k: [] for k in libs}
                for rep in range(a.warmup + a.reps):
                    for name in libs:
                        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        e0.record()
                        for _ in range(a.inner):
                            calls[name][d]()
                        e1.record()
                        e1.synchronize()
                        if rep >= a.warmup:
                            ms[name].append(e0.elapsed_time(e1) * 1e3 / a.inner)
                row = {"dtype": suf, "dir": d, "B": B, "N": N, "max_rel_diff": diff}
                for name in libs:
                    v = np.array(ms[name])
                    row[name + "_us"] = float(np.median(v))
                    row[name + "_spread_us"] = float(v.max() - v.min())
                row["new_over_old"] = row["new_us"] / row["old_us"]
                results.append(row)
                print("%s %s B=%5d N=%4d  new %9.2f us  old %9.2f us  new/old %.3f  (spread new %.2f, old %.2f us)" % (
                    suf, d, B, N, row["new_us"], row["old_us"], row["new_over_old"], row["new_spread_us"],
                    row["old_spread_us"]))
    print(json.dumps({"gpu": gpu, "inner": a.inner, "reps": a.reps, "results": results}))


if __name__ == "__main__":
    main()
