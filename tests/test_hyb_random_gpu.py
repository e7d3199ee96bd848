"""The fused hybrid rollout (dhts_hyb_rollout_{fwd,bwd}_*) against the drop-in RoadNetwork stepped on the CPU
(tests/hyb_random_cases.py), on random plain-mode networks, degenerate networks and every launch shape of
``dhts_hyb_rollout_*`` (csrc/net_hybrid.cu:989-1128).  Bars as in tests/test_hyb_gpu.py: vehicle counts, spawn counters and
the step of every event exact; cells, capacitors and vehicles within 1e-9 absolute; gradients within 1e-8 of the largest
entry.  Launch shapes are read from the profiler trace (kernel, block, grid, dynamic shared memory)."""
import json
import os
import tempfile

import numpy as np
import pytest
import torch

import hyb_random_cases as H
from conftest import relerr
from hyb_random_cases import DEGENERATE, RANDOM, seeds_of

pytestmark = pytest.mark.gpu
F64 = torch.float64
SMEM_MAX = 227 * 1024


# ------------------------------------------------------------------------------------------------ launch-shape restatement
def hyb_threads(topo, R, sms):
    """hyb_threads (net_hybrid.cu:989-995)."""
    NI, sides = topo.NC + topo.L - topo.ML, 2 * topo.L + topo.ML
    w = max(NI, sides)
    if R > sms:
        w = (w + 1) // 2
    t = (w + 31) // 32 * 32
    return min(512, max(32, t))


def hyb_smem(topo, n_par, adj, prefetch, esz=8):
    """hyb_smem (net_hybrid.cu:997-1019); sizeof(HeadRec) is 152 (fp64) / 88 (fp32), sizeof(IdmPar) 6 reals."""
    a8 = lambda x: (x + 7) // 8 * 8
    NC, L, ML, cap, NCAP, n_own, AUX = topo.NC, topo.L, topo.ML, topo.veh_cap, topo.NCAP, topo.n_own, topo.AUX
    NGL, NG, MAXT = sum(len(g) for g in topo.groups), len(topo.groups), topo.MAXT
    el = 8 * NC + 4 * n_own + 2 * AUX + 5 * ML
    by = 0
    if adj:
        el += 3 * NC + NGL * (3 + MAXT)
        el += 3 * NC + 2 * n_own + 3 * ML * cap + NCAP + 6 * L + 5 * ML
        if prefetch:
            el += 4 * NC + 2 * n_own + AUX
        by += 4 * (4 * ML + 4 * NGL)
    NI = NC + (L - ML)
    el += 4 * L + 2 * NI + (4 * (L - ML) if adj else 0)
    by += a8(4 * (L + 1)) + a8(4 * NI) + a8(4 * NC) + esz * 2 * L + (a8(16 * L) + esz * 6 * L if adj and prefetch else 0)
    by += 4 * 6 * NGL + esz
    by += 4 * (NG + 1) + esz
    el += NGL
    by += 6 * esz * n_par + esz
    by += 4 * 2 * ML + esz
    by += 4 * (NG + NGL) + esz
    by += (152 if esz == 8 else 88) * ML + esz
    return esz * el + by + 32


def launches(prof):
    """Kernel launches of the hybrid rollout in a profiler run: name, grid, block, dynamic shared memory."""
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            ev = json.load(f)["traceEvents"]
    out = []
    for e in ev:
        if e.get("cat") == "kernel" and "hyb_rollout" in e.get("name", ""):
            a = e["args"]
            out.append(dict(name=e["name"], grid=tuple(a["grid"]), block=tuple(a["block"]), smem=int(a["shared memory"])))
    return out


def sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count


# ------------------------------------------------------------------------------------------------ run and compare
def run(dev, pairs, topo, dtype=F64, inp=None, T=None, backward=True, profile=False):
    from torch.profiler import ProfilerActivity, profile as prof_ctx

    from dhts_b200 import Flags
    from dhts_b200.hybrid_network import hybrid_rollout
    inp = inp or H.pack(pairs, topo, dev, dtype)
    T = T or inp["T"]
    flags = Flags(dev)
    ctx = prof_ctx(activities=[ProfilerActivity.CUDA]) if profile else None
    if ctx:
        ctx.__enter__()
    try:
        st = hybrid_rollout(topo, inp["r0"], inp["u0"], H.UMAX, H.DT, T, route=inp["route"][:, :T].contiguous(),
                            spawn_route=inp["spawn_route"], own0=inp["own0"], aux0=inp["aux0"], veh_params=inp["veh_params"],
                            flags=flags)
        fwd_bits = flags.read()
        if backward:
            H.kernel_loss(st, pairs, T).backward()
        torch.cuda.synchronize(dev)
    finally:
        if ctx:
            ctx.__exit__(None, None, None)
    return dict(st=st, inp=inp, flags=flags, fwd_bits=fwd_bits, prof=ctx)


def compare(o, pairs, T=None, grads=True, devs=None, replicas=None):
    """Every replica against its reference run; returns the largest deviation per assertion group."""
    st, inp = o["st"], o["inp"]
    topo = st.topo
    T = T or inp["T"]
    devs = devs if devs is not None else {}
    bump = lambda k, x: devs.__setitem__(k, max(devs.get(k, 0.0), float(x)))
    assert o["flags"].read() == (0, 0), "no collision, CFL, NaN, route or overflow flag"
    cells = st.cells.detach().cpu().numpy()
    cnt = st.count.cpu().numpy()
    nsp = st.aux[:, :, topo.A_NSP:topo.A_NSP + topo.ML].detach().round().long().cpu().numpy()
    capac = st.capacitor.detach().cpu().numpy()
    p, v, a, valid = (x.detach().cpu().numpy() for x in st.by_rank())
    for b, (case, ref) in (replicas or list(enumerate(pairs))):
        assert (cnt[:, b] == ref.count[:T + 1]).all(), (case.seed, "vehicle counts per step")
        spawned = np.zeros((T + 1, topo.ML), dtype=np.int64)
        for t, l, _ in ref.spawns:
            if t <= T:
                spawned[t:, topo.mic_of[l]] += 1
        assert (nsp[:, b] == spawned).all(), (case.seed, "spawn counters per step")
        rc = np.stack(ref.cells[:T + 1])
        bump("cells", np.abs(cells[:, b] - rc).max() if rc.size else 0.0)
        if topo.NCAP:
            bump("capacitors", np.abs(capac[:, b] - ref.capac[:T + 1]).max())
        for t in range(T + 1):
            for m in range(topo.ML):
                n = int(ref.count[t, m])
                if n:
                    rv = np.array(ref.veh[t][m])
                    bump("vehicles", np.abs(np.stack([p[t, b, m, :n], v[t, b, m, :n], a[t, b, m, :n]], -1) - rv).max())
        if grads:
            gr, gu = inp["r0"].grad[b].cpu().numpy(), inp["u0"].grad[b].cpu().numpy()
            if topo.NC:
                bump("g_cells", max(relerr(gr, ref.g_r0), relerr(gu, ref.g_u0)))
            if topo.ML:
                gp, gv = inp["p0"].grad[b].cpu().numpy(), inp["v0"].grad[b].cpu().numpy()
                rp = np.concatenate([np.array(x) for x in ref.g_p0]); rv_ = np.concatenate([np.array(x) for x in ref.g_v0])
                if rp.size:
                    op = np.concatenate([gp[m, :len(ref.g_p0[m])] for m in range(topo.ML)])
                    ov = np.concatenate([gv[m, :len(ref.g_v0[m])] for m in range(topo.ML)])
                    bump("g_vehicles", max(relerr(op, rp), relerr(ov, rv_)))
    for k, bar in (("cells", 1e-9), ("capacitors", 1e-9), ("vehicles", 1e-9), ("g_cells", 1e-8), ("g_vehicles", 1e-8)):
        assert devs.get(k, 0.0) < bar, (k, devs[k])
    return devs


def _report(tag, devs, extra=""):
    print("\nDEV %s %s %s" % (tag, " ".join("%s=%.2e" % kv for kv in sorted(devs.items())), extra))


def _pairs(name, layout, R=3, T=None):
    return [H.reference(name, s, layout, T) for s in seeds_of(name, layout, R)]


# ------------------------------------------------------------------------------------------------ random and degenerate networks
@pytest.mark.parametrize("name,layout", RANDOM)
def test_random_network_matches_cpu_reference(dev, name, layout):
    """Three replicas with their own initial states, vehicles, MacroRoutes and spawn routes, 200-300 steps."""
    pairs = _pairs(name, layout)
    topo = H.topology(pairs[0][0], dev)
    o = run(dev, pairs, topo)
    _report("%s-%d" % (name, layout), compare(o, pairs))


@pytest.mark.parametrize("name", DEGENERATE)
def test_degenerate_network_matches_cpu_reference(dev, name):
    """ML = 0, NC = 0 (initial vehicles, hand-offs, drops), a single micro lane, a single macro lane."""
    pairs = _pairs(name, 1)
    topo = H.topology(pairs[0][0], dev)
    assert {"macro_only": topo.ML == 0, "micro_only": topo.NC == 0, "single_micro": topo.L == 1 and topo.NC == 0,
            "single_macro": topo.L == 1 and topo.ML == 0}[name]
    o = run(dev, pairs, topo)
    _report(name, compare(o, pairs))


# ------------------------------------------------------------------------------------------------ launch shapes
def test_512_thread_adjoint_matches_cpu_reference(dev):
    """(a) more than 192 interfaces: hyb_rollout_bwd_kernel<double, 512>, compared with the reference."""
    pairs = _pairs("wide", 1)
    topo = H.topology(pairs[0][0], dev)
    o = run(dev, pairs, topo, profile=True)
    ls = launches(o["prof"])
    thr = hyb_threads(topo, len(pairs), sm_count())
    assert thr > 192
    n_par = len(o["inp"]["veh_params"])
    fwd = [x for x in ls if "hyb_rollout_fwd_kernel<double>" in x["name"]]
    bwd = [x for x in ls if "hyb_rollout_bwd_kernel<double, 512>" in x["name"]]
    assert len(fwd) == 1 and len(bwd) == 1 and len(ls) == 2, ls
    assert bwd[0]["block"] == (thr, 1, 1) and bwd[0]["grid"] == (len(pairs), 1, 1)
    assert bwd[0]["smem"] == hyb_smem(topo, n_par, True, True) <= SMEM_MAX
    assert fwd[0]["smem"] == hyb_smem(topo, n_par, False, False)
    _report("wide", compare(o, pairs), str(ls))


def _tile(pairs, inp, R, place, dev, noise=1e-3, seed=0):
    """R replicas: the reference replicas at the indices `place`, perturbed copies of them (r0 and u0 scaled by
    1 + noise * N(0, 1)) everywhere else."""
    rng = np.random.default_rng(seed)
    src = np.arange(R) % len(pairs)
    src[list(place)] = np.arange(len(pairs))
    idx = torch.tensor(src, device=dev)
    scale = torch.tensor(1 + noise * rng.normal(size=(R, inp["r0"].shape[1])), dtype=F64, device=dev)
    scale[list(place)] = 1.0
    out = dict(inp)
    out["r0"] = (inp["r0"].detach()[idx] * scale).clamp(0.05, 0.9).requires_grad_()
    out["u0"] = (inp["u0"].detach()[idx] * scale).requires_grad_()
    p0, v0 = inp["p0"].detach()[idx].requires_grad_(), inp["v0"].detach()[idx].requires_grad_()
    out["p0"], out["v0"] = p0, v0
    out["aux0_base"] = inp["aux0"].detach()[idx]
    out["own0"] = inp["own0"][idx].contiguous()
    out["route"] = inp["route"][idx].contiguous()
    out["spawn_route"] = inp["spawn_route"][idx].contiguous()
    out["R"] = R
    return out


def _with_leaves(topo, inp):
    """aux0 rebuilt from the p0 / v0 leaves (the rest of the rows as they are)."""
    s = topo.ML * topo.veh_cap
    base = inp["aux0_base"]
    inp = dict(inp)
    inp["aux0"] = torch.cat([inp["p0"].reshape(-1, s), inp["v0"].reshape(-1, s), base[:, 2 * s:]], dim=1)
    return inp


def test_many_replicas_loop_and_match(dev):
    """(b) R > sm_count() and R > the grid of both launches: half-size CTAs whose threads loop over (side, lane) pairs,
    each CTA several replicas in turn.  Four replicas (the last one among them) against the reference; all replicas
    against the same replicas run in batches of at most sm_count() (full-size CTAs, one replica each); permuted replicas
    give permuted results."""
    sms = sm_count()
    ref_pairs = _pairs("many_sides", 1, R=4)
    topo = H.topology(ref_pairs[0][0], dev)
    assert 2 * topo.L + topo.ML > topo.NC + topo.L - topo.ML, "sides must set the thread count"
    base = H.pack(ref_pairs, topo, dev)
    R = 32 * sms + 3                    # above any persistent grid: at most 32 resident CTAs per SM
    place = [0, 1, R // 2, R - 1]
    inp = _with_leaves(topo, _tile(ref_pairs, base, R, place, dev))
    thr = hyb_threads(topo, R, sms)
    assert thr < 2 * topo.L + topo.ML and thr == hyb_threads(topo, 1, sms) // 2
    pairs = [None] * R
    for i, k in enumerate(place):
        pairs[k] = ref_pairs[i]
    loss_pairs = [pairs[k] if pairs[k] is not None else ref_pairs[k % 4] for k in range(R)]
    o = run(dev, loss_pairs, topo, inp=inp, profile=True)
    ls = launches(o["prof"])
    assert len(ls) == 2, ls
    for x in ls:
        assert x["block"] == (thr, 1, 1) and x["grid"][0] < R and x["grid"][0] >= sms, x
    devs = compare(o, ref_pairs, replicas=[(k, ref_pairs[i]) for i, k in enumerate(place)])
    hist, aux = o["st"].hist.detach(), o["st"].aux.detach()
    grads = [inp[k].grad.detach() for k in ("r0", "u0", "p0", "v0")]
    # the same replicas in batches of at most sm_count(): full-size CTAs, one replica per CTA
    worst, bitwise = 0.0, True
    for lo in range(0, R, sms):
        sl = slice(lo, min(R, lo + sms))
        sub = {k: (v[sl] if torch.is_tensor(v) and v.dim() and v.shape[0] == R else v) for k, v in inp.items()}
        sub = {k: (v.detach().requires_grad_() if k in ("r0", "u0", "p0", "v0") else v) for k, v in sub.items()}
        sub["R"] = sl.stop - sl.start
        sub = _with_leaves(topo, sub)
        ob = run(dev, loss_pairs[sl], topo, inp=sub, profile=lo == 0)
        if lo == 0:
            for x in launches(ob["prof"]):
                assert x["block"] == (hyb_threads(topo, 1, sms), 1, 1) and x["grid"][0] == sub["R"], x
        assert ob["flags"].read() == (0, 0)
        pairs_ab = [(hist[:, sl], ob["st"].hist.detach()), (aux[:, sl], ob["st"].aux.detach())]
        pairs_ab += [(g[sl], sub[k].grad) for g, k in zip(grads, ("r0", "u0", "p0", "v0"))]
        for x, y in pairs_ab:
            bitwise &= bool(torch.equal(x, y))
            worst = max(worst, float((x - y).abs().max() / (1e-300 + y.abs().max())))
    assert worst < 1e-13
    # permuting the replicas permutes the results
    perm = torch.tensor(np.random.default_rng(3).permutation(R), device=dev)
    pin = {k: (v.detach()[perm] if torch.is_tensor(v) and v.dim() and v.shape[0] == R else v) for k, v in inp.items()}
    pin = {k: (v.requires_grad_() if k in ("r0", "u0", "p0", "v0") else v) for k, v in pin.items()}
    pin = _with_leaves(topo, pin)
    op = run(dev, [loss_pairs[int(i)] for i in perm.tolist()], topo, inp=pin)
    assert torch.equal(op["st"].hist.detach(), hist[:, perm]) and torch.equal(op["st"].aux.detach(), aux[:, perm])
    for g, k in zip(grads, ("r0", "u0", "p0", "v0")):
        assert torch.equal(pin[k].grad, g[perm])
    _report("many_sides", devs, "R=%d grid=%s threads=%d batched_rel=%.1e bitwise=%s" % (R, [x["grid"][0] for x in ls], thr, worst, bitwise))


def test_adjoint_without_prefetch_matches_cpu_reference(dev):
    """(c) about 1500 macro cells: the fp64 adjoint needs more than 227 KB with prefetch and fits without it."""
    pairs = _pairs("big", 1)
    topo = H.topology(pairs[0][0], dev)
    o = run(dev, pairs, topo, profile=True)
    n_par = len(o["inp"]["veh_params"])
    assert hyb_smem(topo, n_par, True, True) > SMEM_MAX >= hyb_smem(topo, n_par, True, False)
    ls = launches(o["prof"])
    bwd = [x for x in ls if "hyb_rollout_bwd_kernel<double, 512>" in x["name"]]
    assert len(bwd) == 1 and len(ls) == 2, ls
    assert bwd[0]["smem"] == hyb_smem(topo, n_par, True, False) and bwd[0]["block"] == (512, 1, 1)
    _report("big", compare(o, pairs), str(ls))


def test_adjoint_too_large_is_refused_after_a_clean_forward(dev):
    """(d) about 2000 macro cells: the forward fits in shared memory, the adjoint does not even without prefetch.  Today
    the forward runs (and matches the reference) and backward() raises UnsupportedShape without launching."""
    from dhts_b200 import _lib
    pairs = _pairs("huge", 1)
    topo = H.topology(pairs[0][0], dev)
    inp = H.pack(pairs, topo, dev)
    n_par = len(inp["veh_params"])
    assert hyb_smem(topo, n_par, False, False) <= SMEM_MAX < hyb_smem(topo, n_par, True, False)
    o = run(dev, pairs, topo, inp=inp, backward=False)
    devs = compare(o, pairs, grads=False)
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        with pytest.raises(_lib.UnsupportedShape):
            H.kernel_loss(o["st"], pairs, o["inp"]["T"]).backward()
        torch.cuda.synchronize(dev)
    assert not [x for x in launches(prof) if "bwd" in x["name"]]
    assert o["flags"].read() == (0, 0)
    _report("huge", devs)


# ------------------------------------------------------------------------------------------------ fp32, overflow
@pytest.mark.parametrize("name,layout,T", [("branch", 1, 60), ("wide", 1, 60)])
def test_f32_tracks_f64(dev, name, layout, T):
    """fp32 against the fp64 kernel on a horizon where the discrete events agree: states within 2e-4 of the largest
    entry, gradients within 5e-2 (the bars of test_f32_build_tracks_f64_on_a_short_horizon)."""
    pairs = _pairs(name, layout)
    topo = H.topology(pairs[0][0], dev)
    out = {}
    for dt in (F64, torch.float32):
        o = run(dev, pairs, topo, dtype=dt, T=T)
        assert o["flags"].read()[0] & ~4 == 0
        st = o["st"]
        out[dt] = (st.cells.detach().double().cpu().numpy(), st.count.cpu().numpy(), o["inp"]["r0"].grad.double().cpu().numpy(),
                   st.aux[:, :, topo.A_NSP:topo.A_NSP + topo.ML].detach().round().cpu().numpy())
    a, b = out[F64], out[torch.float32]
    assert (a[1] == b[1]).all() and (a[3] == b[3]).all(), "discrete events differ"
    assert a[3].max() >= 1, "the horizon must include a spawn"
    ds, dg = np.abs(a[0] - b[0]).max() / np.abs(a[0]).max(), relerr(b[2], a[2])
    assert ds < 2e-4 and np.isfinite(b[2]).all() and dg < 5e-2
    print("\nDEV f32-%s states=%.2e grads=%.2e" % (name, ds, dg))


def test_vehicle_overflow_is_flagged(dev):
    """A spawn-route list one entry wide for a lane the reference spawns eight vehicles into: the second spawn overflows
    it, the kernel reports FLAG_VEH_OVERFLOW and flags.check() raises."""
    from dhts_b200._lib import FLAG_VEH_OVERFLOW
    pairs = _pairs("merge_drop", 4, R=1)
    topo = H.topology(pairs[0][0], dev)
    assert max(sum(1 for s in pairs[0][1].spawns if s[1] == l) for l in topo.micro) >= 2
    o = run(dev, pairs, topo, inp=H.pack(pairs, topo, dev, KS=1), backward=False)
    bits, _ = o["flags"].read()
    assert bits & FLAG_VEH_OVERFLOW
    with pytest.raises(RuntimeError):
        o["flags"].check()
