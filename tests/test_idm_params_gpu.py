"""Gradients of the IDM kernels with respect to the per-vehicle driver parameters params [6, V] (a_max, a_pref,
v_target, s0, time_pref, length), against autograd through the torch restatement of the step (tests/idm_restate.py,
pinned to the oracle by tests/test_idm_params_host.py).  The state adjoint of a launch that also returns the
parameter adjoint is bit for bit the one of the plain launch."""
import numpy as np
import pytest
import torch

from conftest import relerr
from idm_restate import rollout, step, lane_index

pytestmark = pytest.mark.gpu

UMAX, DT = 30.0, 0.01


def _lanes(sizes, rng):
    off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    V, L = int(off[-1]), len(sizes)
    p0 = np.concatenate([np.arange(n) * 15.0 + rng.uniform(0, 5, n) for n in sizes]) if V else np.zeros(0)
    v0 = rng.uniform(3, 21, V)
    par = np.stack([rng.uniform(1.5, 2.0, V) * UMAX, rng.uniform(1.0, 1.5, V) * UMAX, rng.uniform(0.8, 1.2, V) * UMAX,
                    rng.uniform(1, 2, V), rng.uniform(0.2, 0.6, V), rng.uniform(4.0, 6.0, V)])
    head = np.stack([rng.uniform(15, 1000, L), rng.uniform(-3, 3, L)], -1)
    return p0, v0, par, off, head


def _rows_close(a, b, tol):
    """Every parameter row of a within tol of b's largest entry in that row."""
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    if b.size == 0:
        return a.size == 0
    return all(relerr(a[r], b[r]) < tol for r in range(6))


def _reference(p0, v0, par, off, head, T, wp, wv, g_hist=None):
    """Autograd of the restatement: (g_params, g_p0, g_v0, g_head)."""
    t = lambda a: torch.tensor(np.asarray(a), dtype=torch.float64)
    tp, tv, th, tpar = (t(a).requires_grad_() for a in (p0, v0, head, par))
    pT, vT, ph, vh = rollout(tp, tv, tpar, off, th, DT, T)
    loss = (pT * t(wp)).sum() + (vT * t(wv)).sum()
    if g_hist is not None:
        loss = loss + (ph * t(g_hist[..., 0])).sum() + (vh * t(g_hist[..., 1])).sum()
    loss.backward()
    return tpar.grad.numpy(), tp.grad.numpy(), tv.grad.numpy(), th.grad.numpy()


def _gpu(dev, p0, v0, par, off, head, T, K, wp, wv, with_params, g_hist=None, dtype=torch.float64):
    """The functional API on the GPU; returns (g_params or None, g_p0, g_v0, g_head, flag bits)."""
    import dhts_b200
    from dhts_b200 import functional as F
    t = lambda a: torch.tensor(np.asarray(a), dtype=dtype, device=dev)
    flags = dhts_b200.Flags(dev)
    tp, tv, th, tpar = t(p0).requires_grad_(), t(v0).requires_grad_(), t(head).requires_grad_(), t(par)
    tpar.requires_grad_(with_params)
    off_t = torch.tensor(off, dtype=torch.int32, device=dev)
    if g_hist is None:
        pT, vT = F.idm_rollout(tp, tv, tpar, off_t, th, DT, T, ckpt_every=K, flags=flags)
        loss = (pT * t(wp)).sum() + (vT * t(wv)).sum()
    else:
        pT, vT, ph, vh = F.idm_rollout(tp, tv, tpar, off_t, th, DT, T, ckpt_every=1, flags=flags, return_history=True)
        loss = (pT * t(wp)).sum() + (vT * t(wv)).sum() + (ph * t(g_hist[..., 0])).sum() + (vh * t(g_hist[..., 1])).sum()
    loss.backward()
    bits, _ = flags.read()
    g = (lambda x: None if x is None else x.cpu().numpy())
    return g(tpar.grad), g(tp.grad), g(tv.grad), g(th.grad), bits


def _check_rollout(dev, p0, v0, par, off, head, T, K, g_hist=None, seed=0):
    rng = np.random.default_rng(seed)
    V = p0.shape[0]
    wp, wv = rng.normal(size=V), rng.normal(size=V)
    gpar, gp, gv, gh, bits = _gpu(dev, p0, v0, par, off, head, T, K, wp, wv, True, g_hist)
    _, gp_s, gv_s, gh_s, _ = _gpu(dev, p0, v0, par, off, head, T, K, wp, wv, False, g_hist)
    # the state adjoint of the parameter launch is that of the plain launch, bit for bit
    assert np.array_equal(gp, gp_s) and np.array_equal(gv, gv_s) and np.array_equal(gh, gh_s)
    rpar, rp, rv, rh = _reference(p0, v0, par, off, head, T, wp, wv, g_hist)
    assert _rows_close(gpar, rpar, 1e-9)
    if V:
        assert relerr(gp, rp) < 1e-9 and relerr(gv, rv) < 1e-9
    assert not bits & 2


def test_step_tight_gaps_both_clips(dev):
    """One step, gaps tight enough that both clips are active (no collision): g_params of the step kernel."""
    import dhts_b200
    from dhts_b200 import functional as F
    rng = np.random.default_rng(4)
    L, n = 6, 40
    V = L * n
    off = np.arange(L + 1) * n
    gap = rng.uniform(1.5, 4.0, (L, n))                 # bumper to bumper, to the leader
    v0 = rng.uniform(5, 25, V)
    crawl = rng.choice(V, V // 5, replace=False)
    v0[crawl] = 0.01
    gap.ravel()[crawl] = 0.3
    ln = rng.uniform(4.5, 5.5, (L, n))
    p0 = np.concatenate([np.concatenate([[0.0], np.cumsum(gap[l, :-1] + 0.5 * (ln[l, :-1] + ln[l, 1:]))])
                         for l in range(L)])
    par = np.stack([np.full(V, UMAX), np.full(V, 0.8 * UMAX), np.full(V, 0.9 * UMAX), rng.uniform(0.3, 0.7, V),
                    rng.uniform(0.05, 0.15, V), ln.ravel()])
    head = np.stack([rng.uniform(5, 50, L), rng.uniform(-3, 3, L)], -1)
    wp, wv = rng.normal(size=V), rng.normal(size=V)
    t = lambda a: torch.tensor(np.asarray(a), dtype=torch.float64)
    clips = []
    tpar = t(par).requires_grad_()
    np_, nv_ = step(t(p0), t(v0), tpar, lane_index(off), t(head), DT, clips)
    ((np_ * t(wp)).sum() + (nv_ * t(wv)).sum()).backward()
    ca, cs, col = clips[0]
    assert ca.any() and cs.any() and not col.any()
    outs = []
    for with_params in (True, False):
        d = lambda a: t(a).to(dev)
        flags = dhts_b200.Flags(dev)
        tp, tv, th, dpar = d(p0).requires_grad_(), d(v0).requires_grad_(), d(head).requires_grad_(), d(par)
        dpar.requires_grad_(with_params)
        a, b = F.idm_step(tp, tv, dpar, torch.tensor(off, dtype=torch.int32, device=dev), th, DT, flags)
        ((a * d(wp)).sum() + (b * d(wv)).sum()).backward()
        outs.append((dpar.grad, tp.grad.cpu().numpy(), tv.grad.cpu().numpy(), th.grad.cpu().numpy()))
        assert not flags.read()[0] & 2
    assert all(np.array_equal(x, y) for x, y in zip(outs[0][1:], outs[1][1:]))
    assert outs[1][0] is None
    assert _rows_close(outs[0][0].cpu().numpy(), tpar.grad.numpy(), 1e-9)


@pytest.mark.parametrize("sizes,T", [([0, 3, 0], 7), ([1], 40), ([32, 32], 37), ([33, 1, 0], 37), ([65, 7], 37),
                                     ([130, 2], 37), ([256, 3], 37), ([300, 4], 9)])
@pytest.mark.parametrize("K", [1, 5, 32])
def test_rollout_vs_restatement(dev, sizes, T, K):
    """Empty, single-vehicle and 32 / 33 / 65 / 130 / 256-vehicle lanes (one to eight slots per thread), and a
    300-vehicle lane on the per-step fallback (vehicle 256 starts a CTA of the step kernel mid-lane, so its follower's
    adjoint comes through the recompute path); checkpoint intervals 1, 5 (does not divide T) and 32."""
    rng = np.random.default_rng(sum(sizes) + T + K)
    p0, v0, par, off, head = _lanes(sizes, rng)
    _check_rollout(dev, p0, v0, par, off, head, T, K, seed=K)


@pytest.mark.parametrize("L,n,T", [(6, 64, 40), (33, 10, 25), (4, 200, 12), (3, 300, 6)])
def test_rollout_per_step_head_and_history(dev, L, n, T):
    """Head deltas per step and a loss on the state before every step (return_history=True, g_hist)."""
    rng = np.random.default_rng(L * 100 + n)
    p0, v0, par, off, _ = _lanes([n] * L, rng)
    head = np.stack([rng.uniform(15, 80, (T, L)), rng.uniform(-3, 3, (T, L))], -1)
    g_hist = rng.normal(size=(T, L * n, 2))
    _check_rollout(dev, p0, v0, par, off, head, T, 1, g_hist=g_hist, seed=n)


def test_shared_parameter_leaf_gets_the_sum(dev):
    """A [6, 1] leaf expanded over all vehicles receives the sum of the per-vehicle gradients (<= 1e-12); params is
    the only input that requires a gradient."""
    from dhts_b200 import functional as F
    rng = np.random.default_rng(21)
    p0, v0, par, off, head = _lanes([64] * 5, rng)
    V = p0.shape[0]
    t = lambda a: torch.tensor(np.asarray(a), dtype=torch.float64, device=dev)
    off_t = torch.tensor(off, dtype=torch.int32, device=dev)
    shared = t(par[:, :1]).requires_grad_()
    full = t(np.repeat(par[:, :1], V, axis=1)).requires_grad_()
    for leaf, prm in ((shared, shared.expand(6, V)), (full, full)):
        pT, vT = F.idm_rollout(t(p0), t(v0), prm, off_t, t(head), DT, 30, ckpt_every=8)
        assert pT.requires_grad
        ((pT - t(p0)) ** 2).sum().add((vT ** 2).sum()).backward()
    assert relerr(shared.grad.cpu()[:, 0], full.grad.sum(1).cpu()) < 1e-12


@pytest.mark.parametrize("n,K", [(64, 16), (20, 1), (300, 4)])
def test_parameter_path_nan_flag(dev, n, K):
    """A NaN terminal adjoint raises the NaN-gradient flag on the parameter path too; clean inputs leave it clear."""
    import dhts_b200
    from dhts_b200 import functional as F
    from dhts_b200._lib import FLAG_NAN_GRAD
    rng = np.random.default_rng(n)
    p0, v0, par, off, head = _lanes([n] * 3, rng)
    t = lambda a: torch.tensor(np.asarray(a), dtype=torch.float64, device=dev)
    for poison in (False, True):
        flags = dhts_b200.Flags(dev)
        tpar = t(par).requires_grad_()
        pT, vT = F.idm_rollout(t(p0), t(v0), tpar, torch.tensor(off, dtype=torch.int32, device=dev), t(head), DT, 40,
                               ckpt_every=K, flags=flags)
        w = torch.ones_like(vT)
        if poison:
            w[n + n // 2] = float("nan")
        (vT * w).sum().backward()
        assert bool(flags.read()[0] & FLAG_NAN_GRAD) == poison
        assert bool(torch.isnan(tpar.grad).any()) == poison


def test_fp32_parameter_gradient_vs_fp64(dev):
    """fp32 kernels against the fp64 kernels on the same inputs, T = 100: every parameter row within 5e-4 of its
    largest fp64 entry (measured on a B200: 7.9e-5 in the worst row)."""
    rng = np.random.default_rng(32)
    p0, v0, par, off, head = _lanes([64] * 4 + [20, 130], rng)
    V = p0.shape[0]
    wp, wv = rng.normal(size=V), rng.normal(size=V)
    g64 = _gpu(dev, p0, v0, par, off, head, 100, 16, wp, wv, True)[0]
    g32 = _gpu(dev, p0, v0, par, off, head, 100, 16, wp, wv, True, dtype=torch.float32)[0]
    err = max(relerr(g32[r], g64[r]) for r in range(6))
    print("fp32 vs fp64 g_params, worst row:", err)
    assert err < 5e-4


def test_calibration_end_to_end(dev):
    """Calibrate per-lane IDM parameters from a whole trajectory: 8 lanes x 20 vehicles with heterogeneous gaps, one
    true parameter set per lane, fitted from a +-15 % start with Adam (log-scale parameters) on the mean squared error
    of (p, v) at every step (return_history=True).  The loss falls by >= 10x and every lane's parameter error
    shrinks.  Measured on a B200 with 300 iterations: the loss falls 10 524x, the lanes' relative parameter errors
    (2-norm over the six rows) go from 0.367 to 0.007 - 0.277."""
    from dhts_b200 import functional as F
    rng = np.random.default_rng(5)
    L, n, T, dt = 8, 20, 250, 0.02
    V = L * n
    off = np.arange(L + 1) * n
    gap = rng.uniform(2.0, 30.0, (L, n))
    p0 = np.concatenate([np.concatenate([[0.0], np.cumsum(gap[l, :-1] + 5.0)]) for l in range(L)])
    v0 = rng.uniform(5, 25, V)
    true = np.stack([rng.uniform(1.5, 2.0, L) * UMAX, rng.uniform(1.0, 1.5, L) * UMAX, rng.uniform(0.8, 1.2, L) * UMAX,
                     rng.uniform(1, 2, L), rng.uniform(0.2, 0.6, L), rng.uniform(4.5, 5.5, L)])
    head = np.stack([rng.uniform(10, 40, L), rng.uniform(-2, 2, L)], -1)
    init = true * (1 + 0.15 * rng.choice([-1.0, 1.0], true.shape))
    t = lambda a: torch.tensor(np.asarray(a), dtype=torch.float64, device=dev)
    lane = torch.as_tensor(np.repeat(np.arange(L), n), device=dev)
    off_t = torch.tensor(off, dtype=torch.int32, device=dev)
    run = lambda prm: F.idm_rollout(t(p0), t(v0), prm[:, lane], off_t, t(head), dt, T, ckpt_every=1,
                                    return_history=True)
    with torch.no_grad():
        _, _, ph_o, vh_o = run(t(true))
    u = torch.zeros((6, L), dtype=torch.float64, device=dev, requires_grad=True)
    opt = torch.optim.Adam([u], lr=0.02)

    def loss_fn():
        _, _, ph, vh = run(t(init) * torch.exp(u))
        return ((ph - ph_o) ** 2 + (vh - vh_o) ** 2).mean()
    l0 = None
    for _ in range(300):
        opt.zero_grad()
        loss = loss_fn()
        loss.backward()
        opt.step()
        l0 = loss.item() if l0 is None else l0
    with torch.no_grad():
        lf = loss_fn().item()
    err0 = np.linalg.norm(init / true - 1, axis=0)
    err1 = np.linalg.norm(init * np.exp(u.detach().cpu().numpy()) / true - 1, axis=0)
    print("calibration: loss %.3e -> %.3e (%.0fx); lane errors %s -> %s" % (l0, lf, l0 / lf, err0.round(3), err1.round(3)))
    assert l0 / lf >= 10.0
    assert (err1 < err0).all()

