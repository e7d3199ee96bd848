"""The torch restatement of the IDM step (tests/idm_restate.py) is the reference of the GPU parameter adjoint
(tests/test_idm_params_gpu.py).  Here, on the CPU, it is pinned to the oracle: its forward and its autograd state
gradients match oracle.idm_rollout, and its parameter gradients match central differences of the oracle's forward."""
import ctypes

import numpy as np
import pytest
import torch

from conftest import relerr
from idm_restate import rollout

UMAX, DT = 30.0, 0.01


def _lanes(sizes, rng, spacing=15.0, v_lo=3.0, v_hi=21.0):
    off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    V, L = int(off[-1]), len(sizes)
    p0 = np.concatenate([np.arange(n) * spacing + rng.uniform(0, 5, n) for n in sizes]) if V else np.zeros(0)
    v0 = rng.uniform(v_lo, v_hi, V)
    par = np.stack([rng.uniform(1.5, 2.0, V) * UMAX, rng.uniform(1.0, 1.5, V) * UMAX, rng.uniform(0.8, 1.2, V) * UMAX,
                    rng.uniform(1, 2, V), rng.uniform(0.2, 0.6, V), rng.uniform(4.0, 6.0, V)])
    head = np.stack([rng.uniform(15, 1000, L), rng.uniform(-3, 3, L)], -1)
    return p0, v0, par, off, head


def _clipped_lanes(rng, L=5, n=12):
    """Tight but positive gaps: crawling vehicles behind a close leader clip their acceleration, fast ones behind a much
    faster leader clip s*; no collision within a few steps."""
    off = np.arange(L + 1) * n
    V = L * n
    gap = rng.uniform(1.5, 4.0, (L, n))                 # bumper to bumper, to the leader
    v0 = rng.uniform(5, 25, V)
    crawl = rng.choice(V, V // 5, replace=False)
    v0[crawl] = 0.01
    gap.ravel()[crawl] = 0.3
    p0 = np.concatenate([np.concatenate([[0.0], np.cumsum(gap[l, :-1] + 5.0)]) for l in range(L)])
    par = np.stack([np.full(V, UMAX), np.full(V, 0.8 * UMAX), np.full(V, 0.9 * UMAX), np.full(V, 0.5), np.full(V, 0.1),
                    np.full(V, 5.0)])
    head = np.tile([[1000.0, 0.0]], (L, 1))
    return p0, v0, par, off, head


def _t(a):
    return torch.tensor(np.asarray(a), dtype=torch.float64)


@pytest.mark.parametrize("case", ["ragged", "multi_slot", "clips"])
def test_restatement_matches_oracle(case):
    """Forward <= 1e-12 and autograd gradients wrt (p0, v0, head) <= 1e-10 of the largest entry, collision-free."""
    from oracle import oracle as O
    rng = np.random.default_rng({"ragged": 1, "multi_slot": 2, "clips": 3}[case])
    if case == "ragged":
        (p0, v0, par, off, head), T = _lanes([1, 0, 33, 7, 0, 32, 65, 2], rng), 30
    elif case == "multi_slot":
        (p0, v0, par, off, head), T = _lanes([130, 5, 256], rng), 12
    else:
        (p0, v0, par, off, head), T = _clipped_lanes(rng), 8
    V = p0.shape[0]
    wp, wv = rng.normal(size=V), rng.normal(size=V)
    tp, tv, th = _t(p0).requires_grad_(), _t(v0).requires_grad_(), _t(head).requires_grad_()
    clips = []
    pT, vT, _, _ = rollout(tp, tv, _t(par), off, th, DT, T, clips)
    ((pT * _t(wp)).sum() + (vT * _t(wv)).sum()).backward()
    o = O.idm_rollout(p0, v0, par, off, head, DT, T, g_pT=wp, g_vT=wv)
    assert o["ncol"] == 0 and not any(c[2].any() for c in clips)
    if case == "clips":
        assert sum(int(c[0].sum()) for c in clips) > 0 and sum(int(c[1].sum()) for c in clips) > 0
    assert relerr(pT.detach(), o["pT"]) < 1e-12 and relerr(vT.detach(), o["vT"]) < 1e-12
    assert relerr(tp.grad, o["g_p0"]) < 1e-10 and relerr(tv.grad, o["g_v0"]) < 1e-10
    assert relerr(th.grad, o["g_head"]) < 1e-10


def test_restatement_parameter_gradient_vs_finite_differences():
    """<g_params, d> against (J(par + h d) - J(par - h d)) / 2h of the oracle's forward, for random directions d scaled
    entrywise by par (h = 1e-6), on a clip- and collision-free rollout: <= 1e-5."""
    from oracle import oracle as O
    rng = np.random.default_rng(11)
    p0, v0, par, off, head = _lanes([1, 9, 33, 4], rng, spacing=20.0, v_lo=9.0, v_hi=21.0)
    T, V = 40, p0.shape[0]
    wp, wv = rng.normal(size=V), rng.normal(size=V)
    tpar = _t(par).requires_grad_()
    clips = []
    pT, vT, _, _ = rollout(_t(p0), _t(v0), tpar, off, _t(head), DT, T, clips)
    ((pT * _t(wp)).sum() + (vT * _t(wv)).sum()).backward()
    assert not any(bool(c[0].any() or c[1].any() or c[2].any()) for c in clips)
    g = tpar.grad.numpy()
    def J(q):
        o = O.idm_rollout(p0, v0, q, off, head, DT, T)
        return float((o["pT"] * wp).sum() + (o["vT"] * wv).sum())
    h = 1e-6
    for k in range(4):
        d = rng.normal(size=par.shape) * par
        if k < 3:
            d[2 * k:2 * k + 2] *= 10.0          # weight two parameter rows per direction
        fd = (J(par + h * d) - J(par - h * d)) / (2 * h)
        an = float((g * d).sum())
        assert abs(fd - an) <= 1e-5 * max(abs(an), 1e-12), (k, fd, an)


def test_params_entry_points_reject_null_g_params():
    """dhts_idm_{step,rollout}_bwd_params_* return DHTS_ERR_INVALID for a NULL g_params before touching the device."""
    import dhts_b200
    lib = ctypes.CDLL(dhts_b200.build())
    x = ctypes.c_void_p(16)                      # never dereferenced: the argument check comes first
    for suf, real in (("f64", ctypes.c_double), ("f32", ctypes.c_float)):
        rc = getattr(lib, "dhts_idm_step_bwd_params_" + suf)(x, x, x, x, x, x, real(0.01), 4, 1, x, x, x, x, x,
                                                              ctypes.c_void_p(0), x, ctypes.c_void_p(0))
        assert rc == dhts_b200._lib.ERR_INVALID
        rc = getattr(lib, "dhts_idm_rollout_bwd_params_" + suf)(x, x, x, x, ctypes.c_void_p(0), real(0.01), 4, 1, 4, 3,
                                                                 1, x, x, ctypes.c_void_p(0), x, x, x,
                                                                 ctypes.c_void_p(0), ctypes.c_void_p(0), x,
                                                                 ctypes.c_void_p(0))
        assert rc == dhts_b200._lib.ERR_INVALID
