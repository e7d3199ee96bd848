"""TEST INFRASTRUCTURE ONLY -- one IDM step of CSR lanes restated in plain torch, differentiated by torch.autograd.

It is the independent check of the hand-derived parameter adjoint (csrc/dhts_idm.cuh: idm_par_vjp): the same
arithmetic as idm_eval -- the two clips, the collision reset and the 1e-5 floor of the gap -- written without any
derivative, so that autograd supplies every gradient, those with respect to params [6, V] included.  It is pinned to
the live-reference convention by tests/test_idm_params_host.py (forward and state gradients against the oracle).
"""
from __future__ import annotations

import numpy as np
import torch


def lane_index(off):
    """(lane, is_head, lead) [V] of the CSR offsets `off` [L+1]; the head of a lane is its own `lead` (unused)."""
    off = np.asarray(off, dtype=np.int64)
    V = int(off[-1])
    n = np.diff(off)
    lane = np.repeat(np.arange(len(n)), n)
    is_head = np.zeros(V, dtype=bool)
    is_head[off[1:][n > 0] - 1] = True
    lead = np.arange(V) + 1
    lead[is_head] = np.arange(V)[is_head]
    return torch.as_tensor(lane), torch.as_tensor(is_head), torch.as_tensor(lead)


def step(p, v, par, idx, head, dt, clips=None):
    """(p, v) [V], par [6, V], head [L, 2] -> (np, nv) [V].  `clips`, a list, receives (acc clipped, s* clipped,
    collision) masks of the step."""
    lane, is_head, lead = idx
    a_max, a_pref, v_t, s0, tp, ln = par
    gap = torch.abs(p[lead] - p) - (ln[lead] + ln) * 0.5
    dp = torch.where(is_head, head[lane, 0], gap)
    dv = torch.where(is_head, head[lane, 1], v - v[lead])
    col = dp < 0
    dp = torch.where(col, torch.zeros_like(dp), dp)
    dv = torch.where(col, torch.zeros_like(dv), dv)
    dp = torch.clamp(dp, min=1e-5)
    s = s0 + v * tp + v * dv / (2.0 * torch.sqrt(a_max * a_pref))
    clip_s = s < 0
    s = torch.clamp(s, min=0.0)
    acc = a_max * (1.0 - (v / v_t) ** 4 - (s / dp) ** 2)
    lim = -v / dt
    clip_acc = acc < lim
    acc = torch.where(clip_acc, lim, acc)
    if clips is not None:
        clips.append((clip_acc.detach(), clip_s.detach(), col.detach()))
    return p + dt * v, v + dt * acc


def rollout(p0, v0, par, off, head, dt, T, clips=None):
    """T steps; head [L, 2] or, one pair per step, [T, L, 2].  Returns (pT, vT, p_hist, v_hist), the histories [T, V]
    holding the state BEFORE every step."""
    idx = lane_index(off)
    p, v = p0, v0
    ph, vh = [], []
    for t in range(int(T)):
        ph.append(p); vh.append(v)
        p, v = step(p, v, par, idx, head[t] if head.dim() == 3 else head, dt, clips)
    V = p0.shape[0]
    stack = lambda h: torch.stack(h) if h else p0.new_zeros((0, V))
    return p, v, stack(ph), stack(vh)
