"""Batched, device-resident API of the simulation step.

Each function states which reference loop it stands for.  Tensors are CUDA
tensors (float64 or float32); everything differentiates through the hand-written
adjoint kernels.  Shapes: B macro lanes x N cells; V vehicles in L micro lanes
(CSR ``lane_off``).
"""
from __future__ import annotations

import torch

from . import _lib
from .ops import arz_ckpt_elems as _arz_ckpt_elems
from .ops import (EPSILON, ArzRolloutFn, ArzStepFn, IdmRolloutFn, IdmStepFn, MacroToMicroFn, MicroToMacroFn,
                  csr_expand)


def u_eq(r: torch.Tensor, umax) -> torch.Tensor:
    """ARZ.compute_u_eq (model/macro/_arz.py:133-138), gamma = 0.5; differentiated by autograd like the reference's 0-dim ops."""
    return umax * (1.0 - torch.sqrt(torch.clamp(r, min=0.0) + EPSILON))


def compute_y(r: torch.Tensor, u: torch.Tensor, umax) -> torch.Tensor:
    """ARZ.compute_y (model/macro/_arz.py:121-124)."""
    return r * (u - u_eq(r, umax))


def _per_lane(x, B, like: torch.Tensor) -> torch.Tensor:
    t = torch.as_tensor(x, dtype=like.dtype, device=like.device)
    return t.expand(B).contiguous() if t.dim() == 0 else t.contiguous()


def arz_step(r_pad, y_pad, u_pad, dx, umax, dt, flags, ueq_pad=None, want_case=False):
    """One Godunov step of B lanes: the batched dMacroForwardLayer.apply (dmacro_lane.py:83)
    followed by set_next_state_vector_y's u (``_macro_lane.py:282-299``).
    Inputs are padded [B, N+2] (ghost, cells, ghost); returns (nr, ny, nu)[B, N] (+ case [B, N+1])."""
    B = r_pad.shape[0]
    dx = _per_lane(dx, B, r_pad); umax = _per_lane(umax, B, r_pad)
    return ArzStepFn.apply(r_pad, y_pad, u_pad.detach(), None if ueq_pad is None else ueq_pad.detach(), dx, umax, dt,
                           flags.t, want_case)


def arz_rollout(r0, u0, ghost_r, ghost_u, dx, umax, dt, steps, ckpt_every=32, flags=None, ckpt_buffer=None,
                return_history=False):
    """`steps` x RoadNetwork.forward over B disconnected dMacroLanes, i.e. the loop of
    example/inverse/_inverse.py:91-99 for example/inverse/macro.py, batched:
    set_state_vector_u(r0, u0) -> steps x (boundary, forward, update_state) -> get_state_vector().
    r0, u0 [B, N]; ghost_r, ghost_u [B, 2] (left, right) static ghost cells, or [steps, B, 2]: one pair per step
    (what a lane inside a network sees, road_network.py:364-387; needs ckpt_every = 1).  Returns (rT, yT, uT) [B, N];
    with return_history=True (ckpt_every = 1) also (r_hist, y_hist) [steps, B, N], the state BEFORE every step, both
    differentiable: a loss may read the lane at every step and the adjoint kernel injects its gradient step by step.
    ckpt_buffer: optional flat tensor the state checkpoints are written into instead of a fresh allocation;
    it must stay untouched until this rollout's backward has run (see arz_rollout_plan)."""
    B, N = r0.shape
    flags = flags or _lib.Flags(r0.device)
    # one geometry for all lanes (Python scalars: what the reference's drivers build) travels as two scalars
    uni = not torch.is_tensor(dx) and not torch.is_tensor(umax)
    dxl = None if uni else _per_lane(dx, B, r0); uml = None if uni else _per_lane(umax, B, r0)
    um = float(umax) if uni else uml[:, None]
    y0 = compute_y(r0, u0, um)                       # set_r_u, _arz.py:82-86 (autograd, true derivative)
    ghost = torch.stack([ghost_r, compute_y(ghost_r, ghost_u, um), ghost_u.detach()], dim=-1)   # from_r_u, :74-80
    try:
        out = ArzRolloutFn.apply(r0, y0, u0.detach(), ghost, float(dx) if uni else dxl, float(umax) if uni else uml, dt, steps,
                                 ckpt_every, flags.t, ckpt_buffer, bool(return_history))
        if return_history:
            return out[0], out[1], out[2], out[3][:, 0], out[3][:, 1]
        return out
    except _lib.UnsupportedShape:
        pass
    # lane too long for the register-resident kernel: chain the tiled per-step kernels (still CUDA)
    if uni:
        dxl = _per_lane(dx, B, r0); uml = _per_lane(umax, B, r0)
    r, y, u = r0, y0, u0.detach()
    hist = []
    for t in range(int(steps)):
        g = ghost[t] if ghost.dim() == 4 else ghost
        hist.append((r, y))
        r_pad = torch.cat([g[:, 0:1, 0], r, g[:, 1:2, 0]], dim=1)
        y_pad = torch.cat([g[:, 0:1, 1], y, g[:, 1:2, 1]], dim=1)
        u_pad = torch.cat([g[:, 0:1, 2], u.detach(), g[:, 1:2, 2]], dim=1)
        r, y, u = ArzStepFn.apply(r_pad, y_pad, u_pad, None, dxl, uml, dt, flags.t, False)
    if return_history:
        return r, y, u, torch.stack([h[0] for h in hist]), torch.stack([h[1] for h in hist])
    return r, y, u


def arz_rollout_state(r0, y0, u0, ghost, dx, umax, dt, steps, ckpt_every, flags):
    """The rollout operator on lane STATE as the lanes hold it: (r0, y0)[B, N] differentiable, u0 the speed stored on
    the cells (value only), ghost [B, 2, 3] = (r, y, u) per side, dx / umax [B].  Returns (rT, yT, uT).  What the
    drop-in network's deferred stepping calls (dropin/deferred.py)."""
    return ArzRolloutFn.apply(r0, y0, u0.detach(), ghost, dx, umax, dt, steps, ckpt_every, flags.t, None, False)


def idm_rollout_state(p0, v0, params, lane_off, head, dt, steps, ckpt_every, flags, max_lane):
    """The IDM rollout operator without the per-step fallback of `idm_rollout` (raises UnsupportedShape instead)."""
    return IdmRolloutFn.apply(p0, v0, head, params, lane_off, max_lane, dt, steps, ckpt_every, flags.t, False)


def arz_ckpt_elems(B, N, steps, ckpt_every, dtype) -> int:
    """Elements a caller-owned ``ckpt_buffer`` must hold for a differentiable rollout of this shape: the stored states
    [ceil(steps / ckpt_every), 2, B, N] plus, where the kernels store them, the interface outcomes of every step (a quarter
    byte per cell-step; ``dhts_arz_rollout_ckpt_elems_*``, include/dhts.h)."""
    return _arz_ckpt_elems(B, N, steps, ckpt_every, dtype)[0]


def arz_rollout_plan(B, N, steps, dtype, device, mem_fraction=0.6, min_lanes=296):
    """How to run a differentiable rollout of B lanes within the device's free memory: returns
    (lanes_per_chunk, ckpt_every).  Storing EVERY state (ckpt_every = 1) removes the segment recompute from
    the adjoint -- the fastest mode, 2 * N * steps scalars per lane (+ 1.6 % for the interface outcomes) -- so lanes are processed in chunks
    that fit `mem_fraction` of the free HBM (180 GB on B200: ~6500 lanes of 1024 cells x 1000 steps in
    fp64).  When not even `min_lanes` (two CTAs per SM) fit, fall back to sparse checkpoints + recompute."""
    esz = torch.empty((), dtype=dtype).element_size()
    free, _ = torch.cuda.mem_get_info(device)
    per_lane = -(-arz_ckpt_elems(min_lanes, N, max(int(steps), 1), 1, dtype) // min_lanes) * esz
    fit = int(free * mem_fraction) // per_lane
    if fit >= min(B, min_lanes):
        nchunk = -(-B // min(B, fit))                      # equal chunks (the last one may be a few lanes short)
        chunk = -(-B // nchunk)
        chunk += (-chunk) % 8
        return min(chunk, B), 1
    K = 32
    per_lane = 2 * N * ((int(steps) + K - 1) // K) * esz
    return max(1, min(B, int(free * mem_fraction) // per_lane)), K


def idm_step(p, v, params, lane_off, head, dt, flags, veh_lane=None, want_flags=False):
    """One IDM step of all lanes: the batched dMicroForwardLayer.apply (dmicro_lane.py:75).
    Returns (np, nv)[V] (+ per-vehicle clip / collision bits).  params [6, V] (a_max, a_pref, v_target, s0, time_pref,
    length) is differentiable; for one parameter set shared by many vehicles pass a [6, 1] leaf ``.expand(6, V)``:
    autograd sums the per-vehicle gradients into it."""
    if veh_lane is None:
        veh_lane = csr_expand(lane_off, p.numel())
    return IdmStepFn.apply(p, v, head, params, lane_off, veh_lane, dt, flags.t, want_flags)


def idm_rollout(p0, v0, params, lane_off, head, dt, steps, ckpt_every=32, flags=None, max_lane=None, return_history=False):
    """`steps` x RoadNetwork.forward over L independent dMicroLanes whose heads follow the ghost leader
    (head_position_delta, head_speed_delta): the loop of example/inverse/_inverse.py:91-99 for
    example/inverse/micro.py, batched.  head [L, 2], or [steps, L, 2] for one pair per step (needs no special
    checkpointing).  Returns (pT, vT) [V]; with return_history=True (ckpt_every = 1) also (p_hist, v_hist) [steps, V],
    the state BEFORE every step, differentiable (a loss may read the lanes at every step).  params [6, V] is
    differentiable (calibration of the driver model against trajectories); a parameter set shared by many vehicles is a
    [6, 1] leaf ``.expand(6, V)`` (or, one set per lane, a [6, L] leaf indexed by each vehicle's lane), and autograd
    sums the per-vehicle gradients into it."""
    flags = flags or _lib.Flags(p0.device)
    if max_lane is None:
        max_lane = int((lane_off[1:] - lane_off[:-1]).max().item()) if lane_off.numel() > 1 else 0
    try:
        out = IdmRolloutFn.apply(p0, v0, head, params, lane_off, max_lane, dt, steps, ckpt_every, flags.t, bool(return_history))
        if return_history:
            return out[0], out[1], out[2][:, 0, :p0.numel()], out[2][:, 1, :p0.numel()]
        return out
    except _lib.UnsupportedShape:
        pass
    veh_lane = csr_expand(lane_off, p0.numel())
    p, v = p0, v0
    hist = []
    for t in range(int(steps)):
        hist.append((p, v))
        p, v = IdmStepFn.apply(p, v, head[t] if head.dim() == 3 else head, params, lane_off, veh_lane, dt, flags.t, False)
    if return_history:
        return p, v, torch.stack([h[0] for h in hist]), torch.stack([h[1] for h in hist])
    return p, v


def macro_to_micro(cap, r_last, u_last, free_space, veh_len, dt):
    """Conversion.macro_to_micro (road/network/conversion.py:15-73) for J junctions.
    Returns (cap_out, spawn[int32], v_new, a_new)."""
    return MacroToMicroFn.apply(cap, r_last, u_last, free_space.detach(), veh_len.detach(), dt)


def micro_to_macro(p_head, v_head, a_head, len_head, lane_len, r, y, u, dx, umax):
    """Conversion.micro_to_macro (road/network/conversion.py:75-171) for J junctions x [J, N] downstream cells.
    Returns (r_out, y_out, u_out, absorbed[int32], ntouched[int32])."""
    return MicroToMacroFn.apply(p_head, v_head, a_head, len_head.detach(), lane_len.detach(), r, y, u, dx.detach(),
                                umax.detach())
