"""torch.autograd.Functions over the C ABI of libdhts_b200.so.

These are the B200 counterparts of the reference's per-lane operators
``dMacroForwardLayer`` (road/lane/dmacro_lane.py:234-310) and
``dMicroForwardLayer`` (road/lane/dmicro_lane.py:228-297), batched over lanes,
plus fused T-step rollouts and the macro<->micro exchange of
road/network/conversion.py.  First-order only, like the reference.

Contract notes kept from the reference:
  * the ARZ operators differentiate wrt (r, y) of cells AND ghost cells
    (dmacro_lane.py:296-303); the stored speed ``u`` is a value-only input;
  * the IDM operators fold the ghost leader of dmicro_lane.py:144-151 and return
    the adjoint of (head_position_delta, head_speed_delta);
  * ``nu`` / ``uT`` = compute_u(r', y') is produced inside the operator here (the
    reference does it right after, with 0-dim tensor ops: set_r_y,
    model/macro/_arz.py:88-92); its adjoint uses the true derivative, as autograd
    does there.
"""
from __future__ import annotations

import ctypes

import torch

from . import _lib
from ._lib import check, creal, ptr, stream_ptr, suffix

EPSILON = 1e-5   # model/macro/_arz.py:2


def _c(t):
    return None if t is None else t.contiguous()


def _fn(name, dtype):
    return getattr(_lib.load(), f"dhts_{name}_{suffix(dtype)}")


class ArzStepFn(torch.autograd.Function):
    """(r_pad, y_pad)[B,N+2] -> (nr, ny, nu)[B,N]; u_pad / ueq_pad are stored-value inputs."""

    @staticmethod
    def forward(ctx, r_pad, y_pad, u_pad, ueq_pad, dx, umax, dt, flags, want_case):
        dev = _lib.require_cuda(r_pad, y_pad, u_pad, ueq_pad, dx, umax, flags)
        r_pad, y_pad, u_pad, ueq_pad, dx, umax = map(_c, (r_pad, y_pad, u_pad, ueq_pad, dx, umax))
        B, P = r_pad.shape
        N = P - 2
        dt_ = float(dt)
        nr = torch.empty((B, N), dtype=r_pad.dtype, device=dev)
        ny = torch.empty_like(nr)
        nu = torch.empty_like(nr)
        case = torch.empty((B, N + 1), dtype=torch.int32, device=dev) if want_case else None
        with torch.cuda.device(dev):
            check(_fn("arz_step_fwd", r_pad.dtype)(ptr(r_pad), ptr(y_pad), ptr(u_pad), ptr(ueq_pad), ptr(dx), ptr(umax),
                                                   creal(r_pad.dtype, dt_), B, N, ptr(nr), ptr(ny), ptr(nu), ptr(case),
                                                   ptr(flags), stream_ptr(dev)), "dhts_arz_step_fwd")
        ctx.save_for_backward(r_pad, y_pad, u_pad, ueq_pad, dx, umax, nr, ny)
        ctx.flags = flags          # written in place by kernels and reset by the host: not a versioned autograd input
        ctx.dt = dt_
        ctx.mark_non_differentiable(*([case] if want_case else []))
        if want_case:
            return nr, ny, nu, case
        return nr, ny, nu

    @staticmethod
    def backward(ctx, g_nr, g_ny, g_nu, *_):
        r_pad, y_pad, u_pad, ueq_pad, dx, umax, nr, ny = ctx.saved_tensors
        flags = ctx.flags
        dev = r_pad.device
        B, P = r_pad.shape
        z = lambda g: torch.zeros_like(nr) if g is None else g.contiguous()
        g_nr, g_ny = z(g_nr), z(g_ny)
        g_nu = _c(g_nu)
        g_r = torch.empty_like(r_pad)
        g_y = torch.empty_like(r_pad)
        with torch.cuda.device(dev):
            check(_fn("arz_step_bwd", r_pad.dtype)(ptr(r_pad), ptr(y_pad), ptr(u_pad), ptr(ueq_pad), ptr(dx), ptr(umax),
                                                   creal(r_pad.dtype, ctx.dt), B, P - 2, ptr(nr), ptr(ny), ptr(g_nr),
                                                   ptr(g_ny), ptr(g_nu), ptr(g_r), ptr(g_y), ptr(flags),
                                                   stream_ptr(dev)), "dhts_arz_step_bwd")
        return g_r, g_y, None, None, None, None, None, None, None


class _ArenaLease:
    """Marks a caller-owned checkpoint arena as holding the states of a rollout whose backward has not run yet.
    The kernels write the arena through raw pointers, so autograd's version counter cannot notice that a second
    rollout overwrote it; this lease can: it lives in the first rollout's ctx, ends when its backward has read the
    arena (or when the graph is dropped), and a rollout that finds a live lease on its arena raises."""
    __slots__ = ("active", "__weakref__")

    def __init__(self):
        self.active = True


def _lease_arena(buf):
    import weakref
    ref = getattr(buf, "_dhts_lease", None)
    old = ref() if ref is not None else None
    if old is not None and old.active:
        raise RuntimeError("ckpt_buffer still holds the checkpoints of a rollout whose backward has not run: run that "
                           "backward (or drop its graph) before reusing the arena, or pass another buffer")
    lease = _ArenaLease()
    buf._dhts_lease = weakref.ref(lease)
    return lease


def arz_ckpt_elems(B, N, steps, ckpt_every, dtype):
    """(elements, ckpt_mode) of the checkpoint buffer of a differentiable rollout of this shape (include/dhts.h:
    dhts_arz_rollout_ckpt_elems_*): the ceil(steps / ckpt_every) stored states [S, 2, B, N] and, in mode 1, the interface
    outcomes of every step behind them."""
    mode = ctypes.c_int(0)
    n = int(_fn("arz_rollout_ckpt_elems", dtype)(int(B), int(N), int(steps), int(ckpt_every), ctypes.byref(mode)))
    if n < 0:
        raise ValueError("dhts_arz_rollout_ckpt_elems: invalid shape")
    return n, int(mode.value)


class ArzRolloutFn(torch.autograd.Function):
    """(r0, y0)[B,N], ghost -> (rT, yT, uT)[B,N] (+ hist) after `steps` fused steps.

    ghost [B,2,3]: static ghost cells (r, y, u); ghost [steps,B,2,3]: one pair of ghost cells PER STEP (a lane inside
    a network, road_network.py:364-387).  want_hist (needs ckpt_every = 1): a fourth output hist [steps,2,B,N], the
    (r, y) state BEFORE every step (hist[0] = the input) -- the kernels' checkpoint tensor itself -- so that a loss
    may read the lane at every step; its gradient is injected step by step in the adjoint kernel.
    dx, umax: tensors [B], or two Python floats when every lane has the same geometry (include/dhts.h: dx = umax = NULL
    with dx_all / umax_all -- the kernels then read the lane constants from their parameter block)."""

    @staticmethod
    def forward(ctx, r0, y0, u0, ghost, dx, umax, dt, steps, ckpt_every, flags, ckpt_buffer=None, want_hist=False):
        uni = not torch.is_tensor(dx) and not torch.is_tensor(umax)
        if uni:
            dev = _lib.require_cuda(r0, y0, u0, ghost, flags)
            r0, y0, u0, ghost = map(_c, (r0, y0, u0, ghost))
            dx_all, umax_all, dx, umax = float(dx), float(umax), None, None
        else:
            dev = _lib.require_cuda(r0, y0, u0, ghost, dx, umax, flags)
            r0, y0, u0, ghost, dx, umax = map(_c, (r0, y0, u0, ghost, dx, umax))
            dx_all = umax_all = 0.0
        B, N = r0.shape
        dt_, steps, K = float(dt), int(steps), max(1, int(ckpt_every))
        tv = ghost.dim() == 4
        if tv:
            assert ghost.shape == (steps, B, 2, 3), "per-step ghosts are [steps, B, 2, 3]"
        if (tv or want_hist) and K != 1:
            raise ValueError("per-step ghosts and the state history need ckpt_every = 1 (every state stored)")
        need_grad = any(ctx.needs_input_grad[i] for i in (0, 1, 3))
        S = (steps + K - 1) // K
        ckpt = None
        # what the checkpoint buffer holds: the S states, and behind them the interface outcomes of every step where the
        # kernels take them (ckpt_mode 1, include/dhts.h)
        xmode, n = 0, S * 2 * B * N
        if need_grad and not tv and not want_hist:
            n, xmode = arz_ckpt_elems(B, N, steps, K, r0.dtype)
        if need_grad or want_hist:
            if ckpt_buffer is not None:      # caller-owned arena, reused across sequential rollouts (lane chunks)
                if ckpt_buffer.dtype != r0.dtype or ckpt_buffer.device != dev or ckpt_buffer.numel() < n:
                    raise ValueError("ckpt_buffer must be a %s tensor on %s with >= %d elements" % (r0.dtype, dev, n))
                ckpt = ckpt_buffer.view(-1)[:n]
                ctx.lease = _lease_arena(ckpt_buffer)
            else:
                ckpt = torch.empty((n,), dtype=r0.dtype, device=dev)
        rT = torch.empty_like(r0); yT = torch.empty_like(r0); uT = torch.empty_like(r0)
        with torch.cuda.device(dev):
            check(_fn("arz_rollout_fwd", r0.dtype)(ptr(r0), ptr(y0), ptr(u0), ptr(None if tv else ghost),
                                                   ptr(ghost if tv else None), ptr(dx), ptr(umax),
                                                   creal(r0.dtype, dx_all), creal(r0.dtype, umax_all),
                                                   creal(r0.dtype, dt_), B, N, steps, K, xmode, ptr(ckpt), ptr(rT), ptr(yT),
                                                   ptr(uT), ptr(flags), stream_ptr(dev)), "dhts_arz_rollout_fwd")
        if need_grad:
            if uni:
                ctx.save_for_backward(ckpt, u0, ghost, rT, yT)
            else:
                ctx.save_for_backward(ckpt, u0, ghost, rT, yT, dx, umax)
        ctx.flags = flags
        ctx.cfg = (dt_, steps, K, B, N, tv, bool(want_hist), xmode, dx_all, umax_all)
        if want_hist:
            return rT, yT, uT, ckpt.view(S, 2, B, N)
        return rT, yT, uT

    @staticmethod
    def backward(ctx, g_rT, g_yT, g_uT, g_hist=None):
        ckpt, u0, ghost, rT, yT = ctx.saved_tensors[:5]
        dx, umax = ctx.saved_tensors[5:] if len(ctx.saved_tensors) > 5 else (None, None)
        flags = ctx.flags
        dt_, steps, K, B, N, tv, want_hist, xmode, dx_all, umax_all = ctx.cfg
        dev, dtype = ghost.device, ghost.dtype
        g_rT, g_yT, g_uT, g_hist = map(_c, (g_rT, g_yT, g_uT, g_hist))
        g_r0 = torch.empty((B, N), dtype=dtype, device=dev)
        g_y0 = torch.empty_like(g_r0)
        g_gh = torch.empty((steps, B, 2, 2) if tv else (B, 2, 2), dtype=dtype, device=dev)
        with torch.cuda.device(dev):
            n = _fn("arz_rollout_scratch_elems", dtype)(B, N, K)
            if n < 0:
                raise _lib.UnsupportedShape("dhts_arz_rollout_bwd: lane does not fit the fused kernel")
            scratch = torch.empty((max(int(n), 1),), dtype=dtype, device=dev)
            check(_fn("arz_rollout_bwd", dtype)(ptr(ckpt), ptr(u0), ptr(None if tv else ghost), ptr(ghost if tv else None),
                                                ptr(dx), ptr(umax), creal(dtype, dx_all), creal(dtype, umax_all),
                                                creal(dtype, dt_), B, N, steps, K, xmode, ptr(rT), ptr(yT),
                                                ptr(g_rT), ptr(g_yT), ptr(g_uT), ptr(g_hist), ptr(scratch),
                                                ctypes.c_longlong(int(n)), ptr(g_r0), ptr(g_y0),
                                                ptr(None if tv else g_gh), ptr(g_gh if tv else None), ptr(flags),
                                                stream_ptr(dev)), "dhts_arz_rollout_bwd")
        lease = getattr(ctx, "lease", None)
        if lease is not None:
            lease.active = False          # the arena has been read: the next rollout may overwrite it
        g_ghost = torch.zeros(ghost.shape, dtype=dtype, device=dev)
        g_ghost[..., :2] = g_gh           # ghost u is a value-only input
        return g_r0, g_y0, None, g_ghost, None, None, None, None, None, None, None, None


def csr_expand(lane_off: torch.Tensor, V: int) -> torch.Tensor:
    dev = _lib.require_cuda(lane_off)
    lane_off = lane_off.contiguous()
    veh_lane = torch.empty((max(V, 1),), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        check(_lib.load().dhts_csr_expand(ptr(lane_off), lane_off.numel() - 1, ptr(veh_lane), stream_ptr(dev)),
              "dhts_csr_expand")
    return veh_lane


class IdmStepFn(torch.autograd.Function):
    """(p, v)[V], head[L,2] -> (np, nv)[V]; params [6,V] (differentiable), CSR lane_off[L+1]."""

    @staticmethod
    def forward(ctx, p, v, head, params, lane_off, veh_lane, dt, flags, want_flags):
        dev = _lib.require_cuda(p, v, head, params, lane_off, veh_lane, flags)
        p, v, head, params, lane_off, veh_lane = map(_c, (p, v, head, params, lane_off, veh_lane))
        V, L = p.numel(), lane_off.numel() - 1
        dt_ = float(dt)
        np_ = torch.empty_like(p); nv_ = torch.empty_like(p)
        vf = torch.zeros((V,), dtype=torch.int32, device=dev) if want_flags else None
        with torch.cuda.device(dev):
            check(_fn("idm_step_fwd", p.dtype)(ptr(p), ptr(v), ptr(params), ptr(lane_off), ptr(veh_lane), ptr(head),
                                               creal(p.dtype, dt_), V, L, ptr(np_), ptr(nv_), ptr(vf), ptr(flags),
                                               stream_ptr(dev)), "dhts_idm_step_fwd")
        ctx.save_for_backward(p, v, head, params, lane_off, veh_lane)
        ctx.flags = flags
        ctx.dt = dt_
        if want_flags:
            ctx.mark_non_differentiable(vf)
            return np_, nv_, vf
        return np_, nv_

    @staticmethod
    def backward(ctx, g_np, g_nv, *_):
        p, v, head, params, lane_off, veh_lane = ctx.saved_tensors
        flags = ctx.flags
        dev = p.device
        V, L = p.numel(), lane_off.numel() - 1
        z = lambda g: torch.zeros_like(p) if g is None else g.contiguous()
        g_np, g_nv = z(g_np), z(g_nv)
        g_p = torch.empty_like(p); g_v = torch.empty_like(p)
        g_head = torch.zeros_like(head)
        args = (ptr(p), ptr(v), ptr(params), ptr(lane_off), ptr(veh_lane), ptr(head), creal(p.dtype, ctx.dt), V, L,
                ptr(g_np), ptr(g_nv), ptr(g_p), ptr(g_v), ptr(g_head))
        g_params = None
        with torch.cuda.device(dev):
            if ctx.needs_input_grad[3]:
                g_params = torch.empty_like(params)
                check(_fn("idm_step_bwd_params", p.dtype)(*args, ptr(g_params), ptr(flags), stream_ptr(dev)),
                      "dhts_idm_step_bwd_params")
            else:
                check(_fn("idm_step_bwd", p.dtype)(*args, ptr(flags), stream_ptr(dev)), "dhts_idm_step_bwd")
        return g_p, g_v, g_head, g_params, None, None, None, None, None


class IdmRolloutFn(torch.autograd.Function):
    """(p0, v0)[V], head -> (pT, vT)[V] (+ hist) after `steps` fused steps (one warp per lane).

    head [L,2]: one (head_position_delta, head_speed_delta) pair per lane for the whole rollout; head [steps,L,2]: one
    pair PER STEP (inside a network setup_micro_boundary rewrites them every step, road_network.py:429-580).
    want_hist (ckpt_every = 1): a third output hist [steps,2,V], (p, v) BEFORE every step, differentiable.
    params [6,V] is differentiable too: its adjoint accumulates over every step in the adjoint kernel."""

    @staticmethod
    def forward(ctx, p0, v0, head, params, lane_off, max_lane, dt, steps, ckpt_every, flags, want_hist=False):
        dev = _lib.require_cuda(p0, v0, head, params, lane_off, flags)
        p0, v0, head, params, lane_off = map(_c, (p0, v0, head, params, lane_off))
        V, L = p0.numel(), lane_off.numel() - 1
        lib = _lib.load()
        dt_, steps = float(dt), int(steps)
        K = max(1, min(int(ckpt_every), lib.dhts_idm_rollout_max_ckpt_every()))
        tv = head.dim() == 3
        if tv:
            assert head.shape == (steps, L, 2), "per-step head deltas are [steps, L, 2]"
        if want_hist and K != 1:
            raise ValueError("the state history needs ckpt_every = 1 (every state stored)")
        need_grad = any(ctx.needs_input_grad[i] for i in (0, 1, 2, 3))
        S = (steps + K - 1) // K
        ckpt = torch.empty((S, 2, max(V, 1)), dtype=p0.dtype, device=dev) if (need_grad or want_hist) else None
        pT = torch.empty_like(p0); vT = torch.empty_like(p0)
        with torch.cuda.device(dev):
            check(_fn("idm_rollout_fwd", p0.dtype)(ptr(p0), ptr(v0), ptr(params), ptr(lane_off), ptr(None if tv else head),
                                                   ptr(head if tv else None), creal(p0.dtype, dt_), V, L, int(max_lane),
                                                   steps, K, ptr(ckpt), ptr(pT), ptr(vT), ptr(flags), stream_ptr(dev)),
                  "dhts_idm_rollout_fwd")
        if need_grad:
            ctx.save_for_backward(ckpt, head, params, lane_off)
        ctx.flags = flags
        ctx.cfg = (dt_, steps, K, V, L, int(max_lane), tv)
        if want_hist:
            return pT, vT, ckpt
        return pT, vT

    @staticmethod
    def backward(ctx, g_pT, g_vT, g_hist=None):
        ckpt, head, params, lane_off = ctx.saved_tensors
        flags = ctx.flags
        dt_, steps, K, V, L, max_lane, tv = ctx.cfg
        dev, dtype = head.device, head.dtype
        z = lambda g: torch.zeros((V,), dtype=dtype, device=dev) if g is None else g.contiguous()
        g_pT, g_vT = z(g_pT), z(g_vT)
        g_hist = _c(g_hist)
        g_p0 = torch.empty((V,), dtype=dtype, device=dev); g_v0 = torch.empty_like(g_p0)
        g_head = torch.zeros_like(head)
        args = (ptr(ckpt), ptr(params), ptr(lane_off), ptr(None if tv else head), ptr(head if tv else None),
                creal(dtype, dt_), V, L, max_lane, steps, K, ptr(g_pT), ptr(g_vT), ptr(g_hist), ptr(g_p0), ptr(g_v0),
                ptr(None if tv else g_head), ptr(g_head if tv else None))
        g_params = None
        with torch.cuda.device(dev):
            if ctx.needs_input_grad[3]:
                g_params = torch.empty_like(params)
                check(_fn("idm_rollout_bwd_params", dtype)(*args, ptr(g_params), ptr(flags), stream_ptr(dev)),
                      "dhts_idm_rollout_bwd_params")
            else:
                check(_fn("idm_rollout_bwd", dtype)(*args, ptr(flags), stream_ptr(dev)), "dhts_idm_rollout_bwd")
        return g_p0, g_v0, g_head, g_params, None, None, None, None, None, None, None


class MacroToMicroFn(torch.autograd.Function):
    """Flux capacitor + spawn test of Conversion.macro_to_micro (conversion.py:15-73), per junction [J]."""

    @staticmethod
    def forward(ctx, cap, r_last, u_last, free_space, veh_len, dt):
        dev = _lib.require_cuda(cap, r_last, u_last, free_space, veh_len)
        cap, r_last, u_last, free_space, veh_len = map(_c, (cap, r_last, u_last, free_space, veh_len))
        J = cap.numel()
        dt_ = float(dt)
        cap_out = torch.empty_like(cap); v_new = torch.empty_like(cap); a_new = torch.empty_like(cap)
        spawn = torch.empty((J,), dtype=torch.int32, device=dev)
        with torch.cuda.device(dev):
            check(_fn("m2c_fwd", cap.dtype)(ptr(cap), ptr(r_last), ptr(u_last), ptr(free_space), ptr(veh_len),
                                            creal(cap.dtype, dt_), J, ptr(cap_out), ptr(spawn), ptr(v_new), ptr(a_new),
                                            stream_ptr(dev)), "dhts_m2c_fwd")
        ctx.save_for_backward(r_last, u_last, spawn)
        ctx.dt = dt_
        ctx.mark_non_differentiable(spawn)
        return cap_out, spawn, v_new, a_new

    @staticmethod
    def backward(ctx, g_cap_out, _g_spawn, g_v_new, g_a_new):
        r_last, u_last, spawn = ctx.saved_tensors
        dev = r_last.device
        z = lambda g: torch.zeros_like(r_last) if g is None else g.contiguous()
        g_cap_out, g_v_new, g_a_new = z(g_cap_out), z(g_v_new), z(g_a_new)
        g_cap = torch.empty_like(r_last); g_r = torch.empty_like(r_last); g_u = torch.empty_like(r_last)
        with torch.cuda.device(dev):
            check(_fn("m2c_bwd", r_last.dtype)(ptr(r_last), ptr(u_last), ptr(spawn), creal(r_last.dtype, ctx.dt),
                                               r_last.numel(), ptr(g_cap_out), ptr(g_v_new), ptr(g_a_new), ptr(g_cap),
                                               ptr(g_r), ptr(g_u), stream_ptr(dev)), "dhts_m2c_bwd")
        return g_cap, g_r, g_u, None, None, None


class MicroToMacroFn(torch.autograd.Function):
    """Head-vehicle absorption of Conversion.micro_to_macro (conversion.py:75-171), per junction [J] x cells [J,N]."""

    @staticmethod
    def forward(ctx, p_head, v_head, a_head, len_head, lane_len, r, y, u, dx, umax):
        dev = _lib.require_cuda(p_head, v_head, a_head, len_head, lane_len, r, y, u, dx, umax)
        p_head, v_head, a_head, len_head, lane_len, r, y, u, dx, umax = map(
            _c, (p_head, v_head, a_head, len_head, lane_len, r, y, u, dx, umax))
        J, N = r.shape
        r_out = torch.empty_like(r); y_out = torch.empty_like(r); u_out = torch.empty_like(r)
        absorbed = torch.empty((J,), dtype=torch.int32, device=dev)
        ntouched = torch.empty((J,), dtype=torch.int32, device=dev)
        with torch.cuda.device(dev):
            check(_fn("c2m_fwd", r.dtype)(ptr(p_head), ptr(v_head), ptr(a_head), ptr(len_head), ptr(lane_len), ptr(r),
                                          ptr(y), ptr(u), ptr(dx), ptr(umax), J, N, ptr(r_out), ptr(y_out), ptr(u_out),
                                          ptr(absorbed), ptr(ntouched), stream_ptr(dev)), "dhts_c2m_fwd")
        ctx.save_for_backward(p_head, v_head, a_head, len_head, lane_len, r_out, dx, umax, ntouched)
        ctx.mark_non_differentiable(absorbed, ntouched)
        return r_out, y_out, u_out, absorbed, ntouched

    @staticmethod
    def backward(ctx, g_r_out, g_y_out, g_u_out, *_):
        p_head, v_head, a_head, len_head, lane_len, r_out, dx, umax, ntouched = ctx.saved_tensors
        dev = r_out.device
        J, N = r_out.shape
        z = lambda g: torch.zeros_like(r_out) if g is None else g.contiguous()
        g_r_out, g_y_out, g_u_out = z(g_r_out), z(g_y_out), z(g_u_out)
        g_p = torch.empty_like(p_head); g_v = torch.empty_like(p_head); g_a = torch.empty_like(p_head)
        g_r = torch.empty_like(r_out); g_y = torch.empty_like(r_out); g_u = torch.empty_like(r_out)
        with torch.cuda.device(dev):
            check(_fn("c2m_bwd", r_out.dtype)(ptr(p_head), ptr(v_head), ptr(a_head), ptr(len_head), ptr(lane_len),
                                              ptr(r_out), ptr(dx), ptr(umax), ptr(ntouched), J, N, ptr(g_r_out),
                                              ptr(g_y_out), ptr(g_u_out), ptr(g_p), ptr(g_v), ptr(g_a), ptr(g_r),
                                              ptr(g_y), ptr(g_u), stream_ptr(dev)), "dhts_c2m_bwd")
        return g_p, g_v, g_a, None, None, g_r, g_y, g_u, None, None
