// IDM device math shared by the lane kernels (idm_kernels.cu) and the hybrid network rollout (net_hybrid.cu).
//
// Behaviour restated from the reference (file:line relative to its checkout):
//   model/micro/_idm.py:5-51            acceleration with the two clips
//   road/lane/_micro_lane.py:149-168    collision reset and the 1e-5 floor of the gap
//   model/micro/didm.py:12-102          ego / leader 2x2 Jacobians
#pragma once
#include "dhts_arz.cuh"

namespace dhts {

template <typename T> struct IdmPar { T a_max, v_t_inv, s0, tp, len, sab2_inv; };
//  v_t_inv = 1/target_speed, sab2_inv = 1/(2 sqrt(a_max a_pref)): per-vehicle constants of _idm.py:31-40

template <typename T> __device__ __forceinline__ IdmPar<T> load_par(const T* __restrict__ params, size_t V, size_t i) {
    IdmPar<T> k;
    T a_max = params[i], a_pref = params[V + i], v_t = params[2 * V + i];
    k.a_max = a_max; k.v_t_inv = T(1) / v_t; k.s0 = params[3 * V + i]; k.tp = params[4 * V + i];
    k.len = params[5 * V + i];
    k.sab2_inv = T(1) / (T(2) * t_sqrt(a_max * a_pref));
    return k;
}

template <typename T> struct IdmEval { T acc, s; bool clip_acc, clip_s, col; };

// _micro_lane.py:149-168 (collision reset, 1e-5 floor) + _idm.py:31-51
template <typename T>
__device__ __forceinline__ IdmEval<T> idm_eval(T v, const IdmPar<T>& k, T dp_raw, T dv_raw, T inv_dt) {
    IdmEval<T> e;
    e.col = dp_raw < T(0);
    T dp = e.col ? T(0) : dp_raw, dv = e.col ? T(0) : dv_raw;
    dp = t_max(dp, T(1e-5));
    T s = k.s0 + v * k.tp + (v * dv) * k.sab2_inv;
    e.clip_s = s < T(0);
    s = t_max(s, T(0));
    T q = v * k.v_t_inv; q = q * q;
    T sr = s * f_rcp(dp);              // dp >= 1e-5: branch-free reciprocal (<= 1 ulp) instead of the IEEE division's slow-path call
    T acc = k.a_max * (T(1) - q * q - sr * sr);
    T lim = -v * inv_dt;
    e.clip_acc = acc < lim;
    e.acc = e.clip_acc ? lim : acc;
    e.s = s;
    return e;
}

// didm.py:12-102 with the RAW deltas (dmicro_lane.py:97).  Returns the second
// rows (E10, E11) and (L10, L11); first rows are [1, dt] and [0, 0].
template <typename T>
__device__ __forceinline__ void idm_jac(T v, const IdmPar<T>& k, T dp_raw, T dv_raw, const IdmEval<T>& e, T dt,
                                        T& E10, T& E11, T& L10, T& L11) {
    // Branch-free: the two clips differ per vehicle, so branches here diverge in every warp.  With s* clipped e.s is 0, hence
    // s / dp^2 = 0 and the general expressions reduce to the clipped ones of didm.py:38-56,84-102 (E11 = 1 + dt a_max t1, L11 = 0);
    // the acceleration clip zeroes both second rows.
    T idp = f_rcp(dp_raw);             // raw gap (dmicro_lane.py:97); a zero gap gives a non-finite Jacobian (the reference raises), flagged as NaN gradient
    T sd2 = e.s * idp * idp;          // s / dp^2
    T sd3 = e.s * sd2 * idp;          // s^2 / dp^3
    T l10 = dt * (T(2) * k.a_max * sd3);
    T vt2 = k.v_t_inv * k.v_t_inv;
    T t1 = T(-4) * (v * v * v) * (vt2 * vt2);
    T e11 = T(1) + dt * k.a_max * (t1 - T(2) * sd2 * (k.tp + (v + dv_raw) * k.sab2_inv));
    T l11 = dt * k.a_max * (T(-2) * sd2 * (-v * k.sab2_inv));
    L10 = e.clip_acc ? T(0) : l10;
    E10 = e.clip_acc ? T(0) : -l10;
    E11 = e.clip_acc ? T(0) : e11;
    L11 = e.clip_acc ? T(0) : l11;
}

// Adjoint of the parameters (a_max, a_pref, v_target, s0, time_pref, length) of one vehicle, in factored form.  With
// A = a_max, sd2 = s/dp^2, q = (v/v_t)^2 and acc the unclipped acceleration, nv = v + dt acc has
//   d acc/d a_max  = acc/A + sd2 v dv sab2_inv        d acc/d a_pref = A sd2 v dv sab2_inv / a_pref
//   d acc/d v_t    = 4 A q^2 v_t_inv                  d acc/d s0 = -2 A sd2      d acc/d time_pref = -2 A sd2 v
//   d acc/d length = -A s^2/dp^3 = -(L10 / dt) / 2, for the own length and for the leader's.
// Like idm_jac it uses e.s and the RAW deltas, so at collisions it follows the state Jacobian's convention; the
// acceleration clip zeroes every term, a clipped s* (e.s = 0) every s term.  The per-vehicle constants of the rows are
// left out, so that a rollout adjoint adds one product per step and parameter (idm_par_vjp) and applies them once at
// the end (idm_par_grad).  The length row is not formed here: it is -cpv/2 (cpv = L10 gv, what the vehicle sends to
// its leader) of the vehicle itself -- unless its gap is head_dp, which no length enters -- plus -cpv/2 of its follower.
template <typename T> struct IdmParAdj { T acc, x, q2, sd2, sd2v, len; };

template <typename T>
__device__ __forceinline__ void idm_par_vjp(T v, const IdmPar<T>& k, T dp_raw, T dv_raw, const IdmEval<T>& e, T gv,
                                            IdmParAdj<T>& a) {
    if (e.clip_acc) return;
    T idp = f_rcp(dp_raw);
    T sd2 = e.s * idp * idp;
    T q = (v * v) * (k.v_t_inv * k.v_t_inv);   // not idm_eval's q * q: sharing that product could unfuse its 1 - q*q
    a.acc += gv * e.acc;
    a.x += gv * (sd2 * (v * dv_raw));
    a.q2 += gv * (q * q);
    a.sd2 += gv * sd2;
    a.sd2v += gv * (sd2 * v);
}

// g[6] = d loss / d params of the vehicle from its accumulated IdmParAdj (a_pref: the vehicle's raw parameter)
template <typename T>
__device__ __forceinline__ void idm_par_grad(const IdmParAdj<T>& a, const IdmPar<T>& k, T a_pref, T dt, T* g) {
    const T A = k.a_max, xs = a.x * k.sab2_inv;
    g[0] = dt * (a.acc / A + xs);
    g[1] = dt * (A * xs / a_pref);
    g[2] = dt * (T(4) * A * k.v_t_inv * a.q2);
    g[3] = dt * (T(-2) * A * a.sd2);
    g[4] = dt * (T(-2) * A * a.sd2v);
    g[5] = a.len;
}

}  // namespace dhts
