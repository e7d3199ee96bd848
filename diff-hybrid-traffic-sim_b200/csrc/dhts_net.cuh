// Pieces shared by the connected-network rollouts (net_kernels.cu: macro lanes only; net_hybrid.cu: macro and micro
// lanes with the conversions between them): the per-call argument block, the ghost-source resolution of
// RoadNetwork.get_macro_boundary (road/network/road_network.py:299-362) and the ITSCP signal blend
// (example/control/itscp/_simulator.py:56-142).
#pragma once
#include <cstdint>
#include "dhts_arz.cuh"
#include "dhts_api.h"

namespace dhts {

constexpr int FLAG_ROUTE = 8;      // a lane with several neighbours has none selected by the step's MacroRoute (reference: KeyError)

template <typename T> struct NetArgs {
    // topology, shared by all replicas
    int L, NC, n_own, T_steps, R, mode, soft;
    const int* cell_off;          // [L+1]
    const T* dx;                  // [L]
    const int* nadj;              // [2][L]   number of adjacent lanes per side
    const int* one_adj;           // [2][L]   the adjacent lane when there is exactly one, else -1
    const int* adj_off;           // [2][L+1] CSR of the adjacency lists (side 0: predecessors, 1: successors)
    const int* adj;               // [2][E]
    const int* own_slot;          // [2][L]   slot of the carried own-ghost record, or -1
    const int* route;             // [Rr][T][2][L] MacroRoute per step: (prev lane, next lane) or -1
    long long route_stride;       // 0 when the schedule is shared by all replicas
    T umax, dt, veh_len, static_speed;
    const T* sig;                 // [R][T][L]  lane signals (ITSCP mode)
    const T* incoming;            // [R][T][L]  inflow density of lanes without predecessor (ITSCP mode)
    const T* qk;                  // [T] sigmoid constant of the queue reward, or null (no fused reward)
    const int* kind;              // [L] 0 macro, 1 micro, or null (all macro)
};

template <typename T> __device__ __forceinline__ T sigm(T x) { return f_rcp(T(1) + exp(-x)); }      // |x| <= 16: 1 + e^-x in [1, 9e6]


// u_eq'(r) as autograd differentiates ARZ.compute_u_eq on a tensor (_arz.py:133-138: max(r, 0.) keeps r when r >= 0)
template <typename T> __device__ __forceinline__ T u_eq_true_prime(T r, T umax) {
    return (r >= T(0)) ? T(-0.5) * umax * f_rsqrt(r + DHTS_EPS) : T(0);
}

template <typename T> struct Side {
    int src;        // lane whose edge cell is the green source, -1: own record, -2: incoming (ITSCP left, no predecessor)
    int sig_lane;   // lane whose signal blends this side (left: the route's predecessor; right: the lane itself), -1 none
    T s;            // blend weight actually applied
    T gr_, gu_;     // green (r, u)
    T fr, fu;       // final (r, u)
};

// Resolve the ghost source and the blend of one side of lane l at step t.  `cur_r/cur_u` are the network state.
template <typename T>
__device__ __forceinline__ Side<T> resolve_side(const NetArgs<T>& a, int l, int side, const int* __restrict__ rt,
                                                const T* cur_r, const T* cur_u, const T* own, const T* sig_t,
                                                const T* inc_t, bool& bad_route) {
    Side<T> o;
    const int cnt = a.nadj[side * a.L + l];
    const int sel = rt ? rt[side * a.L + l] : -1;
    int adjl = -1;
    if (cnt == 1) adjl = a.one_adj[side * a.L + l];
    else if (cnt > 1) { adjl = sel; if (sel < 0) bad_route = true; }
    if (adjl >= 0 && a.kind && a.kind[adjl]) adjl = -1;      // micro neighbour: the lane's own ghost record (:353-362)
    o.src = adjl; o.sig_lane = -1; o.s = T(1);
    if (a.mode == 1 && side == 0 && cnt == 0) {
        o.src = -2;
        o.gr_ = inc_t[l]; o.gu_ = u_eq(o.gr_, a.umax);
    } else if (adjl >= 0) {
        const int c = side == 0 ? a.cell_off[adjl + 1] - 1 : a.cell_off[adjl];
        o.gr_ = cur_r[c]; o.gu_ = cur_u[c];
    } else {
        const int sl = a.own_slot[side * a.L + l];
        o.gr_ = sl >= 0 ? own[2 * sl] : T(0); o.gu_ = sl >= 0 ? own[2 * sl + 1] : a.umax;
        o.src = -1;
    }
    if (a.mode == 1) {
        if (side == 0) {
            if (cnt == 0) o.s = T(1);
            else if (sel < 0) o.s = T(0);
            else { o.s = sig_t[sel]; o.sig_lane = sel; }
            o.fr = o.gr_ * o.s + T(0) * (T(1) - o.s);
            o.fu = o.gu_ * o.s + a.umax * (T(1) - o.s);
        } else {
            const T x = sig_t[l];
            if (a.soft) {
                T z = (x - T(0.5)) * T(32);
                z = z < T(-16) ? T(-16) : (z > T(16) ? T(16) : z);
                o.s = sigm(z);
            } else
                o.s = x > T(0.5) ? T(1) : T(0);
            o.sig_lane = l;
            o.fr = o.s * o.gr_ + (T(1) - o.s) * T(1);
            o.fu = o.s * o.gu_ + (T(1) - o.s) * T(0);
        }
    } else {
        o.fr = o.gr_; o.fu = o.gu_;
    }
    return o;
}

}  // namespace dhts
