// Interface-parallel macro step of the connected-network rollouts (net_kernels.cu, net_hybrid.cu).
//
// A network of many SHORT lanes (ITSCP: 1-4 cells) gives one thread per lane a serial chain of up to 5 interface
// solves per step, and the step's latency is that chain.  Here a step is cut into phases that are each one unit of
// work per thread, with the lean per-cell / per-interface math of the lane rollouts (dhts_arz_lean.cuh):
//
//   forward   G  one thread per (lane, side): ghost source + signal blend (resolve_side) -> final ghost (r, u)
//             I  one thread per INTERFACE: record of the cell on its left (or the left ghost), flux through it
//             C  one thread per CELL: Godunov update from its two fluxes, compute_u
//   adjoint   A  one thread per cell: stored-speed adjoint folded into (r, y);  one per (lane, side): ghosts of step t
//             I  one thread per interface: records of both cells, A^T w and B^T w of the flux-difference adjoint
//             C  one thread per cell: new adjoint from its two interfaces;  one per (lane, side): ghost adjoint ->
//                from_r_u -> blend -> published (d green, d signal)
//             (the gathers stay one thread per lane: net_kernels.cu / net_hybrid.cu)
//
// Reference behaviour restated: road/lane/_macro_lane.py:83-146 (update, CFL assert), model/macro/_arz.py:121-332,
// model/macro/darz.py:12-233, road/lane/dmacro_lane.py:96-132,277-310 -- through dhts_arz_lean.cuh.
#pragma once
#include "dhts_net.cuh"
#include "dhts_arz_lean.cuh"

namespace dhts {

// Static per-kernel tables in shared memory.  Macro lane l owns interfaces if_off[l] .. if_off[l] + N (N + 1 of them:
// interface i sits between cell i - 1 and cell i; 0 and N touch the ghosts); micro lanes own none.
template <typename T> struct NetTabs {
    int NI;
    int* if_off;         // [L + 1]
    int* if_lane;        // [NI]
    int* lane_of_cell;   // [NC]
    T* cc;               // [L] dt / dx
    T* dxv;              // [L] dx
    LaneK<T> base;       // the lane-independent constants (u_max, its reciprocals); cc / dx per lane from the two rows above
    __device__ __forceinline__ LaneK<T> lanek(int l) const {
        LaneK<T> k = base;
        k.cc = cc[l]; k.dx = dxv[l];
        return k;
    }
};

__host__ __device__ inline size_t align8(size_t x) { return (x + 7) / 8 * 8; }
template <typename T> __host__ __device__ inline size_t net_tabs_bytes(int L, int NC, int NI) {
    return align8(sizeof(int) * (size_t)(L + 1)) + align8(sizeof(int) * (size_t)NI) + align8(sizeof(int) * (size_t)NC) +
           sizeof(T) * (size_t)2 * L;
}
template <typename T> __device__ __forceinline__ NetTabs<T> net_tabs_carve(unsigned char*& p, const NetArgs<T>& a, int NI) {
    NetTabs<T> t;
    const int L = a.L, NC = a.NC;
    t.NI = NI;
    t.base = make_lanek<T>(a.umax, T(1), a.dt);      // v4 / vmax / veps (the sufficient CFL tests) are not used by the network kernels
    t.cc = reinterpret_cast<T*>(p); t.dxv = t.cc + L; p += sizeof(T) * (size_t)2 * L;
    t.if_off = reinterpret_cast<int*>(p); p += align8(sizeof(int) * (size_t)(L + 1));
    t.if_lane = reinterpret_cast<int*>(p); p += align8(sizeof(int) * (size_t)NI);
    t.lane_of_cell = reinterpret_cast<int*>(p); p += align8(sizeof(int) * (size_t)NC);
    return t;
}
// Every thread calls it once per kernel; ends with a block barrier.
template <typename T> __device__ __forceinline__ void net_tabs_init(const NetArgs<T>& a, const NetTabs<T>& t) {
    for (int l = threadIdx.x; l <= a.L; l += blockDim.x) {
        int nmac = 0;
        if (a.kind) { for (int j = 0; j < l; j++) nmac += a.kind[j] == 0; } else nmac = l;
        t.if_off[l] = a.cell_off[l] + nmac;
        if (l < a.L) { t.cc[l] = a.dt / a.dx[l]; t.dxv[l] = a.dx[l]; }
    }
    __syncthreads();
    for (int l = threadIdx.x; l < a.L; l += blockDim.x) {
        if (a.kind && a.kind[l]) continue;
        const int c0 = a.cell_off[l], N = a.cell_off[l + 1] - c0, i0 = t.if_off[l];
        for (int i = 0; i <= N; i++) t.if_lane[i0 + i] = l;
        for (int i = 0; i < N; i++) t.lane_of_cell[c0 + i] = l;
    }
    __syncthreads();
}

// ---------------------------------------------------------------------------------------------- forward, phase I
// gh [2][L][2]: final ghost (r, u) per (side, lane).  ce: stored u_eq per cell or null.  flux [NI][2].
// Returns true when the CFL condition (_macro_lane.py:137-146) fails at one of this thread's interfaces.  The exact
// per-interface test is evaluated always: the sufficient per-cell tests of the lane rollouts (|u|, |w| < dx / 4 dt)
// never hold on an ITSCP grid (u_max 60, dx 5, 30 Hz: dx / dt = 150), so they would only add work here.
template <typename T>
__device__ __forceinline__ bool net_fwd_flux(const NetArgs<T>& a, const NetTabs<T>& t, const T* cr, const T* cy, const T* cu,
                                             const T* ce, const T* gh, T* flux) {
    bool bad = false;
    for (int it = threadIdx.x; it < t.NI; it += blockDim.x) {
        const int l = t.if_lane[it];
        const int c0 = a.cell_off[l], N = a.cell_off[l + 1] - c0, i = it - t.if_off[l];
        const LaneK<T> k = t.lanek(l);
        FRec<T> L;
        if (i == 0) {
            const T gr = gh[2 * l], gu = gh[2 * l + 1];
            L = frec_stored<T>(gr, gr * (gu - u_eq(gr, a.umax)), gu, T(0), false, k);        // from_r_u, _arz.py:74-80
        } else {
            const int c = c0 + i - 1;
            L = frec_stored<T>(cr[c], cy[c], cu[c], ce ? ce[c] : T(0), ce != nullptr, k);
        }
        const T Rr = i == N ? gh[2 * (a.L + l)] : cr[c0 + i], Rus = i == N ? gh[2 * (a.L + l) + 1] : cu[c0 + i];
        bad |= cfl_exact_bad(L.r, L.us, L.sq, L.w, Rr, Rus, k, a.dt);
        T fr, fy;
        fflux<T, true>(L, Rr, Rus, k, fr, fy);
        flux[2 * it] = fr; flux[2 * it + 1] = fy;
    }
    return bad;
}

// ---------------------------------------------------------------------------------------------- adjoint, phase I
// G: adjoint (gr, gy) of the state after the step, per cell (the stored-speed adjoint already folded in).
// ab [NI][4]: (A^T w).r, (A^T w).y for the cell on the left, (B^T w).r, (B^T w).y for the cell on the right.
template <typename T>
__device__ __forceinline__ void net_adj_flux(const NetArgs<T>& a, const NetTabs<T>& t, const T* cr, const T* cy, const T* cu,
                                             const T* ce, const T* gh, const T* Gr, const T* Gy, T* ab) {
    for (int it = threadIdx.x; it < t.NI; it += blockDim.x) {
        const int l = t.if_lane[it];
        const int c0 = a.cell_off[l], N = a.cell_off[l + 1] - c0, i = it - t.if_off[l];
        const LaneK<T> k = t.lanek(l);
        ARec<T> L, R;
        T gLr = T(0), gLy = T(0), gRr = T(0), gRy = T(0);
        if (i == 0) {
            const T gr = gh[2 * l], gu = gh[2 * l + 1];
            L = arec_stored<T>(gr, gr * (gu - u_eq(gr, a.umax)), gu, T(0), false, k);
        } else {
            const int c = c0 + i - 1;
            L = arec_stored<T>(cr[c], cy[c], cu[c], ce ? ce[c] : T(0), ce != nullptr, k);
            gLr = Gr[c]; gLy = Gy[c];
        }
        if (i == N) {
            const T gr = gh[2 * (a.L + l)], gu = gh[2 * (a.L + l) + 1];
            R = arec_stored<T>(gr, gr * (gu - u_eq(gr, a.umax)), gu, T(0), false, k);
        } else {
            const int c = c0 + i;
            R = arec_stored<T>(cr[c], cy[c], cu[c], ce ? ce[c] : T(0), ce != nullptr, k);
            gRr = Gr[c]; gRy = Gy[c];
        }
        T par, pay, pbr, pby;
        aflux<T, true>(L, R, gRr - gLr, gRy - gLy, k, par, pay, pbr, pby);
        T* o = ab + 4 * (size_t)it;
        o[0] = par; o[1] = pay; o[2] = pbr; o[3] = pby;
    }
}

// Side records kept between the phases of an adjoint step (shared memory, [2][L] each; the final (r, u) are in gh)
template <typename T> struct SideTab {
    int* src; int* sig_lane;
    T* s; T* gr; T* gu;
};
template <typename T> __host__ __device__ inline size_t side_tab_bytes(int L) {
    return align8(sizeof(int) * (size_t)4 * L) + sizeof(T) * (size_t)6 * L;
}
template <typename T> __device__ __forceinline__ SideTab<T> side_tab_carve(unsigned char*& p, int L) {
    SideTab<T> s;
    T* q = reinterpret_cast<T*>(p);
    s.s = q; s.gr = q + 2 * L; s.gu = q + 4 * L;
    p += sizeof(T) * (size_t)6 * L;
    s.src = reinterpret_cast<int*>(p); s.sig_lane = s.src + 2 * L;
    p += align8(sizeof(int) * (size_t)4 * L);
    return s;
}

// ghost adjoint (d loss / d (r, y) of a ghost cell) -> from_r_u -> blend -> own-record recurrence -> published
// (d green r, d green u, d signal);  g_inc_row: this step's row of g_incoming or null.  One call per (lane, side); src,
// sig_lane, s, green_r, green_u: the side's record as resolve_side returned it (kept in a SideTab or recomputed).
template <typename T>
__device__ __forceinline__ void net_adj_side(const NetArgs<T>& a, const T* gh, int l, int side, int src, int sig_lane, T s,
                                             T green_r, T green_u, T g_r, T g_y, T* GO, T* pub, T* g_inc_row) {
    const int L = a.L, q = side * L + l;
    const T fr = gh[2 * q], fu = gh[2 * q + 1];
    const T ue = u_eq(fr, a.umax);
    T gfr = g_r + g_y * (fu - ue - fr * u_eq_true_prime(fr, a.umax));
    T gfu = g_y * fr;
    const int os = a.own_slot[q];
    if (os >= 0) { gfr += GO[2 * os]; gfu += GO[2 * os + 1]; }       // own_{t+1} = final_t
    T ggr = gfr, ggu = gfu, gs = T(0);
    if (a.mode == 1) {
        const T red_r = side == 0 ? T(0) : T(1), red_u = side == 0 ? a.umax : T(0);
        ggr = gfr * s; ggu = gfu * s;
        gs = gfr * (green_r - red_r) + gfu * (green_u - red_u);
        if (side == 1) gs = a.soft ? gs * T(32) * s * (T(1) - s) : T(0);
        if (sig_lane < 0) gs = T(0);
    }
    if (os >= 0) {
        const bool own_src = src == -1;
        GO[2 * os] = own_src ? ggr : T(0); GO[2 * os + 1] = own_src ? ggu : T(0);
    }
    if (side == 0 && g_inc_row) g_inc_row[l] = src == -2 ? ggr + ggu * u_eq_true_prime(green_r, a.umax) : T(0);
    T* pb = pub + ((size_t)l * 2 + side) * 3;
    pb[0] = src >= 0 ? ggr : T(0); pb[1] = src >= 0 ? ggu : T(0); pb[2] = gs;
}

}  // namespace dhts
