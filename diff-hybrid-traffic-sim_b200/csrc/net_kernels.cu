// Fused T-step rollout of a CONNECTED macro network (many replicas per launch), forward and adjoint.
//
// What it replaces in the reference, per simulation step and per replica:
//   RoadNetwork.forward                       road/network/road_network.py:79-111   (boundaries -> forward -> update, Jacobi)
//   RoadNetwork.get_macro_boundary            road/network/road_network.py:299-362  (ghost source: the only neighbour, or the
//                                                                                   lane the MacroRoute of this step selects,
//                                                                                   else the lane's own ghost cell)
//   ItscpRoadNetwork.setup_macro_boundary     example/control/itscp/_simulator.py:56-142  (signal blend of the ghost cells)
//   MacroLane.set_{left,right}most_cell       road/lane/_macro_lane.py:156-162 -> ARZ.FullQ.from_r_u (_arz.py:74-80)
//   dMacroLane.forward / dMacroForwardLayer   road/lane/dmacro_lane.py:68-132,234-310
//   queue-length reward (optional)            example/control/itscp/_env.py:662-742,770-797
// and the autograd chain through all of it (SURVEY 8f rows f1-f3).
//
// Shape of the work: a network is L lanes of a few cells each (ITSCP: 144 lanes of 1-4 cells), coupled every step
// through ghost cells; replicas (scenarios, candidate signal plans) are independent.  One CTA steps one replica:
// the whole network state lives in shared memory for the T steps, one thread per lane (its cells are swept
// serially with the same per-interface math as the lane kernels, dhts_arz_lean.cuh), one block barrier per step.
// Long lanes belong to the lane-batched rollout (arz_rollout.cu); this kernel is for many short coupled lanes.
//
// Ghost cells.  side 0 = left (upstream), 1 = right.  green = (r, u) of the source; the ITSCP blend is
//   left : final = green * s + (0, u_max) * (1 - s),  s = 1 when the lane has no predecessor (green = (incoming,
//          u_eq(incoming))), 0 when the step's MacroRoute gives it no predecessor, else the RAW signal of that lane
//   right: final = s * green + (1 - s) * (1, 0),      s = sigmoid(clamp(32 (sig - 0.5), -16, 16))  [soft]
//                                                     s = sig > 0.5                                 [hard]
// and the lane's own ghost record is overwritten with `final` every step, so a side without a neighbour feeds on
// its own previous value (a recurrence carried in `own`).  mode 0 (plain RoadNetwork): final = green.
//
// Adjoint.  Every state is stored by the forward pass ([T+1][R][3][NC]); the adjoint walks the steps backwards:
// compute_u's true derivative folds the adjoint of the stored speed into (r, y); each lane thread rebuilds its two
// ghosts, runs the flux-difference adjoint over its cells, pulls the ghost adjoint back through from_r_u and the
// blend, and publishes (d green, d signal) per side in shared memory; after one barrier each lane GATHERS what its
// neighbours published for its edge cells and for its signal (fixed order: deterministic, no atomics).
#include <cuda_pipeline.h>
#include "dhts_net_if.cuh"

namespace dhts {

// Shared-memory layout (host and device agree through these two functions).
//   forward:  tabs | state x 2 (r, y, u) | own x 2 | gh [2][L][2] | flux [NI][2] | qc [NC] | red [threads]
//   adjoint:  tabs | side tab | cur, nxt, pre (r, y, u) | G (gr, gy, gu) | own, own_pre, GO | gh | ab [NI][4] | pub [L][2][3] | gq [L]
template <typename T> static size_t net_smem(int L, int NC, int n_own, bool adj, int threads) {
    const int NI = NC + L;
    size_t b = net_tabs_bytes<T>(L, NC, NI);
    if (!adj) return b + sizeof(T) * ((size_t)6 * NC + 4 * n_own + 4 * (size_t)L + 2 * (size_t)NI + NC + threads) + 16;
    return b + side_tab_bytes<T>(L) +
           sizeof(T) * ((size_t)12 * NC + 6 * n_own + 4 * (size_t)L + 4 * (size_t)NI + 6 * (size_t)L + NC) + 16;
}

// ------------------------------------------------------------------------------------------------ forward
// hist  [T+1][R][3][NC]  state (r, y, u) before step t (t = 0..T-1) and after the last step
// ownh  [T+1][R][n_own][2] carried own-ghost records, same indexing
template <typename T>
__global__ void __launch_bounds__(512) net_rollout_fwd_kernel(NetArgs<T> a, const T* __restrict__ r0, const T* __restrict__ y0,
                                                               const T* __restrict__ u0, const T* __restrict__ own0,
                                                               T* __restrict__ hist, T* __restrict__ ownh,
                                                               T* __restrict__ reward, int* __restrict__ flags) {
    extern __shared__ __align__(16) unsigned char raw[];
    const int NC = a.NC, L = a.L, NI = NC + L;
    unsigned char* pp = raw;
    const NetTabs<T> tb = net_tabs_carve<T>(pp, a, NI);
    T* sm = reinterpret_cast<T*>(pp);
    T* buf[2] = {sm, sm + 3 * NC};                         // (r, y, u) x NC, double buffered
    T* own[2] = {sm + 6 * NC, sm + 6 * NC + 2 * a.n_own};
    T* gh = sm + 6 * NC + 4 * a.n_own;                     // [2][L][2] final ghost (r, u) of the step
    T* flux = gh + 4 * L;                                  // [NI][2]
    T* qc = flux + 2 * NI;                                 // [NC] queue-reward terms of the cells
    T* red = qc + NC;                                      // [blockDim] reward reduction
    net_tabs_init(a, tb);
    const T inv_veh_len = T(1) / a.veh_len;
    for (int b = blockIdx.x; b < a.R; b += gridDim.x) {
        __syncthreads();
        for (int c = threadIdx.x; c < NC; c += blockDim.x) {
            buf[0][c] = r0[(size_t)b * NC + c]; buf[0][NC + c] = y0[(size_t)b * NC + c]; buf[0][2 * NC + c] = u0[(size_t)b * NC + c];
        }
        for (int c = threadIdx.x; c < 2 * a.n_own; c += blockDim.x) own[0][c] = own0[(size_t)b * 2 * a.n_own + c];
        __syncthreads();
        bool bad = false, bad_route = false;
        T rew = T(0);
        int p = 0;
        // per-step rows of the inputs and of the stored history: advanced by one stride per step
        const int* rt = a.route ? a.route + (size_t)b * a.route_stride : nullptr;
        const T* sig_t = a.sig ? a.sig + (size_t)b * a.T_steps * L : nullptr;
        const T* inc_t = a.incoming ? a.incoming + (size_t)b * a.T_steps * L : nullptr;
        T* h = hist + (size_t)b * 3 * NC;
        T* oh = ownh + (size_t)b * 2 * a.n_own;
        const size_t h_stride = (size_t)a.R * 3 * NC, oh_stride = (size_t)a.R * 2 * a.n_own;
        for (int t = 0; t <= a.T_steps; t++, h += h_stride, oh += oh_stride) {
            const T* cr = buf[p]; const T* cy = cr + NC; const T* cu = cy + NC;
            // store the state before step t (coalesced)
            for (int c = threadIdx.x; c < 3 * NC; c += blockDim.x) h[c] = cr[c];
            for (int c = threadIdx.x; c < 2 * a.n_own; c += blockDim.x) oh[c] = own[p][c];
            // queue reward of the state after step t - 1, lane by lane (its cell terms were left in qc)
            if (a.qk && t > 0) {
                for (int l = threadIdx.x; l < L; l += blockDim.x) {
                    T q = T(0);
                    for (int c = a.cell_off[l]; c < a.cell_off[l + 1]; c++) q += qc[c];
                    rew -= q * q * a.dt;
                }
            }
            if (t == a.T_steps) break;
            T* nr = buf[p ^ 1]; T* ny = nr + NC; T* nu = ny + NC;
            // ---- G: ghosts, one thread per (side, lane)
            for (int q = threadIdx.x; q < 2 * L; q += blockDim.x) {
                const int side = q >= L, l = q - side * L;
                const Side<T> sd = resolve_side(a, l, side, rt, cr, cu, own[p], sig_t, inc_t, bad_route);
                gh[2 * q] = sd.fr; gh[2 * q + 1] = sd.fu;
                const int os = a.own_slot[q];
                if (os >= 0) { own[p ^ 1][2 * os] = sd.fr; own[p ^ 1][2 * os + 1] = sd.fu; }
            }
            __syncthreads();
            // ---- I: fluxes, one thread per interface
            bad |= net_fwd_flux<T>(a, tb, cr, cy, cu, nullptr, gh, flux);
            __syncthreads();
            // ---- C: update, one thread per cell (_macro_lane.py:83-114; set_r_y refreshes u, _arz.py:88-92)
            for (int c = threadIdx.x; c < NC; c += blockDim.x) {
                const int l = tb.lane_of_cell[c];
                const int it = tb.if_off[l] + (c - a.cell_off[l]);
                const T cc = tb.cc[l];
                const T r = fma(flux[2 * it] - flux[2 * it + 2], cc, cr[c]);
                const T y = fma(flux[2 * it + 1] - flux[2 * it + 3], cc, cy[c]);
                const T u = compute_u(r, y, a.umax);
                nr[c] = r; ny[c] = y; nu[c] = u;
                if (a.qk) {
                    T z = (a.static_speed - u) * a.qk[t];
                    z = z < T(-16) ? T(-16) : (z > T(16) ? T(16) : z);
                    qc[c] = sigm(z) * (r * tb.dxv[l] * inv_veh_len);
                }
            }
            __syncthreads();
            p ^= 1;
            if (rt) rt += 2 * L;
            if (sig_t) sig_t += L;
            if (inc_t) inc_t += L;
        }
        if (reward) {   // fixed-order tree reduction of the per-thread partial sums
            red[threadIdx.x] = rew;
            __syncthreads();
            for (int s = 1; s < (int)blockDim.x; s <<= 1) {
                if ((threadIdx.x & (2 * s - 1)) == 0 && threadIdx.x + s < blockDim.x) red[threadIdx.x] += red[threadIdx.x + s];
                __syncthreads();
            }
            if (threadIdx.x == 0) reward[b] = red[0];
        }
        if (bad) atomicOr(flags, FLAG_CFL);
        if (bad_route) atomicOr(flags, FLAG_ROUTE);
    }
}

// ------------------------------------------------------------------------------------------------ adjoint
// g_states [T][R][3][NC]  optional: dLoss/d(r, y, u) of the state AFTER step t (the last one is the terminal adjoint)
// g_reward [R]            optional: dLoss/d reward (fused queue reward)
// outputs: g_r0, g_y0, g_u0 [R][NC]; g_own0 [R][n_own][2]; g_sig, g_inc [R][T][L]
// MAXTH / MINB: launch bounds.  (512, 1): up to one thread per interface of a large network, 128 registers.  (256, 3): the
// many-replica configuration (half as many threads as interfaces, several CTAs per SM hiding each other's barriers) at 80
// registers -- no spills, three CTAs per SM instead of two.
template <typename T, int MAXTH, int MINB>
__global__ void __launch_bounds__(MAXTH, MINB) net_rollout_bwd_kernel(NetArgs<T> a, const T* __restrict__ hist, const T* __restrict__ ownh,
                                                               const T* __restrict__ g_states, const T* __restrict__ g_reward,
                                                               T* __restrict__ g_r0, T* __restrict__ g_y0, T* __restrict__ g_u0,
                                                               T* __restrict__ g_own0, T* __restrict__ g_sig,
                                                               T* __restrict__ g_inc, int* __restrict__ flags) {
    extern __shared__ __align__(16) unsigned char raw[];
    const int NC = a.NC, L = a.L, NI = NC + L;
    unsigned char* pp = raw;
    const NetTabs<T> tb = net_tabs_carve<T>(pp, a, NI);
    const SideTab<T> sd = side_tab_carve<T>(pp, L);
    T* sm = reinterpret_cast<T*>(pp);
    // three rotating state buffers: state t (cur), state t + 1 (nxt) and the row being prefetched for the next step
    // (pre); the stored rows stream in with cp.async (LDGSTS) one step ahead of the arithmetic
    T* cur = sm;                        // state t      (r, y, u)
    T* nxt = sm + 3 * NC;               // state t + 1  (r, y, u)
    T* pre = sm + 6 * NC;               // state t - 1, in flight
    T* G = sm + 9 * NC;                 // adjoint of state t+1 on entry of a step, of state t on exit: (gr, gy, gu)
    T* own = sm + 12 * NC;              // own records at step t
    T* own_pre = own + 2 * a.n_own;     // own records at step t - 1, in flight
    T* GO = own_pre + 2 * a.n_own;      // adjoint of the own records
    T* gh = GO + 2 * a.n_own;           // [2][L][2] final ghost (r, u) of step t
    T* ab = gh + 4 * L;                 // [NI][4] A^T w, B^T w per interface
    T* pub = ab + 4 * (size_t)NI;       // [L][2 sides][3] published (d green r, d green u, d signal)
    T* gq = pub + (size_t)6 * L;        // [NC] queue-reward sigmoid of every cell of state t + 1
    net_tabs_init(a, tb);
    for (int b = blockIdx.x; b < a.R; b += gridDim.x) {
        __syncthreads();
        {   // terminal state and adjoint
            const T* h = hist + ((size_t)a.T_steps * a.R + b) * 3 * NC;
            for (int c = threadIdx.x; c < 3 * NC; c += blockDim.x) {
                nxt[c] = h[c];
                G[c] = (g_states && a.T_steps > 0) ? g_states[((size_t)(a.T_steps - 1) * a.R + b) * 3 * NC + c] : T(0);
            }
            for (int c = threadIdx.x; c < 2 * a.n_own; c += blockDim.x) GO[c] = T(0);
        }
        const T grew = g_reward ? g_reward[b] : T(0);
        const bool fused = a.qk && g_reward;
        const T inv_veh_len = T(1) / a.veh_len;
        const int* rt0 = a.route ? a.route + (size_t)b * a.route_stride : nullptr;
        const T* sig0 = a.sig ? a.sig + (size_t)b * a.T_steps * L : nullptr;
        const T* inc0 = a.incoming ? a.incoming + (size_t)b * a.T_steps * L : nullptr;
        bool nan = false;
#define DHTS_NET_PREFETCH(TT, DST, ODST)                                                                               \
        {                                                                                                              \
            const T* h_ = hist + ((size_t)(TT) * a.R + b) * 3 * NC;                                                    \
            for (int c = threadIdx.x; c < 3 * NC; c += blockDim.x) __pipeline_memcpy_async((DST) + c, h_ + c, sizeof(T)); \
            const T* oh_ = ownh + ((size_t)(TT) * a.R + b) * 2 * a.n_own;                                              \
            for (int c = threadIdx.x; c < 2 * a.n_own; c += blockDim.x) __pipeline_memcpy_async((ODST) + c, oh_ + c, sizeof(T)); \
            __pipeline_commit();                                                                                       \
        }
        if (a.T_steps > 0) DHTS_NET_PREFETCH(a.T_steps - 1, cur, own)
        for (int t = a.T_steps - 1; t >= 0; t--) {
            __pipeline_wait_prior(0);
            __syncthreads();          // state t has landed; the previous step's gathers are complete
            if (t > 0) DHTS_NET_PREFETCH(t - 1, pre, own_pre)          // pre was state t + 2: nobody reads it any more
            const T* cr = cur; const T* cy = cur + NC; const T* cu = cur + 2 * NC;
            const int* rt = rt0 ? rt0 + (size_t)t * 2 * L : nullptr;
            const T* sig_t = sig0 ? sig0 + (size_t)t * L : nullptr;
            const T* inc_t = inc0 ? inc0 + (size_t)t * L : nullptr;
            bool dummy = false;
            // ---- A0: the queue-reward sigmoid of every cell of state t + 1 (fused queue reward), once
            if (fused) {
                const T qk = a.qk[t];
                for (int c = threadIdx.x; c < NC; c += blockDim.x) {
                    const T zr = (a.static_speed - nxt[2 * NC + c]) * qk;
                    const T z = zr < T(-16) ? T(-16) : (zr > T(16) ? T(16) : zr);
                    gq[c] = sigm(z);
                }
                __syncthreads();
            }
            // ---- A: per cell, reward adjoint and the stored speed's adjoint folded into (r, y); per (side, lane), ghosts of step t
            for (int c = threadIdx.x; c < NC; c += blockDim.x) {
                T gr = G[c], gy = G[NC + c], gu = G[2 * NC + c];
                if (fused) {
                    const int l = tb.lane_of_cell[c];
                    const T w = tb.dxv[l] * inv_veh_len;
                    T q = T(0);                                            // queue length of the cell's lane (<= a few cells)
                    for (int j = a.cell_off[l]; j < a.cell_off[l + 1]; j++) q += gq[j] * (nxt[j] * w);
                    const T glq = -T(2) * q * a.dt * grew;                 // d loss / d (queue length of the lane)
                    const T qk = a.qk[t];
                    const T zr = (a.static_speed - nxt[2 * NC + c]) * qk;
                    const bool in = zr >= T(-16) && zr <= T(16);
                    const T sg = gq[c];
                    gr += glq * sg * w;
                    if (in) gu += glq * nxt[c] * w * sg * (T(1) - sg) * (-qk);
                }
                T dr, dy; du_dry(nxt[c], nxt[NC + c], a.umax, dr, dy);
                G[c] = gr + gu * dr; G[NC + c] = gy + gu * dy;
            }
            for (int q = threadIdx.x; q < 2 * L; q += blockDim.x) {
                const int side = q >= L, l = q - side * L;
                const Side<T> s = resolve_side(a, l, side, rt, cr, cu, own, sig_t, inc_t, dummy);
                gh[2 * q] = s.fr; gh[2 * q + 1] = s.fu;
                sd.src[q] = s.src; sd.sig_lane[q] = s.sig_lane; sd.s[q] = s.s; sd.gr[q] = s.gr_; sd.gu[q] = s.gu_;
            }
            __syncthreads();
            // ---- I: flux-difference adjoint, one thread per interface
            net_adj_flux<T>(a, tb, cr, cy, cu, nullptr, gh, G, G + NC, ab);
            __syncthreads();
            // ---- C: per cell, the adjoint of state t (before the gathers) with the injected adjoint; per (side, lane), the
            // ghost adjoint pulled through from_r_u and the blend
            for (int c = threadIdx.x; c < NC; c += blockDim.x) {
                const int l = tb.lane_of_cell[c];
                const int it = tb.if_off[l] + (c - a.cell_off[l]);      // interface on the cell's left; it + 1 on its right
                const T cc = tb.cc[l];
                T nr_ = fma(cc, ab[4 * (it + 1)] + ab[4 * it + 2], G[c]);
                T ny_ = fma(cc, ab[4 * (it + 1) + 1] + ab[4 * it + 3], G[NC + c]);
                nan |= t_isnan(nr_) || t_isnan(ny_);
                T nu_ = T(0);                                             // the stored speed of state t: filled by the gathers
                if (g_states && t > 0) {
                    const T* gs_ = g_states + ((size_t)(t - 1) * a.R + b) * 3 * NC;
                    nr_ += gs_[c]; ny_ += gs_[NC + c]; nu_ = gs_[2 * NC + c];
                }
                G[c] = nr_; G[NC + c] = ny_; G[2 * NC + c] = nu_;
            }
            for (int q = threadIdx.x; q < 2 * L; q += blockDim.x) {
                const int side = q >= L, l = q - side * L;
                const T cc = tb.cc[l];
                const T* o = ab + 4 * (size_t)(side == 0 ? tb.if_off[l] : tb.if_off[l + 1] - 1);
                const T g_r = cc * (side == 0 ? o[0] : o[2]), g_y = cc * (side == 0 ? o[1] : o[3]);
                net_adj_side<T>(a, gh, l, side, sd.src[q], sd.sig_lane[q], sd.s[q], sd.gr[q], sd.gu[q], g_r, g_y, GO, pub, g_inc ? g_inc + ((size_t)b * a.T_steps + t) * L : nullptr);
            }
            __syncthreads();
            // ---- gathers, one thread per lane: what the neighbours took from this lane's edge cells and from its signal
            for (int l = threadIdx.x; l < L; l += blockDim.x) {
                const int c0 = a.cell_off[l], N = a.cell_off[l + 1] - c0;
                T gsig = pub[((size_t)l * 2 + 1) * 3 + 2];
                // successors whose LEFT ghost came from this lane's last cell / was blended by this lane's signal
                for (int e = a.adj_off[(L + 1) + l]; e < a.adj_off[(L + 1) + l + 1]; e++) {
                    const int n = a.adj[e];
                    const int cnt = a.nadj[n];
                    const int sel = rt ? rt[n] : -1;
                    const int srcn = cnt == 1 ? a.one_adj[n] : (cnt > 1 ? sel : -1);
                    const T* pb = pub + ((size_t)n * 2 + 0) * 3;
                    if (srcn == l) { G[c0 + N - 1] += pb[0]; G[2 * NC + c0 + N - 1] += pb[1]; }
                    if (a.mode == 1 && sel == l) gsig += pb[2];
                }
                // predecessors whose RIGHT ghost came from this lane's first cell
                for (int e = a.adj_off[l]; e < a.adj_off[l + 1]; e++) {
                    const int pl = a.adj[e];
                    const int cnt = a.nadj[L + pl];
                    const int sel = rt ? rt[L + pl] : -1;
                    const int srcp = cnt == 1 ? a.one_adj[L + pl] : (cnt > 1 ? sel : -1);
                    const T* pb = pub + ((size_t)pl * 2 + 1) * 3;
                    if (srcp == l) { G[c0] += pb[0]; G[2 * NC + c0] += pb[1]; }
                }
                if (g_sig) g_sig[((size_t)b * a.T_steps + t) * L + l] = gsig;
                nan |= t_isnan(gsig);
            }
            { T* x_ = nxt; nxt = cur; cur = pre; pre = x_; x_ = own; own = own_pre; own_pre = x_; }     // rotate: no copy, no barrier
        }
#undef DHTS_NET_PREFETCH
        __syncthreads();
        for (int c = threadIdx.x; c < NC; c += blockDim.x) {
            g_r0[(size_t)b * NC + c] = G[c]; g_y0[(size_t)b * NC + c] = G[NC + c]; g_u0[(size_t)b * NC + c] = G[2 * NC + c];
            nan |= t_isnan(G[c]) || t_isnan(G[NC + c]) || t_isnan(G[2 * NC + c]);
        }
        if (g_own0)
            for (int c = threadIdx.x; c < 2 * a.n_own; c += blockDim.x) g_own0[(size_t)b * 2 * a.n_own + c] = GO[c];
        if (nan) atomicOr(flags, FLAG_NAN_GRAD);
    }
}

// ------------------------------------------------------------------------------------------------ host side
// Few replicas (latency-bound: a CTA's step time is what counts): one thread per interface, NC + L of them, up to 512.
// Many replicas (throughput-bound: several CTAs per SM hide each other's barriers): a fraction of that, each thread looping --
// a third for the forward kernel (on the ITSCP grid 2 L = NC = 288 and NI = 432 are then 2, 2 and 3 nearly full iterations of
// 160 threads: 16.1 instead of 17.9 ms at 2048 replicas, r3w), half for the adjoint (three 80-register CTAs per SM; a third
// measured 43.2 instead of 41.5 ms).
constexpr int NET_DIV_FWD = 3, NET_DIV_BWD = 2;
static int net_threads(int L, int NC, int R, bool adj) {
    int ni = NC + L;
    const int div = adj ? NET_DIV_BWD : NET_DIV_FWD;
    if (R > sm_count()) ni = (ni + div - 1) / div;
    int t = (ni + 31) / 32 * 32;
    return t > 512 ? 512 : (t < 32 ? 32 : t);
}


template <typename T>
static int net_check(const NetArgs<T>& a) {
    if (a.L < 1 || a.NC < a.L || a.n_own < 0 || a.T_steps < 0 || a.R < 0 || !a.cell_off || !a.dx || !a.nadj || !a.one_adj ||
        !a.adj_off || !a.own_slot)
        return DHTS_ERR_INVALID;
    if (a.mode == 1 && (!a.sig || !a.incoming)) return DHTS_ERR_INVALID;
    if (a.mode != 0 && a.mode != 1) return DHTS_ERR_INVALID;
    return DHTS_OK;
}

template <typename T>
static int net_fwd(const NetArgs<T>& a, const T* r0, const T* y0, const T* u0, const T* own0, T* hist, T* ownh, T* reward,
                   int* flags, cudaStream_t st) {
    int rc = net_check(a);
    if (rc) return rc;
    if (!r0 || !y0 || !u0 || !hist || !flags || (a.n_own > 0 && (!own0 || !ownh))) return DHTS_ERR_INVALID;
    if (a.R == 0) return DHTS_OK;
    const int threads = net_threads(a.L, a.NC, a.R, false);
    const size_t smem = net_smem<T>(a.L, a.NC, a.n_own, false, threads);
    int grid = 1;
    rc = persistent_grid(net_rollout_fwd_kernel<T>, threads, smem, a.R, &grid);
    if (rc) return rc;
    net_rollout_fwd_kernel<T><<<grid, threads, smem, st>>>(a, r0, y0, u0, own0, hist, ownh, reward, flags);
    return launch_status();
}

template <typename T>
static int net_bwd(const NetArgs<T>& a, const T* hist, const T* ownh, const T* g_states, const T* g_reward, T* g_r0, T* g_y0,
                   T* g_u0, T* g_own0, T* g_sig, T* g_inc, int* flags, cudaStream_t st) {
    int rc = net_check(a);
    if (rc) return rc;
    if (!hist || !g_r0 || !g_y0 || !g_u0 || !flags || (a.n_own > 0 && !ownh)) return DHTS_ERR_INVALID;
    if (a.R == 0) return DHTS_OK;
    const int threads = net_threads(a.L, a.NC, a.R, true);
    const size_t smem = net_smem<T>(a.L, a.NC, a.n_own, true, threads);
    int grid = 1;
    if (threads <= 256 && a.R > sm_count()) {       // many replicas: 80 registers, three CTAs per SM (44.8 -> 41.2 ms)
        rc = persistent_grid(net_rollout_bwd_kernel<T, 256, 3>, threads, smem, a.R, &grid);
        if (rc) return rc;
        net_rollout_bwd_kernel<T, 256, 3><<<grid, threads, smem, st>>>(a, hist, ownh, g_states, g_reward, g_r0, g_y0, g_u0, g_own0,
                                                                       g_sig, g_inc, flags);
    } else {
        rc = persistent_grid(net_rollout_bwd_kernel<T, 512, 1>, threads, smem, a.R, &grid);
        if (rc) return rc;
        net_rollout_bwd_kernel<T, 512, 1><<<grid, threads, smem, st>>>(a, hist, ownh, g_states, g_reward, g_r0, g_y0, g_u0, g_own0,
                                                                       g_sig, g_inc, flags);
    }
    return launch_status();
}

template <typename T> static NetArgs<T> net_args(const dhts_net_topology* tp, const int* route, int route_per_replica, T umax, T dt,
                                                 int steps, int R, int mode, int soft, const T* sig, const T* incoming,
                                                 const T* dx, const T* qk, T veh_len, T static_speed) {
    NetArgs<T> a;
    a.L = tp->L; a.NC = tp->NC; a.n_own = tp->n_own; a.T_steps = steps; a.R = R; a.mode = mode; a.soft = soft;
    a.cell_off = tp->cell_off; a.dx = dx; a.nadj = tp->nadj; a.one_adj = tp->one_adj; a.adj_off = tp->adj_off; a.adj = tp->adj;
    a.own_slot = tp->own_slot; a.route = route; a.route_stride = route_per_replica ? (long long)steps * 2 * tp->L : 0;
    a.umax = umax; a.dt = dt; a.veh_len = veh_len; a.static_speed = static_speed;
    a.sig = sig; a.incoming = incoming; a.qk = qk; a.kind = nullptr;
    return a;
}

}  // namespace dhts

#define DHTS_NET_API(SUF, T)                                                                                           \
    DHTS_EXPORT int dhts_net_rollout_fwd_##SUF(const dhts_net_topology* topo, const T* dx, const int* route,           \
                                               int route_per_replica, const T* sig, const T* incoming, const T* qk,    \
                                               T umax, T dt, T veh_len, T static_speed, int steps, int R, int mode,    \
                                               int soft, const T* r0, const T* y0, const T* u0, const T* own0,         \
                                               T* hist, T* own_hist, T* reward, int* flags, void* stream) {            \
        if (!topo) return DHTS_ERR_INVALID;                                                                            \
        return dhts::net_fwd<T>(dhts::net_args<T>(topo, route, route_per_replica, umax, dt, steps, R, mode, soft, sig, \
                                                  incoming, dx, qk, veh_len, static_speed),                            \
                                r0, y0, u0, own0, hist, own_hist, reward, flags, (cudaStream_t)stream);                \
    }                                                                                                                  \
    DHTS_EXPORT int dhts_net_rollout_bwd_##SUF(const dhts_net_topology* topo, const T* dx, const int* route,           \
                                               int route_per_replica, const T* sig, const T* incoming, const T* qk,    \
                                               T umax, T dt, T veh_len, T static_speed, int steps, int R, int mode,    \
                                               int soft, const T* hist, const T* own_hist, const T* g_states,          \
                                               const T* g_reward, T* g_r0, T* g_y0, T* g_u0, T* g_own0, T* g_sig,      \
                                               T* g_incoming, int* flags, void* stream) {                              \
        if (!topo) return DHTS_ERR_INVALID;                                                                            \
        return dhts::net_bwd<T>(dhts::net_args<T>(topo, route, route_per_replica, umax, dt, steps, R, mode, soft, sig, \
                                                  incoming, dx, qk, veh_len, static_speed),                            \
                                hist, own_hist, g_states, g_reward, g_r0, g_y0, g_u0, g_own0, g_sig, g_incoming, flags, \
                                (cudaStream_t)stream);                                                                 \
    }

DHTS_NET_API(f64, double)
DHTS_NET_API(f32, float)
