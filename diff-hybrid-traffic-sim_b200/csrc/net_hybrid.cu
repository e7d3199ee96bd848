// Fused T-step rollout of a connected HYBRID network (macro ARZ lanes + micro IDM lanes + the conversions between
// them), many replicas per launch, forward and adjoint.  SURVEY 8f rows f1-f3 for configs 3 and 4 (hybrid inverse
// problem, ITSCP hybrid mode).
//
// What it replaces in the reference, per simulation step and per replica:
//   RoadNetwork.forward / conversion*         road/network/road_network.py:79-173   boundaries -> forward -> update ->
//                                                                                   conversions in lane-id order
//   RoadNetwork.get_macro_boundary            road/network/road_network.py:299-362  (a micro neighbour => own ghost record)
//   RoadNetwork.setup_micro_boundary          road/network/road_network.py:429-580  head vehicle's leader along its route
//   ItscpRoadNetwork.setup_macro_boundary     example/control/itscp/_simulator.py:56-142
//   ItscpRoadNetwork.setup_micro_boundary     example/control/itscp/_simulator.py:144-276  signal-blended head deltas,
//                                                                                   running-mean sigmoid constant
//   dMacroLane / dMicroLane operators         road/lane/dmacro_lane.py:68-132,234-310; road/lane/dmicro_lane.py:87-153,228-297
//   Conversion.macro_to_micro                 road/network/conversion.py:15-73     flux capacitor, spawn
//   Conversion.micro_to_macro                 road/network/conversion.py:75-171    head absorbed into the next lane's cells
//   Conversion.micro_to_micro / micro_to_none road/network/conversion.py:174-215   hand-off / drop
// and the autograd chain through all of it.
//
// Shape of the work: as in net_kernels.cu one CTA steps one replica with the whole network state in shared memory
// and one thread per lane.  A micro lane keeps its vehicles in a ring of `cap` slots (a vehicle keeps its slot while
// it is on the lane): front = head vehicle, new vehicles are appended behind the tail.  Every spawned vehicle uses
// default_micro_vehicle's parameters (road/vehicle/micro_vehicle.py:30-72); its route is an INPUT (the reference
// draws it with create_random_route, road_network.py:604-646): spawn_route[m][k] names the route of the k-th
// vehicle spawned into micro lane m.
//
// Conversions are sequential in lane-id order in the reference and they interact (a deposit changes the cell the
// next capacitor reads; a hand-off changes the free space a spawn tests).  The host partitions the lanes that take
// part in conversions into GROUPS (connected components of "touches the same lane"); one thread runs one group in
// lane-id order, groups run in parallel -- the same result as the sequential loop.
//
// State per replica: cells (r, y, u, u_eq) lane by lane -- u_eq is the STORED equilibrium speed, stale on cells a
// deposit rewrote (conversion.py:157-167 refreshes r, u, y only; SURVEY App. B.3) -- own ghost records, and the
// `aux` row: vehicles (p, v, a, route id, route cursor) [ML][cap] each, ring front / count / spawn counter [ML],
// flux capacitors [NCAP], running-mean (sum, count) of the micro signal.
//
// Adjoint: every state row is stored by the forward pass.  The adjoint kernel walks the steps backwards; for step t
// it REPLAYS the forward step from the stored state t (same device function, recording the conversion events and
// the state between update and conversions in shared memory) and then reverses it: conversions in reverse order per
// group, the IDM / ARZ operators per lane, the ghost / head-delta blends, and gathers of everything a lane's
// neighbours took from it (fixed order, no atomics).
#include <cmath>
#include <cuda_pipeline.h>
#include "dhts_net_if.cuh"
#include "dhts_idm.cuh"

// Diagnosis build (-DDHTS_PHASE_TIMING, scripts/hyb_phases.py): thread 0 of CTA 0 accumulates the cycles between the phase
// boundaries of a step (barrier waits included, i.e. the wall time of each phase as the slowest thread sets it).
#ifdef DHTS_PHASE_TIMING
__device__ unsigned long long g_phase_cycles[32];
#define DHTS_PT_DECL unsigned long long pt_last_ = clock64();
#define DHTS_PT(i) if (threadIdx.x == 0 && blockIdx.x == 0) { const unsigned long long now_ = clock64(); atomicAdd(&g_phase_cycles[i], now_ - pt_last_); pt_last_ = now_; }
extern "C" __attribute__((visibility("default"))) int dhts_debug_phase_cycles(unsigned long long* out32) {
    cudaDeviceSynchronize();
    unsigned long long z[32] = {0};
    if (cudaMemcpyFromSymbol(out32, g_phase_cycles, sizeof(z)) != cudaSuccess) return 1;
    return cudaMemcpyToSymbol(g_phase_cycles, z, sizeof(z)) != cudaSuccess;
}
#else
#define DHTS_PT_DECL
#define DHTS_PT(i)
#endif

namespace dhts {

constexpr int FLAG_VEH_OVERFLOW = 16;
constexpr int HYB_THREADS_MAX = 512;

struct AuxL { int P, V, A, RID, CUR, PID, FRONT, CNT, NSP, CAP, RMS, DRAW, AUX; };
__host__ __device__ inline AuxL aux_layout(int ML, int cap, int NCAP) {
    AuxL o;
    const int s = ML * cap;
    o.P = 0; o.V = s; o.A = 2 * s; o.RID = 3 * s; o.CUR = 4 * s; o.PID = 5 * s; o.FRONT = 6 * s; o.CNT = o.FRONT + ML;
    o.NSP = o.CNT + ML; o.CAP = o.NSP + ML; o.RMS = o.CAP + NCAP; o.DRAW = o.RMS + 2; o.AUX = o.DRAW + 1;
    return o;
}

template <typename T> struct HybArgs {
    NetArgs<T> n;             // lane graph, ghost resolution, signals (n.kind != null)
    int ML, cap, NCAP, NGL, NG, RLEN, NR, KS, MAXT;
    const int* mic_of;        // [L]  micro index of a lane, -1 for macro lanes
    const int* mic_lane;      // [ML] lane id of a micro index
    const int* cap_off;       // [L+1] CSR: flux capacitors of a macro lane, one per micro successor
    const int* cap_lane;      // [NCAP] the micro lane a capacitor feeds
    const int* grp_off;       // [NG+1] conversion groups
    const int* grp_lane;      // [NGL] lanes of each group, ascending
    const int* routes;        // [NR][RLEN] lane ids along a vehicle route, -1 terminated
    const T* lane_len;        // [L]
    const int* spawn_route;   // [Rs][ML][KS] route id of the k-th vehicle spawned into a micro lane
    long long spawn_stride;   // 0 when shared by all replicas
    const T* par_tab;         // [NP][6] IDM parameter sets (a_max, a_pref, v_target, s0, T, -); a vehicle names its set (PID), spawns use set 0
    int NP;
    T vlen;                   // length of every vehicle (RoadNetwork.vehicle_length, road_network.py:60)
    const int* src;           // [ML] or null: 1 = boundary micro lane fed from a waiting list (_simulator.py:153-174)
    const T* rnd;             // [Rr][NRAND] the uniform draws of the waiting-list source, in consumption order
    long long rnd_stride;     // 0 when shared by all replicas
    int NRAND;
    int prefetch;             // adjoint: stream the stored rows one step ahead (needs a second set of state buffers in shared memory)
    T head_dp0, head_dv0;     // DEFAULT_HEAD_POSITION_DELTA / DEFAULT_HEAD_SPEED_DELTA (_micro_lane.py:14-15)
    AuxL ax;
};

// dmath.sigmoid(value, constant) = sigma(clamp(value constant, -16, 16)), dmath/operation.py:3-30; ds = d/d value
template <typename T> __device__ __forceinline__ T sigc(T x, T c, T& ds) {
    const T z = x * c;
    const bool in = z >= T(-16) && z <= T(16);
    const T s = sigm(in ? z : (z < T(-16) ? T(-16) : T(16)));
    ds = in ? c * s * (T(1) - s) : T(0);
    return s;
}

template <typename T> __device__ __forceinline__ int route_at(const HybArgs<T>& a, int rid, int k) {
    return (rid >= 0 && rid < a.NR && k >= 0 && k < a.RLEN) ? a.routes[(size_t)rid * a.RLEN + k] : -1;
}

// Head vehicle of a micro lane and everything setup_micro_boundary derives from the state before the step.
template <typename T> struct HeadRec {
    int hs, rid, cur;             // head slot, its route and cursor
    T ph, vh;
    T gdp, gdv;                   // "green" deltas: leader along the route (road_network.py:429-580)
    int lead_m, lead_slot;        // the leader: tail vehicle of micro lane lead_m, or -1 (default deltas)
    bool lead_clamped;
    T red_dp; bool red_live;      // red deltas (_simulator.py:196-198): stop at the end of the lane
    int prev_lane, next_lane;     // lanes whose signals enter final_signal, -1 = absent
    T a, b, c, da, db, dc;        // raw scores (prev, curr, next) and their derivatives wrt ph
    T fin, dfin;                  // final_signal and d final_signal / d ph
};

template <typename T>
__device__ __forceinline__ HeadRec<T> head_rec(const HybArgs<T>& a, int l, int m, const T* auxc, const T* sig_t) {
    const AuxL& x = a.ax;
    HeadRec<T> h;
    const int f = (int)auxc[x.FRONT + m];
    h.hs = f;
    h.ph = auxc[x.P + m * a.cap + f]; h.vh = auxc[x.V + m * a.cap + f];
    h.rid = (int)auxc[x.RID + m * a.cap + f]; h.cur = (int)auxc[x.CUR + m * a.cap + f];
    const T len = a.lane_len[l], vlen = a.vlen;
    // ---- leader along the route
    T acc = len - h.ph - vlen * T(0.5);
    h.gdp = a.head_dp0; h.gdv = a.head_dv0; h.lead_m = -1; h.lead_slot = 0; h.lead_clamped = false;
    for (int k = h.cur; k < a.RLEN; k++) {
        const int nl = route_at(a, h.rid, k + 1);
        if (nl < 0 || a.n.kind[nl] == 0) break;            // end of route or a macro lane: default deltas
        const int m2 = a.mic_of[nl];
        const int n2 = (int)auxc[x.CNT + m2];
        if (n2 > 0) {
            const int ts = ((int)auxc[x.FRONT + m2] + n2 - 1) % a.cap;
            const T plv = auxc[x.P + m2 * a.cap + ts], vlv = auxc[x.V + m2 * a.cap + ts];
            const T d = acc + (plv - vlen * T(0.5));
            h.lead_clamped = d < T(0);                    // max(position_delta, 0.0): the float wins only when d < 0
            h.gdp = h.lead_clamped ? T(0) : d; h.gdv = h.vh - vlv;
            h.lead_m = m2; h.lead_slot = ts;
            break;
        }
        acc += a.lane_len[nl];
    }
    // ---- ITSCP: red deltas and the position-weighted signal (_simulator.py:194-246)
    h.prev_lane = h.cur > 0 ? route_at(a, h.rid, h.cur - 1) : -1;
    h.next_lane = route_at(a, h.rid, h.cur + 1);
    const T rd = len - h.ph - vlen * T(0.5);
    h.red_live = !(rd < T(0)); h.red_dp = h.red_live ? rd : T(0);
    h.a = h.b = h.c = h.da = h.db = h.dc = T(0); h.fin = T(0); h.dfin = T(0);
    if (a.n.mode == 1) {
        if (a.n.soft) {
            T d0, d1;
            if (h.prev_lane >= 0) { h.a = sigc(-h.ph, T(16), d0); h.da = -d0; }
            const T s0 = sigc(h.ph, T(16), d0), s1 = sigc(len - h.ph, T(16), d1);
            h.b = s0 * s1; h.db = d0 * s1 - s0 * d1;
            if (h.next_lane >= 0) { h.c = sigc(h.ph - len, T(16), d0); h.dc = d0; }
            const T S = h.a + h.b + h.c;
            const T sp = h.prev_lane >= 0 ? sig_t[h.prev_lane] : T(0), sc = sig_t[l], sn = h.next_lane >= 0 ? sig_t[h.next_lane] : T(0);
            h.fin = (h.a * sp + h.b * sc + h.c * sn) / S;
            h.dfin = ((h.da * sp + h.db * sc + h.dc * sn) - h.fin * (h.da + h.db + h.dc)) / S;
        } else {
            h.b = T(1); h.fin = sig_t[l];
        }
    }
    return h;
}

// geometry of one touched cell (conversion.py:124-137)
template <typename T>
__device__ __forceinline__ bool dep_cell(int ci, T dx, T len, T v_head, T v_tail, T& overlap, T& dodp) {
    const T c_head = dx * T(ci + 1), c_tail = dx * T(ci);          // Cell.end / Cell.start, _macro_lane.py:46-47
    if (!(c_head > v_tail && c_tail < v_head)) return false;
    const bool head_is_cell = c_head > v_head, tail_is_cell = c_tail < v_tail;
    const T max_head = head_is_cell ? c_head : v_head;
    const T min_tail = tail_is_cell ? c_tail : v_tail;
    overlap = dx + len - (max_head - min_tail);
    dodp = (head_is_cell ? T(0) : T(-1)) + (tail_is_cell ? T(0) : T(1));
    return true;
}

// conversion event log of one step (shared memory, adjoint kernel only): one record per lane of grp_lane
enum { EV_NONE = 0, EV_CAP = 1, EV_SPAWN = 2, EV_DROP = 3, EV_ABSORB = 4, EV_MOVE = 5 };
template <typename T> struct ConvLog {
    int* ei;      // [NGL][4]  type, slot, (capacitor | dest micro index), (spawn slot | dest slot | cells touched)
    T* et;        // [NGL][3 + MAXT]  (r_last, u_last) | (p, v, a of the popped head, n_r of every touched cell)
};

template <typename T> struct HybSm {
    T* st[2];     // (r, y, u, u_eq) x NC
    T* own[2];
    T* aux[2];
    T* fsig;      // [ML][2] final_signal of the head, lane has vehicles
    T* kconst;    // [ML] sigmoid constant of the micro signal blend
    T* headd;     // [ML][2] head deltas the IDM step used
    T* mid;       // adjoint kernel: (r, y, u) x NC between update and conversions
    ConvLog<T> log;
    NetTabs<T> tb;   // interface / cell -> lane tables of the macro lanes (dhts_net_if.cuh)
    T* gh;        // [2][L][2] final ghost (r, u) of the macro lanes at the current step
    T* flux;      // [NI][2] fluxes of the macro lanes' interfaces
    T* ab;        // adjoint kernel: [NI][4] (A^T w, B^T w) per interface; lives in st[1] (dead once the replay is done) + a tail
    SideTab<T> sd;   // adjoint kernel: side records of the current step
    int* walk;    // [NGL][6] lookups of the conversion walk of the current step (lane, kind, next / micro index, capacitor, ...)
    int* goff;    // [NG+1] group offsets (copy of grp_off)
    T* walkT;     // [NGL] length of the lane the walk asks about (macro: the micro successor; micro: the lane itself)
    IdmPar<T>* par;  // [NP] parameter sets with their derived constants
    int* srcf;    // [ML] waiting-list source: the lane had room at this step (one uniform draw consumed)
    int* srcs;    // [ML] waiting-list source: ring slot of the vehicle that entered at this step, -1 = none
    HeadRec<T>* hrec;   // [ML] head-vehicle record of the current step (phase 0), read again by the IDM step and its adjoint
    int* gflag;   // [NG] the group has a conversion candidate at this step (a pop or a spawn may happen): serial walk
    int* gof;     // [NGL] group of a group lane
};

// Parameter sets with their derived constants and the interface tables of the macro lanes.  Every thread calls it once
// per kernel; ends with a block barrier.
template <typename T> __device__ __forceinline__ void hyb_init(const HybArgs<T>& a, const HybSm<T>& s) {
    for (int i = threadIdx.x; i < a.NP; i += blockDim.x) {      // the constants of _idm.py:31-40
        const T* q = a.par_tab + (size_t)i * 6;
        IdmPar<T> k;
        k.a_max = q[0]; k.v_t_inv = T(1) / q[2]; k.s0 = q[3]; k.tp = q[4]; k.len = a.vlen;
        k.sab2_inv = T(1) / (T(2) * t_sqrt(q[0] * q[1]));
        s.par[i] = k;
    }
    // the static part of the conversion walk's lookups (phase 2a fills in what depends on the step's MacroRoute)
    const NetArgs<T>& n = a.n;
    for (int gi = threadIdx.x; gi < a.NGL; gi += blockDim.x) {
        const int l = a.grp_lane[gi];
        int* w = s.walk + gi * 6;
        w[0] = l; w[1] = n.kind[l]; w[2] = -1; w[3] = -1; w[4] = -1; w[5] = n.cell_off[l + 1] - 1;
        s.walkT[gi] = T(0);
        if (w[1] == 1) { w[2] = a.mic_of[l]; s.walkT[gi] = a.lane_len[l]; }
    }
    for (int g = threadIdx.x; g <= a.NG; g += blockDim.x) {
        s.goff[g] = a.grp_off[g];
        if (g < a.NG) for (int gi = a.grp_off[g]; gi < a.grp_off[g + 1]; gi++) s.gof[gi] = g;
    }
    net_tabs_init(a.n, s.tb);
}

// The per-step input rows (MacroRoute, signals, inflow) of replica b at step t.  (Streaming them into shared memory one step
// ahead was measured: no change of the step latency at one replica, 20 % slower at 256 replicas -- the extra cp.async and
// barrier per step cost more than the L2 round trips they hide.)
template <typename T> struct StepRows { const int* rt; const T* sig; const T* inc; };
template <typename T> __device__ __forceinline__ StepRows<T> global_rows(const NetArgs<T>& n, int b, int t) {
    StepRows<T> r;
    r.rt = n.route ? n.route + (size_t)b * n.route_stride + (size_t)t * 2 * n.L : nullptr;
    r.sig = n.sig ? n.sig + ((size_t)b * n.T_steps + t) * n.L : nullptr;
    r.inc = n.incoming ? n.incoming + ((size_t)b * n.T_steps + t) * n.L : nullptr;
    return r;
}
// One simulation step of replica b: state `p` -> state `p ^ 1` of the double buffers.  All threads of the CTA call it.
// REC: keep the state between update and conversions (s.mid) and the conversion events (s.log).
template <typename T, bool REC>
__device__ __forceinline__ void hyb_step(const HybArgs<T>& a, const HybSm<T>& s, int b, int t, int p, const StepRows<T>& rows,
                                         unsigned& fl, int& ncol) {
    const NetArgs<T>& n = a.n;
    const AuxL& x = a.ax;
    const int NC = n.NC, L = n.L;
    const T* cr = s.st[p]; const T* cy = cr + NC; const T* cu = cy + NC; const T* ce = cu + NC;
    T* nr = s.st[p ^ 1]; T* ny = nr + NC; T* nu = ny + NC; T* ne = nu + NC;
    const T* ownc = s.own[p]; T* ownn = s.own[p ^ 1];
    const T* auxc = s.aux[p]; T* auxn = s.aux[p ^ 1];
    const int* rt = rows.rt; const T* sig_t = rows.sig; const T* inc_t = rows.inc;
    const T inv_dt = T(1) / n.dt;
    const bool blend = n.mode == 1 && n.soft && a.ML > 0;
    const T vlen = a.vlen;
    DHTS_PT_DECL
    // ---- phase S: waiting-list sources (ItscpRoadNetwork.setup_micro_boundary, _simulator.py:153-174).  A boundary micro
    // lane with room for a vehicle consumes ONE uniform draw -- lanes in id order within a step, so the draw a lane gets
    // depends on how many lanes before it had room -- and, if the draw is below the scheduled inflow and its waiting list
    // is not exhausted, receives a default vehicle at position 0 BEFORE the step (the row stored for step t does not hold
    // it; the adjoint's replay re-inserts it).
    if (a.src) {
        T* auxw = s.aux[p];
        for (int m = threadIdx.x; m < a.ML; m += blockDim.x) {
            int room = 0;
            if (a.src[m]) {
                const int cnt = (int)auxw[x.CNT + m];
                const T space = cnt > 0 ? auxw[x.P + m * a.cap + ((int)auxw[x.FRONT + m] + cnt - 1) % a.cap] - vlen * T(0.5)
                                        : a.lane_len[a.mic_lane[m]];                  // entering_free_space, _micro_lane.py:289-301
                room = space > vlen * T(0.5);
            }
            s.srcf[m] = room;
        }
        __syncthreads();
        for (int m = threadIdx.x; m < a.ML; m += blockDim.x) {
            int slot = -1;
            if (s.srcf[m]) {
                int idx = (int)auxw[x.DRAW];
                for (int q = 0; q < m; q++) idx += s.srcf[q];
                if (idx >= a.NRAND) fl |= FLAG_VEH_OVERFLOW;
                else {
                    const T u = a.rnd[(size_t)b * a.rnd_stride + idx];
                    const int ord = (int)auxw[x.NSP + m];
                    if (u < inc_t[a.mic_lane[m]] && ord < a.KS) {                     // the list still holds a vehicle and a route
                        const int f = (int)auxw[x.FRONT + m], cnt = (int)auxw[x.CNT + m];
                        if (cnt >= a.cap) fl |= FLAG_VEH_OVERFLOW;
                        else {
                            slot = (f + cnt) % a.cap;
                            const int o = m * a.cap + slot;
                            auxw[x.P + o] = T(0); auxw[x.V + o] = T(0); auxw[x.A + o] = vlen;       // default_micro_vehicle, micro_vehicle.py:30-72
                            auxw[x.RID + o] = (T)a.spawn_route[(size_t)b * a.spawn_stride + (size_t)m * a.KS + ord];
                            auxw[x.CUR + o] = T(0); auxw[x.PID + o] = T(0);
                            auxw[x.CNT + m] = (T)(cnt + 1); auxw[x.NSP + m] = (T)(ord + 1);
                        }
                    }
                }
            }
            s.srcs[m] = slot;
        }
        __syncthreads();
    }
    // ---- phase 0: the head vehicle's record of every micro lane, once per step (final_signal enters the running mean,
    // which visits the micro lanes in id order); the aux row is carried over wholesale, phase 1 writes what changes
    for (int m = (int)blockDim.x - 1 - (int)threadIdx.x; m < a.ML; m += blockDim.x) {
        const bool has = auxc[x.CNT + m] > T(0);
        T fin = T(0);
        if (has) { s.hrec[m] = head_rec(a, a.mic_lane[m], m, auxc, sig_t); fin = s.hrec[m].fin; }
        s.fsig[2 * m] = fin; s.fsig[2 * m + 1] = has ? T(1) : T(0);
    }
    for (int c = threadIdx.x; c < x.AUX; c += blockDim.x) auxn[c] = auxc[c];
    __syncthreads();
    DHTS_PT(0)      // phase S + 0
    // ---- phase 1: every lane takes its step from the state before the step (Jacobi).  Macro lanes in three sub-phases
    // (dhts_net_if.cuh): ghosts per (side, lane), fluxes per interface, update per cell.  The micro lanes -- one thread each,
    // taken from the far end of the CTA so that they do not queue behind the ghost threads -- run beside the ghosts.
    bool bad = false, bad_route = false;
    for (int q = threadIdx.x; q < 2 * L; q += blockDim.x) {
        const int side = q >= L, l = q - side * L;
        if (n.kind[l]) continue;
        const Side<T> sd = resolve_side(n, l, side, rt, cr, cu, ownc, sig_t, inc_t, bad_route);
        s.gh[2 * q] = sd.fr; s.gh[2 * q + 1] = sd.fu;
        const int os = n.own_slot[q];
        if (os >= 0) { ownn[2 * os] = sd.fr; ownn[2 * os + 1] = sd.fu; }
    }
    for (int m = (int)blockDim.x - 1 - (int)threadIdx.x; m < a.ML; m += blockDim.x) {
        {
            const int f = (int)auxc[x.FRONT + m], cnt = (int)auxc[x.CNT + m];
            T dp = a.head_dp0, dv = a.head_dv0, kc = T(0);
            if (cnt > 0) {
                const HeadRec<T>& h = s.hrec[m];
                dp = h.gdp; dv = h.gdv;
                if (n.mode == 1) {
                    if (n.soft) {
                        // signal_rms.update(final_signal) for every micro lane with vehicles, in id order; 32 / |mean|
                        T sum = auxc[x.RMS], num = auxc[x.RMS + 1];
                        for (int q = 0; q <= m; q++) { sum += s.fsig[2 * q] * s.fsig[2 * q + 1]; num += s.fsig[2 * q + 1]; }
                        kc = T(32) / t_abs(sum / num);
                        T ds;
                        const T fs = sigc(h.fin - T(0.5), kc, ds);
                        dp = h.gdp * fs + h.red_dp * (T(1) - fs);
                        dv = h.gdv * fs;
                    } else if (!(h.fin >= T(0.5))) { dp = h.red_dp; dv = T(0); }
                }
                T pl = T(0), vl = T(0);
                for (int j = 0; j < cnt; j++) {
                    const int o = m * a.cap + (f + j) % a.cap;
                    const T pj = auxc[x.P + o], vj = auxc[x.V + o];
                    const T dpr = j == 0 ? dp : t_abs(pl - pj) - vlen;             // (len + len) / 2
                    const T dvr = j == 0 ? dv : vj - vl;
                    const IdmEval<T> e = idm_eval(vj, s.par[(int)auxc[x.PID + o]], dpr, dvr, inv_dt);
                    if (e.col) ncol++;
                    auxn[x.P + o] = pj + n.dt * vj; auxn[x.V + o] = vj + n.dt * e.acc;
                    pl = pj; vl = vj;
                }
            }
            s.headd[2 * m] = dp; s.headd[2 * m + 1] = dv; s.kconst[m] = kc;
            if (m == a.ML - 1) {
                T sum = auxc[x.RMS], num = auxc[x.RMS + 1];
                if (blend) for (int q = 0; q < a.ML; q++) { sum += s.fsig[2 * q] * s.fsig[2 * q + 1]; num += s.fsig[2 * q + 1]; }
                auxn[x.RMS] = sum; auxn[x.RMS + 1] = num;
                T nd = auxc[x.DRAW];
                if (a.src) for (int q = 0; q < a.ML; q++) nd += (T)s.srcf[q];
                auxn[x.DRAW] = nd;
            }
        }
    }
    __syncthreads();
    DHTS_PT(1)      // ghosts + micro lanes
    bad |= net_fwd_flux<T>(n, s.tb, cr, cy, cu, ce, s.gh, s.flux);
    __syncthreads();
    DHTS_PT(2)      // fluxes
    for (int c = threadIdx.x; c < NC; c += blockDim.x) {      // _macro_lane.py:83-114; set_r_y refreshes u and u_eq, _arz.py:88-92
        const int l = s.tb.lane_of_cell[c];
        const int it = s.tb.if_off[l] + (c - n.cell_off[l]);
        const T cc = s.tb.cc[l];
        const T r = fma(s.flux[2 * it] - s.flux[2 * it + 2], cc, cr[c]);
        const T y = fma(s.flux[2 * it + 1] - s.flux[2 * it + 3], cc, cy[c]);
        nr[c] = r; ny[c] = y; nu[c] = compute_u(r, y, n.umax); ne[c] = u_eq(r, n.umax);
    }
    // ---- phase 2a: the table lookups of the conversion walk, one thread per group lane.  The walk itself is serial
    // (lanes of a group in id order, one thread per group); from global memory each of its links -- group -> lane ->
    // kind -> route -> capacitor -> micro index -- is an L2 round trip, which made it half of a step's latency
    for (int gi = threadIdx.x; gi < a.NGL; gi += blockDim.x) {
        int* w = s.walk + gi * 6;
        if (w[1] == 0) {      // macro lane: the micro lane the step's MacroRoute connects it to, and the capacitor that feeds it
            const int l = w[0];
            const int nx = rt ? rt[L + l] : -1;
            int k = -1, m2 = -1, nxm = -1;
            if (nx >= 0 && n.kind[nx] == 1) {
                for (int q = a.cap_off[l]; q < a.cap_off[l + 1]; q++) if (a.cap_lane[q] == nx) k = q;
                nxm = nx; m2 = a.mic_of[nx];
            }
            w[2] = nxm; w[3] = k; w[4] = m2;
            s.walkT[gi] = nx >= 0 ? a.lane_len[nx] : T(0);
        }
    }
    for (int g = threadIdx.x; g < a.NG; g += blockDim.x) s.gflag[g] = 0;
    if (bad) fl |= FLAG_CFL;
    if (bad_route) fl |= FLAG_ROUTE;
    __syncthreads();
    DHTS_PT(3)      // update + walk lookups
    if (REC) for (int c = threadIdx.x; c < 3 * NC; c += blockDim.x) s.mid[c] = nr[c];
    // ---- phase 2b: does a group have a conversion CANDIDATE at this step -- a head vehicle at the end of its lane, a
    // capacitor that has collected a vehicle?  Pops and spawns are rare (a few per lane and episode); without a candidate
    // the serial walk of the group would only add the step's flux to every capacitor, which its lanes do in parallel below.
    for (int gi = threadIdx.x; gi < a.NGL; gi += blockDim.x) {
        const int* w = s.walk + gi * 6;
        bool cand = false;
        if (w[1] == 0) {
            if (w[2] >= 0 && w[3] >= 0) {      // a spawn needs a collected vehicle AND room on the micro lane (exact unless a pop of this step
                const int m2 = w[4];           // empties that lane -- which flags the group by itself)
                const int n2 = (int)auxn[x.CNT + m2];
                const T space = n2 > 0 ? auxn[x.P + m2 * a.cap + ((int)auxn[x.FRONT + m2] + n2 - 1) % a.cap] - vlen * T(0.5) : s.walkT[gi];
                cand = (auxn[x.CAP + w[3]] + nr[w[5]] * nu[w[5]] * n.dt >= vlen) && (space >= vlen);
            }
        } else {
            const int m = w[2];
            if ((int)auxn[x.CNT + m] > 0) cand = auxn[x.P + m * a.cap + (int)auxn[x.FRONT + m]] >= s.walkT[gi];
        }
        if (cand) s.gflag[s.gof[gi]] = 1;
    }
    __syncthreads();
    DHTS_PT(4)      // candidates (+ mid copy)
    // ---- phase 2: conversions (road_network.py:113-173).  Groups without a candidate: one thread per group lane.
    for (int gi = threadIdx.x; gi < a.NGL; gi += blockDim.x) {
        if (s.gflag[s.gof[gi]]) continue;
        const int* w = s.walk + gi * 6;
        int ev = EV_NONE, e2 = 0;
        if (w[1] == 0 && w[2] >= 0 && w[3] >= 0) {                               // macro_to_micro without a spawn, conversion.py:15-73
            const int k = w[3], c = w[5];
            const T rl = nr[c], ul = nu[c];
            auxn[x.CAP + k] = auxn[x.CAP + k] + rl * ul * n.dt;
            ev = EV_CAP; e2 = k;
            if (REC) { s.log.et[gi * (3 + a.MAXT)] = rl; s.log.et[gi * (3 + a.MAXT) + 1] = ul; }
        }
        if (REC) { int* q = s.log.ei + gi * 4; q[0] = ev; q[1] = 0; q[2] = e2; q[3] = 0; }
    }
    // Groups with a candidate: one thread per group, lanes in id order.
    for (int g = threadIdx.x; g < a.NG; g += blockDim.x) {
        if (!s.gflag[g]) continue;
        for (int gi = s.goff[g]; gi < s.goff[g + 1]; gi++) {
            const int* w = s.walk + gi * 6;
            int ev = EV_NONE, e1 = 0, e2 = 0, e3 = 0;
            if (w[1] == 0) {                                                     // conversion_macro
                const int nx = w[2];
                if (nx >= 0) {
                    const int k = w[3];
                    if (k >= 0) {                                                 // macro_to_micro, conversion.py:15-73
                        const int c = w[5];
                        const T rl = nr[c], ul = nu[c];
                        const T flux = auxn[x.CAP + k] + rl * ul * n.dt;
                        const int m2 = w[4];
                        const int f2 = (int)auxn[x.FRONT + m2], n2 = (int)auxn[x.CNT + m2];
                        const T space = n2 > 0 ? auxn[x.P + m2 * a.cap + (f2 + n2 - 1) % a.cap] - vlen * T(0.5) : s.walkT[gi];
                        ev = EV_CAP; e2 = k;
                        if (REC) { s.log.et[gi * (3 + a.MAXT)] = rl; s.log.et[gi * (3 + a.MAXT) + 1] = ul; }
                        if (flux >= vlen && space >= vlen) {
                            const int ord = (int)auxn[x.NSP + m2];
                            if (n2 >= a.cap || ord >= a.KS) { fl |= FLAG_VEH_OVERFLOW; auxn[x.CAP + k] = flux; }
                            else {
                                const int sl_ = (f2 + n2) % a.cap, o = m2 * a.cap + sl_;
                                auxn[x.P + o] = T(0); auxn[x.V + o] = ul; auxn[x.A + o] = flux - (flux - vlen);
                                auxn[x.RID + o] = (T)a.spawn_route[(size_t)b * a.spawn_stride + (size_t)m2 * a.KS + ord];
                                auxn[x.CUR + o] = T(0); auxn[x.PID + o] = T(0);
                                auxn[x.CNT + m2] = (T)(n2 + 1); auxn[x.NSP + m2] = (T)(ord + 1);
                                auxn[x.CAP + k] = flux - vlen;                    // re-created detached, :65-68
                                ev = EV_SPAWN; e1 = m2; e3 = sl_;
                            }
                        } else auxn[x.CAP + k] = flux;
                    }
                }
            } else {                                                             // conversion_micro
                const int m = w[2];
                const int f = (int)auxn[x.FRONT + m], cnt = (int)auxn[x.CNT + m];
                if (cnt > 0) {
                    const int o = m * a.cap + f;
                    const T ph = auxn[x.P + o], vh = auxn[x.V + o], ah = auxn[x.A + o];
                    const int rid = (int)auxn[x.RID + o], cur = (int)auxn[x.CUR + o];
                    const T pid = auxn[x.PID + o];
                    const int nx = route_at(a, rid, cur + 1);
                    const T len = s.walkT[gi];
                    bool pop = false;
                    if (nx < 0) { pop = ph >= len; if (pop) ev = EV_DROP; }       // micro_to_none, :202-215
                    else if (n.kind[nx] == 0) {                                   // micro_to_macro, :75-171
                        pop = ph > len + T(1) * vlen;
                        if (pop) {
                            ev = EV_ABSORB; e2 = nx;
                            const int c0 = n.cell_off[nx], N = n.cell_off[nx + 1] - c0;
                            const T dxn = n.dx[nx], v_hd = ph - len, v_tl = v_hd - vlen;
                            int nt = 0;
                            for (int ci = 0; ci < N; ci++) {
                                T overlap, dodp;
                                if (!dep_cell(ci, dxn, vlen, v_hd, v_tl, overlap, dodp)) break;
                                T n_r = nr[c0 + ci] + (ah / vlen) * (overlap / dxn);
                                if (n_r > T(1) - T(1e-5)) n_r = T(1) - T(1e-5);
                                else if (n_r < T(1e-5)) n_r = T(1e-5);
                                nr[c0 + ci] = n_r; nu[c0 + ci] = vh; ny[c0 + ci] = n_r * (vh - u_eq(n_r, n.umax));
                                if (REC && nt < a.MAXT) s.log.et[gi * (3 + a.MAXT) + 3 + nt] = n_r;
                                nt++;
                            }
                            if (nt > a.MAXT) fl |= FLAG_VEH_OVERFLOW;
                            e3 = nt;
                        }
                    } else {                                                      // micro_to_micro, :174-200
                        pop = ph >= len;
                        if (pop) {
                            const int m2 = a.mic_of[nx];
                            const int f2 = (int)auxn[x.FRONT + m2], n2 = (int)auxn[x.CNT + m2];
                            if (n2 >= a.cap) { fl |= FLAG_VEH_OVERFLOW; pop = false; }
                            else {
                                const int s2 = (f2 + n2) % a.cap, o2 = m2 * a.cap + s2;
                                auxn[x.P + o2] = ph - len; auxn[x.V + o2] = vh; auxn[x.A + o2] = ah;
                                auxn[x.RID + o2] = (T)rid; auxn[x.CUR + o2] = (T)(cur + 1); auxn[x.PID + o2] = pid;
                                auxn[x.CNT + m2] = (T)(n2 + 1);
                                ev = EV_MOVE; e2 = m2; e3 = s2;
                            }
                        }
                    }
                    if (pop) {
                        auxn[x.FRONT + m] = (T)((f + 1) % a.cap); auxn[x.CNT + m] = (T)(cnt - 1);
                        e1 = f;
                        if (REC) { T* q = s.log.et + gi * (3 + a.MAXT); q[0] = ph; q[1] = vh; q[2] = ah; }
                    }
                }
            }
            if (REC) { int* q = s.log.ei + gi * 4; q[0] = ev; q[1] = e1; q[2] = e2; q[3] = e3; }
        }
    }
    __syncthreads();
    DHTS_PT(5)      // conversions
    DHTS_PT(6)      // (nothing: the cost of a marker itself)
#ifdef DHTS_PHASE_TIMING
    if (threadIdx.x == 0 && blockIdx.x == 0) { bool any = false; for (int g = 0; g < a.NG; g++) any |= s.gflag[g] != 0; if (any) atomicAdd(&g_phase_cycles[20], 1ull); }
#endif
}

template <typename T> __device__ __forceinline__ HybSm<T> hyb_carve(const HybArgs<T>& a, unsigned char* raw, bool adj, T*& extra) {
    HybSm<T> s;
    T* q = reinterpret_cast<T*>(raw);
    const int NC = a.n.NC;
    s.st[0] = q; q += 4 * NC; s.st[1] = q; q += 4 * NC;
    s.ab = s.st[1];
    if (adj) q += 4 * (size_t)(a.n.L - a.ML);      // 4 NI = 4 NC + 4 (macro lanes)
    s.own[0] = q; q += 2 * a.n.n_own; s.own[1] = q; q += 2 * a.n.n_own;
    s.aux[0] = q; q += a.ax.AUX; s.aux[1] = q; q += a.ax.AUX;
    s.fsig = q; q += 2 * a.ML; s.kconst = q; q += a.ML; s.headd = q; q += 2 * a.ML;
    s.mid = nullptr; s.log.ei = nullptr; s.log.et = nullptr;
    if (adj) {
        s.mid = q; q += 3 * NC;
        s.log.et = q; q += (size_t)a.NGL * (3 + a.MAXT);
    }
    {
        const int NI = NC + (a.n.L - a.ML);
        s.gh = q; q += 4 * (size_t)a.n.L;
        s.flux = q; q += 2 * (size_t)NI;
        unsigned char* pp = reinterpret_cast<unsigned char*>(q);
        s.tb = net_tabs_carve<T>(pp, a.n, NI);
        s.sd.s = nullptr;
        if (adj && a.prefetch) s.sd = side_tab_carve<T>(pp, a.n.L);
        q = reinterpret_cast<T*>(pp);
    }
    s.walk = reinterpret_cast<int*>(q); q += ((size_t)a.NGL * 6 * sizeof(int) + sizeof(T) - 1) / sizeof(T);
    s.goff = reinterpret_cast<int*>(q); q += ((size_t)(a.NG + 1) * sizeof(int) + sizeof(T) - 1) / sizeof(T);
    s.walkT = q; q += a.NGL;
    s.par = reinterpret_cast<IdmPar<T>*>(q); q += ((size_t)a.NP * sizeof(IdmPar<T>) + sizeof(T) - 1) / sizeof(T);
    s.srcf = reinterpret_cast<int*>(q); q += ((size_t)2 * a.ML * sizeof(int) + sizeof(T) - 1) / sizeof(T);
    s.srcs = s.srcf + a.ML;
    s.gflag = reinterpret_cast<int*>(q); q += ((size_t)(a.NG + a.NGL) * sizeof(int) + sizeof(T) - 1) / sizeof(T);
    s.gof = s.gflag + a.NG;
    s.hrec = reinterpret_cast<HeadRec<T>*>(q); q += ((size_t)a.ML * sizeof(HeadRec<T>) + sizeof(T) - 1) / sizeof(T);
    extra = q;
    return s;
}

// ------------------------------------------------------------------------------------------------ forward
// hist [T+1][R][4][NC], ownh [T+1][R][n_own][2], auxh [T+1][R][AUX]: state before step t and after the last step;
// headh [T][R][ML][2]: head deltas every micro lane used at step t.
template <typename T>
__global__ void __launch_bounds__(HYB_THREADS_MAX) hyb_rollout_fwd_kernel(HybArgs<T> a, const T* __restrict__ r0, const T* __restrict__ y0,
                                                                          const T* __restrict__ u0, const T* __restrict__ ueq0,
                                                                          const T* __restrict__ own0,
                                                                          const T* __restrict__ aux0, T* __restrict__ hist,
                                                                          T* __restrict__ ownh, T* __restrict__ auxh,
                                                                          T* __restrict__ headh, int* __restrict__ flags) {
    extern __shared__ __align__(16) unsigned char raw[];
    T* extra;
    const HybSm<T> s = hyb_carve(a, raw, false, extra);
    hyb_init(a, s);
    const int NC = a.n.NC, AUX = a.ax.AUX, n_own = a.n.n_own;
    unsigned fl = 0; int ncol = 0;
    for (int b = blockIdx.x; b < a.n.R; b += gridDim.x) {
        __syncthreads();
        for (int c = threadIdx.x; c < NC; c += blockDim.x) {
            const T r = r0[(size_t)b * NC + c];
            s.st[0][c] = r; s.st[0][NC + c] = y0[(size_t)b * NC + c]; s.st[0][2 * NC + c] = u0[(size_t)b * NC + c];
            // stored u_eq: as set_r_u leaves it (_arz.py:82-86) unless the caller hands over what the cells hold
            // (cleared cells carry u_max, cells rewritten by micro_to_macro a stale value: conversion.py:157-167)
            s.st[0][3 * NC + c] = ueq0 ? ueq0[(size_t)b * NC + c] : u_eq(r, a.n.umax);
        }
        for (int c = threadIdx.x; c < 2 * n_own; c += blockDim.x) s.own[0][c] = own0[(size_t)b * 2 * n_own + c];
        for (int c = threadIdx.x; c < AUX; c += blockDim.x) { s.aux[0][c] = aux0[(size_t)b * AUX + c]; s.aux[1][c] = T(0); }
        __syncthreads();
        int p = 0;
        for (int t = 0; t <= a.n.T_steps; t++) {
            {
                T* h = hist + ((size_t)t * a.n.R + b) * 4 * NC;
                for (int c = threadIdx.x; c < 4 * NC; c += blockDim.x) h[c] = s.st[p][c];
                T* oh = ownh + ((size_t)t * a.n.R + b) * 2 * n_own;
                for (int c = threadIdx.x; c < 2 * n_own; c += blockDim.x) oh[c] = s.own[p][c];
                T* ah = auxh + ((size_t)t * a.n.R + b) * AUX;
                for (int c = threadIdx.x; c < AUX; c += blockDim.x) ah[c] = s.aux[p][c];
            }
            if (t == a.n.T_steps) break;
            const StepRows<T> rows = global_rows(a.n, b, t);
            hyb_step<T, false>(a, s, b, t, p, rows, fl, ncol);
            if (headh) {
                T* hh = headh + ((size_t)t * a.n.R + b) * 2 * a.ML;
                for (int c = threadIdx.x; c < 2 * a.ML; c += blockDim.x) hh[c] = s.headd[c];
                __syncthreads();      // the next step's phase 1 rewrites s.headd (no barrier before it when phase 0 is skipped)
            }
            p ^= 1;
        }
    }
    if (ncol) { atomicOr(flags, FLAG_COLLISION); atomicAdd(flags + 1, ncol); }
    if (fl) atomicOr(flags, (int)fl);
}

// ------------------------------------------------------------------------------------------------ adjoint
// g_states [T][R][4][NC] optional: dLoss/d(r, y, u, -) of the state AFTER step t;  g_aux [T][R][AUX] optional:
// dLoss/d(p, v, a) of the vehicles AFTER step t, by slot (other entries of the row are ignored).
// outputs: g_r0, g_y0, g_u0 [R][NC]; g_own0 [R][n_own][2]; g_sig, g_inc [R][T][L]; g_aux0 [R][AUX] (p, v, a and
// capacitor entries; the rest zero).
// TMAX: largest CTA this instantiation is launched with: 192 threads (at least two CTAs per SM) or 512 (128 registers; the
// kernel needs 106 since the macro lanes run interface-parallel).  Was: networks of up to 192 lanes (ITSCP 3 x 3: 144) get the
// 170-register budget of two CTAs per SM; larger ones the full register file.
template <typename T, int TMAX>
__global__ void __launch_bounds__(TMAX, TMAX <= 192 ? 2 : 1) hyb_rollout_bwd_kernel(HybArgs<T> a, const T* __restrict__ hist, const T* __restrict__ ownh,
                                                                          const T* __restrict__ auxh, const T* __restrict__ g_states,
                                                                          const T* __restrict__ g_aux, T* __restrict__ g_r0,
                                                                          T* __restrict__ g_y0, T* __restrict__ g_u0,
                                                                          T* __restrict__ g_own0, T* __restrict__ g_sig,
                                                                          T* __restrict__ g_inc, T* __restrict__ g_aux0,
                                                                          int* __restrict__ flags) {
    extern __shared__ __align__(16) unsigned char raw[];
    T* q;
    HybSm<T> s = hyb_carve(a, raw, true, q);
    hyb_init(a, s);
    const NetArgs<T>& n = a.n;
    const AuxL& x = a.ax;
    const int NC = n.NC, L = n.L, AUX = x.AUX, n_own = n.n_own, ML = a.ML, cap = a.cap;
    T* G = q; q += 3 * NC;                     // adjoint of the cells (gr, gy, gu)
    T* GO = q; q += 2 * n_own;                 // adjoint of the own ghost records
    T* GV = q; q += 3 * ML * cap;              // adjoint of the vehicles (gp, gv, ga) x [ML][cap]
    T* GC = q; q += a.NCAP;                    // adjoint of the flux capacitors
    // prefetch targets: the stored rows of step t - 1 stream in with cp.async while step t is processed; the buffers
    // rotate with s.st[0] / s.own[0] / s.aux[0] (no copy)
    // (without a.prefetch -- networks whose buffers would not fit twice -- the rows are loaded at the top of their step)
    T* pre_st = s.st[0]; T* pre_own = s.own[0]; T* pre_aux = s.aux[0];
    if (a.prefetch) { pre_st = q; q += 4 * NC; pre_own = q; q += 2 * n_own; pre_aux = q; q += AUX; }
    T* pub = q; q += (size_t)L * 6;            // [L][2 sides][3] published (d green r, d green u, d signal)
    T* pubm = q; q += (size_t)ML * 5;          // [ML] (d signal prev, curr, next, d leader p, d leader v)
    int* pubi = reinterpret_cast<int*>(q);     // [ML][4] prev lane, next lane, leader micro index, leader slot
    s.log.ei = pubi + 4 * ML;                  // [NGL][4]
    const T inv_dt = T(1) / n.dt;
    const T vlen = a.vlen;
    bool nan = false;
    unsigned fl = 0; int ncol = 0;
    for (int b = blockIdx.x; b < n.R; b += gridDim.x) {
        __syncthreads();
        {   // terminal adjoint (masked to the vehicles that exist in the final state)
            const T* ah = auxh + ((size_t)n.T_steps * n.R + b) * AUX;
            for (int c = threadIdx.x; c < 3 * NC; c += blockDim.x)
                G[c] = (g_states && n.T_steps > 0) ? g_states[((size_t)(n.T_steps - 1) * n.R + b) * 4 * NC + c] : T(0);
            for (int c = threadIdx.x; c < 2 * n_own; c += blockDim.x) GO[c] = T(0);
            for (int c = threadIdx.x; c < a.NCAP; c += blockDim.x) GC[c] = T(0);
            for (int c = threadIdx.x; c < ML * cap; c += blockDim.x) {
                const int m = c / cap, sl_ = c - m * cap;
                const int f = (int)ah[x.FRONT + m], cnt = (int)ah[x.CNT + m];
                const bool occ = ((sl_ - f + cap) % cap) < cnt;
                const T* ga = (g_aux && n.T_steps > 0) ? g_aux + ((size_t)(n.T_steps - 1) * n.R + b) * AUX : nullptr;
                for (int k = 0; k < 3; k++) GV[k * ML * cap + c] = (occ && ga) ? ga[k * ML * cap + c] : T(0);
            }
        }
#define DHTS_HYB_PREFETCH(TT)                                                                                          \
        {                                                                                                              \
            const T* h_ = hist + ((size_t)(TT) * n.R + b) * 4 * NC;                                                    \
            for (int c = threadIdx.x; c < 4 * NC; c += blockDim.x) __pipeline_memcpy_async(pre_st + c, h_ + c, sizeof(T)); \
            const T* oh_ = ownh + ((size_t)(TT) * n.R + b) * 2 * n_own;                                                \
            for (int c = threadIdx.x; c < 2 * n_own; c += blockDim.x) __pipeline_memcpy_async(pre_own + c, oh_ + c, sizeof(T)); \
            const T* ah_ = auxh + ((size_t)(TT) * n.R + b) * AUX;                                                      \
            for (int c = threadIdx.x; c < AUX; c += blockDim.x) __pipeline_memcpy_async(pre_aux + c, ah_ + c, sizeof(T)); \
            __pipeline_commit();                                                                                       \
        }
        if (n.T_steps > 0 && a.prefetch) DHTS_HYB_PREFETCH(n.T_steps - 1)
        DHTS_PT_DECL
        for (int t = n.T_steps - 1; t >= 0; t--) {
            DHTS_PT(15)     // gathers of the previous step
            if (a.prefetch) {
                __pipeline_wait_prior(0);
                __syncthreads();          // rows of step t have landed; the previous step's last readers of s.st[0] are done
                { T* x_ = s.st[0]; s.st[0] = pre_st; pre_st = x_; x_ = s.own[0]; s.own[0] = pre_own; pre_own = x_;
                  x_ = s.aux[0]; s.aux[0] = pre_aux; pre_aux = x_; }
                if (t > 0) DHTS_HYB_PREFETCH(t - 1)
            } else {
                __syncthreads();          // the previous step's last readers of s.st[0] are done
                DHTS_HYB_PREFETCH(t)
                __pipeline_wait_prior(0);
                __syncthreads();
            }
#undef DHTS_HYB_PREFETCH
            DHTS_PT(10)     // rows landed
            const StepRows<T> rows = global_rows(n, b, t);
            hyb_step<T, true>(a, s, b, t, 0, rows, fl, ncol);    // replay: s.mid, s.log, s.kconst, s.aux[1]
            DHTS_PT(11)     // replay (its phases: 0-5)
            const T* cr = s.st[0]; const T* cy = cr + NC; const T* cu = cy + NC; const T* ce = cu + NC;
            const T* auxc = s.aux[0];
            const int* rt = rows.rt; const T* sig_t = rows.sig; const T* inc_t = rows.inc;
            // ---- R1: conversions reversed.  Groups without an event other than the capacitors' flux (s.gflag of the replay):
            // one thread per group lane; the others: one thread per group, last lane first
            for (int gi = threadIdx.x; gi < a.NGL; gi += blockDim.x) {
                if (s.gflag[s.gof[gi]]) continue;
                const int* e = s.log.ei + gi * 4;
                if (e[0] != EV_CAP) continue;
                const int k = e[2], c = s.walk[gi * 6 + 5];
                const T* et = s.log.et + gi * (3 + a.MAXT);
                const T gf = GC[k];
                G[c] += gf * et[1] * n.dt; G[2 * NC + c] += gf * et[0] * n.dt;
            }
            for (int g = threadIdx.x; g < a.NG; g += blockDim.x) {
                if (!s.gflag[g]) continue;
                for (int gi = s.goff[g + 1] - 1; gi >= s.goff[g]; gi--) {
                    const int* e = s.log.ei + gi * 4;
                    const int ev = e[0];
                    if (ev == EV_NONE) continue;
                    const int* w = s.walk + gi * 6;                    // lookups of the replayed step (hyb_step, phase 2a)
                    const int l = w[0];
                    const T* et = s.log.et + gi * (3 + a.MAXT);
                    if (ev == EV_CAP || ev == EV_SPAWN) {
                        const int k = e[2], c = w[5];
                        const T rl = et[0], ul = et[1];
                        T gf = GC[k], gvn = T(0);
                        if (ev == EV_SPAWN) {
                            const int o = e[1] * cap + e[3];
                            gf = GV[2 * ML * cap + o]; gvn = GV[ML * cap + o];
                            GV[o] = T(0); GV[ML * cap + o] = T(0); GV[2 * ML * cap + o] = T(0);
                        }
                        GC[k] = gf;
                        G[c] += gf * ul * n.dt; G[2 * NC + c] += gf * rl * n.dt + gvn;
                    } else if (ev == EV_DROP) {
                        const int o = w[2] * cap + e[1];
                        GV[o] = T(0); GV[ML * cap + o] = T(0); GV[2 * ML * cap + o] = T(0);
                    } else if (ev == EV_MOVE) {
                        const int o = w[2] * cap + e[1], o2 = e[2] * cap + e[3];
                        for (int k = 0; k < 3; k++) { GV[k * ML * cap + o] = GV[k * ML * cap + o2]; GV[k * ML * cap + o2] = T(0); }
                    } else if (ev == EV_ABSORB) {
                        const int o = w[2] * cap + e[1], nx = e[2], nt = e[3] < a.MAXT ? e[3] : a.MAXT;
                        const int c0 = n.cell_off[nx];
                        const T dxn = n.dx[nx], ph = et[0], spd = et[1], ah = et[2];
                        const T v_hd = ph - a.lane_len[l], v_tl = v_hd - vlen;
                        T gp = T(0), gv = T(0), ga = T(0);
                        for (int ci = 0; ci < nt; ci++) {
                            T overlap, dodp;
                            dep_cell(ci, dxn, vlen, v_hd, v_tl, overlap, dodp);
                            const T n_r = et[3 + ci];
                            const T gy = G[NC + c0 + ci];
                            const T gnr = G[c0 + ci] + gy * ((spd - u_eq(n_r, n.umax)) - n_r * u_eq_true_prime(n_r, n.umax));
                            gv += G[2 * NC + c0 + ci] + gy * n_r;
                            ga += gnr * (overlap / dxn) / vlen;
                            gp += gnr * (ah / vlen) * (dodp / dxn);
                            G[c0 + ci] = gnr; G[NC + c0 + ci] = T(0); G[2 * NC + c0 + ci] = T(0);   // old y, u discarded
                        }
                        GV[o] = gp; GV[ML * cap + o] = gv; GV[2 * ML * cap + o] = ga;
                    }
                }
            }
            __syncthreads();
            DHTS_PT(12)     // R1
            // ---- R2: every lane's operator reversed.  Macro lanes in three sub-phases (dhts_net_if.cuh); the micro lanes, one
            // thread each from the far end of the CTA, run beside the first one.
            bool dummy = false;
            T* g_inc_row = g_inc ? g_inc + ((size_t)b * n.T_steps + t) * L : nullptr;
            for (int c = threadIdx.x; c < NC; c += blockDim.x) {      // nu = compute_u(nr, ny): true derivative, at the state before conversions
                T dr, dy; du_dry(s.mid[c], s.mid[NC + c], n.umax, dr, dy);
                const T gu = G[2 * NC + c];
                G[c] += gu * dr; G[NC + c] += gu * dy;
            }
            for (int q = threadIdx.x; q < 2 * L; q += blockDim.x) {
                const int side = q >= L, l = q - side * L;
                if (n.kind[l]) continue;
                const Side<T> sv = resolve_side(n, l, side, rt, cr, cu, s.own[0], sig_t, inc_t, dummy);
                s.gh[2 * q] = sv.fr; s.gh[2 * q + 1] = sv.fu;
                if (s.sd.s) { s.sd.src[q] = sv.src; s.sd.sig_lane[q] = sv.sig_lane; s.sd.s[q] = sv.s; s.sd.gr[q] = sv.gr_; s.sd.gu[q] = sv.gu_; }
            }
            for (int m = (int)blockDim.x - 1 - (int)threadIdx.x; m < ML; m += blockDim.x) {
                const int l = a.mic_lane[m];
                {
                    const int f = (int)auxc[x.FRONT + m], cnt = (int)auxc[x.CNT + m];
                    T* pm = pubm + m * 5; int* pi = pubi + m * 4;
                    pm[0] = pm[1] = pm[2] = pm[3] = pm[4] = T(0); pi[0] = pi[1] = pi[2] = -1; pi[3] = 0;
                    for (int k = 0; k < 6; k++) pub[(size_t)l * 6 + k] = T(0);
                    if (g_inc) g_inc[((size_t)b * n.T_steps + t) * L + l] = T(0);
                    if (cnt > 0) {
                        const HeadRec<T>& h = s.hrec[m];                     // of the replayed step
                        const T dp = s.headd[2 * m], dv = s.headd[2 * m + 1];
                        T pl = T(0), vl = T(0), g_dp = T(0), g_dv = T(0);
                        int oprev = 0;
                        for (int j = 0; j < cnt; j++) {            // g_cur[j] = E_j^T g[j] + L_{j+1}^T g[j+1], dmicro_lane.py:271-297
                            const int o = m * cap + (f + j) % cap;
                            const T pj = auxc[x.P + o], vj = auxc[x.V + o];
                            const T dpr = j == 0 ? dp : t_abs(pl - pj) - vlen;
                            const T dvr = j == 0 ? dv : vj - vl;
                            const IdmPar<T>& ip = s.par[(int)auxc[x.PID + o]];
                            const IdmEval<T> e = idm_eval(vj, ip, dpr, dvr, inv_dt);
                            T E10, E11, L10, L11;
                            idm_jac(vj, ip, dpr, dvr, e, n.dt, E10, E11, L10, L11);
                            const T gp = GV[o], gv = GV[ML * cap + o];
                            T op = gp + E10 * gv, ov = n.dt * gp + E11 * gv;
                            const T sp = L10 * gv, sv = L11 * gv;
                            if (j == 0) { op += sp; ov += sv; g_dp = sp; g_dv = -sv; }     // ghost leader (p + dp, v - dv), dmicro_lane.py:144-151
                            else { GV[oprev] += sp; GV[ML * cap + oprev] += sv; }
                            GV[o] = op; GV[ML * cap + o] = ov;
                            nan |= t_isnan(op) || t_isnan(ov);
                            pl = pj; vl = vj; oprev = o;
                        }
                        // head deltas -> green / red / signal
                        const int oh = m * cap + h.hs;
                        T g_gdp = g_dp, g_gdv = g_dv, g_red = T(0);
                        if (n.mode == 1) {
                            if (n.soft) {
                                T ds;
                                const T fs = sigc(h.fin - T(0.5), s.kconst[m], ds);
                                g_gdp = g_dp * fs; g_gdv = g_dv * fs; g_red = g_dp * (T(1) - fs);
                                const T g_fs = g_dp * (h.gdp - h.red_dp) + g_dv * h.gdv;
                                const T g_fin = g_fs * ds;
                                const T S = h.a + h.b + h.c;
                                pm[0] = g_fin * h.a / S; pm[1] = g_fin * h.b / S; pm[2] = g_fin * h.c / S;
                                pi[0] = h.prev_lane; pi[1] = h.next_lane;
                                GV[oh] += g_fin * h.dfin;
                            } else if (!(h.fin >= T(0.5))) { g_gdp = T(0); g_gdv = T(0); g_red = g_dp; }
                        }
                        if (h.red_live) GV[oh] -= g_red;
                        if (h.lead_m >= 0) {
                            if (!h.lead_clamped) { GV[oh] -= g_gdp; pm[3] = g_gdp; }
                            GV[ML * cap + oh] += g_gdv; pm[4] = -g_gdv;
                            pi[2] = h.lead_m; pi[3] = h.lead_slot;
                        }
                    }
                }
            }
            __syncthreads();
            DHTS_PT(13)     // R2a: fold, ghosts, micro lanes
            net_adj_flux<T>(n, s.tb, cr, cy, cu, ce, s.gh, G, G + NC, s.ab);
            __syncthreads();
            DHTS_PT(14)     // R2b: interfaces
            for (int c = threadIdx.x; c < NC; c += blockDim.x) {
                const int l = s.tb.lane_of_cell[c];
                const int it = s.tb.if_off[l] + (c - n.cell_off[l]);      // interface on the cell's left; it + 1 on its right
                const T cc = s.tb.cc[l];
                const T nr_ = fma(cc, s.ab[4 * (it + 1)] + s.ab[4 * it + 2], G[c]);
                const T ny_ = fma(cc, s.ab[4 * (it + 1) + 1] + s.ab[4 * it + 3], G[NC + c]);
                nan |= t_isnan(nr_) || t_isnan(ny_);
                T nu_ = T(0);                                              // the stored speed of state t: filled by the gathers
                if (g_states && t > 0) {                                   // injected adjoint of state t (the state after step t - 1)
                    const T* gs_ = g_states + ((size_t)(t - 1) * n.R + b) * 4 * NC;
                    G[c] = nr_ + gs_[c]; G[NC + c] = ny_ + gs_[NC + c]; nu_ = gs_[2 * NC + c];
                } else { G[c] = nr_; G[NC + c] = ny_; }
                G[2 * NC + c] = nu_;
            }
            for (int q = threadIdx.x; q < 2 * L; q += blockDim.x) {
                const int side = q >= L, l = q - side * L;
                if (n.kind[l]) continue;
                const T cc = s.tb.cc[l];
                const T* o = s.ab + 4 * (size_t)(side == 0 ? s.tb.if_off[l] : s.tb.if_off[l + 1] - 1);
                const T g_r = cc * (side == 0 ? o[0] : o[2]), g_y = cc * (side == 0 ? o[1] : o[3]);
                if (s.sd.s)
                    net_adj_side<T>(n, s.gh, l, side, s.sd.src[q], s.sd.sig_lane[q], s.sd.s[q], s.sd.gr[q], s.sd.gu[q], g_r, g_y, GO, pub,
                                    g_inc_row);
                else {      // lean shared-memory mode: the side record is resolved again
                    const Side<T> sv = resolve_side(n, l, side, rt, cr, cu, s.own[0], sig_t, inc_t, dummy);
                    net_adj_side<T>(n, s.gh, l, side, sv.src, sv.sig_lane, sv.s, sv.gr_, sv.gu_, g_r, g_y, GO, pub, g_inc_row);
                }
            }
            __syncthreads();
            DHTS_PT(16)     // R2c: cells, sides
            // ---- R3: gathers (edge cells and signals the neighbours used, leaders of other lanes' heads), injected vehicle adjoints.
            // A micro lane's head blends the signals of its own lane and of the lanes before / after it on its route -- neighbours
            // in the lane graph -- so every lane collects those terms while it walks its adjacency lists.
            for (int l = threadIdx.x; l < L; l += blockDim.x) {
                const bool mac = n.kind[l] == 0;
                const int c0 = n.cell_off[l], N = n.cell_off[l + 1] - c0;
                T gsig = mac ? pub[((size_t)l * 2 + 1) * 3 + 2] : pubm[a.mic_of[l] * 5 + 1];
                for (int e = n.adj_off[(L + 1) + l]; e < n.adj_off[(L + 1) + l + 1]; e++) {      // successors
                    const int nn = n.adj[e];
                    if (n.kind[nn]) {                      // its head came from lane l: d (signal of the previous lane)
                        const int m2 = a.mic_of[nn];
                        if (pubi[m2 * 4] == l) gsig += pubm[m2 * 5];
                        continue;
                    }
                    if (!mac) continue;
                    const int cnt = n.nadj[nn];
                    const int sel = rt ? rt[nn] : -1;
                    const int srcn = cnt == 1 ? n.one_adj[nn] : (cnt > 1 ? sel : -1);
                    const T* pb = pub + ((size_t)nn * 2 + 0) * 3;
                    if (srcn == l) { G[c0 + N - 1] += pb[0]; G[2 * NC + c0 + N - 1] += pb[1]; }
                    if (n.mode == 1 && sel == l) gsig += pb[2];
                }
                for (int e = n.adj_off[l]; e < n.adj_off[l + 1]; e++) {                          // predecessors
                    const int pl = n.adj[e];
                    if (n.kind[pl]) {                      // its head goes on to lane l: d (signal of the next lane)
                        const int m2 = a.mic_of[pl];
                        if (pubi[m2 * 4 + 1] == l) gsig += pubm[m2 * 5 + 2];
                        continue;
                    }
                    if (!mac) continue;
                    const int cnt = n.nadj[L + pl];
                    const int sel = rt ? rt[L + pl] : -1;
                    const int srcp = cnt == 1 ? n.one_adj[L + pl] : (cnt > 1 ? sel : -1);
                    const T* pb = pub + ((size_t)pl * 2 + 1) * 3;
                    if (srcp == l) { G[c0] += pb[0]; G[2 * NC + c0] += pb[1]; }
                }
                if (!mac) {
                    const int m = a.mic_of[l];
                    for (int m2 = 0; m2 < ML; m2++) {      // heads whose leader is a vehicle of this lane (possibly lanes ahead of them)
                        const int* pi = pubi + m2 * 4;
                        if (pi[2] == m) { GV[m * cap + pi[3]] += pubm[m2 * 5 + 3]; GV[ML * cap + m * cap + pi[3]] += pubm[m2 * 5 + 4]; }
                    }
                    if (g_aux && t > 0) {
                        const T* ga = g_aux + ((size_t)(t - 1) * n.R + b) * AUX;
                        const int f = (int)auxc[x.FRONT + m], cnt = (int)auxc[x.CNT + m];
                        for (int j = 0; j < cnt; j++) {
                            const int o = m * cap + (f + j) % cap;
                            for (int k = 0; k < 3; k++) GV[k * ML * cap + o] += ga[k * ML * cap + o];
                        }
                    }
                    if (a.src && s.srcs[m] >= 0) {      // the vehicle that entered from the waiting list at step t: a constant
                        const int o = m * cap + s.srcs[m];
                        GV[o] = T(0); GV[ML * cap + o] = T(0); GV[2 * ML * cap + o] = T(0);
                    }
                }
                if (g_sig) g_sig[((size_t)b * n.T_steps + t) * L + l] = gsig;
                nan |= t_isnan(gsig);
            }
        }
        __syncthreads();
        for (int c = threadIdx.x; c < NC; c += blockDim.x) {
            g_r0[(size_t)b * NC + c] = G[c]; g_y0[(size_t)b * NC + c] = G[NC + c]; g_u0[(size_t)b * NC + c] = G[2 * NC + c];
            nan |= t_isnan(G[c]) || t_isnan(G[NC + c]) || t_isnan(G[2 * NC + c]);
        }
        if (g_own0)
            for (int c = threadIdx.x; c < 2 * n_own; c += blockDim.x) g_own0[(size_t)b * 2 * n_own + c] = GO[c];
        if (g_aux0) {
            T* go = g_aux0 + (size_t)b * AUX;
            for (int c = threadIdx.x; c < AUX; c += blockDim.x) {
                T v = T(0);
                if (c < 3 * ML * cap) v = GV[c];
                else if (c >= x.CAP && c < x.CAP + a.NCAP) v = GC[c - x.CAP];
                go[c] = v;
            }
        }
    }
    if (nan) atomicOr(flags, FLAG_NAN_GRAD);
}

// ------------------------------------------------------------------------------------------------ host side
// Few replicas (a CTA's step time is what counts): one thread per interface of the macro lanes, and at least one per (side,
// lane) plus one per micro lane.  Many replicas (several CTAs per SM hide each other's barriers): half as many, looping.
template <typename T> static int hyb_threads(const HybArgs<T>& a) {
    const int NI = a.n.NC + (a.n.L - a.ML), sides = 2 * a.n.L + a.ML;
    int w = NI > sides ? NI : sides;
    if (a.n.R > sm_count()) w = (w + 1) / 2;
    int t = (w + 31) / 32 * 32;
    return t > HYB_THREADS_MAX ? HYB_THREADS_MAX : (t < 32 ? 32 : t);
}

template <typename T> static size_t hyb_smem(const HybArgs<T>& a, bool adj) {
    const size_t NC = a.n.NC, L = a.n.L, ML = a.ML;
    size_t el = 8 * NC + 4 * (size_t)a.n.n_own + 2 * (size_t)a.ax.AUX + 5 * ML;
    size_t bytes = 0;
    if (adj) {
        el += 3 * NC + (size_t)a.NGL * (3 + a.MAXT);                       // mid, log.et
        el += 3 * NC + 2 * (size_t)a.n.n_own + 3 * ML * a.cap + a.NCAP + 6 * L + 5 * ML;
        if (a.prefetch) el += 4 * NC + 2 * (size_t)a.n.n_own + (size_t)a.ax.AUX;   // prefetch targets
        bytes += sizeof(int) * (4 * ML + 4 * (size_t)a.NGL);
    }
    {
        const size_t NI = NC + (L - ML);
        el += 4 * L + 2 * NI + (adj ? 4 * (L - ML) : 0);                    // gh, flux, tail of (A^T w, B^T w) behind st[1]
        bytes += net_tabs_bytes<T>((int)L, (int)NC, (int)NI) + (adj && a.prefetch ? side_tab_bytes<T>((int)L) : 0);
    }
    bytes += sizeof(int) * 6 * (size_t)a.NGL + sizeof(T);                  // walk
    bytes += sizeof(int) * (size_t)(a.NG + 1) + sizeof(T); el += a.NGL;   // goff, walkT
    bytes += sizeof(IdmPar<T>) * (size_t)a.NP + sizeof(T);                // par
    bytes += sizeof(int) * 2 * ML + sizeof(T);                            // srcf, srcs
    bytes += sizeof(int) * (size_t)(a.NG + a.NGL) + sizeof(T);            // gflag, gof
    bytes += sizeof(HeadRec<T>) * ML + sizeof(T);                         // hrec
    return sizeof(T) * el + bytes + 32;
}

template <typename T> static int hyb_check(const HybArgs<T>& a) {
    const NetArgs<T>& n = a.n;
    if (n.L < 1 || n.NC < 0 || n.n_own < 0 || n.T_steps < 0 || n.R < 0 || !n.cell_off || !n.dx || !n.nadj || !n.one_adj || !n.adj_off ||
        !n.own_slot || !n.kind || !a.mic_of || !a.cap_off || !a.grp_off || !a.lane_len)
        return DHTS_ERR_INVALID;
    if (a.ML < 0 || a.cap < 1 || a.NCAP < 0 || a.NG < 0 || a.NGL < 0 || a.RLEN < 1 || a.KS < 0 || a.MAXT < 1) return DHTS_ERR_INVALID;
    if (a.ML > 0 && (!a.mic_lane || !a.routes || (a.NCAP > 0 && (!a.cap_lane || !a.spawn_route || !n.route)))) return DHTS_ERR_INVALID;
    if (n.mode == 1 && (!n.sig || !n.incoming)) return DHTS_ERR_INVALID;
    if (n.mode != 0 && n.mode != 1) return DHTS_ERR_INVALID;
    if (a.NP < 1 || !a.par_tab || !(a.vlen > T(0))) return DHTS_ERR_INVALID;
    if (a.src && (n.mode != 1 || !a.rnd || a.NRAND < 0 || (a.KS > 0 && !a.spawn_route))) return DHTS_ERR_INVALID;
    return DHTS_OK;
}

template <typename T>
static HybArgs<T> hyb_args(const dhts_hyb_topology* tp, const T* dx, const T* lane_len, const int* route, int route_per_replica,
                           const int* spawn_route, int spawn_per_replica, int KS, const T* sig, const T* incoming,
                           const T* veh_par, int n_par, T veh_len, const T* src_rand, int n_rand, int rand_per_replica,
                           T umax, T dt, int steps, int R, int mode, int soft) {
    HybArgs<T> a;
    NetArgs<T>& n = a.n;
    n.L = tp->L; n.NC = tp->NC; n.n_own = tp->n_own; n.T_steps = steps; n.R = R; n.mode = mode; n.soft = soft;
    n.cell_off = tp->cell_off; n.dx = dx; n.nadj = tp->nadj; n.one_adj = tp->one_adj; n.adj_off = tp->adj_off; n.adj = tp->adj;
    n.own_slot = tp->own_slot; n.route = route; n.route_stride = route_per_replica ? (long long)steps * 2 * tp->L : 0;
    n.umax = umax; n.dt = dt; n.veh_len = veh_len; n.static_speed = T(0);
    n.sig = sig; n.incoming = incoming; n.qk = nullptr; n.kind = tp->kind;
    a.ML = tp->ML; a.cap = tp->cap; a.NCAP = tp->NCAP; a.NGL = tp->NGL; a.NG = tp->NG; a.RLEN = tp->RLEN; a.NR = tp->NR;
    a.KS = KS; a.MAXT = tp->MAXT;
    a.mic_of = tp->mic_of; a.mic_lane = tp->mic_lane; a.cap_off = tp->cap_off; a.cap_lane = tp->cap_lane;
    a.grp_off = tp->grp_off; a.grp_lane = tp->grp_lane; a.routes = tp->routes; a.lane_len = lane_len;
    a.spawn_route = spawn_route; a.spawn_stride = spawn_per_replica ? (long long)tp->ML * KS : 0;
    a.par_tab = veh_par; a.NP = n_par; a.vlen = veh_len;
    a.prefetch = 1;
    a.src = tp->src; a.rnd = src_rand; a.NRAND = n_rand; a.rnd_stride = rand_per_replica ? (long long)n_rand : 0;
    a.head_dp0 = T(1000); a.head_dv0 = T(0);
    a.ax = aux_layout(tp->ML, tp->cap, tp->NCAP);
    return a;
}

}  // namespace dhts

#define DHTS_HYB_API(SUF, T)                                                                                           \
    DHTS_EXPORT int dhts_hyb_rollout_fwd_##SUF(const dhts_hyb_topology* topo, const T* dx, const T* lane_len,          \
                                               const int* route, int route_per_replica, const int* spawn_route,        \
                                               int spawn_per_replica, int KS, const T* sig, const T* incoming,         \
                                               const T* veh_par, int n_par, T veh_len, const T* src_rand, int n_rand,  \
                                               int rand_per_replica, T umax, T dt, int steps, int R, int mode,         \
                                               int soft,                                                               \
                                               const T* r0, const T* y0, const T* u0, const T* ueq0, const T* own0,    \
                                               const T* aux0, T* hist, T* own_hist, T* aux_hist, T* head_hist,         \
                                               int* flags, void* stream) {                                             \
        if (!topo || !veh_par || !aux0 || !aux_hist || !flags) return DHTS_ERR_INVALID;                                \
        if (topo->NC > 0 && (!r0 || !y0 || !u0 || !hist)) return DHTS_ERR_INVALID;                                     \
        dhts::HybArgs<T> a = dhts::hyb_args<T>(topo, dx, lane_len, route, route_per_replica, spawn_route,              \
                                               spawn_per_replica, KS, sig, incoming, veh_par, n_par, veh_len,          \
                                               src_rand, n_rand, rand_per_replica, umax, dt, steps, R, mode, soft);   \
        int rc = dhts::hyb_check(a);                                                                                   \
        if (rc) return rc;                                                                                             \
        if (a.n.n_own > 0 && (!own0 || !own_hist)) return DHTS_ERR_INVALID;                                            \
        if (R == 0) return DHTS_OK;                                                                                    \
        const int threads = dhts::hyb_threads(a);                                                                  \
        const size_t smem = dhts::hyb_smem<T>(a, false);                                                               \
        int grid = 1;                                                                                                  \
        rc = dhts::persistent_grid(dhts::hyb_rollout_fwd_kernel<T>, threads, smem, R, &grid);                          \
        if (rc) return rc;                                                                                             \
        dhts::hyb_rollout_fwd_kernel<T><<<grid, threads, smem, (cudaStream_t)stream>>>(a, r0, y0, u0, ueq0, own0,      \
                                                                                         aux0, hist, own_hist,        \
                                                                                         aux_hist, head_hist, flags);  \
        return dhts::launch_status();                                                                                  \
    }                                                                                                                  \
    DHTS_EXPORT int dhts_hyb_rollout_bwd_##SUF(const dhts_hyb_topology* topo, const T* dx, const T* lane_len,          \
                                               const int* route, int route_per_replica, const int* spawn_route,        \
                                               int spawn_per_replica, int KS, const T* sig, const T* incoming,         \
                                               const T* veh_par, int n_par, T veh_len, const T* src_rand, int n_rand,  \
                                               int rand_per_replica, T umax, T dt, int steps, int R, int mode,         \
                                               int soft,                                                               \
                                               const T* hist, const T* own_hist, const T* aux_hist,                    \
                                               const T* g_states, const T* g_aux, T* g_r0, T* g_y0, T* g_u0,           \
                                               T* g_own0, T* g_sig, T* g_incoming, T* g_aux0, int* flags,              \
                                               void* stream) {                                                         \
        if (!topo || !veh_par || !aux_hist || !flags) return DHTS_ERR_INVALID;                                         \
        if (topo->NC > 0 && (!hist || !g_r0 || !g_y0 || !g_u0)) return DHTS_ERR_INVALID;                               \
        dhts::HybArgs<T> a = dhts::hyb_args<T>(topo, dx, lane_len, route, route_per_replica, spawn_route,              \
                                               spawn_per_replica, KS, sig, incoming, veh_par, n_par, veh_len,          \
                                               src_rand, n_rand, rand_per_replica, umax, dt, steps, R, mode, soft);   \
        int rc = dhts::hyb_check(a);                                                                                   \
        if (rc) return rc;                                                                                             \
        if (a.n.n_own > 0 && !own_hist) return DHTS_ERR_INVALID;                                                       \
        if (R == 0) return DHTS_OK;                                                                                    \
        const int threads = dhts::hyb_threads(a);                                                                  \
        size_t smem = dhts::hyb_smem<T>(a, true);                                                                      \
        if (smem > 227 * 1024) { a.prefetch = 0; smem = dhts::hyb_smem<T>(a, true); }                                  \
        int grid = 1;                                                                                                  \
        if (threads <= 192) {                                                                                          \
            rc = dhts::persistent_grid(dhts::hyb_rollout_bwd_kernel<T, 192>, threads, smem, R, &grid);                 \
            if (rc) return rc;                                                                                         \
            dhts::hyb_rollout_bwd_kernel<T, 192><<<grid, threads, smem, (cudaStream_t)stream>>>(                       \
                a, hist, own_hist, aux_hist, g_states, g_aux, g_r0, g_y0, g_u0, g_own0, g_sig, g_incoming, g_aux0,     \
                flags);                                                                                                \
        } else {                                                                                                       \
            rc = dhts::persistent_grid(dhts::hyb_rollout_bwd_kernel<T, dhts::HYB_THREADS_MAX>, threads, smem, R, &grid); \
            if (rc) return rc;                                                                                         \
            dhts::hyb_rollout_bwd_kernel<T, dhts::HYB_THREADS_MAX><<<grid, threads, smem, (cudaStream_t)stream>>>(     \
                a, hist, own_hist, aux_hist, g_states, g_aux, g_r0, g_y0, g_u0, g_own0, g_sig, g_incoming, g_aux0,     \
                flags);                                                                                                \
        }                                                                                                              \
        return dhts::launch_status();                                                                                  \
    }

DHTS_HYB_API(f64, double)
DHTS_HYB_API(f32, float)

DHTS_EXPORT int dhts_hyb_aux_size(const dhts_hyb_topology* topo) {
    if (!topo) return -1;
    return dhts::aux_layout(topo->ML, topo->cap, topo->NCAP).AUX;
}
