// IDM microscopic car-following kernels for sm_100a (K3 forward, K4 adjoint).
//
// Behaviour restated from the reference (file:line relative to its checkout):
//   model/micro/_idm.py:5-51            acceleration with the two clips
//   road/lane/_micro_lane.py:131-214    leader lookup, collision handling, Euler step
//   model/micro/didm.py:12-102          ego / leader 2x2 Jacobians
//   road/lane/dmicro_lane.py:87-153, 271-297   band, ghost leader, VJP
// Vehicles are stored lane by lane (CSR offsets), index 0 = tail; the leader of
// vehicle i is i+1; the head of a lane follows a ghost leader (head_dp, head_dv).
//
//  * idm_step_{fwd,bwd}_kernel: one step, one thread per vehicle, leader state
//    taken from the neighbouring lane of the warp by shuffle.
//  * idm_rollout_{fwd,bwd}_kernel: T fused steps, one warp per lane, VPT vehicles
//    per thread in registers, leaders and follower adjoints exchanged with warp
//    shuffles only (no block barrier in the time loop); checkpoints every K
//    steps, segment recompute with a per-thread stash.
#include "dhts_idm.cuh"
#include "dhts_api.h"

namespace dhts {

// ------------------------------------------------------------------ single step

constexpr int IDM_BLOCK = 256;

template <typename T>
__global__ void __launch_bounds__(IDM_BLOCK)
idm_step_fwd_kernel(const T* __restrict__ p, const T* __restrict__ v, const T* __restrict__ params,
                    const int* __restrict__ lane_off, const int* __restrict__ veh_lane, const T* __restrict__ head,
                    T dt, int V, T* __restrict__ np_, T* __restrict__ nv_, int* __restrict__ vflags,
                    int* __restrict__ flags) {
    const int i = blockIdx.x * IDM_BLOCK + threadIdx.x;
    const bool valid = i < V;
    const int ii = valid ? i : V - 1;
    const unsigned lane = threadIdx.x & 31;
    T pi = p[ii], vi = v[ii];
    IdmPar<T> k = load_par(params, (size_t)V, (size_t)ii);
    // leader state from the next lane of the warp; the warp's last lane reads global
    T lp = __shfl_down_sync(0xffffffffu, pi, 1), lv = __shfl_down_sync(0xffffffffu, vi, 1),
      ll = __shfl_down_sync(0xffffffffu, k.len, 1);
    if (lane == 31 && ii + 1 < V) { lp = p[ii + 1]; lv = v[ii + 1]; ll = params[5 * (size_t)V + ii + 1]; }
    const int l = veh_lane[ii];
    const bool is_head = (ii + 1 == lane_off[l + 1]);
    T dp, dv;
    if (is_head) { dp = head[2 * l]; dv = head[2 * l + 1]; }
    else { dp = t_abs(lp - pi) - (ll + k.len) * T(0.5); dv = vi - lv; }
    IdmEval<T> e = idm_eval(vi, k, dp, dv, T(1) / dt);
    if (valid) {
        np_[i] = pi + dt * vi;
        nv_[i] = vi + dt * e.acc;
        if (vflags) vflags[i] = (int)e.clip_acc | ((int)e.clip_s << 1) | ((int)e.col << 2);
        if (e.col) { atomicOr(flags, FLAG_COLLISION); atomicAdd(flags + 1, 1); }
    }
}

// PAR: also the adjoint of the vehicle parameters, g_params [6][V] (idm_par_vjp); a separate instantiation, so that the
// state adjoint alone stays as it was.
template <typename T, bool PAR>
__global__ void __launch_bounds__(IDM_BLOCK)
idm_step_bwd_kernel(const T* __restrict__ p, const T* __restrict__ v, const T* __restrict__ params,
                    const int* __restrict__ lane_off, const int* __restrict__ veh_lane, const T* __restrict__ head,
                    T dt, int V, const T* __restrict__ g_np, const T* __restrict__ g_nv, T* __restrict__ g_p,
                    T* __restrict__ g_v, T* __restrict__ g_head, int* __restrict__ flags, T* __restrict__ g_params) {
    __shared__ T s_cp[IDM_BLOCK], s_cv[IDM_BLOCK];
    const int i = blockIdx.x * IDM_BLOCK + threadIdx.x;
    const bool valid = i < V;
    const T inv_dt = T(1) / dt;
    IdmParAdj<T> pa = {T(0), T(0), T(0), T(0), T(0), T(0)};
    IdmPar<T> pk;
    // evaluate vehicle j against its leader; returns adjoint pieces (and, for the thread's own vehicle, its parameter ones)
    auto eval = [&](int j, T& E10, T& E11, T& L10, T& L11, bool& is_head, int& l, bool own) {
        T pj = p[j], vj = v[j];
        IdmPar<T> k = load_par(params, (size_t)V, (size_t)j);
        l = veh_lane[j];
        is_head = (j + 1 == lane_off[l + 1]);
        T dp, dv;
        if (is_head) { dp = head[2 * l]; dv = head[2 * l + 1]; }
        else { dp = t_abs(p[j + 1] - pj) - (params[5 * (size_t)V + j + 1] + k.len) * T(0.5); dv = vj - v[j + 1]; }
        IdmEval<T> e = idm_eval(vj, k, dp, dv, inv_dt);
        idm_jac(vj, k, dp, dv, e, dt, E10, E11, L10, L11);
        if constexpr (PAR) if (own) { pk = k; idm_par_vjp(vj, k, dp, dv, e, g_nv[j], pa); }
    };
    T gp = T(0), gv = T(0), cp = T(0), cv = T(0);
    bool is_head = false; int l = 0;
    T E10 = 0, E11 = 0, L10, L11;
    if (valid) {
        eval(i, E10, E11, L10, L11, is_head, l, true);
        gp = g_np[i]; gv = g_nv[i];
        cp = L10 * gv; cv = L11 * gv;     // L^T g: what this vehicle sends to its leader
        if constexpr (PAR) if (!is_head) pa.len = T(-0.5) * cp;
    }
    s_cp[threadIdx.x] = cp; s_cv[threadIdx.x] = cv;
    __syncthreads();
    if (!valid) return;
    T op = gp + E10 * gv;                 // E^T g
    T ov = dt * gp + E11 * gv;
    const bool is_tail = (i == lane_off[l]);
    if (!is_tail) {                       // contribution of the follower i-1
        if (threadIdx.x > 0) {
            op += s_cp[threadIdx.x - 1]; ov += s_cv[threadIdx.x - 1];
            if constexpr (PAR) pa.len += T(-0.5) * s_cp[threadIdx.x - 1];
        } else {
            T e10, e11, l10, l11; bool h; int ll;
            eval(i - 1, e10, e11, l10, l11, h, ll, false);
            T gvf = g_nv[i - 1];
            op += l10 * gvf; ov += l11 * gvf;
            if constexpr (PAR) pa.len += (T(-0.5) * l10) * gvf;     // not l10 * gvf: that product must stay fused into op
        }
    }
    if (is_head) {                        // ghost leader = (p_head + dp, v_head - dv), dmicro_lane.py:144-151
        op += cp; ov += cv;
        if (g_head) { g_head[2 * l] = cp; g_head[2 * l + 1] = -cv; }
    }
    g_p[i] = op; g_v[i] = ov;
    bool nan = t_isnan(op) || t_isnan(ov);
    if constexpr (PAR) {
        T g[6];
        idm_par_grad(pa, pk, params[(size_t)V + i], dt, g);
#pragma unroll
        for (int r = 0; r < 6; r++) { g_params[(size_t)r * V + i] = g[r]; nan |= t_isnan(g[r]); }
    }
    if (nan) atomicOr(flags, FLAG_NAN_GRAD);
}

// lanes with no vehicle get a zero head gradient
template <typename T>
__global__ void idm_zero_empty_head_kernel(const int* __restrict__ lane_off, int L, T* __restrict__ g_head) {
    int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l < L && lane_off[l + 1] == lane_off[l]) { g_head[2 * l] = T(0); g_head[2 * l + 1] = T(0); }
}

__global__ void csr_expand_kernel(const int* __restrict__ lane_off, int L, int* __restrict__ veh_lane) {
    // one warp per lane; writes the lane id of each of its vehicles
    int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, k = threadIdx.x & 31;
    int nw = (gridDim.x * blockDim.x) >> 5;
    for (int l = w; l < L; l += nw)
        for (int i = lane_off[l] + k; i < lane_off[l + 1]; i += 32) veh_lane[i] = l;
}

// ------------------------------------------------------------------ fused rollouts, one warp per lane

constexpr int IDM_KMAX = 32;          // max checkpoint interval of the fused adjoint (stash depth)
constexpr int IDM_ROLL_BLOCK = 128;

template <typename T, int VPT> struct WarpLane {
    T p[VPT], v[VPT];
    IdmPar<T> k[VPT];
    T lead_len[VPT];
    bool valid[VPT], head[VPT];
};

template <typename T, int VPT>
__device__ __forceinline__ void lane_load(WarpLane<T, VPT>& w, const T* __restrict__ p, const T* __restrict__ v,
                                          const T* __restrict__ params, int V, int o, int n, unsigned lane) {
#pragma unroll
    for (int m = 0; m < VPT; m++) {
        int e = m * 32 + (int)lane;
        w.valid[m] = e < n; w.head[m] = (e == n - 1);
        size_t i = (size_t)o + (w.valid[m] ? e : 0);
        if (n > 0) { w.p[m] = p[i]; w.v[m] = v[i]; w.k[m] = load_par(params, (size_t)V, i); }
    }
#pragma unroll
    for (int m = 0; m < VPT; m++) {
        T up = __shfl_down_sync(0xffffffffu, w.k[m].len, 1);
        T ed = __shfl_sync(0xffffffffu, w.k[m + 1 < VPT ? m + 1 : m].len, 0);
        w.lead_len[m] = (lane == 31) ? ed : up;
    }
}

// leader (p, v) of every slot from the OLD state (Jacobi update)
template <typename T, int VPT>
__device__ __forceinline__ void lane_deltas(const WarpLane<T, VPT>& w, T head_dp, T head_dv, unsigned lane, T* dp,
                                            T* dv) {
#pragma unroll
    for (int m = 0; m < VPT; m++) {
        // one rotation per value: lane i takes lane i+1's entry of this slot; lane 31 takes lane 0's entry of the NEXT slot,
        // which lane 0 sends instead of its own (nobody reads lane 0's own entry in a shift by one)
        const T sp_ = (lane == 0) ? w.p[m + 1 < VPT ? m + 1 : m] : w.p[m];
        const T sv_ = (lane == 0) ? w.v[m + 1 < VPT ? m + 1 : m] : w.v[m];
        const T lp = __shfl_sync(0xffffffffu, sp_, (lane + 1) & 31), lv = __shfl_sync(0xffffffffu, sv_, (lane + 1) & 31);
        if (w.head[m]) { dp[m] = head_dp; dv[m] = head_dv; }
        else { dp[m] = t_abs(lp - w.p[m]) - (w.lead_len[m] + w.k[m].len) * T(0.5); dv[m] = w.v[m] - lv; }
    }
}

template <typename T, int VPT>
__device__ __forceinline__ int lane_step(WarpLane<T, VPT>& w, T head_dp, T head_dv, unsigned lane, T dt, T inv_dt) {
    T dp[VPT], dv[VPT];
    lane_deltas(w, head_dp, head_dv, lane, dp, dv);
    int ncol = 0;
#pragma unroll
    for (int m = 0; m < VPT; m++) {
        IdmEval<T> e = idm_eval(w.v[m], w.k[m], dp[m], dv[m], inv_dt);
        if (w.valid[m]) {
            ncol += e.col;
            w.p[m] = w.p[m] + dt * w.v[m];
            w.v[m] = w.v[m] + dt * e.acc;
        }
    }
    return ncol;
}

// EXT = false: no per-step head deltas (head_t is null) -- a separate instantiation, so that the plain rollout does not carry the
// per-step fetches and tests in its time loop (they cost 9 % when they were run-time branches).
template <typename T, int VPT, bool EXT>
__global__ void __launch_bounds__(IDM_ROLL_BLOCK)
idm_rollout_fwd_kernel(const T* __restrict__ p0, const T* __restrict__ v0, const T* __restrict__ params,
                       const int* __restrict__ lane_off, const T* __restrict__ head, const T* __restrict__ head_t_, T dt,
                       int V, int L, int steps, int K, T* __restrict__ ckpt, T* __restrict__ pT, T* __restrict__ vT,
                       int* __restrict__ flags) {
    const T* __restrict__ head_t = EXT ? head_t_ : nullptr;
    const unsigned lane = threadIdx.x & 31;
    const int wid = (blockIdx.x * IDM_ROLL_BLOCK + threadIdx.x) >> 5, nw = (gridDim.x * IDM_ROLL_BLOCK) >> 5;
    const T inv_dt = T(1) / dt;
    int ncol = 0;
    for (int l = wid; l < L; l += nw) {
        const int o = lane_off[l], n = lane_off[l + 1] - o;
        if (n <= 0) continue;
        WarpLane<T, VPT> w;
        lane_load(w, p0, v0, params, V, o, n, lane);
        // head deltas: one pair for the whole rollout, or one per step (head_t [steps][L][2], fetched a step ahead)
        T hdp = head_t ? (steps > 0 ? head_t[2 * l] : T(0)) : head[2 * l];
        T hdv = head_t ? (steps > 0 ? head_t[2 * l + 1] : T(0)) : head[2 * l + 1];
        for (int t = 0; t < steps; t++) {
            T ndp = hdp, ndv = hdv;
            if (head_t && t + 1 < steps) { const T* q = head_t + ((size_t)(t + 1) * L + l) * 2; ndp = q[0]; ndv = q[1]; }
            if (ckpt && t % K == 0) {
                T* cp = ckpt + (size_t)(t / K) * 2 * V + o; T* cv = cp + V;
#pragma unroll
                for (int m = 0; m < VPT; m++)
                    if (w.valid[m]) { cp[m * 32 + lane] = w.p[m]; cv[m * 32 + lane] = w.v[m]; }
            }
            ncol += lane_step(w, hdp, hdv, lane, dt, inv_dt);
            hdp = ndp; hdv = ndv;
        }
#pragma unroll
        for (int m = 0; m < VPT; m++)
            if (w.valid[m]) { pT[o + m * 32 + lane] = w.p[m]; vT[o + m * 32 + lane] = w.v[m]; }
    }
    if (ncol) { atomicOr(flags, FLAG_COLLISION); atomicAdd(flags + 1, ncol); }
}

// EXT = false: no per-step head deltas, no per-step adjoint injection (head_t, g_head_t, g_hist are null).
// PAR = true: also the adjoint of the vehicle parameters, g_params [6][V]: each thread keeps six accumulators per vehicle
// in registers over all segments (idm_par_vjp) and writes them once, after the last step.
template <typename T, int VPT, bool EXT, bool PAR>
__global__ void __launch_bounds__(IDM_ROLL_BLOCK)
idm_rollout_bwd_kernel(const T* __restrict__ ckpt, const T* __restrict__ params, const int* __restrict__ lane_off,
                       const T* __restrict__ head, const T* __restrict__ head_t_, T dt, int V, int L, int steps, int K,
                       const T* __restrict__ g_pT, const T* __restrict__ g_vT, const T* __restrict__ g_hist_,
                       T* __restrict__ g_p0, T* __restrict__ g_v0, T* __restrict__ g_head, T* __restrict__ g_head_t_,
                       int* __restrict__ flags, T* __restrict__ g_params) {
    const T* __restrict__ head_t = EXT ? head_t_ : nullptr;
    const T* __restrict__ g_hist = EXT ? g_hist_ : nullptr;
    T* __restrict__ g_head_t = EXT ? g_head_t_ : nullptr;
    const unsigned lane = threadIdx.x & 31;
    const int wid = (blockIdx.x * IDM_ROLL_BLOCK + threadIdx.x) >> 5, nw = (gridDim.x * IDM_ROLL_BLOCK) >> 5;
    const T inv_dt = T(1) / dt;
    const int S = (steps + K - 1) / K;
    bool bad = false;
    T sp[IDM_KMAX][VPT], sv[IDM_KMAX][VPT];       // per-thread stash of the segment's states
    for (int l = wid; l < L; l += nw) {
        const int o = lane_off[l], n = lane_off[l + 1] - o;
        if (n <= 0) {
            if (g_head && lane == 0) { g_head[2 * l] = T(0); g_head[2 * l + 1] = T(0); }
            if (g_head_t)
                for (int t = (int)lane; t < steps; t += 32) { g_head_t[((size_t)t * L + l) * 2] = T(0); g_head_t[((size_t)t * L + l) * 2 + 1] = T(0); }
            continue;
        }
        T hdp = head_t ? T(0) : head[2 * l], hdv = head_t ? T(0) : head[2 * l + 1];
        WarpLane<T, VPT> w;
        T gp[VPT], gv[VPT], ghp = T(0), ghv = T(0);
        IdmParAdj<T> pa[VPT];
#pragma unroll
        for (int m = 0; m < VPT; m++) {
            int e = m * 32 + (int)lane;
            gp[m] = (e < n) ? g_pT[o + e] : T(0); gv[m] = (e < n) ? g_vT[o + e] : T(0);
            if constexpr (PAR) pa[m] = {T(0), T(0), T(0), T(0), T(0), T(0)};
        }
        for (int seg = S - 1; seg >= 0; seg--) {
            const int t0 = seg * K, ks = min(K, steps - t0);
            const T* cp = ckpt + (size_t)seg * 2 * V; const T* cv = cp + V;
            lane_load(w, cp, cv, params, V, o, n, lane);
            for (int k = 0; k < ks; k++) {
#pragma unroll
                for (int m = 0; m < VPT; m++) { sp[k][m] = w.p[m]; sv[k][m] = w.v[m]; }
                if (head_t) { const T* q = head_t + ((size_t)(t0 + k) * L + l) * 2; hdp = q[0]; hdv = q[1]; }
                if (k + 1 < ks) lane_step(w, hdp, hdv, lane, dt, inv_dt);
            }
            for (int k = ks - 1; k >= 0; k--) {
#pragma unroll
                for (int m = 0; m < VPT; m++) { w.p[m] = sp[k][m]; w.v[m] = sv[k][m]; }
                T dp[VPT], dv[VPT], cpv[VPT], cvv[VPT], np_[VPT], nv_[VPT];
                if (head_t) { const T* q = head_t + ((size_t)(t0 + k) * L + l) * 2; hdp = q[0]; hdv = q[1]; }
                lane_deltas(w, hdp, hdv, lane, dp, dv);
#pragma unroll
                for (int m = 0; m < VPT; m++) {
                    T E10, E11, L10, L11;
                    IdmEval<T> e = idm_eval(w.v[m], w.k[m], dp[m], dv[m], inv_dt);
                    idm_jac(w.v[m], w.k[m], dp[m], dv[m], e, dt, E10, E11, L10, L11);
                    if (!w.valid[m]) { E10 = E11 = L10 = L11 = T(0); }
                    np_[m] = gp[m] + E10 * gv[m];
                    nv_[m] = dt * gp[m] + E11 * gv[m];
                    cpv[m] = L10 * gv[m]; cvv[m] = L11 * gv[m];
                    if (w.head[m]) { np_[m] += cpv[m]; nv_[m] += cvv[m]; ghp += cpv[m]; ghv -= cvv[m]; }
                    if constexpr (PAR)
                        if (w.valid[m]) {
                            idm_par_vjp(w.v[m], w.k[m], dp[m], dv[m], e, gv[m], pa[m]);
                            if (!w.head[m]) pa[m].len += T(-0.5) * cpv[m];
                        }
                }
                // follower (e-1) -> me: within a slot from lane-1, across slots from lane 31 of slot m-1
#pragma unroll
                for (int m = 0; m < VPT; m++) {
                    // one rotation per value (see lane_deltas): lane 31 sends the PREVIOUS slot's entry, which lane 0 needs
                    const T sp_ = (lane == 31) ? (m > 0 ? cpv[m > 0 ? m - 1 : 0] : T(0)) : cpv[m];
                    const T sv_ = (lane == 31) ? (m > 0 ? cvv[m > 0 ? m - 1 : 0] : T(0)) : cvv[m];
                    const T fp = __shfl_sync(0xffffffffu, sp_, (lane + 31) & 31), fv = __shfl_sync(0xffffffffu, sv_, (lane + 31) & 31);
                    if (w.valid[m]) { gp[m] = np_[m] + fp; gv[m] = nv_[m] + fv; }
                    if constexpr (PAR) pa[m].len += T(-0.5) * fp;      // the follower's gap holds this vehicle's length
                }
                if (g_head_t) {       // per-step head deltas: this step's adjoint leaves, the accumulator restarts
                    bool own = false;
#pragma unroll
                    for (int m = 0; m < VPT; m++) own |= w.head[m];
                    if (own) { T* q = g_head_t + ((size_t)(t0 + k) * L + l) * 2; q[0] = ghp; q[1] = ghv; }
                    bad |= t_isnan(ghp) || t_isnan(ghv);
                    ghp = T(0); ghv = T(0);
                }
                if (g_hist) {         // loss terms on the state before this step
                    const T* q = g_hist + (size_t)(t0 + k) * 2 * V + o;
#pragma unroll
                    for (int m = 0; m < VPT; m++)
                        if (w.valid[m]) { gp[m] += q[m * 32 + lane]; gv[m] += q[V + m * 32 + lane]; }
                }
            }
        }
        // NaN test once, on the final adjoint: gp' = gp + ..., gv' = dt gp + E11 gv + ... keep a NaN in its vehicle for good
#pragma unroll
        for (int m = 0; m < VPT; m++) bad |= t_isnan(gp[m]) || t_isnan(gv[m]);
#pragma unroll
        for (int m = 0; m < VPT; m++)
            if (w.valid[m]) { g_p0[o + m * 32 + lane] = gp[m]; g_v0[o + m * 32 + lane] = gv[m]; }
        if constexpr (PAR) {
#pragma unroll
            for (int m = 0; m < VPT; m++)
                if (w.valid[m]) {
                    const size_t i = (size_t)o + m * 32 + lane;
                    T g[6];
                    idm_par_grad(pa[m], w.k[m], params[(size_t)V + i], dt, g);
#pragma unroll
                    for (int r = 0; r < 6; r++) { g_params[(size_t)r * V + i] = g[r]; bad |= t_isnan(g[r]); }
                }
        }
        if (g_head) {
            // exactly one thread of the warp owns the head vehicle
            bool own = false;
#pragma unroll
            for (int m = 0; m < VPT; m++) own |= w.head[m];
            if (own) { g_head[2 * l] = ghp; g_head[2 * l + 1] = ghv; }
        }
    }
    if (bad) atomicOr(flags, FLAG_NAN_GRAD);
}

// ------------------------------------------------------------------ host side

static int idm_grid(int L) {
    int warps_per_block = IDM_ROLL_BLOCK / 32;
    long long want = ((long long)L + warps_per_block - 1) / warps_per_block;
    long long cap = (long long)sm_count() * 16;
    return (int)(want < cap ? (want < 1 ? 1 : want) : cap);
}

template <typename T>
static int idm_step_fwd(const T* p, const T* v, const T* params, const int* lane_off, const int* veh_lane,
                        const T* head, T dt, int V, int L, T* np_, T* nv_, int* vflags, int* flags, cudaStream_t st) {
    if (!p || !v || !params || !lane_off || !veh_lane || !head || !np_ || !nv_ || !flags || V < 0 || L < 0)
        return DHTS_ERR_INVALID;
    if (V == 0) return DHTS_OK;
    idm_step_fwd_kernel<T><<<(V + IDM_BLOCK - 1) / IDM_BLOCK, IDM_BLOCK, 0, st>>>(p, v, params, lane_off, veh_lane, head,
                                                                                  dt, V, np_, nv_, vflags, flags);
    return launch_status();
}

// g_params NULL: the state adjoint only (dhts_idm_step_bwd_*)
template <typename T>
static int idm_step_bwd(const T* p, const T* v, const T* params, const int* lane_off, const int* veh_lane,
                        const T* head, T dt, int V, int L, const T* g_np, const T* g_nv, T* g_p, T* g_v, T* g_head,
                        T* g_params, int* flags, cudaStream_t st) {
    if (!p || !v || !params || !lane_off || !veh_lane || !head || !g_np || !g_nv || !g_p || !g_v || !flags || V < 0 ||
        L < 0)
        return DHTS_ERR_INVALID;
    if (g_head && L > 0) idm_zero_empty_head_kernel<T><<<(L + 255) / 256, 256, 0, st>>>(lane_off, L, g_head);
    if (V == 0) return launch_status();
    const int grid = (V + IDM_BLOCK - 1) / IDM_BLOCK;
    if (g_params)
        idm_step_bwd_kernel<T, true><<<grid, IDM_BLOCK, 0, st>>>(p, v, params, lane_off, veh_lane, head, dt, V, g_np, g_nv,
                                                                 g_p, g_v, g_head, flags, g_params);
    else
        idm_step_bwd_kernel<T, false><<<grid, IDM_BLOCK, 0, st>>>(p, v, params, lane_off, veh_lane, head, dt, V, g_np, g_nv,
                                                                  g_p, g_v, g_head, flags, nullptr);
    return launch_status();
}

#define DHTS_VPT_DISPATCH(max_lane, CALL)        \
    if (max_lane <= 32) { CALL(1) }              \
    else if (max_lane <= 64) { CALL(2) }         \
    else if (max_lane <= 128) { CALL(4) }        \
    else if (max_lane <= 256) { CALL(8) }        \
    else return DHTS_ERR_UNSUPPORTED;

template <typename T>
static int idm_rollout_fwd(const T* p0, const T* v0, const T* params, const int* lane_off, const T* head, const T* head_t,
                           T dt, int V, int L, int max_lane, int steps, int K, T* ckpt, T* pT, T* vT, int* flags,
                           cudaStream_t st) {
    if (!p0 || !v0 || !params || !lane_off || (!head && !head_t) || !pT || !vT || !flags || V < 0 || L < 0 || steps < 0 || max_lane < 0)
        return DHTS_ERR_INVALID;
    if (ckpt && K < 1) return DHTS_ERR_INVALID;
    if (V == 0 || L == 0) return DHTS_OK;
    int grid = idm_grid(L);
    if (K < 1) K = 1;
#define CALL(VPT) { if (head_t) idm_rollout_fwd_kernel<T, VPT, true><<<grid, IDM_ROLL_BLOCK, 0, st>>>(p0, v0, params, lane_off, head, head_t, dt, V, L, steps, K, ckpt, pT, vT, flags); \
                    else idm_rollout_fwd_kernel<T, VPT, false><<<grid, IDM_ROLL_BLOCK, 0, st>>>(p0, v0, params, lane_off, head, nullptr, dt, V, L, steps, K, ckpt, pT, vT, flags); }
    DHTS_VPT_DISPATCH(max_lane, CALL)
#undef CALL
    return launch_status();
}

// g_params NULL: the state adjoint only (dhts_idm_rollout_bwd_*)
template <typename T>
static int idm_rollout_bwd(const T* ckpt, const T* params, const int* lane_off, const T* head, const T* head_t, T dt, int V,
                           int L, int max_lane, int steps, int K, const T* g_pT, const T* g_vT, const T* g_hist, T* g_p0,
                           T* g_v0, T* g_head, T* g_head_t, T* g_params, int* flags, cudaStream_t st) {
    if (!ckpt || !params || !lane_off || (!head && !head_t) || !g_pT || !g_vT || !g_p0 || !g_v0 || !flags || V < 0 || L < 0 ||
        steps < 0 || max_lane < 0 || K < 1)
        return DHTS_ERR_INVALID;
    if ((g_head_t && !head_t) || (g_hist && K != 1)) return DHTS_ERR_INVALID;      // g_hist is laid out like ckpt with K = 1
    if (K > IDM_KMAX) return DHTS_ERR_UNSUPPORTED;
    if (L == 0) return DHTS_OK;
    int grid = idm_grid(L);
    const bool ext = head_t || g_hist || g_head_t;
#define LAUNCH(VPT, EXT, PAR) idm_rollout_bwd_kernel<T, VPT, EXT, PAR><<<grid, IDM_ROLL_BLOCK, 0, st>>>(ckpt, params, lane_off, head, EXT ? head_t : nullptr, dt, V, L, steps, K, g_pT, g_vT, EXT ? g_hist : nullptr, g_p0, g_v0, (EXT && head_t) ? nullptr : g_head, EXT ? g_head_t : nullptr, flags, g_params);
#define CALL(VPT) { if (g_params) { if (ext) LAUNCH(VPT, true, true) else LAUNCH(VPT, false, true) } \
                    else { if (ext) LAUNCH(VPT, true, false) else LAUNCH(VPT, false, false) } }
    DHTS_VPT_DISPATCH(max_lane, CALL)
#undef CALL
#undef LAUNCH
    return launch_status();
}

}  // namespace dhts

#define DHTS_IDM_API(SUF, T)                                                                                           \
    DHTS_EXPORT int dhts_idm_step_fwd_##SUF(const T* p, const T* v, const T* params, const int* lane_off,              \
                                            const int* veh_lane, const T* head, T dt, int V, int L, T* np_, T* nv_,    \
                                            int* vflags, int* flags, void* stream) {                                   \
        return dhts::idm_step_fwd<T>(p, v, params, lane_off, veh_lane, head, dt, V, L, np_, nv_, vflags, flags,        \
                                     (cudaStream_t)stream);                                                            \
    }                                                                                                                  \
    DHTS_EXPORT int dhts_idm_step_bwd_##SUF(const T* p, const T* v, const T* params, const int* lane_off,              \
                                            const int* veh_lane, const T* head, T dt, int V, int L, const T* g_np,     \
                                            const T* g_nv, T* g_p, T* g_v, T* g_head, int* flags, void* stream) {      \
        return dhts::idm_step_bwd<T>(p, v, params, lane_off, veh_lane, head, dt, V, L, g_np, g_nv, g_p, g_v, g_head,   \
                                     nullptr, flags, (cudaStream_t)stream);                                            \
    }                                                                                                                  \
    DHTS_EXPORT int dhts_idm_step_bwd_params_##SUF(const T* p, const T* v, const T* params, const int* lane_off,       \
                                                   const int* veh_lane, const T* head, T dt, int V, int L,             \
                                                   const T* g_np, const T* g_nv, T* g_p, T* g_v, T* g_head,            \
                                                   T* g_params, int* flags, void* stream) {                            \
        if (!g_params) return DHTS_ERR_INVALID;                                                                        \
        return dhts::idm_step_bwd<T>(p, v, params, lane_off, veh_lane, head, dt, V, L, g_np, g_nv, g_p, g_v, g_head,   \
                                     g_params, flags, (cudaStream_t)stream);                                           \
    }                                                                                                                  \
    DHTS_EXPORT int dhts_idm_rollout_fwd_##SUF(const T* p0, const T* v0, const T* params, const int* lane_off,         \
                                               const T* head, const T* head_t, T dt, int V, int L, int max_lane,       \
                                               int steps, int ckpt_every, T* ckpt, T* pT, T* vT, int* flags,           \
                                               void* stream) {                                                         \
        return dhts::idm_rollout_fwd<T>(p0, v0, params, lane_off, head, head_t, dt, V, L, max_lane, steps, ckpt_every, \
                                        ckpt, pT, vT, flags, (cudaStream_t)stream);                                    \
    }                                                                                                                  \
    DHTS_EXPORT int dhts_idm_rollout_bwd_##SUF(const T* ckpt, const T* params, const int* lane_off, const T* head,     \
                                               const T* head_t, T dt, int V, int L, int max_lane, int steps,           \
                                               int ckpt_every, const T* g_pT, const T* g_vT, const T* g_hist,          \
                                               T* g_p0, T* g_v0, T* g_head, T* g_head_t, int* flags, void* stream) {   \
        return dhts::idm_rollout_bwd<T>(ckpt, params, lane_off, head, head_t, dt, V, L, max_lane, steps, ckpt_every,   \
                                        g_pT, g_vT, g_hist, g_p0, g_v0, g_head, g_head_t, nullptr, flags,              \
                                        (cudaStream_t)stream);                                                         \
    }                                                                                                                  \
    DHTS_EXPORT int dhts_idm_rollout_bwd_params_##SUF(const T* ckpt, const T* params, const int* lane_off,             \
                                                      const T* head, const T* head_t, T dt, int V, int L,              \
                                                      int max_lane, int steps, int ckpt_every, const T* g_pT,          \
                                                      const T* g_vT, const T* g_hist, T* g_p0, T* g_v0, T* g_head,     \
                                                      T* g_head_t, T* g_params, int* flags, void* stream) {            \
        if (!g_params) return DHTS_ERR_INVALID;                                                                        \
        return dhts::idm_rollout_bwd<T>(ckpt, params, lane_off, head, head_t, dt, V, L, max_lane, steps, ckpt_every,   \
                                        g_pT, g_vT, g_hist, g_p0, g_v0, g_head, g_head_t, g_params, flags,             \
                                        (cudaStream_t)stream);                                                         \
    }

// C ABI
DHTS_IDM_API(f64, double)
DHTS_IDM_API(f32, float)

DHTS_EXPORT int dhts_csr_expand(const int* lane_off, int L, int* veh_lane, void* stream) {
    if (!lane_off || !veh_lane || L < 0) return DHTS_ERR_INVALID;
    if (L == 0) return DHTS_OK;
    int blocks = (L + 7) / 8;
    if (blocks > 148 * 8) blocks = 148 * 8;
    dhts::csr_expand_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(lane_off, L, veh_lane);
    return dhts::launch_status();
}

DHTS_EXPORT int dhts_idm_rollout_max_ckpt_every(void) { return dhts::IDM_KMAX; }
DHTS_EXPORT int dhts_idm_rollout_max_lane(void) { return 256; }
