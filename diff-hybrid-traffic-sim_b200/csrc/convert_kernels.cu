// Macro <-> micro boundary exchange kernels for sm_100a (K5), batched over junctions.
//
// Behaviour restated from the reference's live exchange, road/network/conversion.py
// (road/hybrid.py is a dead draft, SURVEY section 0):
//   macro_to_micro  conversion.py:15-73   flux capacitor, spawn test, new-vehicle state
//   micro_to_macro  conversion.py:75-171  head removal test, density deposit with
//                                         value-clamp / pass-through gradient
// micro_to_micro / micro_to_none (:174-215) are pure bookkeeping (list hand-off,
// p -= L) and stay on the host side of the operator.
// One thread per junction: the work is scalar and event-like (at most one spawn
// and one absorption per junction per step, SURVEY App. B.8).
#include "dhts_arz.cuh"
#include "dhts_api.h"

namespace dhts {

constexpr int CV_BLOCK = 128;

// conversion.py:32-68.  cap_out is the capacitor AFTER the step; when a vehicle is
// spawned it is re-created detached (:65-68), so its adjoint is cut there.
template <typename T>
__global__ void m2c_fwd_kernel(const T* __restrict__ cap, const T* __restrict__ r_last, const T* __restrict__ u_last,
                               const T* __restrict__ free_space, const T* __restrict__ veh_len, T dt, int J,
                               T* __restrict__ cap_out, int* __restrict__ spawn, T* __restrict__ v_new,
                               T* __restrict__ a_new) {
    int j = blockIdx.x * CV_BLOCK + threadIdx.x;
    if (j >= J) return;
    T len = veh_len[j];
    T flux = cap[j] + r_last[j] * u_last[j] * dt;            // :32-34
    bool sp = (flux >= len) && (free_space[j] >= len * T(1));  // :55
    spawn[j] = sp ? 1 : 0;
    if (sp) {
        v_new[j] = u_last[j];                                // :61
        a_new[j] = flux - (flux - len);                      // :62  value = len, gradient of the capacitor
        cap_out[j] = flux - len;                             // :65-68
    } else {
        v_new[j] = T(0); a_new[j] = T(0);
        cap_out[j] = flux;
    }
}

template <typename T>
__global__ void m2c_bwd_kernel(const T* __restrict__ r_last, const T* __restrict__ u_last,
                               const int* __restrict__ spawn, T dt, int J, const T* __restrict__ g_cap_out,
                               const T* __restrict__ g_v_new, const T* __restrict__ g_a_new, T* __restrict__ g_cap,
                               T* __restrict__ g_r_last, T* __restrict__ g_u_last) {
    int j = blockIdx.x * CV_BLOCK + threadIdx.x;
    if (j >= J) return;
    bool sp = spawn[j] != 0;
    T gf = sp ? g_a_new[j] : g_cap_out[j];                   // adjoint of the pre-spawn capacitor value
    g_cap[j] = gf;
    g_r_last[j] = gf * u_last[j] * dt;
    g_u_last[j] = gf * r_last[j] * dt + (sp ? g_v_new[j] : T(0));
}

// geometry of one touched cell (conversion.py:124-137)
template <typename T>
__device__ __forceinline__ bool c2m_cell(int ci, T dx, T len, T v_head, T v_tail, T& overlap, T& dodp) {
    T c_head = dx * T(ci + 1), c_tail = dx * T(ci);          // Cell.end / Cell.start, _macro_lane.py:46-47
    if (!(c_head > v_tail && c_tail < v_head)) return false;
    bool head_is_cell = c_head > v_head, tail_is_cell = c_tail < v_tail;
    T max_head = head_is_cell ? c_head : v_head;
    T min_tail = tail_is_cell ? c_tail : v_tail;
    overlap = dx + len - (max_head - min_tail);
    dodp = (head_is_cell ? T(0) : T(-1)) + (tail_is_cell ? T(0) : T(1));   // d overlap / d p_head
    return true;
}

// conversion.py:99-171.  r, y, u are [J][N] rows of the downstream macro lanes;
// outputs are full rows (untouched cells copied through).  The stored u_eq of a
// touched cell is NOT refreshed by the reference; callers keep their old u_eq.
template <typename T>
__global__ void c2m_fwd_kernel(const T* __restrict__ p_head, const T* __restrict__ v_head_,
                               const T* __restrict__ a_head, const T* __restrict__ len_head,
                               const T* __restrict__ lane_len, const T* __restrict__ r, const T* __restrict__ y,
                               const T* __restrict__ u, const T* __restrict__ dx_, const T* __restrict__ umax_, int J,
                               int N, T* __restrict__ r_out, T* __restrict__ y_out, T* __restrict__ u_out,
                               int* __restrict__ absorbed, int* __restrict__ ntouched) {
    int j = blockIdx.x * CV_BLOCK + threadIdx.x;
    if (j >= J) return;
    const size_t o = (size_t)j * N;
    T len = len_head[j], dx = dx_[j], umax = umax_[j];
    bool ab = p_head[j] > lane_len[j] + T(1) * len;          // :99
    absorbed[j] = ab ? 1 : 0;
    int nt = 0;
    if (ab) {
        T v_hd = p_head[j] - lane_len[j], v_tl = v_hd - len; // :117-118
        T spd = v_head_[j], a = a_head[j];
        for (int ci = 0; ci < N; ci++) {
            T overlap, dodp;
            if (!c2m_cell(ci, dx, len, v_hd, v_tl, overlap, dodp)) break;   // :169-171
            T n_r = r[o + ci] + (a / len) * (overlap / dx);  // :139-141
            if (n_r > T(1) - T(1e-5)) n_r = T(1) - T(1e-5);  // :149-155 (value clamp)
            else if (n_r < T(1e-5)) n_r = T(1e-5);
            r_out[o + ci] = n_r;
            u_out[o + ci] = spd;                             // :160
            y_out[o + ci] = n_r * (spd - u_eq(n_r, umax));   // :164-167
            nt++;
        }
    }
    ntouched[j] = nt;
    for (int ci = nt; ci < N; ci++) { r_out[o + ci] = r[o + ci]; y_out[o + ci] = y[o + ci]; u_out[o + ci] = u[o + ci]; }
}

template <typename T>
__global__ void c2m_bwd_kernel(const T* __restrict__ p_head, const T* __restrict__ v_head_,
                               const T* __restrict__ a_head, const T* __restrict__ len_head,
                               const T* __restrict__ lane_len, const T* __restrict__ r_out,
                               const T* __restrict__ dx_, const T* __restrict__ umax_, const int* __restrict__ ntouched,
                               int J, int N, const T* __restrict__ g_r_out, const T* __restrict__ g_y_out,
                               const T* __restrict__ g_u_out, T* __restrict__ g_p, T* __restrict__ g_v,
                               T* __restrict__ g_a, T* __restrict__ g_r, T* __restrict__ g_y, T* __restrict__ g_u) {
    int j = blockIdx.x * CV_BLOCK + threadIdx.x;
    if (j >= J) return;
    const size_t o = (size_t)j * N;
    T len = len_head[j], dx = dx_[j], umax = umax_[j];
    T v_hd = p_head[j] - lane_len[j], v_tl = v_hd - len;
    T spd = v_head_[j], a = a_head[j];
    T gp = T(0), gv = T(0), ga = T(0);
    const int nt = ntouched[j];
    for (int ci = 0; ci < nt; ci++) {
        T overlap, dodp;
        c2m_cell(ci, dx, len, v_hd, v_tl, overlap, dodp);
        T n_r = r_out[o + ci];
        // y = n_r (v - u_eq(n_r)) differentiated by autograd: true derivative of _arz.py:133-138
        T ueq = u_eq(n_r, umax);
        T ueqp = (n_r >= T(0)) ? T(-0.5) * umax / t_sqrt(n_r + DHTS_EPS) : T(0);
        T gy = g_y_out[o + ci];
        T gnr = g_r_out[o + ci] + gy * ((spd - ueq) - n_r * ueqp);   // clamp passes the gradient through
        gv += g_u_out[o + ci] + gy * n_r;
        ga += gnr * (overlap / dx) / len;
        gp += gnr * (a / len) * (dodp / dx);
        g_r[o + ci] = gnr; g_y[o + ci] = T(0); g_u[o + ci] = T(0);   // old y, u of the cell are discarded
    }
    for (int ci = nt; ci < N; ci++) { g_r[o + ci] = g_r_out[o + ci]; g_y[o + ci] = g_y_out[o + ci]; g_u[o + ci] = g_u_out[o + ci]; }
    g_p[j] = gp; g_v[j] = gv; g_a[j] = ga;
}

}  // namespace dhts

#define DHTS_CV_API(SUF, T)                                                                                            \
    DHTS_EXPORT int dhts_m2c_fwd_##SUF(const T* cap, const T* r_last, const T* u_last, const T* free_space,            \
                                       const T* veh_len, T dt, int J, T* cap_out, int* spawn, T* v_new, T* a_new,      \
                                       void* stream) {                                                                 \
        if (!cap || !r_last || !u_last || !free_space || !veh_len || !cap_out || !spawn || !v_new || !a_new || J < 0)  \
            return DHTS_ERR_INVALID;                                                                                   \
        if (J == 0) return DHTS_OK;                                                                                    \
        dhts::m2c_fwd_kernel<T><<<(J + dhts::CV_BLOCK - 1) / dhts::CV_BLOCK, dhts::CV_BLOCK, 0,                        \
                                  (cudaStream_t)stream>>>(cap, r_last, u_last, free_space, veh_len, dt, J, cap_out,    \
                                                          spawn, v_new, a_new);                                        \
        return dhts::launch_status();                                                                                  \
    }                                                                                                                  \
    DHTS_EXPORT int dhts_m2c_bwd_##SUF(const T* r_last, const T* u_last, const int* spawn, T dt, int J,                \
                                       const T* g_cap_out, const T* g_v_new, const T* g_a_new, T* g_cap,               \
                                       T* g_r_last, T* g_u_last, void* stream) {                                       \
        if (!r_last || !u_last || !spawn || !g_cap_out || !g_v_new || !g_a_new || !g_cap || !g_r_last || !g_u_last ||  \
            J < 0)                                                                                                     \
            return DHTS_ERR_INVALID;                                                                                   \
        if (J == 0) return DHTS_OK;                                                                                    \
        dhts::m2c_bwd_kernel<T><<<(J + dhts::CV_BLOCK - 1) / dhts::CV_BLOCK, dhts::CV_BLOCK, 0,                        \
                                  (cudaStream_t)stream>>>(r_last, u_last, spawn, dt, J, g_cap_out, g_v_new, g_a_new,   \
                                                          g_cap, g_r_last, g_u_last);                                  \
        return dhts::launch_status();                                                                                  \
    }                                                                                                                  \
    DHTS_EXPORT int dhts_c2m_fwd_##SUF(const T* p_head, const T* v_head, const T* a_head, const T* len_head,           \
                                       const T* lane_len, const T* r, const T* y, const T* u, const T* dx,             \
                                       const T* umax, int J, int N, T* r_out, T* y_out, T* u_out, int* absorbed,       \
                                       int* ntouched, void* stream) {                                                  \
        if (!p_head || !v_head || !a_head || !len_head || !lane_len || !r || !y || !u || !dx || !umax || !r_out ||     \
            !y_out || !u_out || !absorbed || !ntouched || J < 0 || N < 1)                                              \
            return DHTS_ERR_INVALID;                                                                                   \
        if (J == 0) return DHTS_OK;                                                                                    \
        dhts::c2m_fwd_kernel<T><<<(J + dhts::CV_BLOCK - 1) / dhts::CV_BLOCK, dhts::CV_BLOCK, 0,                        \
                                  (cudaStream_t)stream>>>(p_head, v_head, a_head, len_head, lane_len, r, y, u, dx,     \
                                                          umax, J, N, r_out, y_out, u_out, absorbed, ntouched);        \
        return dhts::launch_status();                                                                                  \
    }                                                                                                                  \
    DHTS_EXPORT int dhts_c2m_bwd_##SUF(const T* p_head, const T* v_head, const T* a_head, const T* len_head,           \
                                       const T* lane_len, const T* r_out, const T* dx, const T* umax,                  \
                                       const int* ntouched, int J, int N, const T* g_r_out, const T* g_y_out,          \
                                       const T* g_u_out, T* g_p, T* g_v, T* g_a, T* g_r, T* g_y, T* g_u,               \
                                       void* stream) {                                                                 \
        if (!p_head || !v_head || !a_head || !len_head || !lane_len || !r_out || !dx || !umax || !ntouched ||          \
            !g_r_out || !g_y_out || !g_u_out || !g_p || !g_v || !g_a || !g_r || !g_y || !g_u || J < 0 || N < 1)        \
            return DHTS_ERR_INVALID;                                                                                   \
        if (J == 0) return DHTS_OK;                                                                                    \
        dhts::c2m_bwd_kernel<T><<<(J + dhts::CV_BLOCK - 1) / dhts::CV_BLOCK, dhts::CV_BLOCK, 0,                        \
                                  (cudaStream_t)stream>>>(p_head, v_head, a_head, len_head, lane_len, r_out, dx, umax, \
                                                          ntouched, J, N, g_r_out, g_y_out, g_u_out, g_p, g_v, g_a,    \
                                                          g_r, g_y, g_u);                                              \
        return dhts::launch_status();                                                                                  \
    }

DHTS_CV_API(f64, double)
DHTS_CV_API(f32, float)
