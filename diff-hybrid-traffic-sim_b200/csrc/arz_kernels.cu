// ARZ macroscopic lane kernels for sm_100a (K1 forward, K2 adjoint).
//
//  * arz_step_{fwd,bwd}_kernel   one Godunov step over B lanes x N cells, tiled:
//    each CTA stages a tile of cells plus a one-cell halo per side in shared
//    memory (coalesced loads), solves the tile's interfaces once, then updates.
//    This is the operator behind the reference's per-step autograd contract
//    dMacroForwardLayer (road/lane/dmacro_lane.py:234-310).
//  * the fused T-step rollouts live in arz_rollout.cu.
//
// No tensor cores: nothing here is a contraction (BASELINE.json north_star).
#include "dhts_arz.cuh"
#include "dhts_api.h"

namespace dhts {

constexpr int STEP_TILE = 256;

template <typename T> struct SM {
    T *r, *y, *us, *uc, *w, *sq, *rs, *ri, *uf;   // per padded cell
    T *f0, *f1, *f2, *f3;                         // per interface (flux, or A^T w / B^T w)
    T *gr, *gy;                                   // per padded cell (adjoint)
};

template <typename T, bool ADJ> __device__ __forceinline__ SM<T> carve(unsigned char* raw, int ncell, int nif) {
    SM<T> s;
    T* p = reinterpret_cast<T*>(raw);
    s.r = p; p += ncell; s.y = p; p += ncell; s.us = p; p += ncell; s.uc = p; p += ncell;
    s.w = p; p += ncell; s.sq = p; p += ncell;
    s.f0 = p; p += nif; s.f1 = p; p += nif;
    if (ADJ) {
        s.rs = p; p += ncell; s.ri = p; p += ncell; s.uf = p; p += ncell;
        s.f2 = p; p += nif; s.f3 = p; p += nif;
        s.gr = p; p += ncell; s.gy = p; p += ncell;
    } else {
        s.rs = s.ri = s.uf = s.f2 = s.f3 = s.gr = s.gy = nullptr;
    }
    return s;
}
template <typename T, bool ADJ> __host__ __device__ inline size_t smem_bytes(int ncell, int nif) {
    return sizeof(T) * (size_t)(ADJ ? (11 * ncell + 4 * nif) : (6 * ncell + 2 * nif));
}

template <typename T, bool ADJ> __device__ __forceinline__ void st_cell(const SM<T>& s, int q, const Cell<T>& c) {
    s.r[q] = c.r; s.y[q] = c.y; s.us[q] = c.us; s.uc[q] = c.uc; s.w[q] = c.w; s.sq[q] = c.sq;
    if (ADJ) { s.rs[q] = c.rs; s.ri[q] = c.ri; s.uf[q] = c.uf; }
}
template <typename T, bool ADJ> __device__ __forceinline__ Cell<T> ld_cell(const SM<T>& s, int q) {
    Cell<T> c;
    c.r = s.r[q]; c.y = s.y[q]; c.us = s.us[q]; c.uc = s.uc[q]; c.w = s.w[q]; c.sq = s.sq[q];
    if (ADJ) { c.rs = s.rs[q]; c.ri = s.ri[q]; c.uf = s.uf[q]; }
    else { c.rs = T(0); c.ri = T(0); c.uf = T(0); }
    return c;
}

// ------------------------------------------------------------------ single step, tiled

template <typename T>
__global__ void __launch_bounds__(STEP_TILE)
arz_step_fwd_kernel(const T* __restrict__ r_pad, const T* __restrict__ y_pad, const T* __restrict__ u_pad,
                    const T* __restrict__ ueq_pad, const T* __restrict__ dx, const T* __restrict__ umax_, T dt, int B,
                    int N, int ntile, T* __restrict__ nr, T* __restrict__ ny, T* __restrict__ nu,
                    int* __restrict__ case_out, int* __restrict__ flags) {
    extern __shared__ __align__(16) unsigned char raw[];
    SM<T> s = carve<T, false>(raw, STEP_TILE + 2, STEP_TILE + 1);
    const int b = blockIdx.x / ntile, tile = blockIdx.x % ntile;
    const int c0 = tile * STEP_TILE;
    const int nc = min(STEP_TILE, N - c0);
    const int P = N + 2;
    const T umax = umax_[b], inv_umax = T(1) / umax, inv15 = T(1) / (T(1.5) * umax), dxb = dx[b], cc = dt / dxb;
    const size_t base = (size_t)b * P + c0;
    for (int k = threadIdx.x; k < nc + 2; k += STEP_TILE) {
        T ue = ueq_pad ? ueq_pad[base + k] : T(0);
        st_cell<T, false>(s, k, derive_cell_stored<T, false>(r_pad[base + k], y_pad[base + k], u_pad[base + k], ue,
                                                              ueq_pad != nullptr, umax));
    }
    __syncthreads();
    bool bad = false;
    for (int i = threadIdx.x; i < nc + 1; i += STEP_TILE) {
        Riem<T> o = riemann(ld_cell<T, false>(s, i), ld_cell<T, false>(s, i + 1), umax, inv_umax, inv15, dt, dxb);
        s.f0[i] = o.r0 * o.u0; s.f1[i] = o.y0 * o.u0;
        bad |= o.cfl_bad;
        if (case_out) case_out[(size_t)b * (N + 1) + c0 + i] = o.cas;
    }
    __syncthreads();
    for (int j = threadIdx.x; j < nc; j += STEP_TILE) {
        T r = s.r[j + 1] + (s.f0[j] - s.f0[j + 1]) * cc;
        T y = s.y[j + 1] + (s.f1[j] - s.f1[j + 1]) * cc;
        size_t o = (size_t)b * N + c0 + j;
        nr[o] = r; ny[o] = y; nu[o] = compute_u(r, y, umax);
    }
    if (bad) atomicOr(flags, FLAG_CFL);
}

template <typename T>
__global__ void __launch_bounds__(STEP_TILE)
arz_step_bwd_kernel(const T* __restrict__ r_pad, const T* __restrict__ y_pad, const T* __restrict__ u_pad,
                    const T* __restrict__ ueq_pad, const T* __restrict__ dx, const T* __restrict__ umax_, T dt, int B,
                    int N, int ntile, const T* __restrict__ nr, const T* __restrict__ ny,
                    const T* __restrict__ g_nr, const T* __restrict__ g_ny, const T* __restrict__ g_nu,
                    T* __restrict__ g_r_pad, T* __restrict__ g_y_pad, int* __restrict__ flags) {
    extern __shared__ __align__(16) unsigned char raw[];
    SM<T> s = carve<T, true>(raw, STEP_TILE + 2, STEP_TILE + 1);
    const int b = blockIdx.x / ntile, tile = blockIdx.x % ntile;
    const int c0 = tile * STEP_TILE;
    const int nc = min(STEP_TILE, N - c0);
    const int P = N + 2;
    const T umax = umax_[b], inv_umax = T(1) / umax, inv15 = T(1) / (T(1.5) * umax), dxb = dx[b], cc = dt / dxb;
    const size_t base = (size_t)b * P + c0;
    for (int k = threadIdx.x; k < nc + 2; k += STEP_TILE) {
        T ue = ueq_pad ? ueq_pad[base + k] : T(0);
        st_cell<T, true>(s, k, derive_cell_stored<T, true>(r_pad[base + k], y_pad[base + k], u_pad[base + k], ue,
                                                            ueq_pad != nullptr, umax));
        int j = c0 + k;   // padded index; updated cells are 1..N
        T gr = T(0), gy = T(0);
        if (j >= 1 && j <= N) {
            size_t o = (size_t)b * N + j - 1;
            gr = g_nr[o]; gy = g_ny[o];
            if (g_nu) {   // nu = compute_u(nr, ny) is produced inside the operator
                T dr, dy; du_dry(nr[o], ny[o], umax, dr, dy);
                T gu = g_nu[o]; gr += gu * dr; gy += gu * dy;
            }
        }
        s.gr[k] = gr; s.gy[k] = gy;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < nc + 1; i += STEP_TILE) {
        Cell<T> L = ld_cell<T, true>(s, i), R = ld_cell<T, true>(s, i + 1);
        Riem<T> o = riemann(L, R, umax, inv_umax, inv15, dt, dxb);
        riemann_adj(L, R, o, umax, inv_umax, inv15, s.gr[i + 1] - s.gr[i], s.gy[i + 1] - s.gy[i], s.f0[i], s.f1[i],
                    s.f2[i], s.f3[i]);
    }
    __syncthreads();
    bool bad = false;
    for (int j = threadIdx.x; j < nc; j += STEP_TILE) {
        int k = j + 1;
        T gr = s.gr[k] + cc * (s.f0[k] + s.f2[k - 1]);
        T gy = s.gy[k] + cc * (s.f1[k] + s.f3[k - 1]);
        bad |= t_isnan(gr) || t_isnan(gy);
        g_r_pad[base + k] = gr; g_y_pad[base + k] = gy;
    }
    if (threadIdx.x == 0) {
        if (tile == 0) {
            T gr = cc * s.f0[0], gy = cc * s.f1[0];
            bad |= t_isnan(gr) || t_isnan(gy);
            g_r_pad[(size_t)b * P] = gr; g_y_pad[(size_t)b * P] = gy;
        }
        if (tile == ntile - 1) {
            T gr = cc * s.f2[nc], gy = cc * s.f3[nc];
            bad |= t_isnan(gr) || t_isnan(gy);
            g_r_pad[(size_t)b * P + N + 1] = gr; g_y_pad[(size_t)b * P + N + 1] = gy;
        }
    }
    if (bad) atomicOr(flags, FLAG_NAN_GRAD);
}

// ------------------------------------------------------------------ host-side launch planning

template <typename T>
static int arz_step_fwd(const T* r_pad, const T* y_pad, const T* u_pad, const T* ueq_pad, const T* dx, const T* umax,
                        T dt, int B, int N, T* nr, T* ny, T* nu, int* case_out, int* flags, cudaStream_t st) {
    if (!r_pad || !y_pad || !u_pad || !dx || !umax || !nr || !ny || !nu || !flags || B < 0 || N < 1) return DHTS_ERR_INVALID;
    if (B == 0) return DHTS_OK;
    int ntile = (N + STEP_TILE - 1) / STEP_TILE;
    if ((long long)B * ntile > 2147483647LL) return DHTS_ERR_UNSUPPORTED;
    size_t sm = smem_bytes<T, false>(STEP_TILE + 2, STEP_TILE + 1);
    arz_step_fwd_kernel<T><<<B * ntile, STEP_TILE, sm, st>>>(r_pad, y_pad, u_pad, ueq_pad, dx, umax, dt, B, N, ntile, nr,
                                                              ny, nu, case_out, flags);
    return launch_status();
}

template <typename T>
static int arz_step_bwd(const T* r_pad, const T* y_pad, const T* u_pad, const T* ueq_pad, const T* dx, const T* umax,
                        T dt, int B, int N, const T* nr, const T* ny, const T* g_nr, const T* g_ny, const T* g_nu,
                        T* g_r_pad, T* g_y_pad, int* flags, cudaStream_t st) {
    if (!r_pad || !y_pad || !u_pad || !dx || !umax || !g_nr || !g_ny || !g_r_pad || !g_y_pad || !flags || B < 0 || N < 1)
        return DHTS_ERR_INVALID;
    if (g_nu && (!nr || !ny)) return DHTS_ERR_INVALID;
    if (B == 0) return DHTS_OK;
    int ntile = (N + STEP_TILE - 1) / STEP_TILE;
    if ((long long)B * ntile > 2147483647LL) return DHTS_ERR_UNSUPPORTED;
    size_t sm = smem_bytes<T, true>(STEP_TILE + 2, STEP_TILE + 1);
    int rc = set_smem(arz_step_bwd_kernel<T>, sm);
    if (rc) return rc;
    arz_step_bwd_kernel<T><<<B * ntile, STEP_TILE, sm, st>>>(r_pad, y_pad, u_pad, ueq_pad, dx, umax, dt, B, N, ntile, nr,
                                                              ny, g_nr, g_ny, g_nu, g_r_pad, g_y_pad, flags);
    return launch_status();
}

}  // namespace dhts

// ------------------------------------------------------------------ C ABI (include/dhts.h)

#define DHTS_ARZ_API(SUF, T)                                                                                           \
    DHTS_EXPORT int dhts_arz_step_fwd_##SUF(const T* r_pad, const T* y_pad, const T* u_pad, const T* ueq_pad,          \
                                            const T* dx, const T* umax, T dt, int B, int N, T* nr, T* ny, T* nu,       \
                                            int* case_out, int* flags, void* stream) {                                 \
        return dhts::arz_step_fwd<T>(r_pad, y_pad, u_pad, ueq_pad, dx, umax, dt, B, N, nr, ny, nu, case_out, flags,    \
                                     (cudaStream_t)stream);                                                            \
    }                                                                                                                  \
    DHTS_EXPORT int dhts_arz_step_bwd_##SUF(const T* r_pad, const T* y_pad, const T* u_pad, const T* ueq_pad,          \
                                            const T* dx, const T* umax, T dt, int B, int N, const T* nr, const T* ny,  \
                                            const T* g_nr, const T* g_ny, const T* g_nu, T* g_r_pad, T* g_y_pad,       \
                                            int* flags, void* stream) {                                                \
        return dhts::arz_step_bwd<T>(r_pad, y_pad, u_pad, ueq_pad, dx, umax, dt, B, N, nr, ny, g_nr, g_ny, g_nu,       \
                                     g_r_pad, g_y_pad, flags, (cudaStream_t)stream);                                   \
    }

// C ABI
DHTS_ARZ_API(f64, double)
DHTS_ARZ_API(f32, float)
// end C ABI
