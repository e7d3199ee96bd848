// ARZ macroscopic lane kernels for sm_100a (K1 forward, K2 adjoint).
//
//  * arz_step_{fwd,bwd}_kernel   one Godunov step over B lanes x N cells, tiled:
//    each CTA derives the records of a tile of cells plus a one-cell halo per side
//    into shared memory (coalesced loads), solves the tile's interfaces once, then
//    updates.  The same per-cell records and interface math as the fused rollouts
//    (dhts_arz_lean.cuh), so a step from the same state gives the rollout's first
//    step bit for bit.  This is the operator behind the reference's per-step
//    autograd contract dMacroForwardLayer (road/lane/dmacro_lane.py:234-310).
//  * the fused T-step rollouts live in arz_rollout.cu.
//
// No tensor cores: nothing here is a contraction (BASELINE.json north_star).
#include "dhts_arz_lean.cuh"
#include "dhts_api.h"

namespace dhts {

constexpr int STEP_TILE = 256;
constexpr int STEP_P = STEP_TILE + 2;     // padded cells of a tile
// CTAs per SM the register allocation must allow: the parent kernels' occupancy (fp64 forward 6, fp32 8; fp64 adjoint 5,
// where the compiler's own allocation already gives it).  Without the bound the fp64 forward took 46 registers (5 CTAs)
// and the fp32 adjoint 36 (6 CTAs), 7 % and 15 % slower at 8192 lanes x 1024 cells.
template <typename T, bool ADJ> constexpr int step_min_ctas() { return sizeof(T) == 4 ? 8 : (ADJ ? 5 : 6); }

// Records in shared memory field by field, [NF][STEP_P]: consecutive threads touch consecutive words.
template <typename T, int NF> __device__ __forceinline__ void st_rec(T (*s)[STEP_P], int q, const T* a) {
#pragma unroll
    for (int f = 0; f < NF; f++) s[f][q] = a[f];
}
template <typename T, int NF> __device__ __forceinline__ void ld_rec(const T (*s)[STEP_P], int q, T* a) {
#pragma unroll
    for (int f = 0; f < NF; f++) a[f] = s[f][q];
}

// ------------------------------------------------------------------ single step, tiled

template <typename T>
__global__ void __launch_bounds__(STEP_TILE, step_min_ctas<T, false>())
arz_step_fwd_kernel(const T* __restrict__ r_pad, const T* __restrict__ y_pad, const T* __restrict__ u_pad,
                    const T* __restrict__ ueq_pad, const T* __restrict__ dx, const T* __restrict__ umax_, T dt, int B,
                    int N, int ntile, T* __restrict__ nr, T* __restrict__ ny, T* __restrict__ nu,
                    int* __restrict__ case_out, int* __restrict__ flags) {
    __shared__ T rec[RF_FWD][STEP_P];     // FRec of every padded cell
    __shared__ T ys[STEP_P];
    __shared__ T flux[2][STEP_P - 1];
    const int b = blockIdx.x / ntile, tile = blockIdx.x % ntile;
    const int c0 = tile * STEP_TILE;
    const int nc = min(STEP_TILE, N - c0);
    const LaneK<T> k = make_lanek<T>(umax_[b], dx[b], dt);
    const size_t base = (size_t)b * (N + 2) + c0;
    for (int q = threadIdx.x; q < nc + 2; q += STEP_TILE) {
        const T y = y_pad[base + q];
        T a[RF_FWD];
        pack(frec_stored<T>(r_pad[base + q], y, u_pad[base + q], ueq_pad ? ueq_pad[base + q] : T(0), ueq_pad != nullptr, k), a);
        st_rec<T, RF_FWD>(rec, q, a);
        ys[q] = y;
    }
    __syncthreads();
    bool bad = false;
    for (int i = threadIdx.x; i < nc + 1; i += STEP_TILE) {
        T a[RF_FWD];
        ld_rec<T, RF_FWD>(rec, i, a);
        const FRec<T> L = unpack_f(a);
        const T Rr = rec[0][i + 1], Rus = rec[1][i + 1];
        // the sufficient per-cell tests of the rollouts (dhts_arz_lean.cuh, CFL) rest on a fresh u_eq in w; a stored u_eq
        // (ueq_pad) may be stale, so with one the exact test runs at every interface
        if (ueq_pad || !cell_speed_ok(L.us, L.w, k) || !cell_speed_ok(Rus, rec[3][i + 1], k))
            bad |= cfl_exact_bad(L.r, L.us, L.sq, L.w, Rr, Rus, k, dt);
        bool isL, isM;
        fflux_x<T>(L, Rr, Rus, k, flux[0][i], flux[1][i], isL, isM);
        if (case_out) case_out[(size_t)b * (N + 1) + c0 + i] = isL ? 0 : (isM ? 1 : 2);
    }
    __syncthreads();
    for (int j = threadIdx.x; j < nc; j += STEP_TILE) {
        const T r = fma(flux[0][j] - flux[0][j + 1], k.cc, rec[0][j + 1]);
        const T y = fma(flux[1][j] - flux[1][j + 1], k.cc, ys[j + 1]);
        const size_t o = (size_t)b * N + c0 + j;
        nr[o] = r; ny[o] = y; nu[o] = compute_u(r, y, k.umax);
    }
    if (bad) atomicOr(flags, FLAG_CFL);
}

template <typename T>
__global__ void __launch_bounds__(STEP_TILE, step_min_ctas<T, true>())
arz_step_bwd_kernel(const T* __restrict__ r_pad, const T* __restrict__ y_pad, const T* __restrict__ u_pad,
                    const T* __restrict__ ueq_pad, const T* __restrict__ dx, const T* __restrict__ umax_, T dt, int B,
                    int N, int ntile, const T* __restrict__ nr, const T* __restrict__ ny,
                    const T* __restrict__ g_nr, const T* __restrict__ g_ny, const T* __restrict__ g_nu,
                    T* __restrict__ g_r_pad, T* __restrict__ g_y_pad, int* __restrict__ flags) {
    __shared__ T rec[RF_ADJ][STEP_P];     // ARec and adjoint (gr, gy) of every padded cell
    __shared__ T ab[4][STEP_P - 1];       // per interface: A^T w (left cell), B^T w (right cell)
    const int b = blockIdx.x / ntile, tile = blockIdx.x % ntile;
    const int c0 = tile * STEP_TILE;
    const int nc = min(STEP_TILE, N - c0);
    const int P = N + 2;
    const LaneK<T> k = make_lanek<T>(umax_[b], dx[b], dt);
    const size_t base = (size_t)b * P + c0;
    for (int q = threadIdx.x; q < nc + 2; q += STEP_TILE) {
        const int j = c0 + q;   // padded index; updated cells are 1..N
        T gr = T(0), gy = T(0);
        if (j >= 1 && j <= N) {
            const size_t o = (size_t)b * N + j - 1;
            gr = g_nr[o]; gy = g_ny[o];
            if (g_nu) {   // nu = compute_u(nr, ny) is produced inside the operator
                T dr, dy; du_dry(nr[o], ny[o], k.umax, dr, dy);
                const T gu = g_nu[o]; gr += gu * dr; gy += gu * dy;
            }
        }
        T a[RF_ADJ];
        pack(arec_stored<T>(r_pad[base + q], y_pad[base + q], u_pad[base + q], ueq_pad ? ueq_pad[base + q] : T(0),
                            ueq_pad != nullptr, k), gr, gy, a);
        st_rec<T, RF_ADJ>(rec, q, a);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < nc + 1; i += STEP_TILE) {
        T a[RF_ADJ], c[RF_ADJ];
        ld_rec<T, RF_ADJ>(rec, i, a);
        ld_rec<T, RF_ADJ>(rec, i + 1, c);
        aflux<T>(unpack_a(a), unpack_a(c), c[RF_ADJ - 2] - a[RF_ADJ - 2], c[RF_ADJ - 1] - a[RF_ADJ - 1], k, ab[0][i], ab[1][i], ab[2][i], ab[3][i]);
    }
    __syncthreads();
    bool bad = false;
    for (int j = threadIdx.x; j < nc; j += STEP_TILE) {
        const int q = j + 1;
        const T gr = fma(k.cc, ab[0][q] + ab[2][q - 1], rec[RF_ADJ - 2][q]);
        const T gy = fma(k.cc, ab[1][q] + ab[3][q - 1], rec[RF_ADJ - 1][q]);
        bad |= t_isnan(gr) || t_isnan(gy);
        g_r_pad[base + q] = gr; g_y_pad[base + q] = gy;
    }
    if (threadIdx.x == 0) {
        if (tile == 0) {
            const T gr = k.cc * ab[0][0], gy = k.cc * ab[1][0];
            bad |= t_isnan(gr) || t_isnan(gy);
            g_r_pad[(size_t)b * P] = gr; g_y_pad[(size_t)b * P] = gy;
        }
        if (tile == ntile - 1) {
            const T gr = k.cc * ab[2][nc], gy = k.cc * ab[3][nc];
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
    arz_step_fwd_kernel<T><<<B * ntile, STEP_TILE, 0, st>>>(r_pad, y_pad, u_pad, ueq_pad, dx, umax, dt, B, N, ntile, nr,
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
    arz_step_bwd_kernel<T><<<B * ntile, STEP_TILE, 0, st>>>(r_pad, y_pad, u_pad, ueq_pad, dx, umax, dt, B, N, ntile, nr,
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
