// ARZ (Aw-Rascle-Zhang) device primitives shared by every kernel: flags, constants, the branch-free
// reciprocal / square roots, and the closures u_eq, compute_u and the derivative of compute_u.  The
// per-cell records, the Riemann solver and its adjoint are in dhts_arz_lean.cuh.
//
// Behaviour restated from the reference (file:line relative to its checkout):
//   model/macro/_arz.py:121-149      u_eq, u_eq', compute_u, compute_y
// gamma is the module constant 0.5 (no caller overrides it), so r^gamma =
// sqrt(r), r^(gamma-1) = 1/sqrt(r), x^(1/gamma) = x*x.
#pragma once
#include <cuda_runtime.h>

namespace dhts {

constexpr int FLAG_CFL = 1;        // _macro_lane.py:141-146 assert would fire
constexpr int FLAG_NAN_GRAD = 2;   // dmacro_lane.py:308 assert would fire
constexpr int FLAG_COLLISION = 4;  // _micro_lane.py:151-162 print-and-continue

template <typename T> __device__ __forceinline__ T t_sqrt(T x);
template <> __device__ __forceinline__ double t_sqrt<double>(double x) { return sqrt(x); }
template <> __device__ __forceinline__ float t_sqrt<float>(float x) { return sqrtf(x); }
// fabs folds into the |x| operand modifier of the consuming instruction (a compare-and-select does not)
__device__ __forceinline__ double t_abs(double x) { return fabs(x); }
__device__ __forceinline__ float t_abs(float x) { return fabsf(x); }

// fp64 constants that are not 32-bit immediates can live in constant memory: an FP64 instruction takes a constant-bank operand
// for free, whereas a literal costs two moves into a register pair every time the compiler rematerialises it (it does, under the
// lane rollouts' register caps).  Only translation units that define DHTS_CONSTANT_BANK_LITERALS get this (arz_rollout.cu: the
// forward sweep gains 2 %); elsewhere the compiler hoists the constant loads into registers instead -- the macro-network forward
// kernel went from 62 to 104 registers and lost a third of its occupancy with it (r3f / r3k) -- so the default is literals.
#ifdef DHTS_CONSTANT_BANK_LITERALS
static __constant__ double dhts_kd[5] = {1e-5, 316.22776601683796 /* 1/sqrt(1e-5) */, 0.375, 0.5 / 1.5, 0.0031622776601683794 /* sqrt(1e-5) */};
#define DHTS_KD(i, lit) dhts_kd[i]
#else
#define DHTS_KD(i, lit) (lit)
#endif
template <typename T> struct KC;
template <> struct KC<double> {
    static __device__ __forceinline__ double eps() { return DHTS_KD(0, 1e-5); }
    static __device__ __forceinline__ double rsqrt_eps() { return DHTS_KD(1, 316.22776601683796); }
    static __device__ __forceinline__ double c375() { return DHTS_KD(2, 0.375); }
    static __device__ __forceinline__ double third() { return DHTS_KD(3, 0.5 / 1.5); }
    static __device__ __forceinline__ double sqrt_eps() { return DHTS_KD(4, 0.0031622776601683794); }
};
template <> struct KC<float> {
    static __device__ __forceinline__ float eps() { return 1e-5f; }
    static __device__ __forceinline__ float rsqrt_eps() { return 316.22776601683796f; }
    static __device__ __forceinline__ float c375() { return 0.375f; }
    static __device__ __forceinline__ float third() { return 0.5f / 1.5f; }
    static __device__ __forceinline__ float sqrt_eps() { return 0.0031622776601683794f; }
};

// Branch-free 1/sqrt(x) and 1/x for well-scaled positive x (densities, gaps): hardware
// approximation (MUFU.RSQ64H / MUFU.RCP64H, ~2^-22) refined by one cubic step to ~1 ulp.  The library
// sqrt()/division carry special-case slow paths and long dependent Newton chains that
// dominated the stall profile (profiles/r1a, r1b); parity has >6 digits of headroom.
template <typename T> __device__ __forceinline__ T f_rsqrt(T x);
template <> __device__ __forceinline__ double f_rsqrt<double>(double x) {
    double y;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
    double e = fma(-(x * y), y, 1.0);                 // 1 - x y^2
    return fma(y, e * fma(KC<double>::c375(), e, 0.5), y);         // Halley step: error^3 -> below 1 ulp
}
template <> __device__ __forceinline__ float f_rsqrt<float>(float x) { return rsqrtf(x); }
// the same with the 0.375 as a literal (adjoint kernels: there the compiler does better with literals, see KC)
template <typename T> __device__ __forceinline__ T f_rsqrt_lit(T x) { return f_rsqrt<T>(x); }
template <> __device__ __forceinline__ double f_rsqrt_lit<double>(double x) {
    double y;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
    double e = fma(-(x * y), y, 1.0);
    return fma(y, e * fma(0.375, e, 0.5), y);
}
template <typename T> __device__ __forceinline__ T f_rcp(T x);
template <> __device__ __forceinline__ double f_rcp<double>(double x) {
    double y;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
    double e = fma(-x, y, 1.0);
    return fma(y, fma(e, e, e), y);                   // y (1 + e + e^2): error^3 -> below 1 ulp
}
template <> __device__ __forceinline__ float f_rcp<float>(float x) { return __frcp_rn(x); }
// sqrt(x), x > 0 and well scaled: s0 = x y0 with the hardware seed y0 ~ rsqrt(x) (2^-22), then two coupled Newton
// steps s <- s + (x - s^2) (y0 / 2); the error goes 2^-22 -> 2^-44 -> below the rounding of the last fma.  6
// dependent fp64 operations instead of 9 for "Halley rsqrt, multiply, correct".
template <typename T> __device__ __forceinline__ T f_sqrt_pos(T x);
template <> __device__ __forceinline__ double f_sqrt_pos<double>(double x) {
    double y;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
    const double h = 0.5 * y;
    double s = x * y;
    s = fma(fma(-s, s, x), h, s);
    return fma(fma(-s, s, x), h, s);
}
template <> __device__ __forceinline__ float f_sqrt_pos<float>(float x) {
    float y = rsqrtf(x);
    float s = x * y;
    return fmaf(fmaf(-s, s, x), y * 0.5f, s);
}
template <typename T> __device__ __forceinline__ T t_max(T a, T b) { return a > b ? a : b; }
template <typename T> __device__ __forceinline__ bool t_isnan(T x) { return !(x == x); }

#define DHTS_EPS (KC<T>::eps())
#define DHTS_RSQRT_EPS (KC<T>::rsqrt_eps())   // 1/sqrt(1e-5)
#define DHTS_EPS_LIT (T(1e-5))
#define DHTS_RSQRT_EPS_LIT (T(316.22776601683796))

// u_eq(r) = u_max (1 - (max(r,0)+eps)^gamma)                    _arz.py:133-138
template <typename T> __device__ __forceinline__ T u_eq(T r, T umax) {
    return umax * (T(1) - f_sqrt_pos(t_max(r, T(0)) + DHTS_EPS));      // argument >= eps: branch-free sqrt (<= 1 ulp)
}
// compute_u(r, y)                                               _arz.py:126-131
template <typename T> __device__ __forceinline__ T compute_u(T r, T y, T umax) {
    T rc = t_max(r, DHTS_EPS);
    return y * f_rcp(rc) + umax * (T(1) - f_sqrt_pos(rc + DHTS_EPS));  // rc >= eps: no IEEE division / sqrt slow paths
}

// d compute_u / d(r, y) as autograd differentiates set_r_y OUTSIDE the
// reference's Function (_arz.py:88-92,126-138): the TRUE derivative of
// y/max(r,eps) + u_max (1 - (max(r,eps)+eps)^gamma).
template <typename T> __device__ __forceinline__ void du_dry(T r, T y, T umax, T& du_dr, T& du_dy) {
    if (r >= DHTS_EPS) {
        T ri = f_rcp(r);
        du_dy = ri;
        du_dr = -y * ri * ri - T(0.5) * umax * f_rsqrt(r + DHTS_EPS);
    } else {
        du_dy = T(1) / DHTS_EPS;
        du_dr = T(0);
    }
}

}  // namespace dhts
