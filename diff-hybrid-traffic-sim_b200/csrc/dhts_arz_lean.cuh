// ARZ per-cell records, Riemann solver and its adjoint, for every ARZ kernel: the single step
// (arz_kernels.cu), the fused lane rollouts (arz_rollout.cu) and the network rollouts (dhts_net_if.cuh).
// Everything that depends on ONE cell is evaluated once per cell, in its record; an interface only
// does what couples two cells.
//
// Reference behaviour restated (file:line relative to the reference checkout):
//   model/macro/_arz.py:121-149,155-199,212-332   closures, candidate states, case tree
//   road/lane/_macro_lane.py:83-146               Godunov update, CFL assert
//   model/macro/darz.py:12-233                    dL / dM / dC, flux_prime
//   road/lane/dmacro_lane.py:96-132,277-310       Jacobian band and its VJP
//
// Forward.  The interface flux is selected, not the interface state: for outcome Q_L it is
// (r uc, y uc) of the left cell (per-cell), otherwise (r0 u0, y0 u0) of Q_M / Q_C.  The case tree
// is BRANCH-FREE: with a 86/9/5 % outcome mix nearly every warp holds all three outcomes, so a
// divergent tree executes every path anyway while blocking instruction-level overlap between the
// independent cells of a thread.
//
// CFL.  The reference asserts dt < dx / max(|s|, 1e-5) for two wave speeds per interface
// (_macro_lane.py:137-146), i.e. |s| < dx/dt =: V.  Every non-shock speed is an average of
// u, w = u_max + u - u_eq and lambda_0 = u - (u_max/2) sqrt(r) of the two cells, so two
// per-cell tests (|u| < V/4, |w| < V/4, which bound (u_max/2) sqrt(r) too) imply them.  The shock
// speed (u_L > u_R, r_L >= eps) is s = fd / max(r_m - r_L, eps) with fd = r_m u_R - r_L u_L and
// r_m - r_L = (du/u_max)(2 sqrt(r_L) + du/u_max), du = u_L - u_R > 0, hence
//   fd / (r_m - r_L) = u_R - r_L u_max / (2 sqrt(r_L) + du/u_max),   |.| <= |u_R| + (u_max/2) sqrt(r_L) < V/2,
// and clamping the denominator up to eps only shrinks |s|: the same two per-cell tests cover it.
// Only when one of these SUFFICIENT tests fails (never in a run the reference would accept) is the
// exact per-branch evaluation done (cfl_exact_bad; it evaluates dt < dx / max(|s|, 1e-5) as
// dt * max(|s|, 1e-5) < dx, with no division).
//
// Adjoint.  Not a stored Jacobian band: with A_i = F'(Q0_i) dQ0_i/dQ_left and
// B_i = F'(Q0_i) dQ0_i/dQ_right per interface i, and w_i = g_{i+1} - g_i,
//   gbar_j = g_j + c (A_j^T w_j + B_{j-1}^T w_{j-1})           (SURVEY A.3)
// which is algebraically the band-transpose product of dmacro_lane.py:293-303.  With
// z = F'(Q0)^T w, k = (u0 - u_eq0) - r0 u_eq'(r0), s = z0 + k z1 and a = 2 sqrt(r0), the
// products dQ0/dQ_L^T z and dQ0/dQ_R^T z of darz.py collapse to
//   Q_L:  A^T w = F'(cell L)^T w                       B^T w = 0
//   Q_M:  A^T w = (s a / u_max) P_L                    B^T w = (r0 z1 - s a / u_max) D_R
//   Q_C:  A^T w = (s a / (1.5 u_max) + r0 z1 / 3) P_L  B^T w = 0
// where P_L = (-y/r^2, 1/r) of the left cell (du_L/dQ_L plus the r^(gamma-1) term, which
// cancels u_eq'(r_L)) and D_R = (du_R/dr_R, du_R/dy_R) = (-y/r^2 + u_eq'(r), 1/r) of the
// right cell.  All u_eq' use the reference's convention -u_max gamma max(r,eps)^(gamma-1).
#pragma once
#include "dhts_arz.cuh"

namespace dhts {

template <typename T> struct LaneK {
    T umax, inv_umax, inv15, dx, cc;   // cc = dt / dx
    T hum;                             // u_max / 2
    T v4, vmax, veps;                  // V/4, V = dx/dt, V * 1e-5
};

template <typename T> __host__ __device__ __forceinline__ LaneK<T> make_lanek(T umax, T dx, T dt) {
    LaneK<T> k;
    k.umax = umax; k.inv_umax = T(1) / umax; k.inv15 = T(1) / (T(1.5) * umax); k.dx = dx; k.cc = dt / dx;
    k.hum = T(0.5) * umax;
    k.vmax = dx / dt; k.v4 = T(0.25) * k.vmax;
    k.veps = k.vmax * T(1e-5);
    return k;
}

// Conservative "may be below eps" test on the integer pipe (the high word of a double orders like the value; a
// tie with the high word of eps counts as "maybe").  Used only to choose between the general sweep and the
// vacuum-free one, so a false positive costs time, never correctness.
__device__ __forceinline__ bool maybe_vac(double r) { return __double2hiint(r) <= 0x3EE4F8B5; }   // 1e-5 = 0x3EE4F8B5'88E368F1
__device__ __forceinline__ bool maybe_vac(float r) { return __float_as_int(r) <= __float_as_int(1e-5f); }

// ---------------------------------------------------------------------------- forward
constexpr int RF_FWD = 6;
template <typename T> struct FRec { T r, us, sq, w, fr, fy; };   // fr, fy: flux if this cell is the Q_L outcome

template <typename T> __device__ __forceinline__ void pack(const FRec<T>& c, T* a) {
    a[0] = c.r; a[1] = c.us; a[2] = c.sq; a[3] = c.w; a[4] = c.fr; a[5] = c.fy;
}
template <typename T> __device__ __forceinline__ FRec<T> unpack_f(const T* a) {
    FRec<T> c; c.r = a[0]; c.us = a[1]; c.sq = a[2]; c.w = a[3]; c.fr = a[4]; c.fy = a[5];
    return c;
}

// sufficient per-cell part of the CFL test (see header); false also for NaN.  w - us = u_max - u_eq >=
// u_max sqrt(r), so |us|, |w| < V/4 also bound (u_max/2) sqrt(r) by V/4.
template <typename T> __device__ __forceinline__ bool cell_speed_ok(T us, T w, const LaneK<T>& k) {
    return (t_abs(us) < k.v4) && (t_abs(w) < k.v4);
}

// Per-cell record.  STORED: the cell carries an explicitly stored speed (ghosts, set_r_u at step 0).
// Cells below eps need fix_vacuum afterwards (u_eq(r) = u_max(1 - sqrt(max(r,0)+eps)) differs from the clamped one).
// VAC = false: the caller guarantees r >= eps (no clamp, no vacuum handling).
template <typename T, bool STORED, bool VAC = true>
__device__ __forceinline__ FRec<T> fderive(T r, T y, T us_in, const LaneK<T>& k) {
    FRec<T> c;
    const T rc = VAC ? t_max(r, DHTS_EPS) : r;
    const T rs = f_rsqrt(rc);
    const T ri = rs * rs;
    const T se = f_sqrt_pos(rc + DHTS_EPS);
    const T ueqc = fma(-k.umax, se, k.umax);           // u_eq at the clamped r (compute_u, _arz.py:126-131)
    // every multiply-add of the step is an EXPLICIT fma (or has no product feeding a sum): the compiler's own contraction
    // differs between the kernels this is inlined into, and the segment recompute of the adjoint must reproduce the
    // forward kernel's states bit for bit (tests/test_fullsize_gpu.py: gradients do not depend on ckpt_every)
    const T uc = fma(y, ri, ueqc);
    c.r = r; c.sq = rc * rs;
    c.us = STORED ? us_in : uc;
    c.w = STORED ? ((k.umax + us_in) - ueqc) : fma(y, ri, k.umax);   // u_max + u - u_eq(r)
    c.fr = r * uc; c.fy = y * uc;                       // Q_L re-derives u from (r, y), _arz.py:155-165
    return c;
}
template <typename T> __device__ __forceinline__ T w_vacuum(T r, T us, const LaneK<T>& k) {
    return fma(-k.umax, T(1) - f_sqrt_pos(t_max(r, T(0)) + DHTS_EPS), k.umax + us);
}
// Record of a cell with an explicitly stored speed us, vacuum fix-up included: ghosts built by from_r_u (_arz.py:74-80),
// cells set by set_r_u (:82-86), network cells (nu = compute_u(nr, ny) is stored).  have_ueq: the cell also carries a
// stored u_eq, which then enters w (stale on cells a micro->macro deposit rewrote, conversion.py:157-167).
template <typename T>
__device__ __forceinline__ FRec<T> frec_stored(T r, T y, T us, T ueq_stored, bool have_ueq, const LaneK<T>& k) {
    FRec<T> f = fderive<T, true>(r, y, us, k);
    if (have_ueq) f.w = k.umax + us - ueq_stored;
    else if (r < DHTS_EPS) f.w = w_vacuum(r, us, k);
    return f;
}

// Outcome predicates of the case tree (_arz.py:225-322), shared by forward and adjoint.
template <typename T> struct Tree { bool isL, isM, shock; T b, sc, q, rm, fd; };

template <typename T, bool VAC = true>
__device__ __forceinline__ Tree<T> case_tree(T Lr, T Lus, T Lsq, T Lw, T Rr, T Rus, const LaneK<T>& k) {
    Tree<T> t;
    const bool vacL = VAC && Lr < DHTS_EPS, vacR = VAC && Rr < DHTS_EPS;
    const T du = Lus - Rus;
    const bool same = t_abs(du) < DHTS_EPS;
    const bool shock = du > T(0);
    t.shock = shock;
    const bool rare = Lw > Rus;
    const bool l0 = fma(-k.hum, Lsq, Lus) >= T(0);                 // lambda_0(L) = u - (u_max/2) sqrt(r)
    t.b = fma(du, k.inv_umax, Lsq);                                // Q_M: r_m = b^2
    t.rm = t.b * t.b;
    t.fd = fma(t.rm, Rus, -(Lr * Lus));                            // numerator of the shock speed
    const T rootm = (t.rm >= DHTS_EPS) ? t_abs(t.b) : t.rm * DHTS_RSQRT_EPS;
    const bool m_neg = fma(-k.hum, rootm, Rus) <= T(0);            // lambda_0(Q_M) <= 0
    t.sc = fma(k.umax, Lsq, Lus);                                  // Q_C: r_c = q^2, u_c = sc / 3
    t.q = t.sc * k.inv15;
    // bitwise, not short-circuit: `||` / `&&` made the compiler branch around the lambda_0(Q_M) chain (a divergent
    // 10-instruction block per interface that also splits the sweep into small basic blocks)
    const bool fd_ok = t.fd >= T(0);
    const bool tailL = (shock & fd_ok) | (!shock & l0);
    t.isL = vacL | (vacR ? l0 : (same | tailL));
    t.isM = !t.isL & !vacR & (shock | (rare & m_neg));
    return t;
}

// Exact CFL test of one interface, evaluated only after a sufficient test failed.
template <typename T>
__device__ __forceinline__ bool cfl_exact_bad(T Lr, T Lus, T Lsq, T Lw, T Rr, T Rus, const LaneK<T>& k, T dt) {
    const bool vacL = Lr < DHTS_EPS, vacR = Rr < DHTS_EPS;
    const T du = Lus - Rus;
    const bool same = t_abs(du) < DHTS_EPS, shock = du > T(0), rare = Lw > Rus;
    const T lam0l = Lus - k.hum * Lsq;
    const T b = Lsq + du * k.inv_umax, rm = b * b;
    const T fd = rm * Rus - Lr * Lus;
    const T den = t_max(rm - Lr, DHTS_EPS);
    const T lam0m = Rus - k.hum * ((rm >= DHTS_EPS) ? t_abs(b) : rm * DHTS_RSQRT_EPS);
    const T s_vac = (lam0l + Lw) * T(0.5), s_rare = (lam0l + lam0m) * T(0.5);
    const bool use_shock = !vacL && !vacR && !same && shock;
    const T s0 = (vacL || (!vacR && same)) ? T(0) : (vacR ? s_vac : (rare ? s_rare : s_vac));
    const T s1 = vacL ? Lus : (vacR ? s_vac : Rus);
    const bool ok1 = dt * t_max(t_abs(s1), T(1e-5)) < k.dx;
    const bool ok0s = dt * t_max(t_abs(fd), T(1e-5) * den) < k.dx * den;
    const bool ok0n = dt * t_max(t_abs(s0), T(1e-5)) < k.dx;
    return !((use_shock ? ok0s : ok0n) && ok1);
}

// Flux through the interface between cell L (record) and a right cell (r, stored speed), and the interface's outcome
// (Q_L, Q_M; neither: Q_C).
// The rollouts store the outcome (forward -> adjoint through HBM): two bits per interface and step.  With them the
// adjoint skips the case tree.  (Storing sqrt(r0 + eps) of the selected state as well -- 8 bytes per cell-step, so that the
// adjoint skips that square root too -- was measured: adjoint 629 -> 580 ms per pass but forward 381 -> 411 ms, the forward
// kernel does not take 24 instead of 16 bytes of writes per cell-step for free.)
template <typename T, bool VAC = true>
__device__ __forceinline__ void fflux_x(const FRec<T>& L, T Rr, T Rus, const LaneK<T>& k, T& fr, T& fy, bool& isL, bool& isM) {
    const Tree<T> t = case_tree<T, VAC>(L.r, L.us, L.sq, L.w, Rr, Rus, k);
    const T root = t.isM ? t.b : t.q;
    const T r0 = root * root;
    const T u0 = t.isM ? Rus : t.sc * KC<T>::third();
    const T ueq = fma(-k.umax, f_sqrt_pos(fma(root, root, DHTS_EPS)), k.umax);
    const T y0 = r0 * (u0 - ueq);
    fr = t.isL ? L.fr : r0 * u0;
    fy = t.isL ? L.fy : y0 * u0;
    isL = t.isL; isM = t.isM;
}
template <typename T, bool VAC = true>
__device__ __forceinline__ void fflux(const FRec<T>& L, T Rr, T Rus, const LaneK<T>& k, T& fr, T& fy) {
    bool isL, isM;
    fflux_x<T, VAC>(L, Rr, Rus, k, fr, fy, isL, isM);
}

// ---------------------------------------------------------------------------- adjoint
constexpr int RF_ADJ = 12;
// r, us, sq, w: case tree;  f00, f10, f11: flux_prime at the cell (Q_L outcome);  plr, ri: P_L;  gr, gy: adjoint
template <typename T> struct ARec { T r, us, sq, w, f00, f10, f11, plr, ri, ueqp; };

template <typename T> __device__ __forceinline__ void pack(const ARec<T>& c, T gr, T gy, T* a) {
    a[0] = c.r; a[1] = c.us; a[2] = c.sq; a[3] = c.w; a[4] = c.f00; a[5] = c.f10; a[6] = c.f11; a[7] = c.plr;
    a[8] = c.ri; a[9] = c.ueqp; a[10] = gr; a[11] = gy;
}
template <typename T> __device__ __forceinline__ ARec<T> unpack_a(const T* a) {
    ARec<T> c; c.r = a[0]; c.us = a[1]; c.sq = a[2]; c.w = a[3]; c.f00 = a[4]; c.f10 = a[5]; c.f11 = a[6];
    c.plr = a[7]; c.ri = a[8]; c.ueqp = a[9];
    return c;
}

// Cells below eps need fix_vacuum_adj afterwards.
template <typename T, bool STORED, bool VAC = true>
__device__ __forceinline__ ARec<T> aderive(T r, T y, T us_in, const LaneK<T>& k) {
    ARec<T> c;
    const T rc = VAC ? t_max(r, DHTS_EPS_LIT) : r;
    const T rs = f_rsqrt_lit(rc);
    const T ri = rs * rs;
    const T se = f_sqrt_pos(rc + DHTS_EPS_LIT);
    const T uf = fma(-k.umax, se, k.umax);
    const T yri = y * ri;
    c.r = r; c.sq = rc * rs; c.ri = ri;
    c.us = STORED ? us_in : fma(y, ri, uf);              // bitwise the forward record (fderive)
    c.w = STORED ? ((k.umax + us_in) - uf) : fma(y, ri, k.umax);
    c.ueqp = -k.hum * rs;                               // u_eq'(max(r,eps)), _arz.py:146-149
    c.plr = -yri * ri;
    c.f00 = fma(rc, c.ueqp, uf);                        // flux_prime at (r, y) with the fresh u_eq(r), darz.py:217-233
    c.f10 = fma(y, c.ueqp, -(yri * yri));
    c.f11 = fma(T(2), yri, uf);
    return c;
}
// r < eps: the fresh u_eq(r) enters w, f00 and f11 (the clamped one stays in us)
template <typename T> __device__ __forceinline__ void fix_vacuum_adj(ARec<T>& c, T y, const LaneK<T>& k) {
    const T om = T(1) - f_sqrt_pos(t_max(c.r, T(0)) + DHTS_EPS_LIT);
    const T uf = k.umax * om;
    c.w = fma(-k.umax, om, k.umax + c.us);              // bitwise w_vacuum
    c.f00 = fma(DHTS_EPS_LIT, c.ueqp, uf);
    c.f11 = fma(T(2), y * c.ri, uf);
}
// the adjoint record of frec_stored
template <typename T>
__device__ __forceinline__ ARec<T> arec_stored(T r, T y, T us, T ueq_stored, bool have_ueq, const LaneK<T>& k) {
    ARec<T> c = aderive<T, true>(r, y, us, k);
    if (r < DHTS_EPS) fix_vacuum_adj(c, y, k);
    if (have_ueq) c.w = k.umax + us - ueq_stored;
    return c;
}

// A^T w -> (par, pay) for the left cell, B^T w -> (pbr, pby) for the right cell (see header), given the interface's outcome
// and the roots of its Q_M / Q_C candidates (b and sc of case_tree).  Uses us, sq, f00, f10, f11, plr, ri of L and us, plr,
// ri, ueqp of R.
template <typename T>
__device__ __forceinline__ void aflux_o(const ARec<T>& L, const ARec<T>& R, T wr, T wy, const LaneK<T>& k, bool isL, bool isM,
                                        T b, T sc, T& par, T& pay, T& pbr, T& pby) {
    const T root = isM ? b : sc * k.inv15;
    const T r0 = root * root;
    const T rootr = t_abs(root);
    const T u0 = isM ? R.us : sc * (T(0.5) / T(1.5));
    const T ueq0 = fma(-k.umax, f_sqrt_pos(fma(root, root, DHTS_EPS_LIT)), k.umax);
    const T g = u0 - ueq0;
    const T y0 = r0 * g;
    // flux_prime at Q0 clamps r at eps: with rootc = sqrt(max(r0, eps)) both clamped quantities follow without a select on
    // constants (1 / sqrt(max(r0, eps)) and max(r0, eps); at r0 < eps they differ from the literal 1 / sqrt(eps), eps by an ulp)
    const T rootc = t_max(rootr, KC<T>::sqrt_eps());
    const T inv_sq = f_rcp(rootc);
    const T rr = rootc * rootc;
    const T ueqp0 = -k.hum * inv_sq;
    const T yr = y0 * (inv_sq * inv_sq);
    const T f00 = fma(rr, ueqp0, ueq0);
    const T f10 = fma(y0, ueqp0, -(yr * yr));
    const T f11 = fma(T(2), yr, ueq0);
    const T z0 = fma(f10, wy, f00 * wr);
    const T z1 = fma(f11, wy, wr);
    const T kk = fma(-r0, ueqp0, g);
    const T s = fma(kk, z1, z0);
    const T sa = s * (T(2) * rootr);
    const T cM = sa * k.inv_umax;
    const T r0z1 = r0 * z1;
    const T cC = fma(sa, k.inv15, r0z1 * (T(0.5) / T(1.5)));
    const T coef = isM ? cM : cC;
    const T zl0 = fma(L.f10, wy, L.f00 * wr);
    const T zl1 = fma(L.f11, wy, wr);
    par = isL ? zl0 : coef * L.plr;
    pay = isL ? zl1 : coef * L.ri;
    const T cB = isM ? (r0z1 - cM) : T(0);
    pbr = cB * (R.plr + R.ueqp);
    pby = cB * R.ri;
}
template <typename T, bool VAC = true>
__device__ __forceinline__ void aflux(const ARec<T>& L, const ARec<T>& R, T wr, T wy, const LaneK<T>& k, T& par,
                                      T& pay, T& pbr, T& pby) {
    const Tree<T> t = case_tree<T, VAC>(L.r, L.us, L.sq, L.w, R.r, R.us, k);
    aflux_o<T>(L, R, wr, wy, k, t.isL, t.isM, t.b, t.sc, par, pay, pbr, pby);
}
// the same with the outcome the forward pass stored (fflux_x): no case tree
template <typename T>
__device__ __forceinline__ void aflux_x(const ARec<T>& L, const ARec<T>& R, T wr, T wy, const LaneK<T>& k, bool isL, bool isM,
                                        T& par, T& pay, T& pbr, T& pby) {
    const T b = fma(L.us - R.us, k.inv_umax, L.sq);                // Q_M: r_m = b^2
    const T sc = fma(k.umax, L.sq, L.us);                          // Q_C: r_c = q^2, u_c = sc / 3
    aflux_o<T>(L, R, wr, wy, k, isL, isM, b, sc, par, pay, pbr, pby);
}
// the mailbox record of that path: the 7 fields aflux_x reads of its LEFT cell + that cell's old adjoint
constexpr int RF_ADJX = 9;
template <typename T> __device__ __forceinline__ void pack_x(const ARec<T>& c, T gr, T gy, T* a) {
    a[0] = c.us; a[1] = c.sq; a[2] = c.f00; a[3] = c.f10; a[4] = c.f11; a[5] = c.plr; a[6] = c.ri; a[7] = gr; a[8] = gy;
}
template <typename T> __device__ __forceinline__ ARec<T> unpack_x(const T* a) {
    ARec<T> c; c.r = T(0); c.w = T(0); c.ueqp = T(0);
    c.us = a[0]; c.sq = a[1]; c.f00 = a[2]; c.f10 = a[3]; c.f11 = a[4]; c.plr = a[5]; c.ri = a[6];
    return c;
}

}  // namespace dhts
