// Fused T-step ARZ rollouts for sm_100a, lanes REGISTER-resident.
//
// Each thread owns C consecutive cells of one lane (state, and in the adjoint
// the running adjoint, live in its registers for the whole rollout).  Per step a
// thread derives its cells' records once, solves the C interfaces to the left of
// its cells in one left-to-right sweep, and needs exactly two neighbour items:
//   - the record of the cell left of its chunk  (from thread t-1, before the sweep)
//   - the flux / A^T w at its right edge         (from thread t+1, after the sweep)
// Both travel by warp shuffle; only the two lanes at a warp edge go through a
// small double-buffered shared-memory mailbox (one __syncthreads per exchange).
// Ghost cells are static per lane (road/network/road_network.py:299-387 with no
// neighbouring macro lane) and live in shared memory.
//
// Forward: state checkpoints every K steps to HBM.  Adjoint: segments walked
// backwards; each is recomputed from its checkpoint while stashing every state
// in a per-CTA scratch (L2-resident), then the flux-difference adjoint of
// dhts_arz_lean.cuh is applied step by step, last to first.
//
// Replaces T x (RoadNetwork.forward -> dMacroLane.forward -> dMacroForwardLayer)
// and the autograd chain through them (example/inverse/_inverse.py:91-99,227;
// road/lane/dmacro_lane.py:68-132,234-310).
#include <cstdint>
#include <type_traits>
#define DHTS_CONSTANT_BANK_LITERALS      // see dhts_arz.cuh (KC)
#include "dhts_arz_lean.cuh"
#include "dhts_api.h"

namespace dhts {

constexpr unsigned FULL = 0xffffffffu;

// ---- TMA bulk copies (cp.async.bulk, SASS UBLKCP) completing on an mbarrier: the adjoint's state ring
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_init_fence() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, unsigned bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
// shared -> global bulk store, tracked by bulk async-groups (SASS UBLKCP.G.S)
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void bulk_s2g(void* dst, const void* src, unsigned bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(smem_u32(src)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N_> __device__ __forceinline__ void bulk_wait_read() {
    asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N_) : "memory");
}
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void mbar_wait(uint64_t* bar, unsigned parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "DHTS_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DHTS_DONE;\n"
        "bra DHTS_WAIT;\n"
        "DHTS_DONE:\n"
        "}" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}

// 64-bit shuffles as two explicit 32-bit ones (keeps the register pairs in place)
__device__ __forceinline__ double shfl_up1(double v) {
    int lo = __shfl_up_sync(FULL, __double2loint(v), 1), hi = __shfl_up_sync(FULL, __double2hiint(v), 1);
    return __hiloint2double(hi, lo);
}
__device__ __forceinline__ float shfl_up1(float v) { return __shfl_up_sync(FULL, v, 1); }
__device__ __forceinline__ double shfl_down1(double v) {
    int lo = __shfl_down_sync(FULL, __double2loint(v), 1), hi = __shfl_down_sync(FULL, __double2hiint(v), 1);
    return __hiloint2double(hi, lo);
}
__device__ __forceinline__ float shfl_down1(float v) { return __shfl_down_sync(FULL, v, 1); }

// value held by thread t-1 -> thread t (shuffle; warp edges through the mailbox). All threads must call.
template <typename T, int NF>
__device__ __forceinline__ void from_left(const T* mine, T* out, T* box, int warp, unsigned lane) {
#pragma unroll
    for (int f = 0; f < NF; f++) out[f] = shfl_up1(mine[f]);
    if (lane == 31) {
#pragma unroll
        for (int f = 0; f < NF; f++) box[warp * NF + f] = mine[f];
    }
    __syncthreads();
    if (lane == 0 && warp > 0) {
#pragma unroll
        for (int f = 0; f < NF; f++) out[f] = box[(warp - 1) * NF + f];
    }
}
// value held by thread t+1 -> thread t
template <typename T, int NF>
__device__ __forceinline__ void from_right(const T* mine, T* out, T* box, int warp, int nwarp, unsigned lane) {
#pragma unroll
    for (int f = 0; f < NF; f++) out[f] = shfl_down1(mine[f]);
    if (lane == 0) {
#pragma unroll
        for (int f = 0; f < NF; f++) box[warp * NF + f] = mine[f];
    }
    __syncthreads();
    if (lane == 31 && warp + 1 < nwarp) {
#pragma unroll
        for (int f = 0; f < NF; f++) out[f] = box[(warp + 1) * NF + f];
    }
}

// Chunk loads / stores.  C > 1 is only planned when every row start is 16-byte aligned (fwd_plan, bwd_plan), so the
// vector forms are unconditional.
template <typename T, int C> struct Chunk;
template <typename T> struct Chunk<T, 1> {
    static __device__ __forceinline__ void ld(const T* __restrict__ p, T* v) { v[0] = p[0]; }
    static __device__ __forceinline__ void st(T* __restrict__ p, const T* v) { p[0] = v[0]; }
};
template <> struct Chunk<double, 2> {
    static __device__ __forceinline__ void ld(const double* __restrict__ p, double* v) {
        double2 a = *reinterpret_cast<const double2*>(p); v[0] = a.x; v[1] = a.y;
    }
    static __device__ __forceinline__ void st(double* __restrict__ p, const double* v) {
        *reinterpret_cast<double2*>(p) = make_double2(v[0], v[1]);
    }
};
template <> struct Chunk<double, 4> {
    static __device__ __forceinline__ void ld(const double* __restrict__ p, double* v) {
        double2 a = reinterpret_cast<const double2*>(p)[0], b = reinterpret_cast<const double2*>(p)[1];
        v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
    }
    static __device__ __forceinline__ void st(double* __restrict__ p, const double* v) {
        reinterpret_cast<double2*>(p)[0] = make_double2(v[0], v[1]);
        reinterpret_cast<double2*>(p)[1] = make_double2(v[2], v[3]);
    }
};
template <> struct Chunk<double, 8> {
    static __device__ __forceinline__ void ld(const double* __restrict__ p, double* v) {
        Chunk<double, 4>::ld(p, v); Chunk<double, 4>::ld(p + 4, v + 4);
    }
    static __device__ __forceinline__ void st(double* __restrict__ p, const double* v) {
        Chunk<double, 4>::st(p, v); Chunk<double, 4>::st(p + 4, v + 4);
    }
};
template <> struct Chunk<float, 2> {
    static __device__ __forceinline__ void ld(const float* __restrict__ p, float* v) {
        float2 a = *reinterpret_cast<const float2*>(p); v[0] = a.x; v[1] = a.y;
    }
    static __device__ __forceinline__ void st(float* __restrict__ p, const float* v) {
        *reinterpret_cast<float2*>(p) = make_float2(v[0], v[1]);
    }
};
template <> struct Chunk<float, 4> {
    static __device__ __forceinline__ void ld(const float* __restrict__ p, float* v) {
        float4 a = *reinterpret_cast<const float4*>(p); v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w;
    }
    static __device__ __forceinline__ void st(float* __restrict__ p, const float* v) {
        *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
    }
};
template <> struct Chunk<float, 8> {
    static __device__ __forceinline__ void ld(const float* __restrict__ p, float* v) {
        Chunk<float, 4>::ld(p, v); Chunk<float, 4>::ld(p + 4, v + 4);
    }
    static __device__ __forceinline__ void st(float* __restrict__ p, const float* v) {
        Chunk<float, 4>::st(p, v); Chunk<float, 4>::st(p + 4, v + 4);
    }
};
template <typename T, int C> __device__ __forceinline__ void load_chunk(const T* __restrict__ p, T* v) { Chunk<T, C>::ld(p, v); }
template <typename T, int C> __device__ __forceinline__ void store_chunk(T* __restrict__ p, const T* v) { Chunk<T, C>::st(p, v); }

// Shared-memory layout of a CTA: per-lane constants, per-lane ghost records, two mailboxes x two parities.
constexpr int GH_F = RF_FWD, GH_A = 10;
template <typename T> struct Shm {
    LaneK<T>* lk;     // [lpc]
    T* ghostF;        // [2][lpc][2][GH_F]   left / right ghost forward records (second copy: per-step ghosts, by step parity)
    T* ghostA;        // [2][lpc][2][GH_A]   left / right ghost adjoint records
    T* boxL;          // [2][nwarp][RF_ADJ]
    T* boxR;          // [2][nwarp][4]
};
// fwd: the forward kernel's layout -- no adjoint ghost records, forward-sized mailbox (keeps the 3-stage, 3-row staging
// ring of a 1024-cell lane under the 74 KB of three CTAs per SM)
template <typename T> __host__ __device__ inline size_t shm_bytes(int lpc, int nwarp, bool fwd = false) {
    return sizeof(LaneK<T>) * lpc +
           sizeof(T) * ((size_t)lpc * 4 * (GH_F + (fwd ? 0 : GH_A)) + (size_t)2 * nwarp * ((fwd ? RF_FWD : RF_ADJ) + 4)) + 16;
}
template <typename T> __host__ __device__ inline size_t ring_offset(int lpc, int nwarp, bool fwd = false) {
    return (shm_bytes<T>(lpc, nwarp, fwd) + 127) / 128 * 128;
}
template <typename T> __device__ __forceinline__ Shm<T> carve_shm(unsigned char* raw, int lpc, int nwarp, bool fwd = false) {
    Shm<T> s;
    s.lk = reinterpret_cast<LaneK<T>*>(raw);
    T* p = reinterpret_cast<T*>(raw + sizeof(LaneK<T>) * lpc);
    s.ghostF = p; p += lpc * 4 * GH_F; s.ghostA = p; p += fwd ? 0 : lpc * 4 * GH_A;
    s.boxL = p; p += 2 * nwarp * (fwd ? RF_FWD : RF_ADJ); s.boxR = p;
    return s;
}

// dx == null: every lane has the geometry `kall` (computed on the host; dx and umax are given together or not at all).
template <typename T>
__device__ __forceinline__ void setup_group(const Shm<T>& s, int lane0, int nl, const T* __restrict__ ghost,
                                            const T* __restrict__ dx, const T* __restrict__ umax_, const LaneK<T>& kall, T dt,
                                            bool fwd = false) {
    for (int l = threadIdx.x; l < nl; l += blockDim.x) s.lk[l] = dx ? make_lanek<T>(umax_[lane0 + l], dx[lane0 + l], dt) : kall;
    for (int e = threadIdx.x; e < nl * 2 && ghost; e += blockDim.x) {      // ghost == null: per-step ghosts (step_ghost_record)
        int l = e >> 1, side = e & 1;
        const T* g = ghost + ((size_t)(lane0 + l) * 2 + side) * 3;          // (r, y, u) built by from_r_u
        const LaneK<T> k = dx ? make_lanek<T>(umax_[lane0 + l], dx[lane0 + l], dt) : kall;
        // frec_stored / arec_stored with no stored u_eq, spelled out: through them the compiler schedules the fp64 MODE 2,
        // C = 2 adjoint kernel differently
        FRec<T> f = fderive<T, true>(g[0], g[1], g[2], k);
        if (g[0] < DHTS_EPS) f.w = w_vacuum(g[0], f.us, k);
        pack(f, s.ghostF + (l * 2 + side) * GH_F);
        if (fwd) continue;
        ARec<T> a = aderive<T, true>(g[0], g[1], g[2], k);
        if (g[0] < DHTS_EPS) fix_vacuum_adj(a, g[1], k);
        T tmp[RF_ADJ];
        pack(a, T(0), T(0), tmp);
        for (int i = 0; i < GH_A; i++) s.ghostA[(l * 2 + side) * GH_A + i] = tmp[i];
    }
}

// Per-step ghosts (a lane inside a network gets new ghost cells every step, road_network.py:364-387): thread e < 2 nl
// turns the (r, y, u) it prefetched for side e & 1 of lane e >> 1 into that step's records.
template <typename T, bool ADJ>
__device__ __forceinline__ void step_ghost_record(const Shm<T>& s, int e, int lpc, int par, const T* g) {
    const LaneK<T> k = s.lk[e >> 1];
    if (!ADJ) {
        pack(frec_stored<T>(g[0], g[1], g[2], T(0), false, k), s.ghostF + ((size_t)par * lpc * 2 + e) * GH_F);
    } else {
        T tmp[RF_ADJ];
        pack(arec_stored<T>(g[0], g[1], g[2], T(0), false, k), T(0), T(0), tmp);
#pragma unroll
        for (int i = 0; i < GH_A; i++) s.ghostA[((size_t)par * lpc * 2 + e) * GH_A + i] = tmp[i];
    }
}

// One forward step of this thread's chunk (Godunov update, _macro_lane.py:83-114), STREAMED: only the record
// of the last cell is derived up front (the right neighbour needs it); the sweep then derives cell c, solves
// the interface on its left and finishes the update of cell c-1, so that no per-cell array stays live.
// STORED: the cells carry an explicitly stored speed (set_r_u, step 0).  CHECK: evaluate the CFL condition.
// The sweep exists twice: VAC = false is taken when no cell it touches is below eps (every step of a run
// without vacuum) and drops the clamps, the vacuum predicates and the vacuum fix-ups.
template <typename T, bool STORED, bool VAC>
__device__ __forceinline__ FRec<T> fcell(T r, T y, T us, const LaneK<T>& k) {
    FRec<T> c = fderive<T, STORED, VAC>(r, y, us, k);
    if (VAC) {
        if (r < DHTS_EPS) c.w = w_vacuum(r, c.us, k);      // rare
    }
    return c;
}

// XR: also store the outcome of every interface (dhts_arz_lean.cuh) as warp BALLOTS: for the interface on the left of cell c
// of every thread of the warp, xs[c] = (ballot of Q_L, ballot of Q_M) -- one vote per bit and one 8-byte store by lane 0
// instead of per-thread bit assembly; the adjoint (same thread -> cell mapping) tests its lane's bit.
// DEFER (with CHECK): the sufficient CFL tests of the cells are only AND-ed into okL -- no vote, no branch inside the sweep (one
// basic block); the caller votes once per step and runs the exact test from the stored state (cfl_exact_rows).
template <typename T, int C, bool STORED, bool CHECK, bool VAC, bool XR, bool DEFER = false>
__device__ __forceinline__ bool chunk_fwd_sweep(T* r, T* y, const T* us, const FRec<T>& last, FRec<T>& L,
                                                const LaneK<T>& k, T dt, T* f0, T& fpr, T& fpy, bool& okL, uint2* xs,
                                                unsigned lane) {
    bool bad = false;
#pragma unroll
    for (int c = 0; c < C; c++) {
        const FRec<T> cur = (c == C - 1) ? last : fcell<T, STORED, VAC>(r[c], y[c], STORED ? us[c] : T(0), k);
        T fr, fy;
        if (XR) {
            bool isL, isM;
            fflux_x<T, VAC>(L, cur.r, cur.us, k, fr, fy, isL, isM);
            const unsigned bL = __ballot_sync(FULL, isL), bM = __ballot_sync(FULL, isM);
            if (lane == 0) xs[c] = make_uint2(bL, bM);
        } else fflux<T, VAC>(L, cur.r, cur.us, k, fr, fy);
        if (CHECK) {
            const bool okR = cell_speed_ok(cur.us, cur.w, k);
            if (DEFER) okL &= okR;
            else {
                // never in a valid run; the vote makes the branch warp-uniform (no reconvergence bookkeeping around it): every
                // lane then evaluates the exact test, which is what the flag means anyway
                if (__any_sync(FULL, !okL | !okR)) bad |= cfl_exact_bad(L.r, L.us, L.sq, L.w, cur.r, cur.us, k, dt);
                okL = okR;
            }
        }
        if (c == 0) { f0[0] = fr; f0[1] = fy; }
        else {
            r[c - 1] = fma(fpr - fr, k.cc, r[c - 1]);
            y[c - 1] = fma(fpy - fy, k.cc, y[c - 1]);
        }
        fpr = fr; fpy = fy; L = cur;
    }
    return bad;
}

// xs (XR): the C outcome ballot pairs of this thread's WARP in the step's stage of the staging ring.
// DEFER: returns "a sufficient CFL test failed at a cell this thread's interfaces touch" instead of the exact verdict.
template <typename T, int C, bool STORED, bool CHECK, bool XR = false, bool DEFER = false>
__device__ __forceinline__ bool chunk_fwd_step(T* r, T* y, const T* us, bool first_chunk, bool last_chunk,
                                               const LaneK<T>& k, const T* ghostL, const T* ghostR, T dt, T* boxL,
                                               T* boxR, int warp, int nwarp, unsigned lane, uint2* xs = nullptr) {
    // (the last cell's record always takes the vacuum handling: a second vote before the hand-over, so that it could take the
    // vacuum-free form too, was measured -- 350.9 instead of 348.7 ms, r3o)
    const FRec<T> last = fcell<T, STORED, true>(r[C - 1], y[C - 1], STORED ? us[C - 1] : T(0), k);
    T mine[RF_FWD], left[RF_FWD];
    pack(last, mine);
    from_left<T, RF_FWD>(mine, left, boxL, warp, lane);
    FRec<T> L = first_chunk ? unpack_f(ghostL) : unpack_f(left);
    bool okL = CHECK ? cell_speed_ok(L.us, L.w, k) : true;
    bool anyvac = maybe_vac(L.r);
#pragma unroll
    for (int c = 0; c < C; c++) anyvac |= maybe_vac(r[c]);
    T f0[2], fpr = T(0), fpy = T(0);
    bool bad;
    anyvac = __any_sync(FULL, anyvac);            // one variant per warp (a mixed warp would run both, one after the other)
    if (__builtin_expect(anyvac, 0)) bad = chunk_fwd_sweep<T, C, STORED, CHECK, true, XR, DEFER>(r, y, us, last, L, k, dt, f0, fpr, fpy, okL, xs, lane);
    else bad = chunk_fwd_sweep<T, C, STORED, CHECK, false, XR, DEFER>(r, y, us, last, L, k, dt, f0, fpr, fpy, okL, xs, lane);
    // (XR) the outcomes went into the step's stage; this fence -- before the step's second block barrier, after which the bulk
    // store is issued -- also covers the (r, y) rows written at the top of the step
    if (XR) fence_proxy_async();
    T fR[2];
    from_right<T, 2>(f0, fR, boxR, warp, nwarp, lane);
    if (last_chunk) {   // interface with the right ghost cell
        const FRec<T> G = unpack_f(ghostR);
        fflux<T, true>(L, G.r, G.us, k, fR[0], fR[1]);
        if (CHECK) {
            if (DEFER) okL &= cell_speed_ok(G.us, G.w, k);
            else if (!okL || !cell_speed_ok(G.us, G.w, k)) bad |= cfl_exact_bad(L.r, L.us, L.sq, L.w, G.r, G.us, k, dt);
        }
    }
    r[C - 1] = fma(fpr - fR[0], k.cc, r[C - 1]);
    y[C - 1] = fma(fpy - fR[1], k.cc, y[C - 1]);
    return (CHECK && DEFER) ? !okL : bad;
}

// The exact CFL test of one step (_macro_lane.py:137-146) for the interfaces this thread owns -- the one on the left of each of
// its cells, plus the right ghost's for the last chunk -- evaluated from the state BEFORE the step as the staged forward kernel
// keeps it in shared memory (lr, ly: the lane's rows in the step's stage; lu: the stored speeds of step 0 or null).  Only run
// after a sufficient per-cell test failed somewhere in the warp, i.e. never in a run the reference would accept.
template <typename T, int C>
__device__ __noinline__ bool cfl_exact_rows(const T* lr, const T* ly, const T* lu, int kc, bool last_chunk, const LaneK<T>& k,
                                            const T* ghostL, const T* ghostR, T dt) {
    bool bad = false;
    for (int c = 0; c <= C; c++) {
        if (c == C && !last_chunk) break;
        const int i = kc * C + c;                 // interface between cell i - 1 and cell i (i == N: the right ghost)
        FRec<T> L;
        if (i == 0) L = unpack_f(ghostL);
        else {
            L = lu ? fderive<T, true>(lr[i - 1], ly[i - 1], lu[i - 1], k) : fderive<T, false>(lr[i - 1], ly[i - 1], T(0), k);
            if (lr[i - 1] < DHTS_EPS) L.w = w_vacuum(lr[i - 1], L.us, k);
        }
        T Rr, Rus;
        if (c == C) { const FRec<T> G = unpack_f(ghostR); Rr = G.r; Rus = G.us; }
        else {
            const FRec<T> R = lu ? fderive<T, true>(lr[i], ly[i], lu[i], k) : fderive<T, false>(lr[i], ly[i], T(0), k);
            Rr = R.r; Rus = R.us;
        }
        bad |= cfl_exact_bad(L.r, L.us, L.sq, L.w, Rr, Rus, k, dt);
    }
    return bad;
}

// NS > 0 (every state stored, K == 1): the state rows go to HBM through an NS-stage shared-memory staging ring and
// TMA bulk stores issued by one thread -- no per-thread STG, no store address arithmetic, and the state registers
// are free again as soon as the STS has read them.  NS == 0: per-thread vector stores (sparse checkpoints).
// XR (staged mode only): besides (r, y) every state stores the OUTCOME of each interface of the step taken from it -- warp
// ballots, behind the states in `ckpt` -- which lets the adjoint skip the case tree (aflux_x) for a quarter byte per
// cell-step of HBM traffic.
// Outcome rows: C ballot pairs (8 bytes each) per warp and step, i.e. tpl / 32 * C * 8 = N / 4 bytes per lane and step.
__host__ __device__ inline size_t xlane_bytes(int tpl, int C) { return (size_t)(tpl / 32) * C * 8; }
template <typename T> __host__ __device__ inline size_t xrow_elems(int lpc, int tpl, int C) {      // outcome row of a stage, in elements
    return (((size_t)lpc * xlane_bytes(tpl, C) + 15) / 16 * 16) / sizeof(T);
}
// Launch constants of the staged / ring paths, computed once on the host: as kernel parameters they sit in the constant bank
// and cost no instruction where they are used (the step loops re-derived them every step before: ~10 % of the adjoint's
// instructions were 64-bit index arithmetic).
struct RollK {
    int stage_elems;          // one stage of the ring: (r, y) rows of the CTA's lanes + outcome row, in elements
    int y_off, x_off;         // the y rows / the outcome row inside a stage, in elements
    int ring_off;             // byte offset of the ring in the CTA's dynamic shared memory
    long long step_stride;    // 2 B N: one stored state, in elements
    long long x_stride;       // B x xlane_bytes: the outcome rows of one step, in bytes
};
template <typename T> static RollK make_rollk(int B, int N, int C, int lpc, int nwarp, bool fwd, bool xr) {
    RollK k;
    k.y_off = lpc * N; k.x_off = 2 * lpc * N;
    k.stage_elems = 2 * lpc * N + (xr ? (int)xrow_elems<T>(lpc, N / C, C) : 0);
    k.ring_off = (int)ring_offset<T>(lpc, nwarp, fwd);
    k.step_stride = 2LL * B * N;
    k.x_stride = (long long)B * (long long)xlane_bytes(N / C, C);
    return k;
}

// UNI: all lanes share one geometry (dx == umax_ == null) and the kernel reads the lane constants from its PARAMETERS (`kall`,
// constant bank: free operands of the fp64 instructions) instead of keeping them in 12-14 registers per thread.
template <typename T, int C, int MB, int NS, bool TV = false, bool XR = false, bool UNI = false>
__global__ void __launch_bounds__(1024 / (C < 4 ? C : 4), MB) arz_rollout_fwd_reg_kernel(const T* __restrict__ r0, const T* __restrict__ y0,
                                           const T* __restrict__ u0, const T* __restrict__ ghost,
                                           const T* __restrict__ ghost_t,
                                           const T* __restrict__ dx, const T* __restrict__ umax_, const LaneK<T> kall, T dt, int B, int N,
                                           int steps, int K, int lpc, const RollK rk, T* __restrict__ ckpt, T* __restrict__ rT,
                                           T* __restrict__ yT, T* __restrict__ uT, int* __restrict__ flags) {
    extern __shared__ __align__(128) unsigned char raw[];
    const int nwarp = blockDim.x >> 5, warp = threadIdx.x >> 5;
    const unsigned lane = threadIdx.x & 31;
    Shm<T> s = carve_shm<T>(raw, lpc, nwarp, true);
    const int tpl = N / C;                        // threads per lane
    T* stg = reinterpret_cast<T*>(raw + rk.ring_off);     // [NS][(r, y) x lpc * N | outcomes]
    const int l = threadIdx.x / tpl, kc = threadIdx.x - l * tpl;
    const int ngroup = (B + lpc - 1) / lpc;
    bool bad = false;
    for (int grp = blockIdx.x; grp < ngroup; grp += gridDim.x) {
        const int lane0 = grp * lpc, nl = min(lpc, B - lane0);
        const bool active = l < nl;
        const int ll = active ? l : 0;
        __syncthreads();
        setup_group(s, lane0, nl, ghost, dx, umax_, kall, dt, true);
        __syncthreads();
        const LaneK<T> k = UNI ? kall : s.lk[ll];
        const T* gL = s.ghostF + (ll * 2) * GH_F; const T* gR = gL + GH_F;
        const size_t off = (size_t)(lane0 + ll) * N + (size_t)kc * C;
        const size_t soff = (size_t)ll * N + (size_t)kc * C;
        const bool first_chunk = kc == 0, last_chunk = kc == tpl - 1;
        const size_t BN = (size_t)B * N;
        T gq[3] = {T(0), T(0), T(0)};                           // TV: ghost (r, y, u) of the coming step, thread e < 2 nl
        const bool gthread = TV && (int)threadIdx.x < 2 * nl;
        const T* gsrc = TV ? ghost_t + ((size_t)(lane0 + (threadIdx.x >> 1)) * 2 + (threadIdx.x & 1)) * 3 : nullptr;
        if (gthread && steps > 0) { gq[0] = gsrc[0]; gq[1] = gsrc[1]; gq[2] = gsrc[2]; }
        T r[C], y[C];
        load_chunk<T, C>(r0 + off, r); load_chunk<T, C>(y0 + off, y);
        bool lbad = false;
        T* blA = s.boxL; T* blB = s.boxL + nwarp * RF_FWD;        // double-buffered mailboxes, swapped every step
        T* brA = s.boxR; T* brB = s.boxR + nwarp * 4;
        T* ck = ckpt ? ckpt + off : nullptr;                       // next checkpoint slot of this chunk
        T* ckrow = ckpt ? ckpt + (size_t)lane0 * N : nullptr;      // same, start of the group's rows (bulk stores)
        const unsigned rowbytes = (unsigned)((size_t)nl * N * sizeof(T));
        int next_ck = 0;
        if (NS > 0) {
            // Staged path (every state stored, K == 1): running pointers into the staging ring and into `ckpt`, advanced by the
            // launch constants; step 0 (explicitly stored speeds) is peeled so that the loop holds ONE copy of the step.
            T* sp = stg + soff;                                    // this thread's r chunk in the current stage
            uint2* sx = XR ? reinterpret_cast<uint2*>(stg + rk.x_off) + warp * C : nullptr;     // this warp's ballots, same stage
            unsigned char* xrow = XR ? reinterpret_cast<unsigned char*>(ckpt + (size_t)steps * rk.step_stride) + (size_t)lane0 * xlane_bytes(tpl, C) : nullptr;
            const unsigned xbytes = (unsigned)((size_t)nl * xlane_bytes(tpl, C));
            int stg_i = 0;
            T* bl = s.boxL; T* br = s.boxR;
            int flipl = nwarp * RF_FWD, flipr = nwarp * 4;
            for (int t = 0; t < steps; t++) {
                // Stage t % NS is free: its previous bulk store (step t - NS) was waited for by thread 0 at the top of step
                // t - 1, before that step's block barriers.
                if (active) { store_chunk<T, C>(sp, r); store_chunk<T, C>(sp + rk.y_off, y); }
                if (!XR) fence_proxy_async();
                if (threadIdx.x == 0) bulk_wait_read<(NS > 2 ? NS - 2 : 0)>();
                bool sus;       // a sufficient CFL test failed: the exact one runs from the stage's rows (the state before the step)
                if (t == 0 && u0) {
                    T us[C];
                    load_chunk<T, C>(u0 + off, us);
                    sus = chunk_fwd_step<T, C, true, true, XR, true>(r, y, us, first_chunk, last_chunk, k, gL, gR, dt, bl, br, warp, nwarp, lane, sx);
                } else
                    sus = chunk_fwd_step<T, C, false, true, XR, true>(r, y, nullptr, first_chunk, last_chunk, k, gL, gR, dt, bl, br, warp, nwarp, lane, sx);
                if (__builtin_expect(__any_sync(FULL, sus), 0))
                    lbad |= cfl_exact_rows<T, C>(sp - kc * C, sp - kc * C + rk.y_off, (t == 0 && u0) ? u0 + (size_t)(lane0 + ll) * N : nullptr,
                                                 kc, last_chunk, k, gL, gR, dt);
                bl += flipl; flipl = -flipl; br += flipr; flipr = -flipr;
                // every thread has passed the step's block barriers: the stage is complete and fenced
                if (threadIdx.x == 0) {     // thread 0: soff == 0, sp is the stage
                    bulk_s2g(ckrow, sp, rowbytes);
                    bulk_s2g(ckrow + BN, sp + rk.y_off, rowbytes);
                    if (XR) bulk_s2g(xrow, sp + rk.x_off, xbytes);      // outcome ballots: behind the `steps` stored states
                    bulk_commit();
                }
                ckrow += rk.step_stride;
                if (XR) { xrow += rk.x_stride; sx += (size_t)rk.stage_elems * sizeof(T) / sizeof(uint2); }
                sp += rk.stage_elems;
                if (++stg_i == NS) {
                    stg_i = 0; sp -= (size_t)NS * rk.stage_elems;
                    if (XR) sx -= (size_t)NS * rk.stage_elems * sizeof(T) / sizeof(uint2);
                }
            }
            if (threadIdx.x == 0) bulk_wait_read<0>();      // stages are rewritten by the next lane group
        } else
        for (int t = 0; t < steps; t++) {
            if (TV) {       // this step's ghost records (published by the step's first block barrier), then prefetch the next ones
                if (gthread) {
                    step_ghost_record<T, false>(s, threadIdx.x, lpc, t & 1, gq);
                    if (t + 1 < steps) { const T* q = gsrc + (size_t)(t + 1) * B * 6; gq[0] = q[0]; gq[1] = q[1]; gq[2] = q[2]; }
                }
                gL = s.ghostF + ((size_t)(t & 1) * lpc * 2 + ll * 2) * GH_F; gR = gL + GH_F;
            }
            if (ck && t == next_ck) {
                if (active) { store_chunk<T, C>(ck, r); store_chunk<T, C>(ck + BN, y); }
                ck += 2 * BN;
                next_ck += K;
            }
            if (t == 0 && u0) {
                T us[C];
                load_chunk<T, C>(u0 + off, us);
                lbad |= chunk_fwd_step<T, C, true, true>(r, y, us, first_chunk, last_chunk, k, gL, gR, dt, blA, brA, warp, nwarp, lane);
            } else
                lbad |= chunk_fwd_step<T, C, false, true>(r, y, nullptr, first_chunk, last_chunk, k, gL, gR, dt, blA, brA, warp, nwarp, lane);
            T* x = blA; blA = blB; blB = x; x = brA; brA = brB; brB = x;
        }
        bad |= lbad && active;
        if (active) {
            T u[C];
#pragma unroll
            for (int c = 0; c < C; c++) u[c] = (steps == 0 && u0) ? u0[off + c] : compute_u(r[c], y[c], k.umax);
            store_chunk<T, C>(rT + off, r); store_chunk<T, C>(yT + off, y); store_chunk<T, C>(uT + off, u);
        }
    }
    if (NS > 0 && threadIdx.x == 0) bulk_wait_all();
    if (bad) atomicOr(flags, FLAG_CFL);
}

// One adjoint step of this thread's chunk: (gr, gy) <- VJP of the step taken from state (r, y)
// (flux-difference form of dmacro_lane.py:293-303, SURVEY A.3), streamed like the forward step: interface c
// gives A^T w to cell c-1 and B^T w to cell c, so cell c-1 is finished as soon as interface c is done.
// accL / accR collect the ghost adjoints.  VAC as in the forward sweep.
template <typename T, bool STORED, bool VAC>
__device__ __forceinline__ ARec<T> acell(T r, T y, T us, const LaneK<T>& k) {
    ARec<T> c = aderive<T, STORED, VAC>(r, y, us, k);
    if (VAC) {
        if (r < DHTS_EPS) fix_vacuum_adj(c, y, k);         // rare
    }
    return c;
}

// XR: the forward pass stored the outcome of every interface (xs[c]: warp ballots of Q_L / Q_M for the interface on the left
// of cell c; lm = this lane's bit) -> aflux_x.
template <typename T, int C, bool STORED, bool VAC, bool XR>
__device__ __forceinline__ bool chunk_adj_sweep(const T* r, const T* y, const T* us, T* gr, T* gy, const ARec<T>& last,
                                                ARec<T>& L, T& gLr, T& gLy, const LaneK<T>& k, T* a0, T& bpr, T& bpy,
                                                const uint2* xs, unsigned lm) {
    bool nan = false;
#pragma unroll
    for (int c = 0; c < C; c++) {
        const ARec<T> cur = (c == C - 1) ? last : acell<T, STORED, VAC>(r[c], y[c], STORED ? us[c] : T(0), k);
        const T gcr = gr[c], gcy = gy[c];
        T ar, ay, br, by;
        if (XR) { const uint2 w = xs[c]; aflux_x<T>(L, cur, gcr - gLr, gcy - gLy, k, (w.x & lm) != 0, (w.y & lm) != 0, ar, ay, br, by); }
        else aflux<T, VAC>(L, cur, gcr - gLr, gcy - gLy, k, ar, ay, br, by);
        if (c == 0) { a0[0] = ar; a0[1] = ay; }
        else {
            gr[c - 1] = fma(k.cc, ar + bpr, gLr);
            gy[c - 1] = fma(k.cc, ay + bpy, gLy);
        }
        bpr = br; bpy = by; L = cur; gLr = gcr; gLy = gcy;
    }
    return nan;
}

template <typename T, int C, bool STORED, bool XR = false>
__device__ __forceinline__ bool chunk_adj_step(const T* r, const T* y, const T* us, T* gr, T* gy, bool first_chunk,
                                               bool last_chunk, const LaneK<T>& k, const T* ghostL, const T* ghostR,
                                               T* accL, T* accR, T* boxL, T* boxR, int warp, int nwarp, unsigned lane,
                                               const uint2* xs = nullptr) {
    const T rl = r[C - 1];
    // XR: the vacuum handling only concerns how the thread's OWN cells are derived (the hand-over record carries no r), so the
    // warp's vote comes first and covers the last cell too
    bool anyvac = false;
    if (XR) {
#pragma unroll
        for (int c = 0; c < C; c++) anyvac |= maybe_vac(r[c]);
        anyvac = __any_sync(FULL, anyvac);
    }
    ARec<T> last;
    if (!XR || __builtin_expect(anyvac, 0)) last = acell<T, STORED, true>(rl, y[C - 1], STORED ? us[C - 1] : T(0), k);
    else last = acell<T, STORED, false>(rl, y[C - 1], STORED ? us[C - 1] : T(0), k);
    constexpr int NF = XR ? RF_ADJX : RF_ADJ;     // the stored-outcome path hands over a shorter record (no r, no w)
    T mine[NF], left[NF];
    if (XR) pack_x(last, gr[C - 1], gy[C - 1], mine); else pack(last, gr[C - 1], gy[C - 1], mine);
    from_left<T, NF>(mine, left, boxL, warp, lane);
    ARec<T> L = first_chunk ? unpack_a(ghostL) : (XR ? unpack_x(left) : unpack_a(left));
    T gLr = first_chunk ? T(0) : left[NF - 2], gLy = first_chunk ? T(0) : left[NF - 1];   // OLD adjoint of the cell on the left
    T a0[2], bpr = T(0), bpy = T(0);
    if (!XR) {
        anyvac = maybe_vac(L.r) || maybe_vac(rl);
#pragma unroll
        for (int c = 0; c < C - 1; c++) anyvac |= maybe_vac(r[c]);
        anyvac = __any_sync(FULL, anyvac);        // one variant per warp
    }
    bool nan;
    const unsigned lm = 1u << lane;
    if (__builtin_expect(anyvac, 0)) nan = chunk_adj_sweep<T, C, STORED, true, XR>(r, y, us, gr, gy, last, L, gLr, gLy, k, a0, bpr, bpy, xs, lm);
    else nan = chunk_adj_sweep<T, C, STORED, false, XR>(r, y, us, gr, gy, last, L, gLr, gLy, k, a0, bpr, bpy, xs, lm);
    T aR[2];
    from_right<T, 2>(a0, aR, boxR, warp, nwarp, lane);
    if (last_chunk) {   // interface with the right ghost (its updated-state adjoint is zero)
        const ARec<T> G = unpack_a(ghostR);
        T pbr, pby;
        aflux<T, true>(L, G, -gLr, -gLy, k, aR[0], aR[1], pbr, pby);
        accR[0] = fma(k.cc, pbr, accR[0]); accR[1] = fma(k.cc, pby, accR[1]);
    }
    if (first_chunk) { accL[0] = fma(k.cc, a0[0], accL[0]); accL[1] = fma(k.cc, a0[1], accL[1]); }
    gr[C - 1] = fma(k.cc, aR[0] + bpr, gLr);
    gy[C - 1] = fma(k.cc, aR[1] + bpy, gLy);
    return nan;
}

// MODE 0: every state stored, streamed back through the TMA ring;  1: every state stored, register prefetch;
// 2: checkpoint every K steps, segment recompute with an L2-resident stash.  (Separate instantiations so that
// each gets its own register allocation.)
// EXT (MODE 1 only): per-step ghosts ghost_t [steps][B][2][3] with their adjoints g_ghost_t [steps][B][2][2], and g_hist
// [steps][2][B][N], the adjoint of a loss that reads the state BEFORE every step (added once that step's VJP has run).
// XR (MODE 0 only): the forward pass stored the interface outcomes behind the states (see the forward kernel).
template <typename T, int C, int MB, int MODE, bool EXT = false, bool XR = false, bool UNI = false>
__global__ void __launch_bounds__(1024 / (C < 4 ? C : 4), MB) arz_rollout_bwd_reg_kernel(const T* __restrict__ ckpt, const T* __restrict__ u0,
                                           const T* __restrict__ ghost, const T* __restrict__ ghost_t,
                                           const T* __restrict__ g_hist, T* __restrict__ g_ghost_t,
                                           const T* __restrict__ dx,
                                           const T* __restrict__ umax_, const LaneK<T> kall, T dt, int B, int N, int steps, int K, int lpc,
                                           const T* __restrict__ rT, const T* __restrict__ yT,
                                           const T* __restrict__ g_rT, const T* __restrict__ g_yT,
                                           const T* __restrict__ g_uT, T* __restrict__ scratch,
                                           T* __restrict__ g_r0, T* __restrict__ g_y0, T* __restrict__ g_ghost,
                                           int* __restrict__ flags, int ring_ns, const RollK rk) {
    extern __shared__ __align__(128) unsigned char raw[];
    const int nwarp = blockDim.x >> 5, warp = threadIdx.x >> 5;
    const unsigned lane = threadIdx.x & 31;
    Shm<T> s = carve_shm<T>(raw, lpc, nwarp);
    // state ring of the every-state-stored adjoint: ring_ns stages of (r row, y row) of the CTA's lanes, filled by
    // TMA bulk copies that complete on one mbarrier per stage
    T* ring = reinterpret_cast<T*>(raw + rk.ring_off);
    uint64_t* full = reinterpret_cast<uint64_t*>(ring + (size_t)ring_ns * rk.stage_elems);
    if (MODE == 0) {
        if (threadIdx.x == 0) {
            for (int i = 0; i < ring_ns; i++) mbar_init(full + i, 1);
            mbar_init_fence();
        }
        __syncthreads();
    }
    int fill_st = 0, use_st = 0;              // next stage to fill (thread 0) / to consume (all threads)
    unsigned use_par = 0;
    const int tpl = N / C;
    const int l = threadIdx.x / tpl, kc = threadIdx.x - l * tpl;
    const int ngroup = (B + lpc - 1) / lpc;
    const int S = (steps + K - 1) / K;
    const size_t sstride = (size_t)2 * lpc * N;               // one stashed state of the group
    const size_t BN = (size_t)B * N;
    T* scr = scratch + (size_t)blockIdx.x * K * sstride;
    bool bad = false;
    for (int grp = blockIdx.x; grp < ngroup; grp += gridDim.x) {
        const int lane0 = grp * lpc, nl = min(lpc, B - lane0);
        const bool active = l < nl;
        const int ll = active ? l : 0;
        const bool first_chunk = kc == 0, last_chunk = kc == tpl - 1;
        __syncthreads();
        setup_group(s, lane0, nl, ghost, dx, umax_, kall, dt);
        __syncthreads();
        const LaneK<T> k = UNI ? kall : s.lk[ll];
        const T* gLf = s.ghostF + (ll * 2) * GH_F; const T* gRf = gLf + GH_F;
        const T* gLa = s.ghostA + (ll * 2) * GH_A; const T* gRa = gLa + GH_A;
        const size_t off = (size_t)(lane0 + ll) * N + (size_t)kc * C;
        const size_t soff = (size_t)ll * N + (size_t)kc * C;
        T gr[C], gy[C];
        T accL[2] = {T(0), T(0)}, accR[2] = {T(0), T(0)};     // ghost adjoints of this lane (first / last chunk)
        bool nan = false;
        // terminal adjoint; uT = compute_u(rT, yT) is produced inside the operator
#pragma unroll
        for (int c = 0; c < C; c++) {
            gr[c] = g_rT ? g_rT[off + c] : T(0); gy[c] = g_yT ? g_yT[off + c] : T(0);
            if (g_uT) {
                T dr, dy; du_dry(rT[off + c], yT[off + c], k.umax, dr, dy);
                T gu = g_uT[off + c]; gr[c] += gu * dr; gy[c] += gu * dy;
            }
        }
        T* blA = s.boxL; T* blB = s.boxL + nwarp * RF_ADJ;
        T* brA = s.boxR; T* brB = s.boxR + nwarp * 4;
#define DHTS_SWAP_BOXES { T* x_ = blA; blA = blB; blB = x_; x_ = brA; brA = brB; brB = x_; }
        if (MODE == 0) {
            // every state was stored by the forward pass: one thread streams the rows of the CTA's lanes back through
            // the shared-memory ring, ring_ns steps ahead of the arithmetic.  A stage is refilled at the top of the
            // step after the one that consumed it: by then every thread has passed that step's two block barriers,
            // i.e. has finished reading the stage.
            // Running pointers advanced by the launch constants (RollK) instead of per-step index arithmetic.
            const unsigned rowbytes = (unsigned)((size_t)nl * N * sizeof(T));
            const unsigned xbytes = (unsigned)((size_t)nl * xlane_bytes(tpl, C));
            const T* src = ckpt + (size_t)lane0 * N + (size_t)(steps > 0 ? steps - 1 : 0) * rk.step_stride;      // next state to fetch (thread 0)
            const unsigned char* xsrc = reinterpret_cast<const unsigned char*>(ckpt + (size_t)steps * rk.step_stride) +
                                        (size_t)lane0 * xlane_bytes(tpl, C) + (size_t)(steps > 0 ? steps - 1 : 0) * rk.x_stride;
            int issued = 0;
#define DHTS_RING_ISSUE                                                                                  \
            {                                                                                            \
                uint64_t* bar_ = full + fill_st;                                                         \
                T* dst_ = ring + (size_t)fill_st * rk.stage_elems;                                       \
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");                             \
                mbar_expect_tx(bar_, 2 * rowbytes + (XR ? xbytes : 0u));                                 \
                bulk_g2s(dst_, src, rowbytes, bar_);                                                     \
                bulk_g2s(dst_ + rk.y_off, src + BN, rowbytes, bar_);                                     \
                if (XR) bulk_g2s(dst_ + rk.x_off, xsrc, xbytes, bar_);                                   \
                src -= rk.step_stride; xsrc -= rk.x_stride;                                              \
                issued++;                                                                                \
                if (++fill_st == ring_ns) fill_st = 0;                                                   \
            }
            if (threadIdx.x == 0)
                while (issued < ring_ns && issued < steps) DHTS_RING_ISSUE
            const T* rp = ring + (size_t)use_st * rk.stage_elems + soff;        // this thread's r chunk in the stage to consume
            const uint2* xp = XR ? reinterpret_cast<const uint2*>(ring + (size_t)use_st * rk.stage_elems + rk.x_off) + warp * C : nullptr;
            T* bl = s.boxL; T* br = s.boxR;
            int flipl = nwarp * RF_ADJ, flipr = nwarp * 4;
            for (int t = steps - 1; t >= 0; t--) {
                if (threadIdx.x == 0 && t != steps - 1 && issued < steps) DHTS_RING_ISSUE
                mbar_wait(full + use_st, use_par);
                // cells are read from the stage where the sweep needs them (no register copy of the chunk); the
                // last read precedes the step's second block barrier
                const T* r = rp;
                const T* y = rp + rk.y_off;
                const uint2* ob = xp;
                rp += rk.stage_elems;
                if (XR) xp += (size_t)rk.stage_elems * sizeof(T) / sizeof(uint2);
                if (++use_st == ring_ns) {
                    use_st = 0; use_par ^= 1u; rp -= (size_t)ring_ns * rk.stage_elems;
                    if (XR) xp -= (size_t)ring_ns * rk.stage_elems * sizeof(T) / sizeof(uint2);
                }
                if (t == 0 && u0)
                    { T us_[C]; load_chunk<T, C>(u0 + off, us_); nan |= chunk_adj_step<T, C, true, XR>(r, y, us_, gr, gy, first_chunk, last_chunk, k, gLa, gRa, accL, accR, bl, br, warp, nwarp, lane, ob); }
                else
                    nan |= chunk_adj_step<T, C, false, XR>(r, y, nullptr, gr, gy, first_chunk, last_chunk, k, gLa, gRa, accL, accR, bl, br, warp, nwarp, lane, ob);
                bl += flipl; flipl = -flipl; br += flipr; flipr = -flipr;
            }
#undef DHTS_RING_ISSUE
        } else if (MODE == 1) {
            // register-prefetch variant (rows not 16-byte sized, or no room for the ring): one step ahead of the arithmetic
            // (measured: prefetching only into L2 and loading at the top of the step is 15 % slower)
            T r[C], y[C], rn[C], yn[C];
            const T* cr = ckpt + (size_t)(steps > 0 ? steps - 1 : 0) * 2 * BN + off;
            if (steps > 0) { load_chunk<T, C>(cr, r); load_chunk<T, C>(cr + BN, y); }
            T gq[3] = {T(0), T(0), T(0)};
            const bool tv = EXT && ghost_t != nullptr;
            const bool gthread = tv && (int)threadIdx.x < 2 * nl;
            const T* gsrc = tv ? ghost_t + ((size_t)(lane0 + (threadIdx.x >> 1)) * 2 + (threadIdx.x & 1)) * 3 : nullptr;
            if (gthread && steps > 0) { const T* q = gsrc + (size_t)(steps - 1) * B * 6; gq[0] = q[0]; gq[1] = q[1]; gq[2] = q[2]; }
            const T* gA_L = gLa; const T* gA_R = gRa;
            for (int t = steps - 1; t >= 0; t--) {
                T hr[C], hy[C];
                if (EXT && g_hist) {      // consumed at the end of the step: the loads fly during the step's arithmetic
                    const T* q = g_hist + (size_t)t * 2 * BN + off;
                    load_chunk<T, C>(q, hr); load_chunk<T, C>(q + BN, hy);
                }
                if (tv) {
                    if (gthread) {
                        step_ghost_record<T, true>(s, threadIdx.x, lpc, t & 1, gq);
                        if (t > 0) { const T* q = gsrc + (size_t)(t - 1) * B * 6; gq[0] = q[0]; gq[1] = q[1]; gq[2] = q[2]; }
                    }
                    gA_L = s.ghostA + ((size_t)(t & 1) * lpc * 2 + ll * 2) * GH_A; gA_R = gA_L + GH_A;
                }
                if (t > 0) {
                    cr -= 2 * BN;
                    load_chunk<T, C>(cr, rn); load_chunk<T, C>(cr + BN, yn);
                }
                if (t == 0 && u0)
                    { T us_[C]; load_chunk<T, C>(u0 + off, us_); nan |= chunk_adj_step<T, C, true>(r, y, us_, gr, gy, first_chunk, last_chunk, k, gA_L, gA_R, accL, accR, blA, brA, warp, nwarp, lane); }
                else
                    nan |= chunk_adj_step<T, C, false>(r, y, nullptr, gr, gy, first_chunk, last_chunk, k, gA_L, gA_R, accL, accR, blA, brA, warp, nwarp, lane);
                DHTS_SWAP_BOXES
                if (tv && g_ghost_t && active) {      // this step's ghost adjoints leave; the accumulators restart
                    T* gg = g_ghost_t + ((size_t)t * B + lane0 + ll) * 4;
                    if (first_chunk) { gg[0] = accL[0]; gg[1] = accL[1]; bad |= t_isnan(accL[0]) || t_isnan(accL[1]); }
                    if (last_chunk) { gg[2] = accR[0]; gg[3] = accR[1]; bad |= t_isnan(accR[0]) || t_isnan(accR[1]); }
                }
                if (tv) { accL[0] = accL[1] = accR[0] = accR[1] = T(0); }
                if (EXT && g_hist) {
#pragma unroll
                    for (int c = 0; c < C; c++) { gr[c] += hr[c]; gy[c] += hy[c]; }
                }
#pragma unroll
                for (int c = 0; c < C; c++) { r[c] = rn[c]; y[c] = yn[c]; }
            }
        } else {
            for (int seg = S - 1; seg >= 0; seg--) {
                const int t0 = seg * K, ks = min(K, steps - t0);
                T r[C], y[C];
                {
                    const T* cr = ckpt + ((size_t)seg * 2) * BN + off;
                    load_chunk<T, C>(cr, r); load_chunk<T, C>(cr + BN, y);
                }
                // recompute the segment, stashing every state (the stash stays in L2)
                for (int kk = 0; kk < ks; kk++) {
                    T* sr = scr + (size_t)kk * sstride + soff;
                    if (active) { store_chunk<T, C>(sr, r); store_chunk<T, C>(sr + (size_t)lpc * N, y); }
                    if (kk + 1 < ks) {
                        if (t0 + kk == 0 && u0)
                            { T us_[C]; load_chunk<T, C>(u0 + off, us_); chunk_fwd_step<T, C, true, false>(r, y, us_, first_chunk, last_chunk, k, gLf, gRf, dt, blA, brA, warp, nwarp, lane); }
                        else
                            chunk_fwd_step<T, C, false, false>(r, y, nullptr, first_chunk, last_chunk, k, gLf, gRf, dt, blA, brA, warp, nwarp, lane);
                        DHTS_SWAP_BOXES
                    }
                }
                // adjoint steps, last to first
                for (int kk = ks - 1; kk >= 0; kk--) {
                    if (kk != ks - 1) {
                        const T* sr = scr + (size_t)kk * sstride + soff;
                        load_chunk<T, C>(sr, r); load_chunk<T, C>(sr + (size_t)lpc * N, y);
                    }
                    if (t0 + kk == 0 && u0)
                        { T us_[C]; load_chunk<T, C>(u0 + off, us_); nan |= chunk_adj_step<T, C, true>(r, y, us_, gr, gy, first_chunk, last_chunk, k, gLa, gRa, accL, accR, blA, brA, warp, nwarp, lane); }
                    else
                        nan |= chunk_adj_step<T, C, false>(r, y, nullptr, gr, gy, first_chunk, last_chunk, k, gLa, gRa, accL, accR, blA, brA, warp, nwarp, lane);
                    DHTS_SWAP_BOXES
                }
            }
        }
        // NaN test of the gradients (dmacro_lane.py:308 asserts after every backward step): every step adds to the OLD adjoint
        // of the same cell, so a NaN never leaves a cell once it is there and one test of the final adjoint sees them all
#pragma unroll
        for (int c = 0; c < C; c++) nan |= t_isnan(gr[c]) || t_isnan(gy[c]);
        bad |= nan && active;
        if (active) {
            store_chunk<T, C>(g_r0 + off, gr); store_chunk<T, C>(g_y0 + off, gy);
            if (g_ghost && !(EXT && ghost_t)) {
                T* gg = g_ghost + (size_t)(lane0 + ll) * 4;
                if (first_chunk) { gg[0] = accL[0]; gg[1] = accL[1]; bad |= t_isnan(accL[0]) || t_isnan(accL[1]); }
                if (last_chunk) { gg[2] = accR[0]; gg[3] = accR[1]; bad |= t_isnan(accR[0]) || t_isnan(accR[1]); }
            }
        }
    }
    if (bad) atomicOr(flags, FLAG_NAN_GRAD);
}

// ------------------------------------------------------------------ host-side planning and launch
//
// fwd_plan / bwd_plan alone decide what a call runs: from the shape and the call's options they fix every template argument
// and the launch shape.  fwd_kernel / bwd_kernel map a plan to its instantiation; their lists are every instantiation this
// file compiles.

// Measured on B200 (profiles/r1e sweep, fp64, 8192 lanes x 1024 cells): both kernels are fastest with 4 cells per
// thread capped at 128 registers (2 CTAs of 256 threads per SM) -- forward 57 ms vs 69-89 ms for the other
// shapes, adjoint 97 ms (every state stored) / 149 ms (K = 32) vs 106-226 ms.
constexpr int CELLS = 4;                      // cells per thread where the lane allows (2 or 8: 1530 / 996 ms per pass against 938, r2)
constexpr int RING_NS = 4;                    // adjoint ring stages (3 or 6: 940 / 939 ms per pass against 938, r2)
constexpr int NSF = 4;                        // staging stages of the forward kernel
// Staging ring / state ring per CTA: keeps two CTAs of the 128-register shape on an SM (227 KB usable, 1 KB reserved per CTA).
constexpr size_t RING_BUDGET = 112 * 1024;
// Up to this much shared memory the C = 4 staged forward kernels run at 80 registers, three CTAs per SM (MB = 3): 384 vs
// 393 ms per pass (r2c A/B), 391 vs 405 ms with the stored outcomes (r2u A/B).
constexpr size_t MB3_BUDGET = 74 * 1024;

// Template arguments of a launch.  MB is the register budget in units of "CTAs of 1024/min(C,4) threads per SM": 2 -> 128
// registers (measured best for every C > 1, profiles/r1e sweep), 3 -> 80, 1 -> 255.
struct FwdKey { int C, MB, NS; bool TV, XR, UNI; };
struct BwdKey { int C, MB, MODE; bool EXT, XR, UNI; };
static bool operator==(const FwdKey& a, const FwdKey& b) {
    return a.C == b.C && a.MB == b.MB && a.NS == b.NS && a.TV == b.TV && a.XR == b.XR && a.UNI == b.UNI;
}
static bool operator==(const BwdKey& a, const BwdKey& b) {
    return a.C == b.C && a.MB == b.MB && a.MODE == b.MODE && a.EXT == b.EXT && a.XR == b.XR && a.UNI == b.UNI;
}
template <typename Key> struct Plan {
    Key k;
    int lpc, threads, groups;     // lanes per CTA, threads per CTA, lane groups (CTAs of a non-persistent launch)
    int ring_ns;                  // stages of the adjoint's state ring (MODE 0), else 0
    size_t smem;
    RollK rk;
};

static int round32(int x) { return (x + 31) / 32 * 32; }
// vector chunk loads need 16-byte aligned bases (row offsets are multiples of C elements by construction)
static bool al16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// Cells per thread and lanes per CTA, the same in both directions (the stored outcomes rely on it); no ring, no staging.
template <typename T, typename Key> static int lane_shape(int B, int N, Plan<Key>* p) {
    int C = 1;
    for (int c = CELLS; c > 1; c >>= 1)
        if (N % c == 0 && N / c >= 32) { C = c; break; }
    int tpl = N / C;
    while (tpl > 1024 / (C < 4 ? C : 4) && C < 8 && N % (2 * C) == 0) { C *= 2; tpl = N / C; }   // long lanes: wider chunks
    if (tpl > 1024 / (C < 4 ? C : 4)) return DHTS_ERR_UNSUPPORTED;
    const int target = 128;                       // threads per CTA when lanes are short
    int lpc = tpl >= target ? 1 : target / tpl;
    if (lpc > B) lpc = B;
    if (lpc < 1) lpc = 1;
    p->k.C = C; p->k.MB = C > 1 ? 2 : 1;
    p->lpc = lpc; p->threads = round32(lpc * tpl); p->groups = (B + lpc - 1) / lpc;
    p->ring_ns = 0; p->smem = shm_bytes<T>(lpc, p->threads / 32); p->rk = RollK();
    return DHTS_OK;
}

// Forward.  Every state stored (K == 1, no per-step ghosts) in 16-byte rows: the staging ring with TMA bulk stores, with the
// interface outcomes behind the states when xmode == 1 (the outcomes are warp ballots, stored lane by lane: whole warps per
// lane); the UNI instantiation for uniform geometry exists for the C = 4 kernel with outcomes, the bench's.  Otherwise
// per-thread stores (TV: per-step ghosts).  K == 0: no checkpoints.
template <typename T>
static int fwd_plan(int B, int N, int K, int xmode, bool tv, bool uni, bool aligned, Plan<FwdKey>* p) {
    const int rc = lane_shape<T>(B, N, p);
    if (rc) return rc;
    p->k.NS = 0; p->k.TV = tv; p->k.XR = p->k.UNI = false;
    const int C = p->k.C, nwarp = p->threads / 32;
    if (C > 1 && !aligned) return DHTS_ERR_UNSUPPORTED;          // callers step with the tiled kernels instead
    if (K != 1 || tv || C == 1 || ((size_t)N * sizeof(T)) % 16 != 0) return DHTS_OK;
    const bool xr = xmode == 1 && (N / C) % 32 == 0;
    const size_t stage = ((size_t)2 * p->lpc * N + (xr ? xrow_elems<T>(p->lpc, N / C, C) : 0)) * sizeof(T);
    const size_t smem = ring_offset<T>(p->lpc, nwarp, true) + NSF * stage;
    if (smem > RING_BUDGET) return DHTS_OK;
    p->k = FwdKey{C, C == 4 && smem <= MB3_BUDGET ? 3 : 2, NSF, false, xr, xr && uni && C == 4};
    p->smem = smem;
    p->rk = make_rollk<T>(B, N, C, p->lpc, nwarp, true, xr);
    return DHTS_OK;
}

// Adjoint.  Every state stored (K == 1, no per-step ghosts or history) in 16-byte rows: MODE 0, the state ring filled by
// TMA bulk loads, reading the stored outcomes when xmode == 1.  Otherwise MODE 1 (register prefetch; EXT: per-step ghosts /
// history) or, with sparse checkpoints, MODE 2 (segment recompute).
template <typename T>
static int bwd_plan(int B, int N, int K, int xmode, bool ext, bool uni, bool aligned, Plan<BwdKey>* p) {
    const int rc = lane_shape<T>(B, N, p);
    if (rc) return rc;
    p->k.MODE = K > 1 ? 2 : 1; p->k.EXT = ext; p->k.XR = p->k.UNI = false;
    const int C = p->k.C, nwarp = p->threads / 32;
    if (C > 1 && !aligned) return DHTS_ERR_UNSUPPORTED;
    if (!ext) p->rk = make_rollk<T>(B, N, C, p->lpc, nwarp, false, false);
    // a stage's two rows stay below the 2^20 bytes an mbarrier transaction count holds
    if (K != 1 || ext || C == 1 || ((size_t)N * sizeof(T)) % 16 != 0 || (size_t)p->lpc * N * sizeof(T) >= (1u << 19))
        return DHTS_OK;
    const bool xr = xmode == 1;
    const size_t stage = ((size_t)2 * p->lpc * N + (xr ? xrow_elems<T>(p->lpc, N / C, C) : 0)) * sizeof(T) + 8;  // + mbarrier
    const size_t base = ring_offset<T>(p->lpc, nwarp);
    int ns = RING_NS;
    while (ns >= 2 && base + ns * stage > RING_BUDGET) ns--;
    if (ns < 2) return DHTS_OK;
    p->k = BwdKey{C, 2, 0, false, xr, xr && uni && C == 4};
    p->ring_ns = ns; p->smem = base + ns * stage;
    p->rk = make_rollk<T>(B, N, C, p->lpc, nwarp, false, xr);
    return DHTS_OK;
}

// ckpt_mode 1: the rollouts of this shape store the interface outcomes with the states -- the forward plan is the staged
// kernel with outcomes and the adjoint plan the ring with outcomes (same C and lpc: the rows written are the rows read).
// Callers ask (dhts_arz_rollout_ckpt_elems_*), size `ckpt` accordingly and pass the mode to both calls.
template <typename T> static bool outcomes_stored(int B, int N, int K, Plan<FwdKey>* f) {
    Plan<BwdKey> b;
    return B > 0 && N >= 1 && fwd_plan<T>(B, N, K, 1, false, false, true, f) == DHTS_OK && f->k.XR &&
           bwd_plan<T>(B, N, K, 1, false, false, true, &b) == DHTS_OK && b.k.XR;
}

template <typename T> using FwdFn = decltype(&arz_rollout_fwd_reg_kernel<T, 1, 1, 0>);
template <typename T> using BwdFn = decltype(&arz_rollout_bwd_reg_kernel<T, 1, 1, 1>);
template <typename Key, typename Fn> struct Entry { Key k; Fn fn; };
template <typename T, int C, int MB, int NS, bool TV = false, bool XR = false, bool UNI = false>
static Entry<FwdKey, FwdFn<T>> fwd() { return {FwdKey{C, MB, NS, TV, XR, UNI}, arz_rollout_fwd_reg_kernel<T, C, MB, NS, TV, XR, UNI>}; }
template <typename T, int C, int MB, int MODE, bool EXT = false, bool XR = false, bool UNI = false>
static Entry<BwdKey, BwdFn<T>> bwd() { return {BwdKey{C, MB, MODE, EXT, XR, UNI}, arz_rollout_bwd_reg_kernel<T, C, MB, MODE, EXT, XR, UNI>}; }
template <typename Key, typename Fn, size_t n> static Fn find(const Entry<Key, Fn> (&list)[n], const Key& k) {
    for (const Entry<Key, Fn>& e : list)
        if (e.k == k) return e.fn;
    return nullptr;
}

template <typename T> static FwdFn<T> fwd_kernel(const FwdKey& k) {
    static const Entry<FwdKey, FwdFn<T>> list[] = {
        fwd<T, 1, 1, 0>(),                          // per-thread stores
        fwd<T, 2, 2, 0>(),
        fwd<T, 4, 2, 0>(),
        fwd<T, 8, 2, 0>(),
        fwd<T, 1, 1, 0, true>(),                    // per-step ghosts
        fwd<T, 2, 2, 0, true>(),
        fwd<T, 4, 2, 0, true>(),
        fwd<T, 8, 2, 0, true>(),
        fwd<T, 2, 2, NSF>(),                        // staged
        fwd<T, 4, 3, NSF>(),
        fwd<T, 8, 2, NSF>(),
        fwd<T, 2, 2, NSF, false, true>(),           // staged with outcomes
        fwd<T, 4, 3, NSF, false, true>(),
        fwd<T, 8, 2, NSF, false, true>(),
        fwd<T, 4, 3, NSF, false, true, true>(),     // staged with outcomes, uniform geometry
    };
    return find(list, k);
}

template <typename T> static BwdFn<T> bwd_kernel(const BwdKey& k) {
    static const Entry<BwdKey, BwdFn<T>> list[] = {
        bwd<T, 2, 2, 0>(),                          // ring
        bwd<T, 4, 2, 0>(),
        bwd<T, 8, 2, 0>(),
        bwd<T, 2, 2, 0, false, true>(),             // ring with outcomes
        bwd<T, 4, 2, 0, false, true>(),
        bwd<T, 8, 2, 0, false, true>(),
        bwd<T, 4, 2, 0, false, true, true>(),       // ring with outcomes, uniform geometry
        bwd<T, 1, 1, 1>(),                          // register prefetch (C > 1 gets a ring, except fp32 C = 2 below)
        bwd<T, 1, 1, 1, true>(),                    // per-step ghosts / history
        bwd<T, 2, 2, 1, true>(),
        bwd<T, 4, 2, 1, true>(),
        bwd<T, 8, 2, 1, true>(),
        bwd<T, 1, 1, 2>(),                          // segment recompute
        bwd<T, 2, 2, 2>(),
        bwd<T, 4, 2, 2>(),
        bwd<T, 8, 2, 2>(),
    };
    if constexpr (std::is_same<T, float>::value) {  // fp32 C = 2 lanes with N % 4 == 2: rows that are not 16-byte sized
        static const Entry<BwdKey, BwdFn<T>> fp32[] = {bwd<float, 2, 2, 1>()};
        if (const BwdFn<T> fn = find(fp32, k)) return fn;
    }
    return find(list, k);
}

template <typename T> static long long ckpt_elems(int B, int N, int steps, int K, int* mode) {
    if (B < 0 || N < 1 || steps < 0 || K < 1) return -1;
    Plan<FwdKey> f;
    const bool xr = outcomes_stored<T>(B, N, K, &f);
    if (mode) *mode = xr;
    const long long S = (steps + K - 1) / K;
    long long n = S * 2 * (long long)B * N;
    if (xr) n += ((long long)steps * B * (long long)xlane_bytes(N / f.k.C, f.k.C) + (long long)sizeof(T) - 1) / (long long)sizeof(T);
    return n;
}

template <typename T>
static int rollout_fwd(const T* r0, const T* y0, const T* u0, const T* ghost, const T* ghost_t, const T* dx, const T* umax,
                       T dx_all, T umax_all, T dt, int B, int N, int steps, int K, int xmode, T* ckpt, T* rT, T* yT, T* uT,
                       int* flags, cudaStream_t st) {
    if (!r0 || !y0 || (!ghost && !ghost_t) || (!dx != !umax) || !rT || !yT || !uT || !flags || B < 0 || N < 1 || steps < 0)
        return DHTS_ERR_INVALID;
    const bool uni = !dx;                         // one geometry for all lanes: the lane constants travel as a kernel parameter
    if (uni && !(dx_all > T(0) && umax_all > T(0))) return DHTS_ERR_INVALID;
    const LaneK<T> kall = make_lanek<T>(uni ? umax_all : T(1), uni ? dx_all : T(1), dt);
    if (ckpt && K < 1) return DHTS_ERR_INVALID;
    if (xmode != 0 && xmode != 1) return DHTS_ERR_INVALID;
    Plan<FwdKey> p;
    if (xmode == 1 && (!ckpt || ghost_t || !outcomes_stored<T>(B, N, K, &p))) return DHTS_ERR_INVALID;
    if (B == 0) return DHTS_OK;
    const bool aligned = al16(r0) && al16(y0) && al16(u0) && al16(ckpt) && al16(rT) && al16(yT) && al16(uT);
    int rc = fwd_plan<T>(B, N, ckpt ? K : 0, xmode, ghost_t != nullptr, uni, aligned, &p);
    if (rc) return rc;
    const FwdFn<T> kernel = fwd_kernel<T>(p.k);
    if (!kernel) return DHTS_ERR_CUDA;            // a plan without an instantiation: nothing to launch
    if ((rc = set_smem(kernel, p.smem))) return rc;
    kernel<<<p.groups, p.threads, p.smem, st>>>(r0, y0, u0, ghost_t ? nullptr : ghost, ghost_t, dx, umax, kall, dt, B, N, steps,
                                               K < 1 ? 1 : K, p.lpc, p.rk, ckpt, rT, yT, uT, flags);
    return launch_status();
}

template <typename T> static long long rollout_scratch_elems(int B, int N, int K) {
    Plan<BwdKey> p;
    if (B <= 0) return 0;
    if (K < 1 || bwd_plan<T>(B, N, K, 0, false, false, true, &p)) return -1;
    if (K == 1) return 0;                      // every state comes from the forward pass: nothing to stash
    int grid = 1;
    if (persistent_grid(bwd_kernel<T>(p.k), p.threads, p.smem, p.groups, &grid)) return -1;
    return (long long)grid * K * 2 * p.lpc * N;
}

template <typename T>
static int rollout_bwd(const T* ckpt, const T* u0, const T* ghost, const T* ghost_t, const T* dx, const T* umax, T dx_all,
                       T umax_all, T dt, int B,
                       int N, int steps, int K, int xmode, const T* rT, const T* yT, const T* g_rT, const T* g_yT, const T* g_uT,
                       const T* g_hist, T* scratch, long long scratch_elems, T* g_r0, T* g_y0, T* g_ghost, T* g_ghost_t,
                       int* flags, cudaStream_t st) {
    if (!ckpt || (!ghost && !ghost_t) || (!dx != !umax) || !g_r0 || !g_y0 || !flags || (!scratch && K > 1) || B < 0 || N < 1 || steps < 0 || K < 1)
        return DHTS_ERR_INVALID;
    const bool uni = !dx;
    if (uni && !(dx_all > T(0) && umax_all > T(0))) return DHTS_ERR_INVALID;
    const LaneK<T> kall = make_lanek<T>(uni ? umax_all : T(1), uni ? dx_all : T(1), dt);
    const bool ext = ghost_t || g_hist;
    if (ext && K != 1) return DHTS_ERR_INVALID;        // per-step ghosts / per-step adjoints need every state stored
    if (g_uT && (!rT || !yT)) return DHTS_ERR_INVALID;
    if (xmode != 0 && xmode != 1) return DHTS_ERR_INVALID;
    if (B == 0) return DHTS_OK;
    Plan<FwdKey> f;
    if (xmode == 1 && (ext || !outcomes_stored<T>(B, N, K, &f))) return DHTS_ERR_INVALID;
    // the ring with outcomes uses no scratch
    const bool aligned = al16(ckpt) && al16(u0) && al16(g_r0) && al16(g_y0) && (xmode == 1 || (al16(scratch) && al16(g_hist)));
    Plan<BwdKey> p;
    int rc = bwd_plan<T>(B, N, K, xmode, ext, uni, aligned, &p);
    if (rc) return rc;
    const BwdFn<T> kernel = bwd_kernel<T>(p.k);
    if (!kernel) return DHTS_ERR_CUDA;            // a plan without an instantiation: nothing to launch
    int grid = 1;
    if ((rc = persistent_grid(kernel, p.threads, p.smem, p.groups, &grid))) return rc;
    if (K > 1 && (long long)grid * K * 2 * p.lpc * N > scratch_elems) return DHTS_ERR_INVALID;
    kernel<<<grid, p.threads, p.smem, st>>>(ckpt, u0, ghost_t ? nullptr : ghost, ghost_t, g_hist, ext ? g_ghost_t : nullptr, dx,
                                           umax, kall, dt, B, N, steps, K, p.lpc, rT, yT, g_rT, g_yT, g_uT, scratch, g_r0, g_y0,
                                           g_ghost, flags, p.ring_ns, p.rk);
    return launch_status();
}

}  // namespace dhts

#define DHTS_ARZ_ROLLOUT_API(SUF, T)                                                                                   \
    DHTS_EXPORT int dhts_arz_rollout_fwd_##SUF(const T* r0, const T* y0, const T* u0, const T* ghost, const T* ghost_t, \
                                               const T* dx, const T* umax, T dx_all, T umax_all, T dt, int B, int N,   \
                                               int steps, int ckpt_every, int ckpt_mode, T* ckpt, T* rT, T* yT, T* uT, \
                                               int* flags, void* stream) {                                             \
        return dhts::rollout_fwd<T>(r0, y0, u0, ghost, ghost_t, dx, umax, dx_all, umax_all, dt, B, N, steps, ckpt_every, ckpt_mode, \
                                    ckpt, rT, yT, uT, flags, (cudaStream_t)stream);                                    \
    }                                                                                                                  \
    DHTS_EXPORT long long dhts_arz_rollout_ckpt_elems_##SUF(int B, int N, int steps, int ckpt_every, int* ckpt_mode) { \
        return dhts::ckpt_elems<T>(B, N, steps, ckpt_every, ckpt_mode);                                                \
    }                                                                                                                  \
    DHTS_EXPORT long long dhts_arz_rollout_scratch_elems_##SUF(int B, int N, int ckpt_every) {                         \
        return dhts::rollout_scratch_elems<T>(B, N, ckpt_every);                                                       \
    }                                                                                                                  \
    DHTS_EXPORT int dhts_arz_rollout_bwd_##SUF(const T* ckpt, const T* u0, const T* ghost, const T* ghost_t,           \
                                               const T* dx, const T* umax, T dx_all, T umax_all, T dt, int B, int N, int steps, \
                                               int ckpt_every, int ckpt_mode, const T* rT, const T* yT,                \
                                               const T* g_rT, const T* g_yT, const T* g_uT, const T* g_hist,           \
                                               T* scratch,                                                             \
                                               long long scratch_elems, T* g_r0, T* g_y0, T* g_ghost, T* g_ghost_t,    \
                                               int* flags, void* stream) {                                             \
        return dhts::rollout_bwd<T>(ckpt, u0, ghost, ghost_t, dx, umax, dx_all, umax_all, dt, B, N, steps, ckpt_every, ckpt_mode, rT, \
                                    yT, g_rT, g_yT, g_uT, g_hist, scratch, scratch_elems, g_r0, g_y0, g_ghost, g_ghost_t, flags, \
                                    (cudaStream_t)stream);                                                             \
    }

DHTS_ARZ_ROLLOUT_API(f64, double)
DHTS_ARZ_ROLLOUT_API(f32, float)
