/*
 * dhts.h -- C ABI of libdhts_b200.so: the B200 (sm_100a) simulation-step kernels
 * behind the lane / network object API of SonSang/diff-hybrid-traffic-sim.
 *
 * The reference has no FFI of its own (it is pure Python); the seam these entry
 * points replace is its per-lane autograd operator pair
 *     dMacroForwardLayer  road/lane/dmacro_lane.py:234-310
 *     dMicroForwardLayer  road/lane/dmicro_lane.py:228-297
 * plus the T-step loop that chains them (example/inverse/_inverse.py:91-99,227)
 * and the macro<->micro exchange (road/network/conversion.py:15-215).
 * INTEGRATION.md shows the ctypes binding a reference maintainer would add.
 *
 * Conventions
 *  - Every pointer is a DEVICE pointer owned by the caller (torch tensors on the
 *    Python side); the library never allocates, frees or retains them.
 *  - Every call only ENQUEUES work on `stream` (a cudaStream_t passed as void*)
 *    of the current device and never synchronises.  Re-entrant; no global or
 *    thread-local state besides cached device attributes.
 *  - `_f64` / `_f32`: T = double / float for storage and arithmetic.
 *  - Return value: DHTS_OK or an error code; nothing is enqueued on error.
 *  - `flags` is a caller-zeroed int32[4]: flags[0] is a bit mask OR-ed by the
 *    kernels, flags[1] counts collisions.  The host maps the bits to the
 *    reference's conventions after the rollout:
 *      DHTS_FLAG_CFL       AssertionError "Time step size does not meet CFL
 *                          condition" (road/lane/_macro_lane.py:141-146)
 *      DHTS_FLAG_NAN_GRAD  AssertionError on NaN gradients (dmacro_lane.py:308)
 *      DHTS_FLAG_COLLISION print-and-continue (road/lane/_micro_lane.py:151-162)
 *  - Macro lanes: B lanes x N cells, row-major [B][N]; "padded" arrays are
 *    [B][N+2] = (left ghost, cells, right ghost) exactly like the operator's
 *    input vectors (dmacro_lane.py:134-158).  dx[B], umax[B] are per lane.
 *  - Micro lanes: vehicles lane by lane, index 0 = tail, leader of i is i+1
 *    (road/lane/_micro_lane.py:33-36); lane_off[L+1] are CSR offsets; params is
 *    [6][V] = accel_max, accel_pref, target_speed, min_space, time_pref, length
 *    (road/vehicle/micro_vehicle.py:20-28); head[L][2] = (head_position_delta,
 *    head_speed_delta) (_micro_lane.py:40-43).
 */
#ifndef DHTS_H
#define DHTS_H

#ifdef __cplusplus
extern "C" {
#endif

#define DHTS_OK 0
#define DHTS_ERR_INVALID 1      /* null pointer / negative size / inconsistent arguments */
#define DHTS_ERR_UNSUPPORTED 2  /* shape outside what the fused kernel handles; use the step entry points */
#define DHTS_ERR_CUDA 3         /* launch failed (cudaGetLastError) */

#define DHTS_FLAG_CFL 1
#define DHTS_FLAG_NAN_GRAD 2
#define DHTS_FLAG_COLLISION 4

int dhts_version(void);

/* Measurement helper, not on the simulation path: enqueues `blocks` CTAs of 256 threads that each run 8
 * independent chains of `iters` fp64 fused multiply-adds and store one value per thread into out[blocks*256].
 * Returns the number of DFMA thread-instructions enqueued (-1 on error).  bench.py times it with CUDA events to
 * put a MEASURED fp64 issue peak next to the HBM peak of MEASURED_PEAKS.json (`roofline_fp64`). */
long long dhts_fp64_probe(double* out, int blocks, int iters, void* stream);

/* ---------------------------------------------------------------- ARZ, one step
 * Forward half of dMacroForwardLayer (dmacro_lane.py:236-275 -> MacroLane.forward,
 * _macro_lane.py:83-146; Riemann solver model/macro/_arz.py:212-332).
 *   r_pad, y_pad, u_pad [B][N+2]  cell records incl. ghosts; u_pad is the speed
 *                                 STORED on the cell (the reference does not
 *                                 recompute it at use, SURVEY App. B.3)
 *   ueq_pad [B][N+2] or NULL      stored u_eq; NULL = u_eq(r) (only cells
 *                                 rewritten by micro_to_macro differ)
 *   nr, ny, nu [B][N]             next density, relative flow and
 *                                 nu = compute_u(nr, ny) (set_r_y, _arz.py:88-92)
 *   case_out [B][N+1] or NULL     Riemann outcome per interface (0 Q_L, 1 Q_M, 2 Q_C)
 */
int dhts_arz_step_fwd_f64(const double* r_pad, const double* y_pad, const double* u_pad, const double* ueq_pad,
                          const double* dx, const double* umax, double dt, int B, int N, double* nr, double* ny,
                          double* nu, int* case_out, int* flags, void* stream);
int dhts_arz_step_fwd_f32(const float* r_pad, const float* y_pad, const float* u_pad, const float* ueq_pad,
                          const float* dx, const float* umax, float dt, int B, int N, float* nr, float* ny, float* nu,
                          int* case_out, int* flags, void* stream);

/* Backward half (dmacro_lane.py:96-132 Jacobian band + :277-310 VJP; Jacobians
 * model/macro/darz.py:12-233), evaluated from the saved INPUTS of the step.
 *   g_nr, g_ny [B][N]      adjoint of the outputs;  g_nu [B][N] or NULL adjoint of
 *                          nu (then nr, ny -- the saved outputs -- are required)
 *   g_r_pad, g_y_pad [B][N+2]  adjoint of the padded inputs, ghost entries included
 */
int dhts_arz_step_bwd_f64(const double* r_pad, const double* y_pad, const double* u_pad, const double* ueq_pad,
                          const double* dx, const double* umax, double dt, int B, int N, const double* nr,
                          const double* ny, const double* g_nr, const double* g_ny, const double* g_nu,
                          double* g_r_pad, double* g_y_pad, int* flags, void* stream);
int dhts_arz_step_bwd_f32(const float* r_pad, const float* y_pad, const float* u_pad, const float* ueq_pad,
                          const float* dx, const float* umax, float dt, int B, int N, const float* nr, const float* ny,
                          const float* g_nr, const float* g_ny, const float* g_nu, float* g_r_pad, float* g_y_pad,
                          int* flags, void* stream);

/* ---------------------------------------------------------------- ARZ, fused T-step rollout
 * `steps` x (RoadNetwork.forward over disconnected macro lanes): ghosts are
 * static per lane (road/network/road_network.py:299-387 with no neighbour),
 * lane.forward, update_state.  A lane stays in the REGISTERS of the threads that
 * own it for the whole rollout (1, 2, 4 or 8 consecutive cells per thread).
 *   r0, y0 [B][N]; u0 [B][N] or NULL (stored speed of the initial cells, set_r_u)
 *   ghost [B][2][3]        (r, y, u) of the left / right ghost cell
 *   dx, umax [B]           cell length / speed limit per lane (MacroLane.cell_length, .speed_limit), or BOTH NULL: every
 *                          lane has dx_all / umax_all (what the reference's drivers build: one lane shape per problem) --
 *                          the kernels then read the lane constants from their parameter block instead of registers
 *   ckpt [S][2][B][N] (+ outcomes) or NULL, S = ceil(steps/ckpt_every): state BEFORE steps
 *                          0, K, 2K, ... (needed by the backward entry point)
 *   ckpt_mode              0: ckpt holds the states only.  1: behind the S states it also holds the OUTCOME of every
 *                          interface of every step (Q_L / Q_M / Q_C, _arz.py:324-336: two bits per interface, kept as
 *                          the warp ballots of the kernels' thread -> cell mapping, N / 4 bytes per lane and step),
 *                          which lets the adjoint skip the Riemann case tree for a quarter byte per cell-step of HBM
 *                          traffic.  dhts_arz_rollout_ckpt_elems_*(B, N, steps, ckpt_every,
 *                          &mode) returns the elements `ckpt` must hold and the mode the kernels take for this shape
 *                          (1 where every state is stored, the ghosts are static and the staged forward / ring adjoint
 *                          kernels apply); callers pass that mode to both calls (0 is always accepted)
 *   rT, yT, uT [B][N]      final state, uT = compute_u(rT, yT)
 * Limits of the fused kernels: a lane must fit one CTA -- N <= 1024 cells in general (one or two cells per thread),
 * N <= 2048 when N is a multiple of 8 (256 threads x 8 cells; lane_shape in csrc/arz_rollout.cu) -- and with more than
 * one cell per thread every array must be 16-byte aligned.  Otherwise the call returns DHTS_ERR_UNSUPPORTED and enqueues nothing; the host then chains
 * `steps` launches of the one-step entry points (dhts_b200.functional.arz_rollout does).  The IDM rollouts take lanes
 * of at most dhts_idm_rollout_max_lane() = 256 vehicles and checkpoint intervals up to
 * dhts_idm_rollout_max_ckpt_every() = 32, with the same fallback.
 */
int dhts_arz_rollout_fwd_f64(const double* r0, const double* y0, const double* u0, const double* ghost,
                             const double* ghost_t, const double* dx, const double* umax, double dx_all, double umax_all,
                             double dt, int B, int N, int steps, int ckpt_every, int ckpt_mode, double* ckpt, double* rT,
                             double* yT, double* uT, int* flags, void* stream);
int dhts_arz_rollout_fwd_f32(const float* r0, const float* y0, const float* u0, const float* ghost,
                             const float* ghost_t, const float* dx, const float* umax, float dx_all, float umax_all,
                             float dt, int B, int N, int steps, int ckpt_every, int ckpt_mode, float* ckpt, float* rT,
                             float* yT, float* uT, int* flags, void* stream);

/* Adjoint of the rollout: the chain of dMacroForwardLayer.backward calls autograd makes for the T steps
 * (road/lane/dmacro_lane.py:277-310), flux-difference form, no stored Jacobian band.
 *   ckpt                    what the forward call wrote (same ckpt_every, same ckpt_mode)
 *   dx, umax / dx_all, umax_all  as in the forward call (both arrays, or both NULL with the two scalars)
 *   rT, yT                  final state (only read when g_uT is given: uT = compute_u(rT, yT))
 *   g_rT, g_yT, g_uT [B][N] adjoint of the final state, each may be NULL
 *   scratch                 dhts_arz_rollout_scratch_elems(B, N, ckpt_every) elements (0 when ckpt_every = 1)
 *   g_r0, g_y0 [B][N]       adjoint of the initial (r, y)
 *   g_ghost [B][2][2] or NULL  adjoint of the static ghosts' (r, y), summed over the steps
 * Per-step coupling (both need ckpt_every = 1, i.e. ckpt IS the state history [steps][2][B][N]):
 *   ghost_t [steps][B][2][3] or NULL  ghost (r, y, u) PER STEP instead of `ghost`: a lane inside a network gets new
 *                           ghost cells every step (road/network/road_network.py:364-387); forward and adjoint
 *   g_ghost_t [steps][B][2][2] or NULL  their adjoints, step by step
 *   g_hist [steps][2][B][N] or NULL   adjoint of a loss that reads the state BEFORE every step (a per-step loss such as
 *                           the ITSCP queue length, example/control/itscp/_env.py:662-742, on independent lanes)
 */
int dhts_arz_rollout_bwd_f64(const double* ckpt, const double* u0, const double* ghost, const double* ghost_t,
                             const double* dx, const double* umax, double dx_all, double umax_all, double dt, int B, int N,
                             int steps, int ckpt_every, int ckpt_mode, const double* rT, const double* yT, const double* g_rT, const double* g_yT,
                             const double* g_uT, const double* g_hist, double* scratch, long long scratch_elems,
                             double* g_r0, double* g_y0, double* g_ghost, double* g_ghost_t, int* flags, void* stream);
int dhts_arz_rollout_bwd_f32(const float* ckpt, const float* u0, const float* ghost, const float* ghost_t,
                             const float* dx, const float* umax, float dx_all, float umax_all, float dt, int B, int N,
                             int steps, int ckpt_every, int ckpt_mode, const float* rT, const float* yT, const float* g_rT, const float* g_yT, const float* g_uT,
                             const float* g_hist, float* scratch, long long scratch_elems, float* g_r0, float* g_y0,
                             float* g_ghost, float* g_ghost_t, int* flags, void* stream);
long long dhts_arz_rollout_scratch_elems_f64(int B, int N, int ckpt_every);
long long dhts_arz_rollout_scratch_elems_f32(int B, int N, int ckpt_every);
long long dhts_arz_rollout_ckpt_elems_f64(int B, int N, int steps, int ckpt_every, int* ckpt_mode);
long long dhts_arz_rollout_ckpt_elems_f32(int B, int N, int steps, int ckpt_every, int* ckpt_mode);

/* ---------------------------------------------------------------- IDM, one step
 * Forward half of dMicroForwardLayer (dmicro_lane.py:230-269 -> MicroLane.forward,
 * _micro_lane.py:131-214; model/micro/_idm.py:5-51).
 *   veh_lane [V]        lane index of each vehicle (dhts_csr_expand)
 *   np_, nv_ [V]        next position / speed
 *   vflags [V] or NULL  bit0 acceleration clipped, bit1 s* clipped, bit2 collision
 */
int dhts_csr_expand(const int* lane_off, int L, int* veh_lane, void* stream);
int dhts_idm_step_fwd_f64(const double* p, const double* v, const double* params, const int* lane_off,
                          const int* veh_lane, const double* head, double dt, int V, int L, double* np_, double* nv_,
                          int* vflags, int* flags, void* stream);
int dhts_idm_step_fwd_f32(const float* p, const float* v, const float* params, const int* lane_off,
                          const int* veh_lane, const float* head, float dt, int V, int L, float* np_, float* nv_,
                          int* vflags, int* flags, void* stream);

/* Backward half (dmicro_lane.py:87-127 band, :271-297 VJP; model/micro/didm.py).
 * The ghost leader of dmicro_lane.py:144-151 (p_head + dp, v_head - dv) is folded
 * in: its adjoint is added to the head vehicle and returned as g_head[L][2]
 * (adjoint of head_position_delta, head_speed_delta; may be NULL). */
int dhts_idm_step_bwd_f64(const double* p, const double* v, const double* params, const int* lane_off,
                          const int* veh_lane, const double* head, double dt, int V, int L, const double* g_np,
                          const double* g_nv, double* g_p, double* g_v, double* g_head, int* flags, void* stream);
int dhts_idm_step_bwd_f32(const float* p, const float* v, const float* params, const int* lane_off,
                          const int* veh_lane, const float* head, float dt, int V, int L, const float* g_np,
                          const float* g_nv, float* g_p, float* g_v, float* g_head, int* flags, void* stream);

/* The same, plus the adjoint of the vehicle parameters: g_params [6][V], laid out like params, every entry written
 * (not accumulated).  Like the state Jacobian it is taken with the raw gap and speed difference, so at a collision it
 * follows the same convention; a clipped acceleration contributes nothing, a clipped s* no s-term.  The head vehicle's
 * gap is head_dp, so its own length enters only through its follower's gap.  NULL g_params returns
 * DHTS_ERR_INVALID; a NaN parameter adjoint sets DHTS_FLAG_NAN_GRAD.  g_p, g_v, g_head are those of
 * dhts_idm_step_bwd_*, bit for bit. */
int dhts_idm_step_bwd_params_f64(const double* p, const double* v, const double* params, const int* lane_off,
                                 const int* veh_lane, const double* head, double dt, int V, int L, const double* g_np,
                                 const double* g_nv, double* g_p, double* g_v, double* g_head, double* g_params,
                                 int* flags, void* stream);
int dhts_idm_step_bwd_params_f32(const float* p, const float* v, const float* params, const int* lane_off,
                                 const int* veh_lane, const float* head, float dt, int V, int L, const float* g_np,
                                 const float* g_nv, float* g_p, float* g_v, float* g_head, float* g_params, int* flags,
                                 void* stream);

/* ---------------------------------------------------------------- IDM, fused T-step rollout
 * One warp per lane, vehicles in registers, leaders by warp shuffle.  max_lane =
 * largest lane size (<= dhts_idm_rollout_max_lane()); ckpt [S][2][V];
 * the backward needs ckpt_every <= dhts_idm_rollout_max_ckpt_every(). */
int dhts_idm_rollout_max_lane(void);
int dhts_idm_rollout_max_ckpt_every(void);
int dhts_idm_rollout_fwd_f64(const double* p0, const double* v0, const double* params, const int* lane_off,
                             const double* head, const double* head_t, double dt, int V, int L, int max_lane, int steps,
                             int ckpt_every, double* ckpt, double* pT, double* vT, int* flags, void* stream);
int dhts_idm_rollout_fwd_f32(const float* p0, const float* v0, const float* params, const int* lane_off,
                             const float* head, const float* head_t, float dt, int V, int L, int max_lane, int steps,
                             int ckpt_every, float* ckpt, float* pT, float* vT, int* flags, void* stream);
/* Per-step coupling, as for the ARZ rollouts:
 *   head_t [steps][L][2] or NULL    head deltas PER STEP instead of `head` (inside a network
 *                                   RoadNetwork.setup_micro_boundary rewrites them before every step,
 *                                   road/network/road_network.py:429-580); g_head_t [steps][L][2] their adjoints
 *   g_hist [steps][2][V] or NULL    adjoint of a loss that reads (p, v) BEFORE every step; needs ckpt_every = 1 */
int dhts_idm_rollout_bwd_f64(const double* ckpt, const double* params, const int* lane_off, const double* head,
                             const double* head_t, double dt, int V, int L, int max_lane, int steps, int ckpt_every,
                             const double* g_pT, const double* g_vT, const double* g_hist, double* g_p0, double* g_v0,
                             double* g_head, double* g_head_t, int* flags, void* stream);
int dhts_idm_rollout_bwd_f32(const float* ckpt, const float* params, const int* lane_off, const float* head,
                             const float* head_t, float dt, int V, int L, int max_lane, int steps, int ckpt_every,
                             const float* g_pT, const float* g_vT, const float* g_hist, float* g_p0, float* g_v0,
                             float* g_head, float* g_head_t, int* flags, void* stream);
/* The same, plus the adjoint of the vehicle parameters over the whole rollout: g_params [6][V], with the convention,
 * validation and flags of dhts_idm_step_bwd_params_*.  Per-step head deltas and g_hist are taken as above.  g_p0, g_v0,
 * g_head, g_head_t are those of dhts_idm_rollout_bwd_*, bit for bit. */
int dhts_idm_rollout_bwd_params_f64(const double* ckpt, const double* params, const int* lane_off, const double* head,
                                    const double* head_t, double dt, int V, int L, int max_lane, int steps,
                                    int ckpt_every, const double* g_pT, const double* g_vT, const double* g_hist,
                                    double* g_p0, double* g_v0, double* g_head, double* g_head_t, double* g_params,
                                    int* flags, void* stream);
int dhts_idm_rollout_bwd_params_f32(const float* ckpt, const float* params, const int* lane_off, const float* head,
                                    const float* head_t, float dt, int V, int L, int max_lane, int steps, int ckpt_every,
                                    const float* g_pT, const float* g_vT, const float* g_hist, float* g_p0, float* g_v0,
                                    float* g_head, float* g_head_t, float* g_params, int* flags, void* stream);

/* ---------------------------------------------------------------- macro <-> micro exchange (per junction)
 * macro -> micro, road/network/conversion.py:15-73 (with MacroLane.add_flux_capacitor,
 * road/lane/_macro_lane.py:215-225, and MicroLane.entering_free_space,
 * road/lane/_micro_lane.py:289-301, evaluated by the caller into free_space):
 *   cap' = cap + r_last u_last dt; spawn iff cap' >= veh_len and free_space >= veh_len;
 *   on spawn: v_new = u_last, a_new = veh_len carrying d(cap'), cap_out = cap' - veh_len
 *   with its adjoint cut (the reference re-creates it detached); else cap_out = cap'.
 * All arrays [J].  spawn is int32. */
int dhts_m2c_fwd_f64(const double* cap, const double* r_last, const double* u_last, const double* free_space,
                     const double* veh_len, double dt, int J, double* cap_out, int* spawn, double* v_new,
                     double* a_new, void* stream);
int dhts_m2c_fwd_f32(const float* cap, const float* r_last, const float* u_last, const float* free_space,
                     const float* veh_len, float dt, int J, float* cap_out, int* spawn, float* v_new, float* a_new,
                     void* stream);
int dhts_m2c_bwd_f64(const double* r_last, const double* u_last, const int* spawn, double dt, int J,
                     const double* g_cap_out, const double* g_v_new, const double* g_a_new, double* g_cap,
                     double* g_r_last, double* g_u_last, void* stream);
int dhts_m2c_bwd_f32(const float* r_last, const float* u_last, const int* spawn, float dt, int J,
                     const float* g_cap_out, const float* g_v_new, const float* g_a_new, float* g_cap,
                     float* g_r_last, float* g_u_last, void* stream);

/* micro -> macro, road/network/conversion.py:75-171: when the head vehicle has
 * passed lane_len + len it is absorbed: every downstream cell it overlaps (walking
 * from cell 0 until the first miss) gets r += (a/len)(overlap/dx) value-clamped to
 * [1e-5, 1-1e-5] with pass-through gradient, u = v_head, y = r (u - u_eq(r)).
 *   p_head, v_head, a_head, len_head, lane_len, dx, umax [J]; r, y, u [J][N] rows of
 *   the downstream macro lanes; outputs are full rows; absorbed, ntouched int32 [J].
 * The backward takes the saved r_out / ntouched and returns the adjoints of
 * (p_head, v_head, a_head) and of the input rows. */
int dhts_c2m_fwd_f64(const double* p_head, const double* v_head, const double* a_head, const double* len_head,
                     const double* lane_len, const double* r, const double* y, const double* u, const double* dx,
                     const double* umax, int J, int N, double* r_out, double* y_out, double* u_out, int* absorbed,
                     int* ntouched, void* stream);
int dhts_c2m_fwd_f32(const float* p_head, const float* v_head, const float* a_head, const float* len_head,
                     const float* lane_len, const float* r, const float* y, const float* u, const float* dx,
                     const float* umax, int J, int N, float* r_out, float* y_out, float* u_out, int* absorbed,
                     int* ntouched, void* stream);
int dhts_c2m_bwd_f64(const double* p_head, const double* v_head, const double* a_head, const double* len_head,
                     const double* lane_len, const double* r_out, const double* dx, const double* umax,
                     const int* ntouched, int J, int N, const double* g_r_out, const double* g_y_out,
                     const double* g_u_out, double* g_p, double* g_v, double* g_a, double* g_r, double* g_y,
                     double* g_u, void* stream);
int dhts_c2m_bwd_f32(const float* p_head, const float* v_head, const float* a_head, const float* len_head,
                     const float* lane_len, const float* r_out, const float* dx, const float* umax,
                     const int* ntouched, int J, int N, const float* g_r_out, const float* g_y_out,
                     const float* g_u_out, float* g_p, float* g_v, float* g_a, float* g_r, float* g_y, float* g_u,
                     void* stream);

/* ---------------------------------------------------------------- connected macro network, fused T-step rollout
 * Steps R independent replicas of ONE connected network of macro lanes for `steps` steps in a single launch
 * (one CTA per replica, network state in shared memory), forward and adjoint.  Per step and replica it stands for
 *   RoadNetwork.forward                      road/network/road_network.py:79-111   (Jacobi: boundaries, forward, update)
 *   RoadNetwork.get_macro_boundary           road/network/road_network.py:299-362
 *   ItscpRoadNetwork.setup_macro_boundary    example/control/itscp/_simulator.py:56-142      (mode 1)
 *   set_leftmost_cell / set_rightmost_cell   road/lane/_macro_lane.py:156-162 (FullQ.from_r_u, model/macro/_arz.py:74-80)
 *   dMacroLane.forward + dMacroForwardLayer  road/lane/dmacro_lane.py:68-132,234-310
 *   the queue-length reward (optional)       example/control/itscp/_env.py:662-742,770-797
 * and for the autograd chain through them (SURVEY.md 8f rows f1-f3).
 *
 * Topology (device arrays shared by all replicas; side 0 = predecessors / left ghost, 1 = successors / right ghost):
 *   cell_off [L+1]   CSR of the cells, lane by lane (NC = cell_off[L])
 *   nadj     [2][L]  number of adjacent lanes per side
 *   one_adj  [2][L]  the adjacent lane when there is exactly one, else -1
 *   adj_off  [2][L+1], adj [E]  adjacency lists (absolute offsets into adj)
 *   own_slot [2][L]  slot (0..n_own-1) of the lane's own ghost record for sides that can feed on it, else -1
 * Per call:
 *   dx [L] cell length per lane;  umax, dt, veh_len, static_speed scalars of the network
 *   route [Rr][steps][2][L] int32 or NULL: (prev lane, next lane) chosen by the MacroRoute of each step, -1 = none;
 *                    Rr = R when route_per_replica, else 1
 *   mode 0: ghost = source (plain RoadNetwork); mode 1: ITSCP signal blend with
 *   sig, incoming [R][steps][L]: lane_signal / lane_incoming of each step; soft = 1: sigmoid(32(sig-0.5)) on the right
 *                    side (differentiable=True), 0: sig > 0.5
 *   qk [steps] or NULL: sigmoid constant of the queue reward per step; reward [R] = -sum_t sum_lanes q^2 dt
 *   r0, y0, u0 [R][NC]; own0 [R][n_own][2] initial (r, u) of the own ghost records
 *   ueq0 [R][NC] or NULL     u_eq STORED on the cells at the start (the step reads the stored value: cleared cells carry
 *                            u_max, cells rewritten by micro_to_macro a stale one); NULL = u_eq(r0) as set_r_u leaves it
 *   hist [steps+1][R][3][NC]  every state (r, y, u): before step t, and after the last step (output, kept for bwd)
 *   own_hist [steps+1][R][n_own][2]
 * Backward:
 *   g_states [steps][R][3][NC] or NULL  dLoss/d(r, y, u) of the state AFTER step t (last = terminal adjoint)
 *   g_reward [R] or NULL                dLoss/d reward (needs qk)
 *   g_r0, g_y0, g_u0 [R][NC]; g_own0 [R][n_own][2] or NULL; g_sig, g_incoming [R][steps][L] or NULL
 * Flags: DHTS_FLAG_CFL, DHTS_FLAG_NAN_GRAD, DHTS_FLAG_ROUTE (a lane with several neighbours on one side has none
 * selected by the step's route; the reference raises KeyError there).
 */
#define DHTS_FLAG_ROUTE 8
typedef struct dhts_net_topology {
    int L, NC, n_own;
    const int* cell_off;
    const int* nadj;
    const int* one_adj;
    const int* adj_off;
    const int* adj;
    const int* own_slot;
} dhts_net_topology;

int dhts_net_rollout_fwd_f64(const dhts_net_topology* topo, const double* dx, const int* route, int route_per_replica,
                             const double* sig, const double* incoming, const double* qk, double umax, double dt,
                             double veh_len, double static_speed, int steps, int R, int mode, int soft,
                             const double* r0, const double* y0, const double* u0, const double* own0, double* hist,
                             double* own_hist, double* reward, int* flags, void* stream);
int dhts_net_rollout_fwd_f32(const dhts_net_topology* topo, const float* dx, const int* route, int route_per_replica,
                             const float* sig, const float* incoming, const float* qk, float umax, float dt,
                             float veh_len, float static_speed, int steps, int R, int mode, int soft, const float* r0,
                             const float* y0, const float* u0, const float* own0, float* hist, float* own_hist,
                             float* reward, int* flags, void* stream);
int dhts_net_rollout_bwd_f64(const dhts_net_topology* topo, const double* dx, const int* route, int route_per_replica,
                             const double* sig, const double* incoming, const double* qk, double umax, double dt,
                             double veh_len, double static_speed, int steps, int R, int mode, int soft,
                             const double* hist, const double* own_hist, const double* g_states,
                             const double* g_reward, double* g_r0, double* g_y0, double* g_u0, double* g_own0,
                             double* g_sig, double* g_incoming, int* flags, void* stream);
int dhts_net_rollout_bwd_f32(const dhts_net_topology* topo, const float* dx, const int* route, int route_per_replica,
                             const float* sig, const float* incoming, const float* qk, float umax, float dt,
                             float veh_len, float static_speed, int steps, int R, int mode, int soft,
                             const float* hist, const float* own_hist, const float* g_states, const float* g_reward,
                             float* g_r0, float* g_y0, float* g_u0, float* g_own0, float* g_sig, float* g_incoming,
                             int* flags, void* stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Connected HYBRID network rollout (macro ARZ lanes + micro IDM lanes + the conversions between them), one CTA per
 * replica, forward and adjoint: configs 3 and 4 (hybrid inverse problem, ITSCP hybrid mode) in one launch.  Per step
 * and replica it stands for everything dhts_net_rollout_* does plus
 *   RoadNetwork.setup_micro_boundary        road/network/road_network.py:429-580   leader of a head vehicle along its route
 *   ItscpRoadNetwork.setup_micro_boundary   example/control/itscp/_simulator.py:144-276  signal-blended head deltas (mode 1)
 *   dMicroLane.forward + dMicroForwardLayer road/lane/dmicro_lane.py:87-153,228-297
 *   RoadNetwork.conversion / Conversion.*   road/network/road_network.py:113-173, road/network/conversion.py:15-215
 * and for the autograd chain through them.
 *
 * Topology (device arrays): the dhts_net_topology fields (micro lanes have no cells: cell_off[l+1] == cell_off[l]) and
 *   kind [L] 0 macro / 1 micro;  mic_of [L] micro index or -1;  mic_lane [ML] lane id of a micro index
 *   cap_off [L+1], cap_lane [NCAP]  flux capacitors of a macro lane: one per micro successor (MacroLane.flux_capacitor)
 *   grp_off [NG+1], grp_lane [NGL]  conversion groups: lanes that take part in conversions, partitioned into connected
 *                    components of "may touch the same lane", ascending lane id inside a group
 *   routes [NR][RLEN] lane ids along a vehicle route (MicroRoute.route), -1 terminated
 *   cap   vehicle slots per micro lane;  MAXT  max cells one absorbed vehicle can overlap (ceil(len / min dx) + 1)
 *   src [ML] or NULL (mode 1 only): 1 = micro lane without predecessor that is fed from a WAITING LIST, the stochastic
 *                    source of ITSCP micro mode (ItscpRoadNetwork.setup_micro_boundary, _simulator.py:153-174): while
 *                    the lane has room for a vehicle it consumes one uniform draw per step (lanes in id order) and a
 *                    default vehicle enters at position 0 when the draw is below incoming[.][t][lane] and the lane's
 *                    list (spawn_route row, KS entries, in pop order) is not exhausted
 * Per call (beyond dhts_net_rollout_*):
 *   lane_len [L];  veh_len: the network's vehicle length (RoadNetwork.add_vehicle asserts one length, road_network.py:60)
 *   veh_par [n_par][6] DEVICE array of IDM parameter sets (a_max, a_pref, v_target, s0, T, unused): every vehicle names
 *                    its set (MicroVehicle's own attributes, road/vehicle/micro_vehicle.py:74-122); set 0 is what
 *                    spawned / waiting-list vehicles get (default_micro_vehicle, :30-72)
 *   spawn_route [Rs][ML][KS] int32: route id of the k-th vehicle spawned into a micro lane (Rs = R or 1)
 *   src_rand [Rr][n_rand] (Rr = R or 1) or NULL: the uniform draws of the waiting-list sources in consumption order
 *                    (np.random.random in the reference); DHTS_FLAG_VEH_OVERFLOW when a rollout needs more than n_rand
 *   aux0 [R][AUX] (AUX = dhts_hyb_aux_size): vehicles p, v, a, route id, route cursor, parameter-set id, each [ML][cap]
 *                    by ring slot; ring front, count, spawn counter [ML]; capacitors [NCAP]; running-mean (sum, count) of
 *                    the micro signal (_simulator.py:255-262); number of source draws consumed; integers stored as reals
 *   hist [steps+1][R][4][NC] (r, y, u, stored u_eq);  own_hist;  aux_hist [steps+1][R][AUX];
 *   head_hist [steps][R][ML][2] or NULL: head deltas each micro lane used
 * Backward: g_states [steps][R][4][NC] or NULL;  g_aux [steps][R][AUX] or NULL (p, v, a entries of the vehicles that
 *   exist after step t are read);  g_aux0 [R][AUX] or NULL (p, v, a of the initial vehicles and the capacitors).
 * Flags: as dhts_net_rollout_* plus DHTS_FLAG_COLLISION and DHTS_FLAG_VEH_OVERFLOW (ring, spawn-route list or MAXT
 * exhausted: raise cap / KS).
 */
#define DHTS_FLAG_VEH_OVERFLOW 16
typedef struct dhts_hyb_topology {
    int L, NC, n_own;
    const int* cell_off;
    const int* nadj;
    const int* one_adj;
    const int* adj_off;
    const int* adj;
    const int* own_slot;
    int ML, cap, NCAP, NG, NGL, NR, RLEN, MAXT;
    const int* kind;
    const int* mic_of;
    const int* mic_lane;
    const int* cap_off;
    const int* cap_lane;
    const int* grp_off;
    const int* grp_lane;
    const int* routes;
    const int* src;
} dhts_hyb_topology;

int dhts_hyb_aux_size(const dhts_hyb_topology* topo);
int dhts_hyb_rollout_fwd_f64(const dhts_hyb_topology* topo, const double* dx, const double* lane_len, const int* route,
                             int route_per_replica, const int* spawn_route, int spawn_per_replica, int KS,
                             const double* sig, const double* incoming, const double* veh_par, int n_par, double veh_len,
                             const double* src_rand, int n_rand, int rand_per_replica, double umax, double dt, int steps,
                             int R, int mode, int soft, const double* r0, const double* y0, const double* u0, const double* ueq0,
                             const double* own0, const double* aux0, double* hist, double* own_hist, double* aux_hist, double* head_hist, int* flags,
                             void* stream);
int dhts_hyb_rollout_bwd_f64(const dhts_hyb_topology* topo, const double* dx, const double* lane_len, const int* route,
                             int route_per_replica, const int* spawn_route, int spawn_per_replica, int KS,
                             const double* sig, const double* incoming, const double* veh_par, int n_par, double veh_len,
                             const double* src_rand, int n_rand, int rand_per_replica, double umax, double dt, int steps,
                             int R, int mode, int soft, const double* hist, const double* own_hist, const double* aux_hist,
                             const double* g_states, const double* g_aux, double* g_r0, double* g_y0, double* g_u0, double* g_own0,
                             double* g_sig, double* g_incoming, double* g_aux0, int* flags, void* stream);
int dhts_hyb_rollout_fwd_f32(const dhts_hyb_topology* topo, const float* dx, const float* lane_len, const int* route,
                             int route_per_replica, const int* spawn_route, int spawn_per_replica, int KS,
                             const float* sig, const float* incoming, const float* veh_par, int n_par, float veh_len,
                             const float* src_rand, int n_rand, int rand_per_replica, float umax, float dt, int steps,
                             int R, int mode, int soft, const float* r0, const float* y0, const float* u0, const float* ueq0,
                             const float* own0, const float* aux0, float* hist, float* own_hist, float* aux_hist, float* head_hist, int* flags,
                             void* stream);
int dhts_hyb_rollout_bwd_f32(const dhts_hyb_topology* topo, const float* dx, const float* lane_len, const int* route,
                             int route_per_replica, const int* spawn_route, int spawn_per_replica, int KS,
                             const float* sig, const float* incoming, const float* veh_par, int n_par, float veh_len,
                             const float* src_rand, int n_rand, int rand_per_replica, float umax, float dt, int steps,
                             int R, int mode, int soft, const float* hist, const float* own_hist, const float* aux_hist,
                             const float* g_states, const float* g_aux, float* g_r0, float* g_y0, float* g_u0, float* g_own0,
                             float* g_sig, float* g_incoming, float* g_aux0, int* flags, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DHTS_H */
