/*
 * tcmp.h -- C ABI of libtcmp.so, the B200 (sm_100a) torque-feasibility engine.
 *
 * This is the drop-in boundary for the hot path of
 * HIRO-group/torque_constrained_motion_planning.  Each entry point cites the reference
 * interface it replaces (paths relative to the reference's src/).  The reference has no
 * FFI for this path except the CPython extension `ikfast_panda_arm`; INTEGRATION.md shows
 * the ctypes stubs a maintainer adds to rne.py / panda_primitives.py / ik_utils.py.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes; no C++/torch types cross the boundary.
 *   - Unless the name ends in `_host`, every data pointer is a DEVICE pointer owned by the
 *     caller; the library never frees caller memory and allocates nothing the caller sees.
 *   - Batched arrays are structure-of-arrays: q[j*n + i] is joint j of state i ("[7][n]").
 *   - Calls enqueue on `stream` (a cudaStream_t passed as void*, NULL = legacy default
 *     stream) on the CURRENT device and return without synchronising.
 *   - Return 0 (TCMP_OK) or a negative tcmp_status; tcmp_last_error() gives a thread-local
 *     message.  No global mutable state: the payload mass is an input of every call (the
 *     reference keeps it in module globals, rne.py:143-195).
 *   - dtype: TCMP_F64 computes and stores in double (torques within 1e-9 N.m of the
 *     reference); TCMP_F32 reads/writes float arrays and computes in float (1e-4 relative).
 */
#ifndef TCMP_H_
#define TCMP_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TCMP_ABI_VERSION 1

typedef enum {
    TCMP_OK = 0,
    TCMP_ERR_INVALID_ARG = -1, /* NULL where data is required, n < 0, bad enum, ... */
    TCMP_ERR_CUDA = -2,        /* a CUDA runtime call failed; see tcmp_last_error() */
    TCMP_ERR_NO_DEVICE = -3,   /* no usable sm_100 device */
    TCMP_ERR_UNSUPPORTED = -4  /* combination not implemented */
} tcmp_status;

/* torque_test selector == Problem.torque_test (utils.py:86-93, panda_primitives.py:228-236) */
typedef enum {
    TCMP_MODE_RNE = 0, /* get_torque_limits_not_exceded_test_v4     panda_primitives.py:155-193 */
    TCMP_MODE_NOV = 1, /* get_torque_limits_not_exceded_test_v3_nov panda_primitives.py:118-153 */
    TCMP_MODE_DYN = 2, /* get_torque_limits_not_exceded_test_v2     panda_primitives.py:60-116  */
    TCMP_MODE_BASE = 3 /* get_torque_limits_not_exceded_test_base   panda_primitives.py:13-16   */
} tcmp_mode;

typedef enum { TCMP_F64 = 0, TCMP_F32 = 1 } tcmp_dtype;

/* The reference's closures attach the payload iff mass > 0.01 kg (panda_primitives.py:139,178);
 * rne.add_payload attaches it iff mass > 0 (rne.py:184).  Callers pass the rule explicitly. */
#define TCMP_PAYLOAD_THRESHOLD_TEST 0.01
#define TCMP_PAYLOAD_THRESHOLD_RAW 0.0

int tcmp_abi_version(void);
const char *tcmp_last_error(void);
/* Number of sm_100 devices visible, or a negative status. */
int tcmp_device_count(void);

/*
 * Batched torque test.  Replaces rne.rne(q, qd, qdd) (rne.py:198-254) +
 * add_payload/remove_payload (rne.py:181-195) + the limit compare of the closures
 * (panda_primitives.py:182-188: feasible iff |tau_i| < limit_i for i in 0..5).
 *   q, qd, qdd      [7][n]; qd/qdd may be NULL = zeros (panda_primitives.py:175-177);
 *                   ignored in TCMP_MODE_NOV (panda_primitives.py:136-137).
 *   payload_mass    [n] or NULL (then payload_scalar applies to every state).
 *   payload_threshold  payload attached iff mass > threshold (rne/nov); dyn applies the
 *                   mass unconditionally as a tool-point force (panda_primitives.py:101-110).
 *   tau_out         [7][n] or NULL;  feasible_out [n] (1 = within limits) or NULL.
 * A NaN or infinite joint angle -- joint 1's too, although its value cannot change a torque -- gives NaN torques
 * and, since NaN never compares >= a limit, a feasible verdict, as rne.py does.  The edge, trajectory, IK-select
 * and extend-prefix torque tests follow the same rule.
 */
int tcmp_rne_batch(int mode, int dtype, int64_t n, const void *q, const void *qd, const void *qdd,
                   const void *payload_mass, double payload_scalar, double payload_threshold,
                   void *tau_out, uint8_t *feasible_out, void *stream);

/*
 * The inertial parameters and limits the torque test uses, for callers whose arm is not the stock one (another
 * hand, recalibrated links, tighter limits).  The reference keeps these in module-level lists -- ms, cs,
 * inertia_matrices (rne.py:102,119,138) -- plus the literals 0.14 + 0.025 (rne.py:182,186) and get_max_force
 * (utils.py:1558); SURVEY.md 8b sketches a process-global `tcmp_set_model`.  Here the record is an ARGUMENT of
 * the call instead, so the library keeps no mutable state and stays re-entrant.  The modified-DH geometry
 * (rne.py:47-54) is not part of it: IK, FK and the collision model are built on the same geometry.
 * All doubles, no padding (99 doubles): bindings may pass a flat float64[99].
 */
typedef struct tcmp_model {
    double mass[9];         /* panda_link1..7, panda_link8, panda_hand                      rne.py:125-136 */
    double com[9][3];       /* centre of mass in the body frame (link8 / hand: flange frame) rne.py:106-117 */
    double inertia[9][6];   /* ixx ixy ixz iyy iyz izz about the centre of mass              rne.py:65-75   */
    double payload_radius;  /* payload inertia = diag(m r^2, m r^2, 0), r = 0.165            rne.py:182-187 */
    double tool_z;          /* grasp-target height above the flange, 0.105 (dyn)   panda_mod.urdf:87-91     */
    double torque_limit[7]; /* 87 87 87 87 12 12 12; joint 7 is never tested       panda_primitives.py:182  */
} tcmp_model;
/* Fills *out with the compiled-in Panda (what every other entry point uses). */
int tcmp_model_default(tcmp_model *out);
/*
 * tcmp_rne_batch with a caller-supplied inertial set (host pointer, read during the call; NULL = compiled-in
 * Panda, then identical to tcmp_rne_batch).  The record is folded (link8 + hand onto link 7) and regrouped into
 * base parameters on the host, then handed to the kernel by value.  Masses must be finite and >= 0, limits > 0.
 */
int tcmp_rne_batch_model(const tcmp_model *model, int mode, int dtype, int64_t n, const void *q, const void *qd,
                         const void *qdd, const void *payload_mass, double payload_scalar,
                         double payload_threshold, void *tau_out, uint8_t *feasible_out, void *stream);

/*
 * Joint-space dynamics terms of the model tcmp_rne_batch evaluates, fp64, per state -- what the reference's `dyn`
 * test imports from panda_dynamics_model (get_mass_matrix / get_coriolis_matrix / get_gravity_vector,
 * panda_primitives.py:86-91) plus the tool Jacobian it takes from PyBullet (:93-99):
 *   g_out [7][n]     g(q) = rne(q, 0, 0)
 *   M_out [7][7][n]  joint-space inertia matrix, element (r, c) of state i at (r*7 + c)*n + i; exactly symmetric
 *   C_out [7][7][n]  Christoffel-consistent Coriolis matrix C_ij = sum_k Gamma_ijk qd_k: C qd = rne(q, qd, 0) - g
 *                    and Mdot = C + C^T
 *   J_out [6][7][n]  geometric Jacobian of the grasp-target point (link-7 origin + (0, 0, 0.107 + tool_z)) in the
 *                    base frame, rows [linear; angular]
 * so that M qdd + C qd + g == tcmp_rne_batch(TCMP_MODE_RNE, ..., TCMP_PAYLOAD_THRESHOLD_RAW).
 * M, C and g do not read joint 1's angle: a NaN or infinite q[0] leaves them finite (and J NaN), where
 * tcmp_rne_batch returns NaN torques.
 *   model         host pointer or NULL (compiled-in Panda).
 *   q [7][n]; qd [7][n], required iff C_out != NULL.
 *   payload_mass  [n] or NULL (then payload_scalar): a rigid body on the flange iff m > 0 (rne.py:184); 0 gives the
 *                 arm alone, as panda_dynamics_model does.
 * Each output may be NULL (not computed); at least one is required when n > 0.  n == 0 returns TCMP_OK whatever the
 * buffers (an empty array may have a NULL data pointer).  Enqueues only: no allocation, no synchronisation, so the
 * call can be captured in a CUDA graph.
 */
int tcmp_dynamics_batch(const tcmp_model *model, int64_t n, const double *q, const double *qd,
                        const double *payload_mass, double payload_scalar, double *M_out, double *C_out,
                        double *g_out, double *J_out, void *stream);

/*
 * Forward dynamics, fp64, per state: the joint accelerations a torque produces, and the inverse mass matrix -- the
 * other direction of tcmp_rne_batch, for torque-limited kinodynamic sampling, simulation under torque saturation and
 * operational-space control:
 *   qdd_out  [7][n]     qdd = M(q)^-1 (tau - h(q, qd)),  h = rne(q, qd, 0)
 *   Minv_out [7][7][n]  M(q)^-1, element (r, c) of state i at (r*7 + c)*n + i (tcmp_dynamics_batch's layout); exactly
 *                       symmetric (one triangle computed, the mirror written)
 * It is defined as the exact inverse of the torque test: tcmp_rne_batch(mode, ..., q, qd, qdd_out, ...,
 * TCMP_PAYLOAD_THRESHOLD_RAW) reproduces tau on all 7 joints, within the torque contract (1e-9 N.m).
 *   mode  TCMP_MODE_RNE: the payload is a rigid body on the flange iff m > 0 (tcmp_dynamics_batch's rule), in M and h.
 *         TCMP_MODE_DYN: M is the arm and hand without the payload; h includes the tool-point force m g at the grasp
 *         target for every m (negative too), as the dyn torque test applies it.
 *         Any other mode (NOV ignores qd and qdd, BASE computes nothing) is TCMP_ERR_INVALID_ARG.
 *   model         host pointer or NULL (compiled-in Panda), as in tcmp_dynamics_batch.
 *   q [7][n]; qd [7][n] or NULL (zeros); tau [7][n] or NULL (zeros: free motion under gravity).
 *   payload_mass  [n] or NULL (then payload_scalar applies to every state).
 * M is factored as LDL^T.  Non-finite inputs:
 *   - a NaN or infinite q (joint 1's too), qd, tau or mass of state i makes every qdd entry of state i NaN;
 *   - M^-1 of state i is NaN iff some q (joint 1's too) or the mass is non-finite; it does not read qd or tau;
 *   - other states are unaffected.
 * This follows tcmp_rne_batch, which returns NaN torques for a non-finite joint 1 (no finite qdd reproduces a NaN
 * torque), and deliberately differs from tcmp_dynamics_batch, whose M does not read q[0].
 * A pivot that is not > 0 (a caller record whose tail has no inertia about joint 7's axis, e.g. link 7, link8 and the
 * hand all massless and inertia-free) makes every output of the state NaN.
 * Each output may be NULL; at least one is required when n > 0.  A bad mode, n < 0, a bad record, a NULL q with n > 0
 * or both outputs NULL return TCMP_ERR_INVALID_ARG before any CUDA call; n == 0 otherwise returns TCMP_OK whatever
 * the buffers.  Enqueues only: no allocation, no synchronisation, so the call can be captured in a CUDA graph.
 */
int tcmp_forward_dynamics_batch(const tcmp_model *model, int mode, int64_t n, const double *q, const double *qd,
                                const double *tau, const double *payload_mass, double payload_scalar,
                                double *qdd_out, double *Minv_out, void *stream);

/*
 * Payload-mass intervals: which payload masses a state, or every waypoint of an RRT* edge, can carry within the torque
 * limits -- the inverse of the torque test, in one launch (a bisection over the mass takes ~26 torque-test launches to
 * reach 1e-6 kg over [0, 64] kg, and is wrong when the passing masses do not start at 0: a payload can pull a joint's
 * torque back inside its limit).  fp64 only.
 *
 * Every joint torque of the torque test is affine in the mass: tau(m) = a + m b for every mass the test attaches
 * (m > payload_threshold in rne / nov, every m in dyn).  For one state (q, qd, qdd) and mode:
 *   a [7]  the torque with no payload (mp_inertial = mp_tool = 0);
 *   b [7]  the torque one kilogram adds: rne / nov, the payload rigid body on link 7 (unit mass, axial first moment
 *          0.107, jxx = jyy = payload_radius^2 + 0.107^2, everything else 0); dyn, the tool-point gravity force (moment
 *          arm 0.107 + tool_z).  One forward Newton-Euler pass, a's backward pass, and b's (one wrench carried down).
 * Per joint j in 0..5 (joint 7 is never tested) the passing masses are the open interval {m : |a_j + m b_j| < L_j}:
 *   b_j > 0: ((-L_j - a_j) / b_j, (L_j - a_j) / b_j); b_j < 0: the ends swap;
 *   b_j == 0: (-inf, +inf) if |a_j| < L_j, else the empty (+inf, -inf);
 *   a_j or b_j NaN: (-inf, +inf) -- NaN never compares >= a limit, so the torque test passes the joint at every mass.
 * Outputs per state:
 *   m_lo = max over joints of the lower ends, m_hi = min of the upper ends, over all real m (either may be negative);
 *     the interval is empty iff m_lo >= m_hi.
 *   unloaded_ok = |a_j| < L_j for j = 0..5: the verdict with no payload attached.
 * Contract: for every mass the torque test attaches, its verdict is m_lo < m < m_hi; for a mass it does not attach it
 * is unloaded_ok -- except where some torque lies within 1e-9 N.m of a limit (the torque contract).  So the payload
 * threshold is not an input here: engine.payload_passes / engine.max_payload apply it.
 * A NaN or infinite joint angle (joint 1's too) makes every torque NaN: (-inf, +inf) and unloaded_ok = 1, as
 * tcmp_rne_batch judges such a state feasible at every mass.  TCMP_MODE_BASE writes (-inf, +inf, 1) and reads no input.
 *   model   host pointer or NULL (compiled-in Panda), as in tcmp_dynamics_batch.
 *   q, qd, qdd [7][n]: qd / qdd both given or both NULL (= static), ignored in TCMP_MODE_NOV; q may be NULL in BASE.
 *   m_lo_out, m_hi_out [n] double, unloaded_ok_out [n]: each may be NULL, at least one is required when n > 0.
 * n == 0 returns TCMP_OK whatever the buffers.  Bad mode, n < 0, n_waypoints < 1 or a missing q return
 * TCMP_ERR_INVALID_ARG before any CUDA call.  Enqueues only (no allocation, no synchronisation): graph-capturable.
 *
 * tcmp_edge_payload_interval: per edge qa -> qb, the intersection over its n_waypoints min-jerk samples, which are
 * exactly tcmp_edge_feasibility's (t = linspace(1/W, 1, W); static_only tests (q, 0, 0)): max of m_lo, min of m_hi,
 * AND of unloaded_ok.  Exact, so an edge's result means what a state's does: tcmp_edge_feasibility(..., m) returns
 * n_waypoints iff m lies in the edge's interval (or, for an unattached m, iff unloaded_ok).
 */
int tcmp_payload_interval_batch(const tcmp_model *model, int mode, int64_t n, const double *q, const double *qd,
                                const double *qdd, double *m_lo_out, double *m_hi_out, uint8_t *unloaded_ok_out,
                                void *stream);
int tcmp_edge_payload_interval(const tcmp_model *model, int mode, int64_t n_edges, int n_waypoints,
                               const double *qa, const double *qb, int static_only, double *m_lo_out,
                               double *m_hi_out, uint8_t *unloaded_ok_out, void *stream);

/*
 * Multi-GPU form of tcmp_rne_batch: the feasibility byte of state i is stored into dest_masks[d][dest_offset + i]
 * for every d < n_dest -- the gathered mask buffers of all ranks (this rank's own and its peers', mapped with
 * tcmp_peer_open over NVLink/NVSwitch).  This is the "NCCL all-gather of the masks" of BASELINE.json's
 * north_star fused into the producing kernel as a peer-store epilogue.  fp64 only.  Consumers on other ranks
 * must order their reads after this kernel (stream sync + any cross-rank barrier).
 */
#define TCMP_MAX_PEERS 8
int tcmp_rne_batch_scatter(int mode, int dtype, int64_t n, const void *q, const void *qd, const void *qdd,
                           const void *payload_mass, double payload_scalar, double payload_threshold,
                           void *tau_out, int n_dest, void *const *dest_masks, int64_t dest_offset,
                           void *stream);
/*
 * NVLS form of tcmp_rne_batch_scatter: the gathered buffers are ALSO mapped at one NVSwitch multicast address
 * (mc_masks: cuMulticast* / torch symmetric memory's multicast_ptr; same layout, same dest_offset).  Full warps store
 * their 32 verdicts with two 16-byte multimem.st -- the switch replicates them into every rank's buffer, so a step
 * issues 1/n_dest of the store requests and outgoing NVLink bytes of the unicast form.  The batch's last partial warp
 * (multimem.st has no byte form) goes through dest_masks as in tcmp_rne_batch_scatter, which therefore must be the
 * unicast mappings of the same buffers.  `base` mode and a dest_offset that is not a multiple of 16 take the unicast
 * path entirely.
 */
int tcmp_rne_batch_scatter_mc(int mode, int dtype, int64_t n, const void *q, const void *qd, const void *qdd,
                              const void *payload_mass, double payload_scalar, double payload_threshold,
                              void *tau_out, int n_dest, void *const *dest_masks, void *mc_masks, int64_t dest_offset,
                              void *stream);
/*
 * Completion flags of the fused gathers (no host barrier, no collective call, CUDA-graph capturable).  Every rank owns
 * a sync block (TCMP_PEER_SYNC_BYTES of tcmp_peer_alloc memory, which arrives zeroed; dest_sync[r] = rank r's block as
 * mapped on this rank, dest_sync[rank] = this rank's own).
 *   tcmp_peer_signal, enqueued after a scatter kernel (tcmp_rne_batch_scatter, tcmp_edge_feasibility_scatter), stores
 *     this rank's next epoch into the `arrived[rank]` word of every rank's block: completion of the scatter kernel has
 *     drained its peer stores, a system-scope fence orders the flag behind them.
 *   tcmp_peer_wait holds its stream until every rank has published this rank's current epoch (acquire loads) -- from
 *     then on this rank's gathered buffer holds every rank's results of that step.
 * Both are one-CTA kernels; run them on a side stream behind an event of the scatter kernel and they cost the step
 * nothing (3 us in-stream).  Ordering contract for consumers, with the gathered buffer cycling through 3 copies
 * (distributed.PeerMaskBuffer): reads of step i's copy are enqueued on the stream that carries signal/wait, after
 * wait(i) and before signal(i + 1); the scatter kernel of step i + 3 is ordered after this rank's wait(i + 1) -- every
 * peer has then published i + 1, i.e. finished reading step i.
 */
#define TCMP_PEER_SYNC_BYTES 128
/* The gather as its own small kernel: copy `bytes` of a result block this rank has produced (device pointer src) into
 * dests[d] + dest_offset for every d < n_dest.  On a side stream behind the producing kernel (tcmp_rne_batch,
 * tcmp_edge_feasibility, tcmp_ik_batch counts ...) it overlaps the next step; the alternative to the fused epilogues
 * for results the kernels do not scatter themselves, and measured against them in profiles/r02/. */
int tcmp_peer_push(const void *src, int64_t bytes, int n_dest, void *const *dests, int64_t dest_offset, void *stream);
int tcmp_peer_signal(int rank, int n_dest, void *const *dest_sync, void *stream);
int tcmp_peer_wait(void *own_sync, int n_ranks, void *stream);
/* Peer-shareable device memory (cudaMalloc + CUDA IPC): allocate on the current device and export a 64-byte
 * handle; another process on the same node opens the handle to obtain a pointer valid on ITS current device. */
#define TCMP_IPC_HANDLE_BYTES 64
int tcmp_peer_alloc(void **dev_ptr, int64_t bytes, unsigned char *handle_out);
int tcmp_peer_free(void *dev_ptr);
int tcmp_peer_open(const unsigned char *handle, void **peer_ptr);
int tcmp_peer_close(void *peer_ptr);

/*
 * RRT* edge check: for every edge (qa -> qb) generate n_waypoints samples of the 2-point
 * min-jerk (min_jerk_v2.py:96-142 coefficients, :176-181 t = linspace(1/W, 1, W), :216-220
 * x/v/a) and run the torque test on each (q, qd, qdd); first_fail_out[e] = index of the first
 * infeasible waypoint, or n_waypoints when the edge is feasible (the prefix semantics of
 * safe_path_force_aware, rrt_star.py:90-98, and the stop-at-first-failure of :208-210).
 *   qa, qb [7][n_edges];  static_only != 0 tests (q, 0, 0) per waypoint as tree growth does
 *   (rrt_star.py:95,172 call torque(q) without velocities).
 */
int tcmp_edge_feasibility(int mode, int dtype, int64_t n_edges, int n_waypoints, const void *qa,
                          const void *qb, double payload_scalar, double payload_threshold,
                          int static_only, int32_t *first_fail_out, void *stream);

/* Multi-GPU form of tcmp_edge_feasibility (fp64): the first-failure index of edge e is stored into
 * dest_first_fail[d][dest_offset + e] (int32) for every d < n_dest -- the gathered buffers of all ranks, peers
 * mapped with tcmp_peer_open.  See tcmp_rne_batch_scatter. */
int tcmp_edge_feasibility_scatter(int mode, int64_t n_edges, int n_waypoints, const void *qa, const void *qb,
                                  double payload_scalar, double payload_threshold, int static_only, int n_dest,
                                  void *const *dest_first_fail, int64_t dest_offset, void *stream);

/*
 * Final-trajectory check (rrt_star.py:203-210 + panda_primitives.py:299-316): evaluate the
 * piecewise quintic with coefficients coeffs[seg][joint][6] (a0..a5, unit segment duration,
 * min_jerk_v2.py:121-141) at samples_per_segment points t = linspace(1/S, 1, S) per segment
 * and torque-test every sample.  Sample index s = seg*S + it.  Outputs (each may be NULL):
 *   q_out/qd_out/qdd_out/tau_out [7][n_seg*S], feasible_out [n_seg*S],
 *   first_fail_out[1] = first infeasible sample or n_seg*S.  first_fail_out must be
 *   initialised by the caller to n_seg*S (the kernel atomicMin's into it).
 *   TCMP_MODE_BASE (the constant-true test, panda_primitives.py:13-16): feasible_out is all 1, first_fail_out is
 *   not touched, and q_out / qd_out / qdd_out / tau_out are still written -- the samples are the trajectory the
 *   planner returns and tau_out holds the rne torques (payload_scalar as given) that Conf logs for every sample
 *   regardless of the test mode (utils.py:3376-3378).
 */
int tcmp_traj_feasibility(int mode, int dtype, int n_seg, int samples_per_segment,
                          const double *coeffs, double payload_scalar, double payload_threshold,
                          void *q_out, void *qd_out, void *qdd_out, void *tau_out,
                          uint8_t *feasible_out, int32_t *first_fail_out, void *stream);

/*
 * Batched analytic IK for the Panda link0 -> link8 chain, joint 7 free.  Replaces
 * ComputeIk (ikfast_panda_arm.cpp:12770; IKSolver::ComputeIk :412, rotationfunction0 :3115)
 * and the per-solution expansion of get_ik (:12885-12902, ikfast.h:167-181).
 *   rot9 [9][n] row-major rotation, trans3 [3][n];
 *   free_vals [n_free][n], or [n_free] when free_broadcast != 0;
 *   solve index s = pose*n_free + f;  sols_out [n*n_free][8][7] (may be NULL: counts only),
 *   count_out [n*n_free] = number of solutions (0..8).
 *   status_out [n*n_free] or NULL:
 *     bit 0 (1) = the solve entered a singular branch of the reference's decision tree.  With bit 1 clear the
 *       branch was RESOLVED the way the reference resolves it: shoulder singularity (j2 pinned to 0, :3209-3325),
 *       elbow singularity at j4 = 2.63084142381503 (one member of the one-parameter family, :2774-2835) and at
 *       j4 = 0 (:2436-2598), wrist centre on the joint-6 axis (:509-2346 -- no arm configuration reaches such a
 *       pose and every leaf of that sub-tree rejects it: 0 solutions).
 *     bit 1 (2) = the solve reached a branch of the generated solver that this library does NOT implement and the
 *       solutions of that branch were dropped: the count may be lower than the reference's.  Those branches need an
 *       input that is not a rigid transform (a rotation matrix off orthonormal by more than ~1e-6) or a floating-point
 *       tie on a 1e-6 guard; none is reached by the structured singular-pose sweeps of tests/ (profiles/r02/
 *       ik_reference_coverage.md lists the reference's reached lines).
 *     bit 3 (8) = ill-conditioned count: a duplicate-root test (|d cos|, |d sin| < 1e-6, :495) or a singular-branch
 *       guard came within 1 % of its threshold, or joint 4 lies within 6e-5 rad of the elbow singularity (|K| < 2e-5,
 *       where j5's rounding residue reaches j4 amplified by C^2 / K^2).  Two roots 1e-6 apart come from an asin / acos argument 1.2e-13 from
 *       +-1, where one ulp of the argument moves them by 3e-10: the reference's own count then depends on its libm and
 *       compiler flags.  The host build of the solver (glibc, no contraction) returns the reference's solutions bit
 *       for bit; on the GPU (CUDA libm) 47 of 36 M structured singular solves differed, all with this bit set, and 0 of
 *       100 M random-pose solves.
 *     bit 2 (4) = non-finite input (the reference throws from IKFAST_ASSERT; here the solve returns 0 solutions).
 */
int tcmp_ik_batch(int64_t n, const double *rot9, const double *trans3, const double *free_vals,
                  int n_free, int free_broadcast, double *sols_out, int32_t *count_out,
                  uint8_t *status_out, void *stream);

/*
 * Goal-IK selection: for every pose sweep the free joint (free_vals as in tcmp_ik_batch), solve, keep only
 * solutions inside [q_lo, q_hi] (HOST arrays of 7; ikfast.py:167, franka_ik_fast.py:55-57) that pass the STATIC
 * torque test `mode` with payload `payload_scalar` (panda_primitives.py:263; TCMP_MODE_BASE = no torque test), and
 * return the one nearest to q_ref ([7][n], or [7] when ref_broadcast != 0) in the max norm (use_max_norm != 0,
 * closest_inverse_kinematics ikfast.py:172-188) or the Euclidean norm (ik_utils.select_solution :43-52).
 *   best_q [7][n], best_cost [n] (+inf when no solution survives), n_valid [n] = surviving solutions.
 * Ties keep the first solution in (free value, solver order).  Costs rank in numeric order and a NaN cost after every
 * number, +inf included: a NaN in one joint of q_ref makes every cost NaN (in both norms), and the first surviving
 * solution in (free value, solver order) is returned with best_cost = NaN and n_valid unchanged, as the drop-in's
 * sort does.  +-inf in q_ref makes every cost +inf: again the first survivor, with best_cost = +inf.  With no
 * survivor best_q is all zeros, best_cost +inf and n_valid 0.  A NaN limit bounds nothing (a joint passes unless it
 * is < lo or > hi); lo > hi leaves no survivor.  A non-finite free value gives no solutions; the others are unaffected.
 * NOT the reference's order of operations: the reference takes the nearest IN-LIMIT solution first
 * (closest_inverse_kinematics) and then fails the whole grasp if that single configuration exceeds the torque limits
 * (panda_primitives.py:263), whereas this call picks the nearest solution among those that ALSO pass the torque test --
 * it can succeed where the reference returns None.  For the reference's semantics call it with TCMP_MODE_BASE (limit
 * filter + nearest only) and run tcmp_rne_batch on best_q, which is what panda_primitives.planner_fn_force_aware does.
 */
int tcmp_ik_select(int64_t n, const double *rot9, const double *trans3, const double *free_vals, int n_free,
                   int free_broadcast, const double *q_ref, int ref_broadcast, const double *q_lo_host,
                   const double *q_hi_host, int mode, double payload_scalar, double payload_threshold,
                   int use_max_norm, double *best_q, double *best_cost, int32_t *n_valid, void *stream);

/* Batched FK, replaces ComputeFk (ikfast_panda_arm.cpp:307-395): q [7][n] -> trans3 [3][n],
 * rot9 [9][n] (row-major), link0 -> link8. */
int tcmp_fk_batch(int64_t n, const double *q, double *trans3, double *rot9, void *stream);

/*
 * Synthetic-scene collision predicate (stand-in for utils.get_collision_fn, utils.py:3165-3218, whose PyBullet
 * backend is out of scope): joint-limit test first (utils.py:3177-3178), then link spheres from the DH forward
 * kinematics against axis-aligned boxes / spheres.  Obstacle and limit arrays are HOST memory (copied into the
 * launch parameters).  hit_out[i] = 1 when configuration i collides or violates a joint limit.  As in the NumPy
 * stand-in (collision.get_collision_fn), a NaN joint passes the limit test and the link spheres it moves hit nothing;
 * a +-inf joint is outside any finite limit.
 */
#define TCMP_MAX_OBSTACLES 32
typedef struct {
    int32_t kind;      /* 0 = axis-aligned box, 1 = sphere */
    int32_t reserved;
    double center[3];
    double half[3];    /* box half extents; sphere: half[0] = radius */
} tcmp_obstacle;
int tcmp_collision_batch(int64_t n, const double *q, int n_obs, const tcmp_obstacle *obstacles_host,
                         const double *q_lo_host, const double *q_hi_host, double payload_radius,
                         uint8_t *hit_out, void *stream);
/*
 * RRT* tree-growth edge check, safe_path_force_aware(extend(q1, q2), collision, torque) (rrt_star.py:90-98,172) for
 * MANY candidate edges in one launch.  The extend steps are generated on the device exactly as
 * utils.get_extend_fn / get_refine_fn do (utils.py:3031-3041,3068-3077: floor(||(q2-q1)/resolution||_2) + 1
 * configurations, q1 excluded, q2 included); each is tested for collision and, only if collision-free, with the
 * STATIC torque test `mode` (tree growth never passes velocities, rrt_star.py:95).
 *   q1, q2 [7][n_edges] (device); resolution_host [7];
 *   n_steps_out[e] = number of configurations on edge e, prefix_out[e] = length of the safe prefix (0..n_steps).
 */
int tcmp_extend_prefix(int mode, int64_t n_edges, const double *q1, const double *q2,
                       const double *resolution_host, int n_obs, const tcmp_obstacle *obstacles_host,
                       const double *q_lo_host, const double *q_hi_host, double payload_radius,
                       double payload_scalar, double payload_threshold, int32_t *n_steps_out,
                       int32_t *prefix_out, void *stream);

/*
 * The planner-side entry points with a caller-supplied inertial set: same arguments as the functions of the same
 * name without the suffix, preceded by the record (host pointer, read during the call; NULL = compiled-in Panda).
 * Together with tcmp_rne_batch_model they let a whole plan -- tree growth (extend prefix), goal-IK selection, edge
 * checks, final trajectory check and torque logging -- run on another hand / payload lever / limit set.
 */
int tcmp_edge_feasibility_model(const tcmp_model *model, int mode, int dtype, int64_t n_edges, int n_waypoints,
                                const void *qa, const void *qb, double payload_scalar, double payload_threshold,
                                int static_only, int32_t *first_fail_out, void *stream);
int tcmp_traj_feasibility_model(const tcmp_model *model, int mode, int dtype, int n_seg, int samples_per_segment,
                                const double *coeffs, double payload_scalar, double payload_threshold,
                                void *q_out, void *qd_out, void *qdd_out, void *tau_out, uint8_t *feasible_out,
                                int32_t *first_fail_out, void *stream);
int tcmp_ik_select_model(const tcmp_model *model, int64_t n, const double *rot9, const double *trans3,
                         const double *free_vals, int n_free, int free_broadcast, const double *q_ref,
                         int ref_broadcast, const double *q_lo_host, const double *q_hi_host, int mode,
                         double payload_scalar, double payload_threshold, int use_max_norm, double *best_q,
                         double *best_cost, int32_t *n_valid, void *stream);
int tcmp_extend_prefix_model(const tcmp_model *model, int mode, int64_t n_edges, const double *q1, const double *q2,
                             const double *resolution_host, int n_obs, const tcmp_obstacle *obstacles_host,
                             const double *q_lo_host, const double *q_hi_host, double payload_radius,
                             double payload_scalar, double payload_threshold, int32_t *n_steps_out,
                             int32_t *prefix_out, void *stream);

/*
 * Host-buffer variants: the call a Python/C caller makes with ordinary (ideally pinned) host
 * arrays.  They stage through a caller-created workspace (device buffers + streams), pipeline
 * host->device copies, kernels and device->host copies in chunks, and return after the results
 * are in the host output arrays.
 */
typedef struct tcmp_workspace tcmp_workspace;
/* chunk_states = states per pipeline stage (0 = default 1<<18). */
int tcmp_workspace_create(tcmp_workspace **ws, int64_t chunk_states);
int tcmp_workspace_destroy(tcmp_workspace *ws);
int tcmp_rne_batch_host(tcmp_workspace *ws, int mode, int dtype, int64_t n, const void *q,
                        const void *qd, const void *qdd, const void *payload_mass,
                        double payload_scalar, double payload_threshold, void *tau_out,
                        uint8_t *feasible_out);
/* The same call without the final wait: it enqueues the whole chunk pipeline on the workspace's streams and returns.
 * Consecutive calls on one workspace pipeline across batches (the host->device copies of batch i + 1 run while batch
 * i's last chunk is still computing and reading back); the output arrays of a batch are complete -- and its input
 * arrays may be reused -- after tcmp_workspace_sync.  Host arrays must be pinned for the overlap to happen. */
int tcmp_rne_batch_host_async(tcmp_workspace *ws, int mode, int dtype, int64_t n, const void *q,
                        const void *qd, const void *qdd, const void *payload_mass,
                        double payload_scalar, double payload_threshold, void *tau_out,
                        uint8_t *feasible_out);
int tcmp_workspace_sync(tcmp_workspace *ws);
int tcmp_edge_feasibility_host(tcmp_workspace *ws, int mode, int dtype, int64_t n_edges,
                               int n_waypoints, const void *qa, const void *qb,
                               double payload_scalar, double payload_threshold, int static_only,
                               int32_t *first_fail_out);
int tcmp_ik_batch_host(tcmp_workspace *ws, int64_t n, const double *rot9, const double *trans3,
                       const double *free_vals, int n_free, int free_broadcast, double *sols_out,
                       int32_t *count_out, uint8_t *status_out);
/* Pinned host memory helpers (cudaHostAlloc / cudaFreeHost). */
int tcmp_host_alloc(void **ptr, int64_t bytes);
int tcmp_host_free(void *ptr);

/* FP64 FMA throughput microbenchmark (the roofline denominator the reference never had):
 * runs `iters` dependent-chain DFMA rounds on every SM and writes achieved FLOP/s. */
int tcmp_fp64_peak(int iters, double *flops_out, void *stream);

/* Model constants (read-only): torque limits (7), joint lower/upper (7+7), velocity limits (7). */
int tcmp_get_limits(double *torque7, double *q_lo7, double *q_hi7, double *qd_max7);

#ifdef __cplusplus
}
#endif
#endif /* TCMP_H_ */
