/*
 * r2ik.h -- C ABI of libr2ik.so: B200 (sm_100a) CUDA implementation of the Reachy2
 * symbolic 7-DoF arm IK hot path of pollen-robotics/reachy2_symbolic_ik.
 *
 * The reference is a pure-Python library with no FFI seam; its public surface for this
 * path is two classes.  Each entry point below names the reference interface it replaces
 * (paths relative to the reference checkout):
 *
 *   r2ik_create / r2ik_destroy / r2ik_get_constants
 *        SymbolicIK.__init__                       src/reachy2_symbolic_ik/symbolic_ik.py:26-83
 *        (+ get_singularity_position               src/reachy2_symbolic_ik/utils.py:26-43)
 *   r2ik_symik_solve_f64
 *        SymbolicIK.is_reachable                   symbolic_ik.py:121-282
 *        + theta_to_joints_func = get_joints       symbolic_ik.py:697-863
 *   r2ik_symik_solve_f32
 *        the same, FP32 fast path (float poses in, float results out)
 *   r2ik_symik_no_limits_f64
 *        SymbolicIK.is_reachable_no_limits         symbolic_ik.py:85-119  (+ get_joints)
 *   r2ik_elbow_positions_f64
 *        SymbolicIK.get_elbow_position             symbolic_ik.py:684-695
 *        (on the circle stored by is_reachable :197 or by is_reachable_no_limits :114-116)
 *   r2ik_symik_sweep_f64
 *        theta_to_joints_func called at K elbow angles per pose
 *                                                  symbolic_ik.py:121-282, 85-119, 697-863
 *        (angles placed like get_best_discrete_theta utils.py:366-375)
 *   r2ik_symik_scalar_f64
 *        the scalar call sequence is_reachable / is_reachable_no_limits -> get_elbow_position
 *        -> get_joints of ONE pose in one launch   symbolic_ik.py:121-282, 85-119, 684-695, 697-863
 *        (the reference's consumer calls it once per control tick, src/example/example_control.py:9-27)
 *   r2ik_ctl_discrete_f64
 *        ControlIK.symbolic_inverse_kinematics(name, M, "discrete")
 *                                                  control_ik.py:162-274, 409-462, 464-497
 *        (get_best_discrete_theta utils.py:334-396, limit_theta_to_interval utils.py:93-112,
 *         limit_orbita3d_joints_wrist :508-532, allow_multiturn :493-505,
 *         multiturn_safety_check :535-568)
 *   r2ik_ctl_discrete_scan_f64
 *        the same, exhaustive warp-cooperative scan of the K samples (cross-check)
 *   r2ik_ctl_continuous_f64
 *        ControlIK.symbolic_inverse_kinematics(name, M, "continuous") over trajectories
 *                                                  control_ik.py:276-407
 *        (get_best_continuous_theta2 utils.py:220-264, tend_to_preferred_theta :115-127,
 *         get_best_theta_to_current_joints :267-331, continuity_check :571-589)
 *   r2ik_reach_map_u32
 *        grid sweep of is_reachable (shape of src/benchmark/ik_comparison.py:137-181)
 *   r2ik_reach_map_f64_u32
 *        the same volume, every pair by the all-FP64 flag solve (cross-check)
 *   r2ik_interval_limit
 *        interval_limit + l_arm mirroring          control_ik.py:225-252
 *   r2ik_ctl_ctor_theta_f64
 *        ControlIK.__init__'s previous_theta seed  control_ik.py:142-159 (utils.py:267-331)
 *   r2ik_fk_f64
 *        forward kinematics of the arm chain of config_files/reachy2.urdf (torso -> arm tip).
 *        The reference has no FK of its own: its examples call the Reachy SDK's
 *        (src/example/test_continuous_ik.py:146).  Used for synthetic FK-sampled poses and
 *        the FK round-trip property tests (SURVEY.md 8(f).2).
 *
 * Conventions
 *   - All data pointers are DEVICE pointers unless a parameter says "host".
 *   - Pose buffers (poses / M / current_pose) must be 16-byte aligned (128-bit loads);
 *     a misaligned pointer is R2IK_ERR_ARG.
 *   - Every launch entry takes a cudaStream_t (passed as void*; NULL = legacy default
 *     stream), is asynchronous with respect to the host and allocates nothing.
 *   - Return value: 0 = ok, > 0 = argument error (R2IK_ERR_*), < 0 = -(cudaError_t).
 *   - No exceptions cross this boundary; r2ik_last_error() gives a static message.
 *   - The library has no CPU implementation of any entry point.
 */
#ifndef R2IK_H
#define R2IK_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define R2IK_ABI_VERSION 5 /* 5: + symik_sweep; 4: + ctl_discrete_compact; 3: + symik_scalar, stream_synchronize, host pipelines, ctl_ctor_theta, reach_map_range_u16; no_limits / projected in elbow_positions, prev_joints in
                              no_limits, nullable `reachable`, test hook of the phased continuous entry as a parameter */

/* argument errors */
#define R2IK_ERR_NULL 1
#define R2IK_ERR_ARG 2
#define R2IK_ERR_ARM 3
#define R2IK_ERR_NO_DEVICE 4

/* per-pose state codes; the Python facade maps them to the reference's exact strings */
#define R2IK_STATE_REACHABLE 0           /* "reachable"                  symbolic_ik.py:234 */
#define R2IK_STATE_POSE_OUT_OF_REACH 1   /* "Pose out of reach"          symbolic_ik.py:300 */
#define R2IK_STATE_BACKWARD_POSE 2       /* "Backward pose"              symbolic_ik.py:306 */
#define R2IK_STATE_WRIST_OUT_OF_RANGE 3  /* "wrist out of range"         symbolic_ik.py:159 */
#define R2IK_STATE_LIMITED_BY_WRIST 4    /* "limited by wrist"           symbolic_ik.py:262 */
#define R2IK_STATE_SHOULD_NOT_HAPPEN 5   /* "out of reach - should not happen" :281 */
#define R2IK_STATE_LIMITED_BY_SHOULDER 6 /* "limited by shoulder"        control_ik.py:363,452 */
#define R2IK_STATE_EMPTY 7               /* ""                           control_ik.py:297 */
#define R2IK_STATE_EMERGENCY 8           /* emergency text               utils.py:544-566,584-586 */
#define R2IK_STATE_INVALID_ROTATION 9    /* scipy from_matrix: det <= 0 (ValueError) */

/* pose layouts */
#define R2IK_POSE_EULER6 0 /* n x 6 : x y z roll pitch yaw  (the reference's goal_pose, 2x3)     */
#define R2IK_POSE_MAT4 1   /* n x 16: row-major 4x4; converted like control_ik.py:216 (no snap) */
#define R2IK_POSE_MAT34 2  /* n x 12: the 3x4 top of that matrix (the last row is never read);    */
                           /*   r2ik_symik_solve_f64 and r2ik_symik_sweep_f64 only                 */

/* emergency reason bits (utils.py:544-566, 584-586) */
#define R2IK_EMG_SHOULDER_PITCH 1
#define R2IK_EMG_ELBOW_YAW 2
#define R2IK_EMG_WRIST_YAW 4
#define R2IK_EMG_DISCONTINUITY 8

/* Raw constructor arguments of SymbolicIK for ONE arm (symbolic_ik.py:26-63). */
typedef struct R2ikArmConfig {
  double shoulder_position[3];
  double shoulder_orientation_deg[3]; /* xyz euler, degrees */
  double upper_arm_size;
  double forearm_size;
  double tip_position[3];
  double elbow_limit_deg;         /* 127   */
  double wrist_limit_deg;         /* 42.5  */
  double projection_margin;       /* 1e-8  */
  double backward_limit;          /* 0.02  */
  double normal_vector_margin;    /* 1e-7  */
  double singularity_offset;      /* 0.03; ControlIK: -1.01 (non DVT) / 0.03 (DVT) */
  double singularity_limit_coeff; /* 1.0   */
  int32_t side;                   /* +1 = r_arm, -1 = l_arm */
  int32_t reserved;
} R2ikArmConfig;

/* Derived per-arm constants, readable by the host facade (attributes of SymbolicIK). */
typedef struct R2ikArmConstants {
  double gripper_size;
  double max_arm_length;
  double shoulder_wrist_min_distance;
  double elbow_singularity_position[3];
  double wrist_singularity_position[3];
} R2ikArmConstants;

/* Per-call ControlIK parameters (control_ik.py:162-172, 225-252). */
typedef struct R2ikCtlParams {
  double preferred_theta;      /* per-call value, already mirrored for l_arm             */
  double preferred_theta_ctor; /* ControlIK.preferred_theta[arm] (control_ik.py:133-141)  */
  double interval_limit[2];    /* already mirrored for l_arm (r2ik_interval_limit)        */
  double d_theta_max;          /* 0.01                                                    */
  double orbita3d_max_angle;   /* deg2rad(42.5)                                           */
  int32_t nb_search_points;            /* discrete: 20                                    */
  int32_t nb_search_points_continuous; /* continuous: 10                                  */
} R2ikCtlParams;

/* Per-trajectory controller state = ControlIK's previous_theta / previous_sol / init /
 * emergency_* (control_ik.py:60-84), explicit so trajectories can be chunked and resumed. */
typedef struct R2ikTrajState {
  double previous_theta;
  double previous_sol[7];
  int32_t has_previous_sol; /* 0: next waypoint re-initialises (first call / timeout) */
  int32_t init;
  int32_t emergency_stop;
  int32_t emergency_bits;
} R2ikTrajState;

/* Kinematic chain torso -> tip for r2ik_fk_f64: 7 revolute joints.  fixed[k] is the constant
 * 3x4 row-major transform [R|t] between joint k-1 and joint k (fixed[7]: last joint -> tip),
 * axis[k] the unit rotation axis of joint k in its own frame (URDF <origin>/<axis>). */
typedef struct R2ikFkChain {
  double fixed[8][12];
  double axis[7][3];
} R2ikFkChain;

/* One scalar call sequence of SymbolicIK (r2ik_symik_scalar_f64). */
typedef struct R2ikScalarQuery {
  double goal_pose[6];        /* x y z roll pitch yaw: the reference's goal_pose [[x,y,z],[r,p,y]]  */
  double theta;               /* elbow angle for get_elbow_position / get_joints (has_theta != 0)   */
  double previous_joints[7];  /* get_joints(theta, previous_joints); zeros = the reference default  */
  int32_t no_limits;          /* 0: is_reachable, 1: is_reachable_no_limits                         */
  int32_t has_theta;          /* 0: theta = theta_interval[0]                                       */
} R2ikScalarQuery;

typedef struct R2ikScalarResult {
  double interval[2];              /* theta_interval; NaN when the call failed                          */
  double joints[7];                /* get_joints(theta, previous_joints); NaN when unreachable          */
  double elbow[3];                 /* elbow get_joints returns (after make_elbow_projection, if fired)  */
  double elbow_on_circle[3];       /* get_elbow_position(theta): defined once the circle is stored,     */
                                   /*   i.e. also for "limited by wrist" (symbolic_ik.py:197)           */
  double goal_position_solved[3];  /* self.goal_pose[0] / self.wrist_position after is_reachable or     */
  double wrist_position_solved[3]; /*   is_reachable_no_limits (symbolic_ik.py:143-171, 91-112)         */
  double goal_position[3];         /* ... after get_joints (symbolic_ik.py:711-716)                     */
  double wrist_position[3];
  int32_t reachable;               /* 0 / 1                                                             */
  int32_t state;                   /* R2IK_STATE_*                                                      */
  int32_t projected;               /* 1: make_elbow_projection fired => the reference returns a         */
                                   /*   3-vector elbow instead of [x, y, z, 1] (symbolic_ik.py:714,863) */
  int32_t reserved;
} R2ikScalarResult;

typedef struct r2ik_context *r2ik_handle;

int r2ik_abi_version(void);
const char *r2ik_last_error(void);

/* cfg: host pointer.  device: CUDA ordinal the handle launches on. */
int r2ik_create(const R2ikArmConfig *cfg, int device, r2ik_handle *out);
int r2ik_destroy(r2ik_handle h);
int r2ik_get_constants(r2ik_handle h, R2ikArmConstants *out /* host */);

/* interval_limit of ControlIK for an arm; out: host double[2]. */
int r2ik_interval_limit(int side, int low_elbow, double *out);

/* is_reachable + get_joints(theta) for n independent poses (fresh solver state per pose).
 * theta: nullable; NULL => theta_interval[0].  prev_joints: nullable 7 doubles (device),
 * broadcast; NULL => zeros (the reference default).  Unreachable poses get NaN interval /
 * joints / elbow.  Any output pointer except `state` may be NULL (state == R2IK_STATE_REACHABLE <=> reachable, so a
 * lean host record is state + joints = 57 bytes per pose). */
int r2ik_symik_solve_f64(r2ik_handle h, int pose_kind, const double *poses, const double *theta,
                         const double *prev_joints, int64_t n, uint8_t *reachable, uint8_t *state,
                         double *interval, double *joints, double *elbow, void *stream);

/* FP32 fast path of r2ik_symik_solve_f64 (BASELINE.json north_star: "FP32 path within a stated 1e-4 rad"):
 * float poses (n x 16 row-major 4x4, 16-byte aligned, or n x 6, 8-byte aligned), float outputs.  The solve runs
 * in FP32 with an FP64 front end for the cancelling differences; a pose within FP32 rounding of one of the
 * reference's decisions (state codes, branch cuts, elbow projection) or with an ill-conditioned angle (interval-end
 * lever < 3 mm, shoulder-pitch lever < 1.7 cm, elbow-yaw lever < 3.2 cm, any other atan2 lever < 2 mm) is
 * appended to escalated_idx and re-solved by the FP64 solver on the same inputs in a second kernel of the same
 * call, so states / flags are those of the FP64 path on the widened inputs.
 * Stated bound (against the FP64 solve of the same float inputs; tests/parity.py holds every test set to it, no pose
 * excused): joints and intervals within 1e-4 rad for >= 99.99 % of the poses and within 3e-4 rad for all of them
 * (host soak of 12 M poses, 7.5 M of them reachable, both arms, both layouts, profiles/r2_soak_f32_bound_4242.log:
 * 0 state mismatches, p99.999 <= 9.4e-5, max 2.2e-4, 28 poses over 1e-4 -- nearly straight arms);
 * 2-5 % of FK-sampled poses are re-solved in FP64.
 * escalated_idx: n uint32 of caller-owned device scratch; n_escalated: one uint32 on the device, set by the call
 * to the number of re-solved poses (also for n = 0).  theta / prev_joints as in r2ik_symik_solve_f64 (float).  n < 2^32. */
int r2ik_symik_solve_f32(r2ik_handle h, int pose_kind, const float *poses, const float *theta,
                         const float *prev_joints, int64_t n, uint8_t *reachable, uint8_t *state,
                         float *interval, float *joints, float *elbow, uint32_t *escalated_idx,
                         uint32_t *n_escalated, void *stream);

/* is_reachable_no_limits + get_joints(theta[i], previous_joints).  prev_joints: nullable (zeros); prev_stride 0 = one
 * vector of 7 broadcast, 7 = one per pose.  projected: nullable, 1 where make_elbow_projection fired. */
int r2ik_symik_no_limits_f64(r2ik_handle h, int pose_kind, const double *poses, const double *theta,
                             const double *prev_joints, int32_t prev_stride, int64_t n, double *joints,
                             double *elbow, uint8_t *projected, void *stream);

/* get_elbow_position(thetas[i][k]) after is_reachable(poses[i]) (no_limits = 0) or is_reachable_no_limits (1); NaN
 * when no circle was stored.  projected: nullable n*K, 1 where get_joints(theta) would project the elbow. */
int r2ik_elbow_positions_f64(r2ik_handle h, int pose_kind, const double *poses, const double *thetas,
                             int32_t K, int64_t n, int32_t no_limits, double *elbows /* n*K*3 */,
                             uint8_t *projected, void *stream);

/* Elbow-angle sweep: for every pose i and sample k < K, is_reachable(poses[i]) (no_limits = 1: is_reachable_no_limits)
 * followed by get_joints(theta_ik, previous_joints) as the FIRST call on that solve (symbolic_ik.py:121-282, 85-119,
 * 697-863) -- bit-identical to r2ik_symik_solve_f64 (r2ik_symik_no_limits_f64) on the pose repeated K times with the
 * flattened angles.  The pose is solved once per tile of up to 1 024 of its samples.  The reference's closure, called
 * repeatedly on one solver, leaks state from one call to the next (once the elbow projection fires, later calls see a
 * shifted goal); like r2ik_symik_solve_f64 this entry does not reproduce that leak.
 * Angles: thetas non-NULL: row i at thetas + i * theta_stride, theta_stride = K (one row per pose) or 0 (one row of K
 * shared by all poses).  thetas NULL: K samples on each pose's theta_interval, placed as get_best_discrete_theta places
 * them (utils.py:366-375): linspace(pi/2, 5pi/2, K) for a full circle, a wrapped interval unrolled by +2pi.
 * A pose that is not reachable ("limited by wrist" included) gets NaN thetas_used / joints / elbow and projected = 0 for
 * all K samples.  state: n; interval: n x 2, nullable; thetas_used (the angles used): n x K, nullable; joints:
 * n x K x 7; elbow: n x K x 3, nullable (get_joints' elbow); projected: n x K, nullable, 1 where make_elbow_projection
 * fired.  prev_joints: nullable, 7 doubles broadcast (NULL = zeros).  K >= 1; n * K * 7 must fit int64. */
int r2ik_symik_sweep_f64(r2ik_handle h, int pose_kind, const double *poses, int64_t n, const double *thetas,
                         int32_t theta_stride, int32_t K, int32_t no_limits, const double *prev_joints, uint8_t *state,
                         double *interval, double *thetas_used, double *joints, double *elbow, uint8_t *projected,
                         void *stream);

/* The scalar call sequence of SymbolicIK for one pose in one launch.  query: HOST pointer (passed to the kernel by
 * value).  out: any device-accessible address -- device memory, or pinned host memory (cudaHostAlloc / torch
 * pin_memory: mapped under unified addressing), in which case the call needs no copy at all. */
int r2ik_symik_scalar_f64(r2ik_handle h, const R2ikScalarQuery *query, R2ikScalarResult *out, void *stream);

/* ControlIK.__init__'s seed of previous_theta[arm] (control_ik.py:142-159): is_reachable_no_limits on current_pose,
 * then get_best_theta_to_current_joints as the constructor calls it -- with the list of BOTH arms' joints, so its
 * cost runs over n_rows rows of 7 (utils.py:267-331).  current_joints_rows (n_rows x 7, n_rows <= 7) and
 * current_pose (row-major 4x4): HOST pointers, passed to the kernel by value.  out_theta: one double at any
 * device-accessible address (NaN when the current pose has no valid rotation). */
int r2ik_ctl_ctor_theta_f64(r2ik_handle h, double preferred_theta, const double *current_joints_rows,
                            int32_t n_rows, const double *current_pose, double *out_theta, void *stream);

/* cudaStreamSynchronize(stream): lets a binding without a CUDA runtime of its own wait for a scalar call. */
int r2ik_stream_synchronize(void *stream);

/* ControlIK discrete mode for n poses M (n x 16).  prev_joints / current_joints: 7 doubles
 * each (device), broadcast: ControlIK.previous_sol[arm] and the per-call current_joints.
 * emergency: nullable, per-pose emergency bits. */
int r2ik_ctl_discrete_f64(r2ik_handle h, const R2ikCtlParams *par /* host */, const double *M, int64_t n,
                          const double *prev_joints, const double *current_joints, double *joints,
                          uint8_t *reachable, uint8_t *state, uint8_t *emergency, void *stream);

/* The same with the exhaustive form of the elbow search: every one of the nb_search_points samples is visited,
 * the samples of a pose strided over the lanes of its warp and reduced by a shuffle arg-min (lowest index wins
 * ties).  r2ik_ctl_discrete_f64 finds the same arg-min from the crossings of the two elbow tests without
 * visiting the samples; this entry is the cross-check of that search (identical outputs) at K times the cost. */
int r2ik_ctl_discrete_scan_f64(r2ik_handle h, const R2ikCtlParams *par /* host */, const double *M, int64_t n,
                               const double *prev_joints, const double *current_joints, double *joints,
                               uint8_t *reachable, uint8_t *state, uint8_t *emergency, void *stream);

/* r2ik_ctl_discrete_f64 for large batches, same results: the three sections of the call (is_reachable + preferred-theta
 * shortcut for every pose / elbow search for the poses the shortcut fails on / get_joints + safety chain for the poses
 * with a valid theta) run as separate kernels over compacted index lists, so no warp carries idle lanes through a
 * section its poses do not need.  workspace: r2ik_ctl_discrete_workspace_bytes(n) bytes of device memory, 16-byte
 * aligned, owned by the call until it has completed on `stream`; n < 2^31. */
int64_t r2ik_ctl_discrete_workspace_bytes(int64_t n);
int r2ik_ctl_discrete_compact_f64(r2ik_handle h, const R2ikCtlParams *par /* host */, const double *M, int64_t n,
                                  const double *prev_joints, const double *current_joints, double *joints,
                                  uint8_t *reachable, uint8_t *state, uint8_t *emergency, void *workspace,
                                  int64_t workspace_bytes, void *stream);

/* ControlIK continuous mode: T trajectories x W waypoints, M is T x W x 16.  current_joints
 * (T x 7) and current_pose (T x 16) feed the (re)initialisation; st: T states, in/out. */
int r2ik_ctl_continuous_f64(r2ik_handle h, const R2ikCtlParams *par /* host */, const double *M, int64_t T,
                            int32_t W, const double *current_joints, const double *current_pose,
                            R2ikTrajState *st, double *joints, uint8_t *reachable, uint8_t *state,
                            void *stream);

/* The same computation as r2ik_ctl_continuous_f64 (same flags / states, joints equal to rounding), cut at its data dependences:
 * the per-waypoint work (reachability, target theta, joints for a given theta, Orbita3D limit) runs with one thread per
 * waypoint, and only the rate-limited theta and the unwrap / continuity / emergency chain run as per-trajectory scans --
 * the latter on 16-bit winding codes that the joints kernel emits per waypoint (per-joint change of the winding number
 * against the previous waypoint's raw joints, the continuity verdict, or "irregular"): the scan walks 2 bytes per waypoint
 * and touches a joints row only where the waypoint is irregular, where it runs the reference's statements verbatim; rows
 * of joints that have wound past +-pi get their 2 pi k in a last parallel pass (csrc/r2ik_cont_codes.cuh).
 * workspace: T*W doubles (thetas) followed by T*W uint16 (codes), i.e. at least T*W + (T*W + 3) / 4 doubles of device
 * scratch, caller-owned.
 * test_force_serial_mod: 0 in production; m > 0 sends every m-th waypoint down the serial get_joints route (which no
 * physical pose takes) so that tests can hold that route to the ordinary result. */
int r2ik_ctl_continuous_phased_f64(r2ik_handle h, const R2ikCtlParams *par /* host */, const double *M, int64_t T,
                                   int32_t W, const double *current_joints, const double *current_pose,
                                   R2ikTrajState *st, double *joints, uint8_t *reachable, uint8_t *state,
                                   double *workspace, int32_t test_force_serial_mod, void *stream);

/* Workspace reachability map: counts[v] += #orientations o in [ori_begin, ori_end) with
 * is_reachable(voxel centre, orientations_euler[o]) true.  Voxel (ix,iy,iz) centre =
 * origin + (ix,iy,iz)*step, v = (ix*dims[1] + iy)*dims[2] + iz.  origin/step/dims: host.
 * counts must be zero-initialised by the caller (the kernel overwrites, it does not add). */
int r2ik_reach_map_u32(r2ik_handle h, const double *origin, const double *step, const int32_t *dims,
                       const double *orientations_euler /* device, n_ori x 3 */, int32_t ori_begin,
                       int32_t ori_end, uint32_t *counts, void *stream);

/* The same volume with every (voxel, orientation) pair decided by the all-FP64 flag solve.  r2ik_reach_map_u32 decides
 * a pair with an FP64 front end + FP32 linking test and hands the pairs within the FP32 error bands of a decision to
 * that solve, so the two entries return identical counts; this one is the cross-check (and ~2-3x slower). */
int r2ik_reach_map_f64_u32(r2ik_handle h, const double *origin, const double *step, const int32_t *dims,
                           const double *orientations_euler /* device, n_ori x 3 */, int32_t ori_begin,
                           int32_t ori_end, uint32_t *counts, void *stream);

/* The same counts as r2ik_reach_map_u32 for the voxels [voxel_begin, voxel_end) only (v = (ix*dims[1] + iy)*dims[2] + iz),
 * stored as uint16 into counts[v] (counts = base of the FULL volume).  row_mod > 1: of the rows (ix, iy, :) of that
 * range only those with row % row_mod == row_rem are computed (the range must then be row-aligned) -- the interleaved
 * sharding of the multi-GPU map, where rank r owns every world-th row and the all-reduce adds the disjoint pieces.
 * For the sharded map the volume is produced slab by slab so that the all-reduce of one slab overlaps the kernel of
 * the next, and 16-bit counts halve the bytes on the wire (two counts travel in one int32 lane; <= 65 535
 * orientations cannot carry). */
int r2ik_reach_map_range_u16(r2ik_handle h, const double *origin, const double *step, const int32_t *dims,
                             const double *orientations_euler /* device, n_ori x 3 */, int32_t ori_begin,
                             int32_t ori_end, int64_t voxel_begin, int64_t voxel_end, int32_t row_mod,
                             int32_t row_rem, uint16_t *counts, void *stream);

/* Forward kinematics: M[i] (row-major 4x4) = tip pose in the torso frame for joints[i] (7).
 * chain: host pointer.  device: CUDA ordinal to launch on. */
int r2ik_fk_f64(const R2ikFkChain *chain, int device, const double *joints, int64_t n, double *M, void *stream);

/* Strided copy (cudaMemcpy2DAsync, direction inferred from the pointers): `rows` rows of `width_bytes`
 * between buffers of the given pitches.  Plumbing for the waypoint-chunked host pipeline of the
 * continuous mode (a chunk of waypoints of every trajectory is a strided block of the (T, W, 16)
 * host array).  Host memory should be pinned for the copy to be asynchronous. */
int r2ik_copy2d_async(void *dst, size_t dst_pitch, const void *src, size_t src_pitch, size_t width_bytes,
                      size_t rows, void *stream);

/* ---- host pipelines -------------------------------------------------------------------------------------------
 * A batch in HOST memory, cut into chunks that flow H2D copy -> kernel -> D2H copy on three CUDA streams chained by
 * events (both PCIe directions and the kernel overlap).  The pipeline object owns its device staging buffers, streams
 * and events (created once for a chunk size and a number of in-flight slots); the calls enqueue and return, and
 * r2ik_pipeline_wait blocks until the results are in host memory.  All data pointers below are HOST pointers,
 * ideally pinned (pageable memory makes the copies synchronous).  Batched counterparts of
 * SymbolicIK.is_reachable + get_joints (symbolic_ik.py:121-282, 697-863) and of
 * ControlIK.symbolic_inverse_kinematics(name, M, "discrete") (control_ik.py:162-274, 409-462) for callers whose poses
 * live in host memory -- which is every caller of the reference. */
typedef struct r2ik_pipeline *r2ik_pipeline_t;
int r2ik_pipeline_create(r2ik_handle h, int device, int64_t chunk_poses, int32_t n_slots /* 2 .. 16 */, r2ik_pipeline_t *out);
int r2ik_pipeline_destroy(r2ik_pipeline_t p);
int r2ik_pipeline_wait(r2ik_pipeline_t p);
const char *r2ik_pipeline_last_error(void);

/* Outputs as r2ik_symik_solve_f64 (theta_interval[0], default previous_joints); any output except `state` may be NULL
 * and is then neither computed nor copied: poses n x 6 in + state + joints back is 48 + 57 bytes per pose. */
int r2ik_pipeline_symik_f64(r2ik_pipeline_t p, int pose_kind, const double *poses_host, int64_t n, uint8_t *reachable,
                            uint8_t *state, double *interval, double *joints, double *elbow);
/* FP32 fast path (r2ik_symik_solve_f32): float poses and results; `reachable` is required. */
int r2ik_pipeline_symik_f32(r2ik_pipeline_t p, int pose_kind, const float *poses_host, int64_t n, uint8_t *reachable,
                            uint8_t *state, float *interval, float *joints, float *elbow);
/* r2ik_ctl_discrete_f64 on host matrices M_host (n x 16); prev / current joints: 7 host doubles each. */
int r2ik_pipeline_ctl_discrete_f64(r2ik_pipeline_t p, const R2ikCtlParams *par, const double *M_host, int64_t n,
                                   const double *prev_joints_host, const double *current_joints_host, double *joints,
                                   uint8_t *reachable, uint8_t *state, uint8_t *emergency /* nullable */);

/* FP64 FMA peak probe used by bench.py for the compute roofline: runs `iters` dependent
 * DFMA chains (8 per thread) on a full grid and returns elapsed ms / flop count. */
int r2ik_dfma_probe(int device, int32_t iters, double *out_ms /* host */, double *out_flop /* host */,
                    void *stream);

/* The same with FFMA chains: FP32 FMA peak for the roofline of r2ik_symik_solve_f32. */
int r2ik_ffma_probe(int device, int32_t iters, double *out_ms /* host */, double *out_flop /* host */,
                    void *stream);

#ifdef __cplusplus
}
#endif
#endif /* R2IK_H */
