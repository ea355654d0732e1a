/* wbc.h — C ABI of the batched whole-body controller (libwbc_b200.so).
 *
 * Drop-in boundary for the per-control-step path of vincekurtz/quadruped_drake.
 * Every entry point replaces a block of pydrake calls made by the reference
 * controllers; the citation after each declaration is the reference code it
 * stands in for (paths relative to the reference tree).
 *
 * Conventions
 *   - plain C, no exceptions; every function returns an int status, 0 = WBC_OK;
 *     wbc_last_error() gives the text for the last non-zero return on a handle;
 *   - all arithmetic is FP64; arrays are instance-major (row i = instance i);
 *   - q  = [qw qx qy qz  px py pz  theta(12)]            (19)  Drake position order
 *     v  = [omega_W(3)  pdot_W(3)  thetadot(12)]         (18)  Drake velocity order
 *     joint/velocity order inside theta is given by wbc_model.v_index;
 *   - traj[54] follows lcm_types/trunk_state_t.lcm:10-35 field order:
 *       base p, pd, pdd, rpy, rpyd, rpydd (18),
 *       foot p   LF RF LH RH (12), foot pd (12), foot pdd (12);
 *     contact[4] = planned stance flags LF RF LH RH (trunk_state_t.lcm:38-41,
 *     planners/simple.py:67);
 *   - tau[12] is in actuator (URDF <transmission>) order, like the vector the
 *     reference writes to its `quad_torques` port (basic_controller.py:320);
 *   - metrics[4] = [V, err, res, Vdot] (basic_controller.py:271-283);
 *   - per-instance failures go to status[i] (bit mask below), never abort the batch
 *     (the reference asserts instead: inverse_dynamics_controller.py:224). An instance with ANY status bit set
 *     returns tau = 0 (and f = vd = lam = 0 where requested): an unfinished active-set iterate, a substituted
 *     orientation (bad quaternion, gimbal lock), a rank-deficient problem or a NaN / inf input never leaves the library as
 *     torques (WBC_CTRL_PD excepted: it has no status, and a NaN input gives a NaN torque, as np.clip does in the reference).
 *     metrics[1] (err) is still the tracking error of the state; callers must mask on status;
 *   - "device" entry points take device pointers and a cudaStream_t passed as void*;
 *     "_host" entry points take host pointers and do the copies themselves.
 *   - one handle per device; calls on one handle must be serialised by the caller.
 */
#ifndef WBC_B200_H
#define WBC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define WBC_NQ 19
#define WBC_NV 18
#define WBC_NU 12
#define WBC_NLEG 4
#define WBC_NBODY 13      /* floating base + 4 x (hip/abduct, thigh, shank) after welding */
#define WBC_NTRAJ 54
#define WBC_NMETRIC 4
#define WBC_NLAM 42       /* inequality multipliers: 16 friction rows + 2 controller rows + 24 torque-box rows */

/* return codes */
#define WBC_OK 0
#define WBC_ERR_ARG 1
#define WBC_ERR_CUDA 2
#define WBC_ERR_NOMEM 3

/* per-instance status bits */
#define WBC_ST_OK 0
#define WBC_ST_MAXITER 1       /* active-set iteration cap reached                       */
#define WBC_ST_INFEASIBLE 2    /* QP constraints inconsistent                            */
#define WBC_ST_RANKDEF 4       /* equality constraints rank deficient (e.g. singular leg)  */
                               /* a stance leg counts as singular when |det L_k| <= 2e-3 |c0||c1||c2|, L_k its 3x3 foot
                                * Jacobian block with columns c_j: a test on the sine-volume, independent of the leg's size */
#define WBC_ST_GIMBAL 8        /* |cos(pitch)| < 1e-6: rpy rates undefined (SURVEY A.7)   */
#define WBC_ST_NOTPD 16        /* reduced Hessian not positive definite                   */
#define WBC_ST_BADQUAT 32      /* zero / non-finite quaternion                            */
#define WBC_ST_UNSUPPORTED 64  /* PC controller with no stance foot (the reference raises too) */
#define WBC_ST_DIVERGED 128    /* rollout only: non-finite / runaway velocity, instance frozen   */
#define WBC_ST_NONFINITE 256   /* a NaN / inf among the q, v, traj values of the instance, or a non-finite solution */
#define WBC_ST_BADVARIANT 512  /* perturbed plant only: variant index out of range; the robot is frozen, zero ground forces */
#define WBC_ST_BADTERRAIN 1024 /* terrain plant only: terrain index out of range; the robot is frozen, zero ground forces */
#define WBC_ST_BADPARAMS 2048  /* wbc_step_params only: parameter-set index out of range; zero outputs                  */
#define WBC_ST_BADLOOP 4096    /* wbc_rollout_loop only: bad loop profile; observed without noise, zero applied torque  */
#define WBC_ST_BADMOTOR 8192   /* wbc_rollout_motor / wbc_motor_apply only: motor record index out of range; zero torque */
#define WBC_ST_BADESTIM 16384  /* wbc_rollout_estimator / wbc_estimator_step only: bad record index or failed filter step   */
#define WBC_ST_BADCONTACT 32768 /* wbc_rollout_contact / wbc_contact_step only: bad record index or non-finite force estimate */

/* controller kinds: reference controllers/__init__.py:1-5 */
#define WBC_CTRL_ID 0          /* controllers/inverse_dynamics_controller.py */
#define WBC_CTRL_CLF 1         /* controllers/clf_controller.py              */
#define WBC_CTRL_PC 2          /* controllers/pc_controller.py               */
#define WBC_CTRL_MPTC 3        /* controllers/mptc_controller.py (PC without the passivity rows) */
#define WBC_CTRL_PD 4          /* BasicController.ControlLaw, basic_controller.py:322-352 (joint PD) */

/* Flattened robot: what Drake's Parser + MultibodyPlant::Finalize hold after
 * simulate.py:37-64. Body 0 = floating base, body 1+3*leg+j = link j of leg
 * (legs in foot order LF RF LH RH, basic_controller.py:67-70). Welded links are
 * already merged into their parent. Joint k = 3*leg+j connects body k+1 to its
 * parent (base for j = 0, body k otherwise); all joint frames are unrotated
 * (every moving-joint rpy is 0 in both reference URDFs). */
typedef struct wbc_model {
  double mass[WBC_NBODY];
  double com[WBC_NBODY][3];          /* CoM in the body frame                                  */
  double inertia_com[WBC_NBODY][6];  /* about the CoM, body axes: xx yy zz xy xz yz            */
  double joint_xyz[WBC_NU][3];       /* joint origin in the parent body frame                  */
  double joint_axis[WBC_NU][3];      /* unit axis (same in parent and child frame)             */
  double foot_xyz[WBC_NLEG][3];      /* foot frame origin in the shank frame                   */
  double effort[WBC_NU];             /* URDF effort limit of joint k                           */
  double gravity[3];                 /* world gravity vector, (0,0,-9.81)                      */
  int32_t v_index[WBC_NU];           /* index of joint k in Drake's v (6..17); q index = +1    */
  int32_t act_index[WBC_NU];         /* actuator (output tau) index of joint k                 */
} wbc_model;

/* Gains and weights: the literals inside each reference ControlLaw (SURVEY Appendix G). */
typedef struct wbc_params {
  /* ID  (inverse_dynamics_controller.py:116-128) */
  double id_kp_body_p, id_kd_body_p, id_kp_body_rpy, id_kd_body_rpy;
  double id_kp_foot, id_kd_foot, id_w_body, id_w_foot;
  /* CLF (clf_controller.py:65-78) */
  double clf_q_body_p, clf_q_body_pd, clf_q_body_rpy, clf_q_body_rpyd;
  double clf_q_foot_p, clf_q_foot_pd, clf_r, clf_w_delta;
  /* PC  (pc_controller.py:63-76) */
  double pc_kp_body_p, pc_kd_body_p, pc_kp_body_rpy, pc_kd_body_rpy;
  double pc_kp_foot, pc_kd_foot, pc_w_body, pc_w_foot;
  /* shared (inverse_dynamics_controller.py:19,94) */
  double mu;                 /* friction coefficient, 0.7                      */
  double contact_damping;    /* Kd of the no-slip constraint, 100              */
  /* declared tie-break (SURVEY Appendix E.2): + reg_f/2 |f|^2 + reg_tau/2 |tau|^2
   * + reg_vd/2 |vd|^2 added to the reference cost so the optimum is unique.     */
  double reg_f, reg_tau, reg_vd;
  int32_t torque_limits;     /* 0 = reference QP; 1 = add |tau_k| <= effort_k  */
  int32_t max_iter;          /* active-set iteration cap                       */
  /* Basic PD law (basic_controller.py:331-350): tau = -kp (theta - theta_nom) - kd thetadot, clipped */
  double pd_kp, pd_kd, pd_clip;
  double pd_q_nom[WBC_NU];   /* nominal joint angles in the caller's joint order (q[7:19])       */
} wbc_params;

typedef struct wbc_handle wbc_handle;

/* Optional per-step buffers beyond tau/metrics/status; any pointer may be NULL. */
typedef struct wbc_io {
  const double* q;        /* [N][19] */
  const double* v;        /* [N][18] */
  const double* traj;     /* [N][54] */
  const uint8_t* contact; /* [N][4]  */
  double* tau;            /* [N][12] */
  double* metrics;        /* [N][4]  */
  int32_t* status;        /* [N]     */
  double* vd;             /* [N][18] QP accelerations, Drake velocity order (optional)  */
  double* f;              /* [N][12] contact forces LF RF LH RH, 0 for swing (optional) */
  double* qp_info;        /* [N][4]  objective, max primal violation, delta, #iters (optional) */
  double* lam;            /* [N][42] multipliers (>= 0) of the inequality rows at the returned optimum (optional):
                           *   [4 foot + t]  friction pyramid of foot LF RF LH RH, rows t = +x, -x, +y, -y
                           *                 (inverse_dynamics_controller.py:66-86, A_i row order)
                           *   [16], [17]    controller rows: CLF Vdot row (clf_controller.py:27-45) / PC passivity row
                           *                 (pc_controller.py:14-40, delta eliminated); [17] unused
                           *   [18 + a], [30 + a]   torque box  +tau_a <= effort_a,  -tau_a <= effort_a  (actuator order a)
                           * with these, x = [vd; tau; f] satisfies the KKT conditions of the reference QP (+ tie-break) */
} wbc_io;

/* Fill *p with the reference's constants (SURVEY Appendix G). */
int wbc_default_params(wbc_params* p);

/* BasicController.__init__ (basic_controller.py:21-77): create the plant context
 * equivalent — uploads the model tables and gains to `device`. */
int wbc_create(const wbc_model* model, const wbc_params* params, int device, wbc_handle** out);
int wbc_destroy(wbc_handle* h);
const char* wbc_last_error(const wbc_handle* h);

/* BasicController.CalcDynamics (basic_controller.py:101-115),
 * CalcFramePositionQuantities x4 (:173-196) on device buffers. Outputs (any may be NULL):
 *   M [N][18][18], Cv [N][18], taug [N][18] (= -CalcGravityGeneralizedForces, :112),
 *   Jfeet [N][4][3][18], Jdv [N][4][3], pfeet [N][4][3]; all in Drake velocity order. */
int wbc_dynamics(wbc_handle* h, int64_t n, const double* q, const double* v,
                 double* M, double* Cv, double* taug, double* Jfeet, double* Jdv,
                 double* pfeet, void* stream);

/* BasicController.CalcCoriolisMatrix (basic_controller.py:117-132) and
 * CalcFrameJacobianDot x4 (:198-220): C [N][18][18] with C v = Cv, Jd [N][4][3][18]. */
int wbc_coriolis(wbc_handle* h, int64_t n, const double* q, const double* v,
                 double* C, double* Jd, void* stream);

int wbc_coriolis_host(wbc_handle* h, int64_t n, const double* q, const double* v, double* C, double* Jd);

/* One control step for n instances: DoSetControlTorques -> ControlLaw
 * (basic_controller.py:286-320; inverse_dynamics_controller.py:103-234;
 * clf_controller.py:48-234; pc_controller.py:43-255). Device pointers (or page-locked host memory mapped into the
 * device address space). The step uses per-handle scratch (4.5 KB per instance, at most 262144 instances at a time), so steps
 * of one handle are serialised on the device: a call on a different stream than the previous call of the handle first makes
 * its stream wait for the work submitted to the previous one (an event dependency, no host synchronisation). Host threads must
 * still serialise their calls on one handle; different handles are independent. Batches of 4096 - 65536 instances are issued as
 * two to four chunks, all but the first on library-owned streams that fork from and join `stream` through events: to the caller
 * the step remains one stream-ordered operation on `stream` (not inside a stream capture, where it stays a single chain). */
int wbc_step(wbc_handle* h, int kind, int64_t n, const wbc_io* io, void* stream);
int wbc_step_id(wbc_handle* h, int64_t n, const double* q, const double* v, const double* traj,
                const uint8_t* contact, double* tau, double* metrics, int32_t* status, void* stream);
int wbc_step_clf(wbc_handle* h, int64_t n, const double* q, const double* v, const double* traj,
                 const uint8_t* contact, double* tau, double* metrics, int32_t* status, void* stream);
int wbc_step_pc(wbc_handle* h, int64_t n, const double* q, const double* v, const double* traj,
                const uint8_t* contact, double* tau, double* metrics, int32_t* status, void* stream);
int wbc_step_mptc(wbc_handle* h, int64_t n, const double* q, const double* v, const double* traj,
                  const uint8_t* contact, double* tau, double* metrics, int32_t* status, void* stream);
/* BasicController.ControlLaw (basic_controller.py:322-352); traj / contact are ignored and may be NULL. */
int wbc_step_pd(wbc_handle* h, int64_t n, const double* q, const double* v, double* tau, void* stream);

/* Same step with HOST buffers (what the Python LeafSystem shim calls); returns after tau / metrics / status (and any
 * optional outputs that are non-NULL) are in the caller's buffers. Page-locked buffers (wbc_host_alloc /
 * cudaHostRegister): the kernels write the outputs straight into them; the inputs are read over the host link by the kernels
 * (zero-copy) below 24576 instances (131072 for PC / MPTC) and go through the copy engine into device staging in chunks above.
 * Pageable buffers go through a chunked two-stream copy / compute pipeline in both directions. */
int wbc_step_host(wbc_handle* h, int kind, int64_t n, const wbc_io* host_io);

/* All GPUs of the box from one call (north star: "instances shard trivially across the 8 GPUs of one box, with no NCCL
 * beyond an optional host gather"; SURVEY 8e). wbc_multi_create makes one handle per listed device (devices == NULL: 0 ..
 * n_devices-1; a device may be listed more than once). wbc_multi_step_host splits [0, n) into contiguous shards whose sizes
 * differ by at most one, runs every shard on its device side by side (one host thread, asynchronous enqueue on all devices,
 * then one wait per device) and returns when all outputs are in the caller's host arrays - which is the host gather. Same
 * buffer rules as wbc_step_host; page-locked buffers (wbc_host_alloc) are mapped into every device. */
typedef struct wbc_multi wbc_multi;
int wbc_multi_create(const wbc_model* model, const wbc_params* params, int n_devices, const int* devices, wbc_multi** out);
int wbc_multi_destroy(wbc_multi* m);
const char* wbc_multi_last_error(const wbc_multi* m);
int wbc_multi_device_count(const wbc_multi* m);
int64_t wbc_multi_launch_count(const wbc_multi* m);
int wbc_multi_step_host(wbc_multi* m, int kind, int64_t n, const wbc_io* host_io);

/* Host-buffer version of wbc_dynamics (allocates device scratch per call; a test/debug entry). */
int wbc_dynamics_host(wbc_handle* h, int64_t n, const double* q, const double* v,
                      double* M, double* Cv, double* taug, double* Jfeet, double* Jdv, double* pfeet);

/* Pinned (page-locked) host memory for wbc_step_host buffers. */
void* wbc_host_alloc(size_t bytes);
void wbc_host_free(void* p);

/* Device-side timing helper for benchmarks: runs `reps` back-to-back wbc_step
 * launches on `stream` and returns the mean device time per launch (CUDA events
 * recorded on that same stream). */
int wbc_time_step(wbc_handle* h, int kind, int64_t n, const wbc_io* io, int reps, void* stream,
                  double* ms_per_launch);

/* Per-kernel share of a control step. A step is two stream-ordered kernels: the reduce kernel (state -> dynamics ->
 * reduced QP, one hand-over record per instance in library-owned device scratch) and the solve kernel (active-set QP ->
 * tau / metrics / status). Events are recorded before, between and after them; means over `reps` steps. n <= 262144. */
int wbc_profile_step(wbc_handle* h, int kind, int64_t n, const wbc_io* io, int reps, void* stream,
                     double* ms_reduce, double* ms_solve);

/* Measured-peak helper: FP64 FMA throughput of this device in TFLOP/s (a register
 * resident DFMA loop over all SMs), used as the FP64 roofline denominator. */
int wbc_measure_fp64_peak(int device, double* tflops);

/* ---- LCM wire codecs (SURVEY 8 f3): the byte formats either side of the control step. Messages are packed back
 * to back, `msgs` must be 16-byte aligned; any optional pointer may be NULL. Per-message problems go to status[i]. */
#define WBC_LCM_TRUNK_STATE_BYTES 549   /* lcm_types/trunk_state_t.lcm:1-50: 8 fingerprint + 8 + 1 + 18*24 + 4 + 4*24 */
#define WBC_LCM_ROBOT_STATE_BYTES 204   /* lcm_types/robot_state_control_lcmt.lcm:1-7: 8 fingerprint + 4*(19+18+12)   */
#define WBC_WIRE_BADFINGERPRINT 1       /* the generated decoders raise ValueError("Decode error")                    */
#define WBC_WIRE_OVERFLOW 2             /* finite double beyond float32 range: struct.pack('>f') raises OverflowError */

/* trunk_state_t.decode (lcm_types/trunklcm/trunk_state_t.py:79-120) + the field copy of planners/towr.py:112-145:
 * n messages -> traj [N][54], contact [N][4] (wbc.h layout), optional timestamp [N], finished [N], planned forces
 * f_plan [N][12] (LF RF LH RH, unused by every controller), status [N]. Device pointers. */
int wbc_lcm_decode_trunk_state(wbc_handle* h, int64_t n, const uint8_t* msgs, double* timestamp, uint8_t* finished,
                               double* traj, uint8_t* contact, double* f_plan, int32_t* status, void* stream);
/* trunk_state_t.encode (trunk_state_t.py:54-77), what towr/trunk_mpc.cpp:19-68 publishes per sample. */
int wbc_lcm_encode_trunk_state(wbc_handle* h, int64_t n, const double* timestamp, const uint8_t* finished,
                               const double* traj, const uint8_t* contact, const double* f_plan, uint8_t* msgs, void* stream);
/* robot_state_control_lcmt.decode (lcm_types/cheetahlcm/robot_state_control_lcmt.py:35-47) as used by
 * BasicController.lcm_callback (basic_controller.py:79-87): float32 wire values widened to q [N][19], v [N][18],
 * optional tau [N][12]. */
int wbc_lcm_decode_robot_state(wbc_handle* h, int64_t n, const uint8_t* msgs, double* q, double* v, double* tau,
                               int32_t* status, void* stream);
/* robot_state_control_lcmt.encode (:24-33). q / v may be NULL (zeros: the controller publishes a fresh message that
 * carries only the torques, basic_controller.py:309-314). tau_in_actuator_order != 0: `tau` is the step output of
 * this library (actuator order) and is sent in velocity order like the reference's (S.T @ u)[-12:]; 0: copied as is. */
int wbc_lcm_encode_robot_state(wbc_handle* h, int64_t n, const double* q, const double* v, const double* tau,
                               int tau_in_actuator_order, uint8_t* msgs, int32_t* status, void* stream);
/* The same four with HOST buffers (copies inside, synchronous). */
int wbc_lcm_decode_trunk_state_host(wbc_handle* h, int64_t n, const uint8_t* msgs, double* timestamp, uint8_t* finished,
                                    double* traj, uint8_t* contact, double* f_plan, int32_t* status);
int wbc_lcm_encode_trunk_state_host(wbc_handle* h, int64_t n, const double* timestamp, const uint8_t* finished,
                                    const double* traj, const uint8_t* contact, const double* f_plan, uint8_t* msgs);
int wbc_lcm_decode_robot_state_host(wbc_handle* h, int64_t n, const uint8_t* msgs, double* q, double* v, double* tau,
                                    int32_t* status);
int wbc_lcm_encode_robot_state_host(wbc_handle* h, int64_t n, const double* q, const double* v, const double* tau,
                                    int tau_in_actuator_order, uint8_t* msgs, int32_t* status);

/* ---- Trunk-trajectory sampler (SURVEY 8 f1): TOWR spline solution -> controller input on the device.
 * A plan is what towr's SplineHolder holds after the solve (towr/trunk_mpc.cpp:151-156): cubic Hermite node splines for
 * base position, base Euler angles (rpy), 4 foot positions, 4 foot forces, and the per-foot phase durations. */
#define WBC_TRAJ_CLAMPED 1   /* t outside [0, total]: evaluated at the nearest end (the reference asserts / runs off);
                              * a NaN t is flagged and taken as t = 0, with and without a grid (n_grid > 0: standing
                              * while 0 < wait_time, else the stored sample nearest to 0)                              */
#define WBC_TRAJ_BADPLAN 2   /* plan index out of range: plan 0 used                                                  */

typedef struct wbc_spline_desc {
  int32_t n_poly;            /* number of cubic polynomials                                                        */
  const double* durations;   /* [n_poly]           polynomial durations (Spline::GetPolyDurations)                 */
  const double* nodes;       /* [n_poly + 1][6]    node position (3) and velocity (3), towr Node                   */
} wbc_spline_desc;

typedef struct wbc_plan_desc {
  wbc_spline_desc base_linear, base_angular;   /* SplineHolder::base_linear_, base_angular_                        */
  wbc_spline_desc ee_motion[WBC_NLEG];         /* SplineHolder::ee_motion_ (LF RF LH RH)                           */
  wbc_spline_desc ee_force[WBC_NLEG];          /* SplineHolder::ee_force_                                          */
  int32_t n_phase[WBC_NLEG];                   /* PhaseDurations::GetPhaseDurations().size()                       */
  const double* phase_durations[WBC_NLEG];     /* [n_phase] alternating contact / swing phases of the foot         */
  uint8_t contact_at_start[WBC_NLEG];          /* GaitGenerator::IsInContactAtStart                                */
  /* Planner semantics of planners/towr.py:92-148 (optional, n_grid = 0 -> evaluate the splines at t itself):       */
  int32_t n_grid;                              /* number of stored samples (5001 for trunk_mpc's 1 kHz x 5 s)      */
  const double* grid_timestamps;               /* [n_grid] increasing timestamps of the stored samples             */
  double wait_time;                            /* stand this long before the motion starts (planners/towr.py:35)   */
  double standing[WBC_NTRAJ];                  /* SimpleStanding reference (planners/simple.py:39-85) while waiting */
} wbc_plan_desc;

typedef struct wbc_plan wbc_plan;

/* Upload n_plans plans (host descriptors) and build their device tables; Hermite coefficients
 * (towr/src/polynomial.cc:98-104) are computed on the device. */
int wbc_plan_create(wbc_handle* h, int32_t n_plans, const wbc_plan_desc* plans, wbc_plan** out);
int wbc_plan_destroy(wbc_plan* plan);
/* publish_trunk_state (towr/trunk_mpc.cpp:19-68) + TowrTrunkPlanner.SetTrunkOutputs (planners/towr.py:92-148) for n
 * (plan, time) pairs: traj [N][54], contact [N][4]; optional plan_index [N] (NULL = plan 0), f_plan [N][12],
 * t_eval [N] (the spline time actually evaluated, -1 while standing), status [N]. Device pointers. */
int wbc_sample_trajectory(wbc_handle* h, const wbc_plan* plan, int64_t n, const int32_t* plan_index, const double* t,
                          double* traj, uint8_t* contact, double* f_plan, double* t_eval, int32_t* status, void* stream);
int wbc_sample_trajectory_host(wbc_handle* h, const wbc_plan* plan, int64_t n, const int32_t* plan_index, const double* t,
                               double* traj, uint8_t* contact, double* f_plan, double* t_eval, int32_t* status);

/* Control step with the trunk targets taken from a device-resident plan (TowrTrunkPlanner.SetTrunkOutputs feeding
 * DoSetControlTorques, planners/towr.py:92-148 -> basic_controller.py:286-320) on HOST state buffers: the host sends q, v
 * and the plan time t [N] (+ optional plan_index [N]) - 308 B per instance instead of 736 B - the trajectory rows are sampled on
 * the device into library scratch. Outputs as wbc_step_host. Page-locked buffers are read / written by the kernels directly. */
int wbc_step_plan_host(wbc_handle* h, int kind, const wbc_plan* plan, int64_t n, const double* q, const double* v,
                       const double* t, const int32_t* plan_index, double* tau, double* metrics, int32_t* status);

/* ---- Closed-loop batched rollout (SURVEY 8 f2): the caller of the control step, simulate.py:160-182.
 * wbc_integrate: semi-implicit Euler step of n states with the accelerations vd returned by wbc_step
 * (v += dt vd; q += dt N(q) v, quaternion renormalised); t [N] (optional) is advanced by dt. Device pointers. */
int wbc_integrate(wbc_handle* h, int64_t n, double dt, double* q, double* v, const double* vd, double* t, void* stream);

typedef struct wbc_rollout_io {
  double* q;              /* [N][19] in: initial state (simulate.py:171-179), out: final state                  */
  double* v;              /* [N][18]                                                                             */
  double* t;              /* [N]     in: start time of each instance, out: end time                              */
  const int32_t* plan_index; /* [N] or NULL (plan 0)                                                             */
  double* tau;            /* [N][12] torques of the last step                                                    */
  double* metrics;        /* [N][4]  metrics of the last step                                                    */
  int32_t* status_or;     /* [N]     OR of the per-step status words (optional)                                  */
  double* err_max;        /* [N]     max over the steps of the tracking-error metric (optional)                  */
  double* metrics_log;    /* [n_steps][N][4] every step's output_metrics, what simulate.py:142 logs (optional)   */
} wbc_rollout_io;

/* One time step of n simulated robots on flat ground (the plant half of simulate.py:36-57,160-182): forward dynamics from
 * the APPLIED torques, velocity-level ground contact at the four feet (no penetration, Coulomb pyramid with `mu`; projected
 * Gauss-Seidel, `iters` sweeps from zero; `erp` = fraction of a penetration pushed out per step), semi-implicit Euler. The
 * scheme is defined in csrc/wbc_plant.cuh - Drake's own contact solver is third party and not restatable - and pinned by
 * invariants and by oracle/rollout.py. tau [N][12] in actuator order; q, v updated in place; t (optional) advanced by dt;
 * ctrl_status (optional): robots with a non-zero controller status are frozen; status_or (optional) accumulates;
 * f_contact (optional) [N][12]: ground forces on LF RF LH RH in world axes (impulse / dt). Device pointers. */
typedef struct wbc_plant_opts {
  double mu;        /* ground friction, 1.0 (simulate.py:44-46: static = dynamic = 1.0) */
  double erp;       /* penetration correction per step, 0.2                            */
  int32_t iters;    /* Gauss-Seidel sweeps, 30                                         */
  int32_t reserved;
} wbc_plant_opts;
int wbc_default_plant_opts(wbc_plant_opts* o);
int wbc_plant_step(wbc_handle* h, int64_t n, double dt, const wbc_plant_opts* opts, double* q, double* v, const double* tau,
                   double* t, const int32_t* ctrl_status, int32_t* status_or, double* f_contact, void* stream);
int wbc_plant_step_host(wbc_handle* h, int64_t n, double dt, const wbc_plant_opts* opts, double* q, double* v, const double* tau,
                        double* t, const int32_t* ctrl_status, int32_t* status_or, double* f_contact);

/* n_steps control steps of n robots, entirely on the device: sample the plan at t (wbc_sample_trajectory), run the
 * controller `kind` (wbc_step), integrate (wbc_integrate). No host synchronisation inside; with use_graph != 0 the
 * per-step launches are captured once into a CUDA graph and replayed. Device pointers. */
int wbc_rollout(wbc_handle* h, int kind, const wbc_plan* plan, int64_t n, int32_t n_steps, double dt,
                const wbc_rollout_io* io, int use_graph, void* stream);
int wbc_rollout_host(wbc_handle* h, int kind, const wbc_plan* plan, int64_t n, int32_t n_steps, double dt,
                     const wbc_rollout_io* host_io, int use_graph);
/* The same loop with a choice of plant: plant == 0 integrates the QP's own contact-consistent accelerations ("planned contacts
 * hold", wbc_rollout); plant == 1 applies the controller's TORQUES to the simulated robot on the ground (wbc_plant_step), so a
 * controller can fail physically: slip, land, fall. f_contact (optional, device) receives the last step's ground forces. */
typedef struct wbc_rollout_opts {
  int32_t use_graph;
  int32_t plant;
  wbc_plant_opts plant_opts;
  double* f_contact;      /* [N][12] or NULL */
} wbc_rollout_opts;
int wbc_rollout_ex(wbc_handle* h, int kind, const wbc_plan* plan, int64_t n, int32_t n_steps, double dt,
                   const wbc_rollout_io* io, const wbc_rollout_opts* opts, void* stream);
int wbc_rollout_ex_host(wbc_handle* h, int kind, const wbc_plan* plan, int64_t n, int32_t n_steps, double dt,
                        const wbc_rollout_io* host_io, const wbc_rollout_opts* opts);

/* ---- Perturbed robots for the ground plant: the plant simulates a different robot than the controller believes in, on its
 * own ground friction, and may push it. The controller keeps the handle's model and its own friction pyramid (params.mu).
 *
 * wbc_plant_set_create uploads n_variants robots to the handle's device: models[k] is what the plant simulates for variant k
 * (a payload merged into the base, scaled link masses, another inertia ...); mu[k] >= 0 is that variant's ground friction
 * (mu == NULL: the call's wbc_plant_opts.mu for every variant). Every model must have the handle's v_index and act_index (q, v
 * and tau layouts are shared with the controller), masses > 0, positive definite inertia_com and finite values. Like a
 * plan, a set keeps its device number, not its handle: it may be destroyed after the handle. */
typedef struct wbc_plant_set wbc_plant_set;
int wbc_plant_set_create(wbc_handle* h, int32_t n_variants, const wbc_model* models, const double* mu, wbc_plant_set** out);
int wbc_plant_set_destroy(wbc_plant_set* s);

/* Per-robot perturbation of a plant step or rollout (device pointers for the device entries, host pointers for _host). */
typedef struct wbc_plant_perturb {
  const wbc_plant_set* set;  /* NULL: every robot is the handle's model with opts.mu (one variant, index 0)              */
  const int32_t* variant;    /* [N] variant of each robot, NULL = variant 0. An index < 0 or >= n_variants sets
                              * WBC_ST_BADVARIANT in status_or: that robot keeps its state and gets zero f_contact      */
  const double* push;        /* [N][8] or NULL: force (world, N) [0:3], point of application in base coordinates relative
                              * to the base origin [3:6], t_on [6], t_off [7]; applied during every step whose start time t
                              * satisfies t_on <= t < t_off (t is then required)                                         */
} wbc_plant_perturb;

/* wbc_plant_step for perturbed robots: the step of robot i simulates its variant's model with its variant's friction and adds
 * its push, if active, to the applied forces. perturb == NULL is the nominal model with opts.mu and no push. */
int wbc_plant_step_perturbed(wbc_handle* h, int64_t n, double dt, const wbc_plant_opts* opts, const wbc_plant_perturb* perturb,
                             double* q, double* v, const double* tau, double* t, const int32_t* ctrl_status,
                             int32_t* status_or, double* f_contact, void* stream);
int wbc_plant_step_perturbed_host(wbc_handle* h, int64_t n, double dt, const wbc_plant_opts* opts, const wbc_plant_perturb* perturb,
                                  double* q, double* v, const double* tau, double* t, const int32_t* ctrl_status,
                                  int32_t* status_or, double* f_contact);
/* wbc_rollout_ex with the ground plant (opts->plant must be 1) stepping perturbed robots: the same launches per step, the same
 * graph capture and bookkeeping; only the plant kernel differs. */
int wbc_rollout_perturbed(wbc_handle* h, int kind, const wbc_plan* plan, int64_t n, int32_t n_steps, double dt,
                          const wbc_rollout_io* io, const wbc_rollout_opts* opts, const wbc_plant_perturb* perturb, void* stream);
int wbc_rollout_perturbed_host(wbc_handle* h, int kind, const wbc_plan* plan, int64_t n, int32_t n_steps, double dt,
                               const wbc_rollout_io* host_io, const wbc_rollout_opts* opts, const wbc_plant_perturb* perturb);

/* ---- Uneven ground for the ground plant: each robot stands on its own terrain. The controller is unchanged and sees none of
 * it (its friction pyramid stays about world z, its feet come from the flat-ground plan).
 *
 * A terrain is a plane plus an optional height field,  h(x, y) = z0 + sx x + sy y + H(x, y),  where H is the bilinear
 * interpolant of the row-major grid heights[ny][nx] with origin (x0, y0) and spacing (dx, dy); nx = ny = 0 is no grid (H = 0).
 * Outside the grid the grid coordinates are clamped to its edge (the clamped direction has zero gradient); the cell of a point
 * on the far edge is the last one. H is continuous, so a vertical step in the heights is a ramp one cell wide. Each foot
 * contacts the terrain at its position at the start of the step, along the local normal n = (-h_x, -h_y, 1) / |.|, with the
 * friction pyramid in the frame t1 = normalize(e_x - n_x n), t2 = n x t1, n; its gap is (p_z - h(p_x, p_y)) n_z. f_contact
 * stays in world axes. Only the four foot points touch the ground. On flat terrain (all zero, no grid) the step gives the
 * bits of wbc_plant_step_perturbed.
 *
 * wbc_terrain_set_create uploads n_terrains terrains to the handle's device (heights are copied). Every value must be finite;
 * nx and ny are both 0 or both >= 2; with a grid, dx, dy > 0 and heights != NULL. Like a plan, a set keeps its device number,
 * not its handle: it may be destroyed after the handle. */
typedef struct wbc_terrain_desc {
  double z0, sx, sy;       /* plane z0 + sx x + sy y                                    */
  int32_t nx, ny;          /* grid size, 0 x 0: no grid                                 */
  double x0, y0, dx, dy;   /* world position of heights[0][0], spacing along x and y    */
  const double* heights;   /* [ny][nx] row-major (host), NULL without a grid            */
} wbc_terrain_desc;
typedef struct wbc_terrain_set wbc_terrain_set;
int wbc_terrain_set_create(wbc_handle* h, int32_t n_terrains, const wbc_terrain_desc* terrains, wbc_terrain_set** out);
int wbc_terrain_set_destroy(wbc_terrain_set* s);

/* Per-robot terrain of a plant step or rollout (device pointer for the device entries, host pointer for _host). */
typedef struct wbc_plant_terrain {
  const wbc_terrain_set* set;  /* NULL: flat ground z = 0 for every robot (one terrain, index 0)                        */
  const int32_t* index;        /* [N] terrain of each robot, NULL = terrain 0. An index < 0 or >= n_terrains sets
                                * WBC_ST_BADTERRAIN in status_or: that robot keeps its state and gets zero f_contact  */
} wbc_plant_terrain;

/* wbc_plant_step_perturbed on each robot's terrain. perturb == NULL is the nominal model with opts.mu and no push;
 * terrain == NULL is flat ground. */
int wbc_plant_step_terrain(wbc_handle* h, int64_t n, double dt, const wbc_plant_opts* opts, const wbc_plant_perturb* perturb,
                           const wbc_plant_terrain* terrain, double* q, double* v, const double* tau, double* t,
                           const int32_t* ctrl_status, int32_t* status_or, double* f_contact, void* stream);
int wbc_plant_step_terrain_host(wbc_handle* h, int64_t n, double dt, const wbc_plant_opts* opts, const wbc_plant_perturb* perturb,
                                const wbc_plant_terrain* terrain, double* q, double* v, const double* tau, double* t,
                                const int32_t* ctrl_status, int32_t* status_or, double* f_contact);
/* wbc_rollout_perturbed on each robot's terrain (opts->plant must be 1): the same launches per step, the same graph capture and
 * bookkeeping; only the plant kernel differs. */
int wbc_rollout_terrain(wbc_handle* h, int kind, const wbc_plan* plan, int64_t n, int32_t n_steps, double dt,
                        const wbc_rollout_io* io, const wbc_rollout_opts* opts, const wbc_plant_perturb* perturb,
                        const wbc_plant_terrain* terrain, void* stream);
int wbc_rollout_terrain_host(wbc_handle* h, int kind, const wbc_plan* plan, int64_t n, int32_t n_steps, double dt,
                             const wbc_rollout_io* host_io, const wbc_rollout_opts* opts, const wbc_plant_perturb* perturb,
                             const wbc_plant_terrain* terrain);

/* ---- Per-robot controller parameters: one batched step or rollout runs many gain and weight sets. The controller keeps the
 * handle's model; only the wbc_params differ from robot to robot.
 *
 * wbc_param_set_create uploads n_sets >= 1 parameter sets to the handle's device, each with the constants derived from it
 * (the CLF Riccati solution). Each set must pass the checks of wbc_create (reg_vd == 0, reg_f > 0) and have finite values,
 * max_iter >= 1, torque_limits 0 or 1, mu >= 0, clf_r > 0 and non-negative CLF weights (clf_q_*, clf_w_delta). Like a plan, a
 * set keeps its device number, not its handle: it may be destroyed after the handle. */
typedef struct wbc_param_set wbc_param_set;
int wbc_param_set_create(wbc_handle* h, int32_t n_sets, const wbc_params* params, wbc_param_set** out);
int wbc_param_set_destroy(wbc_param_set* s);

/* Per-robot parameters of a step or rollout (device pointer for the device entries, host pointer for _host). */
typedef struct wbc_ctrl_params {
  const wbc_param_set* set;  /* NULL: the handle's params for every robot (one set, index 0)                            */
  const int32_t* index;      /* [N] set of each robot, NULL = set 0. An index < 0 or >= n_sets sets WBC_ST_BADPARAMS:
                              * that robot returns tau = 0 (and f = vd = lam = 0), its neighbours are unaffected        */
} wbc_ctrl_params;

/* wbc_step / wbc_step_host with robot i controlled by the set index[i]: the same buffer rules, chunking and stream semantics,
 * the same kernels' arithmetic and the same launch count. With a set whose every record equals the handle's params it gives
 * the bits of wbc_step. WBC_CTRL_PD reads pd_kp, pd_kd, pd_clip and pd_q_nom per robot; it writes status[i] (WBC_ST_BADPARAMS
 * or 0) when io->status is non-NULL. p == NULL is the handle's params. */
int wbc_step_params(wbc_handle* h, int kind, int64_t n, const wbc_io* io, const wbc_ctrl_params* p, void* stream);
int wbc_step_params_host(wbc_handle* h, int kind, int64_t n, const wbc_io* host_io, const wbc_ctrl_params* p);

/* The rollout loop of wbc_rollout_ex with per-robot controller parameters (ctrl == NULL: the handle's). With the ground plant
 * (opts->plant = 1) the plant step is the terrain kernel when terrain != NULL, else the variant kernel when perturb != NULL,
 * else the plain one; perturb or terrain without the ground plant is an argument error. The same launches per step, graph
 * capture and bookkeeping as wbc_rollout_ex. A robot flagged WBC_ST_BADPARAMS gets zero torques: the integrator plant freezes
 * it (as any flagged robot); the ground plant lets it go limp, and status_or keeps the flag. */
int wbc_rollout_params(wbc_handle* h, int kind, const wbc_plan* plan, int64_t n, int32_t n_steps, double dt,
                       const wbc_rollout_io* io, const wbc_rollout_opts* opts, const wbc_plant_perturb* perturb,
                       const wbc_plant_terrain* terrain, const wbc_ctrl_params* ctrl, void* stream);
int wbc_rollout_params_host(wbc_handle* h, int kind, const wbc_plan* plan, int64_t n, int32_t n_steps, double dt,
                            const wbc_rollout_io* host_io, const wbc_rollout_opts* opts, const wbc_plant_perturb* perturb,
                            const wbc_plant_terrain* terrain, const wbc_ctrl_params* ctrl);

/* ---- Imperfect sensing and actuation in the ground-plant loop: each robot's controller reads a noisy state, and its torque
 * command reaches a motor of its own strength one or more control steps late.
 *
 * Loop profile of robot i: noise[i][6] = standard deviations of the base orientation (rad), base position (m), joint angles
 * (rad), base angular velocity (rad/s), base linear velocity (m/s) and joint velocities (rad/s); delay[i] in [0, 15] control
 * steps; strength[i] >= 0, a factor on the applied torque; stream[i], a noise stream id (int32 read as uint32). Loop state of
 * robot i: hist[i][16][12], a ring of the last 16 commanded torques, and tick[i], the number of commands issued so far.
 *
 * Noise. Draw j in [0, 18) of step c = tick[i] is Philox4x32-10 (the function of cuRAND's curand_Philox4x32_10, multipliers
 * 0xD2511F53, 0xCD9E8D57, key increments 0x9E3779B9, 0xBB67AE85) of the counter (j, stream, c_lo, c_hi) under the key
 * (seed_lo, seed_hi); its words w0..w3 give u_a = (((w1 << 32) | w0) >> 11) 2^-53 + 2^-54 and u_b the same of (w3, w2), both
 * in (0, 1), and the normals z[2j] = sqrt(-2 ln u_a) cospi(2 u_b), z[2j+1] = sqrt(-2 ln u_a) sinpi(2 u_b). z[0:3] perturb
 * the orientation, z[3:6] the base position, z[6:18] the joint angles (q order), z[18:21] the angular velocity, z[21:24] the
 * linear velocity and z[24:36] the joint velocities. A robot's noise depends on (seed, stream, tick) only: not on its row, the
 * batch size or graph capture.
 *
 * Observe (tick unchanged): delta = sigma_rot z[0:3], theta = |delta|, dq = [cos theta/2, sin theta/2 delta / theta] (identity
 * for theta = 0), observed quaternion normalize(dq (x) q) (a world-frame perturbation, [w x y z]); every other block is
 * value + sigma z. A block with sigma = 0 is copied, so a zero-noise profile observes the true state bit for bit. Time and the
 * plan are not perturbed. The controller runs on the observed state (its metrics are what it observed).
 *
 * Actuate (after the controller, c = tick[i], d = delay[i]): hist[i][c mod 16] = tau_c; the applied torque is
 * strength[i] * hist[i][max(c - d, 0) mod 16] (until d commands exist the first one is held); tick[i] = c + 1. With d = 0 and
 * strength 1 the applied torque is the command bit for bit. The plant applies it to the true state; the controller's status of
 * step c still decides the plant's freeze in step c; io->tau keeps the last COMMANDED torque.
 *
 * Bad profile: a delay outside [0, 15], a sigma or strength that is negative or not finite, or tick < 0. Such a robot is
 * observed without noise, gets applied torque 0 and WBC_ST_BADLOOP in its controller status of the step (kept by status_or);
 * its hist and tick are unchanged. The ground plant does not freeze it: it goes limp, as a WBC_ST_BADPARAMS robot does. */
#define WBC_LOOP_HIST 16
typedef struct wbc_loop {
  const double* noise;      /* [N][6] or NULL: no noise                                                                   */
  const int32_t* delay;     /* [N] or NULL: no delay                                                                      */
  const double* strength;   /* [N] or NULL: strength 1                                                                    */
  const int32_t* stream;    /* [N] or NULL: the row index                                                                 */
  uint64_t seed;
  double* hist;             /* [N][16][12] and tick [N]: both given (in/out) or both NULL (library scratch from tick 0,   */
  int64_t* tick;            /* so each call starts a fresh history); only one of them is WBC_ERR_ARG                      */
} wbc_loop;

/* wbc_rollout_params (opts->plant must be 1) with sample plan -> observe -> controller -> actuate -> ground plant in every
 * step: two more launches per step, captured into the same graph. loop == NULL gives the bits and the launch count of
 * wbc_rollout_params. Device pointers (host pointers for _host; hist and tick are copied in and out). */
int wbc_rollout_loop(wbc_handle* h, int kind, const wbc_plan* plan, int64_t n, int32_t n_steps, double dt,
                     const wbc_rollout_io* io, const wbc_rollout_opts* opts, const wbc_plant_perturb* perturb,
                     const wbc_plant_terrain* terrain, const wbc_ctrl_params* ctrl, const wbc_loop* loop, void* stream);
int wbc_rollout_loop_host(wbc_handle* h, int kind, const wbc_plan* plan, int64_t n, int32_t n_steps, double dt,
                          const wbc_rollout_io* host_io, const wbc_rollout_opts* opts, const wbc_plant_perturb* perturb,
                          const wbc_plant_terrain* terrain, const wbc_ctrl_params* ctrl, const wbc_loop* loop);
/* The observe kernel alone: q_obs [N][19], v_obs [N][18] as the controller of step tick[i] sees them (tick is read, not
 * advanced; hist is not used). loop == NULL observes without noise. */
int wbc_loop_observe(wbc_handle* h, int64_t n, const wbc_loop* loop, const double* q, const double* v, double* q_obs, double* v_obs,
                     void* stream);
int wbc_loop_observe_host(wbc_handle* h, int64_t n, const wbc_loop* loop, const double* q, const double* v, double* q_obs,
                          double* v_obs);

/* ---- Rollout monitor of the ground-plant loop: per-robot fall detection, time to failure and effort statistics, accumulated on
 * the device one control step at a time. It only observes: no existing output changes.
 *
 * The monitor runs once per control step k, after the plant step. It sees the true post-step state q, v (time t_k + dt); the
 * plan sample traj, contact that the step's controller tracked (sampled at t_k); the torque the plant applied (the actuated
 * torque with a loop, else the command); the plant's ground forces f (world axes); and the step's full status word (the
 * controller status plus the plant's bits). The pose is compared with the sample at t_k, not t_k + dt: this one-step lag is exact
 * for a standing plan and adds about |pdot_plan| dt to the errors of a moving one.
 *
 * Per step, with p = q[4:7], q_hat = q[0:4] / |q[0:4]| and q_ref the quaternion of RollPitchYaw traj[9:12] (qz(yaw) (x) qy(pitch)
 * (x) qx(roll), Drake's convention):
 *   e_p     = |p - traj[0:3]|
 *   e_theta = 2 atan2(|u|, |w|) with (w, u) = conj(q_ref) (x) q_hat: the full rotation angle, accurate near 0 and near pi
 *   reasons = WBC_MON_POS if !(e_p <= pos_max), | WBC_MON_ANG if !(e_theta <= ang_max), | WBC_MON_STATUS if the status word is
 *             non-zero. A non-finite error therefore fails; a bound of +inf turns its test off.
 * Per-robot state (caller-owned, in/out; a zeroed state is a fresh one):
 *   steps[i]      steps monitored so far (incremented first)
 *   fail_step[i]  the value of steps at the first step with any reason, 0 while none; written once, never again
 *   fail_why[i]   the reasons at that step
 *   stats[i][11]  sums and maxima over every monitored step, before and after a failure; a maximum is m = e > m ? e : m
 *     SUM_POS2  += e_p^2                      MAX_POS  max e_p
 *     SUM_ANG2  += e_theta^2                  MAX_ANG  max e_theta
 *     TAU2_DT   += dt sum_a tau_a^2           WORK_ABS += dt sum_j |tau_{act_index[j]} v[v_index[j]]|
 *     SAT_MAX   max_j |tau_{act_index[j]}| / effort_j (the handle's model: joint j's effort limit, its actuator's torque)
 *     F_MAX     max over feet of |f_foot|
 *     STANCE_UNLOADED += feet planned in stance whose force is exactly 0 (all three components)
 *     SWING_LOADED    += feet planned in swing whose force is not 0
 *     DIST_XY   += dt |v[3:5]|
 *   why[i] (optional)  the reasons at the latest monitored step: the end-state verdict.
 * WORK_ABS and DIST_XY use the post-step velocities: under the plant's semi-implicit Euler they are exactly tau dtheta and the
 * step's horizontal base travel. The contact counters are exact tests: the plant's Gauss-Seidel starts from zero impulses and its
 * freeze writes 0, so an unloaded or frozen foot has a force of exactly 0. */
#define WBC_MON_NSTAT 11
#define WBC_MON_POS 1
#define WBC_MON_ANG 2
#define WBC_MON_STATUS 4
#define WBC_MON_SUM_POS2 0
#define WBC_MON_MAX_POS 1
#define WBC_MON_SUM_ANG2 2
#define WBC_MON_MAX_ANG 3
#define WBC_MON_TAU2_DT 4
#define WBC_MON_WORK_ABS 5
#define WBC_MON_SAT_MAX 6
#define WBC_MON_F_MAX 7
#define WBC_MON_STANCE_UNLOADED 8
#define WBC_MON_SWING_LOADED 9
#define WBC_MON_DIST_XY 10
typedef struct wbc_monitor {
  double pos_max, ang_max;  /* failure bounds (m, rad), >= 0 (+inf: off); NaN or negative is WBC_ERR_ARG                    */
  double* stats;            /* [N][11]  required                                                                         */
  int64_t* steps;           /* [N]      required                                                                         */
  int64_t* fail_step;       /* [N]      required                                                                         */
  int32_t* fail_why;        /* [N]      required                                                                         */
  int32_t* why;             /* [N] or NULL                                                                               */
} wbc_monitor;

/* wbc_rollout_loop (opts->plant must be 1; loop, perturb, terrain and ctrl may each be NULL) with the monitor after the plant
 * in every step: one more launch per step, captured into the same graph. Every existing output (q, v, t, tau, metrics,
 * status_or, err_max, metrics_log, opts->f_contact) has the bits of the call without a monitor; mon == NULL is wbc_rollout_loop
 * (its bits and launch count). Device pointers (host pointers for _host; the monitor state is copied in and out). */
int wbc_rollout_monitor(wbc_handle* h, int kind, const wbc_plan* plan, int64_t n, int32_t n_steps, double dt,
                        const wbc_rollout_io* io, const wbc_rollout_opts* opts, const wbc_plant_perturb* perturb,
                        const wbc_plant_terrain* terrain, const wbc_ctrl_params* ctrl, const wbc_loop* loop,
                        const wbc_monitor* mon, void* stream);
int wbc_rollout_monitor_host(wbc_handle* h, int kind, const wbc_plan* plan, int64_t n, int32_t n_steps, double dt,
                             const wbc_rollout_io* host_io, const wbc_rollout_opts* opts, const wbc_plant_perturb* perturb,
                             const wbc_plant_terrain* terrain, const wbc_ctrl_params* ctrl, const wbc_loop* loop,
                             const wbc_monitor* mon);
/* The monitor alone on one step's records: q [N][19], v [N][18] (post-step), traj [N][54], contact [N][4], tau_applied [N][12],
 * f_contact [N][12], status [N] (the step's status words, NULL: 0). */
int wbc_monitor_step(wbc_handle* h, int64_t n, double dt, const wbc_monitor* mon, const double* q, const double* v, const double* traj,
                     const uint8_t* contact, const double* tau_applied, const double* f_contact, const int32_t* status, void* stream);
int wbc_monitor_step_host(wbc_handle* h, int64_t n, double dt, const wbc_monitor* mon, const double* q, const double* v,
                          const double* traj, const uint8_t* contact, const double* tau_applied, const double* f_contact,
                          const int32_t* status);

/* ---- Actuator model of the ground-plant loop: per-robot torque-speed limits, motor lag and joint friction between the
 * actuated torque and the plant. Each step is sample plan -> observe -> controller -> actuate -> motor -> ground plant -> monitor.
 *
 * A motor set is K records. A record holds seven per-joint arrays [12] in the model's joint order k (the order of
 * wbc_model.effort): peak torque (N m, >= 0, +inf allowed), speed_knee (rad/s, >= 0, +inf allowed, <= speed_free), speed_free
 * (rad/s, >= 0, +inf allowed), lag (first-order time constant, s), damping (viscous friction, N m s/rad), coulomb (Coulomb
 * friction, N m) and coulomb_speed (regularisation speed, rad/s); the last four finite and >= 0, coulomb_speed > 0 where
 * coulomb > 0. Anything else is WBC_ERR_ARG at creation.
 *
 * Per robot i with record r = set[index[i]], for each joint k with actuator a = act_index[k]:
 *   w   = v[i][v_index[k]], the TRUE joint velocity at the start of the step
 *   u   = the torque reaching actuator a: the actuated torque with a loop, else the command
 *   lag: s = u if count[i] == 0 or lag_k == 0 (the first command primes the filter: no start-up transient, as the loop holds
 *        its first command); else s = m + alpha (u - m) with m = tau_m[i][a], alpha = -expm1(-dt / lag_k)
 *   envelope: L = peak_k, except in the motoring quadrant (s and w non-zero and of one sign) with |w| > speed_knee_k, where
 *        L = 0 if |w| >= speed_free_k, else peak_k (speed_free_k - |w|) / (speed_free_k - speed_knee_k) (with speed_free_k = +inf
 *        its limit, peak_k)
 *   out = s if |s| <= L, else copysign(L, s): a NaN s stays NaN (the plant's DIVERGED rule then freezes the robot)
 *   tau_m[i][a] = out: the clamped value is the state, so nothing winds up
 *   f   = -damping_k w - coulomb_k clamp(w / coulomb_speed_k, -1, 1); a zero coefficient adds nothing (not a signed zero, and
 *         a NaN w does not pass through it); with both zero the plant input is out itself
 *   plant input at a = out + f; count[i] += 1
 * Bad index (< 0 or >= K): motor and plant torque 0 and WBC_ST_BADMOTOR in the step's controller status (kept by status_or);
 * tau_m and count unchanged. No plant freeze mask holds the bit: the robot goes limp, as with WBC_ST_BADLOOP.
 * NULL set: one record with peak = the handle's effort and every other field off (knee = free = +inf, lag = damping =
 * coulomb = 0): saturation at the URDF effort. A record with peak = +inf and every other field off is the ideal motor: the
 * plant gets u bit for bit.
 * The monitor sees out (tau_m), the motor's torque, as the applied torque: SAT_MAX, TAU2_DT and WORK_ABS measure motor effort,
 * not friction (for a robot with a bad index, its unchanged tau_m). io->tau keeps the last COMMANDED torque.
 *
 * Explicit friction: friction uses the pre-step w, so damping_k + coulomb_k / coulomb_speed_k acts like the PD law's Kd and is
 * stable only while (that sum) dt / I < 2 for the joint's effective inertia I (about 1e-3 kg m^2 on the mini_cheetah knee links:
 * 1.5 N m s/rad diverges at dt = 5e-3). Larger values are legal physics at smaller dt and are not rejected; a robot that runs
 * away is flagged WBC_ST_DIVERGED by the plant and frozen. */
typedef struct wbc_motor_desc {
  double peak[WBC_NU];
  double speed_knee[WBC_NU];
  double speed_free[WBC_NU];
  double lag[WBC_NU];
  double damping[WBC_NU];
  double coulomb[WBC_NU];
  double coulomb_speed[WBC_NU];
} wbc_motor_desc;
/* A motor set keeps its device number and may outlive the handle. n_sets >= 1. */
typedef struct wbc_motor_set wbc_motor_set;
int wbc_motor_set_create(wbc_handle* h, int32_t n_sets, const wbc_motor_desc* descs, wbc_motor_set** out);
int wbc_motor_set_destroy(wbc_motor_set* s);

typedef struct wbc_plant_motor {
  const wbc_motor_set* set;  /* NULL: the one record of the handle's effort limits                                         */
  const int32_t* index;      /* [N] record of each robot, NULL = record 0                                                    */
  double* tau_m;             /* [N][12] (actuator order) and count [N]: both given (in/out) or both NULL (library scratch,   */
  int64_t* count;            /* zeroed at the start of each call); only one of them is WBC_ERR_ARG                           */
} wbc_plant_motor;

/* wbc_rollout_monitor (opts->plant must be 1; loop, mon, perturb, terrain and ctrl may each be NULL) with the motor between
 * actuation and the plant in every step: one more launch per step, captured into the same graph. motor == NULL is
 * wbc_rollout_monitor (its bits and launch count). Device pointers (host pointers for _host; tau_m and count are copied in and
 * out). */
int wbc_rollout_motor(wbc_handle* h, int kind, const wbc_plan* plan, int64_t n, int32_t n_steps, double dt,
                      const wbc_rollout_io* io, const wbc_rollout_opts* opts, const wbc_plant_perturb* perturb,
                      const wbc_plant_terrain* terrain, const wbc_ctrl_params* ctrl, const wbc_loop* loop, const wbc_monitor* mon,
                      const wbc_plant_motor* motor, void* stream);
int wbc_rollout_motor_host(wbc_handle* h, int kind, const wbc_plan* plan, int64_t n, int32_t n_steps, double dt,
                           const wbc_rollout_io* host_io, const wbc_rollout_opts* opts, const wbc_plant_perturb* perturb,
                           const wbc_plant_terrain* terrain, const wbc_ctrl_params* ctrl, const wbc_loop* loop,
                           const wbc_monitor* mon, const wbc_plant_motor* motor);
/* The motor alone on one step: v [N][18] (the true pre-step velocities), tau_in [N][12] (u, actuator order) -> tau_plant [N][12]
 * (the plant input); status [N] (or NULL) gets WBC_ST_BADMOTOR ORed in. motor->tau_m and motor->count are required: the motor
 * torque is motor->tau_m afterwards. */
int wbc_motor_apply(wbc_handle* h, int64_t n, double dt, const wbc_plant_motor* motor, const double* v, const double* tau_in,
                    double* tau_plant, int32_t* status, void* stream);
int wbc_motor_apply_host(wbc_handle* h, int64_t n, double dt, const wbc_plant_motor* motor, const double* v, const double* tau_in,
                         double* tau_plant, int32_t* status);

/* ---- State estimation in the ground-plant loop: a per-robot linear Kalman filter fuses a synthesised accelerometer with leg
 * kinematics, and the controller reads the estimated base position and linear velocity instead of observed ones. Each step is
 * sample plan -> observe -> estimate -> controller -> actuate -> motor -> ground plant -> monitor.
 *
 * Robot i has a filter state x[i][18] = (p, v, foot LF, RF, LH, RH), all world frame, its covariance P[i][18][18], v_prev[i][3]
 * (the true base linear velocity at its previous step) and count[i] (steps estimated so far), and uses record r = set[index[i]].
 * At step c = loop tick[i] it reads the loop's observed q_obs, v_obs, the true q, v (for the accelerometer and the statistics
 * only) and the step's planned contact flags. r_k(q) is foot k relative to the base origin in base axes and J_k(q) thetadot its
 * velocity from the leg's joint rates, both from the handle's joint_xyz / joint_axis / foot_xyz; R_true, R_obs are the base
 * rotations of q, q_obs; w_obs = v_obs[0:3] (world frame); g the model's gravity; s_k = 1 for a foot planned in stance and
 * swing_scale for one planned in swing.
 *   accelerometer  a_w = (v[3:6] - v_prev) / dt; f_b = R_true' (a_w - g) + sigma_acc z, z the normals of Philox draws 18 (two) and
 *                  19 (the first) of the loop counter (j, stream, c_lo, c_hi) under the loop seed, so that every draw of the loop
 *                  keeps its bits; sigma_acc = accel_noise[i] (NULL: 0, and 0 draws nothing); input a = R_obs f_b + g
 *   prime          (count <= 0) p = q_obs[4:7], v = v_obs[3:6], foot_k = p + R_obs r_k(q_obs); P = diag(p0_pos^2 (3), p0_vel^2 (3),
 *                  p0_foot^2 (12)); the output is the observed state; v_prev = v[3:6]; count = 1
 *   predict        v += dt a; p += dt v (the plant's semi-implicit Euler); feet unchanged; P = A P A' + Q with
 *                  Q = dt diag(q_pos^2 (3), q_vel^2 (3), (q_foot s_k)^2 (3 per foot)). With a perfect IMU and an exact prime,
 *                  prediction alone reproduces the plant's base position and velocity up to rounding.
 *   update         28 scalar rows with constant H and diagonal R, leg by leg:
 *                  y_p,k = R_obs r_k(q_obs), predicted foot_k - p, std r_pos s_k (3 rows)
 *                  y_v,k = -(w_obs x R_obs r_k + R_obs J_k(q_obs) thetadot_obs,k), predicted v, std r_vel s_k (3 rows: the
 *                          stance-foot zero-velocity constraint)
 *                  y_z,k = 0, predicted foot_k,z, std r_height s_k (flat ground, as the controller assumes)
 *                  A std of +inf drops its row: r_pos = r_vel = r_height = +inf is pure IMU dead reckoning. The batch form is
 *                  S = H P H' + R, K = P H' S^-1, x += K (y - H x), P = (I - K H) P, then P = (P + P') / 2; the kernel makes
 *                  the rows as sequential scalar updates, the same filter in exact arithmetic.
 *   output         the controller reads q_obs with [4:7] = p and v_obs with [3:6] = v, written in place into the loop's observed
 *                  state; orientation, angular velocity and joints stay observed. With an estimator the loop's base-position and
 *                  base-linear-velocity noise (blocks 1 and 4 of its profile) therefore no longer reach the controller (they
 *                  still perturb the prime).
 *                  v_prev = v[3:6]; count += 1; stats[i] (optional, [N][4]) += |p - p_true|^2, max= |p - p_true|,
 *                  += |v - v_true|^2, max= |v - v_true| against the true state at the start of the step, after the update
 *                  (prime steps included)
 *   failure        a scalar innovation variance not > 0, or x or P not finite after the step: the robot is controlled from the
 *                  observed state, count = 0 (a fresh prime next step), x, P, v_prev and stats unchanged, WBC_ST_BADESTIM
 *   bad index      (< 0 or >= K) WBC_ST_BADESTIM, nothing changes
 * WBC_ST_BADESTIM goes into the word the plant ORs its own status into: io->status_or without a monitor, the monitor's per-step
 * word with one (the step then fails with WBC_MON_STATUS, and the bit reaches io->status_or through the monitor). It is not a
 * controller status: no plant freeze mask holds it.
 *
 * Record fields are standard deviations: q_pos (m/sqrt(s)), q_vel (m/s/sqrt(s)), q_foot (m/sqrt(s)) of the process; r_pos (m),
 * r_vel (m/s), r_height (m) of the measurements (+inf allowed); swing_scale >= 1 (finite); p0_pos (m), p0_vel (m/s), p0_foot (m)
 * of the prime. NaN, a negative value, a non-finite process or initial std, or swing_scale < 1 or +inf is WBC_ERR_ARG at creation. */
typedef struct wbc_estimator_desc {
  double q_pos, q_vel, q_foot;
  double r_pos, r_vel, r_height;
  double swing_scale;
  double p0_pos, p0_vel, p0_foot;
} wbc_estimator_desc;
/* An estimator set keeps its device number and may outlive the handle. n_sets >= 1. */
typedef struct wbc_estimator_set wbc_estimator_set;
int wbc_estimator_set_create(wbc_handle* h, int32_t n_sets, const wbc_estimator_desc* descs, wbc_estimator_set** out);
int wbc_estimator_set_destroy(wbc_estimator_set* s);

typedef struct wbc_estimator {
  const wbc_estimator_set* set;  /* required                                                                                  */
  const int32_t* index;          /* [N] record of each robot, NULL = record 0                                                 */
  const double* accel_noise;     /* [N] accelerometer noise std (m/s^2), NULL = 0                                             */
  double* x;                     /* [N][18], P [N][18][18], v_prev [N][3] and count [N]: all given (in/out) or all NULL       */
  double* P;                     /* (library scratch, count 0: each call starts with a fresh prime); anything between is      */
  double* v_prev;                /* WBC_ERR_ARG                                                                               */
  int64_t* count;
  double* stats;                 /* [N][4] or NULL: sum |p err|^2, max |p err|, sum |v err|^2, max |v err| (accumulated)       */
} wbc_estimator;

/* wbc_rollout_motor (opts->plant must be 1, loop required; motor, mon, perturb, terrain and ctrl may each be NULL) with the
 * estimator between observe and the controller in every step: one more launch per step, captured into the same graph.
 * est == NULL is wbc_rollout_motor (its bits and launch count); an estimator without a loop or without the ground plant is
 * WBC_ERR_ARG. Device pointers (host pointers for _host; the estimator state and stats are copied in and out). */
int wbc_rollout_estimator(wbc_handle* h, int kind, const wbc_plan* plan, int64_t n, int32_t n_steps, double dt,
                          const wbc_rollout_io* io, const wbc_rollout_opts* opts, const wbc_plant_perturb* perturb,
                          const wbc_plant_terrain* terrain, const wbc_ctrl_params* ctrl, const wbc_loop* loop,
                          const wbc_monitor* mon, const wbc_plant_motor* motor, const wbc_estimator* est, void* stream);
int wbc_rollout_estimator_host(wbc_handle* h, int kind, const wbc_plan* plan, int64_t n, int32_t n_steps, double dt,
                               const wbc_rollout_io* host_io, const wbc_rollout_opts* opts, const wbc_plant_perturb* perturb,
                               const wbc_plant_terrain* terrain, const wbc_ctrl_params* ctrl, const wbc_loop* loop,
                               const wbc_monitor* mon, const wbc_plant_motor* motor, const wbc_estimator* est);
/* The estimator alone on one step: true q [N][19], v [N][18]; q_obs [N][19], v_obs [N][18] (in/out); contact [N][4]; the loop
 * gives seed, stream and tick (NULL tick: 0; the tick is read, not advanced); status_or [N] (or NULL) gets WBC_ST_BADESTIM ORed
 * in. est->x, P, v_prev and count are required. */
int wbc_estimator_step(wbc_handle* h, int64_t n, double dt, const wbc_estimator* est, const wbc_loop* loop, const double* q,
                       const double* v, double* q_obs, double* v_obs, const uint8_t* contact, int32_t* status_or, void* stream);
int wbc_estimator_step_host(wbc_handle* h, int64_t n, double dt, const wbc_estimator* est, const wbc_loop* loop, const double* q,
                            const double* v, double* q_obs, double* v_obs, const uint8_t* contact, int32_t* status_or);

/* ---- Contact detection in the ground-plant loop: per robot, each foot's ground force is estimated from the joint torques and
 * the motion they produced, and a hysteresis on its world-z component gives the foot's stance flag. The estimator and the
 * controller may read the detected flags instead of the planned ones. Each step is
 * sample plan -> observe -> detect -> estimate -> controller -> actuate -> motor -> ground plant -> record -> monitor.
 *
 * Robot i has the state q_prev[i][19], v_prev[i][18] (what the detector read at its previous step), tau_prev[i][12] (the measured
 * torque of its latest step, actuator order), f_true[i][12] (the plant's ground forces of its latest step, statistics only),
 * f_hat[i][12] (filtered force, world axes, foot k at 3 k), flag[i][4] and count[i], and uses record r = set[index[i]]. At each step
 * it reads q, v: the loop's observed state (before the estimator overwrites it) with a loop, the true state without one.
 *   prime     (count <= 0) flag = the plan's flags, f_hat = 0, q_prev = q, v_prev = v, count = 1
 *   estimate  M, Cv + tau_g (controller sign) and the foot Jacobians J_k taken at q_prev, v_prev with the handle's model; per leg k
 *             the three joint rows of  r = M (v - v_prev) - dt (B tau_prev - Cv - tau_g)  give r_k, and  J_k,leg' p_k = r_k
 *             (J_k,leg the 3 x 3 block of J_k over leg k's joint columns) gives f_raw,k = p_k / dt in world axes.
 *             The plant's step is v+ = v + dt M^-1 (B tau - Cv - tau_g) + M^-1 (J_c' p + push), with a push on base rows only,
 *             so with the true state and the torque the plant received, f_raw reproduces the plant's f_contact up to rounding.
 *   singular  |det J_k,leg| <= 1e-9 |a0| |a1| |a2|, a_j the columns of J_k,leg: f_hat and flag of that foot are held and it adds
 *             nothing to the statistics of the step
 *   filter    f_hat = f_raw on the first estimate after a prime (count == 1) or with tau_f = 0, else
 *             f_hat += alpha (f_raw - f_hat), alpha = -expm1(-dt / tau_f)
 *   flags     a foot at 0 goes to 1 when f_hat_z >= f_on; a foot at 1 goes to 0 when f_hat_z <= f_off
 *   stats     (optional, [N][6], accumulated) sum over estimated steps of sum_k |f_raw,k - f_true,k|^2, the maximum over steps and
 *             feet of |f_raw,k - f_true,k|, then per foot and step the counts of true stance (flag 1, loaded), true swing (0, not
 *             loaded), false stance (1, not loaded) and false swing (0, loaded); a foot is loaded when any component of its
 *             f_true is non-zero (the monitor's rule). f_true is the previous step's: the forces of the step that led to q, v.
 *   then      q_prev = q, v_prev = v, count += 1
 *   failure   a non-finite f_raw of a foot that is not singular: count = 0, everything else unchanged, WBC_ST_BADCONTACT
 *   bad index (< 0 or >= K) WBC_ST_BADCONTACT, nothing changes (the record step leaves the robot alone too)
 * A failed or bad robot outputs the plan's flags for the step. WBC_ST_BADCONTACT goes into the word the plant ORs its own status
 * into, as WBC_ST_BADESTIM does; no plant freeze mask holds it.
 * After the plant, the record step copies the measured torque (the motor torque tau_m with a motor - joint friction is not
 * measured -, else the actuated torque with a loop, else the command: the torque the monitor treats as applied) into tau_prev and
 * the plant's forces into f_true, so that the state carries everything a later call needs.
 *
 * Consumers (feed, a mask): WBC_CONTACT_FEED_ESTIMATOR - the estimator's s_k uses the detected flags instead of the planned ones
 * (WBC_ERR_ARG without an estimator); WBC_CONTACT_FEED_CONTROLLER - the controller's contact input is plan AND detected, so that a
 * late touchdown waits and a slipping or unloaded planned-stance foot carries no QP force, while a loaded foot is still released
 * to swing at lift-off. feed = 0 only observes. The monitor reads the planned flags in every mode.
 *
 * Record fields: tau_f (s) finite and >= 0; f_on, f_off (N) not NaN with f_off <= f_on (+-inf allowed: f_off = -inf never
 * releases a detected foot). Anything else is WBC_ERR_ARG at creation. */
#define WBC_CONTACT_FEED_ESTIMATOR 1
#define WBC_CONTACT_FEED_CONTROLLER 2
typedef struct wbc_contact_desc {
  double tau_f, f_on, f_off;
} wbc_contact_desc;
/* A contact set keeps its device number and may outlive the handle. n_sets >= 1. */
typedef struct wbc_contact_set wbc_contact_set;
int wbc_contact_set_create(wbc_handle* h, int32_t n_sets, const wbc_contact_desc* descs, wbc_contact_set** out);
int wbc_contact_set_destroy(wbc_contact_set* s);

typedef struct wbc_contact {
  const wbc_contact_set* set;    /* required                                                                                  */
  const int32_t* index;          /* [N] record of each robot, NULL = record 0                                                 */
  int32_t feed;                  /* WBC_CONTACT_FEED_* mask                                                                   */
  double* q_prev;                /* [N][19], v_prev [N][18], tau_prev [N][12], f_true [N][12], f_hat [N][12], flag [N][4] and */
  double* v_prev;                /* count [N]: all given (in/out) or all NULL (library scratch, count 0: each call starts with */
  double* tau_prev;              /* a prime); anything between is WBC_ERR_ARG                                                 */
  double* f_true;
  double* f_hat;
  uint8_t* flag;
  int64_t* count;
  double* stats;                 /* [N][6] or NULL (accumulated, see above)                                                   */
} wbc_contact;

/* wbc_rollout_estimator (opts->plant must be 1; loop, est, motor, mon, perturb, terrain and ctrl may each be NULL) with the
 * detector after observe and the record step after the plant: two more launches per step, captured into the same graph.
 * det == NULL is wbc_rollout_estimator (its bits and launch count). Without opts->f_contact the plant's forces go to scratch.
 * Device pointers (host pointers for _host; the detector state and stats are copied in and out). */
int wbc_rollout_contact(wbc_handle* h, int kind, const wbc_plan* plan, int64_t n, int32_t n_steps, double dt,
                        const wbc_rollout_io* io, const wbc_rollout_opts* opts, const wbc_plant_perturb* perturb,
                        const wbc_plant_terrain* terrain, const wbc_ctrl_params* ctrl, const wbc_loop* loop,
                        const wbc_monitor* mon, const wbc_plant_motor* motor, const wbc_estimator* est, const wbc_contact* det,
                        void* stream);
int wbc_rollout_contact_host(wbc_handle* h, int kind, const wbc_plan* plan, int64_t n, int32_t n_steps, double dt,
                             const wbc_rollout_io* host_io, const wbc_rollout_opts* opts, const wbc_plant_perturb* perturb,
                             const wbc_plant_terrain* terrain, const wbc_ctrl_params* ctrl, const wbc_loop* loop,
                             const wbc_monitor* mon, const wbc_plant_motor* motor, const wbc_estimator* est, const wbc_contact* det);
/* The detector alone on one step: q [N][19], v [N][18] (what it reads), contact [N][4] (the plan's flags) -> detected [N][4];
 * status_or [N] (or NULL) gets WBC_ST_BADCONTACT ORed in. tau_prev and f_true are read from the state, which is required;
 * det->feed is ignored. */
int wbc_contact_step(wbc_handle* h, int64_t n, double dt, const wbc_contact* det, const double* q, const double* v,
                     const uint8_t* contact, uint8_t* detected, int32_t* status_or, void* stream);
int wbc_contact_step_host(wbc_handle* h, int64_t n, double dt, const wbc_contact* det, const double* q, const double* v,
                          const uint8_t* contact, uint8_t* detected, int32_t* status_or);

/* Number of kernel launches issued through this handle since creation. */
int64_t wbc_launch_count(const wbc_handle* h);

#ifdef __cplusplus
}
#endif
#endif /* WBC_B200_H */
