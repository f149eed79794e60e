/*
 * farms_b200.h -- C ABI of the B200-native batched FARMS stepping engine.
 *
 * The reference (farmsim/farms_mujoco) has no C ABI of its own for this path:
 * its native code is Cython `cpdef` functions called with Python objects
 * (farms_mujoco/sensors/sensors.pxd:12-29, farms_mujoco/swimming/drag.pyx:152,
 * 389) and its physics is the third-party MuJoCo C library reached through
 * dm_control (farms_mujoco/simulation/simulation.py:53,83-89,156,175).  Each
 * entry point below therefore cites the reference interface it replaces; the
 * binding a reference maintainer would add is shown in INTEGRATION.md.
 *
 * Conventions
 *   - plain C types only; all pointers are HOST pointers unless the name ends
 *     in `_dev` (device pointers, e.g. a torch tensor's data_ptr()).
 *   - every function returns 0 on success, <0 on error; fb_last_error() gives
 *     the message of the last failing call made on the calling thread.
 *   - the engine owns all device buffers; views are borrowed and stay valid
 *     until fb_destroy().
 *   - one handle = one device + one stream; calls on one handle are not
 *     re-entrant.  Handles on different devices may be driven concurrently.
 *   - reals cross the ABI as float64 (the reference's dtype, sensors.pyx:
 *     156-157); the device computes in float32.
 */
#ifndef FARMS_B200_H_
#define FARMS_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FB_ABI_VERSION 2

/* joint / geom enums follow MuJoCo's mjtJoint / mjtGeom numbering */
enum { FB_JNT_FREE = 0, FB_JNT_BALL = 1, FB_JNT_SLIDE = 2, FB_JNT_HINGE = 3 };
enum { FB_GEOM_PLANE = 0, FB_GEOM_SPHERE = 2, FB_GEOM_CAPSULE = 3, FB_GEOM_ELLIPSOID = 4, FB_GEOM_CYLINDER = 5, FB_GEOM_BOX = 6 };

/* Compiled model: the mjModel subset the path reads (SURVEY.md Appendix A).
 * Replaces: mjcf.Physics.from_mjcf_model(mjcf_model), simulation.py:53. */
typedef struct FbModel {
  int32_t nbody, njnt, nq, nv, nu, ngeom, ncand, nM;
  /* <option> (mjcf.py:1326-1403) */
  double timestep;
  double gravity[3];
  double impratio;
  int32_t solver_iterations;
  double tolerance;
  double meaninertia;
  /* bodies [nbody]; body 0 is the world; depth-first order (parent < child) */
  const int32_t *body_parentid, *body_jntid, *body_dofadr, *body_dofnum;
  const double *body_pos, *body_quat, *body_ipos, *body_iquat; /* 3,4,3,4 */
  const double *body_mass, *body_inertia, *body_invweight0;    /* 1,3,2 */
  /* joints [njnt] (<=1 per body) */
  const int32_t *jnt_type, *jnt_bodyid, *jnt_qposadr, *jnt_dofadr, *jnt_limited;
  const double *jnt_pos, *jnt_axis, *jnt_stiffness, *jnt_range, *jnt_margin;
  const double *jnt_solref, *jnt_solimp; /* 2,5 */
  /* dofs [nv] */
  const int32_t *dof_bodyid, *dof_jntid, *dof_parentid, *dof_Madr;
  const double *dof_damping, *dof_armature, *dof_invweight0;
  const double *qpos0, *qpos_spring; /* [nq] */
  /* collision geoms [ngeom] */
  const int32_t *geom_type, *geom_bodyid;
  const double *geom_pos, *geom_quat, *geom_size; /* 3,4,3 */
  /* plane-vs-{sphere, capsule end} candidates [ncand], parameters pre-mixed */
  const int32_t *cand_geom1, *cand_geom2, *cand_end;
  const double *cand_friction, *cand_solref, *cand_solimp, *cand_margin, *cand_gap;
  /* actuators [nu]: force = gain0*ctrl + bias0 + bias1*q + bias2*qvel */
  const int32_t *actuator_trnid, *actuator_ctrllimited, *actuator_forcelimited;
  const double *actuator_gainprm, *actuator_biasprm;          /* 3,3 */
  const double *actuator_ctrlrange, *actuator_forcerange, *actuator_gear;
  /* keyframe 0 (task.py:137 physics.reset(keyframe_id=0)) */
  const double *key_qpos, *key_qvel;
} FbModel;

/* farms-side contract: index maps (physics.py:188-393), swimming tables
 * (drag.pyx:333-387), units (physics.py:428-523).  Replaces:
 * get_physics2data_maps() + SwimmingHandler.__init__(). */
typedef struct FbFarms {
  int32_t n_links, n_joints, n_contacts, n_xfrc, n_swim;
  int32_t link_cols, joint_cols, contact_cols, xfrc_cols; /* 20,18,12,6 */
  /* joint-row column indices (layout.py; farms_core sensor_convention) */
  int32_t col_joint_position, col_joint_velocity, col_joint_torque, col_joint_limit_force;
  const int32_t *link_body;          /* [n_links]  xpos2data == xquat2data == xipos2data */
  const int32_t *joint_qposadr;      /* [n_joints] qpos2data */
  const int32_t *joint_dofadr;       /* [n_joints] qvel2data */
  const int32_t *joint_jntid;        /* [n_joints] joint of jointlimitfrc_<j>, -1 if absent */
  const int32_t *joint_act_position; /* [n_joints] actuator of actuatorfrc_position_<j>, -1 */
  const int32_t *joint_act_velocity; /* [n_joints] actuator of actuatorfrc_velocity_<j>, -1 */
  const int32_t *joint_act_torque;   /* [n_joints] actuator of actuatorfrc_torque_<j>, -1 (empty in the reference, SURVEY.md D-4) */
  const int32_t *cand_sensor;        /* [ncand,4] contact-sensor index for the keys (g1,g2) (g2,g1) (g1,-1) (g2,-1), -1 if absent; signs -1,+1,-1,+1 (sensors.pyx:163-170) */
  const int32_t *xfrc_body;          /* [n_xfrc] data2xfrc */
  /* swimming links (drag.pyx:353-385) */
  const int32_t *swim_links_index, *swim_xfrc_index; /* [n_swim] */
  const double *swim_mass, *swim_height, *swim_density; /* [n_swim] */
  const double *swim_coefficients;   /* [n_swim,2,3] */
  int32_t water_drag, water_sph, water_buoyancy;
  double water_surface, water_density, water_viscosity;
  double water_velocity[3];
  double meters, seconds, kilograms;
} FbFarms;

/* On-device controller (replaces the per-step Python of task.py:288-346):
 * ctrl[act_position[j]] = offset[j] + amplitude[j]*sin(2*pi*frequency[j]*t
 *                         - phase_lag[j] + env_phase[env]),  t = iteration*timestep.
 * Joints with act id -1 are skipped.  All arrays are host pointers. */
typedef struct FbWaveController {
  int32_t n;                  /* number of controlled joints */
  const int32_t *actuator;    /* [n] ctrl index written (maps['ctrl']['pos']) */
  const double *amplitude, *frequency, *phase_lag, *offset; /* [n] */
} FbWaveController;

/* On-device central pattern generator (coupled phase oscillators with amplitude dynamics), the
 * batched stand-in for a farms_core network controller driven through step_control
 * (task.py:288-346).  Per environment and physics step (explicit Euler, dt = timestep):
 *   theta_i' = 2 pi frequency_i + sum_c weight_c r_from(c) sin(theta_from(c) - theta_i - bias_c)
 *   r_i''    = rate_i (rate_i/4 (amplitude_i - r_i) - r_i')
 *   ctrl[out_actuator_o] = out_offset_o + out_gain_o (r_a (1 + cos theta_a) - r_b (1 + cos theta_b))
 *                          (out_osc_b < 0: out_gain_o r_a cos theta_a)
 * ctrl of iteration k is the output after k Euler steps.  A position target writes the joint's
 * position actuator; a torque command writes its motor actuator with out_gain = units.torques
 * (task.py:332).  At most 64 oscillators.  All arrays are host pointers. */
typedef struct FbCpgNetwork {
  int32_t n_osc, n_coupling, n_out;
  const double *frequency, *amplitude, *rate;        /* [n_osc] Hz, nominal amplitude, convergence rate 1/s */
  const int32_t *coupling_from, *coupling_to;        /* [n_coupling] oscillator j acts on oscillator i */
  const double *coupling_weight, *coupling_bias;     /* [n_coupling] w_ij, phi_ij */
  const int32_t *out_actuator, *out_osc_a, *out_osc_b; /* [n_out] */
  const double *out_gain, *out_offset;               /* [n_out] */
} FbCpgNetwork;

typedef struct FbHandle FbHandle;

/* Device log, float32, environment-minor so that the 32 environments of a warp write one
 * contiguous run per store.  A kind with N items and C columns is stored in vectors of V
 * columns (links 4, joints 2, contacts 4, xfrc 2):
 *
 *   <kind>_dev[ (((it*N + item)*(C/V) + col/V)*env_pad + env)*V + col%V ]
 *
 * i.e. the 5-D strided array [ring][N][C/V][env_pad][V]; indexed (env, it, item, col) it holds
 * exactly the reference's data.sensors.<kind>.array[it, item, col] ([buffer_size, n_items,
 * n_cols], task.py:158) of environment env.  fb_export_farms() returns one environment in
 * the reference's own (contiguous, float64) layout; fb_step_host() returns the last row of
 * every environment as dense [n_envs][N][C]. */
typedef struct FbLogView {
  float *links_dev, *joints_dev, *contacts_dev, *xfrc_dev;
  int32_t links_vec, joints_vec, contacts_vec, xfrc_vec; /* V of each kind */
  int32_t ring, n_envs, env_pad;                         /* env_pad = n_envs rounded up to 32 */
} FbLogView;

/* Device state views (float32), one row per environment. */
typedef struct FbStateView {
  float *qpos_dev;   /* [n_envs][nq] */
  float *qvel_dev;   /* [n_envs][nv] */
  float *ctrl_dev;   /* [n_envs][nu] */
  float *xfrc_applied_dev; /* [n_envs][nbody][6] world wrench applied at xipos (force, torque) */
  float *qpos_spring_dev;  /* [n_envs][nq] */
  float *env_phase_dev;    /* [n_envs] */
  int32_t *flags_dev;      /* [n_envs] bit0: non-finite state (PhysicsError analogue, simulation.py:157-161); bit1: contact overflow; bit2: solver not converged */
  int64_t *iteration_dev;  /* [n_envs] batch iteration: physics steps since fb_reset, the same for every environment after each step (fb_get_episode_start maps it to an environment's episode) */
} FbStateView;

/* mjData-like derived quantities of the state at the START of the last step
 * (SURVEY.md Appendix D-1), float32, written when fb_step(..., want_derived=1).
 * These are what physics.data.{xpos,xquat,xipos,sensordata,contact} expose. */
typedef struct FbDerivedView {
  float *xpos_dev, *xquat_dev, *xipos_dev;  /* [n_envs][nbody][3|4|3] */
  float *linvel_dev, *angvel_dev;           /* [n_envs][nbody][3] framelinvel / frameangvel (objtype=body) */
  float *actuator_force_dev;                /* [n_envs][nu] */
  float *jnt_limit_force_dev;               /* [n_envs][njnt] */
  float *qacc_dev;                          /* [n_envs][nv] */
  int32_t *ncon_dev;                        /* [n_envs] */
  int32_t *con_cand_dev;                    /* [n_envs][maxcon] candidate index of each contact */
  float *con_dist_dev;                      /* [n_envs][maxcon] */
  float *con_pos_dev;                       /* [n_envs][maxcon][3] */
  float *con_frame_dev;                     /* [n_envs][maxcon][9] */
  float *con_force_dev;                     /* [n_envs][maxcon][3] mj_contactForce (normal, t1, t2) */
  int32_t maxcon;
} FbDerivedView;

const char *fb_last_error(void);
int fb_abi_version(void);

/* Create an engine for n_envs environments on CUDA device `device`, with a
 * log ring of `ring_steps` rows (task.py:62 buffer_size).  team_lanes = lanes
 * cooperating on one environment (1,2,4,8,16,32; 0 = automatic). */
int fb_create(const FbModel *model, const FbFarms *farms, int n_envs, int device,
              int ring_steps, int team_lanes, FbHandle **out);
void fb_destroy(FbHandle *h);

/* Episode reset (task.py:87-154 + dm_control reset -> mj_forward): state <-
 * qpos0/qvel0 ([n_envs,nq]/[n_envs,nv] host float64, NULL -> keyframe 0),
 * ctrl <- 0, iteration <- 0; runs the forward pass and writes log row 0. */
int fb_reset(FbHandle *h, const double *qpos0, const double *qvel0);

/* Per-environment episodes: restart some environments while the others keep running.  At batch
 * iteration it, a restarted environment e takes the given state (or the keyframe), ctrl, xfrc_applied
 * and flags <- 0, its on-device CPG rows <- the state last set by fb_set_cpg_state (rates 0), and
 * runs the reset's forward pass, which writes its log row it % ring (the episode's row 0; the
 * previous episode's terminal row there is overwritten) and its derived view.  From then on it steps
 * bit for bit as environment e of a fresh batch (fb_reset, fb_set_cpg_state) would: the
 * travelling-wave controller reads the episode's time.  qpos_spring, env_phase and the
 * per-environment parameter tables are kept, as fb_reset keeps them.  Batch-wide nothing changes:
 * the batch iteration, the control sequence and its position, the kernel selection.
 *
 * Restart the environments in envs[n] (host, no duplicates); qpos0 [n][nq] / qvel0 [n][nv] host
 * float64 rows in the order of envs, NULL -> keyframe.  Uploads O(n) rows, not O(n_envs); n = 0
 * enqueues nothing.  Refused, naming the first bad entry: an index out of range or given twice,
 * a non-finite qpos0 / qvel0 value. */
int fb_reset_envs(FbHandle *h, int n, const int32_t *envs, const double *qpos0, const double *qvel0);
/* Same from device memory, stream-ordered, no host synchronisation: mask [n_envs] uint8 (non-zero
 * = restart), qpos0 [n_envs][nq] / qvel0 [n_envs][nv] float32 (rows of unmasked environments are
 * not read; NULL -> keyframe).  Write them on the handle's stream (fb_device_ptr_stream) or
 * synchronise first.  Device data cannot be validated here: a non-finite row shows as flags bit 0
 * after the next step. */
int fb_reset_envs_where(FbHandle *h, const uint8_t *mask, const float *qpos0, const float *qvel0);
/* [n_envs] batch iteration of each environment's episode row 0 (0 after fb_reset).  Accessors of
 * one environment (fb_export_farms) return its current episode; whole-batch ones (fb_export_rows,
 * fb_step_host, FbLogView) keep batch rows. */
int fb_get_episode_start(FbHandle *h, int64_t *out);

/* Control inputs (task.py:307,317,332,343-346). */
int fb_set_ctrl(FbHandle *h, const double *ctrl);                 /* [n_envs][nu] */
int fb_set_qpos_spring(FbHandle *h, const double *qpos_spring);   /* [n_envs][nq] */
/* Open-loop control for the next n_steps physics steps: ctrl[n_steps][n_envs][nu] float32 host
 * (what step_joints_control_* would write before each step, task.py:309-346).  Following
 * fb_step calls consume it in order (a call may not ask for more steps than remain); when it
 * is used up ctrl is held at its last entry.  NULL or n_steps = 0 switches it off; fb_reset
 * clears it.  Actuators driven by the on-device wave controller keep the wave. */
int fb_set_ctrl_sequence(FbHandle *h, const float *ctrl, int n_steps);
int fb_set_env_phase(FbHandle *h, const double *phase);           /* [n_envs] */
int fb_set_wave_controller(FbHandle *h, const FbWaveController *c); /* NULL -> off */
/* On-device CPG (NULL -> off).  While it is on, every fb_step first integrates the network for
 * the steps of the launch and writes their ctrl into the control sequence (the actuators it does
 * not drive keep their held ctrl); a sequence uploaded with fb_set_ctrl_sequence is refused.
 * fb_set_cpg_state: phase [n_envs][n_osc] (and amplitude, NULL -> 0; rates of change start at 0);
 * fb_reset keeps the state (set it again for a new episode). */
int fb_set_cpg(FbHandle *h, const FbCpgNetwork *net);
/* Spring references driven by the network (task.py:338-346: model.qpos_spring[joint] =
 * controller.springrefs()[joint], every iteration): output s sets qpos_spring[qpos_adr[s]] of every
 * step of a launch to offset + gain * (the oscillator expression above), read by the step kernels
 * from the same per-launch sequence as ctrl; qpos_spring ends a launch at the last value used.
 * Call after fb_set_cpg (which clears them); n = 0 clears.  qpos_adr: hinge / slide joints. */
int fb_set_cpg_springrefs(FbHandle *h, int n, const int32_t *qpos_adr, const int32_t *osc_a, const int32_t *osc_b,
                          const double *gain, const double *offset);
int fb_set_cpg_state(FbHandle *h, const double *phase, const double *amplitude);
int fb_get_cpg_state(FbHandle *h, double *phase, double *amplitude);
/* Model edit of ExperimentTask.initialize_control (task.py:262-286): the reference sets
 * actuator_forcelimited / actuator_forcerange ([0, 0]) on the position and velocity
 * actuators of joints whose motor has no 'position' control type.  limited[n], range[n][2]. */
int fb_set_actuator_forcerange(FbHandle *h, int n, const int32_t *actuator, const int32_t *limited,
                               const double *range);
/* Water velocity (drag.pyx:417-419 set_water_velocity). */
int fb_set_water_velocity(FbHandle *h, double vx, double vy, double vz);
/* Drag on/off overrides for the fused swimming step (drag.pyx:393-395). */
int fb_set_swimming(FbHandle *h, int drag, int buoyancy);

/* Per-environment physical parameters (parameter sweeps, domain randomisation): each field is either
 * the model's value for every environment (default) or a table of one value set per environment.
 *   FB_ENV_JNT_STIFFNESS   [n_envs][njnt]     model.jnt_stiffness
 *   FB_ENV_DOF_DAMPING     [n_envs][nv]       model.dof_damping
 *   FB_ENV_DRAG_COEF       [n_envs][n_swim][2][3]  FbFarms.swim_coefficients (linear xyz, angular xyz)
 *   FB_ENV_WATER_VELOCITY  [n_envs][3]        FbFarms.water_velocity
 *   FB_ENV_CAND_FRICTION   [n_envs][ncand]    FbModel.cand_friction: the mixed sliding friction of each
 *                                             collision candidate (the geoms' friction put through the
 *                                             compiler's mixing rule, mjcf_subset.candidate_friction)
 *   FB_ENV_ACT_GAIN        [n_envs][nu]       model.actuator_gainprm[:, 0] (the fixed gain; the other
 *                                             columns are not read)
 *   FB_ENV_ACT_BIAS        [n_envs][nu][3]    model.actuator_biasprm[:, 0:3]
 *                                             (a <position kp> is gain kp, bias [0, -kp, 0]; a
 *                                             <velocity kv> is gain kv, bias [0, 0, -kv])
 * Environment e then steps exactly as the model edited to e's values.  values: host float64; NULL
 * returns the field to the model's value.  Refused, with the field and the first bad index named:
 * non-finite values, negative stiffness or damping (drag coefficients are negative in FARMS and a
 * water velocity has any sign), a non-zero stiffness or damping
 * on the free joint, drag coefficients or water velocity on a model without swimming links, a
 * candidate friction below 0.1 (the pyramid rows stiffen as 1/mu^2 and the fp32 solver's error grows
 * with them), and a friction of an explicit <pair> candidate (cand_end 20 or 21) other than the
 * model's: a pair takes its friction from the pair element.  Gains and biases have no sign check, as
 * in MuJoCo: a velocity gain too large for the explicit Euler step diverges and shows as flags bit
 * 0, like any divergence.  The
 * tables survive fb_reset and fb_reset_envs and are freed by fb_destroy; while FB_ENV_WATER_VELOCITY is set,
 * fb_set_water_velocity is refused.  fb_get_env_param returns the values in the same layout (the
 * model's value broadcast for a field that is not set). */
enum { FB_ENV_JNT_STIFFNESS = 0, FB_ENV_DOF_DAMPING = 1, FB_ENV_DRAG_COEF = 2, FB_ENV_WATER_VELOCITY = 3,
       FB_ENV_CAND_FRICTION = 4, FB_ENV_ACT_GAIN = 5, FB_ENV_ACT_BIAS = 6 };
int fb_set_env_param(FbHandle *h, int field, const double *values);
int fb_get_env_param(FbHandle *h, int field, double *out);

/* Advance every environment by n_steps physics steps (simulation.py:155-156
 * env.step -> mj_step, with task.before_step's sensor logging, the swimming
 * callback and the controller fused in).  Step j writes log row (j+1) % ring.
 * Asynchronous on the handle's stream unless sync != 0. */
int fb_step(FbHandle *h, int n_steps, int want_derived, int sync);
int fb_synchronize(FbHandle *h);
/* CUDA-event time of the last fb_step launch in milliseconds (after sync). */
int fb_last_step_ms(FbHandle *h, float *ms);
/* number of kernels launched by this handle so far */
int64_t fb_launch_count(FbHandle *h);

int fb_log_view(FbHandle *h, FbLogView *out);
int fb_state_view(FbHandle *h, FbStateView *out);
int fb_derived_view(FbHandle *h, FbDerivedView *out);

/* Copy one environment's log to host float64 arrays shaped like the
 * reference's data.sensors.<kind>.array (NULL pointers are skipped).  Rows are those of the
 * environment's current episode: row r is device row (s + r) % ring, s = its episode start; when
 * s > 0, rows the episode has not reached yet are zero (as in a fresh log). */
int fb_export_farms(FbHandle *h, int env, double *links, double *joints,
                    double *contacts, double *xfrc);
/* End-to-end call on HOST buffers (pinned recommended), the batched analogue of
 * one outer iteration of the reference loop (task.py:168-186: control written
 * by host code, env.step, sensors read by host code):
 *   ctrl / qpos / qvel: [n_envs][nu|nq|nv] float32 host, each may be NULL (keep
 *       the device-resident value); uploaded before stepping
 *   n_steps physics steps with the inputs held
 *   links_row / joints_row: [n_envs][n_links][20] / [n_envs][n_joints][joint_cols]
 *       float32 host, the last log row of every environment (NULL -> skipped) */
int fb_step_host(FbHandle *h, const float *ctrl, const float *qpos, const float *qvel,
                 int n_steps, float *links_row, float *joints_row);
/* Pipelined form: returns once everything is enqueued.  The device->host copies run on a
 * second stream, so the transfer of call i overlaps the kernels of call i+1; links_row /
 * joints_row (pinned) are complete after fb_host_wait() or after the NEXT-but-one call
 * returns -- alternate two host buffer pairs.
 * Buffer reuse rule for the INPUTS: a pinned `ctrl` is read by the SMs asynchronously on an upload
 * stream (and pinned qpos / qvel by cudaMemcpyAsync), so ctrl / qpos / qvel must stay unmodified
 * until fb_host_wait_call() of this call's index (fb_host_call_count() before the call; calls that
 * ask for no rows have no index) or fb_host_wait() returns -- rotate as many ctrl buffers as row
 * buffer sets. */
int fb_step_host_async(FbHandle *h, const float *ctrl, const float *qpos, const float *qvel,
                       int n_steps, float *links_row, float *joints_row);
int fb_host_wait(FbHandle *h);
/* Columns of the joints row fb_step_host / fb_step_host_async return: joints_row becomes
 * [n_envs][n_joints][n] with the listed columns (e.g. the four the path writes: position,
 * velocity, torque, limit force; physics.py:481-524 leaves the other 14 zero).  n = 0: all
 * joint_cols columns, the reference's row (default). */
int fb_set_host_joint_columns(FbHandle *h, int n, const int32_t *cols);
/* The same for the links row: links_row becomes [n_envs][n_links][n] with the listed columns of
 * the 20 physics.py:435-466 writes (e.g. CoM position + orientation, 7 columns = 35 % of the
 * bytes, for a host controller that does not read velocities).  n = 0: the full row (default). */
int fb_set_host_link_columns(FbHandle *h, int n, const int32_t *cols);
/* ... and which links: links_row becomes [n_envs][n][columns] with the listed links only (e.g. the
 * head link for a controller that steers by its pose).  n = 0: every link (default). */
int fb_set_host_link_items(FbHandle *h, int n, const int32_t *items);
/* The upload side: `ctrl` of fb_step_host / fb_step_host_async becomes [n_envs][n] and carries the
 * listed actuators only (what step_joints_control_* writes, task.py:309-346: the controlled
 * joints' ctrl entries); the other entries of ctrl keep their device value.  n = 0: all nu. */
int fb_set_host_ctrl_columns(FbHandle *h, int n, const int32_t *cols);
/* Streamed export of whole ring rows of one log kind (0 links, 1 joints, 2 contacts, 3 xfrc) for
 * EVERY environment: rows row0 .. row0+n_rows-1 (ring indices, taken modulo the ring) as dense
 * float32 host memory [n_rows][n_envs][n_items*n_cols] (pinned recommended).  Row r of
 * environment e is the reference's data.sensors.<kind>.array[row] of that environment
 * (task.py:158, simulation.py:198-209 saves exactly these arrays).  Synchronises the step stream
 * first; gathers and device->host copies are double-buffered against each other. */
int fb_export_rows(FbHandle *h, int kind, int row0, int n_rows, float *host);
/* completion of the copies of the latest pipelined call whose index (0, 1, 2, ...) % 2 == slot */
int fb_host_wait_slot(FbHandle *h, int slot);
/* Deeper pipelines (three or more host buffer sets): fb_host_call_count = the index the next
 * call that asks for rows will get; fb_host_wait_call = completion of the copies of that call
 * (copies complete in call order).  Nothing comparable in the reference (its loop is synchronous,
 * simulation.py:149-161). */
long long fb_host_call_count(FbHandle *h);
int fb_host_wait_call(FbHandle *h, long long call);

/* Raw copies between host memory and the engine's device buffers (pointers
 * taken from the views above); for hosts without torch (plain ctypes). */
int fb_copy_to_host(FbHandle *h, const void *dev_ptr, void *host_ptr, int64_t bytes);
int fb_copy_to_device(FbHandle *h, void *dev_ptr, const void *host_ptr, int64_t bytes);

/* Kernel selection.  By default fb_step first runs the environment-per-thread kernel
 * (articulated-body recursion, csrc/fb_fast.h), which advances every environment while
 * no joint limit or contact is active, and then the team kernel (csrc/fb_device.h) on
 * the environments that were handed over.  enable = 0 sends everything to the team
 * kernel (tests compare the two).  fb_fast_path: 0 = team kernel only (disabled or the
 * model is outside the per-thread subset), else environments per block.
 * fb_last_pending: environments the team kernel had to finish in the last fb_step. */
int fb_set_fast_path(FbHandle *h, int enable);
int fb_fast_path(FbHandle *h);
/* Who finishes the environments the per-thread kernel hands over (a joint limit or a plane
 * contact became active): 1 (default) = the per-thread constrained kernel (csrc/fb_fastc.h,
 * matrix-free Newton on the articulated-body recursion), 0 = the team kernel. */
int fb_set_constraint_path(FbHandle *h, int per_thread);
int fb_constraint_path(FbHandle *h);
int fb_fast_smem_bytes_per_env(FbHandle *h);
/* Large-batch (SLIM) layout of the unconstrained per-thread kernel: pose in shared memory,
 * velocities and accumulation slots in the L2 scratch -> 8 instead of 4 warps of environments per
 * SM, in blocks of `enable` = 1 .. 8 warps (2 .. 8: kept in step by a barrier per pass so that
 * they share instruction-cache lines).  fb_create switches it on when the batch has more warps than
 * the regular layout keeps resident (n_envs/32 > 4 x SMs); results are bit-identical to the regular
 * layout.  fb_fast_slim: 0 or the warps per block. */
int fb_set_fast_slim(FbHandle *h, int enable);
/* LEAN variants of the unconstrained kernel: when every joint is a hinge anchored at its body's
 * origin, every inertia axisymmetric, every joint's actuation the unclamped linear form and the
 * joints row the farms layout, fb_step launches a variant with the other paths compiled out (same
 * arithmetic, smaller loops; launches that read a control sequence use the general one).
 * fb_set_fast_lean(h, 0) forces the general variant; fb_fast_lean = 1 when the lean one applies. */
int fb_set_fast_lean(FbHandle *h, int enable);
int fb_fast_lean(FbHandle *h);
/* SPLIT variant of the unconstrained kernel for small batches: the tree of every 32 environments is
 * stepped by several warps (the trunk up to the last branching body on one, the subtrees hanging
 * off it in parallel on the others, two phases per sweep), so that a launch lasts about one trunk +
 * one subtree instead of the whole tree; same per-body arithmetic in the same order along every
 * chain (bit-identical results).  fb_create enables it while the batch leaves schedulers idle;
 * fb_fast_split = warps per 32 environments when it is in use, else 0;
 * fb_fast_split_schedule returns the body lists (n[4], boundary[4] = end of phase A, order[4][64]). */
int fb_set_fast_split(FbHandle *h, int enable);
int fb_fast_split(FbHandle *h);
int fb_fast_split_schedule(FbHandle *h, int32_t *n, int32_t *boundary, uint8_t *order);
int fb_fast_split_blocks_per_sm(FbHandle *h);   /* resident SPLIT blocks per SM (occupancy API), 0 if n/a */
/* SPLIT variant of the CONSTRAINED per-thread kernel (ground-contact batches): the same tree split
 * applied to every sweep of the constrained step (smooth accelerations, the Newton sweeps, the
 * force sweeps); each warp holds the limit rows and collision candidates of its own bodies and the
 * line-search scalars are summed over the warps in a fixed order.  It takes the groups of
 * environments that were ALL handed over before their first step of the launch (a walking batch:
 * every group, every launch) whenever that needs less time by the engine's estimate -- waves of
 * resident blocks x the measured gain per wave; every other group is stepped by the single-warp
 * kernel as before.  Results agree with the single-warp kernel to
 * rounding (the sums are taken in another order), not bit for bit.  fb_con_split = 1 when the
 * next launch uses it. */
int fb_set_con_split(FbHandle *h, int enable);
int fb_con_split(FbHandle *h);
int fb_fast_slim(FbHandle *h);
int fb_last_pending(FbHandle *h, int *count);

/* drag_forces (swimming/drag.pyx:152-268; the operator SwimmingHandler.step calls per swimming link,
 * drag.pyx:389-411) as a stand-alone device operator on n link rows at once, float64 like the
 * reference.  fb_step computes the same forces fused into the step (fp32); this entry point exists
 * for callers that hold link rows of their own.  links [n][20] (the farms links row, SI), coefficients
 * [n][6] (linear x y z, angular x y z), mass / height / density [n] (drag.pyx:353-385), the water
 * surface height, velocity [3] and viscosity, gravity (-9.81 in the reference's call) and the
 * buoyancy flag.  xfrc [n][6] receives force and torque in the CoM frame where the link is at or
 * below the surface and is left untouched where it is above (drag.pyx:192-194); applied [n] says
 * which.  Host pointers; synchronous. */
int fb_drag_forces(int device, int n, const double *links, const double *coefficients, const double *mass,
                   const double *height, const double *density, double surface, const double *water_velocity,
                   double viscosity, double gravity, int use_buoyancy, double *xfrc, int32_t *applied);

/* introspection */
/* Measured FP32 (FFMA, non-tensor) throughput of `device` in TFLOP/s: the denominator bench.py
 * quotes the step kernels' arithmetic against (nothing in the reference; BASELINE.md section 2). */
int fb_measure_fp32_peak(int device, double *tflops_out);
int fb_team_lanes(FbHandle *h);
int fb_smem_bytes_per_env(FbHandle *h);
int fb_device_ptr_stream(FbHandle *h, void **stream_out);

#ifdef __cplusplus
}
#endif
#endif /* FARMS_B200_H_ */
