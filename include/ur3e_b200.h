/* ur3e_b200 -- C ABI of the B200 batched UR3e + Robotiq 2F85 simulator.
 *
 * Drop-in boundary for the reference's hot path  controller -> mj_step x frame_skip -> obs/reward/done.
 * Each entry point names the reference interface it replaces (paths relative to the reference repo).
 *
 * Conventions: every function returns 0 on success or a negative error code (constructors return NULL);
 * ur3e_last_error() gives the thread-local message.  No exceptions cross this boundary.  Pointers named
 * *_dev are device pointers on the batch's CUDA device, owned by the caller (e.g. torch tensors); the
 * library never frees them.  `stream` is a cudaStream_t passed as void* (NULL = legacy default stream);
 * step/reset/get/set are asynchronous on it.  Calls on one batch handle are not thread-safe; different
 * handles are independent.  `dtype`: 0 = float32 (production), 1 = float64 (validation build); all
 * floating-point device buffers of a batch use that element type.
 */
#ifndef UR3E_B200_H
#define UR3E_B200_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef struct ur3e_model ur3e_model;
typedef struct ur3e_batch ur3e_batch;

enum { UR3E_F32 = 0, UR3E_F64 = 1 };
/* object kinds for name lookups: numeric values of mujoco.mjtObj used by utils/utils.py:29-66 */
enum { UR3E_OBJ_BODY = 1, UR3E_OBJ_XBODY = 2 /* body frame (mjOBJ_XBODY); kinematics queries only */, UR3E_OBJ_JOINT = 3, UR3E_OBJ_GEOM = 5, UR3E_OBJ_SITE = 6, UR3E_OBJ_TENDON = 18, UR3E_OBJ_ACTUATOR = 19, UR3E_OBJ_KEY = 23 };
/* controller evaluated inside the step kernel */
enum { UR3E_CTRL_RAW = 0,          /* action = actuator ctrl (imitation_env_direct.py:90) */
       UR3E_CTRL_PD_JOINT = 1,     /* controller_func.py:128-167 pd_joint_ctrl + move_j.py:14-38 */
       UR3E_CTRL_PID_TASK = 2,     /* controller_func.py:68-117 pid_task_ctrl, action = 7-vector trajectory point (move_l_task.py:55-69) */
       UR3E_CTRL_PID_TASK_ENV = 3, /* pid_task_ctrl behind the env action [x,y,z,grip] (ur3e_env2.py:72-82) */
       UR3E_CTRL_PINV = 4          /* controller/move_l.py:15-78: pinv(J) IK + two joint PDs, action = 7-vector trajectory point */ };
enum { UR3E_OBS_STATE = 0, UR3E_OBS_V2 = 1, UR3E_OBS_V0 = 2, UR3E_OBS_DIRECT = 3 };
enum { UR3E_REW_NONE = 0, UR3E_REW_V2 = 1, UR3E_REW_V0 = 2, UR3E_REW_MINUS1 = 3 };
enum { UR3E_TERM_NONE = 0, UR3E_TERM_V2 = 1, UR3E_TERM_V0 = 2 };
enum { UR3E_NOISE_NONE = 0, UR3E_NOISE_LOW = 1, UR3E_NOISE_MED = 2, UR3E_NOISE_HIGH = 3 };   /* gym_utils.py:48-60 */

typedef struct ur3e_model_dims {
  int32_t nq, nv, nu, nbody, njnt, ngeom, nsite, neq, ntendon, npair, nkey;
  double timestep;
} ur3e_model_dims;

/* Environment semantics of a batch (what the four gymnasium env classes + the controller scripts hard-code). */
typedef struct ur3e_env_config {
  int32_t ctrl_mode, obs_kind, reward_kind, term_kind;
  int32_t frame_skip, act_dim, obs_dim, max_steps;
  int32_t reset_key;      /* keyframe index (utils/utils.py:15-24 reset), -1 = qpos0 */
  int32_t reset_noise;    /* UR3E_NOISE_* on the mug x,y (gym_utils.py:63-79) */
  int32_t auto_reset;     /* 1: finished envs are reset inside the step call (SB3 VecEnv semantics) */
  int32_t solver_iterations;   /* Newton iteration cap; 0 = default for dtype */
  double solver_tolerance;     /* scaled-gradient tolerance; 0 = default for dtype */
  double gains[24];       /* PID_TASK*: kp_pos[3] kd_pos[3] kp_rot[3] kd_rot[3]; PD_JOINT: kp[6] kd[6]; PINV: kp_pos[6] kd_pos[6] kp_rot[6] kd_rot[6] */
  double tool_rotvec[3];  /* ur3e_env2.py:74 */
  int64_t env_id_base;    /* global index of env 0 of this batch (multi-GPU sharding: RNG streams are keyed by global id) */
  int32_t single_tier;    /* 1: always step with the full size class (testing aid; default 0 = two-tier stepping where available) */
  int32_t lite_max_contacts, lite_max_rows;   /* lower the lite tier's caps (0 = built-in 8 contacts / 44 rows); the full tier is unaffected */
  int32_t reserved_;
} ur3e_env_config;

const char* ur3e_last_error(void);

/* ---- model: replaces mujoco.MjModel.from_xml_path (utils/utils.py:9-12) and the m.* reads listed in SURVEY 8(b)-2 */
ur3e_model* ur3e_model_load(const char* xml_path);
void ur3e_model_destroy(ur3e_model* m);
int ur3e_model_info(const ur3e_model* m, ur3e_model_dims* out);
/* mujoco.mj_name2id / mj_id2name (utils/utils.py:29-66); -1 / NULL when absent */
int ur3e_model_name2id(const ur3e_model* m, int objtype, const char* name);
const char* ur3e_model_id2name(const ur3e_model* m, int objtype, int id);
/* host view of a model array by its mjModel name (body_mass, jnt_range, actuator_ctrlrange, key_qpos, geom_size, ...);
 * *is_int: 0 float64 / 1 int32; shape has up to 2 entries */
int ur3e_model_array(const ur3e_model* m, const char* field, const void** ptr, int64_t* shape2, int* ndim, int* is_int);
int ur3e_model_num_warnings(const ur3e_model* m);
const char* ur3e_model_warning(const ur3e_model* m, int i);

/* ---- batch: replaces N x (MjData + gymnasium MujocoEnv) behind SubprocVecEnv (train_rl.py:38-44) */
ur3e_batch* ur3e_batch_create(const ur3e_model* m, const ur3e_env_config* cfg, int64_t n_envs, int device, int dtype);
void ur3e_batch_destroy(ur3e_batch* b);
/* MujocoEnv.reset -> reset_model (ur3e_env2.py:101-109): keyframe + noise, forward, obs.  mask_dev: uint8[n_envs] or NULL = all */
int ur3e_batch_reset(ur3e_batch* b, const uint8_t* mask_dev, uint64_t seed, void* obs_out_dev, void* stream);
/* Env.step (ur3e_env2.py:72-99; ur3e_env.py:137-200; imitation_env_*.py step): one launch for all environments.
 * actions_dev [n,act_dim], obs_dev [n,obs_dim], rew_dev [n], term_dev/trunc_dev uint8[n], final_obs_dev [n,obs_dim] or NULL */
int ur3e_batch_step(ur3e_batch* b, const void* actions_dev, void* obs_dev, void* rew_dev, uint8_t* term_dev, uint8_t* trunc_dev, void* final_obs_dev, void* stream);
/* same call with HOST buffers: copies actions in and results out on the batch's stream and synchronises (the e2e path) */
int ur3e_batch_step_host(ur3e_batch* b, const void* actions_host, void* obs_host, void* rew_host, uint8_t* term_host, uint8_t* trunc_host);
/* d.qpos / d.qvel / qacc_warmstart reads and MujocoEnv.set_state + mj_forward (checkpointing, per-step re-seeding in parity tests) */
int ur3e_batch_get_state(ur3e_batch* b, void* qpos_dev, void* qvel_dev, void* qacc_warmstart_dev, void* stream);
int ur3e_batch_set_state(ur3e_batch* b, const void* qpos_dev, const void* qvel_dev, const void* qacc_warmstart_dev, void* stream);
/* d.sensor(name).data of main.xml's logging sensors (assets/main.xml:392-408; readers utils/utils.py:201-245 get_jnt_torques /
 * get_grasp_contact, controller_func.py:191-211): once a buffer [n, UR3E_NSENSOR] of the batch's dtype is attached, every step
 * writes, from the last mj_step of the step, [0..7) actuatorfrc (shoulder_pan .. wrist_3, fingers), [7] touch right_pad1_contact,
 * [8] touch left_pad1_contact, [9..12) d.site("tcp").xpos, [12..21) d.site("tcp").xmat (row-major) as get_task_space_state reads
 * them after mj_step, [21..28) d.ctrl as the in-kernel controller set it (the `u` of pid_task_ctrl that collect_demos.py:139-152
 * records as the "direct" expert action), [28..46) the six <torque> site sensors of assets/main.xml:384-391 (shoulder_pan .. wrist_3,
 * 3 values each: interaction torque between the link and its parent at the site, in the site frame).  NULL detaches (the default: no cost on the step path). */
#define UR3E_NSENSOR 46
int ur3e_batch_set_sensor_buffer(ur3e_batch* b, void* sensors_dev);
/* episode statistics + solver counters since the last reset of the counters: 16 doubles (see UR3E_STAT_*) summed over the batch */
int ur3e_batch_stats(ur3e_batch* b, double* stats16_dev, int reset_counters, void* stream);
enum { UR3E_STAT_EPISODES = 0, UR3E_STAT_RETURN, UR3E_STAT_LENGTH, UR3E_STAT_SUCCESS, UR3E_STAT_TERM_REACH, UR3E_STAT_TERM_TOPPLE,
       UR3E_STAT_TERM_COLLISION, UR3E_STAT_TRUNC, UR3E_STAT_UNSTABLE, UR3E_STAT_NEFC, UR3E_STAT_NCON, UR3E_STAT_ITER, UR3E_STAT_SUBSTEPS, UR3E_STAT_OVERFLOW,
       UR3E_STAT_PAD_CONTACT_STEPS /* env-steps that ended with >= 1 gripper-pad / mug contact */, UR3E_STAT_STEPS /* env-steps */ };
/* kernels launched by this batch so far; bytes of shared memory per environment; environments resident per SM */
int64_t ur3e_batch_launch_count(const ur3e_batch* b);
int ur3e_batch_kernel_info(const ur3e_batch* b, int32_t* arena_bytes, int32_t* warps_per_block, int32_t* blocks_per_sm, int32_t* regs_per_thread);
/* tiered stepping of the float32 main.xml batch (DESIGN.md section 3): out8 = lite arena bytes, lite warps/block, lite blocks/SM,
 * lite registers, two-tier steps, full-only steps (single_tier), environments the full tier stepped at the last observed step, 0; all zero
 * when the batch has a single size class.  Which tier steps an environment is decided per environment on the device (its own
 * recent contact / row counts), so trajectories do not depend on the batch size, the world size or host timing. */
int ur3e_batch_tier_info(const ur3e_batch* b, int64_t* out8);
/* the grasp tier of the float32 main.xml batch (16 contacts / 68 rows, between the lite and the generic size class): shared memory per
 * environment, warps per block, registers per thread; zeros when the batch has none */
int ur3e_batch_mid_tier_info(const ur3e_batch* b, int32_t* arena_bytes, int32_t* warps_per_block, int32_t* regs_per_thread);
/* Measurement aid (bench.py's roofline): while enabled, every step-kernel launch is bracketed by a cudaEvent pair on the launching
 * stream.  ur3e_batch_kernel_times synchronises and returns three {kernel ms, launches} pairs accumulated since the timing was enabled:
 * the lite tier, the grasp / generic tier on the caller's stream (these two are the step's critical path; a batch with one size class
 * reports it here), and the generic tier's launches on the side stream (they overlap the grasp tier). */
int ur3e_batch_kernel_timing(ur3e_batch* b, int enable);
int ur3e_batch_kernel_times(ur3e_batch* b, double* out6);
/* bytes of the persistent per-environment record in HBM (read + written once per step) */
int ur3e_batch_state_bytes(const ur3e_batch* b);
/* Kinematics queries: d.xpos/xmat, d.xipos/ximat, d.geom_xpos/xmat, d.site_xpos/xmat and mj_objectVelocity (utils/utils.py:129-189,
 * utils/gym_utils.py:20-39,207-219) for k objects of every environment.
 * ur3e_batch_query_create compiles k (objtype, id) pairs of the loaded model, 1 <= k <= 256, objtype one of UR3E_OBJ_BODY (inertial
 * frame: xipos / ximat), UR3E_OBJ_XBODY (body frame: xpos / xmat, what d.body(name).xpos returns), UR3E_OBJ_GEOM, UR3E_OBJ_SITE
 * (ids as ur3e_model_name2id returns them); it returns the query's id (>= 0).  The batch owns its queries until ur3e_batch_destroy.
 * ur3e_batch_query writes, for every environment, pos_dev [n, k, 3], mat_dev [n, k, 9] (row-major) and vel_dev [n, k, 6]
 * ([rot(3), lin(3)] as mj_objectVelocity; flg_local = 1: in the object's frame) in the batch's dtype; any of them may be NULL, not
 * all.  Asynchronous on `stream`, one kernel launch; the stored state is not modified.
 * Semantics: the values are evaluated at the STORED state, i.e. what MuJoCo's arrays hold after set_state / reset + mj_forward.
 * After a step, MuJoCo's arrays still hold the last substep's pre-integration kinematics (SURVEY F9); the query is one substep
 * newer than those (the tcp pose of that stale kind is in the sensor record). */
int ur3e_batch_query_create(ur3e_batch* b, const int32_t* objtype, const int32_t* objid, int32_t k);
int ur3e_batch_query(ur3e_batch* b, int query_id, void* pos_dev, void* mat_dev, void* vel_dev, int flg_local, void* stream);
/* mj_jacSite / mj_jacBody / mj_jacBodyCom / mj_jacGeom for the k objects of a kinematics query, plus mj_fullM and d.qfrc_bias,
 * for every environment, at the stored state.  jacp_dev, jacr_dev [n, k, 3, nv]; M_dev [n, nv, nv]; qfrc_bias_dev [n, nv]; batch dtype.
 * query_id = -1: no objects (jacp_dev and jacr_dev must be NULL).  Any output may be NULL, not all.  One launch, asynchronous.
 * The Jacobian of an object is taken at its world point: the site (UR3E_OBJ_SITE, mj_jacSite), the body frame's origin
 * (UR3E_OBJ_XBODY, mj_jacBody), the body's centre of mass (UR3E_OBJ_BODY, mj_jacBodyCom) or the geom (UR3E_OBJ_GEOM, mj_jacGeom);
 * jacp and jacr are MuJoCo's row-major (3, nv) per object.  M is dense and symmetric, armature included.  The stored state is not
 * modified.
 * Semantics: the values are evaluated at the STORED state, i.e. what MuJoCo's arrays hold after set_state / reset + mj_forward.
 * After a step, MuJoCo's d.qfrc_bias and the Jacobian it would compute are the last substep's pre-integration values (SURVEY F9),
 * and so is the cache the fused task-space controllers read; this call is one substep newer than those. */
int ur3e_batch_query_jac(ur3e_batch* b, int query_id, void* jacp_dev, void* jacr_dev, void* M_dev, void* qfrc_bias_dev, void* stream);
/* Forward-dynamics queries: d.ncon, d.contact[k].geom1/geom2/dist/pos/frame, mj_contactForce, d.qacc, d.qfrc_constraint and
 * d.sensordata for every environment (the contact reads of utils/gym_utils.py:98-201 get_robust_block_grasp_state,
 * get_block_grasp_state, get_self_collision, get_table_collision; the sensor reads of utils/utils.py:201-245).
 * C = ur3e_batch_max_contacts(b): contacts stored per environment, the step's largest cap (24 for main.xml, 12 for ur3e_2f85.xml, 0
 * for a model without contact pairs).  Device outputs, any may be NULL, not all; float ones in the batch's dtype:
 *   qacc, qfrc_constraint [n, nv]
 *   info [n, 4] int32: ncon, nefc, solver iterations, overflow bits (1: more contacts / narrow-phase candidates than the caps,
 *        2: more constraint rows than the cap; the bits the step sets)
 *   contact_geom [n, C, 2] int32: geom1, geom2 (ids of the loaded model); contact_dist [n, C]; contact_pos [n, C, 3];
 *   contact_frame [n, C, 9]: MuJoCo's mjContact fields; row 0 of the frame is the normal, from geom1 to geom2
 *   contact_force [n, C, 6]: mj_contactForce in the contact frame, [fn, ft1, ft2, 0, 0, 0] (elliptic cones, condim 3); a contact
 *        without constraint rows (row overflow) reports 0
 *   flags [n] int32: 1 mug - left pad, 2 mug - right pad, 4 gripper - table, 8 self-collision (gym_utils.py:108-201), over all
 *        ncon contacts (the list MuJoCo's d.contact holds); on a row overflow the step's own bits see only the contacts with rows
 *   sensordata [n, 46]: the layout of the step's sensor record (ur3e_batch_set_sensor_buffer)
 * Entries past ncon are written as geom -1 and zeros.  Contacts are in pair-list order (the candidate pairs of the model that survive
 * the static pruning), then in the narrow phase's point order within a pair.
 * ctrl_dev: contiguous [n, nu] (batch dtype; environment e at ctrl_dev + e * nu) or NULL (zero ctrl), the actuation the dynamics see.  When no output needs dynamics (qacc,
 * qfrc_constraint, contact_force, sensordata) only kinematics and collision run: info then reports nefc = 0 and 0 iterations.
 * Rejected: out NULL, every output NULL, a contact_* output when C = 0.  Asynchronous on `stream`, one kernel launch; the stored
 * state is not modified.
 * Semantics: the values are mj_forward's at the STORED state (qpos, qvel and the solver's warm start) with this ctrl, i.e. MuJoCo's
 * d.contact / d.efc_force / d.qacc / d.sensordata after set_state / reset + mj_forward.  After a step, MuJoCo's d.contact still holds
 * the contacts of the last substep before integration (SURVEY F9); this call is one substep newer, the state ur3e_batch_query sees. */
typedef struct ur3e_forward_out {
  void* qacc; void* qfrc_constraint; int32_t* info;
  int32_t* contact_geom; void* contact_dist; void* contact_pos; void* contact_frame; void* contact_force;
  int32_t* flags; void* sensordata;
} ur3e_forward_out;
int ur3e_batch_max_contacts(const ur3e_batch* b);
int ur3e_batch_forward(ur3e_batch* b, const void* ctrl_dev, const ur3e_forward_out* out, void* stream);
/* Inverse dynamics (mj_inverse): the generalised force that produces a given acceleration at a given state, and the constraint and
 * contact forces the soft-constraint model implies at that acceleration.  For feedforward torques of planned motions, inverse-dynamics
 * labels along recorded trajectories and the residual of the forward solver (MuJoCo's mjENBL_FWDINV).
 * State, exactly one source:
 *   qpos_dev and qvel_dev both NULL: the STORED state of the batch's n environments (m must equal n).  As for ur3e_batch_forward,
 *     after a step this is one substep newer than MuJoCo's stale arrays (SURVEY F9).
 *   qpos_dev [m, nq], qvel_dev [m, nv] (batch dtype): m >= 1 given states, independent of n (a [T, m'] trajectory of
 *     ur3e_batch_rollout flattens into one call).  No record is read or written.
 * qacc_dev [m, nv] (batch dtype).  With discrete = 0 it is the continuous acceleration a (MuJoCo's default).  With discrete != 0
 * (mjENBL_INVDISCRETE, mj_discreteAcc) it is the acceleration the Euler step applied, (qvel_next - qvel) / timestep of one mj_step,
 * and a = M^-1 (M + timestep diag(dof_damping)) qacc, the exact inverse of the step's implicit damping; a model without damping has
 * a = qacc.  With frame_skip > 1 one env-step is frame_skip mj_steps: the discrete convention applies per mj_step (substep), not per
 * env-step.
 * Computed, at (qpos, qvel) and a, with no solver iterations and no warm start (ctrl plays no part):
 *   jar = J a - aref;  efc_force = the constraint law at jar (elliptic cones, friction loss, limits: mj_invConstraint);
 *   qfrc_constraint = J^T efc_force;
 *   qfrc_inverse = M a + qfrc_bias - qfrc_passive - qfrc_constraint,  qfrc_passive = -dof_damping qvel - stiffness (q - springref).
 * qfrc_inverse excludes actuation: at a = forward's qacc it equals qfrc_actuator up to the forward solver's residual.  Sensors are not
 * evaluated.
 * Device outputs, any may be NULL, not all; float ones in the batch's dtype; C = ur3e_batch_max_contacts(b):
 *   qfrc_inverse, qfrc_constraint [m, nv]
 *   info [m, 3] int32: ncon, nefc, overflow bits (1 contacts, 2 constraint rows; the bits the step sets)
 *   contact_geom [m, C, 2] int32 and contact_force [m, C, 6]: ur3e_batch_forward's conventions (geom -1 and zeros past ncon;
 *        mj_contactForce [fn, ft1, ft2, 0, 0, 0] in the contact frame at the given acceleration, 0 for a contact without rows)
 * Rejected: qpos_dev without qvel_dev or the reverse, m < 1 or m > 2^31 - 1, m != n for the stored state, qacc_dev NULL, out NULL,
 * every output NULL, a contact output when C = 0.  Asynchronous on `stream`, one kernel launch; no record is modified. */
typedef struct ur3e_inverse_out {
  void* qfrc_inverse; void* qfrc_constraint; int32_t* info; int32_t* contact_geom; void* contact_force;
} ur3e_inverse_out;
int ur3e_batch_inverse(ur3e_batch* b, const void* qpos_dev, const void* qvel_dev, int64_t m, const void* qacc_dev, int32_t discrete,
                       const ur3e_inverse_out* out, void* stream);
/* Offscreen rendering: rgb_array / depth_array images (gymnasium MujocoEnv.render, ur3e_env2.py:25-28) and geom segmentation for
 * selected environments, from a camera anchored to the world or to one object of the loaded model.
 * ur3e_batch_render_create compiles a renderer and returns its id (>= 0); the batch owns it until ur3e_batch_destroy.
 *   cam: anchor objtype -1 = world, UR3E_OBJ_XBODY (body frame) or UR3E_OBJ_SITE with a loaded-model id; pos and xyaxes (MJCF
 *        <camera xyaxes>: x right, y up, the view along -z) in the anchor frame; fovy the vertical field of view in degrees
 *        (0, 180); 0 < znear < zfar in metres.  The aspect ratio is width / height.
 *   geom_ids [k], 1 <= k <= 256: the geoms drawn (box or plane, ids of the loaded model); rgba [k, 4] or NULL = the model's geom_rgba.
 *   width, height in [1, 2048].
 * Scene: all geoms opaque, no shadows, textures, reflections or anti-aliasing.  A plane with size (sx, sy) is |x| <= sx, |y| <= sy
 * of its frame (0 = unbounded) and is seen only from its front (+z) side; boxes are solid, seen from outside.  Shading is a
 * headlight, c = rgb * (0.3 + 0.7 * max(0, -n . d)) with d the unit ray, stored as the nearest uint8 of 255 * clamp(c, 0, 1);
 * the background is black.  One ray per pixel centre, row 0 at the top.
 * ur3e_batch_render renders m environments: env_ids_dev int32 [m] (device) or NULL = all (then m = n).  Outputs, any may be NULL,
 * not all: rgb_dev uint8 [m, H, W, 3]; depth_dev [m, H, W] in the batch's dtype, z-depth in metres along the camera's view axis
 * (what gymnasium's linearised depth_array returns, not the ray length), zfar for a miss or a hit beyond zfar, hits nearer than znear
 * ignored; seg_dev int32 [m, H, W], the hit geom's id, -1 for background.  Equal hit distances go to the lower geom id.  An id
 * outside [0, n) renders as background.  Asynchronous on `stream`, two kernel launches; the stored state is not modified.  The
 * pose scratch is shared by a batch's renderers: calls on different streams must be ordered by the caller.
 * Semantics: the images are of the STORED state, i.e. what MuJoCo's d.geom_xpos / d.geom_xmat hold after set_state / reset +
 * mj_forward.  After a step, MuJoCo's arrays still hold the last substep's pre-integration kinematics (SURVEY F9); the image is one
 * substep newer than those, the state ur3e_batch_query sees. */
typedef struct ur3e_camera {
  int32_t objtype, objid;   /* anchor: objtype -1 = world, else UR3E_OBJ_XBODY or UR3E_OBJ_SITE with a loaded-model id */
  double pos[3], xyaxes[6]; /* in the anchor frame; view along -z */
  double fovy, znear, zfar; /* degrees, metres */
} ur3e_camera;
int ur3e_batch_render_create(ur3e_batch* b, const ur3e_camera* cam, const int32_t* geom_ids, int32_t k, const float* rgba, int32_t width, int32_t height);
int ur3e_batch_render(ur3e_batch* b, int render_id, const int32_t* env_ids_dev, int64_t m, uint8_t* rgb_dev, void* depth_dev, int32_t* seg_dev, void* stream);
/* Rollouts (mujoco.rollout): m independent copies of environments of the batch, each stepped T env-steps with the given actions,
 * with every step's outputs; the batch itself is left untouched.  For lookahead: sampling-based MPC (predictive sampling, MPPI,
 * CEM), lookahead rewards, "what if" evaluation.
 * Source, exactly one of:
 *   src_env_ids_dev int32 [m]: rollout j starts from a copy of environment src[j]'s whole record (state, solver warm start, the
 *     controller's stale-kinematics cache, episode step counter t and tier word), so that its steps are bit-identical to what
 *     ur3e_batch_step would do to environment src[j] with the same actions, up to its first done.  Ids may repeat and m may exceed
 *     n (K branches per environment).  An id outside [0, n) starts from a bad (NaN) state, which the step's own guard
 *     (mj_checkPos/Vel) resets to qpos0 at the first substep; info[j, 0] >= 1 reports it.
 *   qpos0_dev [m, nq], qvel0_dev [m, nv] and optionally qacc_warmstart0_dev [m, nv] (NULL = zero): rollout j starts as
 *     ur3e_batch_set_state leaves a fresh record (forward pass, fresh cache, t = 0, tier 0).
 * Dynamics: T env-steps of the batch's own environment (controller, frame_skip, observation, reward, termination, truncation); a
 * UR3E_CTRL_RAW batch with frame_skip 1 gives mujoco.rollout's semantics.  There is no auto-reset: after a done the rollout keeps
 * stepping and the flags are whatever the environment computes (v2 keeps reporting truncated once t >= max_steps); callers mask the
 * steps after the first done.
 * actions_dev [T, m, act_dim] (batch dtype).  Outputs, time-major (step t's outputs are the contiguous [m, ...] slice t; transpose
 * the first two axes for mujoco.rollout's [nroll, nstep, ...]), device pointers, any may be NULL, not all:
 *   qpos [T, m, nq], qvel [T, m, nv]: the state after each env-step; obs [T, m, obs_dim], reward [T, m], terminated / truncated
 *   uint8 [T, m]: what ur3e_batch_step returns; sensordata [T, m, UR3E_NSENSOR]: the step's logging record (ur3e_batch_set_sensor_buffer)
 *   from each env-step's last mj_step; info int32 [m, 2]: env-steps with a bad-state reset (mj_checkPos/Vel/Acc), env-steps with an
 *   overflow of the contact / row caps.
 * Rejected: m < 1 or m > 2^31 - 1, T < 1, actions NULL, both sources or neither, qpos0 without qvel0 or the reverse, a warm start
 * without qpos0, out NULL, every output NULL.
 * Asynchronous on `stream`: T tiered steps (the kernels of ur3e_batch_step) on a scratch copy.  The batch's records, statistics,
 * attached sensor buffer and ur3e_batch_tier_info's counts are not modified (only the launch count grows); like the queries, the call
 * does not become the stream ur3e_batch_step_host orders itself after.  A batch's rollouts share one workspace (grown to the largest
 * m seen): calls on different streams must be ordered by the caller. */
typedef struct ur3e_rollout_out {
  void* qpos; void* qvel; void* obs; void* reward;
  uint8_t* terminated; uint8_t* truncated;
  void* sensordata; int32_t* info;
} ur3e_rollout_out;
int ur3e_batch_rollout(ur3e_batch* b, const int32_t* src_env_ids_dev, const void* qpos0_dev, const void* qvel0_dev, const void* qacc_warmstart0_dev,
                       int64_t m, int32_t T, const void* actions_dev, const ur3e_rollout_out* out, void* stream);
/* Inverse kinematics (dm_control.utils.inverse_kinematics.qpos_from_site_pose, batched): the joint positions that put one object at a
 * target position and / or orientation.  For reset and goal distributions at sampled tool poses, task-space waypoints converted into
 * joint waypoints for UR3E_CTRL_PD_JOINT, and reachability checks.
 * ur3e_batch_ik_create compiles a problem family and returns its id (>= 0); the batch owns it until ur3e_batch_destroy:
 *   objtype / objid: one object of the kinds ur3e_batch_query_create accepts (UR3E_OBJ_SITE, UR3E_OBJ_XBODY, UR3E_OBJ_BODY,
 *     UR3E_OBJ_GEOM); its world point p(q) and frame R(q) are what a kinematics query returns for it.
 *   joint_ids [nj], 1 <= nj <= nv: distinct hinge or slide joints of the loaded model, the only qpos entries the solve changes.
 * ur3e_batch_ik solves m problems, one warp each.  Start configuration q (all nq entries), exactly one source:
 *   env_ids_dev int32 [m]: the stored qpos of those environments (ids may repeat; an id outside [0, n) gives NaN qpos and err_norm
 *     and status 3);  qpos0_dev [m, nq] (batch dtype): given configurations;  neither: every environment's stored qpos (m = n).
 * Targets (batch dtype, at least one): target_pos_dev [m, 3] world position p*; target_quat_dev [m, 4] world orientation q*
 * (w, x, y, z; normalised first, a zero quaternion is the identity).  For step = 0 .. max_steps - 1:
 *   kinematics at q;  e_pos = p* - p,  e_rot = the rotation vector of R(q*) R(q)^T (world frame);
 *   err_norm = |e_pos| + rot_weight |e_rot| (dm_control's sum of norms);  err_norm < tol: converged (status 0);
 *   J = the r x nj block of [jacp; jacr] at the object's point for the joints' dofs, r = 3 or 6 (rows for the targets given);
 *   lambda = regularization_strength if err_norm > regularization_threshold, else 0;  dq = (J^T J + lambda I)^-1 J^T e, solved as
 *     J^T (J J^T + lambda I)^-1 e when r <= nj (the smaller SPD system, at most 6 x 6); with lambda = 0 a pivot below 1e-13
 *     (float64) / 1e-5 (float32) of the system's largest diagonal entry contributes zero, so dq is the minimum-norm least-squares
 *     step except at exact singularities;
 *   err_norm / |dq| > progress_thresh: insufficient progress (status 2), dq not applied;
 *   dq scaled down to max_update_norm; added to the joints' qpos; every limited joint clamped to its jnt_range.
 * max_steps updates applied without convergence: status 1.
 * Differences from dm_control: the limit clamp (runs whose iterates stay inside the limits are dm_control's); err_norm and steps
 * describe the returned qpos (its error, updates applied; converged means it is within tol); any kinematics-query object, not
 * only sites; with lambda = 0 the minimum-norm step (dm_control's lstsq(J^T J, J^T e, rcond=-1) keeps rounding-noise directions
 * of J^T J when r < nj).  Only the selected joints' qpos entries change (all others are copied bit for bit); equality constraints
 * (the 2F85's four-bar) and contacts are not considered.
 * opt: NULL = the defaults, dm_control's: tol 1e-14 (float64) / 1e-5 (float32), rot_weight 1, regularization_threshold 0.1,
 * regularization_strength 3e-2, max_update_norm 2, progress_thresh 20, max_steps 100.  The float32 tol sits above the float32 noise
 * floor of err_norm (DESIGN §3).
 * Outputs (device, any may be NULL, not all): qpos [m, nq] (batch dtype), err_norm [m] (batch dtype), info int32 [m, 2] = steps,
 * status.
 * Rejected: an unknown id, m < 1 or m > 2^31 - 1, both env_ids_dev and qpos0_dev, m != n when neither is given, no target, out NULL,
 * every output NULL, tol / rot_weight / regularization_threshold / regularization_strength < 0 or NaN, max_update_norm or progress_thresh
 * not > 0, max_steps outside [1, 10000].
 * Asynchronous on `stream`, one kernel launch; no record is read beyond qpos and none is written (like the queries, the call does not
 * become the stream ur3e_batch_step_host orders itself after). */
typedef struct ur3e_ik_options {
  double tol, rot_weight, regularization_threshold, regularization_strength, max_update_norm, progress_thresh;
  int32_t max_steps, reserved_;
} ur3e_ik_options;
typedef struct ur3e_ik_out { void* qpos; void* err_norm; int32_t* info; } ur3e_ik_out;
int ur3e_batch_ik_create(ur3e_batch* b, int32_t objtype, int32_t objid, const int32_t* joint_ids, int32_t nj);
int ur3e_batch_ik(ur3e_batch* b, int ik_id, const int32_t* env_ids_dev, const void* qpos0_dev, int64_t m, const void* target_pos_dev,
                  const void* target_quat_dev, const ur3e_ik_options* opt, const ur3e_ik_out* out, void* stream);
/* Geom distances (mj_geomDistance(m, d, geom1, geom2, distmax, fromto), batched over k pairs and m states): the signed distance and
 * the closest points of box and plane geoms.  For clearance checks of IK solutions, reset samples or waypoints at given
 * configurations, collision-avoidance costs along rollout trajectories, and graded (signed) versions of contact predicates.
 * ur3e_batch_distance_create compiles a pair set and returns its id (>= 0); the batch owns it until ur3e_batch_destroy:
 *   geom1 [k], geom2 [k], 1 <= k <= 256: box or plane geoms of the loaded model (contype / conaffinity and the candidate list play no
 *     part); a geom paired with itself and a plane paired with a plane are rejected.
 * ur3e_batch_distance evaluates the k pairs at m states, one warp each.  Configuration q (all nq entries), exactly one source:
 *   env_ids_dev int32 [m]: the stored qpos of those environments (ids may repeat; an id outside [0, n) gives NaN dist and fromto);
 *   qpos_dev [m, nq] (batch dtype): given configurations;  neither: every environment's stored qpos (m = n).
 * Per pair, at the geoms' world poses of q:
 *   box-box, disjoint (a SAT axis separates): dist = the exact Euclidean distance of the two solids, fromto its closest points;
 *   box-box, overlapping: dist < 0 is the smallest dist of the collider's box-box contacts at margin 0 (for a pair of the step's
 *     candidate list, the deepest contact the step and ur3e_batch_forward see), fromto = pos -/+ dist/2 normal;
 *   plane-box: the plane is an infinite half-space (as in the step's collision); dist = the smallest signed height of the box's 8
 *     vertices over it, fromto = that vertex projected onto the plane and the vertex.
 *   fromto[0:3] lies on geom1 and fromto[3:6] on geom2 (swapping a pair swaps the halves).  When no pair of points is closer than
 *   distmax (dist >= distmax), dist = distmax and fromto = 0.
 * Outputs (device, batch dtype, either may be NULL, not both): dist [m, k], fromto [m, k, 6].
 * Rejected: an unknown id, m < 1 or m > 2^31 - 1, both env_ids_dev and qpos_dev, m != n when neither is given, both outputs NULL,
 * distmax NaN.  Asynchronous on `stream`, one kernel launch; no record is read beyond qpos and none is written. */
int ur3e_batch_distance_create(ur3e_batch* b, const int32_t* geom1, const int32_t* geom2, int32_t k);
int ur3e_batch_distance(ur3e_batch* b, int distance_id, const int32_t* env_ids_dev, const void* qpos_dev, int64_t m, double distmax, void* dist_dev,
                        void* fromto_dev, void* stream);

#ifdef __cplusplus
}
#endif
#endif
