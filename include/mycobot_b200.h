/*
 * mycobot_b200.h -- C ABI of the B200-native batched myCobot physics-and-task engine.
 *
 * Drop-in boundary for the hot path of matinmoezzi/MyCobotGym (SURVEY.md section 8b):
 * every entry point replaces a piece of the reference's per-env Python/MuJoCo path and is
 * what a ctypes / cffi binding on the reference side would bind (INTEGRATION.md).
 *
 * Conventions
 *   - extern "C", plain pointers and sizes, no torch / C++ types in signatures.
 *   - every function returns 0 on success, <0 on error; mcb_last_error() gives the text
 *     (thread-local).  No exceptions cross the ABI.
 *   - all array arguments of the non-`_host` functions are CALLER-OWNED DEVICE pointers
 *     (e.g. torch `data_ptr()`), row-major, env-major.  `stream` is a cudaStream_t passed as
 *     void* (NULL = legacy default stream); all work is enqueued on it, nothing synchronises.
 *   - the library owns only the opaque mcb_model / mcb_batch handles.
 *   - a batch is not thread-safe; one batch per process per GPU is the intended use.
 *
 * Fixed topology: the myCobot 280 joint-variant model (mycobot280.xml) reduced to its 13
 * jointed bodies (fixed children merged by the host-side loader, mycobotgym_b200/flatten.py).
 */
#ifndef MYCOBOT_B200_H_
#define MYCOBOT_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MCB_NB 13     /* jointed bodies: link1..6, rgear, rfinger, lgear, lfinger, rhinge, lhinge, object0 */
#define MCB_NV 18     /* dofs (12 hinges + free cube) */
#define MCB_NQ 19
#define MCB_NU 7
#define MCB_NHINGE 12
#define MCB_NGEOM 5   /* plane, table box, right/left finger-layer boxes, cube box */
#define MCB_MAXPAIR 12
#define MCB_MAXHULL 16   /* convex hulls of the mesh geoms (14 in the myCobot model; base_link.STL is absent from the reference) */
#define MCB_MAXHPAIR 192 /* candidate pairs hull x {hull, box, plane} after MuJoCo's static filters */
#define MCB_OBS_OBJECT 25
#define MCB_OBS_REACH 10
#define MCB_STATE_STRIDE 80 /* doubles per env in the resident state record: qpos19 qvel18 ctrl7 warm18 goal3 qprev6 mocap7 pad2 */

/* Per-env physics parameters: MCB_NPARAM multipliers of fields of the model in use (nominal value 1.0). */
#define MCB_NPARAM 14
#define MCB_P_CUBE_MASS 0    /* mass[12] and the six inertia[12] entries of the cube */
#define MCB_P_FRICTION 1     /* 1..5: sliding friction geom_friction[g][0] of the MCB_NGEOM primitive geoms, g in mcb_model_desc order */
#define MCB_P_GAIN 6         /* 6..12: actuator u: act_gain[u], act_bias[u][1] and act_bias[u][2] (the servo's kp and kv); mocap variant: u = 0 only */
#define MCB_P_ARM_DAMPING 13 /* damping[0..5], in the passive force and in Euler's implicit term */

/* Contact output (mcb_set_contact_output): contact slots per env, and doubles per slot: dist, pos[3], frame[9], force[6]. */
#define MCB_MAXCON 24
#define MCB_CONTACT_DOUBLES 19

/* Flattened, reduced model (host memory; copied to the device by mcb_model_create).
 * Replaces the compiled mjModel the reference builds in MujocoEnv.__init__ (mycobot.py:69-75). */
typedef struct mcb_model_desc {
  /* kinematic tree of jointed bodies, depth-first order == dof order */
  int32_t parent[MCB_NB];        /* jointed parent body or -1 */
  int32_t level[MCB_NB];         /* depth in the jointed tree */
  int32_t subtree_size[MCB_NB];  /* bodies in the subtree rooted here (contiguous in DFS order) */
  int32_t dof_body[MCB_NV];
  uint32_t ancmask[MCB_NB];      /* bit j set: dof j moves this body */
  double Tpos[MCB_NB][3];        /* parent-frame offset of the body frame (through merged fixed bodies) */
  double Tmat[MCB_NB][9];        /* parent-frame orientation of the body frame at q = 0 */
  double axis[MCB_NB][3];        /* hinge axis in the body frame (unused for the free body) */
  double mass[MCB_NB];           /* composite (body + merged fixed children) */
  double ipos[MCB_NB][3];        /* composite centre of mass, body frame */
  double inertia[MCB_NB][6];     /* composite inertia about ipos, body axes: xx yy zz xy xz yz */
  double armature[MCB_NV];
  double damping[MCB_NV];
  double dof_invweight0[MCB_NV];
  double ref_robot[3];           /* world point the robot tree's spatial quantities refer to */
  double qpos0[MCB_NQ];
  /* joint limits (hinges only) */
  int32_t jnt_limited[MCB_NHINGE];
  double jnt_range[MCB_NHINGE][2];
  double jnt_solref[MCB_NHINGE][2];
  double jnt_solimp[MCB_NHINGE][5];
  /* equality: two connects (four-bar closure) + one joint coupling */
  int32_t con_body1[2], con_body2[2];
  double con_anchor1[2][3], con_anchor2[2][3];
  double con_diag[2];            /* body_invweight0 translational sum */
  double con_solref[2][2], con_solimp[2][5];
  int32_t jeq_dof1, jeq_dof2;
  double jeq_polycoef[5];
  double jeq_diag;
  double jeq_solref[2], jeq_solimp[5];
  /* collision geoms (primitives) */
  int32_t geom_type[MCB_NGEOM];  /* 0 plane, 6 box (MuJoCo mjtGeom values) */
  int32_t geom_body[MCB_NGEOM];  /* jointed body index or -1 (static) */
  int32_t geom_condim[MCB_NGEOM];
  double geom_pos[MCB_NGEOM][3]; /* in geom_body frame (world if static) */
  double geom_mat[MCB_NGEOM][9];
  double geom_size[MCB_NGEOM][3];
  double geom_rbound[MCB_NGEOM];
  double geom_friction[MCB_NGEOM][3];
  double geom_solref[MCB_NGEOM][2];
  double geom_solimp[MCB_NGEOM][5];
  double geom_solmix[MCB_NGEOM];
  double geom_invweight[MCB_NGEOM][2]; /* body_invweight0 (translational, rotational) of the geom's body */
  int32_t npair;
  int32_t pair_g1[MCB_MAXPAIR], pair_g2[MCB_MAXPAIR]; /* statically filtered candidate pairs, type1<=type2 */
  /* sites used by the task layer */
  int32_t eef_body;
  double eef_pos[3];
  int32_t obj_body;
  /* staged reward (mycobot.py:402-448): finger-layer / object geoms, target0 site (XML default: only render() moves it, mycobot.py:309-311) */
  int32_t geom_finger_r, geom_finger_l, geom_object;
  double target0_pos[3];
  /* actuators: general, no dynamics, fixed gain, affine bias */
  double act_moment[MCB_NU][MCB_NV];
  double act_gain[MCB_NU];
  double act_bias[MCB_NU][3];
  double act_ctrlrange[MCB_NU][2];
  double act_forcerange[MCB_NU][2];
  int32_t act_ctrllimited[MCB_NU];
  int32_t act_forcelimited[MCB_NU];
  /* options (mycobot280_main.xml:3-5 + MuJoCo defaults) */
  double timestep, gravity[3], tolerance, ls_tolerance, meaninertia, impratio;
  int32_t iterations, ls_iterations;
  /* task constants captured by _env_setup (mycobot.py:450-481) */
  double initial_gripper_xpos[3];
  double height_offset;
  double init_qpos[MCB_NQ];
  double init_ctrl[MCB_NU];
  /* the same four for fetch envs, which start from keyframe 0 (mycobot.py:451-452, mycobot280.xml:4-9) */
  double key_initial_gripper_xpos[3];
  double key_height_offset;
  double key_qpos[MCB_NQ];
  double key_ctrl[MCB_NU];
  /* mocap variant (mycobot280_mocap.xml): one mocap body welded to gripper_tcp (mocap.xml:16-20); nu = 1 there */
  int32_t nu;                    /* actuators in use: 7 (joint variant) or 1 (mocap variant: the finger actuator) */
  int32_t has_weld;
  int32_t weld_body2;            /* jointed body carrying gripper_tcp */
  int32_t reserved0_;
  double Tquat[MCB_NB][4];       /* Tmat as a quaternion (body orientation chain for the weld's orientation error) */
  double weld_anchor1[3];        /* anchor in the mocap body's frame (eq_data[3:6]) */
  double weld_anchor2[3];        /* anchor in weld_body2's frame (gripper_tcp offset + eq_data[0:3]) */
  double weld_relquat[4];        /* orientation of body2 relative to the mocap body at qpos0 (eq_data[6:10]) */
  double weld_torquescale;
  double weld_diag[2];           /* body_invweight0 sums: translational, rotational */
  double weld_solref[2], weld_solimp[5];
  double mocap_pos0[3], mocap_quat0[4];       /* mocap pose from the XML (mocap.xml:3) */
  double key_mocap_pos[3], key_mocap_quat[4]; /* ... and from keyframe 0 for fetch envs (mycobot280_mocap.xml:8-9) */
} mcb_model_desc;

/* Task configuration == the reference constructor kwargs (mycobot.py:30-46) + TimeLimit (__init__.py:34). */
typedef struct mcb_task_cfg {
  int32_t has_object;          /* mycobot.py:33 */
  int32_t block_gripper;       /* mycobot.py:34 */
  int32_t target_in_the_air;   /* mycobot.py:38 */
  int32_t reward_type;         /* 0 sparse (float32 out), 1 dense (float64 out), 2 reward_shaping (float64 out; in reach envs the hidden cube is then simulated,
                                * pass a model whose object geom has size 0 like mycobot.py:475-481 leaves it); mycobot.py:289-298 */
  int32_t max_episode_steps;   /* 50 */
  int32_t frame_skip;          /* 20 */
  int32_t auto_reset;          /* 1: reset inside mcb_step when terminated|truncated */
  int32_t nefc_max;            /* 0 (default): tiered shared-memory layouts (48-row common case, 88-row middle tier for contact-rich envs,
                                * 176-row last tier), one launch each; 88 / 128: start in the middle / last tier (tests) */
  int32_t controller_type;     /* 0 joint (action 7), 1 IK (7, or 4 with fetch_env), 2 mocap (8, or 4 with fetch_env; needs the mocap
                                  model variant); mycobot.py:36,90-103,134-193 */
  int32_t fetch_env;           /* mycobot.py:41: keyframe start, fixed target orientation, 4-d action (IK only) */
  int32_t control_steps;       /* IK: DLS solves per env-step, each followed by frame_skip substeps (5; mycobot.py:35,162) */
  int32_t mesh_collision;      /* 1: the convex hulls registered with mcb_model_set_hulls collide too (mjc_Convex / mjc_PlaneConvex: one MPR
                                * contact per pair); 0: plane / box primitives only */
  int32_t reserved1_;
  int32_t lockstep_warps;      /* scheduling only, results do not depend on it: warps per lockstep group of the step kernel
                                * (1 free-running ... 16 whole CTA); 0 = free-running until the caller runs mcb_autotune() */
  double distance_threshold;   /* 0.01 */
} mcb_task_cfg;

typedef struct mcb_model mcb_model;
typedef struct mcb_batch mcb_batch;

const char* mcb_version(void);
const char* mcb_last_error(void);
int32_t mcb_model_desc_size(void); /* sizeof(mcb_model_desc) as compiled, for binding self-checks */
int32_t mcb_task_cfg_size(void);

/* replaces mujoco.MjModel.from_xml_path + MyCobotEnv._env_setup (mycobot.py:69-82,450-481) */
int32_t mcb_model_create(const mcb_model_desc* host_desc, int32_t device, mcb_model** out);
int32_t mcb_model_destroy(mcb_model* m);

/* Convex hulls of the model's mesh geoms (mycobot280_main.xml:105-250: two identical mesh geoms per robot body; MuJoCo collides
 * their qhull hulls with mjc_Convex = libccd MPR and mjc_PlaneConvex).  All arrays are HOST pointers and are copied.
 * Hull h: jointed body index (or -1: static) `body[h]`, vertices `vert[vadr[h] .. vadr[h] + vnum[h])` (x, y, z in that body's
 * frame), interior point `center[h]` (the mesh geom's frame origin), bounding radius about it, `mult[h]` identical geoms,
 * contact parameters of the geoms.  Pairs: object ids < MCB_NGEOM name a primitive geom of the model, MCB_NGEOM + h a hull;
 * a pair lists the primitive first.  Call once, before mcb_batch_create. */
typedef struct mcb_hull_desc {
  int32_t nhull, npair, nvert, reserved_;
  int32_t body[MCB_MAXHULL], vadr[MCB_MAXHULL], vnum[MCB_MAXHULL], mult[MCB_MAXHULL], condim[MCB_MAXHULL];
  double center[MCB_MAXHULL][3], rbound[MCB_MAXHULL], friction[MCB_MAXHULL][3], solref[MCB_MAXHULL][2], solimp[MCB_MAXHULL][5],
         solmix[MCB_MAXHULL], invweight[MCB_MAXHULL][2];
  uint8_t pair_a[MCB_MAXHPAIR], pair_b[MCB_MAXHPAIR];
  const double* vert;
} mcb_hull_desc;
int32_t mcb_hull_desc_size(void);
int32_t mcb_model_set_hulls(mcb_model* m, const mcb_hull_desc* hulls);

/* replaces constructing n_envs MyCobotEnv instances (train.py:80-85) */
int32_t mcb_batch_create(mcb_model* m, int32_t n_envs, const mcb_task_cfg* cfg, uint64_t seed, mcb_batch** out);
int32_t mcb_batch_destroy(mcb_batch* b);
int32_t mcb_batch_num_envs(const mcb_batch* b);
int32_t mcb_batch_obs_dim(const mcb_batch* b);
int32_t mcb_batch_action_dim(const mcb_batch* b);   /* 7 (joint, IK), 8 (mocap), 4 (fetch IK / fetch mocap); mycobot.py:90-103 */

/* replaces MyCobotEnv.reset / reset_model / _sample_goal (mycobot.py:207-243,506-514).
 * mask: uint8[N] or NULL (= all).  obj_xy: double[N,2] or NULL (device sampler).  goals: double[N,3] or NULL.
 * Injected values are what the reference's seeded sampler produced (bit-exact goals). */
int32_t mcb_reset(mcb_batch* b, const uint8_t* mask, const double* obj_xy, const double* goals,
                  double* obs, double* achieved_goal, double* desired_goal, void* stream);
/* Same call with HOST buffers (any pointer may be NULL): the other half of the drop-in surface next to mcb_step_host
 * (mycobot.py:506-514 returns the first observation).  Synchronises `stream`. */
int32_t mcb_reset_host(mcb_batch* b, const uint8_t* h_mask, const double* h_obj_xy, const double* h_goals,
                       double* h_obs, double* h_achieved_goal, double* h_desired_goal, void* stream);
/* replaces `self._np_random, seed = seeding.np_random(seed)` of MyCobotEnv.reset(seed=) (mycobot.py:509-510) for the
 * device sampler: the masked envs (all if mask == NULL, a device pointer) get Philox key `seed` and draw counter 0, so
 * the goals / cube positions drawn by the following resets are a function of (seed, env index) only.  Their per-env parameter
 * and latency draw counters (mcb_batch_set_param_ranges, mcb_batch_set_latency_range) restart at 0 too. */
int32_t mcb_seed(mcb_batch* b, uint64_t seed, const uint8_t* mask, void* stream);

/* replaces MyCobotEnv.step, joint (mycobot.py:132-133,190-205) and IK (mycobot.py:134-170, utils.py:499-556) controllers
 * incl. TimeLimit truncation.  actions float32[N, action_dim]; reward float32[N] (sparse) or float64[N] (dense); flags uint8[N].
 * final_obs double[N,obs_dim] or NULL: terminal observation of envs that auto-reset in this call. */
int32_t mcb_step(mcb_batch* b, const float* actions, double* obs, double* achieved_goal, double* desired_goal,
                 void* reward, uint8_t* terminated, uint8_t* truncated, uint8_t* success, double* final_obs,
                 void* stream);

/* Same call with HOST buffers: actions are copied host->device and results device->host inside the call;
 * synchronises `stream` before returning.  Page-locked caller buffers are the copy targets themselves, pageable ones go
 * through pinned staging owned by the batch (one extra host memcpy each).  This is the call a reference-side VecEnv
 * adapter holding numpy arrays makes. */
int32_t mcb_step_host(mcb_batch* b, const float* h_actions, double* h_obs, double* h_achieved_goal,
                      double* h_desired_goal, void* h_reward, uint8_t* h_terminated, uint8_t* h_truncated,
                      uint8_t* h_success, double* h_final_obs /* or NULL */, void* stream);

/* state injection / extraction for parity replay (SURVEY 8c): qpos[N,19] qvel[N,18] ctrl[N,7]
 * qacc_warmstart[N,18] goal[N,3] elapsed int32[N]; any pointer may be NULL.  qprev[N,6] = the arm joint
 * positions the reference's *stale* site poses belong to (data.site_xpos is one substep old after mj_step; the IK
 * controller reads it at the start of the next step, mycobot.py:136,151).  Setting qpos without qprev marks the
 * frames fresh (qprev := qpos), which is the state after reset / mj_forward.  mocap[N,7] = data.mocap_pos | mocap_quat
 * (mocap variant; it persists across resets like in the reference, mycobot.py:207-236 never touches it). */
int32_t mcb_get_state(mcb_batch* b, double* qpos, double* qvel, double* ctrl, double* qacc_warmstart, double* goal,
                      int32_t* elapsed, double* qprev, double* mocap, void* stream);
int32_t mcb_set_state(mcb_batch* b, const double* qpos, const double* qvel, const double* ctrl,
                      const double* qacc_warmstart, const double* goal, const int32_t* elapsed, const double* qprev,
                      const double* mocap, void* stream);

/* the rest of a checkpoint: per-env Philox key, draw counter and running episode return (device pointers, any may be NULL).
 * A batch restored with mcb_set_state + mcb_set_rng_state continues the same goal stream and episode statistics. */
int32_t mcb_get_rng_state(mcb_batch* b, uint64_t* env_seed, uint64_t* draw_counter, double* ep_return, void* stream);
int32_t mcb_set_rng_state(mcb_batch* b, const uint64_t* env_seed, const uint64_t* draw_counter, const double* ep_return, void* stream);

/* Per-env physics parameters (domain randomisation).  Each env carries MCB_NPARAM multipliers (slots: MCB_P_*).  A contact pair's
 * friction mixes the scaled sides like mj_contactParam (the larger wins) and everything derived from it follows: the pyramid rows,
 * their first-row diagApprox and their regulariser scale.  Torsional / rolling friction and the constants the model compiler derives
 * (body_invweight0, dof_invweight0, meaninertia and through them con_diag and the pairs' inverse weights) stay as compiled -- MuJoCo
 * behaves the same way when model.body_mass is written between steps without mj_setConst.  Not available with mesh_collision.
 *
 * mcb_batch_set_param_ranges: HOST arrays of MCB_NPARAM bounds; from the next reset on, every reset of an env (mcb_reset,
 * mcb_reset_host, the auto-reset and the bad-simulation reset inside mcb_step) draws slot k from U[lo[k], hi[k]] before its first
 * forward pass, MCB_NPARAM draws per reset whatever the ranges.  The draws come from the env's Philox key (mcb_seed) with a stream tag
 * and a draw counter of their own: the goal / cube stream is unchanged, and mcb_seed restarts the parameter stream of the envs it
 * reseeds.  NULL, NULL stops drawing (the current values stay).  Non-finite bounds, bounds <= 0 and lo > hi are rejected and leave
 * the batch as it was.  The first call turns per-env parameters on (nominal values for every env): it allocates and synchronises
 * the device, so it is not capturable.  Steps and resets enqueued later use the new ranges; a captured CUDA graph keeps the ranges
 * it was captured with. */
int32_t mcb_batch_set_param_ranges(mcb_batch* b, const double* h_lo, const double* h_hi);
/* device pointers params double[N, MCB_NPARAM] and draw_counter uint64[N], either may be NULL.  A batch without per-env parameters
 * reports 1.0 and 0. */
int32_t mcb_get_env_params(mcb_batch* b, double* params, uint64_t* draw_counter, void* stream);
/* fixed per-env values (evaluation, system identification, checkpoints): device pointers as above, either may be NULL.  Turns
 * per-env parameters on if needed (like mcb_batch_set_param_ranges' first call; drawing stays off until ranges are set).  Like
 * mcb_set_state it does not validate device data. */
int32_t mcb_set_env_params(mcb_batch* b, const double* params, const uint64_t* draw_counter, void* stream);

/* Per-env actuation latency (domain randomisation of the control delay).  Each env carries an integer latency d in substeps,
 * 0 <= d <= cfg.frame_skip: every command the controller issues (joint ctrl; mocap pose and gripper ctrl, still computed at substep
 * 0 from the stale frames; each IK block's DLS result) is written before substep d of its block, after the block's last substep
 * when d == frame_skip (before the block_gripper forward pass), and until then the previous command stays in force.  A reset's
 * command is its own (init / key ctrl and the persisting mocap pose).  d == 0 gives the results of a batch without latency bit for
 * bit.  Latency runs in the step kernels of batches with per-env parameters (nominal multipliers if no ranges are set); it is not
 * available with mesh_collision.
 *
 * mcb_batch_set_latency_range: in substeps; from the next reset on, every reset of an env (as for mcb_batch_set_param_ranges)
 * draws d uniformly from the integers [lo, hi]: lo + min(hi - lo, floor(u * (hi - lo + 1))), one draw of the env's Philox key with
 * a stream tag and a draw counter of their own (the goal / cube and parameter streams are unchanged; mcb_seed restarts the
 * counter).  0 <= lo <= hi <= cfg.frame_skip, else rejected and the batch is left as it was; lo = hi = -1 stops drawing (the
 * current values stay).  The first call turns per-env parameters on (nominal multipliers), like mcb_batch_set_param_ranges: it
 * allocates, synchronises and cannot be captured. */
int32_t mcb_batch_set_latency_range(mcb_batch* b, int32_t lo, int32_t hi);
/* device pointers latency int32[N], draw_counter uint64[N], either may be NULL; a batch without latency reports 0 and 0 */
int32_t mcb_get_env_latency(mcb_batch* b, int32_t* latency, uint64_t* draw_counter, void* stream);
/* fixed per-env latencies (evaluation, system identification, checkpoints): device pointers as above, either may be NULL.  Turns
 * per-env parameters on if needed.  It does not validate device data: the step kernels clamp a latency to [0, cfg.frame_skip]. */
int32_t mcb_set_env_latency(mcb_batch* b, const int32_t* latency, const uint64_t* draw_counter, void* stream);

/* Per-env applied forces (MuJoCo's data.qfrc_applied and data.xfrc_applied on the reduced model), persistent state like in MuJoCo:
 * they act on every substep of every mcb_step, on the block_gripper forward pass, on mcb_forward and on mcb_debug_forward (whose
 * qfrc_bias then includes -J' xfrc, so that its qfrc_smooth equals MuJoCo's).  Actuation latency does not delay them.
 *   qfrc: double[N, MCB_NV], a generalized force per dof, added to qfrc_smooth (mj_fwdAcceleration).
 *   xfrc: double[N, MCB_NB, 6], per jointed body (mcb_model_desc order) a world-frame force (0:3) and torque (3:6) applied at the
 *         body's composite centre of mass xpos + xmat * ipos through the body's Jacobian at the current pose (mj_xfrcAccumulate).  For
 *         the cube that is MuJoCo's xipos; for a body with merged fixed children it is the merged body's centre of mass.
 * Every reset of an env (mcb_reset, mcb_reset_host, the auto-reset and the bad-simulation reset inside mcb_step) sets its forces to
 * zero (mj_resetData) before its first forward pass.  In reach envs without reward_shaping the cube is frozen and its forces (body 12,
 * dofs 12..17) are ignored.  Zero forces give the results of a batch without forces bit for bit.  Forces run in the step kernels of
 * batches with per-env parameters (nominal multipliers if no ranges are set); they are not available with mesh_collision.
 *
 * mcb_set_env_applied: device pointers, either may be NULL (that array is left as it is).  It does not validate device data, like
 * mcb_set_state: a non-finite force ends the env's episode through the bad-simulation guard, whose reset clears it.  The first call
 * turns forces on (zero for every env) and per-env parameters with them: it allocates, synchronises and cannot be captured.  Later
 * calls are one kernel on `stream` and can be captured, so a graph replays steps with whatever the caller's arrays hold. */
int32_t mcb_set_env_applied(mcb_batch* b, const double* qfrc, const double* xfrc, void* stream);
/* device pointers as above, either may be NULL; a batch without forces reports zeros */
int32_t mcb_get_env_applied(mcb_batch* b, double* qfrc, double* xfrc, void* stream);

/* Per-env contact output (MuJoCo's data.contact with mj_contactForce).  After every mcb_step, mcb_reset and mcb_forward (and their
 * _host forms), each env that call wrote holds the contacts of its last forward pass, what data.contact / efc_force hold when the
 * reference returns: the last substep's (contacts at its pre-integration state, forces of its Newton solve), the block_gripper forward
 * pass's for block_gripper batches, and the reset's for an env that auto-reset (or hit the bad-simulation reset) in the step, so that
 * the contacts line up with obs.  For such an env the final triple, if registered, receives the contacts of the terminal state before
 * the reset, the ones the step's reward was computed from; like final_obs, rows of the other envs are left untouched.  A masked
 * mcb_reset writes the masked envs only; mcb_set_state writes nothing (the next mcb_forward refreshes the contacts).
 *   ncon: int32[N] contacts in use.
 *   geom: int32[N, MCB_MAXCON, 3] geom1, geom2 (ids of the MCB_NGEOM primitive geoms in mcb_model_desc order), dim (condim).
 *   con:  double[N, MCB_MAXCON, MCB_CONTACT_DOUBLES] dist, pos[3], frame[9] (rows: normal, first and second tangent), force[6]:
 *         mj_contactForce in the contact frame (mju_decodePyramid): force[0] is the sum of the contact's 2 (dim - 1) pyramid forces,
 *         force[i + 1] = (p[2i] - p[2i + 1]) mu[i] for i < dim - 1 with mu = (sliding, sliding[, torsional]), the rest 0.  Sliding
 *         friction is the env's mixed value under its per-env parameters.
 * Slots >= ncon are zero with geom ids -1 and dim 0, so a plain sum over slots is correct.  Contacts that the last layout tier drops
 * because their constraint rows do not fit are not reported (they are counted in stats[5] and absent from ncon).  All six pointers are
 * caller-owned device arrays that stay valid while registered; the final triple may be NULL (no final output), and all NULL turns the
 * output off.  Turning it on turns per-env parameters on (nominal values if no ranges are set).  The call synchronises the device;
 * steps captured in a CUDA graph afterwards write to the registered arrays.  mcb_autotune restores them exactly.  Not available with
 * mesh_collision (hull contacts are out of scope). */
int32_t mcb_set_contact_output(mcb_batch* b, int32_t* ncon, int32_t* geom, double* con, int32_t* final_ncon, int32_t* final_geom,
                               double* final_con);

/* replaces mujoco.mj_forward on every env (mycobot.py:213,229,306); refreshes qacc_warmstart; optional obs out */
int32_t mcb_forward(mcb_batch* b, double* obs, double* achieved_goal, double* desired_goal, void* stream);

/* replaces MyCobotEnv.compute_reward for HER relabelling batches (mycobot.py:289-295, utils.py:24-26) */
int32_t mcb_compute_reward(const double* achieved_goal, const double* goal, int64_t n, double distance_threshold,
                           int32_t reward_type, void* out, void* stream);

/* episode statistics accumulated on device since the last call with reset_after != 0:
 * out[0]=episodes, [1]=successes, [2]=return_sum, [3]=length_sum, [4]=env_steps, [5]=anomalies (constraint rows dropped in the last layout tier + bad-simulation resets),
 * [6]=solver iterations, [7]=substeps.  `out` is a device pointer to 8 doubles. */
int32_t mcb_stats(mcb_batch* b, double* out, int32_t reset_after, void* stream);

/* debug tap for stage-level parity tests: runs mcb_forward() and copies intermediate quantities of env `env`
 * to host memory (`what` is reserved, pass 0).  Layout in doubles: nefc, ncon, solver iterations, overflow |
 * M[18*18] | qfrc_bias, qfrc_smooth, qacc_smooth, qacc, qfrc_constraint [18 each] | xpos[13*3] | xmat[13*9] |
 * efc_J[nefc*18] in MuJoCo row order (equality, limits, contacts) | efc_aref[nefc] | efc_D[nefc] |
 * (dist, pos3, normal3) * ncon.  cap must be >= 4262, the dump's size for the last tier's 176 rows and 24 contacts; a smaller
 * cap fails before anything runs.  Returns the number of doubles written. */
int32_t mcb_debug_forward(mcb_batch* b, int32_t env, int32_t what, double* h_out, int32_t cap, void* stream);

/* Picks the lockstep grouping of the step kernel for this batch (cfg.lockstep_warps == 0): rolls the batch 32 steps
 * ahead (the state right after a reset is not representative), times `steps_per_candidate` (0 -> 4) steps per candidate
 * from that state, keeps the fastest and restores state, episode clocks, RNG streams, per-env parameters, latencies, applied forces, contact output and statistics exactly.  `actions`
 * (device float32 [N, action_dim]) are applied at every tuning step; NULL -> uniform random actions from a private
 * Philox stream.  Synchronises the stream and allocates scratch: it is never called implicitly -- mcb_step only enqueues
 * its three kernels on the caller's stream (no hidden sync, CUDA-graph capturable).  Returns the chosen grouping. */
int32_t mcb_autotune(mcb_batch* b, const float* actions, int32_t steps_per_candidate, void* stream);
int32_t mcb_batch_lockstep_warps(const mcb_batch* b);
/* how many envs of the most recent step overflowed the common shared-memory layout and were redone by the middle-tier
 * kernel (return value) and how many of those also overflowed the middle tier (*last_tier_envs, may be NULL).
 * Synchronises the stream; diagnostics for bench.py. */
int32_t mcb_last_fallback_envs(mcb_batch* b, int32_t* last_tier_envs, void* stream);
/* the env indices behind that count: up to `cap` of the envs of the most recent step that left the common layout are
 * copied to the HOST array h_envs; returns how many there were.  Synchronises the stream (parity tests compare exactly
 * these envs with the oracle). */
int32_t mcb_last_fallback_list(mcb_batch* b, int32_t* h_envs, int32_t cap, void* stream);

/* measurement helpers used by bench.py */
int32_t mcb_last_step_launches(const mcb_batch* b); /* kernels launched by the most recent mcb_step (counted at the launch sites) */
int64_t mcb_total_launches(const mcb_batch* b);     /* all kernels this library launched for the batch since mcb_batch_create */
int32_t mcb_fp64_peak_probe(int32_t device, int32_t iters, double* tflops_out); /* DFMA micro-kernel, CUDA-event timed */

/* ---------------------------------------------------------------------------------------------------------------
 * Device-resident HER replay ("future" strategy) -- replaces stable_baselines3.HerReplayBuffer as
 * mycobotgym/scripts/train.py:89-97 configures it (n_sampled_goal=4, goal_selection_strategy="future"), including its
 * env.compute_reward call on relabelled goals (mycobot.py:289-295).  All array arguments are device pointers.
 * Semantics follow stable_baselines3==2.0.0a0 her_replay_buffer.py: per stored transition ep_start / ep_length,
 * only transitions of complete episodes are sampled, the first int((1 - 1/(n_sampled_goal+1)) * batch) samples get
 * desired_goal := next_achieved_goal of a transition drawn uniformly from [current, episode end) and a recomputed
 * reward (float32), dones are returned as done * (1 - timeout). */
typedef struct mcb_her mcb_her;
int32_t mcb_her_create(int32_t n_envs, int32_t buffer_steps, int32_t obs_dim, int32_t action_dim, int32_t n_sampled_goal,
                       int32_t reward_type, double distance_threshold, uint64_t seed, mcb_her** out);
void mcb_her_destroy(mcb_her* h);
/* HerReplayBuffer.add: one transition per env, [N, .] rows; rewards float32 (rewards_f64 = 0) or float64 (1) */
int32_t mcb_her_add(mcb_her* h, const double* obs, const double* achieved_goal, const double* desired_goal, const double* next_obs,
                    const double* next_achieved_goal, const float* actions, const void* rewards, int32_t rewards_f64,
                    const uint8_t* terminated, const uint8_t* truncated, void* stream);
int64_t mcb_her_size(const mcb_her* h);                       /* stored transitions (all envs) */
/* debugging / tests: copies of the episode table [T, N] (device) and the number of sampleable transitions (host) */
int32_t mcb_her_episode_table(mcb_her* h, int32_t* ep_start, int32_t* ep_length, int64_t* n_valid_host, void* stream);
/* HerReplayBuffer.sample(batch_size).  inj_index [batch] (flat t * N + env) and inj_future [batch] (index inside the
 * episode) replace the device RNG draws when non-null (parity tests).  index_out [batch, 2] (optional) receives the
 * sampled flat index and the relabel source (or -1).  *fail_count (device int) counts samples that found no complete episode. */
int32_t mcb_her_sample(mcb_her* h, int32_t batch_size, const int64_t* inj_index, const int32_t* inj_future, double* obs, double* achieved_goal,
                       double* desired_goal, double* next_obs, double* next_achieved_goal, float* actions, float* rewards, float* dones,
                       int64_t* index_out, int32_t* fail_count, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MYCOBOT_B200_H_ */
