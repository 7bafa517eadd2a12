// mcb_engine.cu -- B200 (sm_100a) batched myCobot physics-and-task engine, C ABI in include/mycobot_b200.h.
//
// One environment per warp; the whole env-step (frame_skip substeps of the MuJoCo-equivalent forward
// dynamics + semi-implicit Euler, then observation / reward / success / auto-reset) is one kernel launch.
// An env's working set lives in the warp's slice of shared memory; HBM sees one 640-byte state record read
// and written per env-step plus the action and the outputs.  All arithmetic is fp64 on the CUDA cores
// (DFMA); tensor cores are deliberately unused: the per-env matrices are 18x18 and smaller and the work is a
// sequence of tree recursions and tiny factorizations, not a dense contraction.
//
// Decisions that set the speed (profiles/README.md has the measurement behind each):
//   * the kernel is latency-bound, so resident envs per SM is the first lever: shared memory per env is
//     ~13.7 KB (16 envs/SM, pinned from the other side by 128 registers per thread) in the common case.  Dead
//     dynamics temporaries and the constraint rows share one union; matrices are packed lower triangles; the
//     constraint Jacobian is stored BLOCKED by row type (robot rows: 12 columns, cube rows: 6, coupled rows: 18,
//     joint-limit rows: none);
//   * capacity comes in three tiers (EnvS<TIER>): 48 rows for the common case, 88 rows / 10 envs per CTA for
//     contact-rich envs (a grasp), 176 rows / five envs per CTA as the last resort.  An env that does not fit its tier
//     aborts untouched, is queued on a device list and is redone by the next tier's launch;
//   * the block structure robot(12) + cube(6) is used everywhere: M's cube block never couples, H couples
//     only through finger-cube contact rows, so the usual factorizations are 12x12 and 6x6, fully unrolled, as
//     L D L' with rows in registers and a branch-free reciprocal (chol_solve_blk);
//   * the kinematic tree is compiled in (kTreeParent): fk and the RNE / CRB passes are register chain walks;
//   * only a quarter of the executed instructions are FP64 math, so instruction count and code footprint matter as
//     much as the math: no division slow paths, explicit 32-bit shuffles, out-of-line helpers on the hot path;
//   * warps of a CTA run free or in lockstep groups (named barriers), chosen per batch by mcb_autotune().
//
// Stage map (what each device function restates; the reference reaches all of it through
// mujoco.mj_step, mycobotgym/envs/mycobot.py:193 -> gymnasium MujocoEnv.do_simulation):
//   fk()              mj_kinematics              cinert_cdof()  mj_comPos
//   crb_mass()        mj_crb                     chol_solve_blk() mj_factorM / mj_solveM (dense L D L' per block)
//   velocity_rne()    mj_comVel, mj_rne          actuation_smooth() mj_passive, mj_fwdActuation
//   collide()         mj_collision (plane-box, box-box)
//   make_rows()       mj_makeConstraint + mj_makeImpedance + mj_referenceConstraint
//   Newton            mj_solNewton (pyramidal cones, exact line search)
//   euler()           mj_Euler + mj_integratePos
//   write_obs() etc.  MyCobotEnv._get_obs / compute_reward / _is_success / reset_model (mycobot.py:207-298,342-400)
//   ik_target() / ik_update_ctrl()  IKController (utils.py:469-556); mocap branch of the step: mycobot.py:172-189
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <math.h>
#include <cmath>
#include <string>
#include <vector>
#include <stdlib.h>

#include "mycobot_b200.h"

#define NB MCB_NB
#define NV MCB_NV
#define NQ MCB_NQ
#define NU MCB_NU
#define NH MCB_NHINGE
#define NTRI 171        // packed lower triangle of an 18 x 18 matrix
#define TRI(i, j) ((i) * ((i) + 1) / 2 + (j))
#define TRIP(i, j) ((((i) >> 1) * (((i) >> 1) + 1) * 2 + ((i) & 1) * ((i) + 1)) + (j))   // row starts padded to even offsets
#define NTRIP 180
#define SR 13           // padded strides of the blocked Jacobian rows (odd => conflict-free lane-per-row reads)
#define SC 7
#define SF 19
#define FULLMASK 0xffffffffu
#define MINVAL 1e-15
#define MINIMP 0.0001
#define MAXIMP 0.9999
#define CUBE 12
#define NMNZ_MAX 96
#define RM_INEQ 0x10000  // rmeta bit: inequality row (limit / contact)
#define NFRC (NV + NB * 6)  // applied forces per env: qfrc_applied[NV], then xfrc_applied[NB][6] (world force 0:3, torque 3:6)

namespace {

thread_local std::string g_err;
int fail(const char* what, cudaError_t e = cudaSuccess) {
  g_err = what;
  if (e != cudaSuccess) { g_err += ": "; g_err += cudaGetErrorString(e); }
  return -1;
}
#define CK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return fail(#call, e_); } while (0)

struct PairParam {
  int g1, g2, dim, ptype;  // ptype: 0 rows touch robot dofs only, 1 cube dofs only, 2 both; g: object ids (>= MCB_NGEOM: hull)
  int b1, b2;              // jointed bodies carrying the two geoms (-1: static)
  double friction[3];
  double KB[2];            // on the device: (K, B) of mj_makeImpedance (the host fills the mixed solref here first, row_constants() converts)
  double solimp[5];        // clamped once at model creation
  double tran, pyr2;       // body_invweight0 sum (translational), 2 mu^2 / impratio / multiplicity (the pyramid's regulariser scale)
};

struct DevModel {
  mcb_model_desc d;
  int nlevel;
  int level_start[NB + 1];
  int level_body[NB];
  int nmnz;
  unsigned char mnz_i[NMNZ_MAX], mnz_j[NMNZ_MAX];
  unsigned char tri_i[176], tri_j[176];   // packed lower-triangle index e -> (row, column)
  PairParam pair[MCB_MAXPAIR];
  // convex hulls of the mesh geoms (mcb_model_set_hulls): what the broad phase needs is staged with the model, vertices and
  // the per-pair contact parameters stay in global memory (read only when a hull pair is actually close)
  int nhull, nhpair;
  int hull_body[MCB_MAXHULL], hull_vadr[MCB_MAXHULL], hull_vnum[MCB_MAXHULL];
  double hull_center[MCB_MAXHULL][3], hull_rbound[MCB_MAXHULL];
  unsigned char hpair_a[MCB_MAXHPAIR], hpair_b[MCB_MAXHPAIR];
  const double* hull_vert;          // [nvert][3], body frames
  const PairParam* hpair_param;     // [nhpair]
};

// The flattened model is staged into the CTA's shared memory (offset 0 of the dynamic segment, before the per-env
// slices): most model tables are indexed by lane (body / dof / pair), which serialises in the constant cache and
// misses in L1 (no L1 is left once shared memory is maxed out); from shared memory they are ordinary LDS.
extern __shared__ __align__(16) unsigned char smem_raw[];
#define MODEL_BYTES ((sizeof(DevModel) + 15) / 16 * 16)
#define MDL (*reinterpret_cast<const DevModel*>(smem_raw))
// contact -> its pair's parameters: primitive pairs from the staged table, hull pairs (ids >= MCB_MAXPAIR) from global memory
#define PP(cp) ((cp) < MCB_MAXPAIR ? MDL.pair[cp] : MDL.hpair_param[(cp) - MCB_MAXPAIR])

static_assert(sizeof(DevModel) % sizeof(double) == 0, "DevModel must be a whole number of doubles");

enum { MODE_STEP = 0, MODE_FORWARD = 1, MODE_RESET = 2 };

// offsets of the arrays in an env's resident state record (MCB_STATE_STRIDE doubles; the record ends in padding)
enum { ST_QPOS = 0, ST_QVEL = ST_QPOS + NQ, ST_CTRL = ST_QVEL + NV, ST_WARM = ST_CTRL + NU, ST_GOAL = ST_WARM + NV, ST_QPREV = ST_GOAL + 3,
       ST_MOCAP = ST_QPREV + 6, ST_END = ST_MOCAP + 7 };
static_assert(ST_END <= MCB_STATE_STRIDE, "the state record must fit its stride");

// The per-env extensions of a batch, read by the PRM kernels only: one record, held by the batch and copied whole into StepArgs.
struct EnvExt {
  // per-env physics parameters
  double* params;            // [N, MCB_NPARAM] multipliers
  unsigned long long* param_ctr;  // [N] parameter draw counters
  int draw_params;           // resets draw new parameters from U[param_lo, param_hi]
  double param_lo[MCB_NPARAM], param_hi[MCB_NPARAM];
  // actuation latency: a new command takes effect latency[env] substeps after it is issued
  int* latency;              // [N] substeps, 0..frame_skip
  unsigned long long* lat_ctr;    // [N] latency draw counters
  int draw_latency, lat_lo, lat_hi;   // resets draw the latency uniformly from the integers [lat_lo, lat_hi]
  // applied forces (null: the batch has none): qfrc_applied (NV) then xfrc_applied (NB x 6) per env
  double* frc;               // [N, NFRC]
  // contact output (caller-owned; null con_n: off): the contacts of each written env's last forward pass, and (con_fn set) those
  // of the terminal state before an auto-reset; ncon [N], geom1 / geom2 / dim [N, MCB_MAXCON, 3], dist pos frame force [N, MCB_MAXCON, 19]
  int *con_n, *con_geom;
  double* con;
  int *con_fn, *con_fgeom;
  double* con_f;
};

struct StepArgs {
  const DevModel* m;
  int n_envs, mode;
  int lockstep_warps;        // warps per lockstep group of the common-layout kernel (1 = free-running), see group_sync()
  int mid_threshold;         // the middle tier only runs when more envs than this left the common layout (else: straight to the last tier)
  mcb_task_cfg cfg;
  const unsigned long long* env_seed;  // [N] Philox key per env (mcb_seed)
  double* state;             // [N, MCB_STATE_STRIDE]
  int* elapsed;              // [N]
  double* ep_return;         // [N]
  unsigned long long* rng_ctr;  // [N]
  double* stats;             // [8]
  int* redo_count;           // [2] envs that overflowed tier 0 / tier 1 in this step
  int* redo_list;            // [2][N]
  const float* actions;      // [N, action_dim]
  const uint8_t* mask;       // reset
  const double* inj_xy;      // reset
  const double* inj_goal;    // reset
  double *obs, *ag, *dg, *final_obs;
  void* reward;
  uint8_t *terminated, *truncated, *success;
  double* debug;             // optional debug dump of env debug_env
  int debug_env;
  int canary_selftest;       // MCB_CANARY build + MCB_CANARY_SELFTEST=1 in the environment: every env writes one double past cpos[] on purpose
  EnvExt x;                  // the batch's per-env extensions (PRM kernels only)
};

// ------------------------------------------------------------------------------------------------
// Per-env shared-memory working set, one layout per capacity tier (DESIGN.md section 3): warps (= envs) per CTA, constraint rows,
// doubles of the blocked Jacobian pool, contacts.  TIER 0: the common case; TIER 1: contact-rich envs -- a grasp, pushing, the
// gripper resting on the table; TIER 2: the last resort (one CTA per SM), rows beyond its capacity are dropped and counted: both
// finger pads flat on the table (8 box-box points each) plus the cube's four corners are 20 condim-4 contacts = 120 rows on top
// of the 13 equality rows and the joint limits -- the IK / mocap soak runs dropped rows at 16 contacts / 128 rows.
template <int TIER> struct Tier;
template <> struct Tier<0> { enum { WARPS = 16, NROW = 48, POOL = 460, MAXC = 8 }; };
template <> struct Tier<1> { enum { WARPS = 10, NROW = 88, POOL = 1230, MAXC = 14 }; };
template <> struct Tier<2> { enum { WARPS = 5, NROW = 176, POOL = 2432, MAXC = 24 }; };
static_assert(Tier<2>::MAXC == MCB_MAXCON, "the contact output holds every contact the last tier keeps");
template <int TIER>
struct EnvCore {
  // MCB_CANARY build (tests/test_gpu_canary.py; compute-sanitizer is closed on the GPU pool): guard words between the arrays of
  // the record, set when an env is loaded and checked when it is stored; a hit is counted in stats[5] and reported.  The pools
  // shrink by the guards' size, which only moves the point where an env changes tier (results do not depend on the tier).
#ifdef MCB_CANARY
#define GUARD(name) double name[2];
#define MCB_NGUARD 8
#else
#define GUARD(name)
#define MCB_NGUARD 0
#endif
  enum { NROW = Tier<TIER>::NROW, POOL = Tier<TIER>::POOL - (MCB_NGUARD ? (TIER == 0 ? 10 : 2 * MCB_NGUARD) : 0),   // (tier 0: the row arrays must stay the union's largest member)
         MAXC = Tier<TIER>::MAXC, IS_BIG = TIER == 2, TIER_ID = TIER };
  double qpos[20], qvel[NV], ctrl[8], warm[NV], goal[4];
  GUARD(g0)
  double xpos[NB * 3], xmat[NB * 9], cdof[NV * 6], refcube[4];
  GUARD(g1)
  double M[NTRI + 1];
  GUARD(g2)
  double H[NTRIP];          // H doubles as the factor storage of chol_solve_blk (padded rows, TRIP)
  GUARD(g3)
  double qfrc_bias[NV], qfrc_smooth[NV], qacc_smooth[NV], qacc[NV], Ma[NV], grad[NV], search[NV], Mv[NV], qfrc_con[NV];
  GUARD(g4)
  double anchors[12];
  double qprev[6];   // arm qpos the frames in shared memory were computed from (the reference's stale site poses)
  double ik[14];     // IK controller: target position (3), target quaternion (4), pose error (6); mocap variant: weld residual (6)
  double mocap[8];   // mocap variant: data.mocap_pos (3) | data.mocap_quat (4)
  double quat5[4];   // mocap variant: orientation quaternion of the body carrying gripper_tcp (composed like mj_kinematics)
  GUARD(g5)
  union {
    struct { union { double lR[NB * 9]; double buf[NV * 6]; }; double cinert[NB * 10], crb[NB * 10], cvel[NB * 6], cacc[NB * 6], cdof_dot[NV * 6]; };  // dead after velocity_rne (lR after fk)
    struct { double pool[POOL], eD[NROW], earef[NROW], eJaref[NROW], eJv[NROW]; };                                              // live from make_rows
    double cscr[152];                                                                                                           // collision scratch (between the two)
  };
  GUARD(g6)
  double cdist[MAXC], cpos[MAXC * 3], cframe[MAXC * 9];
  GUARD(g7)
  int cpair[MAXC], crow[MAXC];
  int rmeta[NROW];   // bits 0-7 index (eq / contact / dof), 8 sign, 9-11 sub-row, 12-14 kind (0 connect 1 joint-eq 2 limit 3 contact 4 weld), 16 inequality
  int nR, nC, nF, nU, nefc, ncon, overflow, iters;
  int mesh, pad_[3];   // mesh: the batch collides the convex hulls too (cfg.mesh_collision)
};
// PRM: the batch has per-env physics parameters (mcb_batch_set_param_ranges / mcb_set_env_params).  Batches without them run the
// PRM = false kernels, whose record is EnvCore itself and whose code does not contain the parameter reads.  With them, the env's
// MCB_NPARAM multipliers and its parameter draw counter are staged after the working set, and so are its actuation latency (substeps,
// clamped to [0, frame_skip] when loaded) and the latency draw counter; `prm_drawn` marks a record a reset redrew (only such records
// are written back).  `frc` points to the env's applied forces in global memory (read there, L1 / L2-resident, not staged): null when
// the batch has none or once a reset in this launch cleared them; the commit zeroes the row of an env whose pointer was cleared.
template <int TIER, bool PRM = false>
struct EnvS : EnvCore<TIER> { enum { HAS_PRM = 0 }; };
template <int TIER>
struct EnvS<TIER, true> : EnvCore<TIER> {
  enum { HAS_PRM = 1 };
  GUARD(gp)
  double prm[MCB_NPARAM];
  unsigned long long prm_ctr, lat_ctr;
  int prm_drawn, lat;
  const double* frc;
};
static_assert(offsetof(EnvCore<0>, H) % 16 == 0 && offsetof(EnvCore<1>, H) % 16 == 0 && offsetof(EnvCore<2>, H) % 16 == 0, "factor storage must be 16-byte aligned (128-bit loads)");
static_assert(sizeof(EnvS<0>) % 16 == 0 && sizeof(EnvS<1>) % 16 == 0 && sizeof(EnvS<2>) % 16 == 0, "per-env records must keep 16-byte alignment");
static_assert(sizeof(EnvS<0, true>) % 16 == 0 && sizeof(EnvS<1, true>) % 16 == 0 && sizeof(EnvS<2, true>) % 16 == 0, "per-env records must keep 16-byte alignment");
static_assert(sizeof(EnvS<0, true>) - sizeof(EnvS<0>) == 144 + 8 * (MCB_NGUARD ? 2 : 0),
              "the parameter record is 14 doubles, two draw counters, a flag, the latency and the applied-force pointer");
template <int TIER, bool PRM = false> constexpr size_t cta_bytes() { return MODEL_BYTES + Tier<TIER>::WARPS * sizeof(EnvS<TIER, PRM>); }
static_assert(cta_bytes<0>() <= 232448 && cta_bytes<1>() <= 232448 && cta_bytes<2>() <= 232448, "a CTA must fit the 227 KB of shared memory an SM offers");
static_assert(cta_bytes<0, true>() <= 232448 && cta_bytes<1, true>() <= 232448 && cta_bytes<2, true>() <= 232448,
              "a CTA with per-env parameters must fit the 227 KB of shared memory an SM offers");


// ------------------------------------------------------------------------------------------------
// fast_rcp(): 1 / d for d >= MINVAL without the library routine's special-case branches: MUFU seed (about 20 bits)
// and two Newton steps (error about 1 ulp; the factorisation does not need a correctly rounded quotient).
__device__ __forceinline__ double fast_rcp(double d) {
  double y;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(d));
  double e = fma(-d, y, 1.0);
  y = fma(y, e, y);
  e = fma(-d, y, 1.0);
  return fma(y, e, y);
}

// 64-bit shuffle as two explicit 32-bit shuffles (the generic double overload left register swaps behind)
__device__ __forceinline__ double shfl_xor_d(double v, int m) {
  int lo = __shfl_xor_sync(FULLMASK, __double2loint(v), m);
  int hi = __shfl_xor_sync(FULLMASK, __double2hiint(v), m);
  return __hiloint2double(hi, lo);
}
__device__ __forceinline__ double shfl_d(double v, int src) {
  int lo = __shfl_sync(FULLMASK, __double2loint(v), src);
  int hi = __shfl_sync(FULLMASK, __double2hiint(v), src);
  return __hiloint2double(hi, lo);
}

// (noinline here and on mulM_row, and one DADD instantiation of the 12 x 12 factorisation for all three uses: the hot code
// footprint is what free-running warps pay for in instruction fetch -- profiles/README.md)
__device__ __noinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += shfl_xor_d(v, o);
  return v;
}
// three warp sums in one butterfly: after two rounds every lane carries one of the (up to four) quantities, so the
// remaining three rounds move one value instead of three -- 9 double shuffles (incl. the broadcasts) instead of 15
__device__ __forceinline__ void warp_sum3(double& a, double& b, double& c, int lane) {   // (out of line the three references live in local memory)
  const bool odd = lane & 1, hi = lane & 2;
  const double r1 = shfl_xor_d(odd ? a : b, 1);      // even lanes collect a and c, odd lanes collect b
  const double r2 = shfl_xor_d(c, 1);
  const double x = (odd ? b : a) + r1, y = odd ? 0.0 : c + r2;
  const double r3 = shfl_xor_d(hi ? x : y, 2);       // lanes 4k: a, 4k+1: b, 4k+2: c (4k+3 carries nothing)
  double z = (hi ? y : x) + r3;
  z += shfl_xor_d(z, 4); z += shfl_xor_d(z, 8); z += shfl_xor_d(z, 16);
  a = shfl_d(z, 0); b = shfl_d(z, 1); c = shfl_d(z, 2);
}
__device__ __forceinline__ double dot3(const double* a, const double* b) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; }
__device__ __forceinline__ void cross3(double* r, const double* a, const double* b) {
  r[0] = a[1] * b[2] - a[2] * b[1]; r[1] = a[2] * b[0] - a[0] * b[2]; r[2] = a[0] * b[1] - a[1] * b[0];
}
__device__ __forceinline__ void mul_inert_vec(double* r, const double* i, const double* v) {
  r[0] = i[0] * v[0] + i[3] * v[1] + i[4] * v[2] - i[8] * v[4] + i[7] * v[5];
  r[1] = i[3] * v[0] + i[1] * v[1] + i[5] * v[2] + i[8] * v[3] - i[6] * v[5];
  r[2] = i[4] * v[0] + i[5] * v[1] + i[2] * v[2] - i[7] * v[3] + i[6] * v[4];
  r[3] = i[8] * v[1] - i[7] * v[2] + i[9] * v[3];
  r[4] = i[6] * v[2] - i[8] * v[0] + i[9] * v[4];
  r[5] = i[7] * v[0] - i[6] * v[1] + i[9] * v[5];
}
__device__ __forceinline__ void cross_motion(double* r, const double* vel, const double* v) {
  r[0] = -vel[2] * v[1] + vel[1] * v[2];
  r[1] = vel[2] * v[0] - vel[0] * v[2];
  r[2] = -vel[1] * v[0] + vel[0] * v[1];
  r[3] = -vel[2] * v[4] + vel[1] * v[5] - vel[5] * v[1] + vel[4] * v[2];
  r[4] = vel[2] * v[3] - vel[0] * v[5] + vel[5] * v[0] - vel[3] * v[2];
  r[5] = -vel[1] * v[3] + vel[0] * v[4] - vel[4] * v[0] + vel[3] * v[1];
}
__device__ __forceinline__ void cross_force(double* r, const double* vel, const double* f) {
  r[0] = -vel[2] * f[1] + vel[1] * f[2] - vel[5] * f[4] + vel[4] * f[5];
  r[1] = vel[2] * f[0] - vel[0] * f[2] + vel[5] * f[3] - vel[3] * f[5];
  r[2] = -vel[1] * f[0] + vel[0] * f[1] - vel[4] * f[3] + vel[3] * f[4];
  r[3] = -vel[2] * f[4] + vel[1] * f[5];
  r[4] = vel[2] * f[3] - vel[0] * f[5];
  r[5] = -vel[1] * f[3] + vel[0] * f[4];
}
__device__ __forceinline__ void quat2mat(double* m, const double* q) {
  double q00 = q[0] * q[0], q01 = q[0] * q[1], q02 = q[0] * q[2], q03 = q[0] * q[3];
  double q11 = q[1] * q[1], q12 = q[1] * q[2], q13 = q[1] * q[3], q22 = q[2] * q[2], q23 = q[2] * q[3], q33 = q[3] * q[3];
  m[0] = q00 + q11 - q22 - q33; m[4] = q00 - q11 + q22 - q33; m[8] = q00 - q11 - q22 + q33;
  m[1] = 2 * (q12 - q03); m[2] = 2 * (q13 + q02); m[3] = 2 * (q12 + q03);
  m[5] = 2 * (q23 - q01); m[6] = 2 * (q13 - q02); m[7] = 2 * (q23 + q01);
}


// kinematic tree of the reduced model (flatten.reduce_model): arm 0..5, gripper sub-chains 6->7, 8->9, 10, 11 under body 5,
// free cube 12.  fk() is written against this table; mcb_model_create checks the descriptor against it.
static const int kTreeParent[NB] = {-1, 0, 1, 2, 3, 4, 5, 6, 5, 8, 5, 5, -1};

// ------------------------------------------------------------------------------------------------
// fk(): body frames of the 13 jointed bodies.  Lane b builds the local transform of body b
// (Tmat * Rot(axis, q)); the chain is then composed along the tree with matrix rows held in registers.
template <class S>
__device__ void fk(S& s, const DevModel* __restrict__ m, int lane, int nba) {
  if (lane < NH) {
    double ang = s.qpos[lane] - MDL.d.qpos0[lane];
    double sn, cs;
    sincos(ang, &sn, &cs);
    const double* ax = MDL.d.axis[lane];
    double oc = 1.0 - cs;
    double R[9];
    R[0] = cs + oc * ax[0] * ax[0];         R[1] = oc * ax[0] * ax[1] - sn * ax[2]; R[2] = oc * ax[0] * ax[2] + sn * ax[1];
    R[3] = oc * ax[0] * ax[1] + sn * ax[2]; R[4] = cs + oc * ax[1] * ax[1];         R[5] = oc * ax[1] * ax[2] - sn * ax[0];
    R[6] = oc * ax[0] * ax[2] - sn * ax[1]; R[7] = oc * ax[1] * ax[2] + sn * ax[0]; R[8] = cs + oc * ax[2] * ax[2];
    const double* T = MDL.d.Tmat[lane];
#pragma unroll
    for (int r = 0; r < 3; r++)
#pragma unroll
      for (int c = 0; c < 3; c++) s.lR[lane * 9 + 3 * r + c] = T[3 * r] * R[c] + T[3 * r + 1] * R[3 + c] + T[3 * r + 2] * R[6 + c];
  } else if (lane == CUBE && nba > CUBE) {
    double* q = s.qpos + 15;
    double n = sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
    if (n < MINVAL) { q[0] = 1; q[1] = q[2] = q[3] = 0; } else { double inv = 1.0 / n; q[0] *= inv; q[1] *= inv; q[2] *= inv; q[3] *= inv; }
    quat2mat(s.xmat + CUBE * 9, q);
    s.xpos[CUBE * 3] = s.qpos[12]; s.xpos[CUBE * 3 + 1] = s.qpos[13]; s.xpos[CUBE * 3 + 2] = s.qpos[14];
  }
  __syncwarp();
  // Chain composition with the tree topology compiled in (kTreeParent; mcb_model_create refuses any other tree): lane
  // 3 g + r carries row r of the accumulated rotation and component r of the position in registers, so the six serial
  // arm levels need no shared-memory round trip and no barrier; the four lane groups g recompute the arm redundantly and
  // then branch to the gripper sub-chains 6->7, 8->9, 10, 11.  Every shared-memory offset of the arm is an immediate.
  if (lane < 12) {
    const int g = lane / 3, r = lane - 3 * g;
    double X0 = s.lR[3 * r], X1 = s.lR[3 * r + 1], X2 = s.lR[3 * r + 2], P = MDL.d.Tpos[0][r];
    if (g == 0) { s.xmat[3 * r] = X0; s.xmat[3 * r + 1] = X1; s.xmat[3 * r + 2] = X2; s.xpos[r] = P; }
#pragma unroll
    for (int b = 1; b <= 5; b++) {
      const double* L = s.lR + b * 9;
      const double* t = MDL.d.Tpos[b];
      P = P + X0 * t[0] + X1 * t[1] + X2 * t[2];
      const double n0 = X0 * L[0] + X1 * L[3] + X2 * L[6], n1 = X0 * L[1] + X1 * L[4] + X2 * L[7], n2 = X0 * L[2] + X1 * L[5] + X2 * L[8];
      X0 = n0; X1 = n1; X2 = n2;
      if (g == 0) { s.xmat[b * 9 + 3 * r] = X0; s.xmat[b * 9 + 3 * r + 1] = X1; s.xmat[b * 9 + 3 * r + 2] = X2; s.xpos[b * 3 + r] = P; }
    }
    {
      const int b = g < 2 ? 6 + 2 * g : 8 + g;        // 6, 8, 10, 11: the children of body 5
      const double* L = s.lR + b * 9;
      const double* t = MDL.d.Tpos[b];
      P = P + X0 * t[0] + X1 * t[1] + X2 * t[2];
      const double n0 = X0 * L[0] + X1 * L[3] + X2 * L[6], n1 = X0 * L[1] + X1 * L[4] + X2 * L[7], n2 = X0 * L[2] + X1 * L[5] + X2 * L[8];
      X0 = n0; X1 = n1; X2 = n2;
      s.xmat[b * 9 + 3 * r] = X0; s.xmat[b * 9 + 3 * r + 1] = X1; s.xmat[b * 9 + 3 * r + 2] = X2; s.xpos[b * 3 + r] = P;
    }
    if (g < 2) {
      const int b = 7 + 2 * g;                        // 7 (child of 6), 9 (child of 8)
      const double* L = s.lR + b * 9;
      const double* t = MDL.d.Tpos[b];
      P = P + X0 * t[0] + X1 * t[1] + X2 * t[2];
      const double n0 = X0 * L[0] + X1 * L[3] + X2 * L[6], n1 = X0 * L[1] + X1 * L[4] + X2 * L[7], n2 = X0 * L[2] + X1 * L[5] + X2 * L[8];
      s.xmat[b * 9 + 3 * r] = n0; s.xmat[b * 9 + 3 * r + 1] = n1; s.xmat[b * 9 + 3 * r + 2] = n2; s.xpos[b * 3 + r] = P;
    }
  }
  __syncwarp();
  if (MDL.d.has_weld) {
    // mocap variant: orientation quaternion of the body carrying gripper_tcp, composed along the arm 0..weld_body2 exactly
    // like mj_kinematics (parent * body_quat, * axis-angle, normalise).  The half-angle rotations are computed by the
    // arm lanes in parallel (scratch: s.cinert, written only after fk); lane 0 does the six serial products.
    double* rq = s.cinert;
    if (lane <= MDL.d.weld_body2 && lane < 6) {
      const double ang = s.qpos[lane] - MDL.d.qpos0[lane];
      double sn, cs;
      sincos(0.5 * ang, &sn, &cs);
      const double* ax = MDL.d.axis[lane];
      if (ang == 0) { cs = 1; sn = 0; }
      rq[lane * 4] = cs; rq[lane * 4 + 1] = ax[0] * sn; rq[lane * 4 + 2] = ax[1] * sn; rq[lane * 4 + 3] = ax[2] * sn;
    }
    __syncwarp();
    if (lane == 0) {
      double* mq = s.mocap + 3;      // mj_kinematics normalises data.mocap_quat in place
      double n = sqrt(mq[0] * mq[0] + mq[1] * mq[1] + mq[2] * mq[2] + mq[3] * mq[3]);
      if (n < MINVAL) { mq[0] = 1; mq[1] = mq[2] = mq[3] = 0; } else { const double in = fast_rcp(n); mq[0] *= in; mq[1] *= in; mq[2] *= in; mq[3] *= in; }
      double q[4] = {1, 0, 0, 0};
      const int nb = MDL.d.weld_body2;      // the arm is a chain: body b's parent is b - 1 (kTreeParent)
      for (int b = 0; b <= nb; b++) {
        const double* tq = MDL.d.Tquat[b];
        const double* r = rq + b * 4;
        double t[4] = {q[0] * tq[0] - q[1] * tq[1] - q[2] * tq[2] - q[3] * tq[3], q[0] * tq[1] + q[1] * tq[0] + q[2] * tq[3] - q[3] * tq[2],
                       q[0] * tq[2] - q[1] * tq[3] + q[2] * tq[0] + q[3] * tq[1], q[0] * tq[3] + q[1] * tq[2] - q[2] * tq[1] + q[3] * tq[0]};
        q[0] = t[0] * r[0] - t[1] * r[1] - t[2] * r[2] - t[3] * r[3];
        q[1] = t[0] * r[1] + t[1] * r[0] + t[2] * r[3] - t[3] * r[2];
        q[2] = t[0] * r[2] - t[1] * r[3] + t[2] * r[0] + t[3] * r[1];
        q[3] = t[0] * r[3] + t[1] * r[2] - t[2] * r[1] + t[3] * r[0];
        const double in = fast_rcp(sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]));
        q[0] *= in; q[1] *= in; q[2] *= in; q[3] *= in;
      }
      s.quat5[0] = q[0]; s.quat5[1] = q[1]; s.quat5[2] = q[2]; s.quat5[3] = q[3];
    }
    __syncwarp();
  }
}


// cinert_cdof(): spatial inertia of every (composite) body and motion axis of every dof, both expressed
// about a per-tree reference point (robot: fixed world point; cube: its own centre of mass).
template <class S>
__device__ void cinert_cdof(S& s, const DevModel* __restrict__ m, int lane, int nba, int nva) {
  if (lane < nba) {
    int b = lane;
    const double* R = s.xmat + b * 9;
    const double* ip = MDL.d.ipos[b];
    double com[3], off[3];
#pragma unroll
    for (int r = 0; r < 3; r++) com[r] = s.xpos[b * 3 + r] + R[3 * r] * ip[0] + R[3 * r + 1] * ip[1] + R[3 * r + 2] * ip[2];
    if (b == CUBE) {
#pragma unroll
      for (int r = 0; r < 3; r++) { s.refcube[r] = com[r]; off[r] = 0; }
    } else {
#pragma unroll
      for (int r = 0; r < 3; r++) off[r] = com[r] - MDL.d.ref_robot[r];
    }
    const double* I = MDL.d.inertia[b];  // xx yy zz xy xz yz
    double Ip[6];
    if constexpr (S::HAS_PRM) {          // the cube's inertia and mass scale together (MCB_P_CUBE_MASS)
      const double p = b == CUBE ? s.prm[MCB_P_CUBE_MASS] : 1.0;
#pragma unroll
      for (int k = 0; k < 6; k++) Ip[k] = I[k] * p;
      I = Ip;
    }
    double A[9];                         // A = R * Ib
#pragma unroll
    for (int r = 0; r < 3; r++) {
      A[3 * r + 0] = R[3 * r] * I[0] + R[3 * r + 1] * I[3] + R[3 * r + 2] * I[4];
      A[3 * r + 1] = R[3 * r] * I[3] + R[3 * r + 1] * I[1] + R[3 * r + 2] * I[5];
      A[3 * r + 2] = R[3 * r] * I[4] + R[3 * r + 1] * I[5] + R[3 * r + 2] * I[2];
    }
    double mass = MDL.d.mass[b];
    if constexpr (S::HAS_PRM) { if (b == CUBE) mass = mass * s.prm[MCB_P_CUBE_MASS]; }
    double* ci = s.cinert + b * 10;
    ci[0] = A[0] * R[0] + A[1] * R[1] + A[2] * R[2] + mass * (off[1] * off[1] + off[2] * off[2]);
    ci[1] = A[3] * R[3] + A[4] * R[4] + A[5] * R[5] + mass * (off[0] * off[0] + off[2] * off[2]);
    ci[2] = A[6] * R[6] + A[7] * R[7] + A[8] * R[8] + mass * (off[0] * off[0] + off[1] * off[1]);
    ci[3] = A[0] * R[3] + A[1] * R[4] + A[2] * R[5] - mass * off[0] * off[1];
    ci[4] = A[0] * R[6] + A[1] * R[7] + A[2] * R[8] - mass * off[0] * off[2];
    ci[5] = A[3] * R[6] + A[4] * R[7] + A[5] * R[8] - mass * off[1] * off[2];
    ci[6] = mass * off[0]; ci[7] = mass * off[1]; ci[8] = mass * off[2]; ci[9] = mass;
  }
  if (lane < nva) {
    int j = lane;
    double* cd = s.cdof + j * 6;
    if (j < NH) {
      const double* R = s.xmat + j * 9;  // hinge j belongs to body j
      const double* a = MDL.d.axis[j];
      double ax[3], off[3];
#pragma unroll
      for (int r = 0; r < 3; r++) { ax[r] = R[3 * r] * a[0] + R[3 * r + 1] * a[1] + R[3 * r + 2] * a[2]; off[r] = MDL.d.ref_robot[r] - s.xpos[j * 3 + r]; }
      cd[0] = ax[0]; cd[1] = ax[1]; cd[2] = ax[2];
      cross3(cd + 3, ax, off);
    } else {
      int k = j - 12;
      if (k < 3) {
        cd[0] = cd[1] = cd[2] = 0; cd[3] = (k == 0); cd[4] = (k == 1); cd[5] = (k == 2);
      } else {
        const double* R = s.xmat + CUBE * 9;
        const double* ip = MDL.d.ipos[CUBE];
        double ax[3] = {R[k - 3], R[k], R[k + 3]}, off[3];
#pragma unroll
        for (int r = 0; r < 3; r++) off[r] = R[3 * r] * ip[0] + R[3 * r + 1] * ip[1] + R[3 * r + 2] * ip[2];  // refcube - xpos
        cd[0] = ax[0]; cd[1] = ax[1]; cd[2] = ax[2];
        cross3(cd + 3, ax, off);
      }
    }
  }
  __syncwarp();
}


// Tree walks with the topology compiled in (kTreeParent).  Lane layout of a walk over NC <= 8 components per body:
// group g = lane / 8 follows one gripper sub-chain (g0: 6 -> 7, g1: 8 -> 9, g2: 10, g3: 11), component c = lane % 8;
// all four groups walk the arm 0..5 redundantly, so a root-to-leaf pass is 8 dependent register updates and needs no
// barrier; group 0 stores the arm's results.
// tree_down(): out[b][c] = out[parent][c] + a[b][c] * w[b]   (b = 0..11; root value `root`)
__device__ __forceinline__ void tree_down(double* out, const double* a, const double* w, double root, int lane) {
  const int g = lane >> 3, c = lane & 7;
  if (c < 6) {
    double v = root;
#pragma unroll
    for (int b = 0; b <= 5; b++) {
      v = fma(a[b * 6 + c], w[b], v);
      if (g == 0) out[b * 6 + c] = v;
    }
    const int b6 = g < 2 ? 6 + 2 * g : 8 + g;
    v = fma(a[b6 * 6 + c], w[b6], v);
    out[b6 * 6 + c] = v;
    if (g < 2) { const int b7 = b6 + 1; v = fma(a[b7 * 6 + c], w[b7], v); out[b7 * 6 + c] = v; }
  }
}
// tree_up(): out[b][c] = in[b][c] + sum over the children's out   (b = 11..0)
__device__ __forceinline__ void tree_up(double* out, const double* in, int lane) {
  const int g = lane >> 3, c = lane & 7;
  const int cc = c < 6 ? c : 0;
  const int b6 = g < 2 ? 6 + 2 * g : 8 + g;
  double v = 0;
  if (g < 2) { v = in[(b6 + 1) * 6 + cc]; if (c < 6) out[(b6 + 1) * 6 + c] = v; }
  v += in[b6 * 6 + cc];
  if (c < 6) out[b6 * 6 + c] = v;
  v += shfl_xor_d(v, 8);
  v += shfl_xor_d(v, 16);                       // all groups: sum over the four children of body 5
#pragma unroll
  for (int b = 5; b >= 0; b--) {
    v += in[b * 6 + cc];
    if (g == 0 && c < 6) out[b * 6 + c] = v;
  }
}

// crb_mass(): composite rigid-body inertias (subtree = contiguous DFS range) and the joint-space inertia M
// (packed lower triangle; the robot-cube block is structurally zero and never written).
template <class S>
__device__ void crb_mass(S& s, const DevModel* __restrict__ m, int lane, int nba, int nva) {
  {
    // subtree sums leaf-to-root: lane 10 g + k, g0: 7 -> 6, g1: 9 -> 8, g2: 10 and 11; then the arm 5..0; lanes 30, 31: cube
    const int g = lane / 10, k = lane - 10 * g;
    double v = 0;
    if (g < 2) {
      const int b7 = 7 + 2 * g;
      v = s.cinert[b7 * 10 + k]; s.crb[b7 * 10 + k] = v;
      v += s.cinert[(b7 - 1) * 10 + k]; s.crb[(b7 - 1) * 10 + k] = v;
    } else if (g == 2) {
      const double a = s.cinert[10 * 10 + k], b = s.cinert[11 * 10 + k];
      s.crb[10 * 10 + k] = a; s.crb[11 * 10 + k] = b;
      v = a + b;
    } else if (nba > CUBE) {
#pragma unroll
      for (int q = 0; q < 5; q++) s.crb[CUBE * 10 + 5 * k + q] = s.cinert[CUBE * 10 + 5 * k + q];
    }
    const double v1 = shfl_d(v, (lane + 10) & 31), v2 = shfl_d(v, (lane + 20) & 31);
    if (g == 0) {
      v += v1 + v2;
#pragma unroll
      for (int b = 5; b >= 0; b--) { v += s.cinert[b * 10 + k]; s.crb[b * 10 + k] = v; }
    }
  }
  __syncwarp();
  if (lane < nva) mul_inert_vec(s.buf + lane * 6, s.crb + MDL.d.dof_body[lane] * 10, s.cdof + lane * 6);
  __syncwarp();
  for (int e = lane; e < MDL.nmnz; e += 32) {
    int i = MDL.mnz_i[e], j = MDL.mnz_j[e];
    if (i >= nva) continue;
    const double* a = s.cdof + j * 6;
    const double* b = s.buf + i * 6;
    double v = a[0] * b[0] + a[1] * b[1] + a[2] * b[2] + a[3] * b[3] + a[4] * b[4] + a[5] * b[5];
    if (i == j) v += MDL.d.armature[i];
    s.M[TRI(i, j)] = v;
  }
  __syncwarp();
}

// chol_solve_blk<N0, N, DADD>(): factorisation A = L D L' (unit lower L) of the diagonal block rows/cols [N0, N0+N) of
// a packed symmetric matrix (src -> dst, may alias) AND the solution of A x = b, in one pass.  Lane i owns row i in
// registers as the UNSCALED entries u_ik = l_ik d_k, so a column step is one dot product with the scaled row j of L
// (broadcast from shared memory), one shuffle of the pivot, one reciprocal and one multiply; finished entries
// l_ij = u_ij / d_j go to dst (strict lower triangle; the diagonal slot receives 1).  Lane 31 carries the right-hand
// side (read from the shared vector `bsrc`) as an extra row, so the forward substitution AND the scaling by D^-1 cost
// nothing extra; its entries reach the lanes through the shared scratch `ytmp`; the back substitution with the unit
// triangle is a shuffle + fma chain without divisions.  DADD: `dadd` is added to the lane's diagonal entry first
// (Euler: h * damping).  Pivots below MINVAL are clamped (mju_cholFactor's mindiag).  Lanes outside the block return 0.
// Fully unrolled: every shared-memory offset is an immediate, no index arithmetic in the inner loops.
// Factor storage: row i of L starts at an even offset TRIP(i, 0), so a row segment starting at an even column is 16-byte
// aligned and the dot products read it with 128-bit loads (NTRIP = 180 doubles for 18 rows instead of NTRI = 171).
template <int N0, int N, bool DADD>
__device__ __noinline__ double chol_solve_blk(const double* src, double* dst, const double* bsrc, double* ytmp, double dadd, int lane) {
  const int i = lane;
  const bool mine = (i >= N0 && i < N0 + N);
  const bool rhs = (i == 31);
  const int ro = i * (i + 1) / 2 + N0;
  const double* base = rhs ? bsrc + N0 : src + ro;      // lane 31 loads b, the others their matrix row (packed, TRI)
  double* wbase = rhs ? ytmp + N0 : dst + TRIP(i, N0);  // ... and stores D^-1 L^-1 b, the others their row of L (padded, TRIP)
  const int ieff = (mine || rhs) ? i : -1;              // entry (i, N0 + k) exists for this lane iff ieff >= N0 + k
  double row[N];
#pragma unroll
  for (int k = 0; k < N; k++) {
    double v = (ieff >= N0 + k) ? base[k] : 0.0;
    if (DADD) v += (N0 + k == i) ? dadd : 0.0;     // (a separate "row[i - N0] += dadd" would index row[] dynamically => local memory)
    row[k] = v;
  }
  __syncwarp();                                         // src may alias dst, whose layout differs: every load precedes every store
#pragma unroll
  for (int j = 0; j < N; j++) {
    const double2* rj = reinterpret_cast<const double2*>(dst + TRIP(N0 + j, N0));      // N0 is even => 16-byte aligned
    double s0 = row[j], s1 = 0.0;
#pragma unroll
    for (int k = 0; k + 1 < j; k += 2) { const double2 l2 = rj[k >> 1]; s0 -= row[k] * l2.x; s1 -= row[k + 1] * l2.y; }
    if (j & 1) s0 -= row[j - 1] * reinterpret_cast<const double*>(rj)[j - 1];
    const double sv = s0 + s1;
    row[j] = sv;
    double d = shfl_d(sv, N0 + j);
    d = (d < MINVAL) ? MINVAL : d;                      // (fmax() drags NaN handling along)
    const double l = sv * fast_rcp(d);
    if (ieff >= N0 + j) wbase[j] = l;
    __syncwarp();
  }
  double x = mine ? ytmp[i] : 0.0;
#pragma unroll
  for (int k = N0 + N - 1; k > N0; k--) {
    const double xk = shfl_d(x, k);
    const double lk = (i < k && i >= N0) ? dst[TRIP(k, 0) + i] : 0.0;
    x = fma(-lk, xk, x);
  }
  return x;
}
// factor + solve with the block structure: coupled => one 18 x 18 block, else robot 12 x 12 and cube 6 x 6.
// b is read from the shared vector bsrc; ytmp is an 18-double shared scratch.
__device__ __forceinline__ double factor_solve(const double* src, double* dst, const double* bsrc, double* ytmp, int lane, int nva, bool coupled) {
  if (coupled) return chol_solve_blk<0, 18, false>(src, dst, bsrc, ytmp, 0.0, lane);
  double x = chol_solve_blk<0, 12, true>(src, dst, bsrc, ytmp, 0.0, lane);
  if (nva > NH) { double xc = chol_solve_blk<12, 6, false>(src, dst, bsrc, ytmp, 0.0, lane); if (lane >= NH) x = xc; }
  return x;
}
// the same for M and M + h*diag(damping): the free cube's block of M is diagonal (rotational dofs are expressed in
// the body's principal frame about its centre of mass), so cube lanes just divide
template <bool DADD>
__device__ __forceinline__ double factor_solve_M(const double* M, double* dst, const double* bsrc, double* ytmp, double dadd, int lane, int nva) {
  double x = chol_solve_blk<0, 12, DADD>(M, dst, bsrc, ytmp, dadd, lane);
  if (lane >= NH && lane < nva) x = bsrc[lane] * fast_rcp(M[TRI(lane, 0) + lane] + dadd);
  return x;
}
// y_i = sum_j M_ij v_j for the lane's row (block diagonal: robot lanes see columns 0..11, cube lanes 12..17)
template <class S>
__device__ __noinline__ double mulM_row(const S& s, int lane, int nva, const double* v) {
  double acc = 0, a1 = 0, a2 = 0;
  const int ro = lane * (lane + 1) / 2;
  if (lane < NH) {
#pragma unroll
    for (int j = 0; j < NH; j += 3) {
      acc += s.M[j <= lane ? ro + j : TRI(j, 0) + lane] * v[j];
      a1 += s.M[j + 1 <= lane ? ro + j + 1 : TRI(j + 1, 0) + lane] * v[j + 1];
      a2 += s.M[j + 2 <= lane ? ro + j + 2 : TRI(j + 2, 0) + lane] * v[j + 2];
    }
  } else if (lane < nva) {
#pragma unroll
    for (int j = NH; j < NV; j += 3) {
      acc += s.M[j <= lane ? ro + j : TRI(j, 0) + lane] * v[j];
      a1 += s.M[j + 1 <= lane ? ro + j + 1 : TRI(j + 1, 0) + lane] * v[j + 1];
      a2 += s.M[j + 2 <= lane ? ro + j + 2 : TRI(j + 2, 0) + lane] * v[j + 2];
    }
  }
  return acc + a1 + a2;
}

// ------------------------------------------------------------------------------------------------
// collision: narrow phase for the statically filtered primitive pairs, one lane per pair
// Narrow phase, warp-cooperative: the candidate pairs that pass the bounding-sphere test are processed one
// after the other by the whole warp, all scratch in shared memory (the dead dynamics union).  Contacts are
// appended to s.cdist / cpos / cframe / cpair in pair order.
//
// scratch layout (doubles) inside s.cscr[]
#define CS_P1 0
#define CS_P2 3
#define CS_S1 6
#define CS_S2 9
#define CS_A 12     // A[i][k]: axis i of box 1 (column i of its rotation), row-major 3x3
#define CS_B 21
#define CS_C 30     // C[i][j] = A_i . B_j
#define CS_SP 39    // separation along the 15 candidate axes
#define CS_T 54     // signed centre distance along the axis
#define CS_PX 69
#define CS_PY 85
#define CS_QX 101
#define CS_QY 117
#define CS_R1 133
#define CS_R2 142
#define CS_N 151

template <class S>
__device__ __forceinline__ void emit_contact(S& s, int idx, int pair, double dist, const double* pos, const double* nrm) {
  s.cdist[idx] = dist;
  s.cpair[idx] = pair;
  double f[9];
  f[0] = nrm[0]; f[1] = nrm[1]; f[2] = nrm[2];
  // mju_makeFrame
  double nn = sqrt(dot3(f, f));
  if (nn < MINVAL) { f[0] = 1; f[1] = f[2] = 0; } else { const double in = fast_rcp(nn); f[0] *= in; f[1] *= in; f[2] *= in; }
  f[3] = f[4] = f[5] = 0;
  if (f[1] < 0.5 && f[1] > -0.5) f[4] = 1; else f[5] = 1;
  double t = dot3(f, f + 3);
  f[3] -= t * f[0]; f[4] -= t * f[1]; f[5] -= t * f[2];
  nn = sqrt(dot3(f + 3, f + 3));
  if (nn < MINVAL) { f[3] = 1; f[4] = f[5] = 0; } else { const double in = fast_rcp(nn); f[3] *= in; f[4] *= in; f[5] *= in; }
  cross3(f + 6, f, f + 3);
#pragma unroll
  for (int k = 0; k < 9; k++) s.cframe[idx * 9 + k] = f[k];
#pragma unroll
  for (int k = 0; k < 3; k++) s.cpos[idx * 3 + k] = pos[k];
}

// world pose of geom g into the shared scratch: lanes [l0, l0+12) write the 9 matrix and 3 position entries
template <class S>
__device__ __forceinline__ void geom_pose(S& s, int g, int lane, int l0, double* pos, double* mat) {
  int e = lane - l0;
  if (e < 0 || e >= 12) return;
  int b = MDL.d.geom_body[g];
  const double* gp = MDL.d.geom_pos[g];
  const double* gm = MDL.d.geom_mat[g];
  if (e < 9) {
    int r = e / 3, c = e % 3;
    double v;
    if (b < 0) v = gm[e];
    else { const double* R = s.xmat + b * 9; v = R[3 * r] * gm[c] + R[3 * r + 1] * gm[3 + c] + R[3 * r + 2] * gm[6 + c]; }
    mat[e] = v;
  } else {
    int r = e - 9;
    double v;
    if (b < 0) v = gp[r];
    else { const double* R = s.xmat + b * 9; v = s.xpos[b * 3 + r] + R[3 * r] * gp[0] + R[3 * r + 1] * gp[1] + R[3 * r + 2] * gp[2]; }
    pos[r] = v;
  }
}

// mjc_PlaneBox: corners below the plane, the first four in corner order.  Lanes 0..7 = corners.
template <class S>
__device__ int plane_box_coop(S& s, int lane, int pair, int ncon, const double* ppos, const double* pmat, const double* bpos, const double* bmat, const double* bsize) {
  double norm[3] = {pmat[2], pmat[5], pmat[8]}, dif[3] = {bpos[0] - ppos[0], bpos[1] - ppos[1], bpos[2] - ppos[2]};
  double dist = dot3(dif, norm);
  int i = lane & 7;
  double vec[3] = {(i & 1 ? bsize[0] : -bsize[0]), (i & 2 ? bsize[1] : -bsize[1]), (i & 4 ? bsize[2] : -bsize[2])};
  double corner[3];
#pragma unroll
  for (int r = 0; r < 3; r++) corner[r] = bmat[3 * r] * vec[0] + bmat[3 * r + 1] * vec[1] + bmat[3 * r + 2] * vec[2];
  double ldist = dot3(norm, corner);
  bool hit = lane < 8 && !(dist + ldist > 0 || ldist > 0);
  unsigned bal = __ballot_sync(FULLMASK, hit);
  int rank = __popc(bal & ((1u << lane) - 1));
  int total = __popc(bal);
  if (total > 4) total = 4;
  if (hit && rank < 4 && ncon + rank < S::MAXC) {
    double cd = dist + ldist, pos[3];
#pragma unroll
    for (int k = 0; k < 3; k++) pos[k] = corner[k] + bpos[k] - norm[k] * cd * 0.5;
    emit_contact(s, ncon + rank, pair, cd, pos, norm);
  }
  return ncon + total;
}

// box_box_coop(): 15-axis separating-axis test (one lane per axis), then a clipped face manifold (<= 8 points,
// Sutherland-Hodgman with one lane per polygon edge) or one edge-edge point.  Normal points from box 1 to box 2.
// Degenerate ties: first face axis wins (a later axis must be better by 1e-10), an edge axis must beat the faces
// by 5%.  Same arithmetic and the same discrete choices as the oracle's box_box().
template <class S>
__device__ int box_box_coop(S& s, int lane, int pair, int ncon, const double* p1, const double* R1, const double* s1, const double* p2, const double* R2, const double* s2) {
  double* cs = s.cscr;
  if (lane < 9) { int i = lane / 3, k = lane % 3; cs[CS_A + lane] = R1[3 * k + i]; cs[CS_B + lane] = R2[3 * k + i]; }   // R1, R2, p1, p2 are in the scratch
  if (lane < 3) { cs[CS_S1 + lane] = s1[lane]; cs[CS_S2 + lane] = s2[lane]; }
  __syncwarp();
  if (lane < 9) { int i = lane / 3, j = lane % 3; cs[CS_C + lane] = dot3(cs + CS_A + 3 * i, cs + CS_B + 3 * j); }
  __syncwarp();
  const double d[3] = {p2[0] - p1[0], p2[1] - p1[1], p2[2] - p1[2]};
  // --- one candidate axis per lane
  {
    double sp = -1e300, t = 0;
    if (lane < 3) {
      int i = lane;
      t = dot3(d, cs + CS_A + 3 * i);
      sp = fabs(t) - (cs[CS_S1 + i] + s2[0] * fabs(cs[CS_C + 3 * i]) + s2[1] * fabs(cs[CS_C + 3 * i + 1]) + s2[2] * fabs(cs[CS_C + 3 * i + 2]));
    } else if (lane < 6) {
      int j = lane - 3;
      t = dot3(d, cs + CS_B + 3 * j);
      sp = fabs(t) - (cs[CS_S2 + j] + s1[0] * fabs(cs[CS_C + j]) + s1[1] * fabs(cs[CS_C + 3 + j]) + s1[2] * fabs(cs[CS_C + 6 + j]));
    } else if (lane < 15) {
      int i = (lane - 6) / 3, j = (lane - 6) % 3;
      double Lx[3];
      cross3(Lx, cs + CS_A + 3 * i, cs + CS_B + 3 * j);
      double l = sqrt(dot3(Lx, Lx));
      if (l >= 1e-6) {
        { const double il = fast_rcp(l); for (int k = 0; k < 3; k++) Lx[k] *= il; }   // (x / l with x == 0 takes div.rn.f64's slow path)
        t = dot3(d, Lx);
        double ra = 0, rb = 0;
        for (int k = 0; k < 3; k++) { ra += s1[k] * fabs(dot3(cs + CS_A + 3 * k, Lx)); rb += s2[k] * fabs(dot3(cs + CS_B + 3 * k, Lx)); }
        sp = fabs(t) - (ra + rb);
      }
    }
    if (lane < 15) { cs[CS_SP + lane] = sp; cs[CS_T + lane] = t; }
    if (__any_sync(FULLMASK, lane < 15 && sp > 0)) return ncon;   // separated (a degenerate edge axis has sp = -1e300)
  }
  __syncwarp();
  // --- sequential choice of the axis (uniform)
  double best = -1e300; int code = -1;
  for (int a = 0; a < 3; a++) { double sp = cs[CS_SP + a]; if (sp > best + (code >= 0 ? 1e-10 : 0.0)) { best = sp; code = a; } }
  for (int a = 3; a < 6; a++) { double sp = cs[CS_SP + a]; if (sp > best + 1e-10) { best = sp; code = a; } }
  for (int a = 6; a < 15; a++) { double sp = cs[CS_SP + a]; if (sp > -1e299 && sp * 1.05 > best + 1e-10 && sp > best) { best = sp; code = a; } }
  if (code < 0) return ncon;
  const double tsel = cs[CS_T + code];
  double bn[3];
  if (code >= 6) {
    int i = (code - 6) / 3, j = (code - 6) % 3;
    const double* Ai = cs + CS_A + 3 * i;
    const double* Bj = cs + CS_B + 3 * j;
    double Lx[3];
    cross3(Lx, Ai, Bj);
    double l = sqrt(dot3(Lx, Lx));
    for (int k = 0; k < 3; k++) { Lx[k] /= l; bn[k] = (tsel < 0 ? -Lx[k] : Lx[k]); }
    double pa[3] = {p1[0], p1[1], p1[2]}, pb[3] = {p2[0], p2[1], p2[2]};
    for (int a = 0; a < 3; a++) {
      if (a == i) continue;
      const double* Aa = cs + CS_A + 3 * a;
      double sg = dot3(Aa, bn) > 0 ? 1.0 : -1.0;
      for (int k = 0; k < 3; k++) pa[k] += sg * cs[CS_S1 + a] * Aa[k];
    }
    for (int b = 0; b < 3; b++) {
      if (b == j) continue;
      const double* Bb = cs + CS_B + 3 * b;
      double sg = dot3(Bb, bn) > 0 ? -1.0 : 1.0;
      for (int k = 0; k < 3; k++) pb[k] += sg * cs[CS_S2 + b] * Bb[k];
    }
    double w[3] = {pa[0] - pb[0], pa[1] - pb[1], pa[2] - pb[2]};
    double b_ = cs[CS_C + 3 * i + j], dd = dot3(Ai, w), e = dot3(Bj, w);
    double den = 1 - b_ * b_;
    double u = (b_ * e - dd) / den, v = (e - b_ * dd) / den;
    double pos[3];
    for (int k = 0; k < 3; k++) { double ca = pa[k] + u * Ai[k], cb = pb[k] + v * Bj[k]; pos[k] = 0.5 * (ca + cb); }
    if (lane == 0 && ncon < S::MAXC) emit_contact(s, ncon, pair, best, pos, bn);
    return ncon + 1;
  }
  // --- face contact: reference box owns the axis
  const bool ref1 = code < 3;
  const int ax = ref1 ? code : code - 3;
  const double* Ar = cs + (ref1 ? CS_A : CS_B);
  const double* Ai = cs + (ref1 ? CS_B : CS_A);
  const double* pr = cs + (ref1 ? CS_P1 : CS_P2);
  const double* pi_ = cs + (ref1 ? CS_P2 : CS_P1);
  const double* sr = cs + (ref1 ? CS_S1 : CS_S2);
  const double* si = cs + (ref1 ? CS_S2 : CS_S1);
  {
    const double* axv = Ar + 3 * ax;
    for (int k = 0; k < 3; k++) bn[k] = (tsel < 0 ? -axv[k] : axv[k]);
  }
  double nref[3];
  for (int k = 0; k < 3; k++) nref[k] = ref1 ? bn[k] : -bn[k];
  int ia = 0; double bestd = -1;
  for (int a = 0; a < 3; a++) { double v = fabs(dot3(Ai + 3 * a, nref)); if (v > bestd) { bestd = v; ia = a; } }
  const double isg = dot3(Ai + 3 * ia, nref) > 0 ? -1.0 : 1.0;
  const int i1 = (ia + 1) % 3, i2 = (ia + 2) % 3, r1 = (ax + 1) % 3, r2 = (ax + 2) % 3;
  const double* Ai1 = Ai + 3 * i1; const double* Ai2 = Ai + 3 * i2; const double* Ar1 = Ar + 3 * r1; const double* Ar2 = Ar + 3 * r2;
  double fc[3];
  for (int k = 0; k < 3; k++) fc[k] = pi_[k] + isg * si[ia] * Ai[3 * ia + k] - pr[k];
  if (lane < 4) {
    const double sg0 = (lane == 0 || lane == 3) ? 1.0 : -1.0, sg1 = (lane < 2) ? 1.0 : -1.0;
    double vz[3];
    for (int k = 0; k < 3; k++) vz[k] = fc[k] + sg0 * si[i1] * Ai1[k] + sg1 * si[i2] * Ai2[k];
    cs[CS_PX + lane] = dot3(vz, Ar1); cs[CS_PY + lane] = dot3(vz, Ar2);
  }
  __syncwarp();
  // Sutherland-Hodgman against |x| <= hx, |y| <= hy: lane i handles the polygon edge (i, i+1)
  const double hx = sr[r1], hy = sr[r2];
  int n = 4;
  // the common case (the cube resting on the table, a pad flat on the cube): all four vertices of the incident face pass all four
  // half-plane tests, so every clipping pass would copy the polygon unchanged -- skip the passes (same tests, same tolerance)
  bool allin;
  {
    bool in = true;
    if (lane < 4) { const double x = cs[CS_PX + lane], y = cs[CS_PY + lane]; in = (hx - x >= -1e-12) && (hx + x >= -1e-12) && (hy - y >= -1e-12) && (hy + y >= -1e-12); }
    allin = __all_sync(FULLMASK, in);
  }
  for (int side = 0; side < (allin ? 0 : 4); side++) {
    const double* px = cs + ((side & 1) ? CS_QX : CS_PX);
    const double* py = cs + ((side & 1) ? CS_QY : CS_PY);
    double* qx = cs + ((side & 1) ? CS_PX : CS_QX);
    double* qy = cs + ((side & 1) ? CS_PY : CS_QY);
    int emit = 0; double ax_ = 0, ay_ = 0, ix = 0, iy = 0; bool keep = false, crossing = false;
    if (lane < n) {
      int j = (lane + 1 == n) ? 0 : lane + 1;
      ax_ = px[lane]; ay_ = py[lane];
      double bx = px[j], by = py[j], da, db;
      if (side == 0) { da = hx - ax_; db = hx - bx; }
      else if (side == 1) { da = hx + ax_; db = hx + bx; }
      else if (side == 2) { da = hy - ay_; db = hy - by; }
      else { da = hy + ay_; db = hy + by; }
      // a vertex within 1e-12 of the clip line counts as inside (an incident edge that coincides with the reference face's border
      // would otherwise be cut at a point chosen by rounding noise; see clip_poly in the oracle)
      keep = da >= -1e-12;
      crossing = keep != (db >= -1e-12);
      if (crossing) { double t = da / (da - db); ix = ax_ + t * (bx - ax_); iy = ay_ + t * (by - ay_); }
      emit = (keep ? 1 : 0) + (crossing ? 1 : 0);
    }
    int incl = emit;
#pragma unroll
    for (int o = 1; o < 16; o <<= 1) { int t = __shfl_up_sync(FULLMASK, incl, o); if (lane >= o) incl += t; }
    int base = incl - emit;
    int total = __shfl_sync(FULLMASK, incl, 15);
    if (keep) { qx[base] = ax_; qy[base] = ay_; base++; }
    if (crossing) { qx[base] = ix; qy[base] = iy; }
    n = total;
    __syncwarp();
    if (n == 0) return ncon;
  }
  // after four sides the polygon is back in PX / PY
  const double o_n = dot3(fc, nref);
  const double u1 = dot3(Ai1, nref), u2 = dot3(Ai2, nref);
  const double a11 = dot3(Ai1, Ar1), a12 = dot3(Ai1, Ar2), a21 = dot3(Ai2, Ar1), a22 = dot3(Ai2, Ar2);
  const double det = a11 * a22 - a12 * a21;
  const double fx = dot3(fc, Ar1), fy = dot3(fc, Ar2);
  bool valid = false; double depth = 0, pt[3] = {0, 0, 0};
  if (lane < n && lane < 16) {
    double x = cs[CS_PX + lane], y = cs[CS_PY + lane];
    double dx = x - fx, dy = y - fy, h;
    if (fabs(det) > 1e-12) {
      const double idet = det < 0 ? -fast_rcp(-det) : fast_rcp(det);
      double al = (dx * a22 - dy * a21) * idet, be = (dy * a11 - dx * a12) * idet;
      h = o_n + al * u1 + be * u2;
    } else h = o_n;
    depth = sr[ax] - h;
    valid = !(-depth >= 0);
    for (int k = 0; k < 3; k++) pt[k] = pr[k] + x * Ar1[k] + y * Ar2[k] + (h + 0.5 * depth) * nref[k];
  }
  // duplicates: a point within 1e-10 of an earlier penetrating point is dropped
  bool dup = false;
  // (an unclipped face with edges longer than 2e-9 has four vertices that are pairwise farther apart than the 1e-10 test radius)
  const bool distinct = allin && si[i1] > 1e-9 && si[i2] > 1e-9;
  for (int e = 0; e < (distinct ? 0 : 15); e++) {
    double ex = __shfl_sync(FULLMASK, pt[0], e), ey = __shfl_sync(FULLMASK, pt[1], e), ez = __shfl_sync(FULLMASK, pt[2], e);
    int ev = __shfl_sync(FULLMASK, (int)valid, e);
    if (e < lane && ev) { double qx_ = pt[0] - ex, qy_ = pt[1] - ey, qz_ = pt[2] - ez; if (qx_ * qx_ + qy_ * qy_ + qz_ * qz_ < 1e-20) dup = true; }
    if (e + 1 >= n) break;
  }
  bool take = valid && !dup;
  unsigned bal = __ballot_sync(FULLMASK, take);
  int rank = __popc(bal & ((1u << lane) - 1));
  int total = __popc(bal);
  if (total > 8) total = 8;
  if (take && rank < 8 && ncon + rank < S::MAXC) emit_contact(s, ncon + rank, pair, -depth, pt, bn);
  return ncon + total;
}


// ------------------------------------------------------------------------------------------------
// Convex hulls (mesh geoms): mjc_Convex / mjc_PlaneConvex.  MuJoCo hands hull pairs to libccd's ccdMPRPenetration (Minkowski
// Portal Refinement, tolerance 1e-6, 50 iterations) with support mappings over the hull vertices / box corners and the geom
// centres as interior points; one contact per pair.  The portal algebra is scalar and runs uniformly on every lane (the portal
// lives in the collision scratch, reads are broadcasts); the support mapping is the parallel part: lanes stride over the hull's
// vertices in global memory and an arg-max butterfly picks the winner (lowest index on ties, like the oracle's first maximum).
#define HS_CEN 0        // world centres of the hulls [MCB_MAXHULL][3]
#define HS_P 48         // portal: 4 points x (v, v1, v2)
#define HS_V4 84        // candidate point (v, v1, v2)
#define CCD_EPS 2.220446049250313e-16
#define HS_POSE 96      // world poses (pos 3, mat 9) of the pair's two vertex frames: kept in the scratch, not on the threads' stacks
struct CvxObj { int kind; int body; const double* verts; int n; const double* size; const double *pos, *mat; };   // kind 0 hull, 1 box; pos / mat: world pose of the vertex frame

template <class S>
__device__ void cvx_support(const S& s, const CvxObj& o, const double* dir, double* out, int lane) {
  double ld[3], best[3];
#pragma unroll
  for (int k = 0; k < 3; k++) ld[k] = o.mat[k] * dir[0] + o.mat[3 + k] * dir[1] + o.mat[6 + k] * dir[2];
  if (o.kind == 1) {
#pragma unroll
    for (int k = 0; k < 3; k++) best[k] = ld[k] >= -1e-11 ? o.size[k] : -o.size[k];      // components within 1e-11 of zero count as positive (see the oracle)
  } else {
    // the lowest-index vertex within 1e-11 of the maximum (two passes): coplanar hull vertices tie up to rounding, see the oracle
    // (both scans are written without early exits and unrolled, so that several vertex loads are in flight: the vertices come
    // from global memory / L2 and a hull has up to 1531 of them)
    double bd = -1e300;
#pragma unroll 4
    for (int i = lane; i < o.n; i += 32) {
      const double* v = o.verts + 3 * i;
      const double t = v[0] * ld[0] + v[1] * ld[1] + v[2] * ld[2];
      bd = t > bd ? t : bd;
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) { const double od = shfl_xor_d(bd, off); if (od > bd) bd = od; }
    int bi = 0x7fffffff;
    const double thr = bd - 1e-11;
#pragma unroll 4
    for (int i = lane; i < o.n; i += 32) {
      const double* v = o.verts + 3 * i;
      const double t = v[0] * ld[0] + v[1] * ld[1] + v[2] * ld[2];
      bi = (t >= thr && i < bi) ? i : bi;
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) { const int oi = __shfl_xor_sync(FULLMASK, bi, off); if (oi < bi) bi = oi; }
    const double* v = o.verts + 3 * bi;
    best[0] = v[0]; best[1] = v[1]; best[2] = v[2];
  }
#pragma unroll
  for (int r = 0; r < 3; r++) out[r] = o.pos[r] + o.mat[3 * r] * best[0] + o.mat[3 * r + 1] * best[1] + o.mat[3 * r + 2] * best[2];
}
// support of the Minkowski difference A - B into a 9-double slot (v, v1, v2) of the scratch
template <class S>
__device__ void mpr_support(S& s, const CvxObj& A, const CvxObj& B, const double* dir, double* slot, int lane) {
  double nd[3] = {-dir[0], -dir[1], -dir[2]}, p1[3], p2[3];
  cvx_support(s, A, dir, p1, lane);
  cvx_support(s, B, nd, p2, lane);
  __syncwarp();
  if (lane == 0) { for (int k = 0; k < 3; k++) { slot[k] = p1[k] - p2[k]; slot[3 + k] = p1[k]; slot[6 + k] = p2[k]; } }
  __syncwarp();
}
__device__ __forceinline__ bool ccd_zero(double x) { return fabs(x) < CCD_EPS; }
__device__ __forceinline__ bool ccd_eq(double a, double b) {
  double ab = fabs(a - b);
  if (ab < CCD_EPS) return true;
  a = fabs(a); b = fabs(b);
  return b > a ? ab < CCD_EPS * b : ab < CCD_EPS * a;
}
__device__ __forceinline__ void normalize3_d(double* v) {
  const double n = sqrt(dot3(v, v));
  if (n < MINVAL) { v[0] = 1; v[1] = 0; v[2] = 0; } else { v[0] /= n; v[1] /= n; v[2] /= n; }
}
__device__ __forceinline__ void copy9(double* d, const double* sarr, int lane) { __syncwarp(); if (lane < 9) d[lane] = sarr[lane]; __syncwarp(); }
__device__ __forceinline__ void portal_dir(const double* P, double* dir) {
  double a[3], b[3];
  for (int k = 0; k < 3; k++) { a[k] = P[18 + k] - P[9 + k]; b[k] = P[27 + k] - P[9 + k]; }
  cross3(dir, a, b);
  normalize3_d(dir);
}
__device__ __forceinline__ bool portal_reach_tol(const double* P, const double* v4, const double* dir, double tol) {
  const double dv4 = dot3(v4, dir);
  double d1 = dv4 - dot3(P + 9, dir), d2 = dv4 - dot3(P + 18, dir), d3 = dv4 - dot3(P + 27, dir);
  d1 = fmin(d1, fmin(d2, d3));
  return ccd_eq(d1, tol) || d1 < tol;
}
__device__ __forceinline__ void expand_portal(double* P, const double* v4, int lane) {
  double v4v0[3];
  cross3(v4v0, v4, P);
  int slot;
  if (dot3(P + 9, v4v0) > 0) slot = dot3(P + 18, v4v0) > 0 ? 1 : 3;
  else slot = dot3(P + 27, v4v0) > 0 ? 2 : 1;
  copy9(P + 9 * slot, v4, lane);
}
// squared distance of the origin to triangle (a, b, c), closest point in w (Ericson 5.1.5; same branches as the oracle)
__device__ double origin_tri_dist2(const double* a, const double* b, const double* c, double* w) {
  double ab[3], ac[3], ap[3], bp[3], cp[3];
  for (int k = 0; k < 3; k++) { ab[k] = b[k] - a[k]; ac[k] = c[k] - a[k]; ap[k] = -a[k]; bp[k] = -b[k]; cp[k] = -c[k]; }
  const double d1 = dot3(ab, ap), d2 = dot3(ac, ap), d3 = dot3(ab, bp), d4 = dot3(ac, bp), d5 = dot3(ab, cp), d6 = dot3(ac, cp);
  double u, v;
  if (d1 <= 0 && d2 <= 0) { u = 0; v = 0; }
  else if (d3 >= 0 && d4 <= d3) { u = 1; v = 0; }
  else if (d1 * d4 - d3 * d2 <= 0 && d1 >= 0 && d3 <= 0) { u = d1 / (d1 - d3); v = 0; }
  else if (d6 >= 0 && d5 <= d6) { u = 0; v = 1; }
  else if (d5 * d2 - d1 * d6 <= 0 && d2 >= 0 && d6 <= 0) { u = 0; v = d2 / (d2 - d6); }
  else if (d3 * d6 - d5 * d4 <= 0 && (d4 - d3) >= 0 && (d5 - d6) >= 0) { v = (d4 - d3) / ((d4 - d3) + (d5 - d6)); u = 1 - v; }
  else { const double va = d3 * d6 - d5 * d4, vb = d5 * d2 - d1 * d6, vc = d1 * d4 - d3 * d2, den = 1 / (va + vb + vc); u = vb * den; v = vc * den; }
  for (int k = 0; k < 3; k++) w[k] = a[k] + u * ab[k] + v * ac[k];
  return dot3(w, w);
}
// ccdMPRPenetration: true and (depth, dir from A to B, pos) if the two convex objects intersect.  Uniform on all lanes.
template <class S>
__device__ __noinline__ bool mpr_penetration(S& s, const CvxObj& A, const CvxObj& B, const double* cA, const double* cB, double& depth, double* dir, double* pos, int lane) {
  const double tol = 1e-6; const int maxiter = 50;
  double* P = s.cscr + HS_P;
  double* V4 = s.cscr + HS_V4;
  double d[3], va[3], vb[3], dot;
  __syncwarp();
  if (lane < 3) { P[3 + lane] = cA[lane]; P[6 + lane] = cB[lane]; P[lane] = cA[lane] - cB[lane]; }
  __syncwarp();
  if (ccd_zero(P[0]) && ccd_zero(P[1]) && ccd_zero(P[2])) { __syncwarp(); if (lane == 0) P[0] += CCD_EPS * 10; __syncwarp(); }
  for (int k = 0; k < 3; k++) d[k] = -P[k];
  normalize3_d(d);
  mpr_support(s, A, B, d, P + 9, lane);
  dot = dot3(P + 9, d);
  if (ccd_zero(dot) || dot < 0) return false;
  cross3(d, P, P + 9);
  if (ccd_zero(dot3(d, d))) {
    depth = sqrt(dot3(P + 9, P + 9));
    for (int k = 0; k < 3; k++) { dir[k] = P[9 + k]; pos[k] = 0.5 * (P[12 + k] + P[15 + k]); }
    normalize3_d(dir);
    return true;
  }
  normalize3_d(d);
  mpr_support(s, A, B, d, P + 18, lane);
  dot = dot3(P + 18, d);
  if (ccd_zero(dot) || dot < 0) return false;
  for (int k = 0; k < 3; k++) { va[k] = P[9 + k] - P[k]; vb[k] = P[18 + k] - P[k]; }
  cross3(d, va, vb);
  normalize3_d(d);
  if (dot3(d, P) > 0) {
    __syncwarp();
    double t = 0;
    if (lane < 9) t = P[9 + lane];
    __syncwarp();
    if (lane < 9) { P[9 + lane] = P[18 + lane]; }
    __syncwarp();
    if (lane < 9) P[18 + lane] = t;
    __syncwarp();
    for (int k = 0; k < 3; k++) d[k] = -d[k];
  }
  for (int guard = 0; guard < 100; guard++) {
    mpr_support(s, A, B, d, P + 27, lane);
    dot = dot3(P + 27, d);
    if (ccd_zero(dot) || dot < 0) return false;
    bool cont = false;
    cross3(va, P + 9, P + 27);
    dot = dot3(va, P);
    if (dot < 0 && !ccd_zero(dot)) { copy9(P + 18, P + 27, lane); cont = true; }
    if (!cont) {
      cross3(va, P + 27, P + 18);
      dot = dot3(va, P);
      if (dot < 0 && !ccd_zero(dot)) { copy9(P + 9, P + 27, lane); cont = true; }
    }
    if (!cont) break;
    for (int k = 0; k < 3; k++) { va[k] = P[9 + k] - P[k]; vb[k] = P[18 + k] - P[k]; }
    cross3(d, va, vb);
    normalize3_d(d);
    if (guard == 99) return false;
  }
  for (int guard = 0;; guard++) {                       // refinePortal
    portal_dir(P, d);
    dot = dot3(d, P + 9);
    if (ccd_zero(dot) || dot > 0) break;
    mpr_support(s, A, B, d, V4, lane);
    dot = dot3(V4, d);
    if (!(ccd_zero(dot) || dot > 0) || portal_reach_tol(P, V4, d, tol)) return false;
    expand_portal(P, V4, lane);
    if (guard > 1000) return false;
  }
  for (int it = 0;; it++) {                             // findPenetr
    portal_dir(P, d);
    mpr_support(s, A, B, d, V4, lane);
    if (portal_reach_tol(P, V4, d, tol) || it > maxiter) {
      double w[3];
      depth = sqrt(origin_tri_dist2(P + 9, P + 18, P + 27, w));
      if (ccd_zero(w[0]) && ccd_zero(w[1]) && ccd_zero(w[2])) { for (int k = 0; k < 3; k++) dir[k] = d[k]; depth = 0; }
      else { for (int k = 0; k < 3; k++) dir[k] = w[k]; normalize3_d(dir); }
      double b[4], t[3], sum;
      cross3(t, P + 9, P + 18); b[0] = dot3(t, P + 27);
      cross3(t, P + 27, P + 18); b[1] = dot3(t, P);
      cross3(t, P, P + 9); b[2] = dot3(t, P + 27);
      cross3(t, P + 18, P + 9); b[3] = dot3(t, P);
      sum = b[0] + b[1] + b[2] + b[3];
      if (ccd_zero(sum) || sum < 0) {
        b[0] = 0;
        cross3(t, P + 18, P + 27); b[1] = dot3(t, d);
        cross3(t, P + 27, P + 9); b[2] = dot3(t, d);
        cross3(t, P + 9, P + 18); b[3] = dot3(t, d);
        sum = b[1] + b[2] + b[3];
      }
      const double inv = 1.0 / sum;
      for (int k = 0; k < 3; k++) {
        const double p1 = b[0] * P[3 + k] + b[1] * P[12 + k] + b[2] * P[21 + k] + b[3] * P[30 + k];
        const double p2 = b[0] * P[6 + k] + b[1] * P[15 + k] + b[2] * P[24 + k] + b[3] * P[33 + k];
        pos[k] = 0.5 * (p1 + p2) * inv;
      }
      return true;
    }
    expand_portal(P, V4, lane);
  }
}
// world centres of the hulls into the scratch
template <class S>
__device__ __forceinline__ void hull_centres(S& s, int lane) {
  double* cen = s.cscr + HS_CEN;
  __syncwarp();
  for (int w = lane; w < MDL.nhull * 3; w += 32) {
    const int h = w / 3, r = w - 3 * h, b = MDL.hull_body[h];
    const double* c = MDL.hull_center[h];
    const double* R = s.xmat + b * 9;
    cen[w] = s.xpos[b * 3 + r] + R[3 * r] * c[0] + R[3 * r + 1] * c[1] + R[3 * r + 2] * c[2];
  }
  __syncwarp();
}
// bounding-sphere test of candidate hull pair p (lane-local)
template <class S>
__device__ __forceinline__ bool hull_pair_near(const S& s, int p, int nba) {
  const double* cen = s.cscr + HS_CEN;
  const int oa = MDL.hpair_a[p], ob = MDL.hpair_b[p], hb = ob - MCB_NGEOM;
  if (oa < MCB_NGEOM) {
    const int g = oa, bg = MDL.d.geom_body[g];
    if (nba <= CUBE && bg == CUBE) return false;
    double pg[3];
    const double* gp = MDL.d.geom_pos[g];
    if (bg < 0) { pg[0] = gp[0]; pg[1] = gp[1]; pg[2] = gp[2]; }
    else { const double* R = s.xmat + bg * 9; for (int r = 0; r < 3; r++) pg[r] = s.xpos[bg * 3 + r] + R[3 * r] * gp[0] + R[3 * r + 1] * gp[1] + R[3 * r + 2] * gp[2]; }
    const double dif[3] = {cen[hb * 3] - pg[0], cen[hb * 3 + 1] - pg[1], cen[hb * 3 + 2] - pg[2]};
    if (MDL.d.geom_type[g] == 0) { const double* gm = MDL.d.geom_mat[g]; const double nrm[3] = {gm[2], gm[5], gm[8]}; return dot3(dif, nrm) <= MDL.hull_rbound[hb]; }
    const double bound = MDL.hull_rbound[hb] + MDL.d.geom_rbound[g];
    return dot3(dif, dif) <= bound * bound;
  }
  const int ha = oa - MCB_NGEOM;
  const double dif[3] = {cen[ha * 3] - cen[hb * 3], cen[ha * 3 + 1] - cen[hb * 3 + 1], cen[ha * 3 + 2] - cen[hb * 3 + 2]};
  const double bound = MDL.hull_rbound[ha] + MDL.hull_rbound[hb];
  return dot3(dif, dif) <= bound * bound;
}
// common-layout tier: broad phase only.  An env with any hull pair inside its bounding spheres leaves for the next tier, whose
// kernel carries the narrow phase -- the MPR code (and its registers / stack) stays out of the kernel every env runs first.
template <class S>
__device__ __noinline__ bool hull_any_near(S& s, int lane, int nba) {
  hull_centres(s, lane);
  bool any = false;
  for (int base = 0; base < MDL.nhpair; base += 32) {
    const int p = base + lane;
    any |= (p < MDL.nhpair) && hull_pair_near(s, p, nba);
  }
  return __any_sync(FULLMASK, any);
}
// hull x {plane, box, hull} for the statically filtered pairs, after the primitive pairs (the oracle's order)
template <class S>
__device__ __noinline__ int collide_hulls(S& s, int lane, int nba, int ncon) {
  double* cen = s.cscr + HS_CEN;
  hull_centres(s, lane);
  for (int base = 0; base < MDL.nhpair; base += 32) {
    const int p = base + lane;
    bool near = (p < MDL.nhpair) && hull_pair_near(s, p, nba);
    unsigned todo = __ballot_sync(FULLMASK, near);
    while (todo) {
      const int q = base + __ffs(todo) - 1;
      todo &= todo - 1;
      const int oa = MDL.hpair_a[q], ob = MDL.hpair_b[q], hb = ob - MCB_NGEOM;
      CvxObj A, B;
      double* poseA = s.cscr + HS_POSE;
      double* poseB = s.cscr + HS_POSE + 12;
      B.kind = 0; B.body = MDL.hull_body[hb]; B.verts = MDL.hull_vert + 3 * (size_t)MDL.hull_vadr[hb]; B.n = MDL.hull_vnum[hb]; B.size = nullptr;
      B.pos = s.xpos + B.body * 3; B.mat = s.xmat + B.body * 9;
      A.kind = 0; A.body = -1; A.verts = nullptr; A.n = 0; A.size = nullptr; A.pos = poseA; A.mat = poseA + 3;
      (void)poseB;
      bool hit = false; double dist = 0, nrm[3] = {0, 0, 1}, pos[3] = {0, 0, 0};
      if (oa < MCB_NGEOM && MDL.d.geom_type[oa] == 0) {
        // mjc_PlaneConvex: the hull's support point against the plane normal (planes are static)
        const double* gm = MDL.d.geom_mat[oa];
        const double* gp = MDL.d.geom_pos[oa];
        const double n[3] = {gm[2], gm[5], gm[8]}, nn[3] = {-gm[2], -gm[5], -gm[8]};
        double sp[3];
        cvx_support(s, B, nn, sp, lane);
        const double dif[3] = {sp[0] - gp[0], sp[1] - gp[1], sp[2] - gp[2]};
        dist = dot3(dif, n);
        if (!(dist > 0)) { hit = true; for (int k = 0; k < 3; k++) { nrm[k] = n[k]; pos[k] = sp[k] - 0.5 * dist * n[k]; } }
      } else {
        double cA[3];
        if (oa < MCB_NGEOM) {
          const int g = oa, bg = MDL.d.geom_body[g];
          A.kind = 1; A.body = bg; A.size = MDL.d.geom_size[g];
          const double* gp = MDL.d.geom_pos[g];
          const double* gm = MDL.d.geom_mat[g];
          __syncwarp();
          if (lane < 12) {
            double v;
            if (bg < 0) v = lane < 3 ? gp[lane] : gm[lane - 3];
            else {
              const double* R = s.xmat + bg * 9;
              if (lane < 3) { const int r = lane; v = s.xpos[bg * 3 + r] + R[3 * r] * gp[0] + R[3 * r + 1] * gp[1] + R[3 * r + 2] * gp[2]; }
              else { const int r = (lane - 3) / 3, c = (lane - 3) % 3; v = R[3 * r] * gm[c] + R[3 * r + 1] * gm[3 + c] + R[3 * r + 2] * gm[6 + c]; }
            }
            poseA[lane] = v;
          }
          __syncwarp();
          for (int k = 0; k < 3; k++) cA[k] = poseA[k];
        } else {
          const int ha = oa - MCB_NGEOM;
          A.kind = 0; A.body = MDL.hull_body[ha]; A.verts = MDL.hull_vert + 3 * (size_t)MDL.hull_vadr[ha]; A.n = MDL.hull_vnum[ha];
          A.pos = s.xpos + A.body * 3; A.mat = s.xmat + A.body * 9;
          for (int k = 0; k < 3; k++) cA[k] = cen[ha * 3 + k];
        }
        const double cB[3] = {cen[hb * 3], cen[hb * 3 + 1], cen[hb * 3 + 2]};
        double depth = 0;
        hit = mpr_penetration(s, A, B, cA, cB, depth, nrm, pos, lane);
        dist = -depth;
      }
      if (hit) {
        __syncwarp();
        if (lane == 0 && ncon < S::MAXC) emit_contact(s, ncon, MCB_MAXPAIR + q, dist, pos, nrm);
        ncon++;
        __syncwarp();
      }
    }
  }
  return ncon;
}

template <class S>
__device__ __noinline__ void collide(S& s, int lane, int nba, bool mesh) {
  // broad phase: lane = candidate pair
  bool near = false;
  if (lane < MDL.d.npair) {
    int g1 = MDL.d.pair_g1[lane], g2 = MDL.d.pair_g2[lane];
    int b1 = MDL.d.geom_body[g1], b2 = MDL.d.geom_body[g2];
    if (!((nba <= CUBE) && (b1 == CUBE || b2 == CUBE))) {
      double p1[3], p2[3];
      {
        const double* gp = MDL.d.geom_pos[g1];
        if (b1 < 0) { p1[0] = gp[0]; p1[1] = gp[1]; p1[2] = gp[2]; }
        else { const double* R = s.xmat + b1 * 9; for (int r = 0; r < 3; r++) p1[r] = s.xpos[b1 * 3 + r] + R[3 * r] * gp[0] + R[3 * r + 1] * gp[1] + R[3 * r + 2] * gp[2]; }
        gp = MDL.d.geom_pos[g2];
        if (b2 < 0) { p2[0] = gp[0]; p2[1] = gp[1]; p2[2] = gp[2]; }
        else { const double* R = s.xmat + b2 * 9; for (int r = 0; r < 3; r++) p2[r] = s.xpos[b2 * 3 + r] + R[3 * r] * gp[0] + R[3 * r + 1] * gp[1] + R[3 * r + 2] * gp[2]; }
      }
      double dif[3] = {p2[0] - p1[0], p2[1] - p1[1], p2[2] - p1[2]};
      if (MDL.d.geom_type[g1] == 0) {
        const double* gm = MDL.d.geom_mat[g1];    // planes are static in this model
        double nrm[3] = {gm[2], gm[5], gm[8]};
        near = dot3(dif, nrm) <= MDL.d.geom_rbound[g2];
      } else {
        double bound = MDL.d.geom_rbound[g1] + MDL.d.geom_rbound[g2];
        near = dot3(dif, dif) <= bound * bound;
      }
    }
  }
  unsigned todo = __ballot_sync(FULLMASK, near);
  int ncon = 0;
  while (todo) {
    int p = __ffs(todo) - 1;
    todo &= todo - 1;
    int g1 = MDL.d.pair_g1[p], g2 = MDL.d.pair_g2[p];
    double* p1 = s.cscr + CS_P1; double* p2 = s.cscr + CS_P2; double* R1 = s.cscr + CS_R1; double* R2 = s.cscr + CS_R2;
    geom_pose(s, g1, lane, 0, p1, R1);
    geom_pose(s, g2, lane, 12, p2, R2);
    __syncwarp();
    if (MDL.d.geom_type[g1] == 0) ncon = plane_box_coop(s, lane, p, ncon, p1, R1, p2, R2, MDL.d.geom_size[g2]);
    else ncon = box_box_coop(s, lane, p, ncon, p1, R1, MDL.d.geom_size[g1], p2, R2, MDL.d.geom_size[g2]);
    __syncwarp();
  }
  if (mesh && MDL.nhull > 0) {
    if (S::TIER_ID == 0) { if (hull_any_near(s, lane, nba) && lane == 0) s.overflow += 1; }
    else ncon = collide_hulls(s, lane, nba, ncon);
  }
  if (lane == 0) {
    if (ncon > S::MAXC) { s.overflow += ncon - S::MAXC; ncon = S::MAXC; }
    s.ncon = ncon;
  }
  __syncwarp();
}

// ------------------------------------------------------------------------------------------------
// solimp arrives clamped (mcb_model_create applies getimpedance's limits once: d0, d1, midpoint in [MINIMP, MAXIMP], power >= 1)
// and with slot 2 holding 1 / width (0 for a width <= MINVAL): IEEE divisions are ~30 dependent instructions each and sat in
// series on every row's critical path (pos / width, then 1 / midpoint); reciprocals by fast_rcp() differ by <= 1 ulp.
__device__ double impedance(const double* solimp, double pos) {
  const double s0 = solimp[0], s1 = solimp[1], iw = solimp[2], s3 = solimp[3], s4 = solimp[4];
  if (s0 == s1 || iw == 0.0) return 0.5 * (s0 + s1);
  double x = fabs(pos * iw);
  if (x >= 1 || x <= 0) return (x >= 1 ? s1 : s0);
  double y;
  if (s4 == 1) y = x;
  else if (s4 == 2) { y = (x <= s3) ? fast_rcp(s3) * (x * x) : 1 - fast_rcp(1 - s3) * ((1 - x) * (1 - x)); }   // pow(v, 2) == v * v, pow(v, 1) == v
  else if (x <= s3) { double a = 1 / pow(s3, s4 - 1); y = a * pow(x, s4); }
  else { double b = 1 / pow(1 - s3, s4 - 1); y = 1 - b * pow(1 - x, s4); }
  return s0 + y * (s1 - s0);
}


// point Jacobian column of dof j for a world point attached to body b (0 if j does not move b)
template <class S>
__device__ __forceinline__ void jac_col(const S& s, const DevModel* __restrict__ m, int b, int j, const double* pt, double* lin, double* rot) {
  if (b >= 0 && ((MDL.d.ancmask[b] >> j) & 1u)) {
    const double* cd = s.cdof + j * 6;
    double off[3];
    if (b == CUBE) { off[0] = pt[0] - s.refcube[0]; off[1] = pt[1] - s.refcube[1]; off[2] = pt[2] - s.refcube[2]; }
    else { off[0] = pt[0] - MDL.d.ref_robot[0]; off[1] = pt[1] - MDL.d.ref_robot[1]; off[2] = pt[2] - MDL.d.ref_robot[2]; }
    double t[3];
    cross3(t, cd, off);
    lin[0] = cd[3] + t[0]; lin[1] = cd[4] + t[1]; lin[2] = cd[5] + t[2];
    rot[0] = cd[0]; rot[1] = cd[1]; rot[2] = cd[2];
  } else {
    lin[0] = lin[1] = lin[2] = 0; rot[0] = rot[1] = rot[2] = 0;
  }
}


// row storage of the blocked Jacobian: robot rows [0, nR) x 12, cube rows [nR, nR+nC) x 6, coupled rows x 18,
// then nU joint-limit rows (a signed unit vector each, no storage)
template <class S> __device__ __forceinline__ double* row_r(S& s, int r) { return s.pool + r * SR; }
template <class S> __device__ __forceinline__ double* row_c(S& s, int r) { return s.pool + s.nR * SR + (r - s.nR) * SC; }
template <class S> __device__ __forceinline__ double* row_f(S& s, int r) { return s.pool + s.nR * SR + s.nC * SC + (r - s.nR - s.nC) * SF; }

// dot product of constraint row r with an 18-vector
template <class S>
__device__ __forceinline__ double row_dot(S& s, int r, const double* v) {
  double acc = 0;
  if (r < s.nR) {
    const double* p = row_r(s, r);
    double a1 = 0, a2 = 0, a3 = 0;
#pragma unroll
    for (int k = 0; k < NH; k += 4) { acc += p[k] * v[k]; a1 += p[k + 1] * v[k + 1]; a2 += p[k + 2] * v[k + 2]; a3 += p[k + 3] * v[k + 3]; }
    acc = (acc + a1) + (a2 + a3);
  } else if (r < s.nR + s.nC) {
    const double* p = row_c(s, r);
    double a1 = 0, a2 = 0;
#pragma unroll
    for (int k = 0; k < 6; k += 3) { acc += p[k] * v[NH + k]; a1 += p[k + 1] * v[NH + k + 1]; a2 += p[k + 2] * v[NH + k + 2]; }
    acc = acc + a1 + a2;
  } else if (r < s.nR + s.nC + s.nF) {
    const double* p = row_f(s, r);
    double a1 = 0, a2 = 0;
#pragma unroll
    for (int k = 0; k < NV; k += 3) { acc += p[k] * v[k]; a1 += p[k + 1] * v[k + 1]; a2 += p[k + 2] * v[k + 2]; }
    acc = acc + a1 + a2;
  } else {
    int meta = s.rmeta[r];
    double x = v[meta & 0xff];
    acc = (meta & 0x100) ? -x : x;
  }
  return acc;
}

// two dot products of constraint row r at once (the row is loaded once)
template <class S>
__device__ __forceinline__ void row_dot2(S& s, int r, const double* v, const double* w, double& dv, double& dw) {
  double a0 = 0, a1 = 0, b0 = 0, b1 = 0;
  if (r < s.nR) {
    const double* p = row_r(s, r);
#pragma unroll
    for (int k = 0; k < NH; k += 2) { a0 += p[k] * v[k]; a1 += p[k + 1] * v[k + 1]; b0 += p[k] * w[k]; b1 += p[k + 1] * w[k + 1]; }
  } else if (r < s.nR + s.nC) {
    const double* p = row_c(s, r);
#pragma unroll
    for (int k = 0; k < 6; k += 2) { a0 += p[k] * v[NH + k]; a1 += p[k + 1] * v[NH + k + 1]; b0 += p[k] * w[NH + k]; b1 += p[k + 1] * w[NH + k + 1]; }
  } else if (r < s.nR + s.nC + s.nF) {
    const double* p = row_f(s, r);
#pragma unroll
    for (int k = 0; k < NV; k += 2) { a0 += p[k] * v[k]; a1 += p[k + 1] * v[k + 1]; b0 += p[k] * w[k]; b1 += p[k + 1] * w[k + 1]; }
  } else {
    int meta = s.rmeta[r];
    double x = v[meta & 0xff], y = w[meta & 0xff];
    a0 = (meta & 0x100) ? -x : x; b0 = (meta & 0x100) ? -y : y;
  }
  dv = a0 + a1; dw = b0 + b1;
}

// make_rows(): equality (7 robot rows), pyramidal contact rows by block type, joint-limit unit rows; then R, D
// and the reference acceleration of every row.  Returns false if the layout's capacity is exceeded.
// Sliding friction of a primitive pair under the env's multipliers, mixed like pair_param() (the larger side wins).  Only batches
// without hull collisions have per-env parameters, so every contact's pair is a primitive one.
template <class S>
__device__ __forceinline__ double env_mu(const S& s, const PairParam& pp) {
  return fmax(MDL.d.geom_friction[pp.g1][0] * s.prm[MCB_P_FRICTION + pp.g1], MDL.d.geom_friction[pp.g2][0] * s.prm[MCB_P_FRICTION + pp.g2]);
}

template <class S>
__device__ bool make_rows(S& s, const DevModel* __restrict__ m, int lane, int nva) {
  // connect anchors (lanes 0..3: constraint e = lane>>1, side = lane&1)
  if (lane < 4) {
    int e = lane >> 1, side = lane & 1;
    int b = side ? MDL.d.con_body2[e] : MDL.d.con_body1[e];
    const double* a = side ? MDL.d.con_anchor2[e] : MDL.d.con_anchor1[e];
    const double* R = s.xmat + b * 9;
    for (int r = 0; r < 3; r++) s.anchors[lane * 3 + r] = s.xpos[b * 3 + r] + R[3 * r] * a[0] + R[3 * r + 1] * a[1] + R[3 * r + 2] * a[2];
  }
  // limits: lane j < 12, lower then upper (both can not be active for a positive-width range)
  int lim = 0, neg = 0;
  if (lane < NH && MDL.d.jnt_limited[lane]) {
    double v = s.qpos[lane];
    if (v - MDL.d.jnt_range[lane][0] < 0) lim = 1;
    else if (MDL.d.jnt_range[lane][1] - v < 0) { lim = 1; neg = 1; }
  }
  unsigned bal = __ballot_sync(FULLMASK, lim);
  const int nU = __popc(bal);
  // row bookkeeping: contacts -> groups.  Lane c owns contact c; group sizes and the contacts' first rows are prefix counts
  // over ballots (a contact has 4 or 6 rows); lane 0 only steps in when the layout overflows.
  {
    const int ne0 = MDL.d.has_weld ? 13 : 7;
    int nc = s.ncon;
    int pt = -1, rows = 0;
    if (lane < nc) { const PairParam& pp = PP(s.cpair[lane]); pt = pp.ptype; rows = 2 * (pp.dim - 1); }
    unsigned m0 = __ballot_sync(FULLMASK, pt == 0), m1 = __ballot_sync(FULLMASK, pt == 1), m2 = __ballot_sync(FULLMASK, pt == 2);
    unsigned m6 = __ballot_sync(FULLMASK, rows == 6);
    auto count = [&](unsigned m) { return 4 * __popc(m) + 2 * __popc(m & m6); };
    int nRc = count(m0), nC = count(m1), nF = count(m2), nR = ne0 + nRc;
    bool fits = (nR + nC + nF + nU <= S::NROW) && (nR * SR + nC * SC + nF * SF <= S::POOL);
    if (!fits) {
      // drop contacts from the end until it fits (tiers 0 and 1 abort the env instead, see the kernel)
      if (lane == 0) s.overflow += 1;
      while (nc > 0 && !fits) {
        nc--;
        const unsigned keep = (nc == 0) ? 0u : (FULLMASK >> (32 - nc));
        m0 &= keep; m1 &= keep; m2 &= keep;
        nRc = count(m0); nC = count(m1); nF = count(m2); nR = ne0 + nRc;
        fits = (nR + nC + nF + nU <= S::NROW) && (nR * SR + nC * SC + nF * SF <= S::POOL);
      }
      if (lane == 0) s.ncon = nc;
    }
    if (lane < nc) {
      const unsigned lt = (1u << lane) - 1;
      const unsigned mg = pt == 0 ? m0 : pt == 1 ? m1 : m2;
      const int start = pt == 0 ? ne0 : pt == 1 ? nR : nR + nC;
      s.crow[lane] = start + count(mg & lt);
    }
    if (lane == 0) { s.nR = nR; s.nC = nC; s.nF = nF; s.nU = nU; s.nefc = nR + nC + nF + nU; }
  }
  __syncwarp();
  const int ne0 = MDL.d.has_weld ? 13 : 7, eq0 = ne0 - 7;      // equality rows: [weld (6)] connect (3 + 3) joint coupling (1)
  if (lane < 7) { s.rmeta[eq0 + lane] = lane < 6 ? ((lane / 3) | ((lane % 3) << 9)) : (1 << 12); }
  if (lane < eq0) { s.rmeta[lane] = (lane << 9) | (4 << 12); }
  for (int w = lane; w < s.ncon * 6; w += 32) {
    int c = w / 6, k = w % 6;
    if (k < 2 * (PP(s.cpair[c]).dim - 1)) {
      int r = s.crow[c] + k;
      s.rmeta[r] = c | (k << 9) | (3 << 12) | RM_INEQ;
    }
  }
  __syncwarp();     // cscr aliases the first pool rows, which the equality fill below overwrites
  if (lim) {
    int u = __popc(bal & ((1u << lane) - 1));
    int r = s.nR + s.nC + s.nF + u;
    s.rmeta[r] = lane | (neg << 8) | (2 << 12) | RM_INEQ;
  }
  // equality Jacobian rows (robot block): item = (connect e, dof j) -> its three rows
  for (int w = lane; w < 2 * NH; w += 32) {
    int e = w / NH, j = w % NH;
    double l1[3], l2[3], rt[3];
    jac_col(s, m, MDL.d.con_body1[e], j, s.anchors + (2 * e) * 3, l1, rt);
    jac_col(s, m, MDL.d.con_body2[e], j, s.anchors + (2 * e + 1) * 3, l2, rt);
    s.pool[(eq0 + 3 * e) * SR + j] = l1[0] - l2[0];
    s.pool[(eq0 + 3 * e + 1) * SR + j] = l1[1] - l2[1];
    s.pool[(eq0 + 3 * e + 2) * SR + j] = l1[2] - l2[2];
  }
  if (eq0) {
    // weld between the (static) mocap body and gripper_tcp (mj_instantiateEquality, mjEQ_WELD): residual in s.ik[0..5]
    const int b2 = MDL.d.weld_body2;
    const double* mq = s.mocap + 3;
    const double* rq = MDL.d.weld_relquat;
    double quat[4] = {mq[0] * rq[0] - mq[1] * rq[1] - mq[2] * rq[2] - mq[3] * rq[3], mq[0] * rq[1] + mq[1] * rq[0] + mq[2] * rq[3] - mq[3] * rq[2],
                      mq[0] * rq[2] - mq[1] * rq[3] + mq[2] * rq[0] + mq[3] * rq[1], mq[0] * rq[3] + mq[1] * rq[2] - mq[2] * rq[1] + mq[3] * rq[0]};
    const double n2[4] = {s.quat5[0], -s.quat5[1], -s.quat5[2], -s.quat5[3]};      // neg(q2)
    const double ts = MDL.d.weld_torquescale;
    double p2[3];
    {
      const double* R = s.xmat + b2 * 9;
      const double* a2 = MDL.d.weld_anchor2;
#pragma unroll
      for (int r = 0; r < 3; r++) p2[r] = s.xpos[b2 * 3 + r] + R[3 * r] * a2[0] + R[3 * r + 1] * a2[1] + R[3 * r + 2] * a2[2];
    }
    if (lane == 0) {
      double Rm[9];
      quat2mat(Rm, mq);
      const double* a1 = MDL.d.weld_anchor1;
      for (int r = 0; r < 3; r++) s.ik[r] = (s.mocap[r] + Rm[3 * r] * a1[0] + Rm[3 * r + 1] * a1[1] + Rm[3 * r + 2] * a1[2]) - p2[r];
      double e[4] = {n2[0] * quat[0] - n2[1] * quat[1] - n2[2] * quat[2] - n2[3] * quat[3], n2[0] * quat[1] + n2[1] * quat[0] + n2[2] * quat[3] - n2[3] * quat[2],
                     n2[0] * quat[2] - n2[1] * quat[3] + n2[2] * quat[0] + n2[3] * quat[1], n2[0] * quat[3] + n2[1] * quat[2] - n2[2] * quat[1] + n2[3] * quat[0]};
      for (int r = 0; r < 3; r++) s.ik[3 + r] = ts * e[1 + r];
    }
    if (lane < NH) {
      const int j = lane;
      double lin[3], rot[3];
      jac_col(s, m, b2, j, p2, lin, rot);
      double ax[3] = {-rot[0], -rot[1], -rot[2]};                                      // jacr(mocap) - jacr(tcp), the mocap body is static
      double qa[4] = {-n2[1] * ax[0] - n2[2] * ax[1] - n2[3] * ax[2], n2[0] * ax[0] + n2[2] * ax[2] - n2[3] * ax[1],
                      n2[0] * ax[1] + n2[3] * ax[0] - n2[1] * ax[2], n2[0] * ax[2] + n2[1] * ax[1] - n2[2] * ax[0]};   // mju_mulQuatAxis
      double q3[4] = {qa[0] * quat[0] - qa[1] * quat[1] - qa[2] * quat[2] - qa[3] * quat[3], qa[0] * quat[1] + qa[1] * quat[0] + qa[2] * quat[3] - qa[3] * quat[2],
                      qa[0] * quat[2] - qa[1] * quat[3] + qa[2] * quat[0] + qa[3] * quat[1], qa[0] * quat[3] + qa[1] * quat[2] - qa[2] * quat[1] + qa[3] * quat[0]};
      s.pool[0 * SR + j] = -lin[0]; s.pool[1 * SR + j] = -lin[1]; s.pool[2 * SR + j] = -lin[2];
      s.pool[3 * SR + j] = 0.5 * q3[1] * ts; s.pool[4 * SR + j] = 0.5 * q3[2] * ts; s.pool[5 * SR + j] = 0.5 * q3[3] * ts;
    }
  }
  if (lane < NH) {
    int j = lane;
    double v = 0;
    if (j == MDL.d.jeq_dof1) v = 1;
    if (j == MDL.d.jeq_dof2) {
      double dif = s.qpos[j] - MDL.d.qpos0[j];
      const double* pc = MDL.d.jeq_polycoef;
      v = -(pc[1] + 2 * pc[2] * dif + 3 * pc[3] * dif * dif + 4 * pc[4] * dif * dif * dif);
    }
    s.pool[(eq0 + 6) * SR + j] = v;
  }
  // contact Jacobian rows: items (contact, dof), enumerated per block type so that only owned columns are visited
  const int ncon = s.ncon;
  const int nRc_ = s.nR - ne0;
#pragma unroll 1
  for (int pt = 0; pt < 3; pt++) {
    if ((pt == 0 && nRc_ == 0) || (pt == 1 && s.nC == 0) || (pt == 2 && s.nF == 0)) continue;
    const int ncol = pt == 0 ? NH : pt == 1 ? 6 : NV, j0 = pt == 1 ? NH : 0;
    for (int w = lane; w < ncon * ncol; w += 32) {
      int c = w / ncol, j = j0 + w % ncol;
      const PairParam& pp = PP(s.cpair[c]);
      if (pp.ptype != pt) continue;
      int b1 = pp.b1, b2 = pp.b2;
      const double* pt3 = s.cpos + c * 3;
      const double* f = s.cframe + c * 9;
      double l1[3], r1[3], l2[3], r2[3];
      jac_col(s, m, b1, j, pt3, l1, r1);
      jac_col(s, m, b2, j, pt3, l2, r2);
      double dl[3] = {l2[0] - l1[0], l2[1] - l1[1], l2[2] - l1[2]}, dr[3] = {r2[0] - r1[0], r2[1] - r1[1], r2[2] - r1[2]};
      double Jn = dot3(f, dl), Jt1 = dot3(f + 3, dl), Jt2 = dot3(f + 6, dl), Jr = dot3(f, dr);
      int r0 = s.crow[c];
      double* p; int st;
      if (pt == 0) { p = row_r(s, r0) + j; st = SR; }
      else if (pt == 1) { p = row_c(s, r0) + (j - NH); st = SC; }
      else { p = row_f(s, r0) + j; st = SF; }
      double mu = pp.friction[0];
      if constexpr (S::HAS_PRM) mu = env_mu(s, pp);
      p[0] = Jn + mu * Jt1;
      p[st] = Jn + (-mu) * Jt1;
      p[2 * st] = Jn + mu * Jt2;
      p[3 * st] = Jn + (-mu) * Jt2;
      if (pp.dim == 4) {
        double mt = pp.friction[1];
        p[4 * st] = Jn + mt * Jr;
        p[5 * st] = Jn + (-mt) * Jr;
      }
    }
  }
  __syncwarp();
  // per-row regularisation and reference acceleration (mj_makeImpedance, mj_referenceConstraint)
  const int nefc = s.nefc;
  for (int r = lane; r < nefc; r += 32) {
    int meta = s.rmeta[r], kind = (meta >> 12) & 7, idx = meta & 0xff, sub = (meta >> 9) & 7;
    const double *solimp, *KB;
    double pos, diag, pyr2 = 0, ipos = -1;     // ipos >= 0: the residual norm the row's impedance is evaluated at (getposdim)
    if (kind == 0) {
      const double* a1 = s.anchors + (2 * idx) * 3;
      const double* a2 = a1 + 3;
      pos = a1[sub] - a2[sub];
      const double e0 = a1[0] - a2[0], e1 = a1[1] - a2[1], e2 = a1[2] - a2[2];
      ipos = sqrt(e0 * e0 + e1 * e1 + e2 * e2);
      KB = MDL.d.con_solref[idx]; solimp = MDL.d.con_solimp[idx]; diag = MDL.d.con_diag[idx];
    } else if (kind == 1) {
      int d1 = MDL.d.jeq_dof1, d2 = MDL.d.jeq_dof2;
      double p1 = s.qpos[d1] - MDL.d.qpos0[d1], dif = s.qpos[d2] - MDL.d.qpos0[d2];
      const double* pc = MDL.d.jeq_polycoef;
      pos = p1 - pc[0] - pc[1] * dif - pc[2] * dif * dif - pc[3] * dif * dif * dif - pc[4] * dif * dif * dif * dif;
      KB = MDL.d.jeq_solref; solimp = MDL.d.jeq_solimp; diag = MDL.d.jeq_diag;
    } else if (kind == 4) {
      pos = s.ik[sub];
      ipos = sqrt(s.ik[0] * s.ik[0] + s.ik[1] * s.ik[1] + s.ik[2] * s.ik[2] + s.ik[3] * s.ik[3] + s.ik[4] * s.ik[4] + s.ik[5] * s.ik[5]);
      // all six rows take the translational inverse weight (2.3.2's mj_diagApprox; pinned by the mocap keyframe, see the oracle)
      KB = MDL.d.weld_solref; solimp = MDL.d.weld_solimp; diag = MDL.d.weld_diag[0];
    } else if (kind == 2) {
      double v = s.qpos[idx];
      pos = (meta & 0x100) ? MDL.d.jnt_range[idx][1] - v : v - MDL.d.jnt_range[idx][0];
      KB = MDL.d.jnt_solref[idx]; solimp = MDL.d.jnt_solimp[idx]; diag = MDL.d.dof_invweight0[idx];
    } else {
      const PairParam& pp = PP(s.cpair[idx]);
      double mu = pp.friction[0];
      if constexpr (S::HAS_PRM) mu = env_mu(s, pp);
      pos = s.cdist[idx];
      KB = pp.KB; solimp = pp.solimp;
      diag = pp.tran + mu * mu * pp.tran;     // the pyramid's first-row diagApprox; all rows share R = 2 mu^2 R_first
      pyr2 = pp.pyr2;
      if constexpr (S::HAS_PRM) { const double pyr = mu / sqrt(MDL.d.impratio); pyr2 = 2 * pyr * pyr; }   // pair_param() with multiplicity 1
    }
    double imp = impedance(solimp, ipos >= 0 ? ipos : pos);
    double R = fmax(MINVAL, (1 - imp) * diag * fast_rcp(imp));      // imp in [MINIMP, MAXIMP]
    if (pyr2 > 0) R = pyr2 * R;
    const double K = KB[0], B = KB[1];
    double vel = row_dot(s, r, s.qvel);
    s.eD[r] = fast_rcp(R);
    s.earef[r] = -B * vel - K * imp * pos;
  }
  __syncwarp();
  return s.overflow == 0;
}

// velocity_rne(): cvel, cdof_dot, bias forces (RNE with zero qacc).  PRM kernels with applied forces: qfrc_bias - J' xfrc_applied.
template <class S>
__device__ void velocity_rne(S& s, const DevModel* __restrict__ m, int lane, int nba, int nva) {
  tree_down(s.cvel, s.cdof, s.qvel, 0.0, lane);
  if (nba > CUBE && (lane & 7) >= 6 && lane < 24) {
    const int c = 2 * (lane >> 3) + (lane & 7) - 6;     // the six idle lanes of groups 0..2 take the cube's six components
    double acc = 0;
#pragma unroll
    for (int j = 12; j < 18; j++) acc = fma(s.cdof[j * 6 + c], s.qvel[j], acc);
    s.cvel[CUBE * 6 + c] = acc;
  }
  __syncwarp();
  if (lane < nva) {
    int j = lane;
    double vel[6];
    if (j < NH) {
      int p = MDL.d.parent[j];
      for (int c = 0; c < 6; c++) vel[c] = (p >= 0 ? s.cvel[p * 6 + c] : 0.0);
      cross_motion(s.cdof_dot + j * 6, vel, s.cdof + j * 6);
    } else if (j < 15) {
      for (int c = 0; c < 6; c++) s.cdof_dot[j * 6 + c] = 0;
    } else {
      vel[0] = vel[1] = vel[2] = 0;
      for (int c = 3; c < 6; c++) vel[c] = s.cdof[12 * 6 + c] * s.qvel[12] + s.cdof[13 * 6 + c] * s.qvel[13] + s.cdof[14 * 6 + c] * s.qvel[14];
      cross_motion(s.cdof_dot + j * 6, vel, s.cdof + j * 6);
    }
  }
  __syncwarp();
  {
    const int c8 = lane & 7;
    tree_down(s.cacc, s.cdof_dot, s.qvel, (c8 >= 3 && c8 < 6) ? -MDL.d.gravity[c8 - 3] : 0.0, lane);
    if (nba > CUBE && c8 >= 6 && lane < 24) {
      const int c = 2 * (lane >> 3) + c8 - 6;
      double acc = (c >= 3 ? -MDL.d.gravity[c - 3] : 0.0);
#pragma unroll
      for (int j = 12; j < 18; j++) acc = fma(s.cdof_dot[j * 6 + c], s.qvel[j], acc);
      s.cacc[CUBE * 6 + c] = acc;
    }
  }
  __syncwarp();
  double f[6];
  if (lane < nba) {
    double t[6], t1[6];
    mul_inert_vec(f, s.cinert + lane * 10, s.cacc + lane * 6);
    mul_inert_vec(t, s.cinert + lane * 10, s.cvel + lane * 6);
    cross_force(t1, s.cvel + lane * 6, t);
    for (int c = 0; c < 6; c++) f[c] += t1[c];
  }
  if constexpr (S::HAS_PRM) {
    // xfrc_applied (mj_xfrcAccumulate): the world wrench at the body's centre of mass joins the body's force as the spatial force
    // about its tree's reference point, with the opposite sign; tree_up and the cdof projection below then give qfrc_bias - J' xfrc
    const double* fr = s.frc;
    if (fr && lane < nba) {
      const double* w = fr + NV + lane * 6;
      double off[3] = {0.0, 0.0, 0.0};   // the cube's reference point is its centre of mass
      if (lane != CUBE) {
        const double* R = s.xmat + lane * 9;
        const double* ip = MDL.d.ipos[lane];
#pragma unroll
        for (int r = 0; r < 3; r++) off[r] = s.xpos[lane * 3 + r] + R[3 * r] * ip[0] + R[3 * r + 1] * ip[1] + R[3 * r + 2] * ip[2] - MDL.d.ref_robot[r];
      }
      double tq[3];
      cross3(tq, off, w);
      f[0] -= w[3] + tq[0]; f[1] -= w[4] + tq[1]; f[2] -= w[5] + tq[2];
      f[3] -= w[0]; f[4] -= w[1]; f[5] -= w[2];
    }
  }
  __syncwarp();
  if (lane < nba) for (int c = 0; c < 6; c++) s.cacc[lane * 6 + c] = f[c];  // cacc now holds cfrc_body
  __syncwarp();
  tree_up(s.cvel, s.cacc, lane);    // cvel now holds the subtree-accumulated cfrc
  if (nba > CUBE && (lane & 7) >= 6 && lane < 24) { const int c = 2 * (lane >> 3) + (lane & 7) - 6; s.cvel[CUBE * 6 + c] = s.cacc[CUBE * 6 + c]; }
  __syncwarp();
  if (lane < nva) {
    const double* a = s.cdof + lane * 6;
    const double* b = s.cvel + MDL.d.dof_body[lane] * 6;
    s.qfrc_bias[lane] = a[0] * b[0] + a[1] * b[1] + a[2] * b[2] + a[3] * b[3] + a[4] * b[4] + a[5] * b[5];
  }
  __syncwarp();
}

// joint damping of dof j under the env's multipliers: the arm's six hinges scale with MCB_P_ARM_DAMPING
template <class S>
__device__ __forceinline__ double env_damping(const S& s, int j) {
  return j < 6 ? MDL.d.damping[j] * s.prm[MCB_P_ARM_DAMPING] : MDL.d.damping[j];
}

// actuation_smooth(): affine PD "general" actuators with ctrl and force clamps, passive damping; qfrc_smooth.
template <class S>
__device__ void actuation_smooth(S& s, const DevModel* __restrict__ m, int lane, int nva) {
  double force = 0;
  if (lane < MDL.d.nu) {
    const double* mom = MDL.d.act_moment[lane];
    double len = 0, vel = 0;
    for (int i = 0; i < NH; i++) { double c = mom[i]; if (c != 0) { len += c * s.qpos[i]; vel += c * s.qvel[i]; } }
    double ctrl = s.ctrl[lane];
    if (MDL.d.act_ctrllimited[lane]) ctrl = fmax(MDL.d.act_ctrlrange[lane][0], fmin(MDL.d.act_ctrlrange[lane][1], ctrl));
    const double* bp = MDL.d.act_bias[lane];
    if constexpr (S::HAS_PRM) {         // one multiplier for the servo's kp (gain, bias[1]) and kv (bias[2]); same expression as below
      const double p = s.prm[MCB_P_GAIN + lane];
      const double g = MDL.d.act_gain[lane] * p, b1 = bp[1] * p, b2 = bp[2] * p;
      force = g * ctrl + bp[0] + b1 * len + b2 * vel;
    } else
    force = MDL.d.act_gain[lane] * ctrl + bp[0] + bp[1] * len + bp[2] * vel;
    if (MDL.d.act_forcelimited[lane]) force = fmax(MDL.d.act_forcerange[lane][0], fmin(MDL.d.act_forcerange[lane][1], force));
  }
  double qa = 0;
#pragma unroll
  for (int a = 0; a < NU; a++) {
    double fa = __shfl_sync(FULLMASK, force, a);
    if (lane < NV) qa += MDL.d.act_moment[a][lane] * fa;
  }
  if constexpr (S::HAS_PRM) {
    if (lane < nva) {
      double q = -env_damping(s, lane) * s.qvel[lane] - s.qfrc_bias[lane] + qa;
      const double* fr = s.frc;
      if (fr) q += fr[lane];       // qfrc_applied (xfrc_applied is in qfrc_bias, velocity_rne)
      s.qfrc_smooth[lane] = q;
    }
  } else
  if (lane < nva) s.qfrc_smooth[lane] = -MDL.d.damping[lane] * s.qvel[lane] - s.qfrc_bias[lane] + qa;
  __syncwarp();
}

// ------------------------------------------------------------------------------------------------
// Newton: primal solver with exact line search over the piecewise-quadratic cost (pyramidal cones).
template <class S>
struct Newton {
  S& s; const DevModel* __restrict__ m; int lane, nva, nefc;
  bool coupled;
  double gauss, cost;

  __device__ __forceinline__ bool active(int r, double jar) const { return !(s.rmeta[r] & RM_INEQ) || jar < 0; }

  // out[r] = J_r . v (- aref_r if sub)
  __device__ void rows_times(const double* v, double* out, bool sub_aref) {
    for (int r = lane; r < nefc; r += 32) {
      double d = row_dot(s, r, v);
      out[r] = sub_aref ? d - s.earef[r] : d;
    }
  }
  // cost and gradient at the current point (Jaref, Ma valid); eJv is used as the efc_force scratch
  // (alpha != 0: the residuals are first advanced along the search direction, Jaref += alpha * J search, in the same pass)
  __device__ void update_cost_grad(double alpha = 0.0) {
    double c = 0;
    for (int r = lane; r < nefc; r += 32) {
      double jar = s.eJaref[r];
      if (alpha != 0.0) { jar += alpha * s.eJv[r]; s.eJaref[r] = jar; }
      bool act = active(r, jar);
      s.eJv[r] = act ? -s.eD[r] * jar : 0.0;
      if (act) c += 0.5 * s.eD[r] * jar * jar;
    }
    double g = 0;
    if (lane < nva) g = 0.5 * (s.Ma[lane] - s.qfrc_smooth[lane]) * (s.qacc[lane] - s.qacc_smooth[lane]);
    __syncwarp();
    gauss = warp_sum(g);
    cost = gauss + warp_sum(c);
    // qfrc_constraint = J' f, by row group.  Robot lanes take the robot rows; the cube rows (the longest group: 6 rows per
    // resting contact) are split over three lanes per cube dof and folded with two shuffles.
    {
      const int nR = s.nR, nC = s.nC, nF = s.nF, nU = s.nU;
      double q = 0, q1 = 0, q2 = 0, q3 = 0;
      if (lane < NH) {
        int r = 0;
        for (; r + 3 < nR; r += 4) { q += s.pool[r * SR + lane] * s.eJv[r]; q1 += s.pool[(r + 1) * SR + lane] * s.eJv[r + 1]; q2 += s.pool[(r + 2) * SR + lane] * s.eJv[r + 2]; q3 += s.pool[(r + 3) * SR + lane] * s.eJv[r + 3]; }
        for (; r < nR; r++) q += s.pool[r * SR + lane] * s.eJv[r];
      } else if (lane < NH + 18 && nva > NH) {
        const int part = (lane - NH) / 6, d = (lane - NH) - 6 * part;
        const double* p = s.pool + nR * SR + d;
        const double* f = s.eJv + nR;
        int r = part;
        for (; r + 9 < nC; r += 12) { q += p[r * SC] * f[r]; q1 += p[(r + 3) * SC] * f[r + 3]; q2 += p[(r + 6) * SC] * f[r + 6]; q3 += p[(r + 9) * SC] * f[r + 9]; }
        for (; r < nC; r += 3) q += p[r * SC] * f[r];
      }
      q = (q + q1) + (q2 + q3);
      const double qa = shfl_d(q, (lane + 6) & 31), qb = shfl_d(q, (lane + 12) & 31);
      if (lane >= NH && lane < NV) q += qa + qb;
      if (lane < nva) {
        { const double* p = s.pool + nR * SR + nC * SC + lane; for (int r = 0; r < nF; r++) q += p[r * SF] * s.eJv[nR + nC + r]; }
        for (int u = 0; u < nU; u++) {
          int r = nR + nC + nF + u, meta = s.rmeta[r];
          if ((meta & 0xff) == lane) q += (meta & 0x100) ? -s.eJv[r] : s.eJv[r];
        }
        s.qfrc_con[lane] = q;
        s.grad[lane] = s.Ma[lane] - s.qfrc_smooth[lane] - q;
      }
    }
    __syncwarp();
  }
  // H = M + J' diag(D * active) J (packed lower triangle), accumulated per block in registers
  __device__ void build_H() {
    const int nR = s.nR, nC = s.nC, nF = s.nF, nU = s.nU;
    int ri[3], rj[3];      // robot-robot entries e = lane + 32 p < 78
#pragma unroll
    for (int p = 0; p < 3; p++) { int e = lane + 32 * p; ri[p] = MDL.tri_i[e]; rj[p] = MDL.tri_j[e]; }
    const int ci = MDL.tri_i[lane], cj = MDL.tri_j[lane];    // cube-cube entry t = lane < 21
    // D_r for active rows, 0 for inactive ones: branch-free accumulation below.  eJv is free here (the constraint
    // forces it held were consumed by update_cost_grad; line_search refills it with J*search).
    double* Da = s.eJv;
    for (int r = lane; r < nefc; r += 32) Da[r] = active(r, s.eJaref[r]) ? s.eD[r] : 0.0;
    __syncwarp();
    double arr[3], ar2[3] = {0, 0, 0}, acc_cc = 0, arc[3] = {0, 0, 0};
#pragma unroll
    for (int p = 0; p < 3; p++) arr[p] = (lane + 32 * p < 78) ? s.M[lane + 32 * p] : 0.0;
    if (lane < 21 && nva > NH) acc_cc = s.M[TRI(NH + ci, NH + cj)];
    {
      const int o0 = ri[0], o1 = rj[0], o2 = ri[1], o3 = rj[1];
      const int o4 = (lane + 64 < 78) ? ri[2] : 0, o5 = (lane + 64 < 78) ? rj[2] : 0;   // lanes past the 78 entries recompute entry (0,0): never stored
      int r = 0;
      for (; r + 1 < nR; r += 2) {
        const double* p = s.pool + r * SR;
        double D0 = Da[r], D1 = Da[r + 1];
        arr[0] += D0 * p[o0] * p[o1]; ar2[0] += D1 * p[SR + o0] * p[SR + o1];
        arr[1] += D0 * p[o2] * p[o3]; ar2[1] += D1 * p[SR + o2] * p[SR + o3];
        arr[2] += D0 * p[o4] * p[o5]; ar2[2] += D1 * p[SR + o4] * p[SR + o5];
      }
      if (r < nR) {
        const double* p = s.pool + r * SR;
        double D0 = Da[r];
        arr[0] += D0 * p[o0] * p[o1]; arr[1] += D0 * p[o2] * p[o3]; arr[2] += D0 * p[o4] * p[o5];
      }
#pragma unroll
      for (int q = 0; q < 3; q++) arr[q] += ar2[q];
    }
    if (nva > NH) {
      {
        const int c0 = (lane < 21) ? ci : 0, c1 = (lane < 21) ? cj : 0;
        const double* p = s.pool + nR * SR;
        const double* Dc = Da + nR;
        double a1 = 0, a2 = 0, a3 = 0;
        int r = 0;
        for (; r + 3 < nC; r += 4) {
          acc_cc += Dc[r] * p[r * SC + c0] * p[r * SC + c1];
          a1 += Dc[r + 1] * p[(r + 1) * SC + c0] * p[(r + 1) * SC + c1];
          a2 += Dc[r + 2] * p[(r + 2) * SC + c0] * p[(r + 2) * SC + c1];
          a3 += Dc[r + 3] * p[(r + 3) * SC + c0] * p[(r + 3) * SC + c1];
        }
        for (; r < nC; r++) acc_cc += Dc[r] * p[r * SC + c0] * p[r * SC + c1];
        acc_cc += (a1 + a2) + a3;
      }
      for (int r = 0; r < nF; r++) {
        int g = nR + nC + r;
        const double* p = s.pool + nR * SR + nC * SC + r * SF;
        double D = Da[g];
#pragma unroll
        for (int q = 0; q < 3; q++) if (lane + 32 * q < 78) arr[q] += D * p[ri[q]] * p[rj[q]];
        if (lane < 21) acc_cc += D * p[NH + ci] * p[NH + cj];
#pragma unroll
        for (int q = 0; q < 3; q++) { int t = lane + 32 * q; if (t < 72) arc[q] += D * p[NH + t / NH] * p[t % NH]; }
      }
    }
#pragma unroll
    for (int p = 0; p < 3; p++) if (lane + 32 * p < 78) s.H[lane + 32 * p] = arr[p];
    if (nva > NH) {
      if (lane < 21) s.H[TRI(NH + ci, NH + cj)] = acc_cc;
#pragma unroll
      for (int q = 0; q < 3; q++) { int t = lane + 32 * q; if (t < 72) s.H[TRI(NH + t / NH, t % NH)] = arc[q]; }
    }
    __syncwarp();
    if (lane == 0) {
      for (int u = 0; u < nU; u++) {
        int r = nR + nC + nF + u;
        int d = s.rmeta[r] & 0xff;
        s.H[TRI(d, d)] += Da[r];
      }
    }
    __syncwarp();
  }
  __device__ void newton_direction() {
    build_H();
    double mg = factor_solve(s.H, s.H, s.grad, s.Mv, lane, nva, coupled);
    if (lane < nva) s.search[lane] = -mg;
    __syncwarp();
  }
  struct Pt { double alpha, cost, d0, d1; };
  __device__ __forceinline__ double line_search(double scale) {
    // per-lane quadratic coefficients of rows lane + 32 t and the Gauss term's: locals of this (inlined) function, so they stay
    // in registers -- as members of a struct whose other methods are out of line they lived in local memory (profiles/r02a)
    double qa[S::NROW / 32 + 1], qb[S::NROW / 32 + 1], qc[S::NROW / 32 + 1], qg0, qg1, qg2;
    auto ls_eval = [&](Pt& p) {
      double a = p.alpha, q0 = 0, q1 = 0, q2 = 0;
#pragma unroll
      for (int t = 0; t < S::NROW / 32 + 1; t++) {
        int r = lane + 32 * t;
        if (r < nefc && active(r, s.eJaref[r] + a * s.eJv[r])) { q0 += qa[t]; q1 += qb[t]; q2 += qc[t]; }
      }
      warp_sum3(q0, q1, q2, lane);
      q0 += qg0; q1 += qg1; q2 += qg2;
      p.cost = a * a * q2 + a * q1 + q0;
      p.d0 = 2 * a * q2 + q1;
      p.d1 = 2 * q2;
      if (p.d1 <= 0) p.d1 = MINVAL;
    };
    // |search|^2 and the two Gauss-term coefficients in one butterfly (M * search is needed for the latter, so it is formed
    // before the zero-norm early-out instead of after it)
    double mv = mulM_row(s, lane, nva, s.search);
    double sn = 0, g1 = 0, g2 = 0;
    if (lane < nva) {
      const double sl = s.search[lane];
      sn = sl * sl; g1 = sl * (s.Ma[lane] - s.qfrc_smooth[lane]); g2 = sl * mv;
      s.Mv[lane] = mv;
    }
    warp_sum3(sn, g1, g2, lane);
    const double snorm = sqrt(sn);
    if (snorm < MINVAL) return 0;
    double gtol = MDL.d.tolerance * MDL.d.ls_tolerance * snorm * (MDL.d.meaninertia * (double)NV);   // 1 / scale
    rows_times(s.search, s.eJv, false);
    qg0 = gauss; qg1 = g1; qg2 = 0.5 * g2;
    __syncwarp();
#pragma unroll
    for (int t = 0; t < S::NROW / 32 + 1; t++) {
      int r = lane + 32 * t;
      if (r < nefc) {
        double D = s.eD[r], ja = s.eJaref[r], jv = s.eJv[r];
        qa[t] = 0.5 * D * ja * ja; qb[t] = D * ja * jv; qc[t] = 0.5 * D * jv * jv;
      } else { qa[t] = qb[t] = qc[t] = 0; }
    }
    const int lsmax = MDL.d.ls_iterations;
    Pt p0, p1, p2, pmid, p1n, p2n;
    p0.alpha = 0; ls_eval(p0);
    p1.alpha = p0.alpha - p0.d0 * fast_rcp(p0.d1); ls_eval(p1);
    if (p0.cost < p1.cost) p1 = p0;
    if (fabs(p1.d0) < gtol) return p1.alpha;
    int dir = p1.d0 < 0 ? 1 : -1, iter = 0, p2update = 0;
    p2 = p1;
    while (p1.d0 * dir <= -gtol && iter < lsmax) {
      p2 = p1; p2update = 1;
      p1.alpha = p1.alpha - p1.d0 * fast_rcp(p1.d1); ls_eval(p1); iter++;
      if (fabs(p1.d0) < gtol) return p1.alpha;
    }
    if (iter >= lsmax || !p2update) return p1.alpha;
    p2n = p1;
    p1n.alpha = p1.alpha - p1.d0 * fast_rcp(p1.d1); ls_eval(p1n);
    while (iter < lsmax) {
      pmid.alpha = 0.5 * (p1.alpha + p2.alpha); ls_eval(pmid); iter++;
      // candidates in the order p1next, p2next, midpoint
      double balpha = 0, bcost = 0; bool found = false;
      if (fabs(p1n.d0) < gtol) { balpha = p1n.alpha; bcost = p1n.cost; found = true; }
      if (fabs(p2n.d0) < gtol && (!found || p2n.cost < bcost)) { balpha = p2n.alpha; bcost = p2n.cost; found = true; }
      if (fabs(pmid.d0) < gtol && (!found || pmid.cost < bcost)) { balpha = pmid.alpha; bcost = pmid.cost; found = true; }
      if (found) return balpha;
      int b1 = 0, b2 = 0;
#define LS_BRACKET(c)                                                                                                   \
      if ((c).d0 * dir < 0 && ((c).alpha - p2.alpha) * dir > 0 && (p1.alpha - (c).alpha) * dir > 0) { p2 = (c); b2 = 1; }     \
      else if ((c).d0 * dir > 0 && (p1.alpha - (c).alpha) * dir > 0 && ((c).alpha - p2.alpha) * dir > 0) { p1 = (c); b1 = 1; }
      { Pt c = p1n; LS_BRACKET(c) }
      { Pt c = p2n; LS_BRACKET(c) }
      { Pt c = pmid; LS_BRACKET(c) }
#undef LS_BRACKET
      if (!b1 && !b2) break;
      if (b1) { p1n.alpha = p1.alpha - p1.d0 * fast_rcp(p1.d1); ls_eval(p1n); }
      if (b2) { p2n.alpha = p2.alpha - p2.d0 * fast_rcp(p2.d1); ls_eval(p2n); }
    }
    return (p1.cost < p2.cost ? p1.alpha : p2.alpha);
  }

  __device__ __forceinline__ void solve() {
    const double scale = fast_rcp(MDL.d.meaninertia * (double)NV);
    coupled = s.nF > 0;
    // warmstart(): better of qacc_warmstart and qacc_smooth.  jar(warm) -> eJaref, jar(smooth) -> eJv
    double cw = 0, cs = 0;      // constraint cost of the two candidates, accumulated while their residuals are formed
    for (int r = lane; r < nefc; r += 32) {
      double dw, ds;
      row_dot2(s, r, s.warm, s.qacc_smooth, dw, ds);
      const double ar = s.earef[r], D = s.eD[r];
      dw -= ar; ds -= ar;
      s.eJaref[r] = dw; s.eJv[r] = ds;
      if (active(r, dw)) cw += 0.5 * D * dw * dw;
      if (active(r, ds)) cs += 0.5 * D * ds * ds;
    }
    double ma = mulM_row(s, lane, nva, s.warm), g = 0;
    if (lane < nva) g = 0.5 * (ma - s.qfrc_smooth[lane]) * (s.warm[lane] - s.qacc_smooth[lane]);
    __syncwarp();
    warp_sum3(cw, cs, g, lane);
    cw += g;
    bool use_smooth = cw > cs;
    if (use_smooth) {
      for (int r = lane; r < nefc; r += 32) s.eJaref[r] = s.eJv[r];
      if (lane < nva) s.qacc[lane] = s.qacc_smooth[lane];
      __syncwarp();
      double ma2 = mulM_row(s, lane, nva, s.qacc);
      if (lane < nva) s.Ma[lane] = ma2;
    } else if (lane < nva) { s.qacc[lane] = s.warm[lane]; s.Ma[lane] = ma; }
    __syncwarp();
    update_cost_grad();
    newton_direction();
    int iter = 0;
    const int maxiter = MDL.d.iterations;
    while (iter < maxiter) {
      double alpha = line_search(scale);
      if (alpha == 0) break;
      if (lane < nva) { s.qacc[lane] += alpha * s.search[lane]; s.Ma[lane] += alpha * s.Mv[lane]; }
      __syncwarp();
      double oldcost = cost;
      update_cost_grad(alpha);
      iter++;
      double gn = 0;
      if (lane < nva) gn = s.grad[lane] * s.grad[lane];
      // gradient norm test on squares: scale * sqrt(gn) < tolerance  <=>  scale^2 gn < tolerance^2 (no sqrt on the critical path)
      double improvement = scale * (oldcost - cost), grad2 = scale * scale * warp_sum(gn);
      if (improvement < MDL.d.tolerance || grad2 < MDL.d.tolerance * MDL.d.tolerance) break;
      newton_direction();
    }
    if (lane == 0) s.iters += iter;
    if (lane < nva) s.warm[lane] = s.qacc[lane];
    __syncwarp();
  }
};

// forward(): everything mj_forward does for this model.  Returns false if the layout overflowed.
// `sync`: the warps of a CTA run the substep loop in lockstep (CTA barriers at the stage boundaries) so that they
// share instruction-cache lines -- the kernel is thousands of straight-line instructions per substep and
// independent warps drifting apart made instruction fetch the top stall (profiles/r01c).  Every path through
// forward() executes exactly NSYNC_FWD barriers when sync is set: one at each of its six stage boundaries.
#define NSYNC_FWD 6
// Lockstep groups: `lw` consecutive warps of the CTA share one named barrier (ids 1..), so the CTA runs 16 / lw groups
// that drift against each other (different stages -> different pipes busy at the same time) while the warps inside a
// group still share instruction-cache lines.  lw = 1: free-running warps, no barriers.  Which grouping wins depends on
// the workload's code footprint (profiles/README.md, r01o / r01q): pick-and-place and reach are fastest free-running
// (2.47 M vs 2.27 M env-steps/s in full lockstep), push and the mocap variant are 2x / 1.4x faster in full lockstep
// (free-running they stall on instruction fetch, `no_instructions` 38 %).  mcb_autotune() measures and picks per batch.
#define LOCKSTEP_CTA 16   // lw >= this: the whole CTA is one group, whatever its tier's warp count (__syncthreads)
__device__ __forceinline__ void group_sync(int lw) {
  if (lw >= LOCKSTEP_CTA) __syncthreads();
  else asm volatile("bar.sync %0, %1;" ::"r"(1 + (int)(threadIdx.x >> 5) / lw), "r"(32 * lw) : "memory");
}
template <class S>
__device__ __noinline__ bool forward(S& s, const DevModel* __restrict__ m, int lane, int nba, int nva, int sync) {
  if (sync) group_sync(sync);
  fk(s, m, lane, nba);
  cinert_cdof(s, m, lane, nba, nva);
  if (sync) group_sync(sync);
  crb_mass(s, m, lane, nba, nva);
  velocity_rne(s, m, lane, nba, nva);
  if (sync) group_sync(sync);
  actuation_smooth(s, m, lane, nva);
  double qs = factor_solve_M<true>(s.M, s.H, s.qfrc_smooth, s.Mv, 0.0, lane, nva);
  if (lane < nva) s.qacc_smooth[lane] = qs;
  __syncwarp();
  if (sync) group_sync(sync);
  collide(s, lane, nba, s.mesh != 0);
  if (sync) group_sync(sync);
  bool ok = make_rows(s, m, lane, nva);
  if (sync) group_sync(sync);
  if (!ok && !S::IS_BIG) return false;
  Newton<S> nw{s, m, lane, nva, s.nefc};
  nw.solve();
  return true;
}

// euler(): (M + h*diag(damping))^-1 (qfrc_smooth + qfrc_constraint), semi-implicit advance.
template <class S>
__device__ __noinline__ void euler(S& s, const DevModel* __restrict__ m, int lane, int nva) {
  const double h = MDL.d.timestep;
  if (lane < NV) s.search[lane] = lane < nva ? s.qfrc_smooth[lane] + s.qfrc_con[lane] : 0.0;   // search / Mv are free outside the solver
  __syncwarp();
  double qacc;
  if constexpr (S::HAS_PRM) qacc = factor_solve_M<true>(s.M, s.H, s.search, s.Mv, lane < nva ? h * env_damping(s, lane) : 0.0, lane, nva);
  else
  qacc = factor_solve_M<true>(s.M, s.H, s.search, s.Mv, lane < nva ? h * MDL.d.damping[lane] : 0.0, lane, nva);
  if (lane < nva) s.qvel[lane] += h * qacc;
  __syncwarp();
  if (lane < NH) s.qpos[lane] += h * s.qvel[lane];
  else if (lane < 15 && nva > NH) s.qpos[lane] += h * s.qvel[lane];
  else if (lane == 15 && nva > NH) {
    double ax[3] = {s.qvel[15], s.qvel[16], s.qvel[17]};
    double n = sqrt(dot3(ax, ax));
    if (n < MINVAL) { ax[0] = 1; ax[1] = ax[2] = 0; } else { const double in = fast_rcp(n); ax[0] *= in; ax[1] *= in; ax[2] *= in; }
    double ang = h * n;
    double qr[4];
    if (ang == 0) { qr[0] = 1; qr[1] = qr[2] = qr[3] = 0; }
    else { double sn, cs; sincos(0.5 * ang, &sn, &cs); qr[0] = cs; qr[1] = ax[0] * sn; qr[2] = ax[1] * sn; qr[3] = ax[2] * sn; }
    double* q = s.qpos + 15;
    double nq = sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
    double a[4];
    if (nq < MINVAL) { a[0] = 1; a[1] = a[2] = a[3] = 0; } else { const double in = fast_rcp(nq); a[0] = q[0] * in; a[1] = q[1] * in; a[2] = q[2] * in; a[3] = q[3] * in; }
    q[0] = a[0] * qr[0] - a[1] * qr[1] - a[2] * qr[2] - a[3] * qr[3];
    q[1] = a[0] * qr[1] + a[1] * qr[0] + a[2] * qr[3] - a[3] * qr[2];
    q[2] = a[0] * qr[2] - a[1] * qr[3] + a[2] * qr[0] + a[3] * qr[1];
    q[3] = a[0] * qr[3] + a[1] * qr[2] - a[2] * qr[1] + a[3] * qr[0];
  }
  __syncwarp();
}

// start-of-episode constants: the model's qpos0 set, or keyframe 0 for fetch envs (mycobot.py:451-472); init_state_kernel reads the model in global memory
__device__ __forceinline__ const double* init_qpos_of(const DevModel& md, int fetch) { return fetch ? md.d.key_qpos : md.d.init_qpos; }
__device__ __forceinline__ const double* init_ctrl_of(const DevModel& md, int fetch) { return fetch ? md.d.key_ctrl : md.d.init_ctrl; }
__device__ __forceinline__ const double* grip0_of(const mcb_task_cfg& c) { return c.fetch_env ? MDL.d.key_initial_gripper_xpos : MDL.d.initial_gripper_xpos; }
__device__ __forceinline__ double hoff_of(const mcb_task_cfg& c) { return c.fetch_env ? MDL.d.key_height_offset : MDL.d.height_offset; }

// Philox4x32-10 counter RNG: one stream per env, key = seed, counter = (env, draw index, stream tag).  Tag GOAL_TAG: goals and cube
// positions; PARAM_TAG: per-env physics parameters, LATENCY_TAG: actuation latency, each with a draw counter of its own, so the goal
// stream is the same with or without them.
#define GOAL_TAG 0x6d79636fu
#define PARAM_TAG 0x7072616du
#define LATENCY_TAG 0x6c61746eu
__device__ __forceinline__ void philox_round(uint32_t* c, uint32_t k0, uint32_t k1) {
  uint32_t hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
  uint32_t hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
  uint32_t n0 = hi1 ^ c[1] ^ k0, n1 = lo1, n2 = hi0 ^ c[3] ^ k1, n3 = lo0;
  c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
}
template <uint32_t TAG = GOAL_TAG>
__device__ double philox_uniform(uint64_t seed, uint32_t env, unsigned long long& ctr) {
  uint32_t c[4] = {(uint32_t)ctr, (uint32_t)(ctr >> 32), env, TAG};
  uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
  for (int i = 0; i < 10; i++) { philox_round(c, k0, k1); k0 += 0x9E3779B9u; k1 += 0xBB67AE85u; }
  ctr++;
  uint64_t bits = ((uint64_t)c[0] << 21) | (uint64_t)(c[1] >> 11);
  return (double)bits * (1.0 / 9007199254740992.0);
}
// _sample_goal (mycobot.py:238-243, utils.py:14-21): same draw structure, device streams
__device__ void sample_goal(const DevModel* __restrict__ m, const mcb_task_cfg& cfg, uint64_t seed, uint32_t env, unsigned long long& ctr, double* g) {
  g[0] = -0.12 + (0.12 - (-0.12)) * philox_uniform(seed, env, ctr);
  g[1] = -0.06 + (0.06 - (-0.06)) * philox_uniform(seed, env, ctr);
  g[2] = hoff_of(cfg);
  if (cfg.target_in_the_air) {
    if (philox_uniform(seed, env, ctr) < 0.5) g[2] += 0.0 + (0.1 - 0.0) * philox_uniform(seed, env, ctr);
  }
}

// EEF site position from the frames in shared memory (its orientation is the body's: the site has no own rotation)
template <class S>
__device__ __forceinline__ void eef_pos_of(const S& s, double* pos) {
  const int eb = MDL.d.eef_body;
  const double* R = s.xmat + eb * 9;
  const double* ep = MDL.d.eef_pos;
#pragma unroll
  for (int r = 0; r < 3; r++) pos[r] = s.xpos[eb * 3 + r] + R[3 * r] * ep[0] + R[3 * r + 1] * ep[1] + R[3 * r + 2] * ep[2];
}
// observation (mycobot.py:342-388): written from the frames currently in shared memory (stale by one
// substep after a step, fresh after forward), qpos / qvel current.  Lanes 0-2: gripper position / velocity,
// 3-5: cube position / velocities, 6: cube Euler angles, 7: gripper joint state; staged through s.grad..s.Mv.
template <class S>
__device__ __noinline__ void write_obs(S& s, const DevModel* __restrict__ m, const mcb_task_cfg& cfg, int lane, int env, double* obs, double* ag, double* dg, double* ag_out3) {
  const double dt = cfg.frame_skip * MDL.d.timestep;
  double* o = s.grad;          // grad, search, Mv are contiguous: 54 doubles of scratch, dead outside the solver
  const bool has_obj = cfg.has_object;
  __syncwarp();
  if (lane < 3) {
    const int r = lane, eb = MDL.d.eef_body;
    double grip[3];
    eef_pos_of(s, grip);
    double off[3] = {grip[0] - MDL.d.ref_robot[0], grip[1] - MDL.d.ref_robot[1], grip[2] - MDL.d.ref_robot[2]};
    double gv = 0;
    unsigned mask = MDL.d.ancmask[eb];
    while (mask) {
      int j = __ffs(mask) - 1; mask &= mask - 1;
      const double* cd = s.cdof + j * 6;
      double t[3];
      cross3(t, cd, off);
      gv += (cd[3 + r] + (r == 0 ? t[0] : r == 1 ? t[1] : t[2])) * s.qvel[j];
    }
    o[40 + r] = (r == 0 ? grip[0] : r == 1 ? grip[1] : grip[2]);
    o[43 + r] = gv;
  } else if (lane < 6 && has_obj) {
    const int r = lane - 3;
    double op[3] = {s.xpos[CUBE * 3], s.xpos[CUBE * 3 + 1], s.xpos[CUBE * 3 + 2]};
    double off[3] = {op[0] - s.refcube[0], op[1] - s.refcube[1], op[2] - s.refcube[2]};
    double vp = 0, vr = 0;
    for (int j = 12; j < 18; j++) {
      const double* cd = s.cdof + j * 6;
      double t[3];
      cross3(t, cd, off);
      vp += (cd[3 + r] + (r == 0 ? t[0] : r == 1 ? t[1] : t[2])) * s.qvel[j];
      vr += cd[r] * s.qvel[j];
    }
    o[46 + r] = (r == 0 ? op[0] : r == 1 ? op[1] : op[2]);
    o[49 + r] = vp;
    o[17 + r] = vr * dt;
  } else if (lane == 6 && has_obj) {
    const double* Ro = s.xmat + CUBE * 9;
    double cy = sqrt(Ro[8] * Ro[8] + Ro[5] * Ro[5]);
    double e0, e1, e2;
    if (cy > 2.220446049250313e-16 * 4.0) { e2 = -atan2(Ro[1], Ro[0]); e1 = -atan2(-Ro[2], cy); e0 = -atan2(Ro[5], Ro[8]); }
    else { e2 = -atan2(-Ro[3], Ro[4]); e1 = -atan2(-Ro[2], cy); e0 = 0.0; }
    o[11] = e0; o[12] = e1; o[13] = e2;
  }
  __syncwarp();
  int nobs;
  if (has_obj) {
    if (lane < 3) {
      const int r = lane;
      double grip = o[40 + r], gv = o[43 + r], op = o[46 + r], vp = o[49 + r];
      o[r] = grip; o[3 + r] = op; o[6 + r] = op - grip;
      o[14 + r] = vp * dt - gv * dt;
      o[20 + r] = gv * dt;
    } else if (lane == 3) {
      o[9] = s.qpos[6]; o[10] = s.qpos[8]; o[23] = s.qvel[6] * dt; o[24] = s.qvel[8] * dt;
    }
    nobs = MCB_OBS_OBJECT;
  } else {
    if (lane < 3) { const int r = lane; o[r] = o[40 + r]; o[5 + r] = o[43 + r] * dt; }
    else if (lane == 3) { o[3] = s.qpos[6]; o[4] = s.qpos[8]; o[8] = s.qvel[6] * dt; o[9] = s.qvel[8] * dt; }
    nobs = MCB_OBS_REACH;
  }
  __syncwarp();
  const int a0 = has_obj ? 3 : 0;     // achieved goal: cube position (object envs) or gripper position (reach)
  if (obs && lane < nobs) obs[(size_t)env * nobs + lane] = o[lane];
  if (lane < 3) {
    if (ag) ag[(size_t)env * 3 + lane] = o[a0 + lane];
    if (dg) dg[(size_t)env * 3 + lane] = s.goal[lane];
  }
  ag_out3[0] = o[a0]; ag_out3[1] = o[a0 + 1]; ag_out3[2] = o[a0 + 2];
  __syncwarp();
}

template <class S>
__device__ void load_state(S& s, const double* __restrict__ st, int lane) {
  for (int w = lane; w < MCB_STATE_STRIDE; w += 32) {
    double v = st[w];
    if (w < ST_QVEL) s.qpos[w - ST_QPOS] = v;
    else if (w < ST_CTRL) s.qvel[w - ST_QVEL] = v;
    else if (w < ST_WARM) s.ctrl[w - ST_CTRL] = v;
    else if (w < ST_GOAL) s.warm[w - ST_WARM] = v;
    else if (w < ST_QPREV) s.goal[w - ST_GOAL] = v;
    else if (w < ST_MOCAP) s.qprev[w - ST_QPREV] = v;
    else if (w < ST_END) s.mocap[w - ST_MOCAP] = v;
  }
  __syncwarp();
}
template <class S>
__device__ void store_state(const S& s, double* __restrict__ st, int lane) {
  for (int w = lane; w < MCB_STATE_STRIDE; w += 32) {
    double v = 0;
    if (w < ST_QVEL) v = s.qpos[w - ST_QPOS];
    else if (w < ST_CTRL) v = s.qvel[w - ST_QVEL];
    else if (w < ST_WARM) v = s.ctrl[w - ST_CTRL];
    else if (w < ST_GOAL) v = s.warm[w - ST_WARM];
    else if (w < ST_QPREV) v = s.goal[w - ST_GOAL];
    else if (w < ST_MOCAP) v = s.qprev[w - ST_QPREV];
    else if (w < ST_END) v = s.mocap[w - ST_MOCAP];
    st[w] = v;
  }
}


// ------------------------------------------------------------------------------------------------
// IK controller (mycobot.py:134-170, utils.py:499-556): damped-least-squares step on the EEF site pose.
// mju_mat2Quat / mju_mulQuat / mju_quat2Vel and rotations.euler2quat restated; scalar work on lane 0.
__device__ void mat2quat_d(double* q, const double* m) {
  if (m[0] + m[4] + m[8] > 0) {
    q[0] = 0.5 * sqrt(1 + m[0] + m[4] + m[8]);
    q[1] = 0.25 * (m[7] - m[5]) / q[0]; q[2] = 0.25 * (m[2] - m[6]) / q[0]; q[3] = 0.25 * (m[3] - m[1]) / q[0];
  } else if (m[0] > m[4] && m[0] > m[8]) {
    q[1] = 0.5 * sqrt(1 + m[0] - m[4] - m[8]);
    q[0] = 0.25 * (m[7] - m[5]) / q[1]; q[2] = 0.25 * (m[1] + m[3]) / q[1]; q[3] = 0.25 * (m[2] + m[6]) / q[1];
  } else if (m[4] > m[8]) {
    q[2] = 0.5 * sqrt(1 - m[0] + m[4] - m[8]);
    q[0] = 0.25 * (m[2] - m[6]) / q[2]; q[1] = 0.25 * (m[1] + m[3]) / q[2]; q[3] = 0.25 * (m[5] + m[7]) / q[2];
  } else {
    q[3] = 0.5 * sqrt(1 - m[0] - m[4] + m[8]);
    q[0] = 0.25 * (m[3] - m[1]) / q[3]; q[1] = 0.25 * (m[2] + m[6]) / q[3]; q[2] = 0.25 * (m[5] + m[7]) / q[3];
  }
  double n = sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
  q[0] /= n; q[1] /= n; q[2] /= n; q[3] /= n;
}
__device__ __forceinline__ void mulquat_d(double* r, const double* a, const double* b) {
  double t0 = a[0] * b[0] - a[1] * b[1] - a[2] * b[2] - a[3] * b[3];
  double t1 = a[0] * b[1] + a[1] * b[0] + a[2] * b[3] - a[3] * b[2];
  double t2 = a[0] * b[2] - a[1] * b[3] + a[2] * b[0] + a[3] * b[1];
  double t3 = a[0] * b[3] + a[1] * b[2] - a[2] * b[1] + a[3] * b[0];
  r[0] = t0; r[1] = t1; r[2] = t2; r[3] = t3;
}
// target pose of this env-step from the (stale) site pose and the clipped float32 action
template <class S>
__device__ void ik_target(S& s, const mcb_task_cfg& cfg, const float* act, int lane) {
  if (lane == 0) {
    double pos[3];
    eef_pos_of(s, pos);
    for (int k = 0; k < 3; k++) s.ik[k] = pos[k] + (double)(act[k] * 0.2f);          // float32 product, float64 sum (numpy semantics)
    if (cfg.fetch_env) { s.ik[3] = 0; s.ik[4] = -0.707; s.ik[5] = 0; s.ik[6] = 0.707; }
    else {
      double e0 = (double)(act[3] * 0.5f), e1 = (double)(act[4] * 0.5f), e2 = (double)(act[5] * 0.5f);
      double ai = e2 / 2, aj = -e1 / 2, ak = e0 / 2;
      double si, ci, sj, cj, sk, ck;
      sincos(ai, &si, &ci); sincos(aj, &sj, &cj); sincos(ak, &sk, &ck);
      double cc = ci * ck, cs = ci * sk, sc = si * ck, ss = si * sk;
      double qr[4] = {cj * cc + sj * ss, cj * cs - sj * sc, -(cj * ss + sj * cc), cj * sc - sj * cs};
      double qe[4];
      mat2quat_d(qe, s.xmat + MDL.d.eef_body * 9);
      mulquat_d(s.ik + 3, qr, qe);
    }
  }
  __syncwarp();
}
// one DLS solve: ctrl[0..5] += (J'J + 0.3 I)^-1 J' err, J = 6 x 6 site Jacobian w.r.t. the arm dofs (all other columns of
// the reference's 6 x 18 Jacobian are zero for this site, so its 18 x 18 least-squares problem decouples exactly)
template <class S>
__device__ void ik_update_ctrl(S& s, int lane, double grip_ctrl, double& cmd) {
  double* Jm = s.grad;          // 36 doubles of scratch: grad, search, Mv are contiguous and dead outside the solver
  double site[3];
  eef_pos_of(s, site);
  if (lane == 0) {
    for (int k = 0; k < 3; k++) s.ik[7 + k] = s.ik[k] - site[k];
    double qe[4], neg[4], er[4];
    mat2quat_d(qe, s.xmat + MDL.d.eef_body * 9);
    neg[0] = qe[0]; neg[1] = -qe[1]; neg[2] = -qe[2]; neg[3] = -qe[3];
    mulquat_d(er, s.ik + 3, neg);
    double ax[3] = {er[1], er[2], er[3]};
    double sn = sqrt(ax[0] * ax[0] + ax[1] * ax[1] + ax[2] * ax[2]);
    if (sn < MINVAL) { ax[0] = 1; ax[1] = ax[2] = 0; } else { ax[0] /= sn; ax[1] /= sn; ax[2] /= sn; }
    double speed = 2 * atan2(sn, er[0]);
    if (speed > 3.14159265358979323846) speed -= 2 * 3.14159265358979323846;
    speed /= 50;
    for (int k = 0; k < 3; k++) s.ik[10 + k] = ax[k] * speed;
  }
  if (lane < 6) {
    const double* cd = s.cdof + lane * 6;
    double off[3] = {site[0] - MDL.d.ref_robot[0], site[1] - MDL.d.ref_robot[1], site[2] - MDL.d.ref_robot[2]};
    double t[3];
    cross3(t, cd, off);
    Jm[0 * 6 + lane] = cd[3] + t[0]; Jm[1 * 6 + lane] = cd[4] + t[1]; Jm[2 * 6 + lane] = cd[5] + t[2];
    Jm[3 * 6 + lane] = cd[0]; Jm[4 * 6 + lane] = cd[1]; Jm[5 * 6 + lane] = cd[2];
  }
  __syncwarp();
  if (lane < 21) {
    int i = MDL.tri_i[lane], j = MDL.tri_j[lane];
    double h = 0;
#pragma unroll
    for (int k = 0; k < 6; k++) h += Jm[k * 6 + i] * Jm[k * 6 + j];
    if (i == j) h += 0.3;
    s.H[lane] = h;
  }
  double b = 0;
  if (lane < 6) {
#pragma unroll
    for (int k = 0; k < 6; k++) b += Jm[k * 6 + lane] * s.ik[7 + k];
  }
  __syncwarp();
  if (lane < 6) s.ik[7 + lane] = b;       // the pose error is consumed (barrier above); reuse its slots for the right-hand side
  __syncwarp();
  double dq = chol_solve_blk<0, 6, false>(s.H, s.H, s.ik + 7, s.Mv, 0.0, lane);
  if constexpr (S::HAS_PRM) cmd = lane < 6 ? s.ctrl[lane] + dq : grip_ctrl;   // lanes 0..6: the new ctrl, held until the latency has passed
  else {
    if (lane < 6) s.ctrl[lane] += dq;
    else if (lane == 6) s.ctrl[6] = grip_ctrl;
  }
  __syncwarp();
}

// reset_model (mycobot.py:207-236): init state, forward, cube xy, forward, goal.  false: layout overflow.
template <class S>
__device__ __noinline__ bool reset_env(S& s, const StepArgs& a, const DevModel* __restrict__ m, int lane, int env, int nba, int nva, unsigned long long& ctr) {
  if constexpr (S::HAS_PRM) {
    // per-env parameters: slot k ~ U[lo_k, hi_k] from draw prm_ctr + k of the parameter stream, before the first forward pass
    if (a.x.draw_params) {
      if (lane < MCB_NPARAM) {
        unsigned long long c = s.prm_ctr + (unsigned long long)lane;
        const double u = philox_uniform<PARAM_TAG>(a.env_seed[env], env, c);
        const double lo = a.x.param_lo[lane], hi = a.x.param_hi[lane];
        s.prm[lane] = fmin(hi, lo + (hi - lo) * u);
      }
      __syncwarp();
      if (lane == 0) { s.prm_ctr += MCB_NPARAM; s.prm_drawn = 1; }
      __syncwarp();
    }
    // actuation latency: one draw of the latency stream, uniform over the integers [lat_lo, lat_hi]
    if (a.x.draw_latency) {
      if (lane == 0) {
        unsigned long long c = s.lat_ctr;
        const double u = philox_uniform<LATENCY_TAG>(a.env_seed[env], env, c);
        const int span = a.x.lat_hi - a.x.lat_lo;
        s.lat = a.x.lat_lo + min(span, (int)floor(u * (span + 1)));
        s.lat_ctr = c; s.prm_drawn = 1;
      }
      __syncwarp();
    }
    // applied forces: every reset clears them (mj_resetData), before its first forward pass; the commit zeroes the env's row
    if (lane == 0) s.frc = nullptr;
  }
  for (int w = lane; w < NQ; w += 32) s.qpos[w] = init_qpos_of(MDL, a.cfg.fetch_env)[w];
  if (lane < NV) s.qvel[lane] = 0;
  if (lane < NU) s.ctrl[lane] = init_ctrl_of(MDL, a.cfg.fetch_env)[lane];
  __syncwarp();
  if (!forward(s, m, lane, nba, nva, false)) return false;
  const double gx0 = grip0_of(a.cfg)[0], gy0 = grip0_of(a.cfg)[1];
  double oxy[2] = {gx0, gy0};
  double g[3];
  if (lane == 0) {
    if (a.cfg.has_object) {
      if (a.inj_xy) { oxy[0] = a.inj_xy[(size_t)env * 2]; oxy[1] = a.inj_xy[(size_t)env * 2 + 1]; }
      else {
        int guard = 0;
        while (sqrt((oxy[0] - gx0) * (oxy[0] - gx0) + (oxy[1] - gy0) * (oxy[1] - gy0)) < 0.1 && guard++ < 10000) {
          sample_goal(m, a.cfg, a.env_seed[env], env, ctr, g);
          oxy[0] = g[0]; oxy[1] = g[1];
        }
      }
      s.qpos[12] = oxy[0]; s.qpos[13] = oxy[1];
    }
    if (a.inj_goal) { g[0] = a.inj_goal[(size_t)env * 3]; g[1] = a.inj_goal[(size_t)env * 3 + 1]; g[2] = a.inj_goal[(size_t)env * 3 + 2]; }
    else {
      int guard = 0;
      sample_goal(m, a.cfg, a.env_seed[env], env, ctr, g);
      while (sqrt((g[0] - oxy[0]) * (g[0] - oxy[0]) + (g[1] - oxy[1]) * (g[1] - oxy[1])) < 0.1 && guard++ < 10000) sample_goal(m, a.cfg, a.env_seed[env], env, ctr, g);
    }
    s.goal[0] = g[0]; s.goal[1] = g[1]; s.goal[2] = g[2];
  }
  __syncwarp();
  bool ok = forward(s, m, lane, nba, nva, false);
  if (lane < 6) s.qprev[lane] = s.qpos[lane];     // frames are fresh after reset
  __syncwarp();
  return ok;
}

// position of row r in MuJoCo's ordering (equality, limits, contacts in detection order) -- debug taps only
template <class S>
__device__ int row_order(const S& s, int r) {
  const int ne0 = MDL.d.has_weld ? 13 : 7;
  const int meta = s.rmeta[r], kind = (meta >> 12) & 7;
  if (kind == 2) return ne0 + (r - (s.nR + s.nC + s.nF));
  if (kind != 3) return r;
  const int c = meta & 0xff, k = (meta >> 9) & 7;
  int o = ne0 + s.nU;
  for (int q = 0; q < c; q++) o += 2 * (PP(s.cpair[q]).dim - 1);
  return o + k;
}
template <class S>
__device__ void debug_dump(S& s, const StepArgs& a, int lane, int nva) {
  // layout (doubles): [0] nefc [1] ncon [2] iters [3] overflow | M(18*18) | bias smooth qacc_smooth qacc qfrc_con | xpos(39) xmat(117)
  //                   | J(nefc*18, MuJoCo row order) aref D | contact(7*ncon)
  double* o = a.debug;
  if (lane == 0) { o[0] = s.nefc; o[1] = s.ncon; o[2] = s.iters; o[3] = s.overflow; }
  o += 4;
  for (int w = lane; w < NV * NV; w += 32) {
    int i = w / NV, j = w % NV;
    o[w] = (i >= j) ? s.M[TRI(i, j)] : s.M[TRI(j, i)];
  }
  o += NV * NV;
  if (lane < NV) { o[lane] = s.qfrc_bias[lane]; o[NV + lane] = s.qfrc_smooth[lane]; o[2 * NV + lane] = s.qacc_smooth[lane]; o[3 * NV + lane] = s.qacc[lane]; o[4 * NV + lane] = s.qfrc_con[lane]; }
  o += 5 * NV;
  for (int w = lane; w < NB * 3; w += 32) o[w] = s.xpos[w];
  o += NB * 3;
  for (int w = lane; w < NB * 9; w += 32) o[w] = s.xmat[w];
  o += NB * 9;
  const int nefc = s.nefc;
  for (int w = lane; w < nefc * NV; w += 32) {
    int r = w / NV, j = w % NV;
    double v = 0;
    if (r < s.nR) v = j < NH ? row_r(s, r)[j] : 0.0;
    else if (r < s.nR + s.nC) v = j >= NH ? row_c(s, r)[j - NH] : 0.0;
    else if (r < s.nR + s.nC + s.nF) v = row_f(s, r)[j];
    else { int meta = s.rmeta[r]; v = ((meta & 0xff) == j) ? ((meta & 0x100) ? -1.0 : 1.0) : 0.0; }
    o[row_order(s, r) * NV + j] = v;
  }
  o += nefc * NV;
  for (int w = lane; w < nefc; w += 32) { const int q = row_order(s, w); o[q] = s.earef[w]; o[nefc + q] = s.eD[w]; }
  o += 2 * nefc;
  for (int w = lane; w < s.ncon; w += 32) {
    o[w * 7] = s.cdist[w];
    for (int k = 0; k < 3; k++) { o[w * 7 + 1 + k] = s.cpos[w * 3 + k]; o[w * 7 + 4 + k] = s.cframe[w * 9 + k]; }
  }
}

// Contact output of env `env` from the last forward pass (PRM kernels): lane c < ncon writes contact c -- geom1, geom2, dim; dist, pos,
// frame, and mj_contactForce in the contact frame (mju_decodePyramid) -- and lanes past ncon zero-fill the empty slots (geom ids -1),
// so every call rewrites the env's whole row.  Pyramid forces are recomputed from eJaref, which is current at every exit of
// Newton::solve (eJv is not: it holds J search or D active there), with the formula of update_cost_grad: -D jar on active rows.
template <class S>
__device__ __noinline__ void write_contacts(const S& s, int* dst_n, int* dst_geom, double* dst_con, int env, int lane) {
  static_assert(S::HAS_PRM, "the contact output runs in the kernels with per-env parameters (env_mu)");
  const int ncon = s.ncon;
  if (lane == 0) dst_n[env] = ncon;
  if (lane < MCB_MAXCON) {
    int* g = dst_geom + ((size_t)env * MCB_MAXCON + lane) * 3;
    double* o = dst_con + ((size_t)env * MCB_MAXCON + lane) * MCB_CONTACT_DOUBLES;
    if (lane < ncon) {
      const PairParam& pp = PP(s.cpair[lane]);
      const int dim = pp.dim, r0 = s.crow[lane];
      g[0] = pp.g1; g[1] = pp.g2; g[2] = dim;
      o[0] = s.cdist[lane];
      for (int k = 0; k < 3; k++) o[1 + k] = s.cpos[lane * 3 + k];
      for (int k = 0; k < 9; k++) o[4 + k] = s.cframe[lane * 9 + k];
      double p[6];
      for (int k = 0; k < 6; k++) {
        const double jar = k < 2 * (dim - 1) ? s.eJaref[r0 + k] : 0.0;   // contact rows are inequalities: active iff jar < 0
        p[k] = jar < 0 ? -s.eD[r0 + k] * jar : 0.0;
      }
      const double mu = env_mu(s, pp);                                     // sliding (both tangents); torsional: pp.friction[1]
      o[13] = p[0] + p[1] + p[2] + p[3] + p[4] + p[5];
      o[14] = (p[0] - p[1]) * mu;
      o[15] = (p[2] - p[3]) * mu;
      o[16] = dim == 4 ? (p[4] - p[5]) * pp.friction[1] : 0.0;
      o[17] = 0.0; o[18] = 0.0;
    } else {
      g[0] = -1; g[1] = -1; g[2] = 0;
      for (int k = 0; k < MCB_CONTACT_DOUBLES; k++) o[k] = 0.0;
    }
  }
  __syncwarp();
}

// ------------------------------------------------------------------------------------------------
// The env kernel: one warp per env, Tier<TIER>::WARPS warps per CTA.  TIER 0 is the first launch over all envs; envs whose
// constraint set overflows a tier's layout leave every output untouched and enqueue themselves on that tier's redo list,
// which the next tier's launch serves (grid-stride over the list; several envs per CTA in the last tier too, for lockstep).
// PRM: the batch has per-env physics parameters (EnvS<TIER, true>); launch() picks the instantiation from the batch.
template <int TIER, bool PRM>
__global__ void __launch_bounds__(32 * Tier<TIER>::WARPS, 1) mcb_env_kernel(const __grid_constant__ StepArgs a) {   // (reset_env takes the arguments by reference: without __grid_constant__ the whole struct is copied to the stack)
  typedef EnvS<TIER, PRM> S;
  constexpr bool BIG = TIER == 2;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int wpb = Tier<TIER>::WARPS;
  S& s = *reinterpret_cast<S*>(smem_raw + MODEL_BYTES + (size_t)wid * sizeof(S));
  const DevModel* __restrict__ m = a.m;
  {  // stage the model (global -> shared), once per CTA
    const double* src = reinterpret_cast<const double*>(a.m);
    double* dst = reinterpret_cast<double*>(smem_raw);
    for (int w = threadIdx.x; w < (int)(sizeof(DevModel) / sizeof(double)); w += blockDim.x) dst[w] = src[w];
    __syncthreads();
  }
  const mcb_task_cfg& cfg = a.cfg;
  // reach envs: the hidden cube (mycobot.py:475-481 only zeroes its geom / site size) is frozen -- it is not observable and the
  // robot's dynamics do not depend on it (SURVEY D.6) -- except under reward_shaping, whose reach term reads its position
  // (mycobot.py:402-448): there it is simulated, with the zero-size box the model variant carries
  const bool sim_cube = cfg.has_object || cfg.reward_type == 2;
  const int nba = sim_cube ? NB : NB - 1;
  const int nva = sim_cube ? NV : NH;
  const int nwork = TIER == 0 ? a.n_envs : a.redo_count[TIER - 1];
  const int* work_list = TIER == 0 ? nullptr : a.redo_list + (size_t)(TIER - 1) * a.n_envs;
  if (TIER > 0 && nwork == 0) return;
  if (TIER == 1 && nwork <= a.mid_threshold) {
    // A tier pass costs the latency of one whole env-step of a single warp whatever the list length, and envs that do not
    // fit here either pay it twice.  A short list is therefore handed to the last tier as it is: its CTAs take it in one or
    // two waves.  The middle tier pays off when many envs are in contact at once (a batch of grasps).
    int* next = a.redo_list + (size_t)a.n_envs;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < nwork; i += gridDim.x * blockDim.x) next[i] = work_list[i];
    if (blockIdx.x == 0 && threadIdx.x == 0) a.redo_count[1] = nwork;
    return;
  }
  // the upper tiers always run their CTA in lockstep (their envs are the divergent, contact-rich ones: free-running they stall on
  // instruction fetch -- held grasp 59 -> 20 ms/step); the batch's grouping (mcb_autotune) only concerns the common-layout kernel
  const int lockstep = TIER == 0 ? (a.lockstep_warps > 1 ? a.lockstep_warps : 0) : LOCKSTEP_CTA;

  // Tier 0: CTA b takes the 16 consecutive envs [16 b, 16 b + 16).  Tier 1: the list is dealt round-robin over the CTAs
  // (item = slot * gridDim.x + b), so a list shorter than one full wave spreads over all SMs with few warps each instead of
  // filling half of them -- the latency of a pass is set by how many heavy envs share an SM.
  for (int item0 = TIER >= 1 ? 0 : blockIdx.x * wpb; item0 < nwork; item0 += gridDim.x * wpb) {
    const int item = TIER >= 1 ? item0 + wid * (int)gridDim.x + (int)blockIdx.x : item0 + wid;
    bool valid = item < nwork;
    const int env = valid ? (TIER == 0 ? item : work_list[item]) : 0;
    if (valid && a.mode == MODE_RESET && a.mask && !a.mask[env]) valid = false;

    // zero what has a static sparsity pattern or is read before it is first written
    for (int w = lane; w < NTRI; w += 32) { s.M[w] = 0; s.H[w] = 0; }
    for (int w = lane; w < NB * 10; w += 32) { s.cinert[w] = 0; s.crb[w] = 0; }
    for (int w = lane; w < NB * 9; w += 32) s.xmat[w] = 0;
    for (int w = lane; w < NB * 3; w += 32) s.xpos[w] = 0;
    for (int w = lane; w < NV * 6; w += 32) { s.cdof[w] = 0; s.cdof_dot[w] = 0; }
    if (lane < NV) { s.qfrc_bias[lane] = 0; s.qfrc_con[lane] = 0; s.qacc[lane] = 0; s.qacc_smooth[lane] = 0; s.qfrc_smooth[lane] = 0; s.Ma[lane] = 0; s.grad[lane] = 0; s.search[lane] = 0; s.Mv[lane] = 0; }
    if (lane == 0) { s.mesh = a.cfg.mesh_collision; s.overflow = 0; s.iters = 0; s.nefc = 0; s.ncon = 0; s.nR = MDL.d.has_weld ? 13 : 7; s.nC = s.nF = s.nU = 0; s.refcube[0] = s.refcube[1] = s.refcube[2] = 0; }
#ifdef MCB_CANARY
    if (lane < 2) { const double c = __longlong_as_double(0x7ff8c0decafe0000ll + lane); s.g0[lane] = c; s.g1[lane] = c; s.g2[lane] = c; s.g3[lane] = c; s.g4[lane] = c; s.g5[lane] = c; s.g6[lane] = c; s.g7[lane] = c; }
    if constexpr (PRM) { if (lane < 2) s.gp[lane] = __longlong_as_double(0x7ff8c0decafe0000ll + lane); }
#endif
    __syncwarp();
    unsigned long long ctr = 0;
    if (valid) { load_state(s, a.state + (size_t)env * MCB_STATE_STRIDE, lane); ctr = a.rng_ctr[env]; }
    if constexpr (PRM) {
      if (valid && lane < MCB_NPARAM) s.prm[lane] = a.x.params[(size_t)env * MCB_NPARAM + lane];
      if (lane == 0) {
        s.prm_ctr = valid ? a.x.param_ctr[env] : 0; s.prm_drawn = 0;
        s.lat_ctr = valid ? a.x.lat_ctr[env] : 0;
        s.lat = valid ? min(max(a.x.latency[env], 0), cfg.frame_skip) : 0;    // mcb_set_env_latency does not validate device data
        s.frc = valid && a.x.frc ? a.x.frc + (size_t)env * NFRC : nullptr;
      }
      __syncwarp();
    }
    double achieved[3];
    int substeps = 0;
    bool ok = valid;

    if (a.mode == MODE_RESET) {
      if (ok) ok = reset_env(s, a, m, lane, env, nba, nva, ctr);
      if (ok) {
        write_obs(s, m, cfg, lane, env, a.obs, a.ag, a.dg, achieved);
        if constexpr (PRM) { if (a.x.con_n) write_contacts(s, a.x.con_n, a.x.con_geom, a.x.con, env, lane); }
        if (lane == 0) { a.elapsed[env] = 0; a.ep_return[env] = 0; }
      }
      substeps = 2;
    } else if (a.mode == MODE_FORWARD) {
      if (ok) ok = forward(s, m, lane, nba, nva, false);
      if (ok) {
        if (lane < 6) s.qprev[lane] = s.qpos[lane];
        __syncwarp();
        write_obs(s, m, cfg, lane, env, a.obs, a.ag, a.dg, achieved);
        if (a.debug && env == a.debug_env) debug_dump(s, a, lane, nva);
        if constexpr (PRM) { if (a.x.con_n) write_contacts(s, a.x.con_n, a.x.con_geom, a.x.con, env, lane); }
      }
      substeps = 1;
    } else {
      const bool ik = cfg.controller_type == 1, mocap = cfg.controller_type == 2;
      const int adim = cfg.fetch_env ? 4 : (mocap ? 8 : NU);
      float act[8];
#pragma unroll
      for (int k = 0; k < 8; k++) act[k] = 0.0f;
      if (ok) {
        // action = clip(action, -1, 1) in float32 (mycobot.py:133)
#pragma unroll
        for (int k = 0; k < 8; k++) if (k < adim) act[k] = fminf(1.0f, fmaxf(-1.0f, a.actions[(size_t)env * adim + k]));
      }
      double grip_ctrl = 0;
      int nblocks = 1;
      // PRM kernels: the command a controller issues is held in `cmd` on the lane that owns its destination `cmd_dst` and written
      // before substep `lat` of its block (after the last one when lat == frame_skip); until then the previous command stays in force
      double cmd = 0;
      double* cmd_dst = nullptr;
      int lat = 0;
      if constexpr (PRM) lat = s.lat;
      if (mocap) {
        // mocap controller (mycobot.py:172-189 + mocap_set_action / reset_mocap2body_xpos): the mocap body goes to the
        // (stale) gripper_tcp pose plus the action deltas; the weld then drags the arm during the 20 substeps
        if (ok) {
          double qsave = lane < 6 ? s.qpos[lane] : 0.0;
          if (lane < 6) s.qpos[lane] = s.qprev[lane];
          __syncwarp();
          fk(s, m, lane, NB - 1);
          if (lane < 6) s.qpos[lane] = qsave;
          __syncwarp();
          if (lane == 0) {
            double* mdst = s.mocap;                // PRM kernels: staged in s.grad (scratch here), then held on lanes 0..7
            if constexpr (PRM) mdst = s.grad;
            double tcp[3];
            const int b2 = MDL.d.weld_body2;
            const double* R = s.xmat + b2 * 9;
            const double* a2 = MDL.d.weld_anchor2;
            for (int r = 0; r < 3; r++) tcp[r] = s.xpos[b2 * 3 + r] + R[3 * r] * a2[0] + R[3 * r + 1] * a2[1] + R[3 * r + 2] * a2[2];
            for (int k = 0; k < 3; k++) mdst[k] = tcp[k] + (double)(act[k] * 0.1f);         // float32 product, float64 sum
            const double fq[4] = {0.5, -0.5, -0.5, 0.5};
            for (int k = 0; k < 4; k++) {
              double tq = s.quat5[k];
              double want = cfg.fetch_env ? fq[k] : (double)act[3 + k];
              mdst[3 + k] = tq + (want - tq);                                                // mocap_quat + (action - tcp_quat)
            }
            float ag = cfg.fetch_env ? act[3] : act[7];
            if constexpr (PRM) s.grad[7] = 0.5 + (double)ag * 0.5;
            else
            s.ctrl[MDL.d.nu - 1] = 0.5 + (double)ag * 0.5;
          }
        }
      } else if (!ik) {
        // joint controller: ctrl = action widened to double (mycobot.py:192-193 -> MujocoEnv.do_simulation)
        if (ok && lane < NU) {
          float v = 0.0f;
#pragma unroll
          for (int k = 0; k < NU; k++) if (lane == k) v = act[k];
          if constexpr (PRM) { cmd = (double)v; cmd_dst = s.ctrl + lane; }
          else
          s.ctrl[lane] = (double)v;
        }
      } else {
        // IK controller (mycobot.py:134-170): the target comes from the site pose the reference still holds from the
        // previous step's last forward pass, i.e. from the frames at qprev
        if (ok) {
          double qsave = lane < 6 ? s.qpos[lane] : 0.0;
          if (lane < 6) s.qpos[lane] = s.qprev[lane];
          __syncwarp();
          fk(s, m, lane, NB - 1);
          cinert_cdof(s, m, lane, NB - 1, NH);
          if (lane < 6) s.qpos[lane] = qsave;
          __syncwarp();
          ik_target(s, cfg, act, lane);
        }
        float ag = 0.0f;
#pragma unroll
        for (int k = 0; k < 8; k++) if (k == adim - 1) ag = act[k];
        grip_ctrl = 0.5 + (double)ag * 0.5;          // actuation_center + action[-1] * actuation_range (mycobot.py:158-160)
        nblocks = cfg.control_steps;
        if constexpr (PRM) { if (ok && lane < NU) cmd_dst = s.ctrl + lane; }
      }
      __syncwarp();
      if constexpr (PRM) {
        if (mocap && ok && lane < 8) { cmd = s.grad[lane]; cmd_dst = lane < 7 ? s.mocap + lane : s.ctrl + (MDL.d.nu - 1); }
        __syncwarp();
      }
      for (int blk = 0; blk < nblocks; blk++) {
        if (ik && ok) ik_update_ctrl(s, lane, grip_ctrl, cmd);
        for (int it = 0; it < cfg.frame_skip; it++) {
          if constexpr (PRM) {
            if (it == lat) { if (cmd_dst) *cmd_dst = cmd; __syncwarp(); }
          }
          if (ok) ok = forward(s, m, lane, nba, nva, lockstep);
          else if (lockstep) { for (int k = 0; k < NSYNC_FWD; k++) group_sync(lockstep); }
          if (lockstep) group_sync(lockstep);
          if (ok) {
            if (lane < 6) s.qprev[lane] = s.qpos[lane];     // the frames now in shared memory belong to this qpos
            euler(s, m, lane, nva);
          }
        }
        if constexpr (PRM) {
          if (lat == cfg.frame_skip) { if (cmd_dst) *cmd_dst = cmd; __syncwarp(); }
        }
      }
      substeps = cfg.frame_skip * nblocks;
      if (ok && cfg.block_gripper) {  // _step_callback (mycobot.py:300-306)
        if (lane == 0) { s.qpos[7] = 0; s.qpos[9] = 0; }
        __syncwarp();
        ok = forward(s, m, lane, nba, nva, false);
        if (lane < 6) s.qprev[lane] = s.qpos[lane];
        __syncwarp();
        substeps++;
      }
      if (ok) {
        int el = a.elapsed[env] + 1;
        double ob_ag[3];
        write_obs(s, m, cfg, lane, env, a.obs, a.ag, a.dg, ob_ag);
        double dx = ob_ag[0] - s.goal[0], dy = ob_ag[1] - s.goal[1], dz = ob_ag[2] - s.goal[2];
        double dist = sqrt(dx * dx + dy * dy + dz * dz);
        bool succ = dist < cfg.distance_threshold;
        bool term = succ, trunc = succ || (el >= cfg.max_episode_steps);
        // bad-simulation guard (the role of mj_checkPos / mj_checkVel / mj_checkAcc in mj_step): a non-finite or exploded
        // state ends the episode (truncated) so that auto-reset restores a sane state; counted in stats[5]
        bool bad = false;
        {
          double v = lane < NQ ? s.qpos[lane] : 0.0, w = lane < NV ? s.qvel[lane] : 0.0;
          bad = __any_sync(FULLMASK, !(fabs(v) < 1e10) || !(fabs(w) < 1e10));
        }
        if (bad) { succ = false; term = false; trunc = true; if (lane == 0) atomicAdd(a.stats + 5, 1.0); }
        double rew = cfg.reward_type == 0 ? -(double)(dist > cfg.distance_threshold) : -dist;
        if (bad) { dist = 1e10; rew = cfg.reward_type == 0 ? -1.0 : 0.0; }
        if (cfg.reward_type == 2 && !bad) {
          // OracleEnv.stage_rewards (oracle/oracle.py; mycobot.py:402-448): reach / grasp / lift from the sites and the contact list of
          // the last forward pass; write_obs left grip_pos in o[0..2]; object_pos = the cube body's origin (site object0 sits on it)
          const double* o = s.grad;
          const double* op = s.xpos + CUBE * 3;
          double gx = o[0] - op[0], gy = o[1] - op[1], gz = o[2] - op[2];
          double r_reach = (1 - tanh(sqrt(gx * gx + gy * gy + gz * gz))) * 0.2;
          bool tr = false, tl = false;
          for (int c = 0; c < s.ncon; c++) {
            const PairParam& pp = PP(s.cpair[c]);
            bool hasobj = pp.g1 == MDL.d.geom_object || pp.g2 == MDL.d.geom_object;
            if (hasobj && (pp.g1 == MDL.d.geom_finger_r || pp.g2 == MDL.d.geom_finger_r)) tr = true;
            if (hasobj && (pp.g1 == MDL.d.geom_finger_l || pp.g2 == MDL.d.geom_finger_l)) tl = true;
          }
          double r_grasp = (tr && tl) ? 0.5 : 0.0, r_lift = 0.0;
          if (r_grasp > 0.0) {
            double tx = op[0] - MDL.d.target0_pos[0], ty = op[1] - MDL.d.target0_pos[1], tz = op[2] - MDL.d.target0_pos[2];
            r_lift = 0.5 + (1 - tanh(sqrt(tx * tx + ty * ty + tz * tz))) * (0.9 - 0.5);
          }
          rew = fmax(fmax(r_reach, r_grasp), r_lift) * 100;
        }
        double epret = a.ep_return[env] + rew;
        bool done = term || trunc;
        double final_stats[4] = {1.0, succ ? 1.0 : 0.0, epret, (double)el};
        if ((done && cfg.auto_reset) || bad) {
          if (a.final_obs) {
            double dummy[3];
            write_obs(s, m, cfg, lane, env, a.final_obs, nullptr, nullptr, dummy);
          }
          if constexpr (PRM) { if (a.x.con_fn) write_contacts(s, a.x.con_fn, a.x.con_fgeom, a.x.con_f, env, lane); }   // the terminal state's
          ok = reset_env(s, a, m, lane, env, nba, nva, ctr);
          if (ok) write_obs(s, m, cfg, lane, env, a.obs, a.ag, a.dg, achieved);
          el = 0; epret = 0; substeps += 2;
        }
        // the last forward pass: the substep loop's or the block_gripper one (euler, write_obs and the reward leave the rows alone),
        // or the reset's for an env that was just reset
        if constexpr (PRM) { if (ok && a.x.con_n) write_contacts(s, a.x.con_n, a.x.con_geom, a.x.con, env, lane); }
        if (ok && lane == 0) {
          if (cfg.reward_type == 0) ((float*)a.reward)[env] = -(float)(dist > cfg.distance_threshold);
          else ((double*)a.reward)[env] = rew;
          a.terminated[env] = term; a.truncated[env] = trunc; a.success[env] = succ;
          if (done) { for (int k = 0; k < 4; k++) atomicAdd(a.stats + k, final_stats[k]); }
          a.elapsed[env] = el; a.ep_return[env] = epret;
        }
      }
    }
    __syncwarp();
#ifdef MCB_CANARY
    if (a.canary_selftest && lane == 0) s.cframe[S::MAXC * 9] = 1.0;      // one past the end: lands on guard g7
    __syncwarp();
    if (lane < 2) {
      const long long c = 0x7ff8c0decafe0000ll + lane;
      const double* g[8] = {s.g0, s.g1, s.g2, s.g3, s.g4, s.g5, s.g6, s.g7};
      for (int k = 0; k < 8; k++)
        if (__double_as_longlong(g[k][lane]) != c) { atomicAdd(a.stats + 5, 1.0e6); printf("MCB_CANARY: guard %d of env %d (tier %d) was overwritten\n", k, env, TIER); }
      if constexpr (PRM) {
        if (__double_as_longlong(s.gp[lane]) != c) { atomicAdd(a.stats + 5, 1.0e6); printf("MCB_CANARY: guard %d of env %d (tier %d) was overwritten\n", 8, env, TIER); }
      }
    }
    __syncwarp();
#endif
    if (valid) {
      if (!ok) {
        // this tier's layout overflowed: leave the env untouched for the next tier's launch
        // (observation rows written above are rewritten by it; state, counters and statistics are not yet committed)
        if (TIER < 2 && lane == 0) { int k = atomicAdd(a.redo_count + TIER, 1); a.redo_list[(size_t)TIER * a.n_envs + k] = env; }
      } else {
        store_state(s, a.state + (size_t)env * MCB_STATE_STRIDE, lane);
        if constexpr (PRM) {
          if (s.prm_drawn) {
            if (lane < MCB_NPARAM) a.x.params[(size_t)env * MCB_NPARAM + lane] = s.prm[lane];
            if (lane == 0) { a.x.param_ctr[env] = s.prm_ctr; a.x.latency[env] = s.lat; a.x.lat_ctr[env] = s.lat_ctr; }
          }
          if (a.x.frc && !s.frc) { for (int w = lane; w < NFRC; w += 32) a.x.frc[(size_t)env * NFRC + w] = 0.0; }   // a reset cleared the forces
        }
        if (lane == 0) {
          a.rng_ctr[env] = ctr;
          if (a.mode == MODE_STEP) atomicAdd(a.stats + 4, 1.0);
          if (BIG && s.overflow) atomicAdd(a.stats + 5, (double)s.overflow);
          atomicAdd(a.stats + 6, (double)s.iters);
          atomicAdd(a.stats + 7, (double)substeps);
        }
      }
    }
    __syncwarp();
  }
}

__global__ void reward_kernel(const double* __restrict__ ag, const double* __restrict__ g, int64_t n, double thr, int type, void* out) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double dx = ag[3 * i] - g[3 * i], dy = ag[3 * i + 1] - g[3 * i + 1], dz = ag[3 * i + 2] - g[3 * i + 2];
  double d = sqrt(dx * dx + dy * dy + dz * dz);
  if (type == 0) ((float*)out)[i] = -(float)(d > thr);
  else ((double*)out)[i] = -d;
}

__global__ void init_state_kernel(double* state, int* elapsed, double* ep_return, unsigned long long* ctr, unsigned long long* env_seed, unsigned long long seed, const DevModel* m, int n, int fetch) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double* st = state + (size_t)i * MCB_STATE_STRIDE;
  for (int k = 0; k < MCB_STATE_STRIDE; k++) st[k] = 0;
  const double* q0 = init_qpos_of(*m, fetch);
  const double* c0 = init_ctrl_of(*m, fetch);
  for (int k = 0; k < NQ; k++) st[ST_QPOS + k] = q0[k];
  for (int k = 0; k < NU; k++) st[ST_CTRL + k] = c0[k];
  for (int k = 0; k < 6; k++) st[ST_QPREV + k] = q0[k];
  const double* mp = fetch ? m->d.key_mocap_pos : m->d.mocap_pos0;
  const double* mq = fetch ? m->d.key_mocap_quat : m->d.mocap_quat0;
  for (int k = 0; k < 3; k++) st[ST_MOCAP + k] = mp[k];
  for (int k = 0; k < 4; k++) st[ST_MOCAP + 3 + k] = mq[k];
  elapsed[i] = 0; ep_return[i] = 0; ctr[i] = 0; env_seed[i] = seed;
}

// DFMA throughput probe: 8 independent chains per thread
__global__ void dfma_probe_kernel(double* out, int iters) {
  double a0 = threadIdx.x * 1e-9, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
  const double b = 1.0000001, c = 1e-9;
  for (int i = 0; i < iters; i++) {
    a0 = fma(a0, b, c); a1 = fma(a1, b, c); a2 = fma(a2, b, c); a3 = fma(a3, b, c);
    a4 = fma(a4, b, c); a5 = fma(a5, b, c); a6 = fma(a6, b, c); a7 = fma(a7, b, c);
  }
  double sum = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
  if (sum == 123.456) out[0] = sum;
}


// uniform float32 actions in [-1, 1) for mcb_autotune's roll-ahead (Philox stream of its own)
__global__ void random_actions_kernel(float* act, int n, uint64_t seed, unsigned step) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  unsigned long long ctr = (unsigned long long)step << 32;
  act[i] = (float)(2.0 * philox_uniform(seed, (uint32_t)i, ctr) - 1.0);
}

// mcb_seed(): MyCobotEnv.reset(seed=) reseeds the env's generator (mycobot.py:509-510) -> new Philox key, draw counter 0
// (pctr, lctr: the parameter and latency draw counters of a batch with per-env parameters, or null)
__global__ void seed_kernel(unsigned long long* env_seed, unsigned long long* ctr, unsigned long long* pctr, unsigned long long* lctr, const uint8_t* mask,
                            unsigned long long seed, int n) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n && (!mask || mask[i])) { env_seed[i] = seed; ctr[i] = 0; if (pctr) pctr[i] = 0; if (lctr) lctr[i] = 0; }
}
// A row copy between a batch's arrays and caller arrays, one thread per (env, column): up to IO_MAXBLK column blocks, each the columns
// [col, col + width) of a batch array with rows of `stride` elements of `elem` (4 or 8) bytes <-> the first `width` columns of a
// caller array with rows of `ustride` elements.  GET: batch -> caller, a null batch array reads as the bit pattern `absent`; SET:
// caller -> batch; FILL: `absent` -> batch.  No two blocks of a list write the same element, so their order does not matter.
enum { IO_GET, IO_SET, IO_FILL, IO_MAXBLK = 8 };
struct IoBlock { char *arr, *user; int stride, col, width, ustride, elem; unsigned long long absent; };
struct IoList {
  int dir, n = 0, width = 0;     // width: the columns of all blocks, per env
  IoBlock blk[IO_MAXBLK];
  // adds a block unless it has no caller array (a GET or SET call leaves such an array alone)
  template <class T> IoList& add(T* arr, int stride, int col, int width, const void* user, T absent = T(), int ustride = 0) {
    static_assert(sizeof(T) == 4 || sizeof(T) == 8, "4- or 8-byte elements");
    if (!user && dir != IO_FILL) return *this;
    IoBlock& c = blk[n++];
    c = {(char*)arr, (char*)user, stride, col, width, ustride ? ustride : width, (int)sizeof(T), 0};
    memcpy(&c.absent, &absent, sizeof(T));
    this->width += width;
    return *this;
  }
};
template <class T> __device__ void copy_element(int dir, const IoBlock& c, size_t ia, size_t iu) {
  T* arr = reinterpret_cast<T*>(c.arr);
  T* user = reinterpret_cast<T*>(c.user);
  const T absent = (T)c.absent;
  if (dir == IO_GET) user[iu] = arr ? arr[ia] : absent;
  else arr[ia] = dir == IO_SET ? user[iu] : absent;
}
__global__ void copy_rows_kernel(const __grid_constant__ IoList l, int n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)n * l.width) return;
  const long long env = i / l.width;
  int k = (int)(i - env * l.width), j = 0;
  while (k >= l.blk[j].width) k -= l.blk[j++].width;
  const IoBlock& c = l.blk[j];
  const size_t ia = (size_t)env * c.stride + c.col + k, iu = (size_t)env * c.ustride + k;
  if (c.elem == 8) copy_element<unsigned long long>(l.dir, c, ia, iu);
  else copy_element<unsigned int>(l.dir, c, ia, iu);
}
__global__ void iota_kernel(int* list, int* count, int n) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) list[i] = i;
  if (i == 0) *count = n;
}

#define DEBUG_DOUBLES (4 + NV * NV + 5 * NV + NB * 12 + Tier<2>::NROW * NV + 2 * Tier<2>::NROW + 7 * Tier<2>::MAXC)

}  // namespace

// ================================================================================================
// ABI calls that need a particular device make it current for their own duration only (the caller's current device is restored)
struct DevGuard {
  int prev = -1; bool ok = true;
  explicit DevGuard(int dev) { ok = cudaGetDevice(&prev) == cudaSuccess && (prev == dev || cudaSetDevice(dev) == cudaSuccess); if (prev == dev) prev = -1; }
  ~DevGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

// Row constants of mj_makeImpedance that do not depend on the state, computed once per model: `si` is clamped to getimpedance's
// limits (slot 2 becomes 1 / width), and `KB` holds the row's solref on entry and its (K, B), refsafe applied, on return.  In the
// DEVICE copy of the model every *_solref pair is overwritten with its (K, B) -- the kernels never need the raw solref.
static void row_constants(double* KB, double* si, double timestep) {
  si[0] = fmin(MAXIMP, fmax(MINIMP, si[0])); si[1] = fmin(MAXIMP, fmax(MINIMP, si[1])); si[2] = fmax(0.0, si[2]) <= MINVAL ? 0.0 : 1.0 / si[2];
  si[3] = fmin(MAXIMP, fmax(MINIMP, si[3])); si[4] = fmax(1.0, si[4]);
  double sr0 = KB[0], sr1 = KB[1];
  if (sr0 > 0) sr0 = fmax(sr0, 2 * timestep);
  const double dmax = si[1];
  if (sr0 > 0) { KB[0] = 1 / fmax(MINVAL, dmax * dmax * sr0 * sr0 * sr1 * sr1); KB[1] = 2 / fmax(MINVAL, dmax * sr0); }
  else { KB[0] = -sr0 / fmax(MINVAL, dmax * dmax); KB[1] = -sr1 / fmax(MINVAL, dmax); }
}

// One side of a candidate contact pair: a primitive geom of the model or a convex hull standing for `mult` identical mesh geoms.
struct Side {
  int condim; const double *friction, *solref, *solimp; double solmix; const double* invweight; int body, mult;
};
static Side geom_side(const mcb_model_desc& d, int g) {
  return {d.geom_condim[g], d.geom_friction[g], d.geom_solref[g], d.geom_solimp[g], d.geom_solmix[g], d.geom_invweight[g], d.geom_body[g], 1};
}
static Side hull_side(const mcb_hull_desc& hd, int h) {
  return {hd.condim[h], hd.friction[h], hd.solref[h], hd.solimp[h], hd.solmix[h], hd.invweight[h], hd.body[h], hd.mult[h]};
}

// Contact parameters of one pair (mj_contactParam, same priority: condim and friction as maxima, solref / solimp mixed by solmix)
// and their row constants.  The caller fills g1 / g2.  Returns false for a condim other than 3 or 4.
static bool pair_param(PairParam& pp, const Side& a, const Side& b, double timestep, double impratio) {
  pp.b1 = a.body; pp.b2 = b.body;
  pp.dim = a.condim > b.condim ? a.condim : b.condim;
  if (pp.dim != 3 && pp.dim != 4) return false;
  for (int k = 0; k < 3; k++) pp.friction[k] = fmax(a.friction[k], b.friction[k]);
  double mix;
  if (a.solmix >= MINVAL && b.solmix >= MINVAL) mix = a.solmix / (a.solmix + b.solmix);
  else if (a.solmix < MINVAL && b.solmix < MINVAL) mix = 0.5;
  else if (a.solmix < MINVAL) mix = 0.0; else mix = 1.0;
  if (a.solref[0] > 0 && b.solref[0] > 0) for (int k = 0; k < 2; k++) pp.KB[k] = mix * a.solref[k] + (1 - mix) * b.solref[k];
  else for (int k = 0; k < 2; k++) pp.KB[k] = fmin(a.solref[k], b.solref[k]);
  for (int k = 0; k < 5; k++) pp.solimp[k] = mix * a.solimp[k] + (1 - mix) * b.solimp[k];
  { const bool c1 = a.body == CUBE, c2 = b.body == CUBE, r1 = a.body >= 0 && !c1, r2 = b.body >= 0 && !c2;
    pp.ptype = ((c1 || c2) && (r1 || r2)) ? 2 : ((c1 || c2) ? 1 : 0); }
  pp.tran = a.invweight[0] + b.invweight[0];
  row_constants(pp.KB, pp.solimp, timestep);
  const double pyr = pp.friction[0] / sqrt(impratio);
  pp.pyr2 = 2 * pyr * pyr / (double)(a.mult * b.mult);      // `mult` identical contacts (twin mesh geoms) == one contact with R / mult
  return true;
}

struct mcb_model {
  int device;
  DevModel* dev;
  DevModel host;
  double* d_hull_vert = nullptr;
  PairParam* d_hpair = nullptr;
};

struct mcb_batch {
  mcb_model* model;
  int n_envs, obs_dim, big_only, mid_only, sm_count;
  int* redo_count; int* redo_list;
  mcb_task_cfg cfg;
  uint64_t seed;
  double* state; int* elapsed; double* ep_return; unsigned long long* rng_ctr; unsigned long long* env_seed; double* stats;
  double* debug;
  int last_launches;
  long long launches_total;   // kernels this library launched on behalf of the batch (counted at the launch sites)
  int lockstep_warps, tuned;
  // per-env extensions: the parameters and latencies are null until a call turns per-env parameters on (enable_params), the applied
  // forces until mcb_set_env_applied, the contact output until mcb_set_contact_output registers the caller's arrays
  EnvExt x;
  // staging for the host-buffer entry point
  float* d_actions; double *d_obs, *d_ag, *d_dg, *d_fobs; void* d_reward; uint8_t* d_flags;
  float* h_actions; double *h_obs, *h_ag, *h_dg, *h_fobs; void* h_reward; uint8_t* h_flags;
};

template <int TIER, bool PRM = false> static cudaError_t set_tier_smem() {
  cudaError_t e = cudaFuncSetAttribute(mcb_env_kernel<TIER, PRM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cta_bytes<TIER, PRM>());
  if (e == cudaSuccess) e = cudaFuncSetAttribute(mcb_env_kernel<TIER, PRM>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
  return e;
}
template <bool PRM>
static cudaError_t launch_tiers(mcb_batch* b, const StepArgs& a, cudaStream_t st) {
  cudaError_t e = cudaMemsetAsync(b->redo_count, 0, 2 * sizeof(int), st);
  if (e != cudaSuccess) return e;
  if (b->big_only) iota_kernel<<<(b->n_envs + 255) / 256, 256, 0, st>>>(b->redo_list + b->n_envs, b->redo_count + 1, b->n_envs);
  else if (b->mid_only) iota_kernel<<<(b->n_envs + 255) / 256, 256, 0, st>>>(b->redo_list, b->redo_count, b->n_envs);
  else mcb_env_kernel<0, PRM><<<(b->n_envs + Tier<0>::WARPS - 1) / Tier<0>::WARPS, 32 * Tier<0>::WARPS, cta_bytes<0, PRM>(), st>>>(a);
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  b->launches_total += 1 + (b->big_only ? 0 : 1) + 1;      // this one, the middle tier (unless last-tier-only), the last tier
  // envs that overflowed the common layout (grid-stride over the device list; empty in contact-free workloads) ...
  if (!b->big_only) mcb_env_kernel<1, PRM><<<b->mid_only ? (b->n_envs + Tier<1>::WARPS - 1) / Tier<1>::WARPS : b->sm_count, 32 * Tier<1>::WARPS, cta_bytes<1, PRM>(), st>>>(a);
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  // ... and the few that overflowed the middle one
  mcb_env_kernel<2, PRM><<<b->big_only ? (b->n_envs + Tier<2>::WARPS - 1) / Tier<2>::WARPS : b->sm_count, 32 * Tier<2>::WARPS, cta_bytes<2, PRM>(), st>>>(a);
  return cudaGetLastError();
}

// The PRM = true kernels are compiled in a translation unit of their own, mcb_engine_prm.cu (this file with MCB_PRM_UNIT defined):
// ptxas allocates registers across the call graph of a module, and the math library's slow paths (sincos argument reduction, pow)
// are functions every env kernel calls, so further env kernels in this module would change the code of the default ones.  Apart,
// the default kernels compile exactly as they would without per-env parameters.  These two calls are the units' interface;
// `args` points to a StepArgs.
cudaError_t prm_launch_tiers(mcb_batch* b, const void* args, cudaStream_t st);
cudaError_t prm_set_tier_smem();
#ifdef MCB_PRM_UNIT
cudaError_t prm_launch_tiers(mcb_batch* b, const void* args, cudaStream_t st) { return launch_tiers<true>(b, *static_cast<const StepArgs*>(args), st); }
cudaError_t prm_set_tier_smem() {
  cudaError_t e = set_tier_smem<0, true>();
  if (e == cudaSuccess) e = set_tier_smem<1, true>();
  if (e == cudaSuccess) e = set_tier_smem<2, true>();
  return e;
}
#else
static int launch(mcb_batch* b, StepArgs& a, cudaStream_t st) {
  a.m = b->model->dev; a.n_envs = b->n_envs; a.cfg = b->cfg; a.env_seed = b->env_seed;
  a.state = b->state; a.elapsed = b->elapsed; a.ep_return = b->ep_return; a.rng_ctr = b->rng_ctr; a.stats = b->stats;
  a.redo_count = b->redo_count; a.redo_list = b->redo_list;
  a.lockstep_warps = b->lockstep_warps;
#ifdef MCB_CANARY
  { const char* st_ = getenv("MCB_CANARY_SELFTEST"); a.canary_selftest = (st_ && st_[0] == '1') ? 1 : 0; }
#endif
  a.mid_threshold = b->mid_only ? -1 : 2 * Tier<2>::WARPS * b->sm_count;    // up to two waves of the last tier are cheaper than a middle-tier pass (profiles/README.md)
  a.x = b->x;
  const cudaError_t e = b->x.params ? prm_launch_tiers(b, &a, st) : launch_tiers<false>(b, a, st);
  if (e != cudaSuccess) return fail("launching the step kernels", e);
  return 0;
}

// Every device array of a batch, described once: its member, its size (bytes per env plus a fixed part), the group it is allocated
// with and whether a Snapshot carries it (what a step changes).  G_CONTACT arrays are the caller's (mcb_set_contact_output); the
// batch allocates and frees the others.  A null array is absent: per-env parameters, applied forces or contact output are off.
enum { G_CORE, G_PARAMS, G_FORCES, G_CONTACT };
struct BatchArray { size_t off, per_env, fixed; int group; bool saved; };
static const BatchArray kBatchArrays[] = {
    {offsetof(mcb_batch, state), MCB_STATE_STRIDE * sizeof(double), 0, G_CORE, true},
    {offsetof(mcb_batch, ep_return), sizeof(double), 0, G_CORE, true},
    {offsetof(mcb_batch, elapsed), sizeof(int), 0, G_CORE, true},
    {offsetof(mcb_batch, rng_ctr), sizeof(unsigned long long), 0, G_CORE, true},
    {offsetof(mcb_batch, stats), 0, 8 * sizeof(double), G_CORE, true},
    {offsetof(mcb_batch, env_seed), sizeof(unsigned long long), 0, G_CORE, false},
    {offsetof(mcb_batch, redo_count), 0, 2 * sizeof(int), G_CORE, false},
    {offsetof(mcb_batch, redo_list), 2 * sizeof(int), 0, G_CORE, false},
    {offsetof(mcb_batch, debug), 0, DEBUG_DOUBLES * sizeof(double), G_CORE, false},
    {offsetof(mcb_batch, x.params), MCB_NPARAM * sizeof(double), 0, G_PARAMS, true},
    {offsetof(mcb_batch, x.param_ctr), sizeof(unsigned long long), 0, G_PARAMS, true},
    {offsetof(mcb_batch, x.latency), sizeof(int), 0, G_PARAMS, true},
    {offsetof(mcb_batch, x.lat_ctr), sizeof(unsigned long long), 0, G_PARAMS, true},
    {offsetof(mcb_batch, x.frc), NFRC * sizeof(double), 0, G_FORCES, true},
    {offsetof(mcb_batch, x.con_n), sizeof(int), 0, G_CONTACT, true},
    {offsetof(mcb_batch, x.con_geom), MCB_MAXCON * 3 * sizeof(int), 0, G_CONTACT, true},
    {offsetof(mcb_batch, x.con), MCB_MAXCON * MCB_CONTACT_DOUBLES * sizeof(double), 0, G_CONTACT, true},
    {offsetof(mcb_batch, x.con_fn), sizeof(int), 0, G_CONTACT, true},
    {offsetof(mcb_batch, x.con_fgeom), MCB_MAXCON * 3 * sizeof(int), 0, G_CONTACT, true},
    {offsetof(mcb_batch, x.con_f), MCB_MAXCON * MCB_CONTACT_DOUBLES * sizeof(double), 0, G_CONTACT, true},
};
enum { NARRAY = sizeof kBatchArrays / sizeof kBatchArrays[0] };
static void*& array_of(mcb_batch* b, const BatchArray& d) { return *reinterpret_cast<void**>(reinterpret_cast<char*>(b) + d.off); }
static size_t bytes_of(const mcb_batch* b, const BatchArray& d) { return (size_t)b->n_envs * d.per_env + d.fixed; }

static void free_group(mcb_batch* b, int group) {
  for (const BatchArray& d : kBatchArrays)
    if (d.group == group) { cudaFree(array_of(b, d)); array_of(b, d) = nullptr; }
}
// Allocates the arrays of one group, zero-filled, all or none (a failure leaves the group null).  Synchronises the device.
static cudaError_t alloc_group(mcb_batch* b, int group) {
  cudaError_t e = cudaSuccess;
  for (const BatchArray& d : kBatchArrays) {
    if (d.group != group || e != cudaSuccess) continue;
    void* p = nullptr;
    e = cudaMalloc(&p, bytes_of(b, d));
    if (e == cudaSuccess) { array_of(b, d) = p; e = cudaMemset(p, 0, bytes_of(b, d)); }
  }
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  if (e != cudaSuccess) free_group(b, group);
  return e;
}

// One launch of copy_rows_kernel over the batch's envs (a list without blocks launches too: one launch per ABI call).
static cudaError_t copy_rows(mcb_batch* b, const IoList& l, cudaStream_t st) {
  const long long n = (long long)b->n_envs * l.width;
  copy_rows_kernel<<<n ? (unsigned)((n + 255) / 256) : 1u, 256, 0, st>>>(l, b->n_envs);
  const cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) b->launches_total++;
  return e;
}

// Turns per-env parameters on: allocates them and the actuation latencies, sets every env to the nominal values (1.0, latency 0, draw
// counters 0) and prepares the PRM kernels.  Synchronises the device.  A failure leaves the batch without per-env parameters.
static int enable_params(mcb_batch* b, const char* who) {
  if (b->x.params) return 0;
  if (b->cfg.mesh_collision) { g_err = who; g_err += ": per-env parameters are not supported with mesh_collision (hull pairs keep the model's friction)"; return -1; }
  DevGuard guard(b->model->device);
  if (!guard.ok) return fail("enable per-env parameters: cannot select the batch's device", cudaGetLastError());
  cudaError_t e = prm_set_tier_smem();
  if (e == cudaSuccess) e = alloc_group(b, G_PARAMS);
  if (e == cudaSuccess) e = copy_rows(b, IoList{IO_FILL}.add(b->x.params, MCB_NPARAM, 0, MCB_NPARAM, nullptr, 1.0), nullptr);
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  if (e != cudaSuccess) { free_group(b, G_PARAMS); return fail("enable per-env parameters", e); }
  return 0;
}

// The staging buffers of mcb_step_host exist all together or not at all (the pointers are null).
static void free_staging(mcb_batch* b) {
  cudaFree(b->d_actions); cudaFree(b->d_obs); cudaFree(b->d_fobs); cudaFree(b->d_ag); cudaFree(b->d_dg); cudaFree(b->d_reward); cudaFree(b->d_flags);
  void* host[7] = {b->h_actions, b->h_obs, b->h_fobs, b->h_ag, b->h_dg, b->h_reward, b->h_flags};
  for (void* p : host) if (p) cudaFreeHost(p);
  b->d_actions = nullptr; b->d_obs = b->d_fobs = b->d_ag = b->d_dg = nullptr; b->d_reward = nullptr; b->d_flags = nullptr;
  b->h_actions = nullptr; b->h_obs = b->h_fobs = b->h_ag = b->h_dg = nullptr; b->h_reward = nullptr; b->h_flags = nullptr;
}
static cudaError_t alloc_staging(mcb_batch* b) {
  const size_t N = (size_t)b->n_envs, od = (size_t)b->obs_dim, ad = (size_t)mcb_batch_action_dim(b);
  cudaError_t e = cudaSuccess;
  auto dev = [&](auto** p, size_t bytes) { if (e == cudaSuccess) e = cudaMalloc(p, bytes); };
  auto host = [&](auto** p, size_t bytes) { if (e == cudaSuccess) e = cudaMallocHost(p, bytes); };
  dev(&b->d_actions, N * ad * sizeof(float)); host(&b->h_actions, N * ad * sizeof(float));
  dev(&b->d_obs, N * od * sizeof(double)); host(&b->h_obs, N * od * sizeof(double));
  dev(&b->d_fobs, N * od * sizeof(double)); host(&b->h_fobs, N * od * sizeof(double));
  dev(&b->d_ag, N * 3 * sizeof(double)); host(&b->h_ag, N * 3 * sizeof(double));
  dev(&b->d_dg, N * 3 * sizeof(double)); host(&b->h_dg, N * 3 * sizeof(double));
  dev(&b->d_reward, N * sizeof(double)); host(&b->h_reward, N * sizeof(double));
  dev(&b->d_flags, N * 3); host(&b->h_flags, N * 3);
  if (e == cudaSuccess) e = cudaMemset(b->d_fobs, 0, N * od * sizeof(double));      // rows of envs that did not auto-reset are never written
  if (e != cudaSuccess) free_staging(b);
  return e;
}

// A device copy of what a step changes in a batch: the arrays of kBatchArrays marked `saved` that the batch has.  The buffers are
// allocated by the first save() and freed with the snapshot.
struct Snapshot {
  mcb_batch* b;
  void* copy[NARRAY] = {};
  explicit Snapshot(mcb_batch* batch) : b(batch) {}
  ~Snapshot() { for (void* p : copy) cudaFree(p); }
  cudaError_t save(cudaStream_t st) { return transfer(true, st); }
  cudaError_t restore(cudaStream_t st) { return transfer(false, st); }

 private:
  cudaError_t transfer(bool save, cudaStream_t st) {
    cudaError_t e = cudaSuccess;
    for (int k = 0; k < NARRAY && e == cudaSuccess; k++) {
      const BatchArray& d = kBatchArrays[k];
      void* live = array_of(b, d);
      if (!d.saved || !live) continue;
      if (save && !copy[k]) e = cudaMalloc(&copy[k], bytes_of(b, d));
      if (e == cudaSuccess) e = cudaMemcpyAsync(save ? copy[k] : live, save ? live : copy[k], bytes_of(b, d), cudaMemcpyDeviceToDevice, st);
    }
    return e;
  }
};

extern "C" {

const char* mcb_version(void) {
  static char buf[320];
  snprintf(buf, sizeof buf, "mycobot_b200 0.5 (sm_100a; shared memory per env: %zu B common layout (%d per CTA), %zu B middle tier (%d per CTA), %zu B last tier (%d per CTA); model %zu B; CTAs %zu / %zu / %zu B)",
           sizeof(EnvS<0>), (int)Tier<0>::WARPS, sizeof(EnvS<1>), (int)Tier<1>::WARPS, sizeof(EnvS<2>), (int)Tier<2>::WARPS, (size_t)MODEL_BYTES,
           cta_bytes<0>(), cta_bytes<1>(), cta_bytes<2>());
  return buf;
}
const char* mcb_last_error(void) { return g_err.c_str(); }
int32_t mcb_model_desc_size(void) { return (int32_t)sizeof(mcb_model_desc); }
int32_t mcb_task_cfg_size(void) { return (int32_t)sizeof(mcb_task_cfg); }

int32_t mcb_model_create(const mcb_model_desc* d, int32_t device, mcb_model** out) {
  if (!d || !out) return fail("mcb_model_create: null argument");
  DevGuard guard(device);
  if (!guard.ok) return fail("mcb_model_create: cannot select the device", cudaGetLastError());
  mcb_model* m = new mcb_model();
  m->device = device;
  DevModel& h = m->host;
  memset(&h, 0, sizeof h);
  h.d = *d;
  // level tables
  int maxl = 0;
  for (int b = 0; b < NB; b++) if (d->level[b] > maxl) maxl = d->level[b];
  h.nlevel = maxl + 1;
  int pos = 0;
  for (int L = 0; L <= maxl; L++) {
    h.level_start[L] = pos;
    for (int b = 0; b < NB; b++) if (d->level[b] == L) h.level_body[pos++] = b;
  }
  h.level_start[maxl + 1] = pos;
  // non-zeros of M: (i, j) with j an ancestor dof of i (or i itself)
  for (int b = 0; b < NB; b++)
    if (d->parent[b] != kTreeParent[b]) { delete m; return fail("mcb_model_create: the kinematic tree differs from the myCobot 280 tree the kernels are written against (kTreeParent)"); }
  if (d->has_weld && (d->weld_body2 < 0 || d->weld_body2 > 5)) { delete m; return fail("mcb_model_create: the weld must attach to an arm body (0..5)"); }
  int n = 0;
  for (int i = 0; i < NV; i++) {
    uint32_t mask = d->ancmask[d->dof_body[i]];
    for (int j = 0; j <= i; j++)
      if ((mask >> j) & 1u) { if (n >= NMNZ_MAX) { delete m; return fail("mcb_model_create: too many M non-zeros"); } h.mnz_i[n] = (unsigned char)i; h.mnz_j[n] = (unsigned char)j; n++; }
  }
  h.nmnz = n;
  for (int i = 0, e = 0; i < NV; i++) for (int j = 0; j <= i; j++, e++) { h.tri_i[e] = (unsigned char)i; h.tri_j[e] = (unsigned char)j; }
  // contact parameter mixing per candidate pair (mj_collideGeoms / mj_contactParam)
  if (d->npair > MCB_MAXPAIR) { delete m; return fail("mcb_model_create: too many pairs"); }
  for (int p = 0; p < d->npair; p++) {
    const int g1 = d->pair_g1[p], g2 = d->pair_g2[p];
    PairParam& pp = h.pair[p];
    pp.g1 = g1; pp.g2 = g2;
    if (!pair_param(pp, geom_side(*d, g1), geom_side(*d, g2), d->timestep, d->impratio)) { delete m; return fail("mcb_model_create: only condim 3 and 4 are supported"); }
  }
  const double ts = h.d.timestep;
  for (int e = 0; e < 2; e++) row_constants(h.d.con_solref[e], h.d.con_solimp[e], ts);
  row_constants(h.d.jeq_solref, h.d.jeq_solimp, ts);
  row_constants(h.d.weld_solref, h.d.weld_solimp, ts);
  for (int j = 0; j < NH; j++) row_constants(h.d.jnt_solref[j], h.d.jnt_solimp[j], ts);
  cudaError_t ce = cudaMalloc(&m->dev, sizeof(DevModel));
  if (ce == cudaSuccess) ce = cudaMemcpy(m->dev, &h, sizeof(DevModel), cudaMemcpyHostToDevice);
  if (ce != cudaSuccess) { cudaFree(m->dev); delete m; return fail("mcb_model_create: upload", ce); }
  *out = m;
  return 0;
}

int32_t mcb_hull_desc_size(void) { return (int32_t)sizeof(mcb_hull_desc); }

int32_t mcb_model_set_hulls(mcb_model* m, const mcb_hull_desc* hd) {
  if (!m || !hd) return fail("mcb_model_set_hulls: null argument");
  if (hd->nhull < 0 || hd->nhull > MCB_MAXHULL || hd->npair < 0 || hd->npair > MCB_MAXHPAIR || hd->nvert < 0 || (hd->nvert > 0 && !hd->vert))
    return fail("mcb_model_set_hulls: counts out of range");
  DevGuard guard(m->device);
  if (!guard.ok) return fail("mcb_model_set_hulls: cannot select the model's device", cudaGetLastError());
  // everything is validated and uploaded into a copy of the host model first: a rejected descriptor or a failed upload leaves the
  // model as it was
  DevModel h = m->host;
  std::vector<PairParam> pps((size_t)hd->npair);
  for (int hq = 0; hq < hd->nhull; hq++) {
    if (hd->body[hq] < 0 || hd->body[hq] >= NB || hd->vadr[hq] < 0 || hd->vnum[hq] <= 0 || hd->vadr[hq] + hd->vnum[hq] > hd->nvert || hd->mult[hq] < 1 ||
        (hd->condim[hq] != 3 && hd->condim[hq] != 4))
      return fail("mcb_model_set_hulls: bad hull (hulls must ride on jointed bodies, condim 3 or 4)");
    h.hull_body[hq] = hd->body[hq]; h.hull_vadr[hq] = hd->vadr[hq]; h.hull_vnum[hq] = hd->vnum[hq];
    for (int k = 0; k < 3; k++) h.hull_center[hq][k] = hd->center[hq][k];
    h.hull_rbound[hq] = hd->rbound[hq];
  }
  for (int p = 0; p < hd->npair; p++) {
    const int oa = hd->pair_a[p], ob = hd->pair_b[p];
    if (ob < MCB_NGEOM || ob >= MCB_NGEOM + hd->nhull || oa >= MCB_NGEOM + hd->nhull || (oa >= MCB_NGEOM && oa >= ob)) return fail("mcb_model_set_hulls: bad pair");
    h.hpair_a[p] = (unsigned char)oa; h.hpair_b[p] = (unsigned char)ob;
    // object a: primitive geom or hull; object b: always a hull
    PairParam& pp = pps[(size_t)p];
    pp.g1 = oa; pp.g2 = ob;
    const Side a = oa >= MCB_NGEOM ? hull_side(*hd, oa - MCB_NGEOM) : geom_side(h.d, oa);
    if (!pair_param(pp, a, hull_side(*hd, ob - MCB_NGEOM), h.d.timestep, h.d.impratio)) return fail("mcb_model_set_hulls: only condim 3 and 4 are supported");
  }
  double* vert = nullptr;
  PairParam* hpair = nullptr;
  const size_t vbytes = (size_t)hd->nvert * 3 * sizeof(double), pbytes = (size_t)hd->npair * sizeof(PairParam);
  cudaError_t e = cudaSuccess;
  if (vbytes) { e = cudaMalloc(&vert, vbytes); if (e == cudaSuccess) e = cudaMemcpy(vert, hd->vert, vbytes, cudaMemcpyHostToDevice); }
  if (pbytes && e == cudaSuccess) { e = cudaMalloc(&hpair, pbytes); if (e == cudaSuccess) e = cudaMemcpy(hpair, pps.data(), pbytes, cudaMemcpyHostToDevice); }
  h.nhull = hd->nhull; h.nhpair = hd->npair; h.hull_vert = vert; h.hpair_param = hpair;
  if (e == cudaSuccess) e = cudaMemcpy(m->dev, &h, sizeof(DevModel), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) { cudaFree(vert); cudaFree(hpair); return fail("mcb_model_set_hulls: upload", e); }
  cudaFree(m->d_hull_vert); cudaFree(m->d_hpair);
  m->d_hull_vert = vert; m->d_hpair = hpair; m->host = h;
  return 0;
}

int32_t mcb_model_destroy(mcb_model* m) {
  if (!m) return 0;
  cudaFree(m->dev); cudaFree(m->d_hull_vert); cudaFree(m->d_hpair);
  delete m;
  return 0;
}


int32_t mcb_batch_create(mcb_model* m, int32_t n_envs, const mcb_task_cfg* cfg, uint64_t seed, mcb_batch** out) {
  if (!m || !cfg || !out || n_envs <= 0) return fail("mcb_batch_create: bad argument");
  { const int lw = cfg->lockstep_warps; if (lw != 0 && lw != 1 && lw != 2 && lw != 4 && lw != 8 && lw != 16) return fail("mcb_batch_create: lockstep_warps must be 0 (auto), 1, 2, 4, 8 or 16"); }
  if (cfg->controller_type < 0 || cfg->controller_type > 2) return fail("mcb_batch_create: controller_type must be 0 (joint), 1 (IK) or 2 (mocap)");
  if ((cfg->controller_type == 2) != (m->host.d.has_weld != 0)) return fail("mcb_batch_create: the mocap controller needs the mocap model variant, the other controllers the joint variant");
  if (cfg->fetch_env && cfg->controller_type == 0) return fail("mcb_batch_create: joint controller is not supported for fetch envs (mycobot.py:96)");
  if (cfg->mesh_collision && m->host.nhull == 0) return fail("mcb_batch_create: mesh_collision needs mcb_model_set_hulls first");
  if (cfg->controller_type == 1 && (cfg->control_steps < 1 || cfg->control_steps > 50)) return fail("mcb_batch_create: control_steps out of range");
  if (cfg->reward_type < 0 || cfg->reward_type > 2) return fail("mcb_batch_create: reward_type must be 0 (sparse), 1 (dense) or 2 (reward_shaping)");
  DevGuard guard(m->device);
  if (!guard.ok) return fail("mcb_batch_create: cannot select the model's device", cudaGetLastError());
  mcb_batch* b = new mcb_batch();
  memset(b, 0, sizeof *b);
  b->model = m; b->n_envs = n_envs; b->cfg = *cfg; b->seed = seed;
  b->obs_dim = cfg->has_object ? MCB_OBS_OBJECT : MCB_OBS_REACH;
  if (cfg->nefc_max != 0 && cfg->nefc_max != 48 && cfg->nefc_max != 88 && cfg->nefc_max != 128) { delete b; return fail("mcb_batch_create: nefc_max must be 0 (tiered), 48, 88 (start in the middle tier) or 128 (last tier only)"); }
  b->big_only = cfg->nefc_max == 128;
  b->mid_only = cfg->nefc_max == 88;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, m->device) != cudaSuccess) { delete b; return fail("mcb_batch_create: cudaGetDeviceProperties", cudaGetLastError()); }
  b->sm_count = prop.multiProcessorCount;
  cudaError_t e = set_tier_smem<0>();
  if (e == cudaSuccess) e = set_tier_smem<1>();
  if (e == cudaSuccess) e = set_tier_smem<2>();
  if (e != cudaSuccess) { delete b; return fail("cudaFuncSetAttribute(shared memory)", e); }
  if ((e = alloc_group(b, G_CORE)) != cudaSuccess) { delete b; return fail("mcb_batch_create: allocating the batch", e); }
  init_state_kernel<<<(n_envs + 127) / 128, 128>>>(b->state, b->elapsed, b->ep_return, b->rng_ctr, b->env_seed, (unsigned long long)seed, m->dev, n_envs, cfg->fetch_env);
  if ((e = cudaGetLastError()) == cudaSuccess) e = cudaDeviceSynchronize();
  if (e != cudaSuccess) { mcb_batch_destroy(b); return fail("mcb_batch_create: init_state_kernel", e); }
  b->launches_total = 1;
  b->lockstep_warps = cfg->lockstep_warps ? cfg->lockstep_warps : 1;   // 0: free-running until mcb_autotune() is called (explicitly: mcb_step never tunes)
  b->tuned = cfg->lockstep_warps != 0;
  *out = b;
  return 0;
}

int32_t mcb_batch_destroy(mcb_batch* b) {
  if (!b) return 0;
  for (const BatchArray& d : kBatchArrays) if (d.group != G_CONTACT) cudaFree(array_of(b, d));
  free_staging(b);
  delete b;
  return 0;
}
int32_t mcb_batch_num_envs(const mcb_batch* b) { return b ? b->n_envs : -1; }
int32_t mcb_batch_obs_dim(const mcb_batch* b) { return b ? b->obs_dim : -1; }
int32_t mcb_batch_action_dim(const mcb_batch* b) { return b ? (b->cfg.fetch_env ? 4 : (b->cfg.controller_type == 2 ? 8 : NU)) : -1; }

int32_t mcb_reset(mcb_batch* b, const uint8_t* mask, const double* obj_xy, const double* goals, double* obs, double* ag, double* dg, void* stream) {
  if (!b) return fail("mcb_reset: null batch");
  StepArgs a; memset(&a, 0, sizeof a);
  a.mode = MODE_RESET; a.mask = mask; a.inj_xy = obj_xy; a.inj_goal = goals; a.obs = obs; a.ag = ag; a.dg = dg;
  return launch(b, a, (cudaStream_t)stream);
}

int32_t mcb_step(mcb_batch* b, const float* actions, double* obs, double* ag, double* dg, void* reward, uint8_t* terminated,
                 uint8_t* truncated, uint8_t* success, double* final_obs, void* stream) {
  if (!b || !actions || !reward || !terminated || !truncated || !success) return fail("mcb_step: null argument");
  StepArgs a; memset(&a, 0, sizeof a);
  a.mode = MODE_STEP; a.actions = actions; a.obs = obs; a.ag = ag; a.dg = dg; a.reward = reward;
  a.terminated = terminated; a.truncated = truncated; a.success = success; a.final_obs = final_obs;
  const long long before = b->launches_total;
  const int rc = launch(b, a, (cudaStream_t)stream);      // nothing but kernel launches on the caller's stream: graph-capturable, no hidden sync
  b->last_launches = (int)(b->launches_total - before);   // one kernel per layout tier (the second and third usually find an empty list)
  return rc;
}

int32_t mcb_batch_lockstep_warps(const mcb_batch* b) { return b ? b->lockstep_warps : -1; }

int32_t mcb_last_fallback_envs(mcb_batch* b, int32_t* last_tier_envs, void* stream) {
  if (!b) return fail("mcb_last_fallback_envs: null batch");
  int n[2] = {0, 0};
  CK(cudaMemcpyAsync(n, b->redo_count, 2 * sizeof(int), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  CK(cudaStreamSynchronize((cudaStream_t)stream));
  if (last_tier_envs) *last_tier_envs = n[1];
  return n[0];
}

int32_t mcb_autotune(mcb_batch* b, const float* actions, int32_t steps_per_candidate, void* stream) {
  if (!b) return fail("mcb_autotune: null batch");
  cudaStream_t st = (cudaStream_t)stream;
  b->tuned = 1;
  if (b->cfg.lockstep_warps != 0 || b->big_only || b->mid_only) return b->lockstep_warps;
  const int K = steps_per_candidate > 0 ? steps_per_candidate : 4;
  const size_t N = (size_t)b->n_envs;
  const size_t adim = (size_t)mcb_batch_action_dim(b);
  // every candidate replays the same K steps from the tuning state; the caller's state is restored at the end
  Snapshot caller(b), tuning(b);
  void* t_reward = nullptr; uint8_t* t_flags = nullptr; float* t_act = nullptr;
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  int best = b->lockstep_warps;
  float best_ms = 1e30f;
  bool okay = true;
#define TCK(call) do { if (okay && (call) != cudaSuccess) okay = false; } while (0)
  TCK(cudaMalloc(&t_reward, N * sizeof(double))); TCK(cudaMalloc(&t_flags, 3 * N));
  if (!actions) TCK(cudaMalloc(&t_act, N * adim * sizeof(float)));
  TCK(cudaEventCreate(&e0)); TCK(cudaEventCreate(&e1));
  TCK(caller.save(st));
  auto one_step = [&](int k) {
    if (!actions) { random_actions_kernel<<<(unsigned)((N * adim + 255) / 256), 256, 0, st>>>(t_act, (int)(N * adim), b->seed ^ 0x74756e65ull, (unsigned)k); b->launches_total++; }
    StepArgs a; memset(&a, 0, sizeof a);
    a.mode = MODE_STEP; a.actions = actions ? actions : t_act; a.reward = t_reward;
    a.terminated = t_flags; a.truncated = t_flags + N; a.success = t_flags + 2 * N;
    if (launch(b, a, st)) okay = false;
  };
  // roll ahead (state right after a reset is not representative: nothing moves yet), then snapshot the tuning state
  for (int k = 0; k < 32 && okay; k++) one_step(k);
  TCK(tuning.save(st));
  const int cand[3] = {LOCKSTEP_CTA, 4, 1};
  for (int c = 0; c < 3 && okay; c++) {
    b->lockstep_warps = cand[c];
    TCK(tuning.restore(st));
    for (int k = 0; k <= K && okay; k++) {          // step 0 is the untimed warm-up of this candidate
      if (k == 1) TCK(cudaEventRecord(e0, st));
      one_step(100 + k);
    }
    TCK(cudaEventRecord(e1, st));
    TCK(cudaEventSynchronize(e1));
    float ms = 0;
    TCK(cudaEventElapsedTime(&ms, e0, e1));
    if (okay && ms < best_ms) { best_ms = ms; best = cand[c]; }
  }
  TCK(caller.restore(st));
  TCK(cudaStreamSynchronize(st));
#undef TCK
  cudaFree(t_reward); cudaFree(t_flags); cudaFree(t_act);
  if (e0) cudaEventDestroy(e0);
  if (e1) cudaEventDestroy(e1);
  b->lockstep_warps = best;
  if (!okay) return fail("mcb_autotune: CUDA error while timing the candidates", cudaGetLastError());
  return best;
}

int32_t mcb_forward(mcb_batch* b, double* obs, double* ag, double* dg, void* stream) {
  if (!b) return fail("mcb_forward: null batch");
  StepArgs a; memset(&a, 0, sizeof a);
  a.mode = MODE_FORWARD; a.obs = obs; a.ag = ag; a.dg = dg;
  return launch(b, a, (cudaStream_t)stream);
}

int32_t mcb_debug_forward(mcb_batch* b, int32_t env, int32_t what, double* h_out, int32_t cap, void* stream) {
  if (!b || env < 0 || env >= b->n_envs) return fail("mcb_debug_forward: bad argument");
  (void)what;
  if (cap < DEBUG_DOUBLES) return fail("mcb_debug_forward: buffer too small");
  StepArgs a; memset(&a, 0, sizeof a);
  a.mode = MODE_FORWARD; a.debug = b->debug; a.debug_env = env;
  if (launch(b, a, (cudaStream_t)stream)) return -1;
  CK(cudaStreamSynchronize((cudaStream_t)stream));
  CK(cudaMemcpy(h_out, b->debug, DEBUG_DOUBLES * sizeof(double), cudaMemcpyDeviceToHost));
  return DEBUG_DOUBLES;
}

// the columns of the state record and the elapsed steps: mcb_get_state / mcb_set_state
static IoList state_cols(mcb_batch* b, int dir, const double* qpos, const double* qvel, const double* ctrl, const double* warm, const double* goal,
                         const int32_t* elapsed, const double* qprev, const double* mocap) {
  const int S = MCB_STATE_STRIDE;
  return IoList{dir}.add(b->state, S, ST_QPOS, NQ, qpos).add(b->state, S, ST_QVEL, NV, qvel).add(b->state, S, ST_CTRL, NU, ctrl).add(b->state, S, ST_WARM, NV, warm)
      .add(b->state, S, ST_GOAL, 3, goal).add(b->elapsed, 1, 0, 1, elapsed).add(b->state, S, ST_QPREV, 6, qprev).add(b->state, S, ST_MOCAP, 7, mocap);
}
int32_t mcb_get_state(mcb_batch* b, double* qpos, double* qvel, double* ctrl, double* warm, double* goal, int32_t* elapsed, double* qprev, double* mocap, void* stream) {
  if (!b) return fail("mcb_get_state: null batch");
  CK(copy_rows(b, state_cols(b, IO_GET, qpos, qvel, ctrl, warm, goal, elapsed, qprev, mocap), (cudaStream_t)stream));
  return 0;
}
int32_t mcb_set_state(mcb_batch* b, const double* qpos, const double* qvel, const double* ctrl, const double* warm, const double* goal,
                      const int32_t* elapsed, const double* qprev, const double* mocap, void* stream) {
  if (!b) return fail("mcb_set_state: null batch");
  IoList l = state_cols(b, IO_SET, qpos, qvel, ctrl, warm, goal, elapsed, qprev, mocap);
  if (qpos && !qprev) l.add(b->state, MCB_STATE_STRIDE, ST_QPREV, 6, qpos, 0.0, NQ);     // qprev := qpos[0:6]
  CK(copy_rows(b, l, (cudaStream_t)stream));
  return 0;
}

int32_t mcb_compute_reward(const double* ag, const double* g, int64_t n, double thr, int32_t type, void* out, void* stream) {
  if (n == 0) return 0;
  if (!ag || !g || !out || n < 0) return fail("mcb_compute_reward: bad argument");
  if (type != 0 && type != 1) return fail("mcb_compute_reward: reward_shaping depends on the simulation state, not on (achieved_goal, goal)");
  reward_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(ag, g, n, thr, type, out);
  CK(cudaGetLastError());
  return 0;
}

int32_t mcb_stats(mcb_batch* b, double* out, int32_t reset_after, void* stream) {
  if (!b || !out) return fail("mcb_stats: null argument");
  CK(cudaMemcpyAsync(out, b->stats, 8 * sizeof(double), cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  if (reset_after) CK(cudaMemsetAsync(b->stats, 0, 8 * sizeof(double), (cudaStream_t)stream));
  return 0;
}

int32_t mcb_step_host(mcb_batch* b, const float* h_actions, double* h_obs, double* h_ag, double* h_dg, void* h_reward, uint8_t* h_term,
                      uint8_t* h_trunc, uint8_t* h_succ, double* h_final_obs, void* stream) {
  if (!b || !h_actions) return fail("mcb_step_host: null argument");
  cudaStream_t st = (cudaStream_t)stream;
  size_t N = (size_t)b->n_envs, od = (size_t)b->obs_dim;
  const size_t ad = (size_t)mcb_batch_action_dim(b);
  size_t rbytes = b->cfg.reward_type == 0 ? sizeof(float) : sizeof(double);
  if (!b->d_actions) CK(alloc_staging(b));
  // Caller buffers that are already page-locked (cudaHostAlloc / cudaHostRegister / torch pin_memory) are used directly;
  // pageable ones go through the batch's pinned staging buffers and cost one extra host memcpy each way.
  auto pinned = [](const void* p) {
    if (!p) return false;
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return at.type == cudaMemoryTypeHost;
  };
  const float* src_actions = h_actions;
  if (!pinned(h_actions)) { memcpy(b->h_actions, h_actions, N * ad * sizeof(float)); src_actions = b->h_actions; }
  CK(cudaMemcpyAsync(b->d_actions, src_actions, N * ad * sizeof(float), cudaMemcpyHostToDevice, st));
  if (mcb_step(b, b->d_actions, b->d_obs, b->d_ag, b->d_dg, b->d_reward, b->d_flags, b->d_flags + N, b->d_flags + 2 * N,
               h_final_obs ? b->d_fobs : nullptr, stream)) return -1;
  struct Out { void* user; void* stage; const void* dev; size_t bytes; bool direct; };
  Out outs[8] = {
      {h_final_obs, b->h_fobs, b->d_fobs, N * od * sizeof(double), false}, {h_obs, b->h_obs, b->d_obs, N * od * sizeof(double), false},
      {h_ag, b->h_ag, b->d_ag, N * 3 * sizeof(double), false},            {h_dg, b->h_dg, b->d_dg, N * 3 * sizeof(double), false},
      {h_reward, b->h_reward, b->d_reward, N * rbytes, false},             {h_term, b->h_flags, b->d_flags, N, false},
      {h_trunc, b->h_flags + N, b->d_flags + N, N, false},                 {h_succ, b->h_flags + 2 * N, b->d_flags + 2 * N, N, false}};
  for (Out& o : outs) {
    if (!o.user) continue;
    o.direct = pinned(o.user);
    CK(cudaMemcpyAsync(o.direct ? o.user : o.stage, o.dev, o.bytes, cudaMemcpyDeviceToHost, st));
  }
  CK(cudaStreamSynchronize(st));
  for (Out& o : outs) if (o.user && !o.direct) memcpy(o.user, o.stage, o.bytes);
  return 0;
}

int32_t mcb_reset_host(mcb_batch* b, const uint8_t* h_mask, const double* h_obj_xy, const double* h_goals, double* h_obs, double* h_ag, double* h_dg, void* stream) {
  if (!b) return fail("mcb_reset_host: null batch");
  cudaStream_t st = (cudaStream_t)stream;
  const size_t N = (size_t)b->n_envs, od = (size_t)b->obs_dim;
  // small per-call device staging (a reset is not the hot path); freed before returning
  uint8_t* d_mask = nullptr; double *d_xy = nullptr, *d_g = nullptr, *d_o = nullptr, *d_a = nullptr, *d_d = nullptr;
  cudaError_t e = cudaSuccess;
  auto up = [&](void** dst, const void* src, size_t bytes) {
    if (!src || e != cudaSuccess) return;
    e = cudaMalloc(dst, bytes);
    if (e == cudaSuccess) e = cudaMemcpyAsync(*dst, src, bytes, cudaMemcpyHostToDevice, st);
  };
  up((void**)&d_mask, h_mask, N); up((void**)&d_xy, h_obj_xy, N * 2 * sizeof(double)); up((void**)&d_g, h_goals, N * 3 * sizeof(double));
  if (e == cudaSuccess && h_obs) e = cudaMalloc(&d_o, N * od * sizeof(double));
  if (e == cudaSuccess && h_ag) e = cudaMalloc(&d_a, N * 3 * sizeof(double));
  if (e == cudaSuccess && h_dg) e = cudaMalloc(&d_d, N * 3 * sizeof(double));
  int rc = 0;
  if (e == cudaSuccess) rc = mcb_reset(b, d_mask, d_xy, d_g, d_o, d_a, d_d, stream);
  if (e == cudaSuccess && rc == 0 && h_obs) e = cudaMemcpyAsync(h_obs, d_o, N * od * sizeof(double), cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess && rc == 0 && h_ag) e = cudaMemcpyAsync(h_ag, d_a, N * 3 * sizeof(double), cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess && rc == 0 && h_dg) e = cudaMemcpyAsync(h_dg, d_d, N * 3 * sizeof(double), cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  cudaFree(d_mask); cudaFree(d_xy); cudaFree(d_g); cudaFree(d_o); cudaFree(d_a); cudaFree(d_d);
  if (e != cudaSuccess) return fail("mcb_reset_host", e);
  return rc;
}

int32_t mcb_seed(mcb_batch* b, uint64_t seed, const uint8_t* mask, void* stream) {
  if (!b) return fail("mcb_seed: null batch");
  seed_kernel<<<(b->n_envs + 255) / 256, 256, 0, (cudaStream_t)stream>>>(b->env_seed, b->rng_ctr, b->x.param_ctr, b->x.lat_ctr, mask, (unsigned long long)seed, b->n_envs);
  CK(cudaGetLastError());
  b->launches_total++;
  if (!mask) b->seed = seed;
  return 0;
}

int32_t mcb_get_rng_state(mcb_batch* b, uint64_t* env_seed, uint64_t* draw_counter, double* ep_return, void* stream) {
  if (!b) return fail("mcb_get_rng_state: null batch");
  CK(copy_rows(b, IoList{IO_GET}.add(b->env_seed, 1, 0, 1, env_seed).add(b->rng_ctr, 1, 0, 1, draw_counter).add(b->ep_return, 1, 0, 1, ep_return),
                (cudaStream_t)stream));
  return 0;
}
int32_t mcb_set_rng_state(mcb_batch* b, const uint64_t* env_seed, const uint64_t* draw_counter, const double* ep_return, void* stream) {
  if (!b) return fail("mcb_set_rng_state: null batch");
  CK(copy_rows(b, IoList{IO_SET}.add(b->env_seed, 1, 0, 1, env_seed).add(b->rng_ctr, 1, 0, 1, draw_counter).add(b->ep_return, 1, 0, 1, ep_return),
                (cudaStream_t)stream));
  return 0;
}

int32_t mcb_batch_set_param_ranges(mcb_batch* b, const double* h_lo, const double* h_hi) {
  if (!b) return fail("mcb_batch_set_param_ranges: null batch");
  if (!h_lo != !h_hi) return fail("mcb_batch_set_param_ranges: pass both bounds, or neither to stop drawing");
  if (!h_lo) { b->x.draw_params = 0; return 0; }
  for (int k = 0; k < MCB_NPARAM; k++)
    if (!(std::isfinite(h_lo[k]) && std::isfinite(h_hi[k]) && h_lo[k] > 0 && h_lo[k] <= h_hi[k]))
      return fail("mcb_batch_set_param_ranges: every range must be finite with 0 < lo <= hi");
  if (enable_params(b, "mcb_batch_set_param_ranges")) return -1;
  memcpy(b->x.param_lo, h_lo, sizeof b->x.param_lo); memcpy(b->x.param_hi, h_hi, sizeof b->x.param_hi);
  b->x.draw_params = 1;
  return 0;
}

// a batch without per-env parameters reads as the nominal 1.0 and draw counter 0
static IoList param_cols(mcb_batch* b, int dir, const double* params, const uint64_t* draw_counter) {
  return IoList{dir}.add(b->x.params, MCB_NPARAM, 0, MCB_NPARAM, params, 1.0).add(b->x.param_ctr, 1, 0, 1, draw_counter);
}
int32_t mcb_get_env_params(mcb_batch* b, double* params, uint64_t* draw_counter, void* stream) {
  if (!b) return fail("mcb_get_env_params: null batch");
  CK(copy_rows(b, param_cols(b, IO_GET, params, draw_counter), (cudaStream_t)stream));
  return 0;
}

int32_t mcb_set_env_params(mcb_batch* b, const double* params, const uint64_t* draw_counter, void* stream) {
  if (!b) return fail("mcb_set_env_params: null batch");
  if (enable_params(b, "mcb_set_env_params")) return -1;
  CK(copy_rows(b, param_cols(b, IO_SET, params, draw_counter), (cudaStream_t)stream));
  return 0;
}

int32_t mcb_batch_set_latency_range(mcb_batch* b, int32_t lo, int32_t hi) {
  if (!b) return fail("mcb_batch_set_latency_range: null batch");
  if (lo == -1 && hi == -1) { b->x.draw_latency = 0; return 0; }
  if (!(0 <= lo && lo <= hi && hi <= b->cfg.frame_skip)) return fail("mcb_batch_set_latency_range: the range must satisfy 0 <= lo <= hi <= frame_skip");
  if (enable_params(b, "mcb_batch_set_latency_range")) return -1;
  b->x.lat_lo = lo; b->x.lat_hi = hi;
  b->x.draw_latency = 1;
  return 0;
}

int32_t mcb_get_env_latency(mcb_batch* b, int32_t* latency, uint64_t* draw_counter, void* stream) {
  if (!b) return fail("mcb_get_env_latency: null batch");
  CK(copy_rows(b, IoList{IO_GET}.add(b->x.latency, 1, 0, 1, latency).add(b->x.lat_ctr, 1, 0, 1, draw_counter), (cudaStream_t)stream));
  return 0;
}

int32_t mcb_set_env_latency(mcb_batch* b, const int32_t* latency, const uint64_t* draw_counter, void* stream) {
  if (!b) return fail("mcb_set_env_latency: null batch");
  if (enable_params(b, "mcb_set_env_latency")) return -1;
  CK(copy_rows(b, IoList{IO_SET}.add(b->x.latency, 1, 0, 1, latency).add(b->x.lat_ctr, 1, 0, 1, draw_counter), (cudaStream_t)stream));
  return 0;
}

// applied forces [N, NFRC] as qfrc [N, NV] and xfrc [N, NB, 6]; a batch without forces reads as zeros
static IoList applied_cols(mcb_batch* b, int dir, const double* qfrc, const double* xfrc) {
  return IoList{dir}.add(b->x.frc, NFRC, 0, NV, qfrc).add(b->x.frc, NFRC, NV, NB * 6, xfrc);
}
int32_t mcb_set_env_applied(mcb_batch* b, const double* qfrc, const double* xfrc, void* stream) {
  if (!b) return fail("mcb_set_env_applied: null batch");
  if (b->cfg.mesh_collision) return fail("mcb_set_env_applied: applied forces are not supported with mesh_collision");
  if (!b->x.frc) {
    // first call: zeroed forces for every env, and the PRM kernels that read them; synchronises (not capturable)
    if (enable_params(b, "mcb_set_env_applied")) return -1;
    DevGuard guard(b->model->device);
    if (!guard.ok) return fail("mcb_set_env_applied: cannot select the batch's device", cudaGetLastError());
    if (const cudaError_t e = alloc_group(b, G_FORCES)) return fail("mcb_set_env_applied: allocating the forces", e);
  }
  if (!qfrc && !xfrc) return 0;
  CK(copy_rows(b, applied_cols(b, IO_SET, qfrc, xfrc), (cudaStream_t)stream));
  return 0;
}

int32_t mcb_get_env_applied(mcb_batch* b, double* qfrc, double* xfrc, void* stream) {
  if (!b) return fail("mcb_get_env_applied: null batch");
  if (!qfrc && !xfrc) return 0;
  CK(copy_rows(b, applied_cols(b, IO_GET, qfrc, xfrc), (cudaStream_t)stream));
  return 0;
}

int32_t mcb_set_contact_output(mcb_batch* b, int32_t* ncon, int32_t* geom, double* con, int32_t* final_ncon, int32_t* final_geom, double* final_con) {
  if (!b) return fail("mcb_set_contact_output: null batch");
  const bool on = ncon || geom || con, fin = final_ncon || final_geom || final_con;
  if (on && !(ncon && geom && con)) return fail("mcb_set_contact_output: ncon, geom and con are given together");
  if (fin && !(final_ncon && final_geom && final_con)) return fail("mcb_set_contact_output: final_ncon, final_geom and final_con are given together");
  if (fin && !on) return fail("mcb_set_contact_output: the final contacts need ncon, geom and con too");
  if (on) {
    if (b->cfg.mesh_collision) return fail("mcb_set_contact_output: contact output is not supported with mesh_collision");
    if (enable_params(b, "mcb_set_contact_output")) return -1;
  }
  // launches already enqueued write to the arrays registered before
  DevGuard guard(b->model->device);
  if (!guard.ok) return fail("mcb_set_contact_output: cannot select the batch's device", cudaGetLastError());
  CK(cudaDeviceSynchronize());
  b->x.con_n = ncon; b->x.con_geom = geom; b->x.con = con;
  b->x.con_fn = final_ncon; b->x.con_fgeom = final_geom; b->x.con_f = final_con;
  return 0;
}

int32_t mcb_last_fallback_list(mcb_batch* b, int32_t* h_envs, int32_t cap, void* stream) {
  if (!b || (cap > 0 && !h_envs) || cap < 0) return fail("mcb_last_fallback_list: bad argument");
  int n = 0;
  CK(cudaMemcpyAsync(&n, b->redo_count, sizeof(int), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  CK(cudaStreamSynchronize((cudaStream_t)stream));
  const int m = n < cap ? n : cap;
  if (m > 0) CK(cudaMemcpy(h_envs, b->redo_list, (size_t)m * sizeof(int), cudaMemcpyDeviceToHost));
  return n;
}

int64_t mcb_total_launches(const mcb_batch* b) { return b ? (int64_t)b->launches_total : -1; }
int32_t mcb_last_step_launches(const mcb_batch* b) { return b ? b->last_launches : -1; }

int32_t mcb_fp64_peak_probe(int32_t device, int32_t iters, double* tflops_out) {
  if (!tflops_out || iters <= 0) return fail("mcb_fp64_peak_probe: bad argument");
  DevGuard guard(device);
  if (!guard.ok) return fail("mcb_fp64_peak_probe: cannot select the device", cudaGetLastError());
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, device));
  double* out;
  CK(cudaMalloc(&out, sizeof(double)));
  int blocks = prop.multiProcessorCount * 8, threads = 256;
  cudaEvent_t e0, e1;
  CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
  dfma_probe_kernel<<<blocks, threads>>>(out, iters);
  CK(cudaDeviceSynchronize());
  float best = 1e30f;
  for (int r = 0; r < 5; r++) {
    CK(cudaEventRecord(e0));
    dfma_probe_kernel<<<blocks, threads>>>(out, iters);
    CK(cudaEventRecord(e1));
    CK(cudaEventSynchronize(e1));
    float ms; CK(cudaEventElapsedTime(&ms, e0, e1));
    if (ms < best) best = ms;
  }
  double flops = 2.0 * 8.0 * (double)iters * (double)blocks * (double)threads;
  *tflops_out = flops / (best * 1e-3) / 1e12;
  cudaFree(out); cudaEventDestroy(e0); cudaEventDestroy(e1);
  return 0;
}


}  // extern "C"

#include "mcb_her.cuh"
#endif  // MCB_PRM_UNIT
