/* mrs_b200.h -- C ABI of the B200-native mrs-gym step path (libmrs_b200.so).
 *
 * The reference (Acciorocketships/mrs-gym) has no FFI: its hot path sits behind the Python
 * class MRS (mrsgym/MRS.py:12) and crosses into C only through ~22+N pybullet calls per
 * agent per step.  This header is the seam a maintainer would bind instead (ctypes stub in
 * INTEGRATION.md); each entry point names the reference interface it replaces.
 *
 * Conventions
 *   - plain pointers and sizes only; every device buffer is CALLER-OWNED (the library never
 *     allocates or frees device memory), all work is ordered on the passed CUDA stream
 *     (a cudaStream_t passed as void*), no hidden synchronisation (except mrs_step_host);
 *   - int return: 0 = OK, <0 = MrsError (mrs_strerror); no C++ exceptions cross the ABI;
 *   - thread-safe for distinct buffer sets; one host thread per GPU: the calls that use the library's internal
 *     side streams (mrs_step_many / mrs_rollout with N > 32, mrs_rollout_host) share one set of streams and events
 *     per device and must not run concurrently on one device.
 *   - there is NO CPU fallback: without a CUDA device every compute call returns
 *     MRS_ERR_CUDA.
 *
 * Layout in HBM (S = E*N agent slots, s = e*N + a):
 *   state  float[13][S]   SoA planes: pos xyz | quat xyzw | vel xyz | angvel xyz (world)
 *   ctrl   float[18][S]   PID planes: int_ori 0-2 | int_pos 3-5 | int_vel 6-8 |
 *                         last_vel_e 9-11 | d_vel_e 12-14 | last_target_vel 15-17.
 *                         last_vel_e.x = NaN marks "controller never called"
 *                         (QuadControl's hasattr laziness, mrsgym/QuadControl.py:55-61).
 *   rpm    float[4][S]    last rotor speeds (Quadcopter.speeds), optional (may be NULL)
 *   X_tape float[L][E][N][D], A_tape float[L][E][N][N]   observation history tapes: the
 *                         host writes slot p-1 at each step (descending) so that slots
 *                         [p, p+K] are the reference's newest-first K_HOPS+1 window
 *                         (mrsgym/MRS.py:87-114) with no per-step copy.
 *   scratch float[P][S]   only for N > 32 (unconstrained velocities, pre-step positions,
 *                         contact-proximity flag between the wide-path kernels; for N > 128
 *                         also the per-slice partial sums of the pair pass).  P =
 *                         mrs_scratch_planes(E, N): 7, or 7 + 2 * slices (<= 32 slices; 1 when
 *                         E is large) for N > 128.  No initial contents required.
 *   wrench float[6][S]    optional (may be NULL) external wrench per agent, SoA planes like state: force fx fy fz
 *                         [N] at the centre of mass (planes 0-2), torque tx ty tz [N m] (planes 3-5), both in the
 *                         WORLD frame.  It enters the Bullet step where the rotor / aero wrench does, in the
 *                         unconstrained velocities before the contact solve:
 *                           v* = clamp(v + dt ((R Fb + F_ext) / m - g z - damping), +-max_coord_vel)
 *                           w*: the body-frame right-hand side gains R^T tau_ext before I^-1
 *                         so it takes part in the contact solve like any other applied force (a grounded agent
 *                         pressed down stays put, a sideways push meets friction).  The buffer persists: every step
 *                         of every stepping call (mrs_step, each of the T steps of mrs_step_many / mrs_rollout /
 *                         mrs_rollout_host, mrs_step_host) reads it until the caller changes it -- unlike
 *                         p.applyExternalForce, which Bullet clears after each stepSimulation.  mrs_set_state,
 *                         mrs_spawn and mrs_autoreset leave it alone.  An agent with a NaN action loses its rotor
 *                         wrench and the downwash it receives but keeps the external wrench.  A NaN / inf component
 *                         is not special-cased: like any non-finite acceleration it meets the +-max_coord_vel clamp
 *                         (fminf / fmaxf return the bound for NaN), so that agent moves at the clamp velocity and
 *                         stays finite (no MRS_STATUS_NONFINITE); no other agent is affected.  NULL: no
 *                         external wrench, the step runs exactly the kernels it runs without this member.  With a
 *                         wrench, N <= 32 runs the run-time-width kernel on small CTAs (no baked constants, no
 *                         chained hand-over in mrs_rollout).
 */
#ifndef MRS_B200_H
#define MRS_B200_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MRS_ABI_VERSION 6
#define MRS_STATE_PLANES 13
#define MRS_CTRL_PLANES 18
#define MRS_STATS_SLOTS 8
#define MRS_SCRATCH_PLANES 7          /* N <= 128 */
#define MRS_SCRATCH_PAIR_SPLITS 32    /* N > 128: + 2 planes (partial pair sum, flag) per partner slice, <= 32 slices */
#define MRS_SYNC_WORDS 8208           /* u64 words of MrsBuffers.sync (launch-to-launch range hand-over of mrs_rollout) */
#define MRS_COMM_MAX_WORLD 16         /* GPUs of one node a peer communicator spans */
#define MRS_COMM_HANDLE_BYTES 64      /* size of the opaque mailbox handle exchanged between ranks */

/* ACTION_TYPE strings of the reference are method names dispatched by getattr
 * (mrsgym/Environment.py:92 -> mrsgym/Quadcopter.py:26-65). */
typedef enum {
    MRS_SET_TARGET_VEL = 0,   /* Quadcopter.set_target_vel   Quadcopter.py:53-55  */
    MRS_SET_TARGET_POS = 1,   /* Quadcopter.set_target_pos   Quadcopter.py:58-60  */
    MRS_SET_TARGET_ACCEL = 2, /* Quadcopter.set_target_accel Quadcopter.py:48-50  */
    MRS_SET_FORCE = 3,        /* README "set_force" := set_target_accel(F/Mass)   */
    MRS_SET_TARGET_ORI = 4,   /* Quadcopter.set_target_ori   Quadcopter.py:63-65  */
    MRS_SET_CONTROL = 5,      /* Quadcopter.set_control      Quadcopter.py:26-34  */
    MRS_SET_SPEEDS = 6,       /* Quadcopter.set_speeds       Quadcopter.py:38-45  */
    MRS_NO_ACTION = 7         /* MRS.step(actions=None): no forces (MRS.py:243)   */
} MrsActionType;

/* Built-in fused state_fn layouts (user state_fn: MRS.py:16, Environment.py:84-87). */
typedef enum {
    MRS_X_NONE = 0,           /* X written by the caller (python state_fn)        */
    MRS_X_POS_VEL = 1,        /* D=6  cat(get_pos, get_vel)  README.md:28-29      */
    MRS_X_FULL = 2            /* D=13 pos, quat, vel, angvel                      */
} MrsStateLayout;

typedef enum {
    MRS_OK = 0,
    MRS_ERR_ARG = -1,
    MRS_ERR_CUDA = -2,
    MRS_ERR_UNSUPPORTED = -3
} MrsError;

/* status word bits (device, sticky; the host reads them lazily) */
#define MRS_STATUS_NAN_ACTION 1u   /* mirrors the NaN guard of mrsgym/MRS.py:247-248 */
#define MRS_STATUS_NONFINITE 2u    /* a state component left the finite range        */
#define MRS_STATUS_CONTACT_OVERFLOW 16u /* N > 32: an env had more agents / pairs in contact than the solver holds */
#define MRS_STATUS_SYNC_TIMEOUT 8u /* a chained launch of mrs_rollout waited > 2 s for its predecessor's range    */
#define MRS_STATUS_COMM_TIMEOUT 4u /* mrs_stats_allreduce / mrs_comm_barrier gave up waiting for a peer */
#define MRS_STATUS_NEIGHBOR_OVERFLOW 32u /* mrs_neighbors: an agent had more neighbours than max_nbr (list truncated) */

/* stats slots (unsigned long long, device; summed across GPUs per rollout; never reset by a step).  The unit of
 * each counter is the same on every step path unless noted; a warp-chunk holds 32 / pow2ceil(N) envs. */
#define MRS_STAT_AGENT_CONTACTS 0  /* per agent-step: sphere-sphere pair rows of the agent whose normal impulse
                                      ended > 0 (a pushing pair counts once for each of its two agents) */
#define MRS_STAT_GROUND_CONTACTS 1 /* agent-steps whose ground rows pushed (sum of the four normal impulses > 0) */
#define MRS_STAT_NONFINITE 2       /* agent-steps that end with a non-finite state component */
#define MRS_STAT_NAN_ACTIONS 3     /* agent-steps whose action has a NaN component (MRS_STATUS_NAN_ACTION) */
#define MRS_STAT_CONTACT_CHUNKS 4  /* N <= 32 (0 otherwise): warp-chunk steps on the contact path.  Single-step
                                      launches (mrs_step, mrs_rollout): one per chunk and step that has an agent
                                      below the ground-skip height, a pair within contact range or a NaN action.
                                      mrs_step_many: T - t0 per chunk whose first such step is t0 (the chunk
                                      stays on the contact path for the rest of the launch) */
#define MRS_STAT_SOLVER_SWEEPS 5   /* N <= 32 (0 otherwise): per contact-path chunk step, the largest number of
                                      Gauss-Seidel sweeps among its envs */
#define MRS_STAT_NEIGHBOR_OVERFLOW 6 /* mrs_neighbors: rows whose list was truncated at max_nbr */

/* cf2x.urdf properties (mrsgym/models/cf2x.urdf:5,11-12,42-78), the derived ones of
 * Quadcopter.calculate_parameters (Quadcopter.py:153-168) and the QuadControl gains
 * (QuadControl.py:14-32). */
typedef struct {
    float mass, ixx, iyy, izz;           /* file inertia: set_control scaling only */
    float kf, km, arm;
    float gnd_eff_coeff, prop_radius, gnd_hclip;
    float drag_xy, drag_z;
    float dw1, dw2, dw3;
    float prop_x[4], prop_y[4];
    float pos_p, pos_i, pos_d;
    float vel_p, vel_i, vel_d;
    float ori_p[3], ori_i[3], ori_d[3];
    float min_pwm, max_pwm, pwm2rpm_a, pwm2rpm_b;
    float ctrl_dt, ctrl_gravity;         /* QuadControl always uses DefaultSim: 0.01 / 9.81 */
    float mix_ainv[16];                  /* inverse of the 'x' mixer, Quadcopter.py:164-165 */
    float mix_a[16];
    float nnls_tab[16 * 16];             /* per active set: least-squares solve matrix */
} MrsQuadParams;

/* What p.stepSimulation() does to this scene (mrsgym/BulletSim.py:46-47); Bullet3 is not
 * vendored in the reference: see oracle/bullet_model.py for the restated algorithm. */
typedef struct {
    float mass;
    float inertia[3];                    /* AABB-box inertia Bullet uses without URDF_USE_INERTIA_FROM_FILE */
    float lin_damping, ang_damping;
    float max_coord_vel;
    int gyro;
    float ang_motion_threshold;
    float erp2, slop, contact_margin;
    float mu_ground, ground_z;
    float col_radius, col_halfheight, col_margin;
    int ground_contact, agent_contact;
    float agent_radius;                  /* MRS.AGENT_RADIUS, MRS.py:28: minimum start separation / 2 (mrs_spawn) */
    float contact_radius;                /* agent-agent contact sphere (north star: = AGENT_RADIUS; 0.06 = the cf2x hull) */
    float mu_agent;                      /* quad-quad friction: link default 0.5 x 0.5 */
    int solver_iters;                    /* Gauss-Seidel sweeps of the contact solver (Bullet numSolverIterations 50) */
    float solver_tol;                    /* early exit: largest change of a row's contact-point velocity in a sweep [m/s] */
} MrsPhysicsParams;

typedef struct {
    int E, N, K, L;                      /* envs (this GPU's shard), agents/env, K_HOPS, tape slots */
    int action_type;                     /* MrsActionType */
    int state_layout;                    /* MrsStateLayout */
    float dt, gravity;                   /* BulletSim.DT / GRAVITY, BulletSim.py:13-14 */
    float comm_range;                    /* MRS.COMM_RANGE (inf => ones - eye), MRS.py:117-124 */
    MrsQuadParams quad;
    MrsPhysicsParams phys;
} MrsConfig;

typedef struct {
    float* state;                        /* [13][S] */
    float* ctrl;                         /* [18][S] */
    float* rpm;                          /* [4][S] or NULL */
    float* X_tape;                       /* [L][E][N][D] or NULL */
    float* A_tape;                       /* [L][E][N][N] or NULL */
    float* scratch;                      /* [mrs_scratch_planes(E, N)][S], needed iff N > 32 */
    unsigned int* status;                /* [1] */
    unsigned long long* stats;           /* [MRS_STATS_SLOTS] */
    unsigned long long* sync;            /* [MRS_SYNC_WORDS], zero-initialised once by the caller, owned by the library
                                            afterwards; NULL = mrs_rollout falls back to grid-wide dependencies */
    float* wrench;                       /* [6][S] or NULL: external force / torque per agent, world frame (see above) */
} MrsBuffers;

int mrs_abi_version(void);
const char* mrs_strerror(int err);

/* D of a built-in layout (0 for MRS_X_NONE). */
int mrs_state_dim(int state_layout);
/* ACTION_DIM of an action type. */
int mrs_action_dim(int action_type);

/* Planes of MrsBuffers.scratch E envs of N agents need (0 for N <= 32). */
int mrs_scratch_planes(int E, int N);

/* sizeof(MrsConfig) / sizeof(MrsBuffers) as compiled: lets a foreign binding check its mirror. */
size_t mrs_sizeof_config(void);
size_t mrs_sizeof_buffers(void);

/* Fills quad/phys/dt/gravity with the reference's constants (cf2x.urdf, QuadControl gains,
 * BulletSim defaults) and the mixer tables.  E,N,K,L,action_type,... are left to the caller.
 * Replaces Quadcopter.read_attributes/calculate_parameters (Quadcopter.py:119-168). */
int mrs_default_config(MrsConfig* cfg);

/* 1 when cfg carries exactly the reference's constants (every field mrs_default_config fills:
 * cf2x.urdf, QuadControl gains, Bullet defaults, DT 0.01, GRAVITY 9.81, AGENT_RADIUS 0.3), 0
 * otherwise.  For such a configuration the N <= 32 step runs kernels that hold these constants
 * as immediates (generated csrc/mrs_baked.cuh); any other configuration runs the generic kernels
 * that read them from MrsConfig.  Same arithmetic, same results; no reference counterpart. */
int mrs_config_is_baked(const MrsConfig* cfg);

/* Debug / build tooling: copies the host-derived constants of cfg (struct Derived of
 * csrc/mrs_device.cuh, out_bytes must equal its size) to `out`.  tools/gen_baked.py reads the
 * library's own numbers through this call when it generates csrc/mrs_baked.cuh. */
int mrs_debug_derived(const MrsConfig* cfg, void* out, size_t out_bytes);

/* One env.step for all E envs: actions -> controller -> rotor wrench + aero (ground
 * effect, drag, downwash) -> Bullet step (contact) -> newest X slice into X tape slot
 * `slot_x`, newest A slice into A tape slot `slot_a` (the reference shifts its X and A deques
 * independently, MRS.py:87-114).  actions: device float[E][N][ACTION_DIM] (ignored for
 * MRS_NO_ACTION).  bufs->wrench (NULL or [6][S]) is added to every agent's wrench in this step.
 * Replaces MRS.step's set_actions + step_sim + calc_Xk + calc_Ak (MRS.py:252-257). */
int mrs_step(const MrsConfig* cfg, const MrsBuffers* bufs, const float* actions, int slot_x, int slot_a,
             void* stream);

/* T consecutive steps in one call (N <= 32: one launch, state stays in registers); step t
 * reads actions[t] (device float[T][E][N][ACTION_DIM]) and writes tape slots
 * slot_x_first - t / slot_a_first - t.  Every step reads the same bufs->wrench.  The rollout loop of
 * examples/simulating_data/helper/DataGenerator.py:8-48 with pre-computed actions. */
int mrs_step_many(const MrsConfig* cfg, const MrsBuffers* bufs, const float* actions, int T,
                  int slot_x_first, int slot_a_first, void* stream);

/* T consecutive steps as T single-step launches (every step reads and writes the whole state in HBM / L2, one
 * launch per env.step as in a closed loop) with pre-computed actions float[T][E][N][ACTION_DIM]; tape slots as in
 * mrs_step_many.  For N in {8, 16, 32} and jobs that fill the GPU the launches are CHAINED: environments are
 * independent, so the chunk range a CTA of step t has finished is handed to a CTA of step t+1 through
 * bufs->sync (a queue in completion order) instead of waiting for the whole grid of step t -- an SM never waits
 * for the slowest SM of the previous step (not with bufs->wrench set: then every step is a plain launch of the
 * wrench kernel).  Everything else behaves like T calls of mrs_step, the wrench included.  Capturable in a
 * CUDA graph.  The rollout loop of examples/simulating_data/helper/DataGenerator.py:8-48. */
int mrs_rollout(const MrsConfig* cfg, const MrsBuffers* bufs, const float* actions, int T, int slot_x_first,
                int slot_a_first, void* stream);

/* Observation only: X (state layout) and/or A (adjacency) of the CURRENT state into tape
 * slot `slot`.  Replaces MRS.calc_Xk / MRS.calc_Ak+calc_A (MRS.py:87-124) outside step. */
int mrs_observe(const MrsConfig* cfg, const MrsBuffers* bufs, int slot, int write_X, int write_A,
                void* stream);

/* Adjacency of arbitrary float32 positions: pos device float[E][N][3] -> A float[E][N][N].
 * MRS.calc_A (MRS.py:117-124): bit-exact with torch CPU on identical positions. */
int mrs_adjacency(const MrsConfig* cfg, const float* pos, float* A, void* stream);

/* Neighbour lists of the COMM_RANGE graph of the current positions (bufs->state planes 0-2).
 * For every agent i of every env:
 *   cnt[e][i]              = number of j != i with A[e][i][j] == 1 (the exact predicate of
 *                            mrs_adjacency / the step kernels, COMM_RANGE = inf included);
 *   idx[e][i][0 .. min(cnt, max_nbr))
 *                          = those j in ascending order; the remaining entries of the row are -1.
 * idx: device int32 [E][N][max_nbr] (may be NULL when max_nbr == 0: degrees only);
 * cnt: device int32 [E][N].  A degree above max_nbr keeps the first max_nbr neighbours, reports
 * the true degree in cnt, sets MRS_STATUS_NEIGHBOR_OVERFLOW and adds the truncated rows to
 * stats[MRS_STAT_NEIGHBOR_OVERFLOW] (max_nbr == 0 asks for the degrees alone and reports no
 * overflow).  Deterministic, stream-ordered, capturable.  MRS_ERR_ARG for a negative max_nbr or a
 * missing cnt, MRS_ERR_UNSUPPORTED when E * N * 32 does not fit in 32 bits.
 * A graph learner's form of MRS.calc_A (MRS.py:117-124): 4 (max_nbr + 1) bytes per agent instead of 4 N. */
int mrs_neighbors(const MrsConfig* cfg, const MrsBuffers* bufs, int max_nbr, int* idx, int* cnt, void* stream);

/* Upload start states: device float[E][N][3] each (ori = euler 'xyz' roll,pitch,yaw), NULL
 * pointer = keep that component; env_mask device uint8[E] or NULL (= all envs).  PID state
 * is NOT reset (reference quirk, SURVEY.md §3.3).
 * Replaces Environment.set_state -> Object.set_state (Environment.py:97-103, Object.py:42-65). */
int mrs_set_state(const MrsConfig* cfg, const MrsBuffers* bufs, const float* pos, const float* ori_euler,
                  const float* vel, const float* angvel, const unsigned char* env_mask, void* stream);

/* Tape maintenance.  which: 1 = X, 2 = A.  Copies slot src into `count` slots starting at
 * dst_first (src < 0: fill with zeros).  Used for the reference's ring padding after
 * reset (X: copies of X0, A: zeros; MRS.py:92-93,107-108) and for window compaction. */
int mrs_tape_fill(const MrsConfig* cfg, const MrsBuffers* bufs, int which, int src, int dst_first,
                  int count, void* stream);

/* End-to-end step over HOST buffers (pinned recommended): H2D actions, mrs_step, D2H of the
 * newest X slice ([E][N][D]) and A slice ([E][N][N], and / or its bit-packed form, see mrs_pack_adjacency); X_host /
 * A_host / Abits_host may be NULL.
 * dev_actions: caller-owned device staging float[E][N][ACTION_DIM].  bufs->wrench applies as in mrs_step (it stays
 * on the device; no copy).  Synchronises the stream before returning (the reference's step is synchronous). */
int mrs_step_host(const MrsConfig* cfg, const MrsBuffers* bufs, const float* actions_host,
                  float* dev_actions, float* X_host, float* A_host, unsigned int* Abits_host,
                  unsigned int* dev_Abits, int slot_x, int slot_a, void* stream);

/* Compact adjacency for the wire (opt-in; the float32 {0,1} matrix of MRS.calc_A stays the default): A float[E][N][N]
 * -> bits u32[E][N][ceil(N/32)], bit j of word w of row i = A[i][32 w + j] != 0.  At C5 the newest A slice shrinks from
 * 16.8 MB to 2.1 MB; the host paths are PCIe-bound, so this is what the caller with a bandwidth problem asks for:
 * mrs_step_host / mrs_rollout_host take Abits_host (pinned host u32, [T] x that shape) + dev_Abits (caller-owned
 * device staging: one such array for mrs_step_host, TWO for mrs_rollout_host) next to or instead of A_host. */
int mrs_pack_adjacency(const MrsConfig* cfg, const float* A, unsigned int* bits, void* stream);

/* On-device reset with the reference's DEFAULT start distribution for the envs selected by
 * env_mask (NULL = all; only the 13 state planes of the selected envs are written), any N.
 * Round 0: every agent draws xy ~ N(0, xy_sigma) pulled onto the disc of radius xy_radius and z ~ U[z_lo, z_hi];
 * then agent i is flagged iff some j < i of its env is closer than 2*AGENT_RADIUS (squared distance < 4 r^2,
 * this round's positions).  Every later round re-draws the flagged agents and tests again; an env stops when no
 * agent is flagged.  An env still flagged after max_rounds rounds keeps its last positions and counts once in
 * *failed_envs (device u32, added to, may be NULL).  yaw ~ U[yaw_lo, yaw_hi], roll = pitch = 0; velocities zero.
 * Counter-based RNG (splitmix64 keyed by seed, global env index env_offset + e, agent and round): the result
 * depends on (seed, env_offset + e, N, the spawn arguments, AGENT_RADIUS) only, not on E, env_mask or the launch
 * shape -- env_offset is the global index of this shard's first env, so the ranks of a sharded job draw
 * different environments from one seed.  N <= 32 and N > 32 use different key packings (a warp per env / a CTA
 * per env), so their streams differ.  E*N must fit 32-bit slot indices (MRS_ERR_UNSUPPORTED otherwise).
 * Replaces MRS.generate_start_pos / generate_start_ori / default_spawn_dist + the set_state of
 * MRS.reset (MRS.py:69-78,127-161,174-184) without the host round trip. */
int mrs_spawn(const MrsConfig* cfg, const MrsBuffers* bufs, const unsigned char* env_mask,
              unsigned long long seed, unsigned long long env_offset, float z_lo, float z_hi, float xy_radius, float xy_sigma, float yaw_lo,
              float yaw_hi, int max_rounds, unsigned int* failed_envs, void* stream);

/* Closed-loop episode bookkeeping and auto-reset, once per step after the step: the tail of the loop of
 * examples/simulating_data/helper/DataGenerator.py:8-48 (done -> masked reset -> calc_Ak) without a host decision,
 * so that a closed loop can be captured in a CUDA graph.  For every env e, with n = env_steps[e] (steps since its
 * last reset, counted BEFORE this step's increment, as MRS.done_fn sees it):
 *   done = (done_in && done_in[e]) || (max_timesteps >= 0 && n >= max_timesteps)
 *          || (episode_length > 0 && n + 1 >= episode_length);
 *   done_out[e] = done.
 * A done env starts episode episode[e] + 1: its start state is redrawn with the default distribution and the
 * 2*AGENT_RADIUS rejection rule of mrs_spawn (at most max_rounds rounds; an env still flagged keeps its last draw and
 * counts once in *failed_envs), keyed by (seed, env_offset + e, episode[e] + 1) with ONE key packing for every N --
 * the draw depends neither on E, the launch shape nor the step the reset falls on; velocities and angular
 * velocities become zero, the PID planes are left alone (reference quirk, SURVEY.md §3.3); X0 (state_layout) is
 * written into the K+1 X window slots (slot_x + k) mod L, A0 (the dense adjacency of the new positions, the
 * predicate of mrs_adjacency) into slot_a and zeros into the K older A slots (slot_a + k) mod L; episode[e] += 1,
 * env_steps[e] = 0.  Any other env only gets env_steps[e] += 1: no byte of its state, PID planes or tapes changes.
 * A warp per env for N <= 32, a CTA per env above.  Stream-ordered, no host synchronisation, capturable.
 * MRS_ERR_ARG: missing env_steps / episode / done_out, an X tape with MRS_X_NONE, a slot outside [0, L);
 * MRS_ERR_UNSUPPORTED: E*N does not fit 32-bit slot indices. */
typedef struct {
    unsigned long long seed, env_offset;     /* as mrs_spawn */
    float z_lo, z_hi, xy_radius, xy_sigma, yaw_lo, yaw_hi;
    int max_rounds;
    int episode_length;                      /* 0 = no limit */
    int max_timesteps;                       /* MRS.MAX_TIMESTEPS as the default done_fn sees it; <0 = inf */
} MrsAutoResetArgs;

int mrs_autoreset(const MrsConfig* cfg, const MrsBuffers* bufs, const MrsAutoResetArgs* a,
                  const unsigned char* done_in,   /* device [E] or NULL: the user's done_fn result */
                  int* env_steps,                 /* device [E], steps since the env's last reset, in/out */
                  unsigned* episode,              /* device [E], episodes started per env, in/out */
                  unsigned char* done_out,        /* device [E]: the dataset's done[t] */
                  int slot_x, int slot_a,         /* newest X / A slots; window slots are (slot + k) mod L */
                  unsigned* failed_envs, void* stream);

/* Analytic sensors on the primitives of the 'simple' world (ground box top at ground_z, agents as
 * phys.contact_radius spheres: the contact geometry of the step's pair rows; phys.agent_radius is only
 * the spawn separation), for all agents of all envs at once.
 * mrs_proximity: per agent the gap to the nearest other agent (centre distance - 2*contact_radius) and
 * its index (the lowest index among equal distances; -1 and an infinite gap when N == 1), the gap of the
 * collision cylinder to the ground, and collision = any gap < threshold (strict; the reference uses 0.04).  The
 * ground gap is that of the lowest of the four rim points (+-col_radius, 0, cz), (0, +-col_radius, cz) that the
 * step's ground rows use: z - col_radius*max(|R20|,|R21|) - col_halfheight*|R22| - col_margin - ground_z.
 * Any output pointer may be NULL.  Device arrays of E*N elements.
 * Replaces Object.collision / get_dist / get_contact_points distances (Object.py:98-140).
 * mrs_raycast: n_rays rays per agent, directions device float[n_rays][3] in the body frame
 * (body_frame != 0) or the world frame, start = position + R * offset3 (HOST float[3], may be NULL);
 * hit_dist float[E*N][n_rays] (inf = nothing within range), hit_id int[E*N][n_rays]: -1 none,
 * N = ground, j = agent j of the same env; the first hit at t < range wins, ties go to the ground, then the
 * lowest index.  A direction counts by its orientation only: any finite nonzero magnitude (denormal to FLT_MAX)
 * gives the result of its unit vector; a zero direction or one with a NaN or infinite component hits nothing
 * (-1 / inf, never NaN).  MRS_ERR_UNSUPPORTED (outputs untouched) when E*N*n_rays >= 2^32 - 1.
 * Replaces Object.raycast (Object.py:143-174). */
int mrs_proximity(const MrsConfig* cfg, const MrsBuffers* bufs, float threshold, float* gap_agent, int* nearest,
                  float* gap_ground, unsigned char* collision, void* stream);
int mrs_raycast(const MrsConfig* cfg, const MrsBuffers* bufs, const float* directions, int n_rays,
                const float* offset3, int body_frame, float range, float* hit_dist, int* hit_id, void* stream);

/* T steps over HOST buffers with the copies pipelined against the kernels (H2D of step t+1 and
 * D2H of step t-1 overlap the kernel of step t on two internal copy streams).  actions_host
 * float[T][E][N][ACTION_DIM] (pinned), dev_actions: caller-owned device staging, TWO action
 * buffers float[2][E][N][ACTION_DIM]; X_host float[T][E][N][D] / A_host float[T][E][N][N] (pinned,
 * may be NULL) receive the newest slice of every step.  Step t writes tape slots
 * slot_x_first - t / slot_a_first - t (the caller guarantees they exist); every step reads bufs->wrench.
 * Synchronises before returning.  The open-loop rollout of examples/simulating_data/helper/DataGenerator.py:8-48 for a
 * caller whose actions and trajectory buffers live in host memory. */
int mrs_rollout_host(const MrsConfig* cfg, const MrsBuffers* bufs, const float* actions_host,
                     float* dev_actions, float* X_host, float* A_host, unsigned int* Abits_host,
                     unsigned int* dev_Abits, int T, int slot_x_first, int slot_a_first, void* stream);

/* ---- the one exchange step of the path: per-rollout statistics reduction across env shards (SURVEY.md §8b/§8e;
 * the reference runs one environment per process and has no counterpart, examples/simulating_data/helper/
 * DataGenerator.py:8-48 gathers its episodes on the host).
 *
 * Environments shard across the GPUs of one node with no traffic on the step; only the MRS_STATS_SLOTS counters
 * are summed across ranks, once per rollout.  64 bytes are a latency problem, so instead of an ncclComm_t the
 * library carries its own peer-memory communicator: every rank owns a small device mailbox (the one device
 * allocation this library makes), all mailboxes are mapped into every process, and the reduction is ONE
 * 32-thread kernel per GPU that pushes its counters into the peers' mailboxes with NVLink stores, waits on
 * local flags and sums in rank order -- stream-ordered, no host involvement, capturable in a CUDA graph.
 *
 *   one process per GPU:  mrs_comm_create -> mrs_comm_handle -> exchange the world x 64 handle bytes by any
 *                         means (torch.distributed, MPI, a file) -> mrs_comm_connect.
 *   one process, N GPUs:  mrs_comm_create per device -> mrs_comm_mailbox -> mrs_comm_connect_ptrs.
 * All calls of one communicator are collective: every rank issues the same sequence of mrs_stats_allreduce /
 * mrs_comm_barrier calls.  A rank that waits more than 4 s for a peer gives up, raises MRS_STATUS_COMM_TIMEOUT in
 * its status word and reports its local counters. */
typedef struct MrsPeerComm MrsPeerComm;
int mrs_comm_create(int rank, int world, MrsPeerComm** out);          /* on the CURRENT device; world <= MRS_COMM_MAX_WORLD */
int mrs_comm_handle(const MrsPeerComm* comm, unsigned char* out_handle /* [MRS_COMM_HANDLE_BYTES] */);
int mrs_comm_connect(MrsPeerComm* comm, const unsigned char* handles /* [world][MRS_COMM_HANDLE_BYTES], rank order */);
void* mrs_comm_mailbox(const MrsPeerComm* comm);
int mrs_comm_connect_ptrs(MrsPeerComm* comm, void* const* mailboxes /* [world] */, const int* devices /* [world] or NULL */);
int mrs_comm_destroy(MrsPeerComm* comm);
/* Device-side barrier across the ranks on `stream` (bench: aligns the start of a timed region on the device). */
int mrs_comm_barrier(MrsPeerComm* comm, unsigned int* status /* device, may be NULL */, void* stream);
/* out[i] (device u64[MRS_STATS_SLOTS], caller-owned) = sum over ranks of bufs->stats[i]; bufs->stats is left as
 * it is.  cfg is unused today (kept for the survey's signature). */
int mrs_stats_allreduce(const MrsConfig* cfg, const MrsBuffers* bufs, MrsPeerComm* comm, unsigned long long* out,
                        void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MRS_B200_H */
