/* diygym_b200.h - C ABI of the B200 batched simulation backend (libdiygym_b200.so).
 *
 * Plain pointers and sizes only; no C++ or torch types cross this boundary.  The reference has no FFI of its
 * own for this path: its step path calls the third-party `pybullet` C extension function by function
 * (SURVEY.md 2.3).  Each entry point below names the reference call sites it replaces for N environments at
 * once; INTEGRATION.md shows the ctypes binding the reference-side `DIYGym` would use.
 *
 * Conventions: every function returns 0 on success or a negative DG_E_* code and never throws; the message of
 * the last failure is available from dg_last_error().  Device buffers are OWNED BY THE CALLER (PyTorch in this
 * repo); the library keeps only an immutable copy of the compiled scene and borrowed pointers.  All launches
 * are asynchronous on the caller's stream (`stream` is a cudaStream_t passed as void*; NULL = default stream);
 * no entry point except dg_step_host / dg_world_create / dg_world_destroy synchronises.
 */
#ifndef DIYGYM_B200_H
#define DIYGYM_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct DgWorld DgWorld;

enum { DG_OK = 0, DG_E_ARG = -1, DG_E_SCENE = -2, DG_E_CUDA = -3, DG_E_UNBOUND = -4, DG_E_NOMEM = -5 };

/* dg_query() keys */
enum {
  DG_Q_STATE_SIZE = 0,   /* floats per environment in the state row                */
  DG_Q_PARAM_SIZE = 1,   /* floats per environment in the parameter row            */
  DG_Q_N_ACT = 2, DG_Q_N_OBS = 3, DG_Q_N_REW = 4, DG_Q_N_TERM = 5,
  DG_Q_N_ENVS = 6,
  DG_Q_TEAM = 7,         /* lanes cooperating on one environment                   */
  DG_Q_BLOCK_THREADS = 8,
  DG_Q_GRID_BLOCKS = 9,
  DG_Q_SMEM_BYTES = 10,  /* dynamic shared memory per block of the step kernel      */
  DG_Q_WS_FLOATS = 11,   /* workspace floats per environment                        */
  DG_Q_N_CAMERAS = 12,
  DG_Q_LAUNCHES = 13,    /* kernels launched by this world since creation           */
  DG_Q_RS_ASHARED = 14,  /* floats of shared memory per environment holding the contact solver's row-space matrix */
  DG_Q_SOLVER = 15,      /* 1: row-space team solver for contact environments, 0: per-body sweeps */
  DG_Q_MAX_CONTACTS = 16,     /* contact-point capacity per environment (YAML extension key `max_contacts`) */
  DG_Q_CONTACTS_DROPPED = 17, /* contacts lost to that capacity since the world was created (synchronises the device) */
  DG_Q_SPLIT = 18             /* 1: a step is several stage launches around the contact-sweep kernel, 0: one fused launch */
};

/* Buffers of one world, all DEVICE pointers, row-major with the environment as the leading dimension. */
typedef struct DgBufferTable {
  float* state;    /* [n_envs][state_size]  dynamic state (base pose/twist, q, qd, motor targets, link cache, ...) */
  float* param;    /* [n_envs][param_size]  per-environment parameters (mass, inertia, damping, friction, spawn pose) */
  float* action;   /* [n_envs][n_act]       flattened add-on actions, read by dg_step                     */
  float* obs;      /* [n_envs][n_obs]       flattened add-on observations, written by dg_step / dg_reset   */
  float* reward;   /* [n_envs][n_rew]       one entry per reward add-on                                     */
  uint8_t* term;   /* [n_envs][n_term]      one entry per terminal add-on                                   */
} DgBufferTable;

/* Compile a scene for n_envs environments on CUDA device `device`.
 * (ibuf, fbuf) are the section buffers emitted by diy_gym_b200/compiler/scene.py (layout: csrc/scene_sections.h).
 * team = lanes per environment (1,2,4,8,16,32) or 0 for the built-in choice.
 * DG_E_NOMEM when the scene does not fit the device's shared memory: the step workspace, the ray_sensor shapes, or a scene with
 * a camera whose visual shapes' records exceed one render block (about 1350 visual shapes at 227 KB, DESIGN.md section 4.3).
 * Replaces: p.connect / p.resetSimulation / p.setPhysicsEngineParameter / p.setGravity / p.loadURDF ...
 *           (/root/reference/diy_gym/diy_gym.py:68-86, diy_gym/model.py:65-83) */
int dg_world_create(const int32_t* ibuf, int n_ibuf, const double* fbuf, int n_fbuf, int n_envs, int device, int team,
                    DgWorld** out);
/* Replaces p.disconnect (/root/reference/diy_gym/diy_gym.py:225) */
void dg_world_destroy(DgWorld* w);
const char* dg_last_error(const DgWorld* w);   /* w may be NULL: last dg_world_create failure */
int64_t dg_query(const DgWorld* w, int key);

/* Borrow the caller's device buffers. */
int dg_bind_buffers(DgWorld* w, const DgBufferTable* t);
/* Per-environment RNG stream id = env_id_offset + local index (so results do not depend on the GPU count). */
int dg_set_seed(DgWorld* w, uint32_t seed, int env_id_offset);
/* Which action ops take part in the next dg_step calls: op_enabled[k] == 0 skips op k (HOST array, one byte per
 * scene op).  Mirrors the reference's rule that only add-ons present in the action dict are updated
 * (/root/reference/diy_gym/diy_gym.py:202-204).  Default: all enabled. */
int dg_set_action_mask(DgWorld* w, const uint8_t* op_enabled, int n_ops);
/* Fill state and parameter rows with the scene defaults (what loadURDF + resetBasePositionAndOrientation leave). */
int dg_init_state(DgWorld* w, void* stream);

/* One DIYGym.step for every environment: add-on update(action) -> stepSimulation -> observe/reward/is_terminal.
 * Replaces /root/reference/diy_gym/diy_gym.py:187-209 (p.stepSimulation at :207 and every add-on hook it fans out to).
 * Scenes with ray_sensor add-ons: their distances (and hit body ids) are part of obs, cast by one more launch on `stream`
 * after the step (dg_ray_kernel); the same holds for dg_reset (masked environments only), dg_observe and dg_step_host. */
int dg_step(DgWorld* w, void* stream);
/* Measurement aid (no reference counterpart): per-block, per-phase cycle sums of the step kernel.  enable != 0 allocates and
 * clears a [grid][64] table keyed by (source line of the phase in dg_env.cuh) & 63; dg_debug_read copies n <= grid * 64
 * entries out and clears the table; enable == 0 frees it.  tools/phase_probe.py prints the result. */
int dg_debug_phase_cycles(DgWorld* w, int enable);
int dg_debug_read(DgWorld* w, unsigned long long* out, int n);
/* DIYGym.reset for the environments whose mask byte is non-zero (mask_dev == NULL: all).
 * Replaces /root/reference/diy_gym/diy_gym.py:130-148 (add-on reset hooks, hot-start steps, observe).  Ray_sensor rays of the
 * masked environments are cast after it (see dg_step); the other environments' obs rows are not touched. */
int dg_reset(DgWorld* w, const uint8_t* mask_dev, void* stream);
/* DIYGym.observe / reward / is_terminal on the state rows as they are (no physics): refreshes the link-pose cache the sensors
 * read and evaluates every sensor / reward / terminal op into obs / reward / term (ray_sensor rays included, see dg_step).
 * Replaces /root/reference/diy_gym/diy_gym.py:211-222 (observe, reward, is_terminal -> walk_addons). */
int dg_observe(DgWorld* w, void* stream);
/* Camera add-on number `cam`: rgb [n_envs][H][W][3] float in [0,1], depth [n_envs][H][W] eye-space z (negative).
 * Replaces p.getCameraImage + post-processing (/root/reference/diy_gym/addons/sensors/camera.py:58-92). */
int dg_render(DgWorld* w, int cam, float* rgb_dev, float* depth_dev, void* stream);
/* The same with the segmentation mask of sensors/camera.py:54-56,89-90 (`use_segmentation_mask`): seg_dev [n_envs][H][W] gets
 * the unique id (body index in load order) of the body visible in each pixel, -1 for the background; NULL = no mask. */
int dg_render_seg(DgWorld* w, int cam, float* rgb_dev, float* depth_dev, float* seg_dev, void* stream);
/* The same with the colour image as bytes: rgb_dev [n_envs][H][W][3] uint8 = round(255 c) - the renderer's own output format,
 * which the reference divides by 255 (sensors/camera.py:76-78); a quarter of the colour bytes to move.  seg_dev may be NULL.
 * All three render calls store whole 16-byte pieces: float buffers must be 16-byte aligned, colour bytes 8-byte aligned. */
int dg_render_u8(DgWorld* w, int cam, uint8_t* rgb_dev, float* depth_dev, float* seg_dev, void* stream);

/* Rigid-body dynamics of body `body` (load order) for every environment, from its state and parameter rows: one launch on `stream`.
 * Generalized velocity nu: [omega_base, v_base (world axes, base COM), qd] for a floating base, qd for a fixed one; n = len(nu) <=
 * DG_DYN_MAX_N.  q_dev [n_envs][n_dof] joint positions (the base pose always comes from the state row), qd_dev / qdd_dev
 * [n_envs][n]; NULL: the state row's q, the state row's nu, zero.  Outputs, NULL = not computed:
 *   jac_dev  [n_envs][6][n]  Jacobian of the point `point` (link COM frame; NULL = the COM) of link `link` (-1 = base), world axes,
 *                            linear rows first (p.calculateJacobian)
 *   mass_dev [n_envs][n][n]  M(q) (p.calculateMassMatrix)
 *   tau_dev  [n_envs][n]     M(q) qdd + C(q, nu) nu + G(q), the scene's gravity; a floating base's first six entries are the base
 *                            wrench [torque about the base COM, force] (p.calculateInverseDynamics)
 * Masses and inertias are the parameter row's (dynamics_randomizer is honoured); joint damping, motors, limits, contacts and welds
 * are not part of it.  Writes nothing but the outputs.  DG_E_ARG for a body without degrees of freedom, n > DG_DYN_MAX_N or a
 * link out of range. */
enum { DG_DYN_MAX_N = 64 };
int dg_body_dynamics(DgWorld* w, int body, int link, const float point[3], const float* q_dev, const float* qd_dev, const float* qdd_dev,
                     float* jac_dev, float* mass_dev, float* tau_dev, void* stream);

/* Inverse kinematics of body `body` (load order) for every environment (p.calculateInverseKinematics): one launch on `stream`.
 * The solve is the ik_controller op's damped least squares: at most max_iters iterations while the position residual of the last
 * iterate exceeds `threshold`, on the URDF frame of link `link` (0 <= link < links of the body) in the coordinates of the base,
 * whose pose is the state row's and stays fixed.
 *   target_pos_dev [n_envs][3]            world position of the link frame
 *   target_orn_dev [n_envs][4] or NULL     world orientation (xyzw, normalised here); NULL: position only (3 task rows)
 *   q0_dev         [n_envs][nd] or NULL     seed (nd = the body's DoF); NULL: the state row's q
 *   limits_dev     [n_envs][4][nd] or NULL  lower, upper, range, rest: adds the null-space term (SURVEY App. A.4); NULL: none
 *   q_out_dev      [n_envs][nd]             the solution, the body's DoF in order
 *   err_dev        [n_envs][2] or NULL      at q_out: distance of the link frame from the target (m), angle of the remaining
 *                                           rotation (rad; 0 without target_orn)
 * Writes nothing but the outputs and a scratch buffer the world allocates on the first call (calls on different streams must not
 * overlap).  DG_E_ARG for no such body, a body without degrees of freedom, nd > DG_IK_MAX_ND, a link out of range,
 * max_iters < 1, a negative or NaN threshold, or a NULL target_pos_dev / q_out_dev. */
enum { DG_IK_MAX_ND = 64 };
int dg_body_ik(DgWorld* w, int body, int link, const float* target_pos_dev, const float* target_orn_dev, const float* q0_dev,
               const float* limits_dev, int max_iters, float threshold, float* q_out_dev, float* err_dev, void* stream);

/* Host-buffer form of dg_step (the reference-facing call when the caller keeps numpy arrays): copies the actions
 * host->device, steps, copies obs / reward / terminal device->host and waits.  Any output pointer may be NULL. */
int dg_step_host(DgWorld* w, const float* action_host, float* obs_host, float* reward_host, uint8_t* term_host, void* stream);

/* Measured non-tensor FP32 FMA issue rate of the device in TFLOP/s (the physics kernels' compute roofline). */
int dg_measure_fp32_peak(int device, double* tflops_out);

#ifdef __cplusplus
}
#endif
#endif
