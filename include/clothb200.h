/*
 * clothb200.h - C ABI of libclothb200.so: the B200-native batched replacement for the per-step
 * hot path of gym-cloth's ClothEnv.
 *
 * The reference exposes NO C ABI for this path: the boundary is three CPython extension modules
 * built from Cython (setup.py:39-43) whose classes are called by gym_cloth/envs/cloth_env.py.
 * Every entry point below therefore cites the reference *method* it replaces (paths relative to
 * the reference checkout).  The Python facade in gym_cloth_b200/ binds these symbols with ctypes
 * and re-exposes the reference's own names (Cloth.update, Gripper.grab_top, ClothEnv.step ...);
 * INTEGRATION.md shows the binding a gym-cloth maintainer would add.
 *
 * Conventions
 *  - plain C types only; every pointer documented as HOST or DEVICE; the library never owns
 *    persistent device memory (PyTorch tensors do) except small per-thread scratch caches
 *    used by the *_host convenience entry points and for the derived rows of the *_phys_* ones.
 *  - `stream` is a cudaStream_t passed as void* (NULL = default stream).  Device entry points are
 *    asynchronous on that stream; *_host entry points synchronise the stream before returning.
 *  - return value: 0 = CLOTHB200_OK, negative = error (clothb200_error_string()).  No exceptions
 *    cross the boundary.  Per-environment problems (tear, out-of-bounds, nothing gripped,
 *    coincident points / non-finite state) are reported in the `flags` word, not as errors.
 *  - scalar type by suffix: *_f32 (production) and *_f64 (parity build: bit-exact with the
 *    reference's IEEE-double arithmetic; compiled with -fmad=false).
 *  - state layout in HBM (zero-copy tensors):  pos[n_env][N][4], prev[n_env][N][4] scalars,
 *    N = num_width_points*num_height_points, point index p = r*W + c (cloth.pyx:92-93):
 *        pos [e][p] = { Point.x,  Point.y,  Point.z,  Point.pinned (0 or 1) }   (point.pyx:34-50)
 *        prev[e][p] = { Point.px, Point.py, Point.pz, multiplicity of p in Gripper.grabbed_pts }
 */
#ifndef CLOTHB200_H_
#define CLOTHB200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CLOTHB200_VERSION 110 /* 0.1.1: ClothB200Params.reward_type */

/* error codes */
#define CLOTHB200_OK 0
#define CLOTHB200_ERR_ARG (-1)         /* bad argument (NULL pointer, n_env < 0, misaligned tensor) */
#define CLOTHB200_ERR_CONFIG (-2)      /* config the reference rejects (cloth.pyx:85,91,132) or we cannot run */
#define CLOTHB200_ERR_CUDA (-3)        /* CUDA runtime error, see clothb200_last_cuda_error() */
#define CLOTHB200_ERR_UNSUPPORTED (-4) /* grid too large for one CTA's shared memory, unknown mode */
#define CLOTHB200_ERR_NO_DEVICE (-5)   /* no CUDA device / not sm_100 */

/* per-environment flag bits (int32 flags[n_env], DEVICE, in/out) */
#define CLOTHB200_FLAG_TEAR 1      /* Cloth.cloth_have_tear, sticky (cloth.pyx:272-273); input bit is honoured */
#define CLOTHB200_FLAG_OOB 2       /* ClothEnv._out_of_bounds() after the call (cloth_env.py:1020-1045) */
#define CLOTHB200_FLAG_NOGRAB 4    /* len(gripper.grabbed_pts)==0 -> exit_early (cloth_env.py:490-493) */
#define CLOTHB200_FLAG_BADSTATE 8  /* coincident points (reference: ZeroDivisionError, cloth.pyx:232,331) or non-finite */

/* relaxation ordering */
#define CLOTHB200_MODE_REFERENCE_ORDER 0 /* replays the Cython Gauss-Seidel order exactly */
#define CLOTHB200_MODE_COLOURED 1        /* graph-coloured parallel Gauss-Seidel (not bit-comparable) */

/* cfg env.reward_type: the two types the reference admits (`assert 'coverage' in self.reward_type`, cloth_env.py:130) */
#define CLOTHB200_REWARD_COVERAGE_DELTA 0 /* rew += coverage - previous coverage (cloth_env.py:660-662) */
#define CLOTHB200_REWARD_COVERAGE 1       /* rew += coverage (cloth_env.py:657-659) */

/* initial grid types (cfg init.type, cloth.pyx:94-132) */
#define CLOTHB200_INIT_TIER1 1
#define CLOTHB200_INIT_TIER2 2
#define CLOTHB200_INIT_TIER3 3

/* Everything Cloth.update and ClothEnv.step read from the cfg dict
 * (cloth.pyx:53-56,175-186; cloth_env.py:91-106; gripper.pyx:10-21). */
typedef struct ClothB200Params {
    int32_t num_width_points, num_height_points; /* cfg.cloth.num_*_points; must be equal (cloth.pyx:91) */
    double width, height;                        /* cfg.cloth.width/height */
    double density, ks, damping, thickness, plane_friction, tear_thresh;
    double gravity, minimum_z;                   /* Cloth.__init__ defaults -9.8, 0 (cloth.pyx:24-26) */
    int32_t frames_per_sec, simulation_steps;
    double iters_up, iters_up_rest, iters_grip_rest, iters_rest; /* doubles: tier-3 reset uses a float (cloth_env.py:960) */
    int32_t iters_pull_max, max_actions;
    double reduce_factor, grip_radius, gripper_height;
    int32_t clip_act_space, delta_actions;
    int32_t force_grab;
    int32_t reserved0;                           /* coloured mode: limit passes per update (relax_iters); 0/1 = one pass */
    int32_t reward_type;                         /* cfg env.reward_type (cloth_env.py:657-662): CLOTHB200_REWARD_* */
    int32_t reserved1;
} ClothB200Params;

/* One decoded pull action (cloth_env.py:401-470): where to grip, the per-substep pull delta and
 * the number of pull substeps. */
typedef struct ClothB200Plan {
    double gx, gy;      /* grip point passed to Gripper.grab_top (cloth_env.py:431) */
    double dxr, dyr;    /* x_dir_r, y_dir_r (cloth_env.py:455-456) */
    int32_t iters_pull; /* cloth_env.py:460-470 */
    int32_t reserved;   /* bit 0 = CLOTHB200_PLAN_BAD_ACTION: the action held a NaN.  The reference's iters_pull loop
                           (cloth_env.py:462-467) never exits on one; here the step grips nothing, runs no substep and
                           sets CLOTHB200_FLAG_BADSTATE | CLOTHB200_FLAG_NOGRAB. */
} ClothB200Plan;
#define CLOTHB200_PLAN_BAD_ACTION 1
#define CLOTHB200_MAX_ITERS_PULL (1 << 24) /* bound of the iters_pull accumulation loop (degenerate reduce_factor) */

/* All per-environment tensors one step touches.  DEVICE pointers.  Optional ones may be NULL. */
typedef struct ClothB200Step {
    void *pos, *prev;          /* [n_env][N][4] scalar, in/out (layout above) */
    const void *rest;          /* rest lengths Spring.rest_length (cloth.pyx:417), slot q*6+k for the k-th spring
                                  created by point q (cloth.pyx:135-146), [6N] or [n_env][6N]; NULL = constants of
                                  the flat tier-1/3 grid (f32 only) */
    int64_t rest_env_stride;   /* elements between environments in `rest` (0 = one table shared by all) */
    int32_t *flags;            /* [n_env] in/out, CLOTHB200_FLAG_* */
    int32_t *sim_steps;        /* [n_env] out: Cloth.update() calls executed by this call */
    int32_t *n_grabbed;        /* [n_env] out (optional): len(gripper.grabbed_pts) after grab_top */
    uint32_t *grab_mask;       /* [n_env][ceil(N/32)] out (optional): bit p set <=> p in grabbed_pts after grab_top */
    double *coverage;          /* [n_env] out (optional): ClothEnv._compute_coverage() after the call */
    double *variance_inv;      /* [n_env] out (optional): ClothEnv._compute_variance() */
    void *obs;                 /* [n_env][3N] scalar out (optional): ClothEnv.state for obs_type '1d' (cloth_env.py:196-200) */
    /* episode bookkeeping of ClothEnv.step/_reward/_terminal (cloth_env.py:519-534, 536-715); all or none */
    double *prev_coverage;     /* [n_env] in/out: self._prev_reward */
    int32_t *num_steps;        /* [n_env] in/out: self.num_steps */
    int32_t *num_sim_steps;    /* [n_env] in/out: self.num_sim_steps */
    double *reward;            /* [n_env] out */
    int32_t *done;             /* [n_env] out */
    const double *iters_up_env;/* [n_env] optional per-env override of iters_up (tier-3 reset, cloth_env.py:960) */
    const int32_t *env_order;  /* [n_env] optional: explicit order in which CTAs pick environments; also selects a subset
                                  (n_env entries of a larger batch).  Overrides the built-in scheduling. */
    float *cost;               /* [n_env] optional out: measured SM cycles per substep of each environment's last step
                                  (diagnostics; it does not predict the next step and is not used for scheduling) */
    void *sched_scratch;       /* optional DEVICE scratch.  When given (and env_order is NULL) step_plans / step_actions /
                                  step_host order environments by the substeps their plan will run (0 if the grip catches
                                  nothing), longest first; needs >= 8*pow2ceil(n_env) + 4*n_env bytes. */
    int64_t sched_scratch_bytes; /* size of sched_scratch.  With >= clothb200_sched_scratch_bytes(n_env) bytes and more
                                  environments than resident CTAs (at most 65536), the step runs time-sliced: a
                                  persistent grid runs CLOTHB200_SLICE (default 64) substeps of a cloth at a time and
                                  swaps it for a waiting cloth that has more substeps left (longest remaining first), so
                                  that a launch ends at max(longest action, total work / resident CTAs) rather than
                                  with the last whole action.  Results do not depend on it. */
} ClothB200Step;

/* ---- library / device ---- */
int clothb200_version(void);
const char *clothb200_error_string(int code);
const char *clothb200_last_cuda_error(void);
size_t clothb200_sizeof_params(void);
size_t clothb200_sizeof_plan(void);
size_t clothb200_sizeof_step(void);
/* sm count, compute capability, shared memory per SM of `device` (-1 = current). */
int clothb200_device_info(int device, int *sm_count, int *cc_major, int *cc_minor, int *smem_per_sm);
/* resident cloths per SM / shared memory per cloth for this grid size, f32 (is_f64=0) or f64. */
int clothb200_occupancy(const ClothB200Params *params, int is_f64, int *ctas_per_sm, int *smem_bytes, int *threads);
/* the step kernel step_plans would launch for this grid, mode, rest-table choice (rest_table != 0: ClothB200Step.rest
 * given) and material (per_env_physics != 0: the `_phys` entry points) on the current device, as the runtime reports
 * it: resident CTAs per SM (cudaOccupancyMaxActiveBlocksPerMultiprocessor), registers per thread, local memory
 * (spill) bytes per thread and dynamic shared memory per CTA.  Nothing is launched. */
int clothb200_step_kernel_info(const ClothB200Params *params, int is_f64, int mode, int rest_table, int per_env_physics,
                               int *ctas_per_sm, int *registers, int *local_bytes, int *smem_bytes);

/* values of cfg/t1_rgbd.yaml (identical in t2/t3 apart from init.type). */
int clothb200_params_default(ClothB200Params *params);
/* validation the reference performs in Cloth.__init__ (cloth.pyx:85,91,132). */
int clothb200_params_validate(const ClothB200Params *params);

/* ---- construction: Cloth.__init__ grid + Spring.rest_length (cloth.pyx:92-146, 411-417) ----
 * HOST computation in IEEE double exactly as the reference, rounded to the scalar type on output.
 * noise: N doubles `np_random.rand()*0.01-0.005` (tier2 only; NULL otherwise).  pos4/prev4: HOST [N][4];
 * rest6: HOST [6N] (slot q*6+k; unused slots 0).  Any output may be NULL. */
int clothb200_init_grid_f32(const ClothB200Params *params, int init_type, const double *noise, int init_side,
                            float *pos4, float *prev4, float *rest6);
int clothb200_init_grid_f64(const ClothB200Params *params, int init_type, const double *noise, int init_side,
                            double *pos4, double *prev4, double *rest6);
/* replicate one [N][4] state (DEVICE) into n_env environments (DEVICE). */
int clothb200_broadcast_state_f32(int n_points, int n_env, const float *pos4, const float *prev4, float *pos, float *prev, void *stream);
int clothb200_broadcast_state_f64(int n_points, int n_env, const double *pos4, const double *prev4, double *pos, double *prev, void *stream);

/* ---- action decode: ClothEnv.step lines 401-470 ----
 * host: IEEE double with libm pow() for `**2`, i.e. exactly what CPython computes (bit-exact drop-in).
 * device: same arithmetic with x*x for `**2` (differs from CPython's pow in the last ulp for ~0.085 % of
 * inputs); actions are DEVICE [n_env][4] scalars in env.step's format, plans DEVICE [n_env]. */
int clothb200_decode_actions_host(const ClothB200Params *params, int n_env, const double *actions, ClothB200Plan *plans);
int clothb200_decode_actions_f32(const ClothB200Params *params, int n_env, const float *actions, ClothB200Plan *plans, void *stream);
int clothb200_decode_actions_f64(const ClothB200Params *params, int n_env, const double *actions, ClothB200Plan *plans, void *stream);

/* ---- THE hot path ----
 * clothb200_step_plans_*: for every environment: Gripper.grab_top (gripper.pyx:23-42), then the substep loop of
 * ClothEnv.step (cloth_env.py:472-515): _pull schedule (:352-367) + Cloth.update() (cloth.pyx:169-214) with tear
 * break, then coverage / variance / out-of-bounds and, if the bookkeeping tensors are given, reward and done.
 * One CTA per cloth, whole state resident in shared memory for the entire action.
 * `initialize` != 0 mirrors step(action, initialize=True): no bookkeeping update (cloth_env.py:499-500,517-518). */
int clothb200_step_plans_f32(const ClothB200Params *params, int mode, int n_env, const ClothB200Plan *plans,
                             const ClothB200Step *io, int initialize, void *stream);
int clothb200_step_plans_f64(const ClothB200Params *params, int mode, int n_env, const ClothB200Plan *plans,
                             const ClothB200Step *io, int initialize, void *stream);
/* decode on device + step_plans (plans_scratch: DEVICE [n_env] ClothB200Plan). */
int clothb200_step_actions_f32(const ClothB200Params *params, int mode, int n_env, const float *actions,
                               ClothB200Plan *plans_scratch, const ClothB200Step *io, int initialize, void *stream);
int clothb200_step_actions_f64(const ClothB200Params *params, int mode, int n_env, const double *actions,
                               ClothB200Plan *plans_scratch, const ClothB200Step *io, int initialize, void *stream);
/* n_updates x Cloth.update() with no gripper motion and no tear break - the settle loops of the tier-2/3 resets
 * (cloth_env.py:902-903, 948-949, 980-981) and a bare `cloth.update()` of the facade. */
int clothb200_update_n_f32(const ClothB200Params *params, int mode, int n_env, int n_updates, const ClothB200Step *io, void *stream);
int clothb200_update_n_f64(const ClothB200Params *params, int mode, int n_env, int n_updates, const ClothB200Step *io, void *stream);

/* ---- per-environment material (domain randomisation of the physics) ----
 * The six cfg values Cloth.update turns into constants (cloth.pyx:53-56, 175-186, 240-241), one row per environment.
 * The `_phys` twins below take `physics`, a DEVICE array [n_env] indexed by environment index (the index of `pos`, not
 * the launch position: env_order subsets and the built-in longest-first order work unchanged).  Each row's constants
 * are derived in double and rounded once, exactly as from ClothB200Params, so a row equal to the batch's values gives
 * the plain entry point's bits.  physics == NULL is the plain entry point.  A row with a non-finite value or
 * density <= 0 is invalid: that environment is treated like a CLOTHB200_PLAN_BAD_ACTION plan (no substep, state kept,
 * CLOTHB200_FLAG_BADSTATE | CLOTHB200_FLAG_NOGRAB; update_n: no update, BADSTATE).  The other fields of
 * ClothB200Params (grid, thickness, schedule, gripper) stay per batch. */
typedef struct ClothB200Physics {
    double density, ks, damping, plane_friction, tear_thresh, gravity;
    double reserved[2];        /* 0 */
} ClothB200Physics;            /* 64 bytes */
size_t clothb200_sizeof_physics(void);
int clothb200_step_plans_phys_f32(const ClothB200Params *params, int mode, int n_env, const ClothB200Plan *plans,
                                  const ClothB200Step *io, int initialize, const ClothB200Physics *physics, void *stream);
int clothb200_step_plans_phys_f64(const ClothB200Params *params, int mode, int n_env, const ClothB200Plan *plans,
                                  const ClothB200Step *io, int initialize, const ClothB200Physics *physics, void *stream);
int clothb200_step_actions_phys_f32(const ClothB200Params *params, int mode, int n_env, const float *actions,
                                    ClothB200Plan *plans_scratch, const ClothB200Step *io, int initialize,
                                    const ClothB200Physics *physics, void *stream);
int clothb200_step_actions_phys_f64(const ClothB200Params *params, int mode, int n_env, const double *actions,
                                    ClothB200Plan *plans_scratch, const ClothB200Step *io, int initialize,
                                    const ClothB200Physics *physics, void *stream);
int clothb200_update_n_phys_f32(const ClothB200Params *params, int mode, int n_env, int n_updates, const ClothB200Step *io,
                                const ClothB200Physics *physics, void *stream);
int clothb200_update_n_phys_f64(const ClothB200Params *params, int mode, int n_env, int n_updates, const ClothB200Step *io,
                                const ClothB200Physics *physics, void *stream);
int clothb200_step_host_phys_f32(const ClothB200Params *params, int mode, int n_env, const double *actions,
                                 const ClothB200Step *io, int initialize, float *obs, double *reward, int32_t *done,
                                 double *coverage, double *variance_inv, int32_t *flags, int32_t *sim_steps,
                                 const ClothB200Physics *physics, void *stream);
int clothb200_step_host_phys_f64(const ClothB200Params *params, int mode, int n_env, const double *actions,
                                 const ClothB200Step *io, int initialize, double *obs, double *reward, int32_t *done,
                                 double *coverage, double *variance_inv, int32_t *flags, int32_t *sim_steps,
                                 const ClothB200Physics *physics, void *stream);

/* ---- pieces, for the facade and the parity tests ---- */
/* Gripper.grab_top(x, y) (gripper.pyx:23-42); xy DEVICE [n_env][2] doubles; grip_radius as Gripper.grip_radius. */
int clothb200_grab_top_f32(const ClothB200Params *params, int n_env, const double *xy, double grip_radius,
                           const ClothB200Step *io, void *stream);
int clothb200_grab_top_f64(const ClothB200Params *params, int n_env, const double *xy, double grip_radius,
                           const ClothB200Step *io, void *stream);
/* Gripper.adjust(x,y,z) (gripper.pyx:55-66) with one delta for all environments, and Gripper.release() (:68-73). */
int clothb200_gripper_adjust_f32(int n_points, int n_env, double x, double y, double z, float *pos, float *prev, void *stream);
int clothb200_gripper_adjust_f64(int n_points, int n_env, double x, double y, double z, double *pos, double *prev, void *stream);
int clothb200_gripper_release_f32(int n_points, int n_env, float *pos, float *prev, void *stream);
int clothb200_gripper_release_f64(int n_points, int n_env, double *pos, double *prev, void *stream);
/* coverage / variance_inv / OOB flag of the current state without stepping (cloth_env.py:1075-1098, 1020-1045). */
int clothb200_measure_f32(const ClothB200Params *params, int n_env, const ClothB200Step *io, void *stream);
int clothb200_measure_f64(const ClothB200Params *params, int n_env, const ClothB200Step *io, void *stream);

/* ---- host-buffer entry point (what a CPU-side caller such as ClothEnv.step binds) ----
 * actions HOST [n_env][4] doubles (env.step format).  State stays in the DEVICE tensors of `io`; per-step results
 * are copied back into the HOST arrays (any may be NULL): obs [n_env][3N] scalar, reward/coverage/variance_inv
 * [n_env] double, done/flags/sim_steps [n_env] int32.  Decode is done on the host (bit-exact with CPython).
 * Copies run on `stream` inside the call; the call returns after the stream is synchronised. */
int clothb200_step_host_f32(const ClothB200Params *params, int mode, int n_env, const double *actions,
                            const ClothB200Step *io, int initialize, float *obs, double *reward, int32_t *done,
                            double *coverage, double *variance_inv, int32_t *flags, int32_t *sim_steps, void *stream);
int clothb200_step_host_f64(const ClothB200Params *params, int mode, int n_env, const double *actions,
                            const ClothB200Step *io, int initialize, double *obs, double *reward, int32_t *done,
                            double *coverage, double *variance_inv, int32_t *flags, int32_t *sim_steps, void *stream);

/* ---- image observations (SURVEY.md §8 row f-4): the scene gym_cloth/blender/get_image_rep_279.py builds, rendered on
 * the GPU instead of exporting an .obj and starting Blender per observation (cloth_env.py:212-330).  Blender is not
 * available to pin pixel values; geometry (camera, planes, mesh, which side is visible) follows the script. ---- */
typedef struct ClothB200Scene {
    int32_t height, width;       /* 224 x 224 (cloth_env.py:150-151) */
    int32_t samples;             /* colour image: samples x samples sub-pixel grid (depth images use the pixel centre) */
    int32_t reserved;
    float lens_mm, sensor_mm;    /* 40 / 36 (get_image_rep_279.py:267-277) */
    float cam_pos[3];            /* 0.5, 0.5, 1.45 (:114-117) */
    float cam_deg[3];            /* XYZ Euler degrees, 0 = straight down (:119-122) */
    float lamp_pos[3];           /* the default scene's point lamp; NOSHADOW, CONSTANT falloff (:467-468) */
    float lamp_energy;           /* 1.5 (:469) */
    float diffuse_intensity;     /* 0.8, Blender's material default */
    float horizon;               /* world colour behind everything, linear (0.051) */
    float bed_z, bed_x0, bed_x1, bed_y0, bed_y1;            /* frame0.obj placed by set_bed_pose (:143-156): unit square, z = -0.05 */
    float floor_z, floor_x0, floor_x1, floor_y0, floor_y1;  /* floor.obj, depth images only (:126-140, :455-462): z = -0.25 */
    float front[3], back[3], bed[3];                        /* linear RGB (:249-253, :171) */
} ClothB200Scene;
/* optional per-environment values (domain randomisation, cloth_env.py:786-794), DEVICE pointers, NULL = scene value */
typedef struct ClothB200SceneEnv {
    const float *cam_pos_offset; /* [n_env][3] added to cam_pos */
    const float *cam_deg;        /* [n_env][3] added to cam_deg */
    const float *front, *back, *bed; /* [n_env][3] */
    const int32_t *swap_sides;   /* [n_env] nonzero: colours of the two sides exchanged (tier2 && init_side == -1, :236-238) */
} ClothB200SceneEnv;
size_t clothb200_sizeof_scene(void);
int clothb200_scene_default(ClothB200Scene *scene);
/* colour image, uint8 BGR [n_env][height][width][3] (the channel order cv2.imread returns, cloth_env.py:292) */
int clothb200_render_rgb_f32(const ClothB200Params *params, const ClothB200Scene *scene, const ClothB200SceneEnv *env, int n_env,
                             const float *pos, uint8_t *out_bgr, void *stream);
int clothb200_render_rgb_f64(const ClothB200Params *params, const ClothB200Scene *scene, const ClothB200SceneEnv *env, int n_env,
                             const double *pos, uint8_t *out_bgr, void *stream);
/* depth image as Blender writes it: camera-space Z normalised over the frame, display transform, uint8 [n_env][height][width].
 * zbuf_scratch DEVICE float [n_env][height][width], minmax_scratch DEVICE uint32 [n_env][2]. */
int clothb200_render_depth_f32(const ClothB200Params *params, const ClothB200Scene *scene, const ClothB200SceneEnv *env, int n_env,
                               const float *pos, float *zbuf_scratch, uint32_t *minmax_scratch, uint8_t *out_gray, void *stream);
int clothb200_render_depth_f64(const ClothB200Params *params, const ClothB200Scene *scene, const ClothB200SceneEnv *env, int n_env,
                               const double *pos, float *zbuf_scratch, uint32_t *minmax_scratch, uint8_t *out_gray, void *stream);
/* what cloth_env.py does to the loaded PNG (:296-315).  Depth: cv2.bilateralFilter(img, 7, 50, 50), subtract `sub`
 * ([n_env] or NULL = 50), optional noise, written as three equal-source channels [n_env][h][w][3].  Colour: gamma
 * lookup table ([n_env][256] uint8 as _adjust_gamma builds it, or NULL) and optional noise, in place.
 * noise: DEVICE float [n_env][h][w][3] or NULL. */
int clothb200_post_depth(int n_env, int height, int width, const uint8_t *gray, const float *sub, const float *noise,
                         uint8_t *out_3ch, void *stream);
int clothb200_post_rgb(int n_env, int height, int width, uint8_t *bgr, const uint8_t *lut, const float *noise, void *stream);

/* ---- measurement helpers used by bench.py (microbenchmarks of this GPU's shared-memory and FP32 peaks) ---- */
int clothb200_bench_smem_bandwidth(int iters, double *gb_per_s, void *stream);
int clothb200_bench_fp32_flops(int iters, double *tflop_per_s, void *stream);
/* number of kernels this library has launched since load (bench.py's gpu_launches). */
int64_t clothb200_launch_count(void);
/* bytes of ClothB200Step.sched_scratch that enable the time-sliced step for n_env environments */
size_t clothb200_sched_scratch_bytes(int n_env);
/* tests: pretend the GPU holds `resident_ctas` cloths at once and slice every `slice_substeps` substeps (0, 0 = automatic) */
int clothb200_debug_set_slicing(int resident_ctas, int slice_substeps);
/* debug: DEVICE int64 [n_env][16]; when set, the step kernel records per-phase SM cycles of thread 0 and event counts
 * (0..9 phases of Cloth.update, 10 substeps, 11 replayed buckets, 12 limit-queue pops, 13 springs shortened). NULL = off. */
int clothb200_debug_set_profile(void *dev_int64_nenv_x16);

#ifdef __cplusplus
}
#endif
#endif /* CLOTHB200_H_ */
