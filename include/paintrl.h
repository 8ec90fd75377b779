/*
 * paintrl.h -- C ABI of the B200-native batched paint-simulation step.
 *
 * The reference (translearn/PaintRL) has no FFI boundary of its own: the step path sits behind a
 * Python "operator API" of module functions keyed by PyBullet body id
 * (PaintRLEnv/bullet_paint_wrapper.py:1327-1400) and behind gym.Env
 * (PaintRLEnv/robot_gym_env.py:207-422).  This header is the batched, device-resident mirror of
 * exactly that path; each entry point names the reference interface it replaces.
 *
 * Conventions
 *   - plain C, no torch / CUDA types in signatures: device pointers are `void*`/typed pointers to
 *     device memory, the stream is an opaque `void*` holding a cudaStream_t (NULL = default).
 *   - every call returns 0 on success or a negative PAINTRL_E_* code; the message is available
 *     from paintrl_last_error() (thread-local).
 *   - the library owns per-environment state and its device copy of the part tables; the caller
 *     owns every I/O buffer (contiguous, 16-byte aligned) and the stream.
 *   - *_dev calls are asynchronous on the given stream and never synchronise; *_host calls copy
 *     host<->device inside the call and return after the stream has drained.
 *   - a handle is not thread-safe; different handles (one per GPU) are independent.  All calls on one
 *     handle must be issued on ONE stream (or on streams the caller orders): the two kernels of a step hand
 *     over per environment through device flags.
 *   - there is NO CPU fallback: without a CUDA device paintrl_create fails with PAINTRL_E_CUDA.
 */
#ifndef PAINTRL_H_
#define PAINTRL_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PAINTRL_ABI_VERSION 2
#define PAINTRL_STATE_SCALARS 12   /* doubles per environment in the `scalars` of paintrl_get_state / paintrl_set_state */

enum {
    PAINTRL_OK = 0,
    PAINTRL_E_INVALID = -1,   /* bad argument / unsupported configuration            */
    PAINTRL_E_CUDA = -2,      /* CUDA runtime error (no device, launch failure, OOM) */
    PAINTRL_E_STATE = -3      /* call not valid in the current state                 */
};

/* robot_gym_env.py:126-132 class attributes */
enum { PAINTRL_ACTION_DISCRETE = 0, PAINTRL_ACTION_CONTINUOUS = 1 };
enum { PAINTRL_OBS_SECTION = 0, PAINTRL_OBS_GRID = 1, PAINTRL_OBS_SIMPLE = 2, PAINTRL_OBS_DISCRETE = 3 };
/* robot_gym_env.py:134-157 extra_config */
enum { PAINTRL_COLOR_RGB = 0, PAINTRL_COLOR_HSI = 1 };
enum { PAINTRL_TERM_LATE = 0, PAINTRL_TERM_EARLY = 1, PAINTRL_TERM_HYBRID = 2 };
/* robot.py:172 Robot.PAINT_METHOD */
enum { PAINTRL_PAINT_FAST = 0, PAINTRL_PAINT_NORMAL = 1 };

/*
 * Constant per-part tables (SURVEY.md section 8a row P), all host pointers, row-major, FP64
 * unless noted.  They are the outputs of the reference's load-time preprocessing
 * (bullet_paint_wrapper.py:622-648, 599-620, 816-832, 922-963, 740-783); paintrl_create copies
 * what it needs to the device and builds its own acceleration tables from them.
 */
typedef struct PaintrlPartPack {
    int32_t abi_version;          /* PAINTRL_ABI_VERSION */
    int32_t width, height;        /* texture size (bullet_paint_wrapper.py:714-718) */
    int32_t axis0, axis1;         /* principal axes (bullet_paint_wrapper.py:1294-1300) */

    int32_t n_texels;             /* front-side texels: len(profile[front]) */
    const double *texel_pos;      /* [n_texels,3]  pixel_positions[front]   */
    const int32_t *texel_ij;      /* [n_texels,2]  profile[front] (i,j)     */

    int32_t n_planes;             /* collision hull half-spaces n.x <= off (shim S1) */
    const double *plane_n;        /* [n_planes,3] */
    const double *plane_off;      /* [n_planes]   */

    int32_t n_vertices;           /* side-masked vertex set (bullet_paint_wrapper.py:599-620) */
    const double *vertices;       /* [n_vertices,3] */
    const int32_t *vtri_start;    /* [n_vertices+1] CSR of uv_map restricted to front triangles */
    const int32_t *vtri_idx;      /* [vtri_start[n_vertices]] in uv_map order */

    int32_t n_tris;               /* front triangles (BarycentricInterpolator, :123-146) */
    const double *tri_a;          /* [n_tris,3] */
    const double *tri_v0;         /* [n_tris,3] */
    const double *tri_v1;         /* [n_tris,3] */
    const double *tri_d00, *tri_d01, *tri_d11, *tri_inv_denom;   /* [n_tris] each */
    const double *tri_n;          /* [n_tris,3] corrected normals (:650-698) */

    double range0_min, range0_max;   /* ranges along axis0 / axis1 (:1282-1285) */
    double range1_min, range1_max;
    double length_width_ratio;       /* :817 */

    int32_t grid_granularity;     /* Part.GRID_GRANULARITY = 100 (:447) */
    const double *grid_lo;        /* [grid_granularity] silhouette table grid_dict[front] (:922-963) */
    const double *grid_hi;

    int32_t n_starts;             /* start points of the configured START_POINT_MODE (:749-783) */
    const double *start_pos;      /* [n_starts,3] */
    const double *start_normal;   /* [n_starts,3] */

    int32_t status_init;          /* first-channel value of a fresh front texel: 191 RGB / 255 HSI (:586) */

    /* PAINTRL_PAINT_NORMAL only (may be NULL otherwise): for every front texel, the texel that the reference's
     * cKDTree.query(k = 1) (bullet_paint_wrapper.py:565) returns among the texels sharing its exact 3-D position (UV
     * seams map a few texels to the same point: 109 groups on the door).  Which twin the kd-tree reports is fixed
     * by the tree's leaf order, not by the query, so it is a constant table; identity for unique positions. */
    const int32_t *texel_nn_rep;  /* [n_texels] */
} PaintrlPartPack;

/* Everything PaintGymEnv reads at construction (robot_gym_env.py:126-157, 240-252). */
typedef struct PaintrlConfig {
    int32_t abi_version;
    int32_t action_mode;            /* PAINTRL_ACTION_*            ACTION_MODE  */
    int32_t action_shape;           /* 1 or 2                      ACTION_SHAPE */
    int32_t discrete_granularity;   /* DISCRETE_GRANULARITY */
    /* [discrete_granularity + 1,3] host table (u1, u2, turning angle) for the discrete actions 0..n; row n
     * serves every action >= n (the reference clips, robot.py:390-393), actions < 0 use row 0;
     * computed by the host exactly as robot_gym_env.py:342-347 + robot.py:151-160,352-358 do
     * (NumPy cos/sin, libm atan), so discrete directions are bit-identical to the reference. */
    const double *discrete_table;
    int32_t obs_mode;               /* PAINTRL_OBS_*               OBS_MODE */
    int32_t obs_grad;               /* OBS_GRAD */
    int32_t color_mode;             /* PAINTRL_COLOR_*             COLOR_MODE */
    int32_t termination_mode;       /* PAINTRL_TERM_*              TERMINATION_MODE */
    double switch_threshold;        /* SWITCH_THRESHOLD */
    int32_t expected_episode_length;/* Expected_Episode_Length */
    int32_t episode_max_length;     /* EPISODE_MAX_LENGTH */
    int32_t turning_penalty;        /* TURNING_PENALTY (bool) */
    int32_t overlap_penalty;        /* OVERLAP_PENALTY (bool) */
    double max_possible_point;      /* Part_Dict[Part_NO][1] (robot_gym_env.py:106-117) */
    /* Not in the reference (one env per process there): what to do when an episode ends.
     * 0: nothing -- the caller resets by index with paintrl_reset (gym semantics, :370-387).
     * 1: same-step auto-reset -- `obs` still receives the terminal observation (:358); the env is
     *    then reset and the first observation of the new episode goes to `next_obs`.          */
    int32_t auto_reset;
    uint64_t seed;                  /* start-index stream for auto-reset (uniform over n_starts) */
    /* Robot.PAINT_METHOD (robot.py:172, 414-417).  PAINTRL_PAINT_FAST: every shot is the ball query of its centre
     * (Part.fast_paint, bullet_paint_wrapper.py:568-570) -- the reference's default.  PAINTRL_PAINT_NORMAL: every shot
     * casts the beam fan `beam_plain` from the TCP (Robot._paint / _generate_paint_beams, robot.py:251-258, 280-285)
     * and paints the texel nearest to each hit (Part.paint, bullet_paint_wrapper.py:562-566).
     * beam_plain: host float64 [n_beams, 3], the ray end points in the TCP frame (Robot._paint_plain: the uniform
     * disc of robot.py:23-36 for RGB, the beta-distributed rings of :39-69 for HSI; both at z = 0.2). */
    int32_t paint_method;
    int32_t n_beams;
    const double *beam_plain;
} PaintrlConfig;

typedef struct PaintrlEngine *PaintrlHandle;

/* Batched PaintGymEnv.__init__ after load_part (robot_gym_env.py:207-229, 271-287): allocates
 * `num_envs` environments on CUDA device `device`.  State is undefined until paintrl_reset. */
int paintrl_create(const PaintrlPartPack *pack, const PaintrlConfig *cfg, int32_t num_envs,
                   int32_t device, PaintrlHandle *out);
/* PaintGymEnv.close (robot_gym_env.py:417-418). */
void paintrl_destroy(PaintrlHandle h);

int32_t paintrl_num_envs(PaintrlHandle h);
int32_t paintrl_obs_dim(PaintrlHandle h);    /* observation_space.shape[0] (robot_gym_env.py:166-173) */
int32_t paintrl_action_dim(PaintrlHandle h); /* 1 (discrete, int64) or ACTION_SHAPE (float64) */
int32_t paintrl_num_texels(PaintrlHandle h);
int32_t paintrl_status_bytes(PaintrlHandle h); /* bytes per texel of the status plane: 1 RGB, 2 HSI */
/* device bytes of per-environment state the step reads and writes: flip-bit plane (+ int16 thickness plane in HSI,
 * + grid-cell counters in grid mode) + the 128-byte record, move output, counters and hand-off flag */
int64_t paintrl_state_bytes_per_env(PaintrlHandle h);

/* PaintGymEnv.reset (robot_gym_env.py:370-387) = Part.reset_part (bullet_paint_wrapper.py:706-712)
 * + Robot.reset (robot.py:366-372) + _augmented_observation.
 *   env_ids_dev : int32[n] environments to reset, or NULL for all (then n == num_envs)
 *   start_idx_dev: int32[n] index into the start-point table per reset env (the reference draws
 *                  it with random.randint; rollout mode uses 0), or NULL for the seeded stream
 *   obs_dev     : float64[n, obs_dim] first observation of each reset env, or NULL */
int paintrl_reset(PaintrlHandle h, const int32_t *env_ids_dev, int32_t n,
                  const int32_t *start_idx_dev, double *obs_dev, void *stream);

/* Robot.reset(pose) alone (robot.py:366-372), as spiral.py:28-38 calls it after env.reset():
 * places the TCP at pos/normal without touching the texture or the episode counters.
 *   pos_dev, normal_dev: float64[n,3];  obs_dev: float64[n, obs_dim] or NULL */
int paintrl_set_pose(PaintrlHandle h, const int32_t *env_ids_dev, int32_t n, const double *pos_dev,
                     const double *normal_dev, double *obs_dev, void *stream);

/* PaintGymEnv.step for every environment (robot_gym_env.py:349-368 and everything under it:
 * robot.py:383-433, bullet_paint_wrapper.py:865-880, 568-577, 965-978, 1045-1061, 1126-1139).
 *   actions_dev   : int64[num_envs] (discrete) or float64[num_envs, action_shape] (continuous)
 *   obs_dev       : float64[num_envs, obs_dim]  observation after the step (terminal obs if done)
 *   reward_dev    : float64[num_envs]  info['reward']   = newly painted / 100
 *   penalty_dev   : float64[num_envs]  info['penalty']
 *   actual_dev    : float64[num_envs]  the step's return value reward - penalty
 *   done_dev      : uint8[num_envs]
 *   new_texels_dev: int32[num_envs] texels newly painted by this step (RGB) / thickness units
 *                   removed (HSI); may be NULL
 *   next_obs_dev  : float64[num_envs, obs_dim] observation to act on next (== obs unless the env
 *                   auto-reset in this call); may be NULL; only written when cfg.auto_reset
 *   reset_start_idx_dev: int32[num_envs] start index to use if env e auto-resets in this call;
 *                   NULL = seeded stream */
int paintrl_step(PaintrlHandle h, const void *actions_dev, double *obs_dev, double *reward_dev,
                 double *penalty_dev, double *actual_dev, uint8_t *done_dev,
                 int32_t *new_texels_dev, double *next_obs_dev,
                 const int32_t *reset_start_idx_dev, void *stream);

/* paintrl_step for the environments env_ids_dev[0..n) (device int32, unique), or, when env_ids_dev is NULL,
 * for env_lo .. env_lo + n - 1.  Every I/O buffer has n rows, row k = the k-th listed environment.
 * What the step does to a listed environment is exactly what paintrl_step does to it (record, planes,
 * counters, the seeded auto-reset stream); the other environments are not touched.  The kernel shape
 * (one or two launches) follows n.  Ids outside [0, num_envs) are skipped by the device code; unique ids
 * are the caller's contract.  PAINTRL_E_INVALID for n outside [1, num_envs], a range outside the batch or
 * env_lo != 0 together with a list. */
int paintrl_step_subset(PaintrlHandle h, const int32_t *env_ids_dev, int32_t env_lo, int32_t n,
                        const void *actions_dev, double *obs_dev, double *reward_dev, double *penalty_dev,
                        double *actual_dev, uint8_t *done_dev, int32_t *new_texels_dev, double *next_obs_dev,
                        const int32_t *reset_start_idx_dev, void *stream);

/* Same step with HOST buffers: copies the actions host->device, runs the step, copies
 * obs/reward/penalty/actual/done (and next_obs if given) device->host, and returns once they
 * have landed.  This is the call the gym / VectorEnv surface makes. */
int paintrl_step_host(PaintrlHandle h, const void *actions_host, double *obs_host,
                      double *reward_host, double *penalty_host, double *actual_host,
                      uint8_t *done_host, double *next_obs_host, void *stream);

/* The same host-buffer step, split in two so that consecutive steps overlap: `submit` queues the host->device copy of
 * the actions (on a copy stream of the library's own), the step (on `stream`) and the device->host copy of the results
 * (on a second copy stream) and returns at once; `wait` blocks until the results of that slot have landed.  Two slots
 * (0 and 1) with separate device staging: step t + 1 may be submitted on the other slot before step t is waited for --
 * its copy-in and kernels then run while step t's results travel and the host wakes up.  Steps execute in submission
 * order.  The host buffers of a slot (actions included) belong to the library between submit and wait; pinned memory
 * is needed for the copies to be asynchronous.  A slot resubmitted without a wait first waits for its own copy-out. */
int paintrl_step_host_submit(PaintrlHandle h, int32_t slot, const void *actions_host, double *obs_host,
                             double *reward_host, double *penalty_host, double *actual_host,
                             uint8_t *done_host, double *next_obs_host, void *stream);
/* paintrl_step_host_submit for the range env_lo .. env_lo + n - 1: host buffers of n rows; completed by
 * paintrl_step_host_wait(slot).  Two slots = two groups in flight: a closed-loop host policy computes one group's
 * next actions while the other group steps.  Results come back in the same obs | reward | penalty | actual |
 * [next_obs] | done order, sized for n rows. */
int paintrl_step_host_submit_range(PaintrlHandle h, int32_t slot, int32_t env_lo, int32_t n, const void *actions_host,
                                   double *obs_host, double *reward_host, double *penalty_host, double *actual_host,
                                   uint8_t *done_host, double *next_obs_host, void *stream);
int paintrl_step_host_wait(PaintrlHandle h, int32_t slot);

/* State access (the reference keeps it in Part.texels / Robot._pose,_orn / PaintGymEnv counters,
 * robot_gym_env.py:219-221, robot.py:201-218, bullet_paint_wrapper.py:467,483).
 * status_dev: int16[n, n_texels] first-channel value per front texel in part-pack order
 *             (== get_texture_image's R plane restricted to profile[front]);
 * pose_dev  : float64[n,3]; quat_dev: float64[n,4];
 * scalars_dev: float64[n, PAINTRL_STATE_SCALARS] = total_reward, total_return, step_counter, terminate_counter,
 *             last_on_part, terminate, last_turning_angle, angle_diff, has_overlap_reference,
 *             overlap_reference_centre[3].  The last four carry Part._last_painted_pixels
 *             (bullet_paint_wrapper.py:483, 575-576) exactly: that set is the ball query of the previous shot's
 *             centre, so a state saved mid-episode and restored into another handle continues bit for bit,
 *             OVERLAP_PENALTY included.  paintrl_set_state with a status plane but without scalars clears the
 *             reference (as reset_part does, :708).  Any pointer may be NULL.
 * env_ids must be in [0, num_envs) and unique; ids out of range are ignored by the device code. */
int paintrl_get_state(PaintrlHandle h, const int32_t *env_ids_dev, int32_t n, int16_t *status_dev,
                      double *pose_dev, double *quat_dev, double *scalars_dev, void *stream);
int paintrl_set_state(PaintrlHandle h, const int32_t *env_ids_dev, int32_t n,
                      const int16_t *status_dev, const double *pose_dev, const double *quat_dev,
                      const double *scalars_dev, void *stream);

/* get_job_status / get_job_limit (bullet_paint_wrapper.py:727-735): painted front texels per env.
 * painted_dev: int32[num_envs] */
int paintrl_job_status(PaintrlHandle h, int32_t *painted_dev, void *stream);

/* Per-handle counters since creation (device-side, read back synchronously): env-steps run,
 * episodes ended, sum of footprint-union texels, kernels launched by this library. */
typedef struct PaintrlStats {
    uint64_t env_steps;
    uint64_t episodes_ended;
    uint64_t footprint_texels;
    uint64_t kernel_launches;
    uint64_t ray_full_scans;   /* rays that needed the full plane list (5 rays per env-step) */
    uint64_t move_bailouts;    /* env-steps whose move phase left the fast kernel and ran in the paint warp */
} PaintrlStats;
int paintrl_stats(PaintrlHandle h, PaintrlStats *out);

/* Load-time texel rasterisation (Part.preprocess + BarycentricInterpolator.get_uv_pixels,
 * bullet_paint_wrapper.py:604-618, 191-212) at an arbitrary texture size, on the GPU: the front
 * texels (i, j) and their 3-D positions from the front triangles' corners and UV coordinates.
 * This is what makes textures other than the reference's 240x240 usable (the reference's own loader
 * is O(W * H * n) Python).  All pointers are HOST pointers; synchronous.
 *   tri_a/b/c : float64[n_tris,3] corners, tri_uv: float64[n_tris,3,2], both in bary_list order;
 *   capacity  : rows available in the outputs; 0 = only count (outputs may be NULL);
 *   texel_ij_out: int32[capacity,2], texel_pos_out: float64[capacity,3], sorted by (i, j);
 *   *n_texels_out: number of front texels. */
int paintrl_rasterize_texels(const double *tri_a, const double *tri_b, const double *tri_c,
                             const double *tri_uv, int32_t n_tris, int32_t width, int32_t height,
                             int32_t device, int32_t capacity, int32_t *texel_ij_out,
                             double *texel_pos_out, int32_t *n_texels_out);

/* Load-time silhouette scans (Part._get_exact_boundary, bullet_paint_wrapper.py:906-920, called by _set_grid_dict
 * :922-963 for the left and the right end of every row of the 100-row grid): from `points[k]` march along
 * `proof_axis` in 1 mm steps (towards smaller values where is_min[k]) and test, at every step, a ray along
 * `non_principal_axis` (end points 1, 2, 3 ... beyond the point on either side, as the reference accumulates them)
 * against the collision hull  plane_n . x <= plane_off  with shim S1's slab arithmetic; boundary_out[k] is the coordinate
 * of the first step whose ray misses, found_out[k] = 0 when none of the `steps_range` steps does (the reference then
 * returns None).  One warp per scan on the GPU.  All pointers are HOST pointers; synchronous. */
int paintrl_silhouette_march(const double *plane_n, const double *plane_off, int32_t n_planes, const double *points,
                             const int8_t *is_min, int32_t n_scans, int32_t proof_axis, int32_t non_principal_axis,
                             int32_t steps_range, int32_t device, double *boundary_out, int8_t *found_out);

/*
 * The grid-world ParamTestEnv (PaintRLEnv/param_test_env.py:96-246; driven by param_test_*.py), batched:
 * one handle = num_envs independent size x size worlds on one GPU.  Same conventions as above.
 */
enum { PAINTRL_PARAM_OBS_SECTION = 0, PAINTRL_PARAM_OBS_SIMPLE = 1, PAINTRL_PARAM_OBS_DIRECT = 2, PAINTRL_PARAM_OBS_GRID = 3 };
typedef struct PaintrlParamConfig {
    int32_t abi_version;            /* PAINTRL_ABI_VERSION */
    int32_t size;                   /* ParamTestEnv(size, ...)                      (param_test_env.py:110) */
    int32_t max_len;                /* EPISODE_MAX_LENGTH = max(max_len, (size-2)^2) (:112) */
    int32_t termination_by_repeat;  /* (:146) */
    int32_t obs_mode;               /* class attribute OBS_MODE (:101): section 4+2, simple 2, direct size^2+2, grid 100+2 */
    int32_t auto_reset;             /* reset a finished world inside the step; next_obs gets reset()'s observation */
} PaintrlParamConfig;
typedef struct PaintrlParamEngine *PaintrlParamHandle;

int paintrl_param_create(const PaintrlParamConfig *cfg, int32_t num_envs, int32_t device, PaintrlParamHandle *out);
void paintrl_param_destroy(PaintrlParamHandle h);
int32_t paintrl_param_obs_dim(PaintrlParamHandle h);
/* ParamTestEnv.reset (:150-160); env_ids_dev NULL = all; obs_dev float64[n, obs_dim] or NULL */
int paintrl_param_reset(PaintrlParamHandle h, const int32_t *env_ids_dev, int32_t n, double *obs_dev, void *stream);
/* ParamTestEnv.step (:218-240): actions int64[num_envs] in 0..3.  The reference raises IndexError for anything else
 * (:173-174); here such a world is left untouched, its output row is written as (current observation, reward 0,
 * penalty 0, done 1) and the bad-action flag of paintrl_param_stats is raised (reported once, then cleared) --
 * the host mirror checks the actions before the launch and raises IndexError like the reference. */
int paintrl_param_step(PaintrlParamHandle h, const int64_t *actions_dev, double *obs_dev, double *reward_dev,
                       double *penalty_dev, double *actual_dev, uint8_t *done_dev, double *next_obs_dev, void *stream);
/* world / visit_table (:113-131) of the listed worlds as int32[n, size*size] (visit counts saturate at 65535) */
int paintrl_param_tables(PaintrlParamHandle h, const int32_t *env_ids_dev, int32_t n, int32_t *world_dev,
                         int32_t *visit_dev, void *stream);
int paintrl_param_stats(PaintrlParamHandle h, uint64_t *env_steps, uint64_t *episodes_ended,
                        uint64_t *kernel_launches, int32_t *bad_action_seen);

/*
 * The rollout policy of the reference's PPO script (paint_ppo.py:179-183: fully connected obs -> 256 -> 128 ->
 * {logits | mean, value}, tanh, value branch sharing the hidden layers) evaluated and sampled for a whole batch in
 * ONE kernel launch per environment step (layer 2 on the tcgen05 tensor cores, BF16 inputs, FP32 accumulation):
 * observations come straight from paintrl_step's obs buffer, actions go straight into the next paintrl_step.
 * Weights are host pointers, row-major FP32: w1 [obs_dim][256], b1 [256], w2 [256][128], b2 [128],
 * w3 [128][n_out + 1] (last column = value head), b3 [n_out + 1].  obs_dim <= 32, n_out <= 15.
 */
typedef struct PaintrlPolicyConfig {
    int32_t abi_version;
    int32_t obs_dim;
    int32_t n_out;          /* discrete: number of actions (logits); continuous: action dimensions (means) */
    int32_t discrete;       /* 1: Gumbel-max sample of the logits (int64 actions); 0: tanh(mean) + unit Gaussian (float64) */
    int32_t capacity;       /* largest batch (one random-number counter per environment) */
    uint64_t seed;
    const float *w1, *b1, *w2, *b2, *w3, *b3;
} PaintrlPolicyConfig;
typedef struct PaintrlPolicyEngine *PaintrlPolicyHandle;

int paintrl_policy_create(const PaintrlPolicyConfig *cfg, int32_t device, PaintrlPolicyHandle *out);
void paintrl_policy_destroy(PaintrlPolicyHandle h);
/* obs_dev float64 [batch, obs_dim]; actions_dev int64 [batch] (discrete) or float64 [batch, n_out]; logp_dev /
 * value_dev float32 [batch]; logits_dev float32 [batch, n_out + 1] or NULL (logits | means, then the value).
 * sample = 0 evaluates value (and logits) only -- the bootstrap value at the end of a fragment -- and draws nothing. */
int paintrl_policy_act(PaintrlPolicyHandle h, const double *obs_dev, int32_t batch, void *actions_dev, float *logp_dev,
                       float *value_dev, float *logits_dev, int32_t sample, void *stream);

/*
 * Training the policy on the GPU: the PPO learner of the reference's training script (RLlib PPO, ray 0.x).
 * Parameters travel as one flat FP32 device vector, w1 | b1 | w2 | b2 | w3 | b3, each row-major as in
 * PaintrlPolicyConfig; paintrl_policy_num_params gives its length (PAINTRL_E_INVALID for shapes the kernels do not take).
 * paintrl_policy_set_params packs such a vector into the policy engine's device weights on `stream`, at the addresses
 * the engine already uses: a CUDA graph captured around paintrl_policy_act samples with the new weights on its next replay.
 */
int32_t paintrl_policy_num_params(int32_t obs_dim, int32_t n_out);
int paintrl_policy_set_params(PaintrlPolicyHandle h, const float *params_dev, void *stream);

typedef struct PaintrlPpoConfig {
    int32_t abi_version;
    int32_t obs_dim, n_out, discrete;   /* as PaintrlPolicyConfig */
    int32_t max_minibatch;              /* largest n of paintrl_ppo_grad (sizes the partial-gradient workspace) */
    float clip_param;                   /* surrogate clip epsilon (RLlib default 0.3) */
    float vf_clip_param;                /* value clip (RLlib default 10) */
    float vf_loss_coeff;                /* RLlib default 1 */
    float entropy_coeff;                /* RLlib default 0 */
} PaintrlPpoConfig;
typedef struct PaintrlPpoEngine *PaintrlPpoHandle;

int paintrl_ppo_create(const PaintrlPpoConfig *cfg, int32_t device, PaintrlPpoHandle *out);
void paintrl_ppo_destroy(PaintrlPpoHandle h);
/* The loss gradient of one minibatch, asynchronous on `stream` (two launches, no synchronisation).  Row k of the
 * minibatch is row idx_dev[k] of the flattened fragment (idx int32 [n]; the indices are the caller's contract):
 * obs float64 [rows][obs_dim], actions int64 [rows] (discrete) or float64 [rows][n_out], logp_old / value_old / adv /
 * vtarg float32 [rows], logits_old float32 [rows][n_out + 1] (the act kernel's logits output).  Loss, averaged over the
 * n rows: -min(A r, A clip(r, 1 +- clip)) + kl_coeff KL(old || new) + vf_loss_coeff max((v - R)^2, (v_old + clip(v -
 * v_old, +-vf_clip) - R)^2) - entropy_coeff H.  Writes grad_dev float32 [num_params] (overwritten, not accumulated) and
 * stats_dev float32 [6]: policy loss, value loss, KL, entropy, clip fraction, mean ratio.  Bitwise reproducible. */
int paintrl_ppo_grad(PaintrlPpoHandle h, const float *params_dev, const int32_t *idx_dev, int32_t n, const double *obs_dev,
                     const void *actions_dev, const float *logp_old_dev, const float *value_old_dev, const float *logits_old_dev,
                     const float *adv_dev, const float *vtarg_dev, float kl_coeff, float *grad_dev, float *stats_dev, void *stream);
/* The learner kernel's forward pass alone: out_dev float32 [n][n_out + 1], logits | means, then the value -- equal to
 * paintrl_policy_act's logits output for the same weights, bit for bit. */
int paintrl_ppo_forward(PaintrlPpoHandle h, const float *params_dev, const int32_t *idx_dev, int32_t n, const double *obs_dev,
                        float *out_dev, void *stream);
/* Adam (torch.optim.Adam's arithmetic, bias-corrected, no gradient clipping) over n_params FP32 values; m / v are the
 * caller's moment buffers (zero before step 1); step counts from 1. */
int paintrl_adam_step(float *params_dev, const float *grad_dev, float *m_dev, float *v_dev, int32_t n_params, float lr,
                      float beta1, float beta2, float eps, int32_t step, void *stream);

/*
 * PPO with a learned log-std (RLlib's DiagGaussian for a Box action space) on a continuous engine with n_out = 2 A:
 * head column o is the mean mu_o and column A + o is log sigma_o of action dimension o < A, then the value.  Both calls
 * return PAINTRL_E_INVALID for a discrete handle or an odd n_out.
 *
 * paintrl_policy_act_diag_gaussian: a_o = fl(fl(sigma_o z_o) + mu_o), sigma_o = expf(log sigma_o), z_o the Box-Muller
 * draw paintrl_policy_act's continuous head uses (pol_uniform k = 2o, 2o + 1); no tanh and no clamp (the environment
 * clips).  actions_dev float64 [batch, A] (FP32 values), logp_dev float32 [batch] = log N(a; mu, diag sigma^2) computed
 * from those FP32 actions by the function the learner also uses, value_dev float32 [batch], logits_dev float32
 * [batch, n_out + 1] or NULL.  Always samples; the bootstrap value comes from paintrl_policy_act with sample = 0.
 *
 * paintrl_ppo_grad_diag_gaussian: paintrl_ppo_grad's arguments and loss on this distribution, actions float64 [rows][A]:
 * KL(old || new) = sum_o (log sigma_o - log sigma_old,o + (sigma_old,o^2 + (mu_old,o - mu_o)^2) / (2 sigma_o^2) - 1/2)
 * and H = sum_o (log sigma_o + log(2 pi e) / 2).  The same six statistics; the first minibatch after a collection has
 * ratios of exactly 1.
 */
int paintrl_policy_act_diag_gaussian(PaintrlPolicyHandle h, const double *obs_dev, int32_t batch, double *actions_dev, float *logp_dev,
                                     float *value_dev, float *logits_dev, void *stream);
int paintrl_ppo_grad_diag_gaussian(PaintrlPpoHandle h, const float *params_dev, const int32_t *idx_dev, int32_t n, const double *obs_dev,
                                   const void *actions_dev, const float *logp_old_dev, const float *value_old_dev,
                                   const float *logits_old_dev, const float *adv_dev, const float *vtarg_dev, float kl_coeff,
                                   float *grad_dev, float *stats_dev, void *stream);

/*
 * Double DQN with a dueling head on the same network (RLlib DQN's dueling combination, without its extra hidden layer
 * per stream): the n_out head outputs are the advantages A, the value column is V, and Q(s, a) = V + A_a - mean_o A_o.
 * "Greedy" is the first maximum of Q (the lowest action index on ties), in the act kernel and in the target alike.
 *
 * paintrl_policy_act_epsilon: epsilon-greedy actions of a discrete policy engine (PAINTRL_E_INVALID for a continuous
 * one).  epsilon_dev is one float32 in device memory, read by the kernel on every launch, so a CUDA graph captured
 * around this call follows an exploration schedule written into it between replays.  Per environment and launch the
 * engine's counter ctr gives the draws pol_uniform(seed, env, ctr, k) of paintrl_policy.cuh: k = 0 explores when it is
 * < epsilon, k = 1 then picks the action min(floor(u * n_out), n_out - 1); the counter advances by one either way.
 * value_dev float32 [batch]; logits_dev float32 [batch, n_out + 1] or NULL, the same bits as paintrl_policy_act's.
 */
int paintrl_policy_act_epsilon(PaintrlPolicyHandle h, const double *obs_dev, int32_t batch, void *actions_dev, float *value_dev,
                               float *logits_dev, const float *epsilon_dev, void *stream);

typedef struct PaintrlDqnConfig {
    int32_t abi_version;
    int32_t obs_dim, n_out;             /* as PaintrlPolicyConfig (discrete actions only) */
    int32_t max_minibatch;              /* largest n of paintrl_dqn_grad (sizes the partial-gradient and s' workspaces) */
    float gamma;                        /* discount, in (0, 1] */
} PaintrlDqnConfig;
typedef struct PaintrlDqnEngine *PaintrlDqnHandle;

int paintrl_dqn_create(const PaintrlDqnConfig *cfg, int32_t device, PaintrlDqnHandle *out);
void paintrl_dqn_destroy(PaintrlDqnHandle h);
/* The double-DQN loss gradient of one minibatch, asynchronous on `stream` (four launches, no synchronisation).  Row k
 * of the minibatch is row idx_dev[k] of the transition arrays (idx int32 [n]): obs / next_obs float64 [rows][obs_dim],
 * actions int64 [rows], reward float32 [rows], done uint8 [rows].  y = r + gamma (1 - done) Q_target(s', argmax_o
 * Q_online(s', o)) with Q_online from params_dev and Q_target from target_params_dev; loss = mean Huber(Q(s, a) - y),
 * delta 1.  Writes grad_dev float32 [num_params] (overwritten) and stats_dev float32 [4]: mean Huber loss, mean |td|,
 * mean Q(s, a), mean y.  Bitwise reproducible. */
int paintrl_dqn_grad(PaintrlDqnHandle h, const float *params_dev, const float *target_params_dev, const int32_t *idx_dev, int32_t n,
                     const double *obs_dev, const int64_t *actions_dev, const float *reward_dev, const double *next_obs_dev,
                     const uint8_t *done_dev, float *grad_dev, float *stats_dev, void *stream);
/* paintrl_dqn_grad with a per-sample importance weight (prioritized replay): weight_dev float32 [n] and td_out_dev
 * float32 [n], both in minibatch order.  loss = mean w_k Huber(td_k), its gradient per sample
 * (clamp(td, -1, 1) * w) / n, so all-ones weights give paintrl_dqn_grad's gradient and statistics bit for bit.  td_out_dev
 * receives td_k = Q(s, a) - y for the priority update; stats_dev float32 [5]: mean weighted Huber loss, mean |td|,
 * mean Q(s, a), mean y, mean weight.  Bitwise reproducible. */
int paintrl_dqn_grad_weighted(PaintrlDqnHandle h, const float *params_dev, const float *target_params_dev, const int32_t *idx_dev,
                              int32_t n, const double *obs_dev, const int64_t *actions_dev, const float *reward_dev,
                              const double *next_obs_dev, const uint8_t *done_dev, const float *weight_dev, float *td_out_dev,
                              float *grad_dev, float *stats_dev, void *stream);

/*
 * Prioritized replay (RLlib's PrioritizedReplayBuffer) over a ring of `capacity` rows: a sum tree and a min tree, both
 * float64 [2 * tree_leaves] in device memory and owned by the caller.  tree_leaves is a power of two >= capacity; node 1
 * is the root, node i has children 2i and 2i + 1, and row r is leaf tree_leaves + r.  A filled leaf holds p^alpha in
 * both trees; the caller initialises every leaf and node to 0 in the sum tree and +inf in the min tree.  After every
 * leaf write the calls below rebuild each internal node from its two children (sum: left + right, min: fmin), so the
 * trees are a pure function of their leaves.  max_priority_dev is one float64 in device memory (RLlib starts it at 1).
 * All three are asynchronous on `stream`.
 *
 * paintrl_prio_fill: rows [start, start + count) mod capacity get max_priority^alpha, as new transitions do in RLlib.
 * paintrl_prio_update: for k < n, row idx_dev[k] (int32, in [0, capacity)) gets (|td_k| + eps)^alpha from the float32
 *   td_dev [n] (paintrl_dqn_grad_weighted's td_out), computed in float64, and max_priority rises to max(|td_k| + eps).
 *   Duplicate rows must carry identical td (as one minibatch's do).
 * paintrl_prio_sample: n rows, row k from the float64 uniform u_dev[k] in [0, 1): the leaf where the prefix sum of the
 *   sum tree passes u * root, never a row of priority 0 (so never one at or beyond size, the filled rows [0, size)).
 *   idx_out_dev int32 [n]; weight_out_dev float32 [n] = (p_i / p_min)^(-beta) in float64, p_min the min-tree root: RLlib's
 *   (N P(i))^-beta / max_j (N P(j))^-beta, at most 1.
 * Requirements: alpha finite and >= 0, eps finite and > 0, beta in [0, 1], size in [1, capacity], count in [1, capacity],
 * start in [0, capacity), n in [1, 2^24].
 */
int paintrl_prio_fill(double *sum_tree_dev, double *min_tree_dev, int32_t tree_leaves, int32_t capacity, int32_t start, int32_t count,
                      const double *max_priority_dev, double alpha, void *stream);
int paintrl_prio_update(double *sum_tree_dev, double *min_tree_dev, int32_t tree_leaves, int32_t capacity, const int32_t *idx_dev,
                        const float *td_dev, int32_t n, double *max_priority_dev, double alpha, double eps, void *stream);
int paintrl_prio_sample(const double *sum_tree_dev, const double *min_tree_dev, int32_t tree_leaves, int32_t capacity, int32_t size,
                        const double *u_dev, int32_t n, double beta, int32_t *idx_out_dev, float *weight_out_dev, void *stream);

/* Global-norm clipping of n float32 values in place (torch.nn.utils.clip_grad_norm_'s rule: scaled by
 * max_norm / (norm + 1e-6) only when the L2 norm exceeds max_norm, untouched otherwise).  norm_out_dev float32 [1]
 * receives the norm before clipping.  Fixed-order reduction: the same norm on every run. */
int paintrl_clip_grad_norm(float *grad_dev, int32_t n, float max_norm, float *norm_out_dev, void *stream);

const char *paintrl_last_error(void);
int32_t paintrl_abi_version(void);

#ifdef __cplusplus
}
#endif
#endif /* PAINTRL_H_ */
