/*
 * mate_b200.h -- C ABI of the B200-native batched MultiAgentTracking simulator.
 *
 * The reference (XuehaiPan/mate) is pure Python and has NO native/FFI layer; its boundary
 * for the step path is the Python class ``mate.environment.MultiAgentTracking``
 * (mate/environment.py:288) reached through ``mate.make`` (mate/__init__.py:24-43).  This
 * header is the C-ABI a binding for that class calls instead of the per-entity Python
 * loops.  Each entry point cites the reference method it replaces.  The Python binding
 * (ctypes) that mirrors the reference class on top of it is ``mate_b200/environment.py``;
 * INTEGRATION.md shows the stub a reference maintainer would add.
 *
 * Conventions
 *   - plain C types only; no torch / CUDA types in signatures (streams are passed as
 *     ``void*`` holding a ``cudaStream_t``; NULL = legacy default stream);
 *   - every function returns 0 on success or a negative MateStatus; the message is
 *     available from mate_b200_last_error() (thread-local);
 *   - "dev" pointers are device pointers owned by the caller (e.g. PyTorch tensors) on the
 *     device the handle was created for; "host" pointers are ordinary host memory;
 *   - batched I/O is row-major [B, N, D] float32 in the reference's feature order
 *     (mate/environment.py:908-983, mate/constants.py:267-300); the observation rows
 *     (the ``float* cam_obs / tgt_obs`` arguments) may instead be float16 per handle, see
 *     mate_b200_set_observation_format: the arguments then address buffers of that type;
 *   - a handle is not re-entrant; different handles are independent (one per GPU);
 *   - step/reset/observe/save_state/load_state enqueue work on the given stream and never synchronise the host.
 */
#ifndef MATE_B200_H_
#define MATE_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MATE_B200_ABI_VERSION 2
#define MATE_NUM_WAREHOUSES 4   /* mate/constants.py:70-75 */
#define MATE_MAX_CAMERAS 32
#define MATE_MAX_TARGETS 32
#define MATE_MAX_OBSTACLES 64

typedef enum MateStatus {
    MATE_OK = 0,
    MATE_EINVAL = -1,   /* bad argument / unsupported configuration */
    MATE_ECUDA = -2,    /* CUDA runtime error (message has the cudaError string) */
    MATE_ENOMEM = -3,   /* allocation failure */
    MATE_ESTATE = -4    /* handle in the wrong state for this call */
} MateStatus;

/* Validated configuration, flattened from the YAML/dict the reference's read_config()
 * produces (mate/environment.py:113-269).  Per-entity parameters are common to all
 * entities of a kind, exactly as in the reference's config schema. */
typedef struct MateConfig {
    int32_t num_cameras;                /* Nc >= 0 */
    int32_t num_targets;                /* Nt >= 1 */
    int32_t num_obstacles;              /* No >= 0 */
    int32_t max_episode_steps;          /* environment.py:199-203 */
    int32_t num_cargoes_per_target;     /* environment.py:223-229 (>= 4) */
    int32_t num_high_capacity_targets;  /* int(Nt * high_capacity_target_split), environment.py:1527-1535 */
    int32_t targets_start_with_cargoes; /* bool */
    int32_t shuffle_entities;           /* bool */
    int32_t reward_sparse;              /* reward_type == 'sparse' */
    int32_t reserved0;
    double bounty_factor;
    double camera_radius;
    double camera_min_viewing_angle;
    double camera_max_sight_range;
    double camera_rotation_step;
    double camera_zooming_step;
    double target_step_size;
    double target_sight_range;
    double obstacle_transmittance;
    double obstacle_radius_low;   /* radius_random_range (low == high for a fixed radius) */
    double obstacle_radius_high;
    /* host arrays [N][4] = (x_low, x_high, y_low, y_high); a fixed location has low == high */
    const double* camera_location_ranges;
    const double* target_location_ranges;
    const double* obstacle_location_ranges;
} MateConfig;

/* Host-side view of the simulator state for get/set (checkpoint, parity harness).
 * These are the quantities SURVEY.md section 8a lists as carried between steps; the
 * reference has state() (environment.py:894-906) but no set_state.  All arrays are
 * host pointers, batched row-major; any pointer may be NULL to skip that field. */
typedef struct MateStateView {
    double* cam_xy;          /* [B, Nc, 2]  Camera.location                      */
    double* cam_phi;         /* [B, Nc]     Camera.orientation, degrees [-180,180) */
    double* cam_theta;       /* [B, Nc]     Camera.viewing_angle, degrees         */
    double* tgt_xy;          /* [B, Nt, 2]  Target.location                       */
    double* obs_xyr;         /* [B, No, 3]  Obstacle.location, radius             */
    int32_t* tgt_capacity;   /* [B, Nt]     1 or 2 (step_size = cfg step / capacity) */
    int32_t* tgt_goal;       /* [B, Nt]     target_goals, -1 = no cargo           */
    int32_t* tgt_weight;     /* [B, Nt]     target_goal_bits[t, goal] (cargo weight) */
    int32_t* tgt_bounty;     /* [B, Nt]     bounties                              */
    int32_t* tgt_empty_bits; /* [B, Nt]     bit w = Target.empty_bits[w]          */
    int32_t* remaining;      /* [B, 4, 4]   remaining_cargoes                     */
    int32_t* awaiting;       /* [B, 4]      awaiting_cargo_counts                 */
    int32_t* num_delivered;  /* [B]         num_delivered_cargoes                 */
    int32_t* episode_step;   /* [B]                                               */
    int32_t* episode_id;     /* [B]         counter-based RNG episode counter     */
    double* episode_reward;  /* [B, 2]      target_team_episode_reward, delayed_* */
} MateStateView;

/* Optional per-step auxiliary outputs (all dev pointers; NULL = not wanted).
 * These are the reference's public per-step attributes / info-dict entries
 * (environment.py:634-661) as tensors. */
typedef struct MateStepAux {
    uint8_t* mask_ct;        /* [B, Nc, Nt] camera_target_view_mask   */
    uint8_t* mask_cc;        /* [B, Nc, Nc] camera_camera_view_mask   */
    uint8_t* mask_co;        /* [B, Nc, No] camera_obstacle_view_mask */
    uint8_t* mask_tc;        /* [B, Nt, Nc] target_camera_view_mask   */
    uint8_t* mask_to;        /* [B, Nt, No] target_obstacle_view_mask */
    uint8_t* mask_tt;        /* [B, Nt, Nt] target_target_view_mask   */
    float* coverage;         /* [B, 3] coverage_rate, real_coverage_rate, mean_transport_rate */
    int32_t* num_delivered;  /* [B]                                                          */
    uint8_t* target_dones;   /* [B, Nt] environment.py:1320-1322                             */
    uint8_t* is_colliding;   /* [B, Nt] Target.is_colliding, entities.py:668                 */
    float* warehouse_dist;   /* [B, Nt, 4] target_warehouse_distances                        */
    int32_t* episode_step;   /* [B] episode_step after this step (before auto-reset)         */
    int32_t* tgt_goal;       /* [B, Nt] target_goals (-1 = none), environment.py:1271-1324   */
    uint8_t* tgt_empty_bits; /* [B, Nt] Target.empty_bits as bit set (bit w = warehouse w)   */
} MateStepAux;

/* Parity mode: recorded outcomes of the reference's two stochastic step-path draws
 * (dev pointers).  NULL members / NULL struct => the counter-based Philox stream is used. */
typedef struct MateReplay {
    const uint8_t* transmit;   /* [B, Nc, Nt] outcome of binomial(1, transmittance), entities.py:503 */
    const int8_t* goal_choice; /* [B, Nt] outcome of np_random.choice(...), environment.py:1303; -1 = none */
} MateReplay;

typedef struct MateSim MateSim;

/* Flags for mate_b200_step. */
#define MATE_STEP_AUTO_RESET 1u /* reset finished episodes inside the call; returned obs are the new episode's */
/* mate_b200_step_host only: the caller passes the same cam_obs / tgt_obs buffers as in its previous mate_b200_step_host
 * call on this handle and has not written to them since.  The library then sends and rewrites only the 64-byte groups of
 * the rows that differ from the previous call's rows (which it keeps on the device); the buffers hold the complete rows of
 * this step either way.  Without the flag, or with other buffers than the previous call's, every byte of the rows is
 * written. */
#define MATE_STEP_HOST_ROWS_KEPT 2u

const char* mate_b200_last_error(void);
int mate_b200_abi_version(void);

/* MultiAgentTracking.__init__ (environment.py:330-562): allocate the struct-of-arrays
 * state for num_envs environments on CUDA device `device`.  env_index_base is the global
 * index of local env 0 (multi-GPU sharding: RNG streams are keyed on the global index so
 * results do not depend on the number of GPUs). */
int mate_b200_create(const MateConfig* cfg, int32_t num_envs, int32_t device,
                     int64_t env_index_base, MateSim** out);
int mate_b200_destroy(MateSim* sim);

/* Observation row widths: Dc, Dt (constants.py:267-300). */
int mate_b200_obs_dims(const MateSim* sim, int32_t* cam_dim, int32_t* tgt_dim);

/* Element type of the observation rows this handle writes: MATE_OBS_FORMAT_F32 (the default) or MATE_OBS_FORMAT_F16.
 * The float16 rows are the float32 rows of the same call rounded once to nearest even; the simulation, the masks, the
 * registered observation wrappers, rewards, done, auxiliary outputs and actions are unchanged (float32).  After
 * MATE_OBS_FORMAT_F16 the `float* cam_obs / tgt_obs` arguments of mate_b200_reset, _step, _observe and _step_host
 * address float16 buffers of the same shapes (cast the pointers), and mate_b200_transform_observations is refused
 * (register the wrappers with mate_b200_set_observation_ops instead).  Allowed only before the handle's first reset,
 * step, step_host or observe (MATE_ESTATE afterwards); an unknown code is MATE_EINVAL. */
#define MATE_OBS_FORMAT_F32 0
#define MATE_OBS_FORMAT_F16 1
int mate_b200_set_observation_format(MateSim* sim, int32_t format);

/* MultiAgentTracking.reset (environment.py:679-834) for the envs with env_mask[b] != 0
 * (dev, NULL = all); Philox streams keyed on (seed, global env index, episode id).
 * Writes the first joint observation of the reset envs (other rows are rewritten with
 * their current observation); cam_obs / tgt_obs in the handle's observation format.  Either may be NULL: that
 * team's rows are then neither composed nor written (one team learning against built-in agents). */
int mate_b200_reset(MateSim* sim, const uint8_t* env_mask, uint64_t seed,
                    float* cam_obs, float* tgt_obs, void* stream);

/* MultiAgentTracking.seed / reset(seed=...) (environment.py:700-701, 1203-1227): an explicit seed makes the
 * following resets reproducible.  Stores `seed` as the key of the handle's Philox streams and rewinds the
 * episode counter (the RNG counter field mate_b200_reset advances) of the envs with env_mask[b] != 0 (dev,
 * NULL = all), so that seed(s) followed by reset gives the same initial states every time.  Without this call
 * successive resets draw independent episodes, like the reference's reset() without a seed. */
int mate_b200_seed(MateSim* sim, const uint8_t* env_mask, uint64_t seed, void* stream);

/* MultiAgentTracking.step (environment.py:590-676) for all envs: _simulate,
 * _update_view, _assign_goals, joint_observation, reward/done.
 *   cam_act [B,Nc,2], tgt_act [B,Nt,2] float32 dev (finite);
 *   cam_obs [B,Nc,Dc], tgt_obs [B,Nt,Dt] dev, float32 or float16 (mate_b200_set_observation_format); either may be
 *     NULL: that team's rows are neither composed nor written, and everything else is what a call with both
 *     buffers computes;
 *   rewards [B,2] float32 dev = (camera_team_reward, target_team_reward);
 *   done [B] uint8 dev. */
int mate_b200_step(MateSim* sim, const float* cam_act, const float* tgt_act,
                   float* cam_obs, float* tgt_obs, float* rewards, uint8_t* done,
                   const MateStepAux* aux, const MateReplay* replay, uint32_t flags,
                   void* stream);

/* joint_observation() of the current state without stepping (_update_view +
 * joint_observation, environment.py:1356-1388, 908-983); used after set_state.  cam_obs / tgt_obs in the
 * handle's observation format; either may be NULL (that team's rows are not written). */
int mate_b200_observe(MateSim* sim, float* cam_obs, float* tgt_obs,
                      const MateStepAux* aux, const MateReplay* replay, void* stream);

/* Same as mate_b200_step but with HOST buffers (pinned or pageable): actions are copied
 * host->device, results device->host, chunked over internal streams so that copies
 * overlap the kernel.  Returns after the results are in the host buffers.
 * Ordering: the chunks run on internal non-blocking streams that first wait for everything
 * already queued on the legacy default stream (and on blocking streams, e.g. torch's default
 * stream); a caller that queued reset / step / set_state work on a NON-BLOCKING stream of its
 * own synchronises that stream before this call.  Auto-resets adopt the prepared next
 * episodes exactly like mate_b200_step (the refill runs on the side stream).
 * The observation rows reach cam_obs / tgt_obs as a dense copy or, depending on the host threads the process has
 * (INTEGRATION.md), compacted: non-zero 16-byte chunks only, or -- with MATE_STEP_HOST_ROWS_KEPT -- only the 64-byte
 * groups that differ from the previous call's rows; host threads of the library put them in place before the call
 * returns.  The buffers hold the same bytes in every case.  Row buffers must be 4-byte aligned (16-byte aligned for full
 * speed) and of the handle's observation format (float16 rows halve the bytes on the link).  cam_obs or tgt_obs may be
 * NULL: that team's rows are not composed and nothing of them crosses the link.  MATE_STEP_HOST_ROWS_KEPT needs the same
 * pointers, NULL included, as the previous call: a call that switches a team between NULL and a buffer writes every
 * byte of the rows it is given. */
int mate_b200_step_host(MateSim* sim, const float* cam_act, const float* tgt_act,
                        float* cam_obs, float* tgt_obs, float* rewards, uint8_t* done,
                        uint32_t flags);

/* State view / injection (host arrays; synchronises the device).  A view, not a complete checkpoint: it leaves out the
 * running coverage sum, the line-of-sight cache, the Philox seed and the episode statistics; use mate_b200_save_state
 * to save and restore a batch exactly.  A set_state refused for a value out of range (MATE_EINVAL) leaves the handle
 * unchanged. */
int mate_b200_get_state(MateSim* sim, MateStateView* view);
int mate_b200_set_state(MateSim* sim, const MateStateView* view);

/* Device-side state snapshots: the complete per-environment state of a batch, saved to and loaded from a device buffer
 * without leaving the device, for exact resume (checkpoints) and for branching (environment d takes the state of
 * environment s).  The payload is a caller-owned device buffer on the handle's device, 16-byte aligned, of
 * mate_b200_snapshot_bytes(count) bytes; its layout is private to the library and tagged with MATE_SNAPSHOT_VERSION.
 * The library allocates nothing for snapshots.  Both calls only enqueue work on `stream`, like mate_b200_step.
 *
 * What a snapshot holds: every live state array of the environments (entities, target and cargo integers, episode
 * step / id / rewards / coverage sum, the per-episode line-of-sight cache), copied verbatim, plus the handle's 16
 * episode-statistics accumulators.  Observation rows and MateStepAux outputs are not saved: mate_b200_observe
 * recomputes them.
 *
 * Random draws after a load: a reset is a function of (seed, global environment index, episode id) and the step's
 * draws (transmission, goal choice) of (seed, global environment index, episode id, episode step).  An environment
 * restored at its own global index under the saving handle's seed therefore replays exactly.  A clone at another index
 * shares the state but draws its own outcomes from its next step on, unless the step is given a MateReplay. */
#define MATE_SNAPSHOT_VERSION 1
typedef struct MateSnapshotInfo {      /* host-side header of a device payload */
    int32_t version;                   /* MATE_SNAPSHOT_VERSION */
    int32_t num_cameras, num_targets, num_obstacles;
    int32_t count;                     /* environments in the payload */
    int32_t reserved;
    uint64_t config_hash;              /* fingerprint of the MateConfig the saving handle was created with: 64-bit FNV-1a
                                          over its scalar fields (reserved0 excepted) and the values of its three range
                                          arrays, in declaration order */
    uint64_t seed;                     /* the saving handle's Philox key */
    uint64_t payload_bytes;
} MateSnapshotInfo;

/* Bytes of the payload of a snapshot of `count` (> 0) environments of this handle's shape. */
int mate_b200_snapshot_bytes(const MateSim* sim, int32_t count, uint64_t* bytes);

/* Save: payload entry i gets the state of environment env[i] (dev int32 [count]; NULL = every environment, which
 * requires count == num_envs).  An entry of env outside [0, num_envs) leaves payload entry i unwritten.  Fills *info
 * on the host without reading device memory (it never synchronises). */
int mate_b200_save_state(MateSim* sim, const int32_t* env, int32_t count, void* payload,
                         MateSnapshotInfo* info, void* stream);

/* Load: environment d takes payload entry src[d] (dev int32 [num_envs]; NULL = entry d for every d, which requires
 * info->count == num_envs); a negative or out-of-range entry keeps environment d as it is.  Only the mapped environments
 * change; the handle's seed and statistics stay.  With MATE_LOAD_STATE_RESUME (requires src == NULL) the handle also
 * takes the saving handle's seed (info->seed) and statistics, so that the batch continues bit for bit.
 * The saving and the loading handle need the same (Nc, Nt, No) and configuration (config_hash); their observation
 * format, env_index_base and num_envs may differ.  A load is allowed before the first reset and does not fix the
 * observation format.  The prepared next episodes of the loaded environments are discarded and prepared again (on
 * the side stream, ordered after the load); the load waits for a prepare still running with an event, not by
 * synchronising the host.  MATE_EINVAL, with the handle unchanged, for another version, shape or configuration, a
 * count <= 0, a NULL map with a count other than num_envs, RESUME with a map, or a misaligned payload. */
#define MATE_LOAD_STATE_RESUME 1u
int mate_b200_load_state(MateSim* sim, const void* payload, const MateSnapshotInfo* info,
                         const int32_t* src, uint32_t flags, void* stream);

/* Episode statistics accumulated on device since the last call with reset_after != 0:
 * out[0]=episodes finished, [1]=sum return (target team), [2]=sum length,
 * [3]=sum delivered cargoes, [4]=sum of per-episode mean coverage, [5]=env-steps,
 * [6]=auto-resets served from the prepared next-episode state, [7]=auto-resets computed in place,
 * [8..15] reserved (0).  `out16` is a dev pointer to 16 floats; the optional multi-GPU
 * all-reduce of this vector is done by the caller (torch.distributed / NCCL). */
int mate_b200_episode_stats(MateSim* sim, float* out16, int32_t reset_after, void* stream);

/* The reference's observation wrappers applied IN PLACE to the joint observations of the current state, in
 * the given order, in one pass over the tensors (SURVEY.md section 8f, N1):
 *   MATE_OBS_ENHANCED_CAMERA / _TARGET  EnhancedObservation.observation, mate/wrappers/enhanced_observation.py:72-123
 *   MATE_OBS_SHARED_CAMERA / _TARGET    SharedFieldOfView.observation,   mate/wrappers/shared_field_of_view.py:74-145
 *   MATE_OBS_RELATIVE                   convert_coordinates,  mate/agents/utils.py:40-94  (RelativeCoordinates)
 *   MATE_OBS_RESCALED                   normalize_observation, mate/agents/utils.py:97-127 (RescaledObservation)
 * `ops` is a HOST array of num_ops <= MATE_MAX_OBS_OPS codes, in the order the reference's wrappers admit:
 *   (ENHANCED_* | SHARED_*)*  RELATIVE?  RESCALED?
 * i.e. no mask code after RELATIVE or RESCALED, neither of those twice, and no RELATIVE after RESCALED; any other
 * sequence is MATE_EINVAL and leaves the registered wrappers as they were.  cam_affine [Dc][2] / tgt_affine [Dt][2] are dev
 * arrays of (scale, shift) per observation column, needed (non-NULL) only with MATE_OBS_RESCALED.  cam_obs /
 * tgt_obs must hold the observations the last step/reset/observe call wrote for this handle.  float32 handles only
 * (MATE_EINVAL after MATE_OBS_FORMAT_F16). */
#define MATE_OBS_ENHANCED_CAMERA 1
#define MATE_OBS_ENHANCED_TARGET 2
#define MATE_OBS_SHARED_CAMERA 3
#define MATE_OBS_SHARED_TARGET 4
#define MATE_OBS_RELATIVE 5
#define MATE_OBS_RESCALED 6
#define MATE_MAX_OBS_OPS 8   /* codes per stack, ordered (ENHANCED_* | SHARED_*)* RELATIVE? RESCALED? (above) */
int mate_b200_transform_observations(MateSim* sim, float* cam_obs, float* tgt_obs, const int32_t* ops,
                                     int32_t num_ops, const float* cam_affine, const float* tgt_affine,
                                     void* stream);

/* The same wrappers REGISTERED with the simulator: from now on every mate_b200_reset / _step / _step_host / _observe
 * applies them to an environment's rows while they are still in shared memory (the packer of the step kernel), i.e.
 * without the extra read + write pass over the observation tensors mate_b200_transform_observations costs.
 * num_ops = 0 unregisters.  The same order rule holds: a refused sequence leaves the registered wrappers in effect.
 * The affine tables must stay valid until they are replaced. */
int mate_b200_set_observation_ops(MateSim* sim, const int32_t* ops, int32_t num_ops,
                                  const float* cam_affine, const float* tgt_affine);

/* Camera.sight_range_at (mate/entities.py:507-511): value of the sampled field-of-view polyline of camera
 * camera[i] of environment env[i] at bearing angle_deg[i] (any angle; normalised like the reference), for n
 * queries.  The polyline (Camera.add_obstacles, entities.py:362-479) is never materialised: this evaluates the
 * same routine the step kernel uses for its occlusion tests, which makes the routine testable against the
 * reference's tables directly.  All pointers are dev pointers. */
int mate_b200_fov_range(MateSim* sim, const int32_t* env, const int32_t* camera, const double* angle_deg,
                        double* out, int64_t n, void* stream);

/* rgb_array frames of chosen environments, drawn from the live state by a CUDA kernel (DESIGN.md section 7k).
 * out: dev uint8 [count][size][size][3]; frame i is environment env[i] (dev int32 [count]; NULL = every environment,
 * which requires count == num_envs).  An entry of env outside [0, num_envs) leaves frame i unwritten.  The call only
 * enqueues work on `stream`: it never synchronises, changes nothing in the handle and reads the state as it is, like
 * mate_b200_fov_range.  MATE_EINVAL, nothing launched, for a NULL sim or out, count <= 0, a NULL env with count !=
 * num_envs, or a size outside [MATE_RENDER_MIN_SIZE, MATE_RENDER_MAX_SIZE].
 *
 * The picture.  Row 0 is the top (y = +V), column 0 the left (x = -V), V = MATE_RENDER_HALF_EXTENT.  Pixel (i, j) is
 * decided at its centre x_j = ((2j + 1 - S) V) / S, y_i = ((S - 2i - 1) V) / S (fp64: one exact product, one correctly
 * rounded division); the pixel pitch is p = 2V / S.  Colours are 0xRRGGBB, stored as the bytes R, G, B.  Layers, in order:
 *   1. MATE_RENDER_TERRAIN where |x| <= 1000 and |y| <= 1000, else MATE_RENDER_OUTSIDE;
 *   2. warehouse w (centre MATE_RENDER_WAREHOUSE_CENTER * (+-1, +-1) in the order (+,+), (-,+), (-,-), (+,-)) where
 *      max(|x - wx|, |y - wy|) <= MATE_RENDER_WAREHOUSE_HALF_SIZE, colour MATE_RENDER_WAREHOUSE_<w>;
 *   3. with k the number of cameras that would see a target at the pixel centre (Camera.perceive with a transmission draw
 *      of 0: the step's range + sector test and its occlusion test dist <= sight_range_at(bearing) * (1 + 1e-6)),
 *      MATE_RENDER_FOV blended k times: dst = (dst * (255 - a) + src * a + 127) / 255 per channel, a = MATE_RENDER_FOV_ALPHA;
 *   4. MATE_RENDER_OBSTACLE where dx^2 + dy^2 <= r^2;
 *   5. MATE_RENDER_CAMERA where dx^2 + dy^2 <= camera_radius^2;
 *   6. targets in index order, with r_in = max(MATE_RENDER_TARGET_INNER, MATE_RENDER_TARGET_INNER_PITCH * p) and r_out =
 *      max(MATE_RENDER_TARGET_OUTER, MATE_RENDER_TARGET_OUTER_PITCH * p): d^2 <= r_in^2 gets the colour of the goal
 *      warehouse if the target is loaded (goal >= 0 and weight > 0), else MATE_RENDER_TARGET_EMPTY; r_in^2 < d^2 <= r_out^2
 *      gets MATE_RENDER_TRACKED if some camera sees the target's location by the predicate of layer 3.
 * Layers 2, 4, 5 and 6 compute in fp64 without fused multiply-add.  A frame is a function of its environment's state. */
#define MATE_RENDER_MIN_SIZE 16
#define MATE_RENDER_MAX_SIZE 4096
#define MATE_RENDER_HALF_EXTENT 1050.0          /* 1.05 * terrain size */
#define MATE_RENDER_WAREHOUSE_CENTER 925.0
#define MATE_RENDER_WAREHOUSE_HALF_SIZE 75.0
#define MATE_RENDER_FOV_ALPHA 64
#define MATE_RENDER_TARGET_INNER 12.0
#define MATE_RENDER_TARGET_INNER_PITCH 1.25
#define MATE_RENDER_TARGET_OUTER 22.0
#define MATE_RENDER_TARGET_OUTER_PITCH 2.25
#define MATE_RENDER_TERRAIN 0xF4F4F4u
#define MATE_RENDER_OUTSIDE 0x404040u
#define MATE_RENDER_WAREHOUSE_0 0xE69F00u
#define MATE_RENDER_WAREHOUSE_1 0x56B4E9u
#define MATE_RENDER_WAREHOUSE_2 0x009E73u
#define MATE_RENDER_WAREHOUSE_3 0xCC79A7u
#define MATE_RENDER_FOV 0x0072B2u
#define MATE_RENDER_OBSTACLE 0x808080u
#define MATE_RENDER_CAMERA 0x003E7Du
#define MATE_RENDER_TRACKED 0xD55E00u
#define MATE_RENDER_TARGET_EMPTY 0x202020u
int mate_b200_render(MateSim* sim, const int32_t* env, int32_t count, int32_t size, uint8_t* out, void* stream);

/* Per-agent terms of the reference's auxiliary-reward and training-information wrappers (SURVEY.md section
 * 8f, N3) from the auxiliary outputs of the LAST step (so they describe the finished step even where the
 * environment was auto-reset), one pass, no host round trip:
 *   cam_terms [B, Nc, MATE_CAM_TERMS]: the keys of AuxiliaryCameraRewards.ACCEPTABLE_KEYS in order
 *     (mate/wrappers/auxiliary_camera_rewards.py:38-46, 140-149): raw_reward, coverage_rate, real_coverage_rate,
 *     mean_transport_rate, soft_coverage_score (0 unless soft_matrix is given), num_tracked, baseline; then is_sensed
 *     (mate/wrappers/more_training_information.py:61-65);
 *   tgt_terms [B, Nt, MATE_TGT_TERMS]: the keys of AuxiliaryTargetRewards.ACCEPTABLE_KEYS in order
 *     (mate/wrappers/auxiliary_target_rewards.py:135-177): raw_reward, coverage_rate, real_coverage_rate,
 *     mean_transport_rate, normalized_goal_distance, sparse_delivery, soft_coverage_score (0), is_tracked,
 *     is_colliding, baseline; then goal, goal_distance and the four clipped warehouse distances of
 *     MoreTrainingInformation (more_training_information.py:68-82).
 * `aux` must be the struct the last mate_b200_step / observe call filled, with mask_ct, mask_tc, coverage,
 * target_dones, is_colliding, warehouse_dist, tgt_goal and tgt_empty_bits non-NULL; rewards [B, 2] as written
 * by mate_b200_step. */
#define MATE_CAM_TERMS 8
#define MATE_TGT_TERMS 16
int mate_b200_auxiliary_terms(MateSim* sim, const MateStepAux* aux, const float* rewards, const float* soft_matrix,
                              float* cam_terms, float* tgt_terms, void* stream);

/* AuxiliaryCameraRewards.compute_soft_coverage_scores (mate/wrappers/auxiliary_camera_rewards.py:182-233): the
 * [B, Nc, Nt] matrix of signed distances of every target to the boundary of every camera's field of view (outer
 * polyline of Camera.add_obstacles / boundary_between(outer=True), mate/entities.py:362-479, 484-511, restricted
 * to the current sector), in units of the inscribed-circle radius.  mask_ct [B, Nc, Nt] as written by the last
 * step; `done` (nullable, [B]) marks the environments that were auto-reset in that step: they get zeros.  Pass the
 * result as `soft_matrix` to mate_b200_auxiliary_terms to fill the soft_coverage_score columns. */
int mate_b200_soft_coverage(MateSim* sim, const uint8_t* mask_ct, const uint8_t* done, float* soft_matrix, void* stream);

/* Batched opponents for the single-team wrappers (SURVEY.md section 8f, N4): GreedyTargetAgent
 * (mate/agents/greedy.py:235-365) for every target of every environment, driven like MultiCamera drives its
 * opponents (mate/wrappers/single_team.py:79-92, 261-279: observe -> communicate -> act).
 *   memory     dev double [MATE_AGENT_MEMORY, Nt, B] (field-major), owned by the caller, carried from step to step: goal (-1 = none),
 *              remembered non-empty warehouses (bit set), previous location x, y, previous noise x, y;
 *   reset_mask dev uint8 [B], nullable: environments whose agents are reset on the current state first
 *              (GreedyTargetAgent.reset: after env.reset and after an auto-reset);
 *   seed / serial  key and per-step counter of the agents' counter-based (Philox) draws;
 *   replay     parity mode: recorded outcomes of the agents' draws (NULL members = live draws);
 *   tgt_act    dev float [B, Nt, 2]: the joint target action for mate_b200_step. */
#define MATE_AGENT_MEMORY 6
typedef struct MateAgentReplay {
    const uint8_t* binomial;     /* [B, Nt] outcome of binomial(1, prob), greedy.py:315            */
    const double* sample;        /* [B, Nt, 2] action_space.sample() of a redraw, greedy.py:316     */
    const int8_t* choice;        /* [B, Nt] np_random.choice(non-empty warehouses), greedy.py:303   */
    const double* reset_sample;  /* [B, Nt, 2] action_space.sample() in reset(), greedy.py:271      */
} MateAgentReplay;
int mate_b200_greedy_target_actions(MateSim* sim, double* memory, const uint8_t* reset_mask, double noise_scale,
                                    uint64_t seed, uint64_t serial, const MateAgentReplay* replay, float* tgt_act,
                                    void* stream);

/* GreedyCameraAgent (mate/agents/greedy.py:14-232) for every camera of every environment, driven like MultiTarget
 * drives its opponents.  memory: dev double [6 Nt + Nc + 4, B, Nc] owned by the caller, FIELD-MAJOR (per camera the
 * fields are: remembered target states [Nt][4], time2forget [Nt], never_loaded [Nt], previous action [2], communication
 * delay [Nc], known teammates (bit set), own-state message pending); tracked: dev uint8 [B, Nc, Nt], the target flags of the cameras' CURRENT
 * observations; cam_act: dev float [B, Nc, 2].  Other arguments as for mate_b200_greedy_target_actions. */
typedef struct MateCameraAgentReplay {
    const int8_t* binomial;   /* [B, Nc] outcome of binomial(1, 0.1), greedy.py:96 (-1 = not drawn)          */
    const double* sample;     /* [B, Nc, 2] action_space.sample(), greedy.py:97                                */
    const int32_t* delay;     /* [B, Nc, Nc] randint(memory_period // 4, 2 * memory_period) per message sent   */
} MateCameraAgentReplay;
int mate_b200_greedy_camera_actions(MateSim* sim, double* memory, const uint8_t* tracked, const uint8_t* reset_mask,
                                    uint64_t seed, uint64_t serial, const MateCameraAgentReplay* replay, float* cam_act,
                                    void* stream);

/* The reference's communication wrappers (RestrictedCommunicationRange, RandomMessageDropout, NoCommunication,
 * mate/wrappers/message_filter.py) applied to the messages the batched greedy teams exchange inside
 * mate_b200_greedy_target_actions / _camera_actions (DESIGN.md section 7h).  A message is one routed copy (sender,
 * recipient) of a team: a target's broadcast of its non-empty warehouse set is one copy per teammate, its own
 * included; a camera sends at most one message (state bit and target byte) to each other camera per call.  A
 * message is delivered iff
 *   - the Euclidean distance of sender and recipient, taken in fp64 without fused multiply-add from the state the
 *     agents act on, is <= range_limit[team], and
 *   - its dropout draw keeps it: a 32-bit Philox word keyed on (the handle's seed, see mate_b200_seed, the global
 *     environment index) with counter (the call's serial, team, sender, recipient) below
 *     floor(keep_probability[team] * 2^32).  Several dropout wrappers compose into the product of their keep
 *     probabilities: equal in distribution to the reference, not draw for draw.
 * A dropped message changes only what the recipient receives; the sender's communication delay is drawn as before.
 * Every call also writes, when the pointers are given, the team's delivered set (delivered[team][b], bit 8 s + r:
 * s's message reached r) and adds it to total_edges[team] [B, N, N] (sender-major, int32); an environment's totals
 * restart from this call's set when its agents are reset (reset_mask).  Edges are counted with or without a
 * restriction.  The handle copies the struct; NULL = deliver everything, count nothing (the default).  MATE_EINVAL,
 * with the handle unchanged, for a range_limit that is negative or NaN, a keep_probability outside [0, 1], misaligned
 * pointers, or a restriction or edge pointer for a team of more than 8 agents. */
typedef struct MateMessageFilter {
    double range_limit[2];         /* per team, 0 = cameras, 1 = targets; INFINITY = unrestricted                     */
    double keep_probability[2];    /* per team; 1 = no dropout, 0 = no communication                                  */
    uint64_t* delivered[2];        /* dev [B]: bit 8 s + r = s's message reached r in the team's last call; nullable   */
    int32_t* total_edges[2];       /* dev [B, N, N]: delivered since the environment's agents were reset; nullable    */
} MateMessageFilter;
int mate_b200_set_message_filter(MateSim* sim, const MateMessageFilter* filter);

/* The tensor message channel of a learning team (DESIGN.md section 7i): every agent s of the team sends one message of
 * `dim` floats, content[b][s][:], to the teammates r with recipients[b][s][r] != 0 (NULL = broadcast: to every
 * teammate, its own copy included, like a broadcast Message).  A routed message is delivered iff it passes the team's
 * registered filter (mate_b200_set_message_filter) exactly as the greedy teams' messages do: the range rule on the
 * positions of the current state, then the dropout draw, word r % 4 of the Philox call keyed on (the handle's seed, the
 * global environment index, 'COMM') with counter (serial, 22 << 16 | team << 8 | s << 2 | r >> 2).  The caller advances
 * `serial` once per call; the draws do not depend on the batch split.
 *   - MATE_MESSAGES_NONE: inbox [B, N(r), N(s), dim]; inbox[b][r][s] is s's message, bit for bit, if it reached r, else 0.
 *   - MATE_MESSAGES_SUM:  inbox [B, N(r), dim], the float32 sum of the delivered messages, added in ascending s from 0.
 *   - MATE_MESSAGES_MEAN: that sum divided (IEEE, round to nearest) by the number of delivered senders; 0 without any.
 * A message that is not delivered is never read.  Every element of inbox (and of delivered) is written.  delivered
 * [B, N(r), N(s)] (nullable) gets 1 where s's message reached r, else 0.  When the team's edge tensors are registered
 * the call writes the delivered set to delivered[team][b] (bit 8 s + r) and adds it to total_edges[team]; an
 * environment's totals restart from this call's set when its episode id differs from episode[b], which is then set to
 * it (the caller sets episode[b] = -1 to restart them at the next call).  The call enqueues one kernel on `stream` and
 * never synchronises.  MATE_EINVAL, nothing launched, for a team other than 0 / 1, a team of 0 or more than 8 agents,
 * dim < 1 (or N * N * dim above 2^31 - 1), an unknown reduction, a NULL content, inbox or episode, or content / inbox /
 * episode not 4-byte aligned. */
#define MATE_MESSAGES_NONE 0
#define MATE_MESSAGES_SUM 1
#define MATE_MESSAGES_MEAN 2
typedef struct MateMessageExchange {
    const float* content;          /* dev [B, N, dim]                                                                 */
    const uint8_t* recipients;     /* dev [B, N(s), N(r)]: non-zero = s sends to r; NULL = broadcast                  */
    float* inbox;                  /* dev [B, N, N, dim] (NONE) or [B, N, dim] (SUM / MEAN)                           */
    uint8_t* delivered;            /* dev [B, N(r), N(s)]: 1 = s's message reached r; nullable                        */
    int32_t* episode;              /* dev [B]: the episode id the team's totals belong to, -1 = restart them          */
    int32_t team;                  /* 0 = cameras, 1 = targets                                                        */
    int32_t dim;                   /* floats per message, >= 1                                                        */
    int32_t reduction;             /* MATE_MESSAGES_NONE / _SUM / _MEAN                                               */
    int32_t reserved;              /* 0                                                                               */
} MateMessageExchange;
int mate_b200_exchange_messages(MateSim* sim, const MateMessageExchange* exchange, uint64_t serial, void* stream);

/* DiscreteCamera / DiscreteTarget.action (mate/wrappers/discrete_action_spaces.py:98-117, 204-228): grid
 * indices (dev int64 [count]) -> continuous actions (dev float32 [count][2]) through the wrapper's table
 * (dev float32 [table_size][2]). */
int mate_b200_decode_actions(const int64_t* index, const float* table, int32_t table_size, float* out,
                             int64_t count, void* stream);

/* Number of kernels this handle has launched since creation (bench bookkeeping). */
int64_t mate_b200_launch_count(const MateSim* sim);

/* What the last mate_b200_step_host call on this handle did on its device -> host leg (bench bookkeeping): *leg = 0 the rows
 * were copied densely, 1 their non-zero 16-byte chunks crossed the link and the rows were rebuilt in the caller's buffers,
 * 2 only the 64-byte groups that differ from the previous call's rows crossed and were patched in (MATE_STEP_HOST_ROWS_KEPT);
 * *row_bytes_on_link = bytes of observation rows (and their bitmaps) that crossed the link in that call (the teams with a
 * NULL buffer contribute none). */
int mate_b200_host_leg_info(const MateSim* sim, int32_t* leg, uint64_t* row_bytes_on_link);

#ifdef __cplusplus
}
#endif
#endif /* MATE_B200_H_ */
