/*
 * rover_b200.h -- C ABI of the B200-native rover hot path (librover_b200.so).
 *
 * The reference (abmoRobotics/isaac_rover_2.0) has no FFI: its boundary for this path is a set of
 * Python call signatures (SURVEY.md 8b).  Each entry point below replaces the arithmetic behind one of
 * those calls and cites it (paths relative to omniisaacgymenvs/tasks/).  The Python mirror in
 * isaac_rover_2.0_b200/ keeps the reference's names and signatures and binds these symbols with ctypes
 * (INTEGRATION.md shows the stub).
 *
 * Conventions
 *   - every pointer is a BORROWED DEVICE pointer into caller-owned memory unless the name ends in _host;
 *     fp16 buffers are passed as uint16_t* (IEEE binary16 bits); outputs are pre-allocated by the caller;
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*; NULL = legacy default stream);
 *     no hidden synchronisation except where stated;
 *   - return value: 0 = ok, <0 = rvb_status; rvb_last_error() gives a thread-local message;
 *   - nothing throws across this boundary; arguments are validated on the host before any launch;
 *   - `sem` selects which torch backend's rounding is reproduced where torch-CPU and torch-CUDA differ
 *     (division by a Python scalar is a reciprocal multiply on CUDA, and fp16-vs-scalar compares are done
 *     in fp32 on CUDA but in fp16 on CPU).  The reference hard-wires 'cuda:0' (rover.py:90), so
 *     RVB_SEM_TORCH_CUDA is the product default; RVB_SEM_TORCH_CPU exists so the CPU oracle / golden
 *     vectors can be matched bit for bit.
 */
#ifndef ROVER_B200_H
#define ROVER_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RVB_ABI_VERSION 5

typedef enum rvb_status {
    RVB_OK = 0,
    RVB_ERR_INVALID = -1,   /* bad argument (null pointer, shape, range) */
    RVB_ERR_CUDA = -2,      /* CUDA runtime error, see rvb_last_error() */
    RVB_ERR_NOMEM = -3,
    RVB_ERR_UNSUPPORTED = -4
} rvb_status;

typedef enum rvb_semantics { RVB_SEM_TORCH_CUDA = 0, RVB_SEM_TORCH_CPU = 1 } rvb_semantics;

int rvb_abi_version(void);
const char* rvb_last_error(void);

/* ------------------------------------------------------------------------------------------------
 * Terrain layer handle: the grid-bucketed K-nearest-triangle index + mesh of ONE layer (terrain or
 * big_rock_layer).  Replaces Camera._load_triangles_with_indices (utils/camera/camera.py:154-161) and
 * Rock_Detection._load_triangles_with_indices (utils/rock_detection/rock_detect.py:151-158).
 *
 * map_indices is the [G0,G1,K] *view* the reference indexes (element strides given, so the permuted
 * [K,G,G] tensor of camera.py:157-158 is accepted as is).  The handle owns a K-contiguous copy of the
 * index and one pre-resolved 32-byte record per triangle (a = v2, b = v1-a, c = v0-a, b x c, all fp16
 * with the reference's roundings, ray_casting.py:34-40).  Immutable after creation => usable from any
 * stream concurrently.  Synchronises `stream` before returning.
 * ---------------------------------------------------------------------------------------------- */
typedef struct rvb_terrain rvb_terrain;

int rvb_terrain_create(rvb_terrain** out,
                       const int32_t* map_indices, int64_t G0, int64_t G1, int64_t K,
                       int64_t stride_g0, int64_t stride_g1, int64_t stride_k,
                       const int32_t* triangles, int64_t T,
                       const uint16_t* vertices, int64_t V,
                       float res, float shift_x, float shift_y,
                       int sem, int flags, void* stream);
/* flags (0 = a heightmap layer with every list):
 *   RVB_LAYER_INDEX_ONLY  build the K-contiguous index and the triangle records only, not the block / superblock lists of the
 *                         heightmap ray-cast's production kernels: the layer of a Rock_Detection (rock_detect.py:151-158), whose
 *                         kernel scans the K-lists themselves -- 3.2 GB instead of 6 GB for the reference's rock index.
 *                         rvb_heightmap_raycast on such a layer runs the per-cell kernels (variants 1 / 2 and what 0 / 3 fall back to). */
#define RVB_LAYER_INDEX_ONLY 1
int rvb_terrain_destroy(rvb_terrain* t);
/* bytes of device memory owned by the handle */
int64_t rvb_terrain_bytes(const rvb_terrain* t);
/* Gives back the handle's K-contiguous copy of map_indices (G0*G1*K int32 -- the same size as the reference's tensor,
 * camera.py:154-157; more than half of a layer).  The production heightmap ray-cast (variants 0 and 3 of rvb_heightmap_raycast,
 * rvb_env_post) never reads it; afterwards variants 1 / 2, rvb_cast_rays and rvb_rock_collision on THIS handle return
 * RVB_ERR_INVALID.  Needs the block lists (K <= 255).  Synchronises the device.  rvb_terrain_has_index: 1 / 0. */
int rvb_terrain_release_index(rvb_terrain* t);
int rvb_terrain_has_index(const rvb_terrain* t);
/* Triangles of the layer whose fp16 determinant is within rounding of zero even for a vertical ray (zero area, edge-on): the shadow
 * kernel has no culling bound for them.  More than 2 % of T => variant 0 of rvb_heightmap_raycast runs the tiled kernel for the
 * whole layer; fewer => a tile that meets more than 128 of them is handed to the tiled kernel.  Results never depend on it. */
int64_t rvb_terrain_unbounded_triangles(const rvb_terrain* t);

/* ------------------------------------------------------------------------------------------------
 * Camera.get_depths (utils/camera/camera.py:60-145) = _depth_transform (:165-212) + _height_lookup
 * (:233-264) + the partitioned gather / ray_distance / min-over-K loop (:77-127).
 *   pos, euler   f32 [N,3]           pattern f64 [P,3] (Heightmap.get_distribution())
 *   trig         optional f32 [N,6] = sin,cos of -roll,-pitch,-yaw; NULL => computed with sinf/cosf
 *   dist         f16 [N,P]  (required)         hit_slot i32 [N,P] (argmin position in the K list, optional)
 *   hit_tri      i32 [N,P]  triangle id        pt, sources f16 [N,P,3] (optional)
 *   obs/obs_ld/col_a/col_b: optional fused Heightmap.get_sparse_vector/get_dense_vector + rover.py:324-325:
 *        obs[n*obs_ld + col_a[p]] = obs[n*obs_ld + col_b[p]] = f32(fp16(dist/2))  for columns >= 0.
 *   obs_h16/obs_h16_ld/obs_h16_col0: optional PACKED form of the same columns -- they are fp16 values by construction
 *        (rover.py:324-325 stores fp16(dist / 2) into the f32 obs_buf), so a consumer that wants half the bytes passes
 *        obs_h16[n*obs_h16_ld + (col - obs_h16_col0)] = fp16(dist/2)  for col in col_a/col_b >= 0  (obs may then be NULL).
 *        Not available with variant 1.  rvb_env_post uses it for rvb_step_io.obs_h16.
 * `variant`: 0 = production ("shadow" kernel: enumerates triangles, not (ray, candidate) pairs; needs the layer's block
 * lists, i.e. K <= 255, otherwise the tiled kernel on per-cell lists runs), 1 = simple per-pair kernel kept for
 * cross-checking, 2 = tiled kernel on per-cell lists, 3 = tiled kernel on 3x3-cell block lists.  All four are
 * bit-identical by construction.
 * ---------------------------------------------------------------------------------------------- */
int rvb_heightmap_raycast(const rvb_terrain* t, const float* pos, const float* euler, const float* trig,
                          const double* pattern, int64_t P, int64_t N,
                          uint16_t* dist, int32_t* hit_slot, int32_t* hit_tri, uint16_t* pt, uint16_t* sources,
                          float* obs, int64_t obs_ld, uint16_t* obs_h16, int64_t obs_h16_ld, int obs_h16_col0,
                          const int32_t* col_a, const int32_t* col_b, int variant, void* stream);

/* Cast pre-computed fp16 rays (sources/directions [R,3], directions NOT normalised, as handed to
 * ray_distance by camera.py:110) against a layer: _height_lookup + gather + ray_distance + min over K. */
int rvb_cast_rays(const rvb_terrain* t, const uint16_t* sources, const uint16_t* directions, int64_t R,
                  uint16_t* dist, int32_t* hit_slot, int32_t* hit_tri, uint16_t* pt, void* stream);

/* ray_distance(sources, directions, triangles) (utils/camera/ray_casting.py:3-66): n rays vs n triangles,
 * fp16.  sources, directions [n,3]; triangles [n,3,3]; k [n]; pt [n,3] (optional). */
int rvb_ray_distance(const uint16_t* sources, const uint16_t* directions, const uint16_t* triangles, int64_t n,
                     uint16_t* k, uint16_t* pt, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Rock_Detection.get_collisions (utils/rock_detection/rock_detect.py:52-149: _get_wheel_rays :160-319,
 * _get_body_rays :321-371, lookup + ray-cast against the big_rock_layer index) and
 * RoverTask.check_collision (rover.py:663-668).
 *   joints f32 [N,13] (DOF order rock_detect.py:174-188)    wheel_dist f16 [N,24]   body_dist f16 [N,2]
 *   hit_tri i32 [N,26] optional    collision i64 [N] optional (|min wheel| < 0.8 or |min body| < 0.45)
 *   rays_out f16 [N,26,6] optional (source xyz, direction xyz as fed to the ray-cast; for tests)
 *   joint_trig f32 [N,18] optional = (sin j_i, cos j_i) for the DOFs i = 0..8 the wheel chain uses (rock_detect.py:248-291),
 *        NULL = sinf/cosf on the device.  Like `trig` for the body rotation: libm results differ in the last ulp between
 *        torch-CPU, torch-CUDA and CUDA's sinf, and parity tests that demand bit-identical rays inject the oracle's values.
 * ---------------------------------------------------------------------------------------------- */
int rvb_rock_collision(const rvb_terrain* rocks, const float* pos, const float* euler, const float* trig,
                       const float* joints, const float* joint_trig, int64_t N,
                       uint16_t* wheel_dist, uint16_t* body_dist, int32_t* hit_tri, int64_t* collision,
                       uint16_t* rays_out, void* stream);
/* check_collision alone (rover.py:663-668) on caller-provided distances.  Both torch backends round the thresholds to fp16
 * before the compare, so the flags do not depend on `sem` and the call takes none. */
int rvb_check_collision(const uint16_t* wheel_dist, const uint16_t* body_dist, int64_t N, int64_t* collision, void* stream);

/* tensor_quat_to_eul (utils/math/tensor_quat_to_euler.py:6-31): wxyz f32 [N,4] -> (roll,pitch,yaw) f32 [N,3] */
int rvb_quat_to_euler(const float* quat, int64_t N, float* euler, void* stream);

/* Ackermann (utils/kinematics.py:14-67) + joint-target mapping (rover.py:396-409).
 *   lin/ang: f32 with element strides (the reference passes column views of actions[N,2], rover.py:391)
 *   steer, vel f32 [N,6] (FL,FR,ML,MR,RL,RR); pos_targets f32 [N,4] (FR,RR,FL,RL), vel_targets f32 [N,6]
 *   (FR,CR,RR,FL,CL,RL), both optional. */
int rvb_ackermann(const float* lin, int64_t lin_stride, const float* ang, int64_t ang_stride, int64_t N,
                  float* steer, float* vel, float* pos_targets, float* vel_targets, int sem, void* stream);

/* Memory.input_state (rover.py:76-77): hist f32 [N,H] shift right by one, newest at column 0. */
int rvb_history_push(float* hist, int64_t N, int64_t H, const float* newest, int64_t newest_stride, void* stream);

/* RoverTask.get_observations, proprioceptive part (rover.py:279-283, 320-323): heading f32 [N] and
 * obs[:,0:4] = (|target-pos|/9, heading/pi, lin_now, ang_now).  obs row stride obs_ld (elements). */
int rvb_obs_proprio(const float* pos, const float* euler, const float* target, const float* lin_now,
                    const float* ang_now, int64_t N, float* obs, int64_t obs_ld, float* heading, int sem,
                    void* stream);
/* Heightmap.get_sparse_vector/get_dense_vector + rover.py:324-325 on an existing dist buffer:
 * obs[n, col0 + i] = f32(fp16(dist[n, idx[i]] / 2)). */
int rvb_obs_gather(const uint16_t* dist, int64_t P, int64_t N, const int64_t* idx, int64_t n_idx,
                   float* obs, int64_t obs_ld, int64_t col0, void* stream);

/* ------------------------------------------------------------------------------------------------
 * RoverTask.calculate_metrics (rover.py:460-531) + RoverTask.is_done (:610-647), one pass.
 * ---------------------------------------------------------------------------------------------- */
typedef struct rvb_reward_params {
    float pos_reward, heading_contraint_reward, motion_contraint_reward, goal_angle_reward,
          boogie_contraint_reward;                 /* cfg/task/Rover.yaml:37-46 */
    int32_t max_episode_length;                    /* rover.py:119 (3000) */
    int32_t curriculum_level;                      /* rover.py:104,353 */
    int64_t num_envs_total;                        /* collision_penalty = flag * num_envs (rover.py:517) */
    int32_t sem;
    int32_t reserved;
} rvb_reward_params;

#define RVB_N_STATS 16
/* stats (f64 [16], optional, overwritten): 0 envs, 1 sum rew, 2 sum pos_reward, 3 collisions, 4 sum
 * uprightness, 5 sum heading pen., 6 sum motion pen., 7 sum goal-angle pen., 8 resets, 9 timeouts,
 * 10 tilt resets, 11 too-far resets, 12 goals reached, 13 collision resets, 14 sum target dist, 15 0.
 * Deterministic (fixed-order two-stage reduction).  `stats_scratch` f64 [rvb_stats_scratch_len(N)]. */
int64_t rvb_stats_scratch_len(int64_t N);
int rvb_reward_reset(const rvb_reward_params* p,
                     const float* pos, const float* target, const float* heading, const float* rover_rot,
                     const float* lin, const float* lin_prev, const float* ang, const float* ang_prev,
                     const float* joints, const int64_t* progress, const int64_t* rock_collision, int64_t N,
                     float* rew, int64_t* reset,
                     float* ex_pos_reward, int64_t* ex_collision, float* ex_uprightness, float* ex_heading,
                     float* ex_motion, float* ex_goal_angle,
                     double* stats, double* stats_scratch, void* stream);

/* ------------------------------------------------------------------------------------------------
 * One env step with two host calls, split at the simulator's boundary, for the loop this library is built into:
 *   obs_t -> policy -> pre_physics_step(a_t) -> simulator steps -> post_physics_step() -> obs_{t+1}.
 * PhysX is outside this library: a caller without a simulator step between the calls passes the same poses to both.
 *
 * rvb_env_pre is the action half of RoverTask.pre_physics_step (rover.py:338-414) on the PRE-physics pose: rover_rot =
 * tensor_quat_to_eul(quat) (rover.py:343; is_done reads it one post half later, :615-616), Memory.input_state x2 (:379-380,389),
 * Ackermann + joint targets (:391,400-409): rvb_quat_to_euler, rvb_history_push x2 and rvb_ackermann in one launch.  It reads
 * no goal, progress or reset state, so it may run before or after the reset half of pre_physics_step.
 *   quat f32 [N,4] (16-byte aligned)  actions f32 [N,2]  lin_hist/ang_hist f32 [N,H] (shifted in place)  rover_rot f32 [N,3]
 *   pos_targets f32 [N,4] (FR,RR,FL,RL), vel_targets f32 [N,6] (FR,CR,RR,FL,CL,RL), both optional.
 *
 * rvb_env_post is RLTask.post_physics_step (rl_task.py:239-259) on the POST-physics poses in io: progress += 1, get_observations
 * (euler -> io.euler, heading, proprioceptive columns with this step's action read from lin_hist/ang_hist[:, 0], heightmap
 * ray-cast into obs or obs_h16, rock layer), calculate_metrics + is_done with the rover_rot of rvb_env_pre.  Equivalent to
 * calling rvb_quat_to_euler, rvb_obs_proprio, rvb_heightmap_raycast (obs fused), rvb_rock_collision and rvb_reward_reset in
 * that order; the rock layer is cast on an internal forked stream, concurrently with the heightmap.
 *   lin_hist/ang_hist f32 [N,H] (Memory.tracker, newest first; as rvb_env_pre left them)   progress i64 [N] (incremented in place)
 *   euler f32 [N,3]  heading f32 [N]
 *   obs f32 [N,obs_ld>=4+sparse+dense]  dist f16 [N,P]  wheel_dist f16 [N,24]  body_dist f16 [N,2]  rock_collision i64 [N]
 *   (rock outputs and the `rocks` layer may be NULL when curriculum_level < 2); rew, reset, ex_*, stats as rvb_reward_reset.
 * ---------------------------------------------------------------------------------------------- */
typedef struct rvb_step_io {
    const float* pos; const float* quat; const float* joints; const float* target;
    float* lin_hist; float* ang_hist; int64_t* progress;
    float* euler; float* heading;
    float* obs; int64_t obs_ld;
    uint16_t* dist; uint16_t* wheel_dist; uint16_t* body_dist; int64_t* rock_collision;
    float* rew; int64_t* reset;
    float* ex_pos_reward; int64_t* ex_collision; float* ex_uprightness; float* ex_heading; float* ex_motion; float* ex_goal_angle;
    double* stats; double* stats_scratch;
    /* optional packed observation (ABI 2): obs_h16 f16 [N, obs_h16_ld >= sparse+dense] receives the heightmap columns
     * (obs column c -> obs_h16 column c - 4) as the fp16 values they are by construction (fp16(dist / 2), rover.py:324-325);
     * obs[:, 4:] is then NOT written (obs[:, 0:4] still is).  Halves the bytes a host-side consumer has to read back.  The teacher-data
     * recorder then reads the observation from obs_h16 and obs[:, 0:4] (rvb_teacher_record_packed), never from obs[:, 4:]. */
    uint16_t* obs_h16; int64_t obs_h16_ld;
} rvb_step_io;
int rvb_env_pre(const float* quat, const float* actions, int64_t N, int64_t H, float* lin_hist, float* ang_hist,
                float* rover_rot, float* pos_targets, float* vel_targets, int sem, void* stream);
int rvb_env_post(const rvb_terrain* terrain, const rvb_terrain* rocks, const rvb_reward_params* p, const rvb_step_io* io,
                 const float* rover_rot, const double* pattern, int64_t P, const int32_t* col_a, const int32_t* col_b,
                 int64_t N, int64_t H, void* stream);

/* Device timing of the heightmap ray-cast inside rvb_env_post (CUDA events on the caller's stream, calling thread only):
 * enable, run steps, then read the per-step durations in ms (host array; returns the count or <0; synchronises). */
int rvb_timing_enable(int on);
int rvb_timing_read(float* ms_host, int cap);

/* ------------------------------------------------------------------------------------------------
 * stone_info validation (rover.py:533-542 check_goal_collision, :649-661 avoid_pos_rock_collision):
 * nearest[m] = min_s(cdist(xy[m], stone[s].xy) - stone[s].radius), flag[m] = nearest <= thr.
 *   xy f32 with row stride xy_ld; stones f32 [S,7]; nearest/flag/count optional; count i32 [1] += #flags.
 * torch.cdist switches to its matmul formulation when M>25 or S>25; `force_mode` 0 = same rule,
 * 1 = direct, 2 = matmul formulation.
 * ---------------------------------------------------------------------------------------------- */
int rvb_stone_validate(const float* xy, int64_t xy_ld, int64_t M, const float* stones, int64_t S, float thr,
                       int force_mode, float* nearest, int64_t* flag, int32_t* count, void* stream);
/* avoid_pos_rock_collision: the whole fixed-point loop on the device (x += 0.05 while nearest <= 1.4).
 * pos f32 [N,3] updated in place; iterations i32 [1] optional (number of sweeps executed). */
int rvb_spawn_validate(float* pos, int64_t N, const float* stones, int64_t S, int32_t max_iter,
                       int32_t* iterations, void* stream);
/* get_pos_height (rover.py:588-608): out[m] = heightmap[round(clamp((xy-shift)/hscale,0,H-1))] * vscale */
int rvb_height_lookup(const float* heightmap, int64_t H0, int64_t H1, const float* xy, int64_t xy_ld, int64_t M,
                      float hscale, float vscale, float shift_x, float shift_y, float* out, int sem, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Device-side reset path (SURVEY.md 8f-2): RoverTask.pre_physics_step's work for the envs whose reset_buf is set
 * (rover.py:356-361) in ONE launch and without the reference's host synchronisations (reset_buf.nonzero() + len(),
 * rover.py:356-357; the `while reset_buf_len > 0` goal loop, :547-549):
 *   reset_idx book-keeping (rover.py:451-452): progress[n] = 0, reset_out[n] = 0 (both optional; reset_out may alias reset_in);
 *   generate_goals (rover.py:544-564): a goal on the circle of `radius` around initial_pos[n], re-drawn (at most max_attempts
 *     times) until min_s(|goal - stone_s| - radius_s) > thr (rover.py:533-542, direct distance formula);
 *   set_targets (rover.py:582-583): target[n,2] = heightmap value at the goal (rvb_height_lookup arithmetic).
 * The reference draws torch.rand numbers in resetting-env order, which no device-side scheme can reproduce; here the k-th
 * draw of env g at call `epoch` is Philox4x32-10(counter = (g lo, g hi, k, epoch lo), key = (seed lo, seed hi ^ epoch hi)),
 * u = (x0 >> 8) * 2^-24, so results depend on (seed, epoch, global env id) only -- not on sharding.  env_offset = global id of
 * local env 0.  The reference's re-draw of env 0 on every retry (rover.py:540) is not reproduced.
 * counters i32 [3] optional, overwritten: envs reset, goals drawn, envs that exhausted max_attempts.
 * ---------------------------------------------------------------------------------------------- */
int rvb_reset_targets(const int64_t* reset_in, int64_t N, int64_t env_offset, uint64_t seed, uint64_t epoch,
                      const float* initial_pos, float radius, const float* stones, int64_t S, float thr,
                      int32_t max_attempts, const float* heightmap, int64_t H0, int64_t H1, float hscale, float vscale,
                      float shift_x, float shift_y, float* target, int64_t* progress, int64_t* reset_out,
                      int32_t* counters, int sem, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Offline index builder (utils/rover_utils.py:52-118 _get_knn_triangles): for cell (i,j) at fp16
 * coordinates (cell_x[i], cell_y[j]) -- torch.arange(0, G*res, res, dtype=float16), rover_utils.py:77-78 --
 * the K triangles with the smallest fp16 centroid distance; ties ordered by triangle id (torch.topk leaves
 * them unspecified).  out int32 [K,G0,G1] like map_indices.pt.  Synchronises `stream` once (bounding box).
 * ---------------------------------------------------------------------------------------------- */
int rvb_build_knn_index(const int32_t* triangles, int64_t T, const uint16_t* vertices, int64_t V,
                        const uint16_t* cell_x, const uint16_t* cell_y, int64_t G0, int64_t G1, int64_t K,
                        int32_t* out, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Policy-inference epilogue (SURVEY.md 8f-3): the consumer of obs_buf.  Replaces
 * StochasticActorHeightmap.compute and DeterministicHeightmap.compute (../learning/model.py:152-195,197-241):
 *   x0 = encoder0(obs[:, p:p+S]); x1 = encoder1(obs[:, p+S:p+S+D]); x = cat(obs[:, 0:p], x0, x1)   (model.py:183-189)
 *   x = mlp(x); out = head(x) [tanh for the actor, model.py:176]                                   (model.py:190-191)
 * every hidden layer being Linear + activation (model.py:86-116).  The layer widths are the ones the reference
 * hard-wires (../train.py:95, ../cfg/trainSKRL/RoverPPOSKRL.yaml:4-9): encoders [80,60], mlp [256,160,128]; other widths
 * return RVB_ERR_UNSUPPORTED.  p <= 8, S and D are free (the C5 patterns change them), head width 1..4.
 * rvb_linear = one torch nn.Linear: weight f32 [out_features, in_features] row-major, bias f32 [out_features], both
 * borrowed DEVICE pointers that may be released when rvb_policy_create returns (it re-packs them into k-major panels
 * owned by the handle and synchronises `stream`).  enc_sparse / enc_dense point at 2 layers, mlp at 3, head at 1.
 * `device` must be the calling thread's current CUDA device (the library never switches devices).
 * fp32-grade arithmetic like the reference's (TF32 off); accumulation order differs from cuBLAS, parity gate 2e-5 absolute.
 * rvb_policy_forward: obs f32 [N, obs_ld] (obs_ld >= p+S+D) -> out f32 [N, out_ld] columns 0..head-1, asynchronous on `stream`;
 * the handle is immutable => usable from any stream.  Two kernels on the tensor cores (tcgen05, tf32 hi + lo operands,
 * accumulators in TMEM): the first encoder layers, then the rest of the network as a programmatic dependent launch.  Shapes that
 * path refuses (p != 4, odd S, D or obs_ld, obs not 8-byte aligned) run one fp32 FFMA2 kernel instead, which computes the same
 * layers in another summation order.
 * ---------------------------------------------------------------------------------------------- */
typedef struct rvb_policy rvb_policy;
typedef struct rvb_linear {
    const float* weight;
    const float* bias;
    int32_t in_features, out_features;
} rvb_linear;
typedef enum rvb_activation {   /* the keys of Layer.activation_functions, model.py:104-111 */
    RVB_ACT_LEAKYRELU = 0, RVB_ACT_RELU = 1, RVB_ACT_ELU = 2, RVB_ACT_TANH = 3, RVB_ACT_SIGMOID = 4, RVB_ACT_RELU6 = 5
} rvb_activation;

int rvb_policy_create(rvb_policy** out, int32_t n_proprio, int32_t n_sparse, int32_t n_dense,
                      const rvb_linear* enc_sparse, const rvb_linear* enc_dense, const rvb_linear* mlp,
                      const rvb_linear* head, int32_t activation, int32_t head_tanh, int device, void* stream);
int rvb_policy_destroy(rvb_policy* policy);
int64_t rvb_policy_bytes(const rvb_policy* policy);
int rvb_policy_forward(const rvb_policy* policy, const float* obs, int64_t obs_ld, int64_t N, float* out, int64_t out_ld,
                       void* stream);
/* Policy dispatch, process-wide: 2 = default (tensor-core path where the shape allows it, FFMA2 kernel otherwise), 1 = the FFMA2
 * kernel for every shape.  The hook bench.py (`ffma2_kernel_ms`) and the tests use to force the FFMA path.  1 or 2 sets the
 * dispatch and returns the previous value; a negative argument only queries it; anything else (0 and 3 selected kernels that are
 * gone) returns RVB_ERR_INVALID and leaves the setting unchanged. */
int rvb_policy_variant(int variant);
/* Two networks on the same observations in ONE launch (grid.y = network): what a PPO step asks for -- policy.compute and
 * value.compute on the same states.  Twice the CTAs for the same obs tile (second read served by L2). */
int rvb_policy_forward_pair(const rvb_policy* a, const rvb_policy* b, const float* obs, int64_t obs_ld, int64_t N,
                            float* out_a, int64_t out_a_ld, float* out_b, int64_t out_b_ld, void* stream);
/* The same networks on the packed observation of the fused step (rvb_step_io.obs_h16): proprio f32 [N, proprio_ld >= p] (obs[:, 0:p],
 * e.g. the strided view obs_buf[:, :4]) and heightmap f16 [N, heightmap_ld >= S+D] (the sparse then the dense columns, as raw fp16
 * bits).  b = NULL runs network a alone (out_b is ignored); otherwise a and b as in rvb_policy_forward_pair.  The result is bit for bit
 * that of rvb_policy_forward(_pair) on the widened rows cat(proprio, float(heightmap)), on either path: the heightmap's fp16 values
 * are exact in tf32, so the tensor-core path reads them as they are (half the bytes) and splits nothing.  It takes the tensor-core
 * path when p == 4, S and D are even, heightmap_ld is even and heightmap is 4-byte aligned (and rvb_policy_variant is 2); the FFMA2
 * kernel otherwise, for any 2-byte aligned heightmap.  Null pointers, short rows and mismatched networks are refused on the host. */
int rvb_policy_forward_packed(const rvb_policy* a, const rvb_policy* b, const float* proprio, int64_t proprio_ld,
                              const uint16_t* heightmap, int64_t heightmap_ld, int64_t N, float* out_a, int64_t out_a_ld,
                              float* out_b, int64_t out_b_ld, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Observation hooks and the teacher-data recorder (SURVEY.md 8f-4).
 * rvb_obs_hooks: the four in-place epilogues of RoverTask.get_observations the reference keeps commented out
 * (rover.py:326-329), applied in the reference's order on obs f32 [N, obs_ld] columns [0, C):
 *   columns >= col0:  v += noise_std * z           (rover.py:326, sqrt(0.20) * randn; 0 = off)
 *   columns >= col0:  v  = dropped ? 0 : v / (1 - dropout_p)      (rover.py:327, F.dropout p=0.1; 0 = off)
 *   every column:     v -= offset                  (rover.py:328, 0.02)
 *   zero_mask[c]!=0:  v  = 0                       (rover.py:329, remove_idx + 4 as a u8 [C] column mask; NULL = off)
 * Draws: Philox4x32-10, counter = (global env id lo, hi, column, epoch lo), key = (seed lo, seed hi ^ epoch hi);
 * normal by Box-Muller from x0, x1, dropout from x2 -- a function of (seed, epoch, env_offset + n, column) only, so shards
 * reproduce the unsharded run (torch's own generator stream is not reproduced).
 * rvb_teacher_record: one row of the teacher data set per env (rover.py:299-300,364,374-375):
 *   record[n] = [reset_info[n], actions[n,0], actions[n,1], obs[n, 0..C)],  record f32 [N, record_ld >= C+3].
 * ---------------------------------------------------------------------------------------------- */
int rvb_obs_hooks(float* obs, int64_t obs_ld, int64_t N, int64_t C, int64_t col0, float noise_std, float dropout_p,
                  float offset, const uint8_t* zero_mask, uint64_t seed, uint64_t epoch, int64_t env_offset, void* stream);
int rvb_teacher_record(const float* reset_info, const float* actions, int64_t actions_ld, const float* obs, int64_t obs_ld,
                       int64_t N, int64_t C, float* record, int64_t record_ld, void* stream);
/* rvb_teacher_record on the packed observation of the fused step (rvb_step_io.obs_h16): proprio f32 [N, proprio_ld >= p] = obs[:, 0:p]
 * (e.g. the strided view obs_buf[:, :4]; may be NULL when p == 0), heightmap f16 [N, heightmap_ld >= E] = obs_h16 (raw fp16 bits).
 *   rec16 == NULL: rec[n] = [reset_info[n], a0, a1, proprio[n, 0..p), f32(heightmap[n, 0..E))]   rec_ld >= 3 + p + E
 *                  -- bit for bit what rvb_teacher_record writes for the widened row cat(proprio, heightmap.float()).
 *   rec16 != NULL: rec[n] = [reset_info[n], a0, a1, proprio[n, 0..p)]   rec_ld >= 3 + p,   rec16[n, 0..E) = heightmap[n, 0..E)
 *                  (the bits copied: half the bytes of the f32 row; fp16 -> f32 is exact, so widening rec16 later gives the same rows).
 * Any 2-byte aligned heightmap / rec16 and any row strides, odd ones included; 64-bit row offsets.  p in 0..8, E >= 1; N == 0 is a
 * no-op.  Null pointers, short rows and misaligned pointers are refused on the host. */
int rvb_teacher_record_packed(const float* reset_info, const float* actions, int64_t actions_ld, const float* proprio,
                              int64_t proprio_ld, int64_t p, const uint16_t* heightmap, int64_t heightmap_ld, int64_t E, int64_t N,
                              float* rec, int64_t rec_ld, uint16_t* rec16, int64_t rec16_ld, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* ROVER_B200_H */
