// Fused env step: everything the action half of RoverTask.pre_physics_step (rover.py:366-414) and RLTask.post_physics_step
// (rl_task.py:239-259) compute for one step, enqueued by two host calls, one on each side of the simulator's step:
//   rvb_env_pre            env_pre_kernel: tensor_quat_to_eul of the pre-physics pose (rover_rot), Memory.input_state x2,
//                          Ackermann + joint targets                                    (one thread per env)
//   rvb_env_post           env_post_kernel: progress += 1, euler of the post-physics pose, proprioceptive columns + heading
//                          (one thread per env), then:
//     heightmap ray-cast   Camera.get_depths with the sparse/dense gather fused into obs_buf[:, 4:]
//     rock collision       Rock_Detection.get_collisions + check_collision, on a forked stream (independent of the ray-cast)
//     reward_reset         calculate_metrics + is_done + episode statistics (rvb_reward_reset)
// The per-call entry points of rover_b200.h stay the reference-shaped API; this pair removes ~25 Python/ctypes round trips
// per step (the host side was the bottleneck once the ray-cast dropped below 1.5 ms).
#include "task_dev.cuh"
#include "raycast_common.cuh"

// action half alone: rover_rot is the euler of the pose BEFORE physics (rover.py:343), is_done reads it one post half later
__global__ void env_pre_kernel(const float* __restrict__ quat, const float* __restrict__ actions, int64_t N, int H,
                               float* __restrict__ lin_hist, float* __restrict__ ang_hist, float* __restrict__ rover_rot,
                               float* __restrict__ pos_t, float* __restrict__ vel_t, int sem) {
    const int64_t n = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (n >= N) return;
    const float4 q = reinterpret_cast<const float4*>(quat)[n];
    float r, p, y;
    quat_to_euler_dev(q.x, q.y, q.z, q.w, r, p, y);
    rover_rot[n * 3 + 0] = r; rover_rot[n * 3 + 1] = p; rover_rot[n * 3 + 2] = y;
    const float lin = actions[n * 2 + 0], ang = actions[n * 2 + 1];
    float* hl = lin_hist + n * H;
    float* ha = ang_hist + n * H;
    for (int i = H - 1; i > 0; --i) { hl[i] = hl[i - 1]; ha[i] = ha[i - 1]; }  // rover.py:76-77
    hl[0] = lin; ha[0] = ang;
    float st[6], ve[6];
    ackermann_dev(lin, ang, sem, st, ve);
    ackermann_store(n, st, ve, nullptr, nullptr, pos_t, vel_t);
}

// per-env start of the observation half on the post-physics pose; this step's action is hist[:, 0], pushed by the pre half
__global__ void env_post_kernel(rvb_step_io io, int64_t N, int H, int sem) {
    const int64_t n = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (n >= N) return;
    io.progress[n] += 1;                                                       // rl_task.py:241
    const float4 q = reinterpret_cast<const float4*>(io.quat)[n];
    float r, p, y;
    quat_to_euler_dev(q.x, q.y, q.z, q.w, r, p, y);
    io.euler[n * 3 + 0] = r; io.euler[n * 3 + 1] = p; io.euler[n * 3 + 2] = y;
    obs_proprio_dev(io.pos[n * 3 + 0], io.pos[n * 3 + 1], y, io.target[n * 3 + 0], io.target[n * 3 + 1], io.lin_hist[n * H],
                    io.ang_hist[n * H], sem, io.obs + n * io.obs_ld, io.heading + n);
}

#include <vector>

namespace {
// optional device timing of the heightmap ray-cast inside rvb_env_post (bench.py's roofline figure)
struct Timing {
    bool on = false;
    std::vector<cudaEvent_t> ev;     // start, end, start, end, ...
    size_t used = 0;
};
thread_local Timing g_timing;

}  // namespace

extern "C" int rvb_env_pre(const float* quat, const float* actions, int64_t N, int64_t H, float* lin_hist, float* ang_hist,
                           float* rover_rot, float* pos_targets, float* vel_targets, int sem, void* stream) {
    RVB_REQUIRE(N >= 0, "rvb_env_pre: N < 0");
    if (N == 0) return RVB_OK;
    RVB_REQUIRE(quat && actions && lin_hist && ang_hist && rover_rot, "rvb_env_pre: null pointer");
    RVB_REQUIRE(((uintptr_t)quat & 15) == 0, "rvb_env_pre: quat must be 16-byte aligned");
    RVB_REQUIRE(H >= 2 && H <= 64, "rvb_env_pre: history length out of range");
    env_pre_kernel<<<(unsigned)ceil_div(N, 256), 256, 0, as_stream(stream)>>>(quat, actions, N, (int)H, lin_hist, ang_hist, rover_rot,
                                                                             pos_targets, vel_targets, sem);
    RVB_LAUNCH_CHECK();
    return RVB_OK;
}

extern "C" int rvb_env_post(const rvb_terrain* terrain, const rvb_terrain* rocks, const rvb_reward_params* p, const rvb_step_io* io_,
                            const float* rover_rot, const double* pattern, int64_t P, const int32_t* col_a, const int32_t* col_b,
                            int64_t N, int64_t H, void* stream) {
    RVB_REQUIRE(N >= 0, "rvb_env_post: N < 0");
    if (N == 0) return RVB_OK;
    RVB_REQUIRE(terrain && p && io_ && rover_rot && pattern && col_a && col_b, "rvb_env_post: null pointer");
    const rvb_step_io io = *io_;
    RVB_REQUIRE(io.pos && io.quat && io.joints && io.target && io.lin_hist && io.ang_hist && io.euler && io.heading && io.obs &&
                    io.dist && io.rew && io.reset && io.progress, "rvb_env_post: null pointer in rvb_step_io");
    RVB_REQUIRE(((uintptr_t)io.quat & 15) == 0, "rvb_env_post: quat must be 16-byte aligned");
    RVB_REQUIRE(H >= 2 && H <= 64 && io.obs_ld >= 4, "rvb_env_post: bad history length or obs_ld");
    RVB_REQUIRE(!io.obs_h16 || io.obs_h16_ld > 0, "rvb_env_post: obs_h16 needs obs_h16_ld");
    RVB_REQUIRE(p->curriculum_level < 2 || (rocks && io.wheel_dist && io.body_dist && io.rock_collision),
                "rvb_env_post: curriculum_level >= 2 needs the rock layer and its outputs");
    cudaStream_t st = as_stream(stream);
    // the knobs are read and the ray-cast's arguments checked before the first launch, so that a bad knob or argument fails the
    // call before anything is launched
    RaycastKnobs knobs;
    const int krc = read_raycast_knobs(knobs);
    if (krc != RVB_OK) return krc;
    // packed observation requested: the heightmap columns go to obs_h16 (fp16, what they are by construction) and the f32
    // columns 4.. of obs are left alone
    rc::TiledParams q{};
    q.pos = io.pos; q.euler = io.euler; q.pattern = pattern; q.dist = (__half*)io.dist;
    q.obs = io.obs_h16 ? nullptr : io.obs; q.obs_ld = io.obs_ld; q.col_a = col_a; q.col_b = col_b;
    q.obs16 = (__half*)io.obs_h16; q.obs16_ld = io.obs_h16_ld; q.obs16_col0 = 4;
    const int prc = fill_tiled_params(terrain, P, N, 0, q);
    if (prc != RVB_OK) return prc;
    env_post_kernel<<<(unsigned)ceil_div(N, 256), 256, 0, st>>>(io, N, (int)H, p->sem);
    RVB_LAUNCH_CHECK();
    cudaEvent_t t0 = nullptr, t1 = nullptr;
    if (g_timing.on) {
        if (g_timing.used + 2 > g_timing.ev.size()) {
            cudaEvent_t a, b;
            RVB_CUDA(cudaEventCreate(&a));
            RVB_CUDA(cudaEventCreate(&b));
            g_timing.ev.push_back(a);
            g_timing.ev.push_back(b);
        }
        t0 = g_timing.ev[g_timing.used];
        t1 = g_timing.ev[g_timing.used + 1];
        g_timing.used += 2;
        // the timed ray-cast includes its env order, as a standalone rvb_heightmap_raycast (which builds the order inside) does
        RVB_CUDA(cudaEventRecord(t0, st));
    }
    // one env order (from this step's euler) for the ray-cast and the rock kernel; declared before the join guard, so that st
    // waits for the rock kernel before the order goes back to the pool
    RvbTemp<int32_t> order;
    RVB_CUDA(order.alloc_pool((size_t)N, st));
    const int orc = build_env_order(q, N, knobs.cos_steep, order.p, st);
    if (orc != RVB_OK) return orc;
    const bool with_rocks = rocks && io.wheel_dist && io.body_dist;
    RvbJoinGuard guard(st);          // on every exit path below: st waits for the rock layer's kernel
    if (with_rocks) {
        RvbSide* side = nullptr;
        RVB_CUDA(rvb_side_stream(0, &side));
        RVB_CUDA(cudaEventRecord(side->fork, st));
        RVB_CUDA(cudaStreamWaitEvent(side->s, side->fork, 0));
        const int rc = rock_collision(rocks, io.pos, io.euler, nullptr, io.joints, nullptr, N, io.wheel_dist, io.body_dist, nullptr,
                                      io.rock_collision, nullptr, order.p, side->s);
        if (rc != RVB_OK) return rc;
        RVB_CUDA(cudaEventRecord(side->join, side->s));
        guard.join = side->join;
    }
    const int rc = heightmap_raycast(terrain, q, N, 0, knobs, order.p, st);
    if (rc != RVB_OK) return rc;
    if (t1) RVB_CUDA(cudaEventRecord(t1, st));
    if (guard.join) {
        RVB_CUDA(cudaStreamWaitEvent(st, guard.join, 0));
        guard.join = nullptr;
    }
    // hist[:, 0] = this step's action, hist[:, 1] = the previous one (rover.py:498-501)
    return launch_reward_reset(p, io.pos, io.target, io.heading, rover_rot, io.lin_hist, io.lin_hist + 1, io.ang_hist, io.ang_hist + 1, H,
                            io.joints, io.progress, p->curriculum_level >= 2 ? io.rock_collision : nullptr, N, io.rew, io.reset,
                            io.ex_pos_reward, io.ex_collision, io.ex_uprightness, io.ex_heading, io.ex_motion, io.ex_goal_angle,
                            io.stats, io.stats_scratch, st);
}

extern "C" int rvb_timing_enable(int on) {
    g_timing.on = on != 0;
    g_timing.used = 0;
    return RVB_OK;
}

extern "C" int rvb_timing_read(float* ms_host, int cap) {
    int n = 0;
    for (size_t i = 0; i + 1 < g_timing.used && n < cap; i += 2, ++n) {
        if (cudaEventSynchronize(g_timing.ev[i + 1]) != cudaSuccess) return rvb_set_error(RVB_ERR_CUDA, "rvb_timing_read", "event sync failed");
        if (cudaEventElapsedTime(ms_host + n, g_timing.ev[i], g_timing.ev[i + 1]) != cudaSuccess)
            return rvb_set_error(RVB_ERR_CUDA, "rvb_timing_read", "elapsed time failed");
    }
    g_timing.used = 0;
    return n;
}
