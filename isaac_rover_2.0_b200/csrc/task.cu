// Per-env fp32 task arithmetic: tensor_quat_to_eul, Ackermann + joint-target mapping, Memory.input_state,
// the proprioceptive observation columns, calculate_metrics + is_done with fused episode statistics.
// All of it is HBM-streaming SoA/AoS work: one thread per env, coalesced loads, no FMA contraction.
#include "task_dev.cuh"

__global__ void quat_to_euler_kernel(const float4* __restrict__ quat, int64_t N, float* __restrict__ euler) {
    int64_t n = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (n >= N) return;
    const float4 q = quat[n];
    float r, p, y;
    quat_to_euler_dev(q.x, q.y, q.z, q.w, r, p, y);
    euler[n * 3 + 0] = r;
    euler[n * 3 + 1] = p;
    euler[n * 3 + 2] = y;
}

extern "C" int rvb_quat_to_euler(const float* quat, int64_t N, float* euler, void* stream) {
    if (N <= 0) return RVB_OK;
    RVB_REQUIRE(quat && euler, "rvb_quat_to_euler: null pointer");
    RVB_REQUIRE(((uintptr_t)quat & 15) == 0, "rvb_quat_to_euler: quat must be 16-byte aligned");
    quat_to_euler_kernel<<<(unsigned)ceil_div(N, 256), 256, 0, as_stream(stream)>>>((const float4*)quat, N, euler);
    RVB_LAUNCH_CHECK();
    return RVB_OK;
}

// ---------------------------------------------------------------- Ackermann
__global__ void ackermann_kernel(const float* __restrict__ lin_p, int64_t lin_stride, const float* __restrict__ ang_p,
                                 int64_t ang_stride, int64_t N, float* __restrict__ steer, float* __restrict__ vel,
                                 float* __restrict__ pos_t, float* __restrict__ vel_t, int sem) {
    int64_t n = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (n >= N) return;
    float st[6], ve[6];
    ackermann_dev(lin_p[n * lin_stride], ang_p[n * ang_stride], sem, st, ve);
    ackermann_store(n, st, ve, steer, vel, pos_t, vel_t);
}

extern "C" int rvb_ackermann(const float* lin, int64_t lin_stride, const float* ang, int64_t ang_stride, int64_t N,
                             float* steer, float* vel, float* pos_targets, float* vel_targets, int sem, void* stream) {
    if (N <= 0) return RVB_OK;
    RVB_REQUIRE(lin && ang && steer && vel, "rvb_ackermann: null pointer");
    RVB_REQUIRE(lin_stride >= 0 && ang_stride >= 0, "rvb_ackermann: negative stride");
    ackermann_kernel<<<(unsigned)ceil_div(N, 256), 256, 0, as_stream(stream)>>>(lin, lin_stride, ang, ang_stride, N, steer,
                                                                              vel, pos_targets, vel_targets, sem);
    RVB_LAUNCH_CHECK();
    return RVB_OK;
}

// ---------------------------------------------------------------- Memory.input_state
__global__ void history_push_kernel(float* __restrict__ hist, int64_t N, int H, const float* __restrict__ newest,
                                    int64_t stride) {
    int64_t n = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (n >= N) return;
    float* h = hist + n * H;
    for (int i = H - 1; i > 0; --i) h[i] = h[i - 1];
    h[0] = newest[n * stride];
}

extern "C" int rvb_history_push(float* hist, int64_t N, int64_t H, const float* newest, int64_t newest_stride,
                                void* stream) {
    if (N <= 0) return RVB_OK;
    RVB_REQUIRE(hist && newest, "rvb_history_push: null pointer");
    RVB_REQUIRE(H >= 1 && H <= 64, "rvb_history_push: horizon out of range");
    history_push_kernel<<<(unsigned)ceil_div(N, 256), 256, 0, as_stream(stream)>>>(hist, N, (int)H, newest, newest_stride);
    RVB_LAUNCH_CHECK();
    return RVB_OK;
}

// ---------------------------------------------------------------- observation columns 0..3 + heading
__global__ void obs_proprio_kernel(const float* __restrict__ pos, const float* __restrict__ euler,
                                   const float* __restrict__ target, const float* __restrict__ lin_now,
                                   const float* __restrict__ ang_now, int64_t N, float* __restrict__ obs, int64_t ld,
                                   float* __restrict__ heading, int sem) {
    int64_t n = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (n >= N) return;
    obs_proprio_dev(pos[n * 3 + 0], pos[n * 3 + 1], euler[n * 3 + 2], target[n * 3 + 0], target[n * 3 + 1], lin_now[n], ang_now[n],
                    sem, obs + n * ld, heading ? heading + n : nullptr);
}

extern "C" int rvb_obs_proprio(const float* pos, const float* euler, const float* target, const float* lin_now,
                               const float* ang_now, int64_t N, float* obs, int64_t obs_ld, float* heading, int sem,
                               void* stream) {
    if (N <= 0) return RVB_OK;
    RVB_REQUIRE(pos && euler && target && lin_now && ang_now && obs, "rvb_obs_proprio: null pointer");
    RVB_REQUIRE(obs_ld >= 4, "rvb_obs_proprio: obs_ld < 4");
    obs_proprio_kernel<<<(unsigned)ceil_div(N, 256), 256, 0, as_stream(stream)>>>(pos, euler, target, lin_now, ang_now, N,
                                                                                obs, obs_ld, heading, sem);
    RVB_LAUNCH_CHECK();
    return RVB_OK;
}

__global__ void obs_gather_kernel(const __half* __restrict__ dist, int64_t P, int64_t N, const int64_t* __restrict__ idx,
                                  int n_idx, float* __restrict__ obs, int64_t ld, int64_t col0) {
    const int64_t n = blockIdx.y;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_idx) return;
    const __half d = dist[n * P + idx[i]];
    obs[n * ld + col0 + i] = __half2float(h_mul(d, __float2half_rn(0.5f)));
}

extern "C" int rvb_obs_gather(const uint16_t* dist, int64_t P, int64_t N, const int64_t* idx, int64_t n_idx, float* obs,
                              int64_t obs_ld, int64_t col0, void* stream) {
    if (N <= 0 || n_idx <= 0) return RVB_OK;
    RVB_REQUIRE(dist && idx && obs, "rvb_obs_gather: null pointer");
    RVB_REQUIRE(N <= 65535, "rvb_obs_gather: at most 65535 envs per call");
    dim3 grid((unsigned)ceil_div(n_idx, 256), (unsigned)N);
    obs_gather_kernel<<<grid, 256, 0, as_stream(stream)>>>((const __half*)dist, P, N, idx, (int)n_idx, obs, obs_ld, col0);
    RVB_LAUNCH_CHECK();
    return RVB_OK;
}

// ---------------------------------------------------------------- calculate_metrics + is_done
#define RR_THREADS 256

extern "C" int64_t rvb_stats_scratch_len(int64_t N) { return ceil_div(N > 0 ? N : 1, RR_THREADS) * RVB_N_STATS; }

__global__ void __launch_bounds__(RR_THREADS)
reward_reset_kernel(rvb_reward_params p, const float* __restrict__ pos, const float* __restrict__ target,
                    const float* __restrict__ heading, const float* __restrict__ rover_rot,
                    const float* __restrict__ lin_p, const float* __restrict__ lin_prev_p, const float* __restrict__ ang_p,
                    const float* __restrict__ ang_prev_p, const float* __restrict__ joints,
                    const int64_t* __restrict__ progress, const int64_t* __restrict__ rock, int64_t N, int64_t hs,
                    float* __restrict__ rew, int64_t* __restrict__ reset, float* __restrict__ ex_pos,
                    int64_t* __restrict__ ex_col, float* __restrict__ ex_up, float* __restrict__ ex_head,
                    float* __restrict__ ex_motion, float* __restrict__ ex_goal, double* __restrict__ partial) {
    const int64_t n = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    double s[RVB_N_STATS];
#pragma unroll
    for (int i = 0; i < RVB_N_STATS; ++i) s[i] = 0.0;
    if (n < N) {
        const float lin = lin_p[n * hs], lin_prev = lin_prev_p[n * hs], ang = ang_p[n * hs], ang_prev = ang_prev_p[n * hs];
        const float ddx = F::sub(target[n * 3 + 0], pos[n * 3 + 0]), ddy = F::sub(target[n * 3 + 1], pos[n * 3 + 1]);
        const float td = __fsqrt_rn(F::add(F::mul(ddx, ddx), F::mul(ddy, ddy)));                 // rover.py:482
        const float head_pen = F::mul(lin < 0.f ? -1.f : 0.f, p.heading_contraint_reward);       // :486
        const float up = F::mul(F::add(F::add(fabsf(joints[n * 13 + 0]), fabsf(joints[n * 13 + 1])),
                                       fabsf(joints[n * 13 + 2])), p.boogie_contraint_reward);   // :492
        const float h = heading[n];
        const float goal_pen = (fabsf(h) > 2.f) ? -fabsf(F::mul(F::mul(h, 0.3f), p.goal_angle_reward)) : 0.f;   // :495
        const float dl = fabsf(F::sub(F::mul(lin, 3.f), F::mul(3.f, lin_prev)));
        const float da = fabsf(F::sub(F::mul(ang, 3.f), F::mul(3.f, ang_prev)));
        const float p1 = (dl > 0.05f) ? F::mul(dl, dl) : 0.f;                                    // :498
        const float p2 = (da > 0.05f) ? F::mul(da, da) : 0.f;
        float motion = F::mul(F::mul(p1, p1), p.motion_contraint_reward);                        // :500
        motion = F::add(motion, F::mul(F::mul(p2, p2), p.motion_contraint_reward));              // :502
        float pos_rew = F::mul(__fdiv_rn(1.f, F::add(1.f, F::mul(F::mul((float)(0.33 * 0.33), td), td))), p.pos_reward);
        const int64_t prog = progress[n];
        if (td <= 0.18f) pos_rew = F::mul(1.03f, (float)((int64_t)p.max_episode_length - prog));  // :506
        float reward = F::add(F::add(F::add(pos_rew, head_pen), motion), goal_pen);              // :512
        const bool col = (p.curriculum_level >= 2) && rock && rock[n] == 1;
        if (col) reward = F::sub(reward, 300.f);                                                 // :519
        reward = div_scalar(reward, 3000.f, 1.0f / 3000.f, p.sem);                               // :522
        rew[n] = reward;
        if (ex_pos) ex_pos[n] = pos_rew;
        if (ex_col) ex_col[n] = col ? p.num_envs_total : 0;                                      // :517
        if (ex_up) ex_up[n] = up;
        if (ex_head) ex_head[n] = head_pen;
        if (ex_motion) ex_motion[n] = motion;
        if (ex_goal) ex_goal[n] = goal_pen;
        // is_done (:610-647)
        const bool timeout = prog >= (int64_t)p.max_episode_length;
        const float lim = (float)(0.78 * 1.5);
        const bool tilt = fabsf(rover_rot[n * 3 + 0]) >= lim || fabsf(rover_rot[n * 3 + 1]) >= lim;
        const bool far_away = td >= 11.f, goal = td <= 0.18f;
        const bool r = timeout || tilt || far_away || goal || col;
        reset[n] = r ? 1 : 0;
        s[0] = 1.0; s[1] = reward; s[2] = pos_rew; s[3] = col; s[4] = up; s[5] = head_pen; s[6] = motion; s[7] = goal_pen;
        s[8] = r; s[9] = timeout; s[10] = tilt; s[11] = far_away; s[12] = goal; s[13] = col; s[14] = td;
    }
    if (!partial) return;
    // fixed-order block reduction: warp shuffle tree, then warp 0 adds the 8 warp sums in order
    __shared__ double sm[RR_THREADS / 32][RVB_N_STATS];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int i = 0; i < RVB_N_STATS; ++i) {
        double v = s[i];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
        if (lane == 0) sm[warp][i] = v;
    }
    __syncthreads();
    if (threadIdx.x < RVB_N_STATS) {
        double v = 0.0;
        for (int w = 0; w < RR_THREADS / 32; ++w) v += sm[w][threadIdx.x];
        partial[(int64_t)blockIdx.x * RVB_N_STATS + threadIdx.x] = v;
    }
}

__global__ void stats_final_kernel(const double* __restrict__ partial, int64_t nblocks, double* __restrict__ stats) {
    // one block of 32 x 16 threads; each of 32 strided partial sums is added in a fixed order
    __shared__ double sm[32][RVB_N_STATS];
    const int i = threadIdx.x % RVB_N_STATS, r = threadIdx.x / RVB_N_STATS;
    double v = 0.0;
    for (int64_t b = r; b < nblocks; b += 32) v += partial[b * RVB_N_STATS + i];
    sm[r][i] = v;
    __syncthreads();
    if (r == 0) {
        double t = 0.0;
        for (int k = 0; k < 32; ++k) t += sm[k][i];
        stats[i] = t;
    }
}

int launch_reward_reset(const rvb_reward_params* p, const float* pos, const float* target, const float* heading,
                        const float* rover_rot, const float* lin, const float* lin_prev, const float* ang,
                        const float* ang_prev, int64_t hs, const float* joints, const int64_t* progress,
                        const int64_t* rock_collision, int64_t N, float* rew, int64_t* reset, float* ex_pos_reward,
                        int64_t* ex_collision, float* ex_uprightness, float* ex_heading, float* ex_motion,
                        float* ex_goal_angle, double* stats, double* stats_scratch, cudaStream_t st) {
    RVB_REQUIRE(p && pos && target && heading && rover_rot && lin && lin_prev && ang && ang_prev && joints && progress &&
                    rew && reset, "rvb_reward_reset: null pointer");
    RVB_REQUIRE(p->curriculum_level < 2 || rock_collision, "rvb_reward_reset: curriculum_level >= 2 needs rock_collision");
    RVB_REQUIRE(!stats || stats_scratch, "rvb_reward_reset: stats needs stats_scratch");
    if (N <= 0) {
        if (stats) RVB_CUDA(cudaMemsetAsync(stats, 0, sizeof(double) * RVB_N_STATS, st));
        return RVB_OK;
    }
    const int64_t blocks = ceil_div(N, RR_THREADS);
    reward_reset_kernel<<<(unsigned)blocks, RR_THREADS, 0, st>>>(*p, pos, target, heading, rover_rot, lin, lin_prev, ang,
                                                                ang_prev, joints, progress, rock_collision, N, hs, rew, reset,
                                                                ex_pos_reward, ex_collision, ex_uprightness, ex_heading,
                                                                ex_motion, ex_goal_angle, stats ? stats_scratch : nullptr);
    RVB_LAUNCH_CHECK();
    if (stats) {
        stats_final_kernel<<<1, 32 * RVB_N_STATS, 0, st>>>(stats_scratch, blocks, stats);
        RVB_LAUNCH_CHECK();
    }
    return RVB_OK;
}

extern "C" int rvb_reward_reset(const rvb_reward_params* p, const float* pos, const float* target, const float* heading,
                                const float* rover_rot, const float* lin, const float* lin_prev, const float* ang,
                                const float* ang_prev, const float* joints, const int64_t* progress,
                                const int64_t* rock_collision, int64_t N, float* rew, int64_t* reset, float* ex_pos_reward,
                                int64_t* ex_collision, float* ex_uprightness, float* ex_heading, float* ex_motion,
                                float* ex_goal_angle, double* stats, double* stats_scratch, void* stream) {
    return launch_reward_reset(p, pos, target, heading, rover_rot, lin, lin_prev, ang, ang_prev, 1, joints, progress,
                               rock_collision, N, rew, reset, ex_pos_reward, ex_collision, ex_uprightness, ex_heading, ex_motion,
                               ex_goal_angle, stats, stats_scratch, as_stream(stream));
}
