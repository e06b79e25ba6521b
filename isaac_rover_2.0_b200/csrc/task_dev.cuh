// Per-env fp32 task arithmetic shared by task.cu (one kernel per reference call) and step.cu (fused env step).
#pragma once
#include <math_constants.h>

#include "common.cuh"

// calculate_metrics + is_done with the episode statistics (task.cu; rvb_reward_reset and the end of rvb_env_post).
// hs: element stride between consecutive envs in lin / lin_prev / ang / ang_prev (1 for packed columns, H for [N,H] histories)
int launch_reward_reset(const rvb_reward_params* p, const float* pos, const float* target, const float* heading,
                        const float* rover_rot, const float* lin, const float* lin_prev, const float* ang,
                        const float* ang_prev, int64_t hs, const float* joints, const int64_t* progress,
                        const int64_t* rock_collision, int64_t N, float* rew, int64_t* reset, float* ex_pos_reward,
                        int64_t* ex_collision, float* ex_uprightness, float* ex_heading, float* ex_motion,
                        float* ex_goal_angle, double* stats, double* stats_scratch, cudaStream_t st);

#define PI_F32 3.1415927410125732f   // tensor_quat_to_euler.py:4

using F = Ops<float>;

// torch divides a tensor by a Python scalar with a true division on the CPU and with a multiplication by
// fp32(1/scalar) on CUDA (ATen div_true_kernel_cuda); `inv` must be 1.0f / c computed in fp32.
__device__ __forceinline__ float div_scalar(float v, float c, float inv, int sem) {
    return sem == RVB_SEM_TORCH_CPU ? __fdiv_rn(v, c) : __fmul_rn(v, inv);
}

// ---------------------------------------------------------------- tensor_quat_to_eul
__device__ __forceinline__ void quat_to_euler_dev(float w, float x, float y, float z, float& roll, float& pitch,
                                                  float& yaw) {
    const float sinr = F::mul(2.f, F::add(F::mul(w, x), F::mul(y, z)));
    const float cosr = F::sub(1.f, F::mul(2.f, F::add(F::mul(x, x), F::mul(y, y))));
    roll = atan2f(sinr, cosr);
    const float sinp = F::mul(2.f, F::sub(F::mul(w, y), F::mul(z, x)));
    // sign(sinp - 1) >= 0  <=>  sinp - 1 >= 0 (NaN -> false)   (:23)
    pitch = (F::sub(sinp, 1.f) >= 0.f) ? copysignf(F::mul(PI_F32, 0.5f), sinp) : asinf(sinp);
    const float siny = F::mul(2.f, F::add(F::mul(w, z), F::mul(x, y)));
    const float cosy = F::sub(1.f, F::mul(2.f, F::add(F::mul(y, y), F::mul(z, z))));
    yaw = atan2f(siny, cosy);
}

static __constant__ float c_wheel_xy[6][2] = {{-0.385f, 0.438f}, {0.385f, 0.438f},   {-0.447f, 0.0f},
                                       {0.447f, 0.0f},    {-0.385f, -0.411f}, {0.385f, -0.411f}};   // kinematics.py:20-25

// Ackermann for one env (kinematics.py:14-67): steering angles st[6] and motor velocities ve[6] (FL,FR,ML,MR,RL,RR)
__device__ __forceinline__ void ackermann_dev(float lin, const float ang, int sem, float* st, float* ve) {
    float P = copysignf(__fdiv_rn(lin, ang), -ang);                      // :34-35
    P = (fabsf(P) > 0.45f) ? P : 0.f;                                    // :38
    lin = (P != 0.f) ? lin : 0.f;                                        // :39
#pragma unroll
    for (int w = 0; w < 6; ++w) {
        const float wx = c_wheel_xy[w][0], wy = c_wheel_xy[w][1];
        const float ddx = F::sub(P, wx), ddy = F::sub(0.f, wy);
        const float dist = __fsqrt_rn(F::add(F::mul(ddx, ddx), F::mul(ddy, ddy)));   // :43
        const float side = (w & 1) ? 1.f : -1.f;
        const float omega = (lin != 0.f) ? copysignf(ang, lin) : F::mul(ang, side);  // :49-52
        float v = F::mul(dist, omega);
        v = (dist > 1000.f) ? lin : v;                                   // :58
        ve[w] = div_scalar(v, 0.2f, 1.0f / 0.2f, sem);                   // :61
        float a = atan2f(wy, F::sub(wx, P));                             // :63
        a = (a < (float)(-3.14 / 2)) ? F::add(a, (float)M_PI) : a;       // :64
        a = (a > (float)(3.14 / 2)) ? F::sub(a, (float)M_PI) : a;        // :65
        st[w] = a;
    }
}

__device__ __forceinline__ void ackermann_store(int64_t n, const float* st, const float* ve, float* __restrict__ steer,
                                                float* __restrict__ vel, float* __restrict__ pos_t, float* __restrict__ vel_t) {
#pragma unroll
    for (int w = 0; w < 6; ++w) {
        if (steer) steer[n * 6 + w] = st[w];
        if (vel) vel[n * 6 + w] = ve[w];
    }
    if (pos_t) {   // rover.py:400-403  FR, RR, FL, RL
        pos_t[n * 4 + 0] = st[1]; pos_t[n * 4 + 1] = st[5]; pos_t[n * 4 + 2] = st[0]; pos_t[n * 4 + 3] = st[4];
    }
    if (vel_t) {   // rover.py:404-409  FR, CR, RR, FL, CL, RL
        vel_t[n * 6 + 0] = ve[1]; vel_t[n * 6 + 1] = ve[3]; vel_t[n * 6 + 2] = ve[5];
        vel_t[n * 6 + 3] = ve[0]; vel_t[n * 6 + 4] = ve[2]; vel_t[n * 6 + 5] = ve[4];
    }
}

// proprioceptive observation columns + heading for one env (rover.py:279-283, 320-323)
__device__ __forceinline__ void obs_proprio_dev(float px, float py, float yaw, float tgx, float tgy, float lin_now, float ang_now,
                                                int sem, float* __restrict__ obs_row, float* __restrict__ heading_out) {
    const float dx = cosf(yaw), dy = sinf(yaw);                                    // rover.py:280-281
    const float tx = F::sub(tgx, px), ty = F::sub(tgy, py);
    const float h = -atan2f(F::sub(F::mul(tx, dy), F::mul(ty, dx)), F::add(F::mul(tx, dx), F::mul(ty, dy)));   // :283
    if (heading_out) *heading_out = h;
    const float nrm = __fsqrt_rn(F::add(F::mul(tx, tx), F::mul(ty, ty)));
    obs_row[0] = div_scalar(nrm, 9.f, 1.0f / 9.f, sem);                            // :320
    obs_row[1] = div_scalar(h, (float)M_PI, 1.0f / (float)M_PI, sem);              // :321
    obs_row[2] = lin_now;
    obs_row[3] = ang_now;
}
