// Per-step observation epilogues the reference's authors toggled by hand (SURVEY.md 8f-4), one pass over obs_buf each:
//
//   rvb_obs_hooks       rover.py:326-329 (commented out in the reference, applied here in its order when enabled):
//                         obs[:, 4:] += sqrt(0.20) * randn            -> noise_std
//                         obs[:, 4:]  = F.dropout(obs[:, 4:], p=0.1)  -> dropout_p (kept values scaled by 1/(1-p))
//                         obs         = obs - 0.02                    -> offset (every column)
//                         obs[:, remove_idx + 4] = 0                  -> zero_mask (u8 per column)
//   rvb_teacher_record  rover.py:298-300,364,374-375: one row [reset_info, a0, a1, obs...] per env of the teacher data set.
//
// Random numbers: torch's generator stream (one randn tensor per step, then one bernoulli tensor) cannot be reproduced
// per element on a sharded device path; like the reset path (stones.cu) the draws are Philox4x32-10 with
// counter = (global env id lo, hi, column, epoch lo), key = (seed lo, seed hi ^ epoch hi): x0, x1 -> Box-Muller normal
// (u1 = ((x0 >> 8) + 1) 2^-24 in (0, 1], u2 = (x1 >> 8) 2^-24), x2 -> dropout (drop iff (x2 >> 8) < round(p 2^24)) --
// a pure function of (seed, epoch, env, column), independent of how envs are sharded.  oracle/hooks_oracle.py restates it.
// HBM-streaming: 2 x 4 B per element (28.7 MB each way at 4096 envs); one thread per element, coalesced along columns.
#include "common.cuh"

__global__ void obs_hooks_kernel(float* __restrict__ obs, int64_t obs_ld, int64_t N, int C, int col0, float noise_std,
                                 uint32_t drop_thr, float keep_scale, float offset, const uint8_t* __restrict__ zero_mask,
                                 uint32_t k0, uint32_t k1, uint32_t epoch_lo, int64_t env_offset) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t n = blockIdx.y;
    if (c >= C) return;
    float v = obs[n * obs_ld + c];
    if (c >= col0 && (noise_std != 0.f || drop_thr != 0u)) {
        const uint64_t gid = (uint64_t)(n + env_offset);
        uint32_t x0, x1, x2, x3;
        philox4x32_10((uint32_t)gid, (uint32_t)(gid >> 32), (uint32_t)c, epoch_lo, k0, k1, x0, x1, x2, x3);
        if (noise_std != 0.f) {
            const float u1 = __fmul_rn((float)((x0 >> 8) + 1u), 5.9604644775390625e-8f);
            const float u2 = __fmul_rn((float)(x1 >> 8), 5.9604644775390625e-8f);
            const float r = sqrtf(__fmul_rn(-2.f, logf(u1)));
            const float z = __fmul_rn(r, cosf(__fmul_rn(6.2831854820251465f, u2)));
            v = __fadd_rn(v, __fmul_rn(noise_std, z));
        }
        if (drop_thr != 0u) v = ((x2 >> 8) < drop_thr) ? 0.f : __fmul_rn(v, keep_scale);
    }
    v = __fsub_rn(v, offset);
    if (zero_mask && zero_mask[c]) v = 0.f;
    obs[n * obs_ld + c] = v;
}

extern "C" int rvb_obs_hooks(float* obs, int64_t obs_ld, int64_t N, int64_t C, int64_t col0, float noise_std, float dropout_p,
                             float offset, const uint8_t* zero_mask, uint64_t seed, uint64_t epoch, int64_t env_offset,
                             void* stream) {
    if (N <= 0 || C <= 0) return RVB_OK;
    RVB_REQUIRE(obs, "rvb_obs_hooks: null pointer");
    RVB_REQUIRE(obs_ld >= C && C < (1 << 30) && col0 >= 0 && N <= 0x7fffffff, "rvb_obs_hooks: bad shape");
    RVB_REQUIRE(dropout_p >= 0.f && dropout_p < 1.f && noise_std >= 0.f, "rvb_obs_hooks: dropout_p must be in [0,1), noise_std >= 0");
    RVB_REQUIRE(env_offset >= 0, "rvb_obs_hooks: negative env_offset");
    const uint32_t thr = (uint32_t)llrintf(dropout_p * 16777216.0f);
    const float keep = 1.0f / (1.0f - dropout_p);
    // grid.y = env: up to 65,535 per launch
    for (int64_t n0 = 0; n0 < N; n0 += 65535) {
        const int64_t nb = (N - n0 < 65535) ? N - n0 : 65535;
        dim3 grid((unsigned)ceil_div(C, 256), (unsigned)nb);
        obs_hooks_kernel<<<grid, 256, 0, as_stream(stream)>>>(obs + n0 * obs_ld, obs_ld, nb, (int)C, (int)(col0 < C ? col0 : C), noise_std,
                                                              thr, keep, offset, zero_mask, (uint32_t)seed,
                                                              (uint32_t)(seed >> 32) ^ (uint32_t)(epoch >> 32), (uint32_t)epoch,
                                                              env_offset + n0);
    }
    RVB_LAUNCH_CHECK();
    return RVB_OK;
}

// record[n] = [reset_info[n], actions[n,0], actions[n,1], obs[n, 0..C)]   (rover.py:299,364,374-375)
__global__ void teacher_record_kernel(const float* __restrict__ reset_info, const float* __restrict__ actions, int64_t actions_ld,
                                      const float* __restrict__ obs, int64_t obs_ld, int C, float* __restrict__ record,
                                      int64_t record_ld) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;      // column of the record row
    const int64_t n = blockIdx.y;
    if (c >= C + 3) return;
    float v;
    if (c == 0) v = reset_info[n];
    else if (c < 3) v = actions[n * actions_ld + (c - 1)];
    else v = obs[n * obs_ld + (c - 3)];
    record[n * record_ld + c] = v;
}

extern "C" int rvb_teacher_record(const float* reset_info, const float* actions, int64_t actions_ld, const float* obs,
                                  int64_t obs_ld, int64_t N, int64_t C, float* record, int64_t record_ld, void* stream) {
    if (N <= 0) return RVB_OK;
    RVB_REQUIRE(reset_info && actions && obs && record, "rvb_teacher_record: null pointer");
    RVB_REQUIRE(C > 0 && C < (1 << 30) && obs_ld >= C && record_ld >= C + 3 && actions_ld >= 2, "rvb_teacher_record: bad shape");
    for (int64_t n0 = 0; n0 < N; n0 += 65535) {
        const int64_t nb = (N - n0 < 65535) ? N - n0 : 65535;
        dim3 grid((unsigned)ceil_div(C + 3, 256), (unsigned)nb);
        teacher_record_kernel<<<grid, 256, 0, as_stream(stream)>>>(reset_info + n0, actions + n0 * actions_ld, actions_ld,
                                                                   obs + n0 * obs_ld, obs_ld, (int)C, record + n0 * record_ld, record_ld);
    }
    RVB_LAUNCH_CHECK();
    return RVB_OK;
}

// The recorder on the packed observation of the fused step (rvb_step_io.obs_h16): the row's lead [reset_info, a0, a1, proprio[0..p)]
// in f32, then the E heightmap columns -- widened with __half2float (what torch's .float() does on the device, so the row is bit for
// bit teacher_record_kernel's on cat(proprio, heightmap.float())) or copied as fp16 bits into their own block (rec16).
// HBM-streaming.  One CTA per (row, chunk of TRP_CHUNK columns); the shipped row (1746 columns) is one chunk.  A 1746-half row is
// only 4-byte aligned and every pointer and row stride may be odd, so the chunk is staged in shared memory: 16-byte loads aligned
// on the source, then 16-byte streaming stores aligned on the destination, scalar accesses only for the partial lines at either end.
// Bytes per env-step: 4 (reset) + 8 (actions) + 4p (proprio) + 2E read; 4(3 + p + E) written (f32 block) or 4(3 + p) + 2E (rec16).
constexpr int TRP_THREADS = 128;
constexpr int TRP_LINES = 2;                                      // 16-byte source lines per thread
constexpr int TRP_CHUNK = TRP_LINES * TRP_THREADS * 8 - 8;       // 2040 columns: at any alignment they span <= 256 lines

template <bool WIDEN>
__global__ void __launch_bounds__(TRP_THREADS)
teacher_record_packed_kernel(const float* __restrict__ reset_info, const float* __restrict__ actions, int64_t actions_ld,
                             const float* __restrict__ proprio, int64_t proprio_ld, int p, const uint16_t* __restrict__ hm,
                             int64_t hm_ld, int E, float* __restrict__ rec, int64_t rec_ld, uint16_t* __restrict__ rec16,
                             int64_t rec16_ld) {
    __shared__ __align__(16) uint16_t s[TRP_CHUNK + 8];
    const int64_t n = blockIdx.y;
    const int j0 = blockIdx.x * TRP_CHUNK;
    const int m = min(TRP_CHUNK, E - j0);
    float* row = rec + n * rec_ld;
    const int t = threadIdx.x;
    if (blockIdx.x == 0 && t < 3 + p) {
        float v;
        if (t == 0) v = reset_info[n];
        else if (t < 3) v = actions[n * actions_ld + (t - 1)];
        else v = proprio[n * proprio_ld + (t - 3)];
        row[t] = v;
    }
    // column j of the chunk goes to s[a + j]: the source's 16-byte lines land on 16-byte lines of s
    const uint16_t* src = hm + n * hm_ld + j0;
    const int a = (int)((reinterpret_cast<uintptr_t>(src) >> 1) & 7);
    uint4 v[TRP_LINES];
#pragma unroll
    for (int k = 0; k < TRP_LINES; ++k) {                   // every full line's load is in flight before the first is stored
        const int lo = (t + k * TRP_THREADS) * 8 - a;
        if (lo >= 0 && lo + 8 <= m) v[k] = __ldg(reinterpret_cast<const uint4*>(src + lo));
    }
#pragma unroll
    for (int k = 0; k < TRP_LINES; ++k) {
        const int l = t + k * TRP_THREADS, lo = l * 8 - a;
        if (lo >= 0 && lo + 8 <= m) *reinterpret_cast<uint4*>(s + l * 8) = v[k];
        else
            for (int q = max(lo, 0); q < min(lo + 8, m); ++q) s[a + q] = src[q];
    }
    __syncthreads();
    if (WIDEN) {
        float* dst = row + 3 + p + j0;
        const int b = (int)((reinterpret_cast<uintptr_t>(dst) >> 2) & 3);
        for (int l = t; l < (b + m + 3) >> 2; l += TRP_THREADS) {
            const int lo = l * 4 - b;
            if (lo >= 0 && lo + 4 <= m) {
                const uint16_t* h = s + a + lo;
                __stcs(reinterpret_cast<float4*>(dst + lo), make_float4(__half2float(__ushort_as_half(h[0])), __half2float(__ushort_as_half(h[1])),
                                                                        __half2float(__ushort_as_half(h[2])), __half2float(__ushort_as_half(h[3]))));
            } else {
                for (int q = max(lo, 0); q < min(lo + 4, m); ++q) dst[q] = __half2float(__ushort_as_half(s[a + q]));
            }
        }
    } else {
        uint16_t* dst = rec16 + n * rec16_ld + j0;
        const int b = (int)((reinterpret_cast<uintptr_t>(dst) >> 1) & 7);
        for (int l = t; l < (b + m + 7) >> 3; l += TRP_THREADS) {
            const int lo = l * 8 - b;
            if (lo >= 0 && lo + 8 <= m) {
                uint4 w;
                if (a == b) {
                    w = *reinterpret_cast<const uint4*>(s + l * 8);
                } else {
                    const uint16_t* h = s + a + lo;
                    w = make_uint4(h[0] | (uint32_t)h[1] << 16, h[2] | (uint32_t)h[3] << 16, h[4] | (uint32_t)h[5] << 16,
                                   h[6] | (uint32_t)h[7] << 16);
                }
                __stcs(reinterpret_cast<uint4*>(dst + lo), w);
            } else {
                for (int q = max(lo, 0); q < min(lo + 8, m); ++q) dst[q] = s[a + q];
            }
        }
    }
}

extern "C" int rvb_teacher_record_packed(const float* reset_info, const float* actions, int64_t actions_ld, const float* proprio,
                                         int64_t proprio_ld, int64_t p, const uint16_t* heightmap, int64_t heightmap_ld, int64_t E,
                                         int64_t N, float* rec, int64_t rec_ld, uint16_t* rec16, int64_t rec16_ld, void* stream) {
    if (N == 0) return RVB_OK;
    RVB_REQUIRE(reset_info && actions && heightmap && rec && (proprio || p == 0), "rvb_teacher_record_packed: null pointer");
    RVB_REQUIRE(p >= 0 && p <= 8, "rvb_teacher_record_packed: p must be in 0..8");
    RVB_REQUIRE(N > 0 && E > 0 && E < (1 << 30), "rvb_teacher_record_packed: bad shape");
    RVB_REQUIRE(actions_ld >= 2 && proprio_ld >= p && heightmap_ld >= E && rec_ld >= 3 + p + (rec16 ? 0 : E) && (!rec16 || rec16_ld >= E),
                "rvb_teacher_record_packed: short row");
    RVB_REQUIRE(!((uintptr_t)reset_info & 3) && !((uintptr_t)actions & 3) && !((uintptr_t)proprio & 3) && !((uintptr_t)heightmap & 1) &&
                    !((uintptr_t)rec & 3) && !((uintptr_t)rec16 & 1),
                "rvb_teacher_record_packed: misaligned pointer");
    const unsigned chunks = (unsigned)ceil_div(E, TRP_CHUNK);
    for (int64_t n0 = 0; n0 < N; n0 += 65535) {             // grid.y = row: up to 65,535 per launch
        const int64_t nb = (N - n0 < 65535) ? N - n0 : 65535;
        const dim3 grid(chunks, (unsigned)nb);
        const float* pr = proprio ? proprio + n0 * proprio_ld : nullptr;
        if (rec16)
            teacher_record_packed_kernel<false><<<grid, TRP_THREADS, 0, as_stream(stream)>>>(
                reset_info + n0, actions + n0 * actions_ld, actions_ld, pr, proprio_ld, (int)p, heightmap + n0 * heightmap_ld,
                heightmap_ld, (int)E, rec + n0 * rec_ld, rec_ld, rec16 + n0 * rec16_ld, rec16_ld);
        else
            teacher_record_packed_kernel<true><<<grid, TRP_THREADS, 0, as_stream(stream)>>>(
                reset_info + n0, actions + n0 * actions_ld, actions_ld, pr, proprio_ld, (int)p, heightmap + n0 * heightmap_ld,
                heightmap_ld, (int)E, rec + n0 * rec_ld, rec_ld, nullptr, 0);
    }
    RVB_LAUNCH_CHECK();
    return RVB_OK;
}
