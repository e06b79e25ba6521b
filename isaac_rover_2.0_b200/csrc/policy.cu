// Policy-inference epilogue (SURVEY.md 8f-3): the direct consumer of obs_buf.
//
// Replaces StochasticActorHeightmap.compute / DeterministicHeightmap.compute (learning/model.py:152-195, 197-241):
//   x0 = encoder0(obs[:, p : p+S])            Linear(S,80)  + act, Linear(80,60) + act      (model.py:118-144,186)
//   x1 = encoder1(obs[:, p+S : p+S+D])        Linear(D,80)  + act, Linear(80,60) + act      (model.py:187)
//   x  = cat(obs[:, 0:p], x0, x1)             (model.py:188-189)
//   x  = Linear(124,256)+act, Linear(256,160)+act, Linear(160,128)+act, Linear(128,A) [+ Tanh for the actor] (model.py:169-177,190-191)
// with the layer widths the reference hard-wires (train.py:95, cfg/trainSKRL/RoverPPOSKRL.yaml:4-9).
//
// Arithmetic: the reference runs torch fp32 nn.Linear (TF32 is off by default for matmuls), and a single-pass bf16/TF32
// contraction would change the answer by 1e-3.  The default path (policy_l1_tc_kernel + policy_tail_tc_kernel, below) runs the
// network on tcgen05 with every operand split into tf32 hi + lo parts, which is fp32-grade.  policy_forward_kernel, an fp32 FFMA2
// chain, is the fall-back for the shapes the tensor-core path refuses (tc_usable) and what rvb_policy_variant(1) forces.  Both
// differ from cuBLAS in the summation order (unspecified there).  Tests hold the tensor-core path to an fp64 oracle bit for bit
// on exact probes (tests/policy_probe.py) and, on dense random inputs, within max(32 x the error of torch fp32, 1e-7).
//
// policy_forward_kernel: sums are accumulated in k order per output with packed fp32 FMAs (ffma2, IEEE fma per element).
// One CTA of 256 threads per tile of TM = 32 envs; every activation of the tile stays in shared memory from the
// observation row to the action (k-major [k][env], row stride 36 floats), so obs is read exactly once from HBM/L2 and
// nothing but the A outputs is written.  Weights are re-packed once per handle into k-major, 32-column-padded panels
// (Wt[k][OUTP]) that every CTA streams from L2 through a 16 KB staging buffer.  Thread (mg = warp, ng = lane) owns
// 4 envs x CN columns {ng + 32 j}: per k one broadcast 128-bit activation load + CN conflict-free weight loads feed
// 4 CN FMAs.  99 KB shared memory -> 2 CTAs per SM.
#include <memory>
#include <new>
#include <stdlib.h>
#include <type_traits>

#include "common.cuh"

#define PL_TM 32
#define PL_LDA 36
#define PL_THREADS 256
#define PL_WS_FLOATS 4096          // weight staging buffer: KC x OUTP floats
#define PL_E1 80
#define PL_E2 60
#define PL_M1 256
#define PL_M2 160
#define PL_M3 128
#define PL_MAX_PROPRIO 8
#define PL_MAX_HEAD 4

static inline int pad32(int n) { return (n + 31) / 32 * 32; }

struct PackedLinear {
    float* wt;     // [in][outp]  k-major, zero padded columns
    float* bias;   // [outp]
    int in, out, outp;
};

// What the kernel reads: a copy lives at the start of the handle's device allocation, so one launch can serve two
// networks (blockIdx.y) without indexing kernel parameters dynamically.
struct PolicyDev {
    PackedLinear es1, es2, ed1, ed2, m1, m2, m3;
    float* head_w;   // [A][PL_M3]  torch layout
    float* head_b;   // [A]
    int n_proprio, n_sparse, n_dense, n_head;
    int act, head_tanh;
    // tensor-core path of the two first encoder layers (policy_l1_tc_kernel): the torch-layout weights [80][K] split into tf32
    // hi + lo parts, K padded to chunks of 32, stored as the exact shared-memory image of each chunk (K-major, SWIZZLE_128B):
    // [chunk][part][80 rows][32 floats]
    const float* tc_img_s;
    const float* tc_img_d;
    int tc_cs, tc_cd;     // chunks of the sparse / dense encoder
    const float* tc_tail; // weight stream of the remaining layers in the order policy_tail_tc_kernel consumes it (TT_* below)
};

struct rvb_policy : PolicyDev {
    int device;
    float* storage;        // the one allocation everything points into: [PolicyDev | panels | head]
    int64_t storage_floats;
    const PolicyDev* dev;  // = storage
};
#define PL_DESC_FLOATS 128   // room reserved for the descriptor (keeps the panels 512-byte aligned)
static_assert(sizeof(PolicyDev) <= PL_DESC_FLOATS * sizeof(float), "descriptor does not fit its slot");

__device__ __forceinline__ float pl_act(float v, int kind) {
    switch (kind) {
        case RVB_ACT_LEAKYRELU: return v > 0.f ? v : __fmul_rn(v, 0.01f);   // nn.LeakyReLU() default slope (model.py:107)
        case RVB_ACT_RELU: return fmaxf(v, 0.f);
        case RVB_ACT_ELU: return v > 0.f ? v : expm1f(v);
        case RVB_ACT_TANH: return tanhf(v);
        case RVB_ACT_SIGMOID: return __fdiv_rn(1.f, __fadd_rn(1.f, expf(-v)));
        case RVB_ACT_RELU6: return fminf(fmaxf(v, 0.f), 6.f);
        default: return v;
    }
}

// Sixteen values at once with the switch OUTSIDE the loop: inlined sixteen times, pl_act's switch (with its expm1f / tanhf / expf
// arms) cost 270 cycles per element in the tensor-core kernels' epilogues.
__device__ __forceinline__ void pl_act16(float* v, int kind) {
    if (kind == RVB_ACT_LEAKYRELU) {
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = v[j] > 0.f ? v[j] : __fmul_rn(v[j], 0.01f);
    } else if (kind == RVB_ACT_RELU) {
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = fmaxf(v[j], 0.f);
    } else {          // statically indexed (a rolled loop would push v[] into local memory for every caller)
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = pl_act(v[j], kind);
    }
}

// torch [out][in] -> k-major padded panel
__global__ void pl_pack_kernel(const float* __restrict__ w, const float* __restrict__ b, int in, int out, int outp,
                               float* __restrict__ wt, float* __restrict__ bias) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < (int64_t)in * outp) {
        const int k = (int)(i / outp), n = (int)(i % outp);
        wt[i] = n < out ? w[(int64_t)n * in + k] : 0.f;
    }
    if (i < outp) bias[i] = i < out ? b[i] : 0.f;
}

// an observation value as f32: the f32 rows as they are, the packed fp16 heightmap widened (exact)
__device__ __forceinline__ float pl_ldg(const float* p) { return __ldg(p); }
__device__ __forceinline__ float pl_ldg(const __half* p) { return __half2float(__ldg(p)); }

// One dense layer of the tile.  Input activations: shared memory `act_in` [K][PL_LDA] (GLOBAL_IN = false) or columns
// [col0, col0 + K) of the tile's observation rows in global memory (f32 or fp16), staged transposed through `xs` as f32
// (GLOBAL_IN = true).  Output: act(in . Wt + bias) into shared memory `act_out` [n][PL_LDA], rows n < OUT only.
template <typename T> struct pl_given { using type = T; };      // T as the caller names it (the layers on shared memory pass nullptr)
template <int CN, bool GLOBAL_IN, typename T = float>
__device__ __forceinline__ void pl_dense(const float* __restrict__ act_in, const typename pl_given<T>::type* __restrict__ obs, int64_t obs_ld, int64_t m0,
                                         int64_t N, int col0, int K, const PackedLinear& L, float* __restrict__ xs,
                                         float* __restrict__ ws, float* __restrict__ act_out, int act_kind) {
    constexpr int OUTP = 32 * CN;
    constexpr int KC = (PL_WS_FLOATS / OUTP) < 32 ? (PL_WS_FLOATS / OUTP) : 32;
    const int tid = threadIdx.x, ng = tid & 31, mg = tid >> 5;
    float acc[4][CN];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < CN; ++j) acc[i][j] = 0.f;

    // Software pipeline: chunk i+1 travels global -> registers while chunk i is multiplied out of shared memory.
    constexpr int WV = (KC * (OUTP / 4) + PL_THREADS - 1) / PL_THREADS;
    float4 wreg[WV];
    float xreg[PL_TM / 8];
    auto fetch = [&](int k0) {
        const int kc = min(KC, K - k0);
        const float4* src = reinterpret_cast<const float4*>(L.wt + (int64_t)k0 * OUTP);   // contiguous rows, 16-byte aligned
#pragma unroll
        for (int v = 0; v < WV; ++v) {
            const int i = tid + v * PL_THREADS;
            wreg[v] = i < kc * (OUTP / 4) ? __ldg(src + i) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        if (GLOBAL_IN) {                                   // a warp reads 32 consecutive floats of one env's row
#pragma unroll
            for (int r = 0; r < PL_TM / 8; ++r) {
                const int m = mg + 8 * r;
                xreg[r] = (ng < kc && m0 + m < N) ? pl_ldg(obs + (m0 + m) * obs_ld + col0 + k0 + ng) : 0.f;
            }
        }
    };
    fetch(0);
    for (int k0 = 0; k0 < K; k0 += KC) {
        const int kc = min(KC, K - k0);
        __syncthreads();                                   // previous chunk fully consumed (and act_in fully written)
#pragma unroll
        for (int v = 0; v < WV; ++v) {
            const int i = tid + v * PL_THREADS;
            if (i < kc * (OUTP / 4)) reinterpret_cast<float4*>(ws)[i] = wreg[v];
        }
        if (GLOBAL_IN) {                                   // transposed: xs[k][env]
#pragma unroll
            for (int r = 0; r < PL_TM / 8; ++r) xs[ng * PL_LDA + mg + 8 * r] = xreg[r];
        }
        __syncthreads();
        if (k0 + KC < K) fetch(k0 + KC);
        const float* a_base = GLOBAL_IN ? xs : act_in + (int64_t)k0 * PL_LDA;
        auto step = [&](int kk) {
            const float4 a = *reinterpret_cast<const float4*>(a_base + kk * PL_LDA + mg * 4);
            float w[CN];
#pragma unroll
            for (int j = 0; j < CN; ++j) w[j] = ws[kk * OUTP + ng + 32 * j];
#pragma unroll
            for (int j = 0; j < CN; ++j) {
                ffma2(acc[0][j], acc[1][j], a.x, a.y, w[j]);
                ffma2(acc[2][j], acc[3][j], a.z, a.w, w[j]);
            }
        };
        if (kc == KC) {                                    // full chunks: no loop overhead
#pragma unroll
            for (int kk = 0; kk < KC; ++kk) step(kk);
        } else {
#pragma unroll 4
            for (int kk = 0; kk < kc; ++kk) step(kk);
        }
    }
#pragma unroll
    for (int j = 0; j < CN; ++j) {
        const int n = ng + 32 * j;
        if (n < L.out) {
            const float b = __ldg(L.bias + n);
            float4 o;
            o.x = pl_act(__fadd_rn(acc[0][j], b), act_kind);
            o.y = pl_act(__fadd_rn(acc[1][j], b), act_kind);
            o.z = pl_act(__fadd_rn(acc[2][j], b), act_kind);
            o.w = pl_act(__fadd_rn(acc[3][j], b), act_kind);
            *reinterpret_cast<float4*>(act_out + n * PL_LDA + mg * 4) = o;
        }
    }
}

// shared-memory plan (floats)
#define PL_SM_A 0                                   // concat [<=128][LDA], later the third hidden layer [128][LDA]
#define PL_SM_B (PL_SM_A + 128 * PL_LDA)            // first hidden layer [256][LDA]
#define PL_SM_C (PL_SM_B + PL_M1 * PL_LDA)          // encoder hidden [80][LDA], later the second hidden layer [160][LDA]
#define PL_SM_XS (PL_SM_C + PL_M2 * PL_LDA)         // obs chunk [32][LDA]
#define PL_SM_WS (PL_SM_XS + 32 * PL_LDA)           // weight chunk
#define PL_SM_FLOATS (PL_SM_WS + PL_WS_FLOATS)
#define PL_SMEM_BYTES (PL_SM_FLOATS * 4)

// The observation of a row: proprio[0, p) and the heightmap's sparse | dense columns, which start at column p of hm's row
// (hm_after_proprio: the f32 rows, passed as both sources) or at column 0 (the packed form: obs_buf[:, :p] and the fp16 heightmap).
template <typename T>
__device__ __forceinline__ void policy_forward_body(const PolicyDev* __restrict__ p0, const PolicyDev* __restrict__ p1,
                                                    const float* __restrict__ proprio, int64_t proprio_ld, const T* __restrict__ hm,
                                                    int64_t hm_ld, bool hm_after_proprio, int64_t N, float* __restrict__ out0,
                                                    int64_t out0_ld, float* __restrict__ out1, int64_t out1_ld) {
    // blockIdx.y selects the network (actor / critic of one PPO step read the same obs tile, hot in L2)
    const PolicyDev& P = *(blockIdx.y ? p1 : p0);
    float* __restrict__ out = blockIdx.y ? out1 : out0;
    const int64_t out_ld = blockIdx.y ? out1_ld : out0_ld;
    extern __shared__ __align__(16) float sm[];
    float* A = sm + PL_SM_A;
    float* B = sm + PL_SM_B;
    float* Cb = sm + PL_SM_C;
    float* xs = sm + PL_SM_XS;
    float* ws = sm + PL_SM_WS;
    const int tid = threadIdx.x;
    const int64_t m0 = (int64_t)blockIdx.x * PL_TM;
    const int p = P.n_proprio;

    // proprioceptive columns -> concat rows 0..p-1 (model.py:188)
    if (tid < PL_TM * p) {
        const int m = tid & 31, k = tid >> 5;
        A[k * PL_LDA + m] = (m0 + m < N) ? __ldg(proprio + (m0 + m) * proprio_ld + k) : 0.f;
    }
    const int hm_col0 = hm_after_proprio ? p : 0;
    // sparse encoder (model.py:186) -> concat rows p .. p+59
    pl_dense<3, true, T>(nullptr, hm, hm_ld, m0, N, hm_col0, P.n_sparse, P.es1, xs, ws, Cb, P.act);
    pl_dense<2, false>(Cb, nullptr, 0, 0, 0, 0, PL_E1, P.es2, xs, ws, A + p * PL_LDA, P.act);
    // dense encoder (model.py:187) -> concat rows p+60 .. p+119
    pl_dense<3, true, T>(nullptr, hm, hm_ld, m0, N, hm_col0 + P.n_sparse, P.n_dense, P.ed1, xs, ws, Cb, P.act);
    pl_dense<2, false>(Cb, nullptr, 0, 0, 0, 0, PL_E1, P.ed2, xs, ws, A + (p + PL_E2) * PL_LDA, P.act);
    // MLP (model.py:190-191)
    pl_dense<8, false>(A, nullptr, 0, 0, 0, 0, p + 2 * PL_E2, P.m1, xs, ws, B, P.act);
    pl_dense<5, false>(B, nullptr, 0, 0, 0, 0, PL_M1, P.m2, xs, ws, Cb, P.act);
    pl_dense<4, false>(Cb, nullptr, 0, 0, 0, 0, PL_M2, P.m3, xs, ws, A, P.act);
    __syncthreads();
    // head: Linear(128, A) [+ Tanh] -- warp o computes output o for the tile's 32 envs
    const int m = tid & 31, o = tid >> 5;
    if (o < P.n_head && m0 + m < N) {
        const float* w = P.head_w + o * PL_M3;
        float acc = 0.f;
#pragma unroll 8
        for (int k = 0; k < PL_M3; ++k) acc = fmaf(A[k * PL_LDA + m], __ldg(w + k), acc);
        acc = __fadd_rn(acc, __ldg(P.head_b + o));
        out[(m0 + m) * out_ld + o] = P.head_tanh ? tanhf(acc) : acc;
    }
}

__global__ void __launch_bounds__(PL_THREADS, 2)
policy_forward_kernel(const PolicyDev* __restrict__ p0, const PolicyDev* __restrict__ p1, const float* __restrict__ obs,
                      int64_t obs_ld, int64_t N, float* __restrict__ out0, int64_t out0_ld, float* __restrict__ out1,
                      int64_t out1_ld) {
    policy_forward_body(p0, p1, obs, obs_ld, obs, obs_ld, true, N, out0, out0_ld, out1, out1_ld);
}

// the packed observation: any 2-byte aligned heightmap, any hm_ld (scalar loads)
__global__ void __launch_bounds__(PL_THREADS, 2)
policy_forward_h16_kernel(const PolicyDev* __restrict__ p0, const PolicyDev* __restrict__ p1, const float* __restrict__ proprio,
                          int64_t proprio_ld, const __half* __restrict__ hm, int64_t hm_ld, int64_t N, float* __restrict__ out0,
                          int64_t out0_ld, float* __restrict__ out1, int64_t out1_ld) {
    policy_forward_body(p0, p1, proprio, proprio_ld, hm, hm_ld, false, N, out0, out0_ld, out1, out1_ld);
}


// ------------------------------------------------------------------------------------------------------------
// Tensor-core path of the two first encoder layers (58 % of the network's multiply-adds): Linear(634, 80) and
// Linear(1112, 80) of model.py:118-144 on tcgen05 (sm_100a), fp32-grade accuracy.
//   * Operands are split into tf32 hi + lo parts (x = hi + lo to 2^-22 relative): A.W = Ah.Wh + Ah.Wl + Al.Wh to fp32 accuracy,
//     accumulated in fp32 in TMEM.  The weights are split once per handle; the observation chunk is split by the threads that
//     load it.  The heightmap observation columns are fp16 values by construction (rover.py:324-325) and every fp16 value is
//     EXACTLY representable in tf32 (10 explicit mantissa bits, 8-bit exponent), so their lo part is zero: the loaders flag a
//     chunk whose lo part is zero everywhere and the third MMA of its k-steps is skipped (two MMAs per k-step on the step's
//     obs_buf; three when a caller feeds arbitrary fp32 rows, e.g. after the noise hook).
//   * One CTA per 128 envs, 6 warps: warps 0-3 load their env's row chunk (32 columns = 128 bytes) and write it into shared
//     memory in the canonical K-major SWIZZLE_128B layout, then run the epilogue (TMEM -> registers, + bias, activation, store);
//     warp 5 streams the weight chunks with cp.async.bulk (the image in global memory IS the shared-memory image) onto the
//     stage's mbarrier; warp 4 issues the MMAs (M = 128, N = 80 per network, K = 8) and commits them to the stage's "empty"
//     barrier.  Three stages of 32 KB (A hi + lo) + 20 KB per network (W hi + lo).  Both networks of a PPO step share the A tiles.
// Output: h1 [N][nets * 160] = act(obs_sparse . W^T + b) | act(obs_dense . W^T + b) per network; the rest of the network (42 % of
// the multiply-adds) runs in policy_tail_tc_kernel from there.
// ------------------------------------------------------------------------------------------------------------
#define TC_M 128
#define TC_KC 32
#define TC_STAGES 3
#define TC_THREADS 320

__global__ void pl_tc_image_kernel(const float* __restrict__ w, int in, int chunks, float* __restrict__ img) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;          // one thread per (chunk, row, k in chunk)
    if (i >= (int64_t)chunks * PL_E1 * TC_KC) return;
    const int kk = (int)(i % TC_KC), row = (int)((i / TC_KC) % PL_E1), chunk = (int)(i / (TC_KC * PL_E1));
    const int k = chunk * TC_KC + kk;
    const float v = k < in ? w[(int64_t)row * in + k] : 0.f;
    uint32_t hi, lo;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(hi) : "f"(v));
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(lo) : "f"(__fsub_rn(v, __uint_as_float(hi))));
    const int c16 = kk >> 2, e = kk & 3;
    const int64_t at = (int64_t)row * TC_KC + (((c16 ^ (row & 7)) << 2) + e);
    img[((int64_t)chunk * 2 + 0) * PL_E1 * TC_KC + at] = __uint_as_float(hi);
    img[((int64_t)chunk * 2 + 1) * PL_E1 * TC_KC + at] = __uint_as_float(lo);
}

__device__ __forceinline__ uint32_t tc_smem(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint64_t tc_desc(uint32_t saddr) {
    // K-major, SWIZZLE_128B, 8-row groups 1024 B apart: start >> 4 | LBO 1 << 16 | SBO 64 << 32 | version 1 << 46 | layout 2 << 61
    return (uint64_t)((saddr >> 4) & 0x3FFFu) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
__device__ __forceinline__ void tc_mma(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d),
                 "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
                 : "memory");
}
// bounded wait: a wrong descriptor or a lost arrival must end in a trap, not in a hung GPU
__device__ __forceinline__ void tc_wait(uint64_t* bar, uint32_t parity) {
    const uint32_t a = tc_smem(bar);
    for (uint32_t it = 0; it < (1u << 26); ++it) {
        uint32_t done;
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(done)
                     : "r"(a), "r"(parity)
                     : "memory");
        if (done) return;
    }
    __trap();
}

// T = float: the f32 observation rows (the encoders' columns start at p).  T = __half: the packed heightmap rows (they start at 0),
// fp16 values, exact in tf32: the loaders widen them and store the hi tile only -- no lo part, no lo flag, so the MMA warp issues
// the two MMAs per k-step it issues for f32 rows holding the same values.
template <int NETS, typename T>
__device__ __forceinline__ void policy_l1_tc_body(const PolicyDev* __restrict__ p0, const PolicyDev* __restrict__ p1,
                                                  const T* __restrict__ obs, int64_t obs_ld, int64_t N, float* __restrict__ h1) {
    constexpr bool H16 = std::is_same<T, __half>::value;
    constexpr int NB = PL_E1 * NETS;                      // MMA N: 80 columns per network
    constexpr int A_FLOATS = 2 * TC_M * TC_KC;            // hi + lo, 2 x 16 KB
    constexpr int W_FLOATS = 2 * NB * TC_KC;              // hi + lo, 20 KB per network
    constexpr int STAGE_FLOATS = A_FLOATS + W_FLOATS;
    constexpr uint32_t TMEM_COLS = NETS == 2 ? 256u : 128u;      // 80 x NETS accumulator columns, a power of two
    constexpr int LOADERS = 8 * 32;                       // warps 0-7; warp 8 issues the MMAs, warp 9 streams the weights
    extern __shared__ unsigned char tc_smem_raw[];
    // SWIZZLE_128B operands want 1024-byte aligned tiles: align by hand (the launch reserves 1 KB of slack)
    float* stages = reinterpret_cast<float*>(tc_smem_raw + ((1024u - (tc_smem(tc_smem_raw) & 1023u)) & 1023u));
    __shared__ __align__(8) uint64_t full[TC_STAGES], empty[TC_STAGES], dready;
    __shared__ uint32_t tmem_base_s;
    __shared__ uint32_t s_lo[64];                         // chunk c of this tile has a non-zero lo part of A
    __shared__ float s_bias[PL_E1 * 2];                   // [network][80] of this CTA's encoder
    const PolicyDev& P0 = *p0;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    // blockIdx.y = encoder (0 sparse, 1 dense): the two first layers of a tile run as two CTAs, 20 and 35 chunks long -- the
    // latency of a tile (what a small batch sees) is the longer one, not their sum
    const bool dense = blockIdx.y != 0;
    const int nchunks = dense ? P0.tc_cd : P0.tc_cs;
    const int act_kind = P0.act;                          // rvb_policy_forward_pair requires the same activation of both networks
    if (tid < 64) s_lo[tid] = 0u;
    for (int i = tid; i < NB; i += TC_THREADS) {
        const int net = i / PL_E1, col = i % PL_E1;
        const PolicyDev& P = (NETS == 2 && net) ? *p1 : P0;
        s_bias[i] = __ldg((dense ? P.ed1.bias : P.es1.bias) + col);
    }
    const int64_t m0 = (int64_t)blockIdx.x * TC_M;
    if (tid == 0) {
        for (int s = 0; s < TC_STAGES; ++s) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(tc_smem(&full[s])), "r"(LOADERS + 1));
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(tc_smem(&empty[s])));
        }
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(tc_smem(&dready)));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 8) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tc_smem(&tmem_base_s)), "r"(TMEM_COLS));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = tmem_base_s;
    // programmatic dependent launch: the tail kernel's CTAs may be scheduled from here on (they allocate TMEM, initialise their
    // barriers and start streaming their weight images, then wait for THIS grid to complete before they read h1)
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

    if (warp < 8) {
        // ---- loaders: warp w owns rows [16 w, 16 w + 16) of the tile, four rows per pass: lane = (row of the pass, 16-byte column
        // group), so a row's 128 bytes are read by eight lanes with two 8-byte loads each and stored with ONE 16-byte store per
        // part.  (A thread-per-row layout made every load 32 L1 wavefronts; a lane-per-column layout needed two 4-byte stores per
        // element: the loaders, not the tensor core, set the pace -- 2.2 us per chunk.)  Chunk c+1 travels global -> registers
        // while chunk c is split and stored (two register buffers in ping-pong: a copy would wait for the loads it should hide).
        // The fp16 rows keep the lane map: a chunk row is 64 bytes, eight lanes read 8 bytes each as two 4-byte loads (a dense block
        // S halves into the row is only 4-byte aligned) and store the lane's 16-byte group of the f32 hi tile with one store.
        const int ri = lane >> 3, c16 = lane & 7;
        const int64_t rbase = m0 + warp * 16 + ri;
        const T* obase = obs + (H16 ? 0 : P0.n_proprio) + (dense ? P0.n_sparse : 0) + c16 * 4;
        const int kall = dense ? P0.n_dense : P0.n_sparse;
        using V = typename std::conditional<H16, __half2, float2>::type;
        auto fetch = [&](int c, V* v) {
            const int k0 = c * TC_KC;
            const int kmax = kall - k0;                                             // valid columns of this chunk (even)
            const T* src = obase + k0;
#pragma unroll
            for (int it = 0; it < 4; ++it) {
                const int64_t row = rbase + 4 * it;
                const V* q = reinterpret_cast<const V*>(src + row * obs_ld);
                const bool ok = row < N;
                v[2 * it] = (ok && c16 * 4 < kmax) ? __ldg(q) : V{};
                v[2 * it + 1] = (ok && c16 * 4 + 2 < kmax) ? __ldg(q + 1) : V{};
            }
        };
        auto process = [&](int c, const V* v) {
            const int s = c % TC_STAGES;
            const uint32_t ph = (uint32_t)(c / TC_STAGES) & 1u;
            tc_wait(&empty[s], ph ^ 1u);
            float* tile = stages + s * STAGE_FLOATS;
            bool any_lo = false;
#pragma unroll
            for (int it = 0; it < 4; ++it) {
                const int r = warp * 16 + 4 * it + ri;
                if constexpr (H16) {
                    float* dst = tile + (r >> 3) * 256 + (r & 7) * 32 + ((c16 ^ (r & 7)) << 2);
                    const float2 a = __half22float2(v[2 * it]), b = __half22float2(v[2 * it + 1]);
                    float x[4] = {a.x, a.y, b.x, b.y};
                    // +-inf: the f32 rows' split gives lo = inf - inf = NaN, which turns the row's sums into NaN; so does NaN as hi
#pragma unroll
                    for (int e = 0; e < 4; ++e) x[e] = isinf(x[e]) ? __int_as_float(0x7fffffff) : x[e];
                    *reinterpret_cast<float4*>(dst) = make_float4(x[0], x[1], x[2], x[3]);
                } else {
                    const float x[4] = {v[2 * it].x, v[2 * it].y, v[2 * it + 1].x, v[2 * it + 1].y};
                    float hi[4], lo[4];
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        uint32_t h, l;
                        asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(h) : "f"(x[e]));
                        asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(l) : "f"(__fsub_rn(x[e], __uint_as_float(h))));
                        hi[e] = __uint_as_float(h); lo[e] = __uint_as_float(l);
                        any_lo |= (l << 1) != 0u;
                    }
                    float* dst = tile + (r >> 3) * 256 + (r & 7) * 32 + ((c16 ^ (r & 7)) << 2);
                    *reinterpret_cast<float4*>(dst) = make_float4(hi[0], hi[1], hi[2], hi[3]);
                    *reinterpret_cast<float4*>(dst + TC_M * TC_KC) = make_float4(lo[0], lo[1], lo[2], lo[3]);
                }
            }
            if (!H16 && __any_sync(0xffffffffu, any_lo) && lane == 0) atomicOr(&s_lo[c & 63], 1u);
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(tc_smem(&full[s])) : "memory");
        };
        V va[8], vb[8];
        fetch(0, va);
        for (int c = 0; c < nchunks; c += 2) {
            if (c + 1 < nchunks) fetch(c + 1, vb);
            process(c, va);
            if (c + 1 < nchunks) {
                if (c + 2 < nchunks) fetch(c + 2, va);
                process(c + 1, vb);
            }
        }
        // ---- epilogue: TMEM lane = row of the tile, columns [0, NB) = (network, 80); a warp reads the TMEM quarter warp % 4, warps
        // 0-3 the first half of the columns, warps 4-7 the second
        const int q = warp & 3, half = warp >> 2;
        const int64_t row = m0 + q * 32 + lane;
        const bool live = row < N;
        tc_wait(&dready, 0);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        constexpr int G = NB / 16;                          // groups of 16 columns: 5 (one network) or 10
#pragma unroll 1
        for (int c0 = (half ? (G + 1) / 2 : 0) * 16; c0 < (half ? G : (G + 1) / 2) * 16; c0 += 16) {
            uint32_t r[16];
            const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)c0;
            asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                         : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
                           "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                         : "r"(taddr));
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            if (live) {
                float4 o[4];
                float* of = reinterpret_cast<float*>(o);
#pragma unroll
                for (int j = 0; j < 16; ++j) of[j] = __fadd_rn(__uint_as_float(r[j]), s_bias[c0 + j]);
                pl_act16(of, act_kind);
                float4* dst = reinterpret_cast<float4*>(h1 + row * (2 * NB) + (dense ? NB : 0) + c0);
#pragma unroll
                for (int j = 0; j < 4; ++j) dst[j] = o[j];
            }
        }
    } else if (warp == 9) {
        // ---- weight producer: the global image of a chunk is its shared-memory image -> bulk copies onto the stage's barrier
        if (lane == 0) {
            for (int c = 0; c < nchunks; ++c) {
                const int s = c % TC_STAGES;
                const uint32_t ph = (uint32_t)(c / TC_STAGES) & 1u;
                tc_wait(&empty[s], ph ^ 1u);
                const int kc = c;
                constexpr uint32_t PART_BYTES = PL_E1 * TC_KC * 4;          // 10 KB: one network, one part
                asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(tc_smem(&full[s])), "r"(2u * NETS * PART_BYTES) : "memory");
                float* wdst = stages + s * STAGE_FLOATS + A_FLOATS;
#pragma unroll
                for (int net = 0; net < NETS; ++net) {
                    const PolicyDev& P = net ? *p1 : P0;
                    const float* img = (dense ? P.tc_img_d : P.tc_img_s) + (int64_t)kc * 2 * PL_E1 * TC_KC;
#pragma unroll
                    for (int part = 0; part < 2; ++part)
                        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                                         tc_smem(wdst + (part * NB + net * PL_E1) * TC_KC)),
                                     "l"(img + (int64_t)part * PL_E1 * TC_KC), "r"(PART_BYTES), "r"(tc_smem(&full[s]))
                                     : "memory");
                }
            }
        }
    } else {
        // ---- MMA issuer
        if (lane == 0) {
            const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(NB >> 3) << 17) | ((uint32_t)(TC_M >> 4) << 24);
            for (int c = 0; c < nchunks; ++c) {
                const int s = c % TC_STAGES;
                const uint32_t ph = (uint32_t)(c / TC_STAGES) & 1u;
                tc_wait(&full[s], ph);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t d_tmem = tmem_base;
                const float* st = stages + s * STAGE_FLOATS;
                const uint64_t da = tc_desc(tc_smem(st)), dal = tc_desc(tc_smem(st + TC_M * TC_KC)), dh = tc_desc(tc_smem(st + A_FLOATS)),
                               dl = tc_desc(tc_smem(st + A_FLOATS + NB * TC_KC));
                uint32_t acc = c == 0 ? 0u : 1u;
                const bool with_lo = !H16 && *reinterpret_cast<volatile uint32_t*>(&s_lo[c & 63]) != 0u;
#pragma unroll
                for (int k = 0; k < 4; ++k) {                    // 8 tf32 = 32 bytes = 2 descriptor units per MMA
                    tc_mma(d_tmem, da + 2 * k, dh + 2 * k, idesc, acc);
                    tc_mma(d_tmem, da + 2 * k, dl + 2 * k, idesc, 1u);
                    if (with_lo) tc_mma(d_tmem, dal + 2 * k, dh + 2 * k, idesc, 1u);
                    acc = 1u;
                }
                asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(tc_smem(&empty[s])) : "memory");
                if (c == nchunks - 1) asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(tc_smem(&dready)) : "memory");
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 8) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS));
}

template <int NETS>
__global__ void __launch_bounds__(TC_THREADS, 1)
policy_l1_tc_kernel(const PolicyDev* __restrict__ p0, const PolicyDev* __restrict__ p1, const float* __restrict__ obs, int64_t obs_ld,
                    int64_t N, float* __restrict__ h1) {
    policy_l1_tc_body<NETS>(p0, p1, obs, obs_ld, N, h1);
}

// the packed heightmap: hm_ld even and hm 4-byte aligned (tc_usable)
template <int NETS>
__global__ void __launch_bounds__(TC_THREADS, 1)
policy_l1_tc_h16_kernel(const PolicyDev* __restrict__ p0, const PolicyDev* __restrict__ p1, const __half* __restrict__ hm, int64_t hm_ld,
                        int64_t N, float* __restrict__ h1) {
    policy_l1_tc_body<NETS>(p0, p1, hm, hm_ld, N, h1);
}

static size_t tc_smem_bytes(int nets) { return (size_t)TC_STAGES * (2 * TC_M * TC_KC + 2 * PL_E1 * nets * TC_KC) * sizeof(float) + 1024; }


// ------------------------------------------------------------------------------------------------------------
// The rest of the network on tcgen05 (policy_tail_tc_kernel): Linear(80,60) x2, Linear(124,256), Linear(256,160),
// Linear(160,128) of one network for a tile of 128 envs, chained through TMEM and shared memory, then the head.
// Every layer: the input activations (fp32) are split into tf32 hi + lo by the four converter warps (thread = env row) and
// written as SWIZZLE_128B operand tiles of 32 features; the weights arrive as a pre-built stream of tile images (hi + lo)
// through two 40 KB stages filled by cp.async.bulk; one thread issues Ah.Wh + Ah.Wl + Al.Wh per 8-feature step into a TMEM
// accumulator; the converters read it back (tcgen05.ld), add the bias, apply the activation and produce the next operand.
// Operand space is 4 x 32 features (128 KB with hi + lo), so the 256- and 160-wide inputs are fed in two passes that
// accumulate into the same TMEM columns.  TMEM columns: D2s [0,64) D2d [64,128) | D3 [160,416) | D4 [0,160) | D5 [160,288).
// ------------------------------------------------------------------------------------------------------------
#define TT_THREADS 320
#define TT_ENTRIES 27
#define TT_A_CHUNK (2 * TC_M * TC_KC)              // floats: hi + lo tile of one 32-feature chunk
#define TT_W_STAGE (2 * PL_M2 * TC_KC)             // floats: the largest weight chunk (160 rows, hi + lo) = 40 KB
#define TT_OFF_L2S 0
#define TT_OFF_L2D (3 * 2 * 64 * TC_KC)
#define TT_OFF_M1 (TT_OFF_L2D + 3 * 2 * 64 * TC_KC)
#define TT_OFF_M2 (TT_OFF_M1 + 8 * 2 * 128 * TC_KC)
#define TT_OFF_M3 (TT_OFF_M2 + 8 * 2 * PL_M2 * TC_KC)
#define TT_FLOATS (TT_OFF_M3 + 5 * 2 * 128 * TC_KC)
#define TT_D2S 0u
#define TT_D2D 64u
#define TT_D3 160u
#define TT_D4 0u
#define TT_D5 160u

struct TailEntry {
    int pass, achunk, rows, first, last;
    uint32_t dcol;
    int64_t woff;
};
__device__ __forceinline__ TailEntry tail_entry(int e) {
    TailEntry t;
    if (e < 3) t = {0, e, 64, e == 0, e == 2, TT_D2S, (int64_t)TT_OFF_L2S + (int64_t)e * 2 * 64 * TC_KC};
    else if (e < 6) t = {1, e - 3, 64, e == 3, e == 5, TT_D2D, (int64_t)TT_OFF_L2D + (int64_t)(e - 3) * 2 * 64 * TC_KC};
    else if (e < 14) { const int i = e - 6; t = {2, i >> 1, 128, (i >> 1) == 0, i == 7, TT_D3 + 128u * (uint32_t)(i & 1), (int64_t)TT_OFF_M1 + (int64_t)i * 2 * 128 * TC_KC}; }
    else if (e < 22) { const int i = e - 14; t = {3 + (i >> 2), i & 3, PL_M2, i == 0, (i & 3) == 3, TT_D4, (int64_t)TT_OFF_M2 + (int64_t)i * 2 * PL_M2 * TC_KC}; }
    else { const int i = e - 22; t = {5 + (i >> 2), i & 3, 128, i == 0, i == 3 || i == 4, TT_D5, (int64_t)TT_OFF_M3 + (int64_t)i * 2 * 128 * TC_KC}; }
    return t;
}

// one image block of the weight stream: rows [row0, row0 + rows) x features [32 kc, 32 kc + 32) of a torch-layout weight
__global__ void pl_tail_image_kernel(const float* __restrict__ w, int in, int out, int row0, int rows, int kc, float* __restrict__ dst) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= rows * TC_KC) return;
    const int kk = i % TC_KC, r = i / TC_KC;
    const int k = kc * TC_KC + kk, row = row0 + r;
    const float v = (k < in && row < out) ? w[(int64_t)row * in + k] : 0.f;
    uint32_t hi, lo;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(hi) : "f"(v));
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(lo) : "f"(__fsub_rn(v, __uint_as_float(hi))));
    const int at = r * TC_KC + ((((kk >> 2) ^ (r & 7)) << 2) + (kk & 3));
    dst[at] = __uint_as_float(hi);
    dst[rows * TC_KC + at] = __uint_as_float(lo);
}

__global__ void __launch_bounds__(TT_THREADS, 1)
policy_tail_tc_kernel(const PolicyDev* __restrict__ p0, const PolicyDev* __restrict__ p1, const float* __restrict__ proprio,
                      int64_t proprio_ld, int64_t N, const float* h1, int h1_nets, float* __restrict__ out0, int64_t out0_ld,
                      float* __restrict__ out1, int64_t out1_ld) {
    const PolicyDev& P = *(blockIdx.y ? p1 : p0);
    float* __restrict__ out = blockIdx.y ? out1 : out0;
    const int64_t out_ld = blockIdx.y ? out1_ld : out0_ld;
    extern __shared__ unsigned char tt_smem_raw[];
    float* abuf = reinterpret_cast<float*>(tt_smem_raw + ((1024u - (tc_smem(tt_smem_raw) & 1023u)) & 1023u));      // 4 chunks x (hi, lo)
    float* wbuf = abuf + 4 * TT_A_CHUNK;                                                                              // 2 stages
    __shared__ __align__(8) uint64_t a_full, d_ready, w_full[2], w_empty[2];
    __shared__ uint32_t tmem_base_s;
    __shared__ float s_b[64 + 64 + PL_M1 + PL_M2 + PL_M3];          // biases: es2 | ed2 | m1 | m2 | m3
    __shared__ float s_head[PL_MAX_HEAD * PL_M3 + PL_MAX_HEAD];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t m0 = (int64_t)blockIdx.x * TC_M;
    const int act_kind = P.act;
    for (int i = tid; i < 64 + 64 + PL_M1 + PL_M2 + PL_M3; i += TT_THREADS) {
        float v;
        if (i < 64) v = i < PL_E2 ? __ldg(P.es2.bias + i) : 0.f;
        else if (i < 128) v = i - 64 < PL_E2 ? __ldg(P.ed2.bias + i - 64) : 0.f;
        else if (i < 128 + PL_M1) v = __ldg(P.m1.bias + i - 128);
        else if (i < 128 + PL_M1 + PL_M2) v = __ldg(P.m2.bias + i - 128 - PL_M1);
        else v = __ldg(P.m3.bias + i - 128 - PL_M1 - PL_M2);
        s_b[i] = v;
    }
    for (int i = tid; i < P.n_head * PL_M3 + P.n_head; i += TT_THREADS)
        s_head[i] = i < P.n_head * PL_M3 ? __ldg(P.head_w + i) : __ldg(P.head_b + i - P.n_head * PL_M3);
    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(tc_smem(&a_full)), "r"(2 * TC_M));
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(tc_smem(&d_ready)));
        for (int s = 0; s < 2; ++s) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(tc_smem(&w_full[s])));
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(tc_smem(&w_empty[s])));
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 8) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tc_smem(&tmem_base_s)), "r"(512));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = tmem_base_s;

    if (warp < 8) {
        // ---- converters: two threads per env row of the tile (= TMEM lane; a warp reaches the TMEM quarter warp % 4): warps 0-3 take
        // the even groups of 16 features, warps 4-7 the odd ones
        const int r = (warp & 3) * 32 + lane, half = warp >> 2;
        const int64_t row = m0 + r;
        const bool live = row < N;
        float* arow = abuf + (r >> 3) * 256 + (r & 7) * 32;
        // four consecutive features f .. f+3 (f % 4 == 0) of this row -> hi / lo tiles of chunk f / 32
        auto store4 = [&](int f, float x0, float x1, float x2, float x3) {
            const float x[4] = {x0, x1, x2, x3};
            float hi[4], lo[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                uint32_t h, l;
                asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(h) : "f"(x[e]));
                asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(l) : "f"(__fsub_rn(x[e], __uint_as_float(h))));
                hi[e] = __uint_as_float(h); lo[e] = __uint_as_float(l);
            }
            float* dst = arow + (f >> 5) * TT_A_CHUNK + ((((f & 31) >> 2) ^ (r & 7)) << 2);
            *reinterpret_cast<float4*>(dst) = make_float4(hi[0], hi[1], hi[2], hi[3]);
            *reinterpret_cast<float4*>(dst + TC_M * TC_KC) = make_float4(lo[0], lo[1], lo[2], lo[3]);
        };
        auto publish = [&]() {
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(tc_smem(&a_full)) : "memory");
        };
        auto tmem16 = [&](uint32_t col, float* v) {          // 16 consecutive accumulator columns of this row
            uint32_t q[16];
            const uint32_t taddr = tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + col;
            asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                         : "=r"(q[0]), "=r"(q[1]), "=r"(q[2]), "=r"(q[3]), "=r"(q[4]), "=r"(q[5]), "=r"(q[6]), "=r"(q[7]), "=r"(q[8]),
                           "=r"(q[9]), "=r"(q[10]), "=r"(q[11]), "=r"(q[12]), "=r"(q[13]), "=r"(q[14]), "=r"(q[15])
                         : "r"(taddr));
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
            for (int j = 0; j < 16; ++j) v[j] = __uint_as_float(q[j]);
        };
        // accumulator columns [col, col + n) + bias + activation -> features [f0, f0 + n) of the operand (n % 16 == 0 here)
        auto convert = [&](uint32_t col, const float* bias, int n, int f0, int nvalid) {
            for (int j0 = 16 * half; j0 < n; j0 += 32) {
                float v[16];
                tmem16(col + j0, v);
#pragma unroll
                for (int j = 0; j < 16; ++j) v[j] = __fadd_rn(v[j], bias[j0 + j]);
                pl_act16(v, act_kind);
#pragma unroll
                for (int j = 0; j < 16; ++j) v[j] = (j0 + j < nvalid) ? v[j] : 0.f;
#pragma unroll
                for (int g = 0; g < 4; ++g)
                    if (j0 + 4 * g < nvalid) store4(f0 + j0 + 4 * g, v[4 * g], v[4 * g + 1], v[4 * g + 2], v[4 * g + 3]);
            }
        };
        int pass = 0;
        auto wait_pass = [&]() {                     // the MMAs of pass `pass` are complete: accumulator readable, operand space free
            tc_wait(&d_ready, (uint32_t)pass & 1u);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            ++pass;
        };
        // P0 / P1: the first encoder layers (policy_l1_tc_kernel's output) -> operand of the second ones.  Launched as a programmatic
        // dependent of that kernel: everything above ran beside its last CTAs; its results are visible after this wait.
        asm volatile("griddepcontrol.wait;" ::: "memory");
        const float* hrow = h1 + (live ? row : 0) * (2 * PL_E1 * h1_nets) + (int)blockIdx.y * PL_E1;
        for (int enc = 0; enc < 2; ++enc) {
            if (enc) wait_pass();
            const float4* src = reinterpret_cast<const float4*>(hrow + enc * PL_E1 * h1_nets);
#pragma unroll 5
            for (int g = half; g < PL_E1 / 4; g += 2) {
                // a plain (coherent) load, and h1 is not __restrict__: under programmatic dependent launch the producer grid was
                // still writing h1 while this one was resident, so the non-coherent read-only path is not allowed here
                const float4 x = live ? src[g] : make_float4(0.f, 0.f, 0.f, 0.f);
                store4(4 * g, x.x, x.y, x.z, x.w);
            }
            for (int f = PL_E1 + 4 * half; f < 96; f += 8) store4(f, 0.f, 0.f, 0.f, 0.f);
            publish();
        }
        // P2: x = cat(proprio, x0, x1) (model.py:188-189), 4 + 60 + 60 = 124 features (+ 4 zeros)
        wait_pass();
        {
            const float* orow = proprio + (live ? row : 0) * proprio_ld;
            if (half == 0) {
                const float4 pr = live ? make_float4(__ldg(orow), __ldg(orow + 1), __ldg(orow + 2), __ldg(orow + 3)) : make_float4(0.f, 0.f, 0.f, 0.f);
                store4(0, pr.x, pr.y, pr.z, pr.w);          // n_proprio == 4 on this path (tc_usable)
            } else {
                store4(124, 0.f, 0.f, 0.f, 0.f);
            }
            convert(TT_D2S, s_b, 64, 4, PL_E2);
            convert(TT_D2D, s_b + 64, 64, 4 + PL_E2, PL_E2);
            publish();
        }
        // P3 / P4: first hidden layer (256) in two halves
        wait_pass();
        convert(TT_D3, s_b + 128, 128, 0, 128);
        publish();
        wait_pass();
        convert(TT_D3 + 128, s_b + 128 + 128, 128, 0, 128);
        publish();
        // P5 / P6: second hidden layer (160): 128 + 32 features
        wait_pass();
        convert(TT_D4, s_b + 128 + PL_M1, 128, 0, 128);
        publish();
        wait_pass();
        convert(TT_D4 + 128, s_b + 128 + PL_M1 + 128, 32, 0, 32);
        publish();
        // head: Linear(128, A) [+ tanh] on the third hidden layer
        wait_pass();
        if (half == 0) {
            float acc[PL_MAX_HEAD] = {0.f, 0.f, 0.f, 0.f};
            const int n_head = P.n_head;
            const float* b3 = s_b + 128 + PL_M1 + PL_M2;
            for (int j0 = 0; j0 < PL_M3; j0 += 16) {
                float v[16];
                tmem16(TT_D5 + j0, v);
#pragma unroll
                for (int j = 0; j < 16; ++j) v[j] = __fadd_rn(v[j], b3[j0 + j]);
                pl_act16(v, act_kind);
#pragma unroll
                for (int j = 0; j < 16; ++j) {
#pragma unroll
                    for (int o = 0; o < PL_MAX_HEAD; ++o)
                        if (o < n_head) acc[o] = fmaf(v[j], s_head[o * PL_M3 + j0 + j], acc[o]);
                }
            }
            if (live)
                for (int o = 0; o < P.n_head; ++o) {
                    const float y = __fadd_rn(acc[o], s_head[P.n_head * PL_M3 + o]);
                    out[row * out_ld + o] = P.head_tanh ? tanhf(y) : y;
                }
        }
    } else if (warp == 9) {
        // ---- weight producer
        if (lane == 0) {
            const float* stream = P.tc_tail;
            for (int e = 0; e < TT_ENTRIES; ++e) {
                const TailEntry t = tail_entry(e);
                const int s = e & 1;
                tc_wait(&w_empty[s], ((uint32_t)(e >> 1) & 1u) ^ 1u);
                const uint32_t bytes = (uint32_t)(2 * t.rows * TC_KC * 4);
                asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(tc_smem(&w_full[s])), "r"(bytes) : "memory");
                asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                                 tc_smem(wbuf + s * TT_W_STAGE)),
                             "l"(stream + t.woff), "r"(bytes), "r"(tc_smem(&w_full[s]))
                             : "memory");
            }
        }
    } else {
        // ---- MMA issuer
        if (lane == 0) {
            int pass = -1;
            for (int e = 0; e < TT_ENTRIES; ++e) {
                const TailEntry t = tail_entry(e);
                if (t.pass != pass) {                          // a new operand: wait for the converters
                    pass = t.pass;
                    tc_wait(&a_full, (uint32_t)pass & 1u);
                }
                const int s = e & 1;
                tc_wait(&w_full[s], (uint32_t)(e >> 1) & 1u);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(t.rows >> 3) << 17) | ((uint32_t)(TC_M >> 4) << 24);
                const float* at = abuf + t.achunk * TT_A_CHUNK;
                const float* wt = wbuf + s * TT_W_STAGE;
                const uint64_t ah = tc_desc(tc_smem(at)), al = tc_desc(tc_smem(at + TC_M * TC_KC)), wh = tc_desc(tc_smem(wt)),
                               wl = tc_desc(tc_smem(wt + t.rows * TC_KC));
                const uint32_t d = tmem_base + t.dcol;
                uint32_t acc = t.first ? 0u : 1u;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    tc_mma(d, ah + 2 * k, wh + 2 * k, idesc, acc);
                    tc_mma(d, ah + 2 * k, wl + 2 * k, idesc, 1u);
                    tc_mma(d, al + 2 * k, wh + 2 * k, idesc, 1u);
                    acc = 1u;
                }
                asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(tc_smem(&w_empty[s])) : "memory");
                if (t.last) asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(tc_smem(&d_ready)) : "memory");
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 8) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512));
}

static size_t tt_smem_bytes() { return (size_t)(4 * TT_A_CHUNK + 2 * TT_W_STAGE) * sizeof(float) + 1024; }

static int check_linear(const rvb_linear* L, int in, int out, const char* what) {
    if (!L || !L->weight || !L->bias) return rvb_set_error(RVB_ERR_INVALID, "rvb_policy_create: null layer", what);
    if (L->in_features != in || L->out_features != out)
        return rvb_set_error(RVB_ERR_UNSUPPORTED, "rvb_policy_create: layer shape differs from the reference network "
                             "(encoders [80,60], mlp [256,160,128]; train.py:95)", what);
    return RVB_OK;
}

extern "C" int rvb_policy_create(rvb_policy** out, int32_t n_proprio, int32_t n_sparse, int32_t n_dense,
                                 const rvb_linear* enc_sparse, const rvb_linear* enc_dense, const rvb_linear* mlp,
                                 const rvb_linear* head, int32_t activation, int32_t head_tanh, int device, void* stream) {
    RVB_REQUIRE(out, "rvb_policy_create: null pointer");
    *out = nullptr;
    RVB_REQUIRE(enc_sparse && enc_dense && mlp && head, "rvb_policy_create: null pointer");
    RVB_REQUIRE(n_proprio >= 0 && n_proprio <= PL_MAX_PROPRIO && n_sparse > 0 && n_dense > 0,
                "rvb_policy_create: bad observation split");
    RVB_REQUIRE(activation >= RVB_ACT_LEAKYRELU && activation <= RVB_ACT_RELU6, "rvb_policy_create: unknown activation");
    RVB_REQUIRE(head->out_features >= 1 && head->out_features <= PL_MAX_HEAD, "rvb_policy_create: head width must be 1..4");
    int rc;
    if ((rc = check_linear(&enc_sparse[0], n_sparse, PL_E1, "sparse encoder layer 0"))) return rc;
    if ((rc = check_linear(&enc_sparse[1], PL_E1, PL_E2, "sparse encoder layer 1"))) return rc;
    if ((rc = check_linear(&enc_dense[0], n_dense, PL_E1, "dense encoder layer 0"))) return rc;
    if ((rc = check_linear(&enc_dense[1], PL_E1, PL_E2, "dense encoder layer 1"))) return rc;
    if ((rc = check_linear(&mlp[0], n_proprio + 2 * PL_E2, PL_M1, "mlp layer 0"))) return rc;
    if ((rc = check_linear(&mlp[1], PL_M1, PL_M2, "mlp layer 1"))) return rc;
    if ((rc = check_linear(&mlp[2], PL_M2, PL_M3, "mlp layer 2"))) return rc;
    if ((rc = check_linear(head, PL_M3, head->out_features, "head"))) return rc;

    int cur_dev = -1;                  // like every other entry point: the caller's current device, never changed here
    RVB_CUDA(cudaGetDevice(&cur_dev));
    RVB_REQUIRE(device == cur_dev, "rvb_policy_create: `device` is not the calling thread's current CUDA device");
    // value-initialised (storage null), so on a failure rvb_policy_destroy frees exactly what was built
    std::unique_ptr<rvb_policy, int (*)(rvb_policy*)> P(new (std::nothrow) rvb_policy(), rvb_policy_destroy);
    if (!P) return rvb_set_error(RVB_ERR_NOMEM, "rvb_policy_create", "host allocation failed");
    P->n_proprio = n_proprio; P->n_sparse = n_sparse; P->n_dense = n_dense; P->n_head = head->out_features;
    P->act = activation; P->head_tanh = head_tanh ? 1 : 0; P->device = device;
    struct Slot { PackedLinear* dst; const rvb_linear* src; };
    Slot slots[7] = {{&P->es1, &enc_sparse[0]}, {&P->es2, &enc_sparse[1]}, {&P->ed1, &enc_dense[0]}, {&P->ed2, &enc_dense[1]},
                     {&P->m1, &mlp[0]}, {&P->m2, &mlp[1]}, {&P->m3, &mlp[2]}};
    int64_t total = 0;
    for (auto& s : slots) {
        s.dst->in = s.src->in_features; s.dst->out = s.src->out_features; s.dst->outp = pad32(s.src->out_features);
        total += (int64_t)s.dst->in * s.dst->outp + s.dst->outp;
    }
    total += (int64_t)P->n_head * PL_M3 + 32 + PL_DESC_FLOATS;
    // tensor-core images of the two first layers: [chunks][hi, lo][80][32] floats each, 256-byte aligned
    P->tc_cs = (n_sparse + TC_KC - 1) / TC_KC;
    P->tc_cd = (n_dense + TC_KC - 1) / TC_KC;
    const int64_t img_s = (int64_t)P->tc_cs * 2 * PL_E1 * TC_KC, img_d = (int64_t)P->tc_cd * 2 * PL_E1 * TC_KC;
    total = (total + 63) / 64 * 64;
    const int64_t img_at = total;
    total += img_s + img_d + TT_FLOATS;
    const cudaError_t e = cudaMalloc((void**)&P->storage, sizeof(float) * total);
    if (e != cudaSuccess) {
        cudaGetLastError();          // reported here, not again by the next launch check (common.cuh: RVB_CUDA)
        return rvb_set_error(RVB_ERR_NOMEM, "rvb_policy_create: cudaMalloc", cudaGetErrorString(e));
    }
    P->storage_floats = total;
    cudaStream_t st = as_stream(stream);
    P->dev = reinterpret_cast<const PolicyDev*>(P->storage);
    float* cur = P->storage + PL_DESC_FLOATS;
    for (auto& s : slots) {
        PackedLinear& L = *s.dst;
        L.wt = cur; cur += (int64_t)L.in * L.outp;       // every panel size is a multiple of 32 floats: 16-byte alignment holds
        L.bias = cur; cur += L.outp;
        const int64_t n = (int64_t)L.in * L.outp;
        pl_pack_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, st>>>(s.src->weight, s.src->bias, L.in, L.out, L.outp, L.wt, L.bias);
    }
    P->head_w = cur; cur += (int64_t)P->n_head * PL_M3;
    P->head_b = cur;
    {
        float* is_ = P->storage + img_at;
        float* id_ = is_ + img_s;
        P->tc_img_s = is_; P->tc_img_d = id_;
        pl_tc_image_kernel<<<(unsigned)ceil_div((int64_t)P->tc_cs * PL_E1 * TC_KC, 256), 256, 0, st>>>(enc_sparse[0].weight, n_sparse, P->tc_cs, is_);
        pl_tc_image_kernel<<<(unsigned)ceil_div((int64_t)P->tc_cd * PL_E1 * TC_KC, 256), 256, 0, st>>>(enc_dense[0].weight, n_dense, P->tc_cd, id_);
        // the weight stream of policy_tail_tc_kernel, block by block in consumption order (tail_entry)
        float* tail = id_ + img_d;
        P->tc_tail = tail;
        auto block = [&](const rvb_linear& L, int row0, int rows, int kc, int64_t off) {
            pl_tail_image_kernel<<<(unsigned)ceil_div((int64_t)rows * TC_KC, 256), 256, 0, st>>>(L.weight, L.in_features, L.out_features, row0, rows, kc, tail + off);
        };
        for (int kc = 0; kc < 3; ++kc) block(enc_sparse[1], 0, 64, kc, (int64_t)TT_OFF_L2S + (int64_t)kc * 2 * 64 * TC_KC);
        for (int kc = 0; kc < 3; ++kc) block(enc_dense[1], 0, 64, kc, (int64_t)TT_OFF_L2D + (int64_t)kc * 2 * 64 * TC_KC);
        for (int i = 0; i < 8; ++i) block(mlp[0], 128 * (i & 1), 128, i >> 1, (int64_t)TT_OFF_M1 + (int64_t)i * 2 * 128 * TC_KC);
        for (int i = 0; i < 8; ++i) block(mlp[1], 0, PL_M2, i, (int64_t)TT_OFF_M2 + (int64_t)i * 2 * PL_M2 * TC_KC);
        for (int i = 0; i < 5; ++i) block(mlp[2], 0, 128, i, (int64_t)TT_OFF_M3 + (int64_t)i * 2 * 128 * TC_KC);
    }
    RVB_CUDA(cudaMemcpyAsync(P->head_w, head->weight, sizeof(float) * P->n_head * PL_M3, cudaMemcpyDeviceToDevice, st));
    RVB_CUDA(cudaMemcpyAsync(P->head_b, head->bias, sizeof(float) * P->n_head, cudaMemcpyDeviceToDevice, st));
    // the descriptor the kernel reads (P outlives the copy: the stream is synchronised below)
    RVB_CUDA(cudaMemcpyAsync(P->storage, static_cast<const PolicyDev*>(P.get()), sizeof(PolicyDev), cudaMemcpyHostToDevice, st));
    RVB_LAUNCH_CHECK();
    RVB_CUDA(cudaFuncSetAttribute(policy_forward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, PL_SMEM_BYTES));
    RVB_CUDA(cudaFuncSetAttribute(policy_l1_tc_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc_smem_bytes(1)));
    RVB_CUDA(cudaFuncSetAttribute(policy_l1_tc_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc_smem_bytes(2)));
    RVB_CUDA(cudaFuncSetAttribute(policy_forward_h16_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, PL_SMEM_BYTES));
    RVB_CUDA(cudaFuncSetAttribute(policy_l1_tc_h16_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc_smem_bytes(1)));
    RVB_CUDA(cudaFuncSetAttribute(policy_l1_tc_h16_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc_smem_bytes(2)));
    RVB_CUDA(cudaFuncSetAttribute(policy_tail_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tt_smem_bytes()));
    RVB_CUDA(cudaStreamSynchronize(st));   // the caller may free its weight tensors on return
    *out = P.release();
    return RVB_OK;
}

extern "C" int rvb_policy_destroy(rvb_policy* P) {
    if (!P) return RVB_OK;
    cudaFree(P->storage);
    delete P;
    return RVB_OK;
}

extern "C" int64_t rvb_policy_bytes(const rvb_policy* P) { return P ? P->storage_floats * (int64_t)sizeof(float) : 0; }

// 2 (default) = the whole network on tcgen05 (policy_l1_tc_kernel + policy_tail_tc_kernel: faster than the FFMA path from a single
// 128-env tile upwards) where tc_usable allows it, policy_forward_kernel otherwise; 1 = policy_forward_kernel for every shape (what
// bench.py's ffma2_kernel_ms and the tests force).  The two sum in different orders; both return the fp64 oracle's answer on the
// exact probes of tests/policy_probe.py and stay within max(32 x torch fp32's error, 1e-7) of it on dense random inputs.
static int g_policy_variant = 2;
extern "C" int rvb_policy_variant(int v) {
    if (v < 0) return g_policy_variant;
    RVB_REQUIRE(v == 1 || v == 2, "rvb_policy_variant: 1 (FFMA2 kernel) or 2 (default dispatch); variants 0 (scalar FFMA) and 3 are removed");
    const int prev = g_policy_variant;
    g_policy_variant = v;
    return prev;
}

// What the kernels read of a row: the f32 observation (hm16 == nullptr: proprio = obs, the heightmap follows at column p of the same
// row) or the packed form (proprio f32 [N, proprio_ld], the fp16 heightmap hm16 [N, hm_ld]).
struct PolicyIn {
    const float* proprio;
    int64_t proprio_ld;
    const __half* hm16;
    int64_t hm_ld;
};

// the tensor-core path reads f32 observation rows with 8-byte loads and fp16 heightmap rows with 4-byte loads
static bool tc_usable(const PolicyDev* P, const PolicyIn& in) {
    const bool aligned = in.hm16 ? (in.hm_ld % 2 == 0) && (((uintptr_t)in.hm16 & 3u) == 0)
                                 : (in.proprio_ld % 2 == 0) && (((uintptr_t)in.proprio & 7u) == 0);
    return g_policy_variant == 2 && aligned && (P->n_proprio == 4) && (P->n_sparse % 2 == 0) && (P->n_dense % 2 == 0);
}

static int check_forward(const rvb_policy* P, const float* obs, int64_t obs_ld, const float* out, int64_t out_ld) {
    RVB_REQUIRE(obs && out, "rvb_policy_forward: null pointer");
    RVB_REQUIRE(obs_ld >= (int64_t)P->n_proprio + P->n_sparse + P->n_dense, "rvb_policy_forward: obs rows are shorter than the network's input");
    RVB_REQUIRE(out_ld >= P->n_head, "rvb_policy_forward: out rows are shorter than the head");
    int cur_dev = -1;
    RVB_CUDA(cudaGetDevice(&cur_dev));
    RVB_REQUIRE(P->device == cur_dev, "rvb_policy_forward: the network lives on another device than the calling thread's current one");
    return RVB_OK;
}

// The tail kernel as a programmatic dependent of the first-layer kernel in front of it on `st`.
static cudaError_t launch_tail_tc(dim3 grid, cudaStream_t st, const PolicyDev* a, const PolicyDev* b, const float* proprio,
                                  int64_t proprio_ld, int64_t N, const float* h1, int nets, float* out0, int64_t out0_ld, float* out1,
                                  int64_t out1_ld) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = dim3(TT_THREADS);
    cfg.dynamicSmemBytes = tt_smem_bytes();
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, policy_tail_tc_kernel, a, b, proprio, proprio_ld, N, h1, nets, out0, out0_ld, out1, out1_ld);
}

// One network (B == nullptr) or two on the same observations (grid.y = network; the pair's first layers share the observation tiles).
static int policy_launch(const rvb_policy* A, const rvb_policy* B, const PolicyIn& in, int64_t N,
                         float* out_a, int64_t out_a_ld, float* out_b, int64_t out_b_ld, cudaStream_t st) {
    RVB_REQUIRE(N <= (int64_t)PL_TM * 0x7fffffff, "rvb_policy_forward: too many envs");
    const int nets = B ? 2 : 1;
    const PolicyDev* db = B ? B->dev : nullptr;
    RvbTemp<float> h1;
    if (tc_usable(A, in)) {
        RVB_CUDA(h1.alloc_pool((size_t)N * nets * 2 * PL_E1, st));
        const dim3 grid((unsigned)ceil_div(N, TC_M), 2);
        if (in.hm16) {
            if (B) policy_l1_tc_h16_kernel<2><<<grid, TC_THREADS, tc_smem_bytes(2), st>>>(A->dev, db, in.hm16, in.hm_ld, N, h1.p);
            else policy_l1_tc_h16_kernel<1><<<grid, TC_THREADS, tc_smem_bytes(1), st>>>(A->dev, db, in.hm16, in.hm_ld, N, h1.p);
        } else {
            if (B) policy_l1_tc_kernel<2><<<grid, TC_THREADS, tc_smem_bytes(2), st>>>(A->dev, db, in.proprio, in.proprio_ld, N, h1.p);
            else policy_l1_tc_kernel<1><<<grid, TC_THREADS, tc_smem_bytes(1), st>>>(A->dev, db, in.proprio, in.proprio_ld, N, h1.p);
        }
        RVB_CUDA(launch_tail_tc(dim3((unsigned)ceil_div(N, TC_M), nets), st, A->dev, db, in.proprio, in.proprio_ld, N, h1.p, nets, out_a,
                                out_a_ld, out_b, out_b_ld));
    } else {
        const dim3 grid((unsigned)ceil_div(N, PL_TM), nets);
        if (in.hm16)
            policy_forward_h16_kernel<<<grid, PL_THREADS, PL_SMEM_BYTES, st>>>(A->dev, db, in.proprio, in.proprio_ld, in.hm16, in.hm_ld, N,
                                                                               out_a, out_a_ld, out_b, out_b_ld);
        else
            policy_forward_kernel<<<grid, PL_THREADS, PL_SMEM_BYTES, st>>>(A->dev, db, in.proprio, in.proprio_ld, N, out_a, out_a_ld,
                                                                           out_b, out_b_ld);
    }
    RVB_LAUNCH_CHECK();
    return RVB_OK;
}

extern "C" int rvb_policy_forward(const rvb_policy* P, const float* obs, int64_t obs_ld, int64_t N, float* out, int64_t out_ld,
                                  void* stream) {
    RVB_REQUIRE(P, "rvb_policy_forward: null handle");
    if (N <= 0) return RVB_OK;
    int rc;
    if ((rc = check_forward(P, obs, obs_ld, out, out_ld))) return rc;
    return policy_launch(P, nullptr, PolicyIn{obs, obs_ld, nullptr, 0}, N, out, out_ld, nullptr, 0, as_stream(stream));
}

extern "C" int rvb_policy_forward_pair(const rvb_policy* A, const rvb_policy* B, const float* obs, int64_t obs_ld, int64_t N,
                                       float* out_a, int64_t out_a_ld, float* out_b, int64_t out_b_ld, void* stream) {
    RVB_REQUIRE(A && B, "rvb_policy_forward_pair: null handle");
    if (N <= 0) return RVB_OK;
    int rc;
    if ((rc = check_forward(A, obs, obs_ld, out_a, out_a_ld))) return rc;
    if ((rc = check_forward(B, obs, obs_ld, out_b, out_b_ld))) return rc;
    RVB_REQUIRE(A->device == B->device, "rvb_policy_forward_pair: the two networks live on different devices");
    RVB_REQUIRE(A->n_proprio == B->n_proprio && A->n_sparse == B->n_sparse && A->n_dense == B->n_dense,
                "rvb_policy_forward_pair: the two networks read different observation splits");
    RVB_REQUIRE(A->act == B->act, "rvb_policy_forward_pair: the two networks use different activations");
    return policy_launch(A, B, PolicyIn{obs, obs_ld, nullptr, 0}, N, out_a, out_a_ld, out_b, out_b_ld, as_stream(stream));
}

static int check_packed(const rvb_policy* P, int64_t proprio_ld, int64_t heightmap_ld, int64_t out_ld) {
    RVB_REQUIRE(proprio_ld >= P->n_proprio, "rvb_policy_forward_packed: proprio rows are shorter than the network's proprioceptive input");
    RVB_REQUIRE(heightmap_ld >= (int64_t)P->n_sparse + P->n_dense,
                "rvb_policy_forward_packed: heightmap rows are shorter than the network's sparse + dense input");
    RVB_REQUIRE(out_ld >= P->n_head, "rvb_policy_forward_packed: out rows are shorter than the head");
    int cur_dev = -1;
    RVB_CUDA(cudaGetDevice(&cur_dev));
    RVB_REQUIRE(P->device == cur_dev, "rvb_policy_forward_packed: the network lives on another device than the calling thread's current one");
    return RVB_OK;
}

// The pointers are checked before the handle: every malformed call is refused before the handle is read.
extern "C" int rvb_policy_forward_packed(const rvb_policy* A, const rvb_policy* B, const float* proprio, int64_t proprio_ld,
                                         const uint16_t* heightmap, int64_t heightmap_ld, int64_t N, float* out_a, int64_t out_a_ld,
                                         float* out_b, int64_t out_b_ld, void* stream) {
    RVB_REQUIRE(N <= 0 || (proprio && heightmap && out_a && (!B || out_b)), "rvb_policy_forward_packed: null pointer");
    RVB_REQUIRE(A, "rvb_policy_forward_packed: null handle");
    if (N <= 0) return RVB_OK;
    int rc;
    if ((rc = check_packed(A, proprio_ld, heightmap_ld, out_a_ld))) return rc;
    if (B) {
        if ((rc = check_packed(B, proprio_ld, heightmap_ld, out_b_ld))) return rc;
        RVB_REQUIRE(A->device == B->device, "rvb_policy_forward_packed: the two networks live on different devices");
        RVB_REQUIRE(A->n_proprio == B->n_proprio && A->n_sparse == B->n_sparse && A->n_dense == B->n_dense,
                    "rvb_policy_forward_packed: the two networks read different observation splits");
        RVB_REQUIRE(A->act == B->act, "rvb_policy_forward_packed: the two networks use different activations");
    }
    return policy_launch(A, B, PolicyIn{proprio, proprio_ld, reinterpret_cast<const __half*>(heightmap), heightmap_ld}, N, out_a, out_a_ld,
                         out_b, out_b_ld, as_stream(stream));
}
