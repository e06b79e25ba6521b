// Shared device/host helpers for librover_b200 (sm_100a only).
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/rover_b200.h"

// ---------------------------------------------------------------- errors (thread-local, never thrown)
int rvb_set_error(int code, const char* what, const char* detail);

// A failed call also sets the runtime's last error (a failed cudaMalloc does).  Once reported it is cleared: otherwise the next
// launch check -- this library's or the caller's own -- would report it again.  A device fault stays: it is sticky.
#define RVB_CUDA(expr)                                                                   \
    do {                                                                                 \
        cudaError_t e_ = (expr);                                                         \
        if (e_ != cudaSuccess) {                                                         \
            cudaGetLastError();                                                          \
            return rvb_set_error(RVB_ERR_CUDA, #expr, cudaGetErrorString(e_));           \
        }                                                                                \
    } while (0)
#define RVB_REQUIRE(cond, msg)                                                           \
    do {                                                                                 \
        if (!(cond)) return rvb_set_error(RVB_ERR_INVALID, msg, #cond);                  \
    } while (0)
#define RVB_LAUNCH_CHECK() RVB_CUDA(cudaGetLastError())

// Stream-ordered scratch memory from the library's own per-device pool.  The pool keeps what it has been given (release
// threshold = max): the default pool hands its memory back at every synchronisation, and a caller that synchronises once
// per env step (the host pipeline) then pays a driver re-allocation of several ms inside the next call.
cudaError_t rvb_scratch_alloc(void** p, size_t bytes, cudaStream_t st);

// Side stream + fork / join events of the calling thread for the current device (slot 0: rock layer beside the heightmap in
// rvb_env_post; slot 1: steep envs beside the shadow kernel), created once per (thread, device, slot) and kept.
struct RvbSide {
    cudaStream_t s;
    cudaEvent_t fork, join;
};
cudaError_t rvb_side_stream(int slot, RvbSide** out);

// Runs on EVERY exit path of a launcher that forked work onto a side stream: the caller's stream waits for the side stream's join
// event (once it has been recorded).
struct RvbJoinGuard {
    cudaStream_t st;
    cudaEvent_t join = nullptr;      // set after cudaEventRecord(join, side)
    explicit RvbJoinGuard(cudaStream_t s) : st(s) {}
    ~RvbJoinGuard() {
        if (join) cudaStreamWaitEvent(st, join, 0);
    }
};

// A temporary device array of n T, freed on EVERY exit path of its scope.  alloc_pool: stream-ordered scratch from the library's
// pool, given back on its stream.  alloc: a plain cudaMalloc buffer, for the layer build's temporaries -- the pool keeps what it
// is given, so gigabytes of sort keys would stay reserved for the life of the process.
template <typename T>
struct RvbTemp {
    T* p = nullptr;
    cudaStream_t st = nullptr;
    bool pooled = false;
    RvbTemp() = default;
    RvbTemp(const RvbTemp&) = delete;
    RvbTemp& operator=(const RvbTemp&) = delete;
    cudaError_t alloc(size_t n) { return cudaMalloc((void**)&p, sizeof(T) * n); }
    cudaError_t alloc_pool(size_t n, cudaStream_t s) {
        pooled = true;
        st = s;
        return rvb_scratch_alloc((void**)&p, sizeof(T) * n, s);
    }
    ~RvbTemp() {
        if (!p) return;
        if (pooled) cudaFreeAsync(p, st);
        else cudaFree(p);
    }
};

// ---------------------------------------------------------------- terrain handle
// One pre-resolved record per triangle, 32 B = one L2 sector, two 16-byte loads.
// halves: a.xyz | b.xyz | c.xyz | n.xyz (n = b x c) | 4 x pad      (ray_casting.py:34-40)
struct __align__(16) TriRec {
    __half a[3], b[3], c[3], n[3], pad[4];
};
static_assert(sizeof(TriRec) == 32, "TriRec must be one 32-byte sector");

// One 32-byte record (TriRec, S1Rec: 32-byte aligned) through the read-only path in ONE instruction: sm_100's 256-bit load
// (LDG.E.256) instead of a 128-bit + a 64/128-bit one -- half the LSU instructions and L1 wavefronts of the record gathers.
__device__ __forceinline__ void ldg_rec32(const void* p, uint4& lo, uint4& hi) {
    asm("ld.global.nc.v8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
        : "=r"(lo.x), "=r"(lo.y), "=r"(lo.z), "=r"(lo.w), "=r"(hi.x), "=r"(hi.y), "=r"(hi.z), "=r"(hi.w)
        : "l"(p));
}

// Per-triangle inputs of the shadow kernel's stage 1 (raycast_shadow.cu), pre-computed once per layer with the very fp32
// operations the kernel used to run per (env, triangle): centroid, bounding radius, b x c, and the two magnitudes the
// error bounds scale with (rounded UP to fp16: a larger value only widens the bounds).
struct __align__(16) S1Rec {
    float qx, qy, qz, r;      // centroid a + (b + c) / 3; 2/3 of the longest edge (+ slack)
    float nx, ny, nz;         // b x c in fp32
    uint32_t cb_amax;         // fp16 bits: max |b_i|, |c_i|  |  max |a_i| << 16
};
static_assert(sizeof(S1Rec) == 32, "S1Rec must be one 32-byte sector");

// Bounds of the stage-1 inputs of 32 consecutive superblock-list entries (window w = entries [32 w, 32 w + 32) of sb_ids, whatever
// lists they belong to): the shadow kernel tests a whole window against a superblock item's ray rectangle before it enumerates
// the window's triangles (raycast_shadow.cu: chunk_cull; numpy statement + proof by comparison with stage 1: tests/shadow_proto.py).
struct __align__(16) ChunkRec {
    float x0, x1, y0, y1, z0, z1;      // centroid box (x0 = NaN: the window holds a non-finite record -- never culled)
    float rmax, cbmax, amax;            // max of S1Rec.r, cb, amax
    float nxlo, nxhi, nylo, nyhi, nzlo, nzhi;      // component ranges of b x c
    float pad;
};
static_assert(sizeof(ChunkRec) == 64, "ChunkRec");

struct rvb_terrain {
    int32_t* index;    // [G0,G1,Ks] device; row stride Ks = K rounded up to even (8-byte aligned id pairs), pad ids = 0
    TriRec* recs;      // [T], device
    S1Rec* s1recs;     // [T], device
    int64_t G0, G1, K, Ks, T, V;
    float res, shift_x, shift_y;
    int sem;
    int device;
    // Block lists (built when K <= 255): the grid is cut into RVB_BLK x RVB_BLK cell blocks; a block's list is the
    // union of its cells' K-lists, one entry per distinct triangle (sorted by id, padded to an even count): its id
    // and, for each of the block's cells, the slot the triangle holds in that cell's list (0xFF = not in that list).
    // Rays of neighbouring cells then share one fetch of every candidate record while each ray still sees exactly
    // its own cell's list and slots.
    int32_t nBx, nBy;
    uint32_t* blk_off;   // [nBx*nBy + 1] entry offsets (even)
    int32_t* blk_ids;    // [n_ent]  triangle ids (pad entries: 0)
    uint4* blk_slots;    // [n_ent]  byte s = slot in sub-cell s (s = (cx % BLK) * BLK + cy % BLK), other bytes 0xFF
    int64_t n_ent;
    // Superblock lists (built with the block lists): the union of the K-lists of RVB_SB x RVB_SB blocks, sorted by id.
    // The shadow ray-cast kernel enumerates these (a superset of every member cell's candidates) and, for the few candidates a
    // ray can actually hit, reads membership + slot in the ray's own K-list from the entry's per-cell table (sb_slot9).
    int32_t nSBx, nSBy;
    uint32_t* sb_off;    // [nSBx*nSBy + 1]
    int32_t* sb_ids;     // [n_sb_ent]
    unsigned char* sb_slot9;   // [n_sb_ent][24][24]  slot of the triangle in the K-list of cell (cx % 24, cy % 24) of the superblock; 0xFF = absent
    int64_t n_sb_ent;
    ChunkRec* sb_chunk;  // [ceil(n_sb_ent / 32)]
    int64_t n_ill;       // triangles whose determinant is rounding noise even for a vertical ray (no culling bound exists for them)
};
#define RVB_BLK 3
#define RVB_SB 8

// ---------------------------------------------------------------- fp16 arithmetic with torch's roundings
// ATen computes every Half element-wise op as fp32 op + one rounding; for + - * that equals the
// correctly rounded fp16 op, so the *_rn intrinsics are used (they also forbid mul+add contraction).
// Division goes through IEEE fp32 division and one rounding (innocuous double rounding).
__device__ __forceinline__ __half h_add(__half a, __half b) { return __hadd_rn(a, b); }
__device__ __forceinline__ __half h_sub(__half a, __half b) { return __hsub_rn(a, b); }
__device__ __forceinline__ __half h_mul(__half a, __half b) { return __hmul_rn(a, b); }
__device__ __forceinline__ __half h_div(__half a, __half b) {
    return __float2half_rn(__fdiv_rn(__half2float(a), __half2float(b)));
}
__device__ __forceinline__ __half h_from_bits(unsigned short b) { return __ushort_as_half(b); }
__device__ __forceinline__ unsigned short h_bits(__half h) { return __half_as_ushort(h); }

#define RVB_H_LO 0xAE66u    // fp16(0 - 0.1)  = -0.0999755859375   (ray_casting.py:26)
#define RVB_H_HI 0x3C66u    // fp16(1 + 0.1)  =  1.099609375       (ray_casting.py:27)
#define RVB_H_MISS 0x4980u  // fp16(1.1 * 10) = 11.0               (ray_casting.py:28)

struct H3 {
    __half x, y, z;
};

__device__ __forceinline__ H3 h3_sub(H3 u, H3 v) { return {h_sub(u.x, v.x), h_sub(u.y, v.y), h_sub(u.z, v.z)}; }
// Tensor.cross on Half: (u1*v2 - u2*v1, u2*v0 - u0*v2, u0*v1 - u1*v0), each op rounded.
__device__ __forceinline__ H3 h3_cross(H3 u, H3 v) {
    return {h_sub(h_mul(u.y, v.z), h_mul(u.z, v.y)), h_sub(h_mul(u.z, v.x), h_mul(u.x, v.z)),
            h_sub(h_mul(u.x, v.y), h_mul(u.y, v.x))};
}
// left-to-right dot product (ray_casting.py:41)
__device__ __forceinline__ __half h3_dot(H3 u, H3 v) {
    return h_add(h_add(h_mul(u.x, v.x), h_mul(u.y, v.y)), h_mul(u.z, v.z));
}

// One (ray, triangle) test given pre-resolved a, b, c, n = b x c and d = -normalize(dir).
// Returns k_after_check (ray_casting.py:40-59).
__device__ __forceinline__ __half pair_test(H3 s, H3 d, H3 a, H3 b, H3 c, H3 n) {
    const __half lo = h_from_bits(RVB_H_LO), hi = h_from_bits(RVB_H_HI), miss = h_from_bits(RVB_H_MISS);
    H3 g = h3_sub(s, a);
    __half det = h3_dot(n, d);
    __half nn = h_div(h3_dot(h3_cross(g, c), d), det);
    if (__heq(det, lo)) nn = miss;
    __half mm = h_div(h3_dot(h3_cross(b, g), d), det);
    if (__heq(det, hi)) mm = miss;
    __half kk = h_div(h3_dot(n, g), det);
    if (__heq(det, hi)) kk = miss;
    bool ok = __hge(nn, lo) && __hge(mm, lo) && __hle(h_add(nn, mm), hi);
    return ok ? kk : miss;
}

// -normalize(dir) (ray_casting.py:31): L2 norm accumulated in fp32, rounded to fp16, clamp_min(eps -> 0 in
// fp16), fp16 division, negation.
__device__ __forceinline__ H3 neg_normalize(H3 v) {
    float x = __half2float(v.x), y = __half2float(v.y), z = __half2float(v.z);
    float ss = __fadd_rn(__fadd_rn(__fmul_rn(x, x), __fmul_rn(y, y)), __fmul_rn(z, z));
    __half nrm = __float2half_rn(__fsqrt_rn(ss));
    __half den = __hmax_nan(nrm, __float2half_rn(1e-12f));
    return {__hneg(h_div(v.x, den)), __hneg(h_div(v.y, den)), __hneg(h_div(v.z, den))};
}

// torch.min ordering on fp16: NaN first (propagates), -0 == +0, ties -> lower slot.
__device__ __forceinline__ uint32_t min_key(__half k, uint32_t slot) {
    unsigned short b = h_bits(k);
    uint32_t key;
    if ((b & 0x7fffu) > 0x7c00u) key = 0u;
    else {
        if ((b & 0x7fffu) == 0u) b = 0u;
        key = (b & 0x8000u) ? (uint32_t)(unsigned short)~b : (uint32_t)(b | 0x8000u);
    }
    return (key << 16) | slot;
}

// Two fp32 FMAs in one issue slot (Blackwell FFMA2: d.xy = a.xy * b + d.xy; ptxas folds the {b, b} pair into the
// instruction's broadcast operand).  Each half is an IEEE fma, so the result equals two fmaf() calls bit for bit.
__device__ __forceinline__ void ffma2(float& d0, float& d1, float a0, float a1, float b) {
    asm("{\n\t.reg .b64 ra, rb, rc;\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %4};\n\tmov.b64 rc, {%0, %1};\n\t"
        "fma.rn.f32x2 rc, ra, rb, rc;\n\tmov.b64 {%0, %1}, rc;\n\t}"
        : "+f"(d0), "+f"(d1)
        : "f"(a0), "f"(a1), "f"(b));
}

// f64 -> fp16 the way torch casts (double -> float -> half, two roundings) (camera.py:212)
__device__ __forceinline__ __half h_from_double(double v) { return __float2half_rn(__double2float_rn(v)); }

// (xy - shift)/res -> clamp -> round-half-even -> cell (camera.py:241-253).  torch-CUDA divides by a Python
// scalar as a multiplication by fp32(1/res); torch-CPU performs a true division.
__device__ __forceinline__ int cell_coord(__half v16, float shift, float res, float inv_res, int gmax, int sem) {
    float v = __fsub_rn(__half2float(v16), shift);
    v = (sem == RVB_SEM_TORCH_CPU) ? __fdiv_rn(v, res) : __fmul_rn(v, inv_res);
    v = fminf(fmaxf(v, 0.0f), (float)gmax);     // NaN -> 0 (the reference would fault on NaN input)
    return (int)rintf(v);
}

// Body transform shared by camera.py:197-199 and rock_detect.py:305-307,356-358 (no FMA contraction).
template <typename T>
struct Ops;
template <>
struct Ops<double> {
    static __device__ __forceinline__ double mul(double a, double b) { return __dmul_rn(a, b); }
    static __device__ __forceinline__ double add(double a, double b) { return __dadd_rn(a, b); }
    static __device__ __forceinline__ double sub(double a, double b) { return __dsub_rn(a, b); }
};
template <>
struct Ops<float> {
    static __device__ __forceinline__ float mul(float a, float b) { return __fmul_rn(a, b); }
    static __device__ __forceinline__ float add(float a, float b) { return __fadd_rn(a, b); }
    static __device__ __forceinline__ float sub(float a, float b) { return __fsub_rn(a, b); }
};

struct Trig {
    float sx, cx, sy, cy, sz, cz;   // sin/cos of -roll, -pitch, -yaw (camera.py:184-189)
};

__device__ __forceinline__ Trig make_trig(const float* euler, const float* trig, int64_t n) {
    Trig t;
    if (trig) {
        const float* p = trig + n * 6;
        t = {p[0], p[1], p[2], p[3], p[4], p[5]};
    } else {
        float r = -euler[n * 3 + 0], p = -euler[n * 3 + 1], y = -euler[n * 3 + 2];
        t = {sinf(r), cosf(r), sinf(p), cosf(p), sinf(y), cosf(y)};
    }
    return t;
}

template <typename T>
__device__ __forceinline__ void body_transform(T x, T y, T z, const Trig& t, T tx, T ty, T tz, T& xo, T& yo, T& zo) {
    using O = Ops<T>;
    T sx = (T)t.sx, cx = (T)t.cx, sy = (T)t.sy, cy = (T)t.cy, sz = (T)t.sz, cz = (T)t.cz;
    T A = O::add(O::mul(y, cx), O::mul(z, sx));
    T C = O::sub(O::mul(z, cx), O::mul(y, sx));
    T B = O::sub(O::mul(x, cy), O::mul(sy, C));
    xo = O::add(O::add(tx, O::mul(sz, A)), O::mul(cz, B));
    yo = O::sub(O::add(ty, O::mul(cz, A)), O::mul(sz, B));
    zo = O::add(O::add(tz, O::mul(x, sy)), O::mul(cy, C));
}

// Philox4x32-10 (Salmon et al., SC'11; Random123 known answers in oracle/reset_oracle.py): the counter-based generator of
// the device-side reset path (stones.cu) and of the observation hooks (hooks.cu).
__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1,
                                              uint32_t& o0, uint32_t& o1, uint32_t& o2, uint32_t& o3) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        c0 = hi1 ^ c1 ^ k0; c1 = lo1; c2 = hi0 ^ c3 ^ k1; c3 = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    o0 = c0; o1 = c1; o2 = c2; o3 = c3;
}

static inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }
static inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }
