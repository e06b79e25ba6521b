// Pieces shared by the heightmap ray-cast kernels (raycast.cu, raycast_tiled.cu, raycast_shadow.cu) and the rock layer's
// cast (rock.cu), and the host functions of rvb_heightmap_raycast that one of those files calls in another.
#pragma once
#include <initializer_list>

#include "common.cuh"

// Tuning knobs of the heightmap ray-cast: parameters of the shipped design that tools/ sweep (DESIGN.md 6, "Tuning knobs").
// read_raycast_knobs (raycast_shadow.cu) takes them from the environment on every call, so a process can change them between
// calls; an unset variable means the shipped default, a value that does not parse or lies outside its range is RVB_ERR_INVALID.
struct RaycastKnobs {
    int force;            // RVB_SHADOW_FORCE: -1 = unset (the layer's count of triangles without a bound decides), 0 / 1 = off / on
    float cos_steep;      // RVB_COS_STEEP: envs whose ray direction has |d_z| below it are cast by the tiled kernel
    int min_sh;           // RVB_SHADOW_SH: finest bins of the shadow kernel, 2^sh x 2^sh cells
    int task_rays;        // RVB_SHADOW_TASK_RAYS: rays per stage-3L task
    int64_t split;        // RVB_SHADOW_SPLIT: envs cast by two half-ray CTAs at the end of the launch; -1 = unset (depends on N)
    bool dbg;             // RVB_SHADOW_DBG: per-stage counters of each launch on stderr
};
int read_raycast_knobs(RaycastKnobs& k);

namespace rc { struct TiledParams; }
// rvb_heightmap_raycast (raycast.cu) and rvb_env_post (step.cu) set the call's inputs and outputs in one parameter block and hand
// it to heightmap_raycast.
// fill_tiled_params (raycast_tiled.cu): checks a ray-cast of P rays over N envs with `variant` and q's inputs and outputs, and
// fills in the rest of q (zero-initialised by the caller): the layer's lists and grid, P and the tiling of the P rays.  With
// N == 0 it checks N and P alone and leaves q as it is.
int fill_tiled_params(const rvb_terrain* t, int64_t P, int64_t N, int variant, rc::TiledParams& q);
// launch_tiled (raycast_tiled.cu): q.work_list / q.work_count set: `grid` CTAs loop over the list; otherwise one CTA per
// (env, tile).  `blocks`: the 3x3-cell block lists instead of the K-contiguous index.
int launch_tiled(const rc::TiledParams& q, bool blocks, int64_t grid, cudaStream_t st);
// build_env_order (raycast_shadow.cu): order[0 .. N) = the envs of q (filled by fill_tiled_params) in the order the shadow kernel
// and the rock kernel cast them: envs with tilted rays first (the slow CTAs of the shadow kernel must not start last), within
// each class by map position (Z-order of 0.8 m cells of the layer's grid), so that the envs resident on the GPU at one time share
// their terrain data in L2.  Deterministic: equal keys keep index order.
int build_env_order(const rc::TiledParams& q, int64_t N, float cos_steep, int32_t* order, cudaStream_t st);
// launch_shadow (raycast_shadow.cu): the shadow kernel over N envs in `order` (null: it builds the order itself), with the tiled
// kernel for the envs and tiles it leaves.
int launch_shadow(rc::TiledParams q, int64_t N, const RaycastKnobs& knobs, const int32_t* order, cudaStream_t st);
// heightmap_raycast (raycast.cu): the ray-cast of q (filled by fill_tiled_params) with the knobs already read and, for the shadow
// route, the env order of the shadow kernel (or null).
int heightmap_raycast(const rvb_terrain* t, const rc::TiledParams& q, int64_t N, int variant, const RaycastKnobs& knobs,
                      const int32_t* order, cudaStream_t st);
// rock_collision (rock.cu): rvb_rock_collision with the envs taken in `order` (null: index order); outputs stay indexed by env.
int rock_collision(const rvb_terrain* t, const float* pos, const float* euler, const float* trig, const float* joints,
                   const float* joint_trig, int64_t N, uint16_t* wheel_dist, uint16_t* body_dist, int32_t* hit_tri,
                   int64_t* collision, uint16_t* rays_out, const int32_t* order, cudaStream_t st);

// Raises each kernel's dynamic shared-memory limit to its size, once per (thread, device): the attribute belongs to the
// current device.  `configured_device` is the caller's thread_local record of the device it was last set on.
struct SmemLimit {
    const void* kernel;
    size_t bytes;
};
inline int set_smem_limits(int& configured_device, std::initializer_list<SmemLimit> kernels) {
    int dev = 0;
    RVB_CUDA(cudaGetDevice(&dev));
    if (configured_device == dev) return RVB_OK;
    for (const SmemLimit& k : kernels)
        RVB_CUDA(cudaFuncSetAttribute(k.kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k.bytes));
    configured_device = dev;
    return RVB_OK;
}

namespace rc {

constexpr uint32_t KEY_INIT = 0xC9800000u;     // (11.0, slot 0): the result when every candidate misses
constexpr uint32_t ORD_MISS = 0xC980u;        // order key of fp16 11.0 (0x4980 | 0x8000)

struct TiledParams {
    const int32_t* index;
    const TriRec* recs;
    const S1Rec* s1;          // stage-1 records of the shadow kernel
    const uint32_t* blk_off;
    const int32_t* blk_ids;
    const uint4* blk_slots;
    int nBy;
    int G0, G1, K, Ks;
    float res, inv_res, shift_x, shift_y;
    int sem;
    const float* pos;
    const float* euler;
    const float* trig;
    const double* pattern;
    int P, tiles, tile_size;
    __half* dist;
    int32_t* hit_slot;
    int32_t* hit_tri;
    __half* pt;
    __half* sources;
    float* obs;
    int64_t obs_ld;
    __half* obs16;            // optional packed observation: obs16[n * obs16_ld + (column - obs16_col0)] = fp16(dist / 2)
    int64_t obs16_ld;
    int obs16_col0;
    const int32_t* col_a;
    const int32_t* col_b;
    // shadow kernel (raycast_shadow.cu): superblock candidate lists + the list of (env, tile) work items it hands back
    const uint32_t* sb_off;
    const int32_t* sb_ids;
    const unsigned char* sb_slot9;
    const ChunkRec* sb_chunk;   // bounds per window of 32 list entries (window cull)
    int nSBy;
    float cos_steep;          // envs whose ray direction is flatter than this go to the fall-back list
    int* fb_count;            // [1]
    int32_t* fb_list;         // [N * tiles]  env * tiles + tile
    // tiled kernel in work-list mode: CTAs loop over fb_list[0 .. *fb_count) instead of blockIdx
    const int* work_count;
    const int32_t* work_list;
    int work_slices;
    // shadow kernel: env order (envs with tilted rays first: they are the slow CTAs, so they must not start last), written by
    // hm_classify_kernel with the list of steep envs (cast by the tiled kernel on a second stream, concurrently)
    const int32_t* order;     // [N]
    int min_sh;              // bins are 2^sh x 2^sh cells, sh >= min_sh (0 = one cell; tuning knob)
    int task_rays;            // shadow kernel: rays per task of stage 3L (1..32: one mask bit each; tuning knob)
    int64_t split_from;       // shadow kernel: order positions >= split_from are cast by two CTAs (half the rays each); -1 = none
    int split_at;             // first ray of the second half
    unsigned long long* dbg;  // optional [24] work counters / cycle counts of the shadow kernel (RVB_SHADOW_DBG=1)
};

// Cell (cx, cy) of an fp16 source: the x and y look-ups of camera.py:241-253.  Both axes clamp to size(0) - 1 (camera.py:243),
// then y also to G1 - 1.  The scalars are references so that, inlined, each is read where its axis needs it: with copies made
// before the call, ptxas schedules hm_tiled_kernel<3> differently (12952 instead of 12960 SASS instructions, nvcc 12.9).
__device__ __forceinline__ int2 ray_cell(__half x, __half y, const float& shift_x, const float& shift_y, const float& res,
                                         const float& inv_res, const int& G0, const int& G1, const int& sem) {
    return make_int2(cell_coord(x, shift_x, res, inv_res, G0 - 1, sem),
                     min(cell_coord(y, shift_y, res, inv_res, G0 - 1, sem), G1 - 1));
}

// The env's ray direction d = -normalize(dir) in fp16: dir is the body transform of the appended point (0, 0, -1) minus the
// translation, cast to fp16 (camera.py:179-181,202-207; ray_casting.py:31).
__device__ __forceinline__ H3 env_dir16(const Trig& tr, double tx, double ty, double tz) {
    double xo, yo, zo;
    body_transform<double>(0.0, 0.0, -1.0, tr, tx, ty, tz, xo, yo, zo);
    return neg_normalize({h_from_double(__dsub_rn(xo, tx)), h_from_double(__dsub_rn(yo, ty)), h_from_double(__dsub_rn(zo, tz))});
}

// two candidates of one cell, component-wise packed: .x = candidate j, .y = candidate j+1
struct Tri2 {
    __half2 ax, ay, az, bx, by, bz, cx, cy, cz, nx, ny, nz;
};

__device__ __forceinline__ __half2 u2h(uint32_t u) { return *reinterpret_cast<__half2*>(&u); }
__device__ __forceinline__ uint32_t h2u(__half2 h) { return *reinterpret_cast<uint32_t*>(&h); }
__device__ __forceinline__ __half2 add2(__half2 a, __half2 b) { return __hadd2_rn(a, b); }
__device__ __forceinline__ __half2 sub2(__half2 a, __half2 b) { return __hsub2_rn(a, b); }
__device__ __forceinline__ __half2 mul2(__half2 a, __half2 b) { return __hmul2_rn(a, b); }

__device__ __forceinline__ Tri2 pack_tri2(const uint4& p0, const uint2& p1, const uint4& q0, const uint2& q1) {
    // record halves: q0 = [a.x a.y | a.z b.x | b.y b.z | c.x c.y], q1 = [c.z n.x | n.y n.z]
    Tri2 t;
    t.ax = u2h(__byte_perm(p0.x, q0.x, 0x5410)); t.ay = u2h(__byte_perm(p0.x, q0.x, 0x7632));
    t.az = u2h(__byte_perm(p0.y, q0.y, 0x5410)); t.bx = u2h(__byte_perm(p0.y, q0.y, 0x7632));
    t.by = u2h(__byte_perm(p0.z, q0.z, 0x5410)); t.bz = u2h(__byte_perm(p0.z, q0.z, 0x7632));
    t.cx = u2h(__byte_perm(p0.w, q0.w, 0x5410)); t.cy = u2h(__byte_perm(p0.w, q0.w, 0x7632));
    t.cz = u2h(__byte_perm(p1.x, q1.x, 0x5410)); t.nx = u2h(__byte_perm(p1.x, q1.x, 0x7632));
    t.ny = u2h(__byte_perm(p1.y, q1.y, 0x5410)); t.nz = u2h(__byte_perm(p1.y, q1.y, 0x7632));
    return t;
}

// ------------------------------------------------------------------------------------------------------------
// Conservative fp16 pre-filter.  With q_n = N/det, q_m = M/det (exact rationals of fp16 values), n = fp16(q_n),
// m = fp16(q_m), a candidate passes ray_casting.py:59 only if
//     n >= fp16(-0.1)        <=>  q_n >= -3277/32768   (rounding boundary below -0x1.998p-4, tie -> even = -0.1)
//     m >= fp16(-0.1)        <=>  q_m >= -3277/32768
//     fp16(n + m) <= fp16(1.1) =>  q_n + q_m < 2253/2048 + 2^-9   (n, m are within 2^-11 relative of q_n, q_m, both
//                                                                   in [-0.11, 1.31] there, so n + m moves by < 2^-9)
// Multiplying by |det| (N' = N*sgn(det), M' likewise):  N' >= -C_LO*|det|,  M' >= -C_LO*|det|,  N'+M' < C_FAIL*|det|.
// The filter evaluates these in packed fp16 against thresholds rounded OUTWARDS:
//     tlo = -RN(|det| * 0x2E68 + 2^-23)   <= -C_LO*|det|      (0x2E68 = 0.10009766 >= C_LO / (1 - 2^-11))
//     thi =  RN(|det| * 0x3C6B + 2^-23)   >= RN16(x) for every x < C_FAIL*|det|   (0x3C6B = 1.10449 >= C_FAIL*(1+2^-11)^2)
// (the 2^-23 term covers the absolute rounding error 2^-25 of subnormal results).  NaN thresholds or numerators
// compare false -- exactly the cases the reference rejects (det = 0/NaN gives n, m = +-inf/NaN; a NaN numerator
// gives a NaN quotient).  Every candidate the filter lets through is re-evaluated with the literal op sequence
// (pair_test, divisions included), so the filter only has to be conservative, never exact.
// ------------------------------------------------------------------------------------------------------------
#define H_C1 0x2E68u
#define H_C2 0x3C6Bu
#define H_TINY 0x0002u

struct Cand2 {
    uint32_t sgn;      // sign bits of det = (b x c) . d in both halves   (ray_casting.py:41; d is per env)
    __half2 tlo, thi;  // outward-rounded thresholds; NaN for a slot beyond K
};

__device__ __forceinline__ Cand2 make_cand2(const Tri2& t, __half2 dx, __half2 dy, __half2 dz, bool v0, bool v1) {
    Cand2 c;
    const __half2 det = add2(add2(mul2(t.nx, dx), mul2(t.ny, dy)), mul2(t.nz, dz));
    c.sgn = h2u(det) & 0x80008000u;
    const __half2 da = u2h(h2u(det) & 0x7fff7fffu);
    const __half2 tiny = u2h(H_TINY | (H_TINY << 16));
    c.tlo = __hneg2(__hfma2(da, u2h(H_C1 | (H_C1 << 16)), tiny));
    c.thi = __hfma2(da, u2h(H_C2 | (H_C2 << 16)), tiny);
    if (!v0) c.tlo = u2h((h2u(c.tlo) & 0xffff0000u) | 0x7fffu);
    if (!v1) c.tlo = u2h((h2u(c.tlo) & 0x0000ffffu) | 0x7fff0000u);
    return c;
}

// 0xffff in the half of every candidate that may pass
__device__ __forceinline__ uint32_t prefilter2(__half2 sx, __half2 sy, __half2 sz, __half2 dx, __half2 dy, __half2 dz,
                                               const Tri2& t, const Cand2& c) {
    const __half2 gx = sub2(sx, t.ax), gy = sub2(sy, t.ay), gz = sub2(sz, t.az);                 // ray_casting.py:37
    const __half2 ux = sub2(mul2(gy, t.cz), mul2(gz, t.cy));                                     // g x c  (:44)
    const __half2 uy = sub2(mul2(gz, t.cx), mul2(gx, t.cz));
    const __half2 uz = sub2(mul2(gx, t.cy), mul2(gy, t.cx));
    const __half2 Nn = add2(add2(mul2(ux, dx), mul2(uy, dy)), mul2(uz, dz));                     // :45 numerator
    const __half2 vx = sub2(mul2(t.by, gz), mul2(t.bz, gy));                                     // b x g  (:49)
    const __half2 vy = sub2(mul2(t.bz, gx), mul2(t.bx, gz));
    const __half2 vz = sub2(mul2(t.bx, gy), mul2(t.by, gx));
    const __half2 Mn = add2(add2(mul2(vx, dx), mul2(vy, dy)), mul2(vz, dz));                     // :50 numerator
    const __half2 Ns = u2h(h2u(Nn) ^ c.sgn), Ms = u2h(h2u(Mn) ^ c.sgn);
    return __hge2_mask(Ns, c.tlo) & __hge2_mask(Ms, c.tlo) & __hle2_mask(add2(Ns, Ms), c.thi);
}

// key of torch.min's total order: NaN < everything, -0 == +0, ties -> lower slot; bit 0 remembers a negative zero.
__device__ __forceinline__ uint32_t make_key(unsigned short b, uint32_t slot) {
    uint32_t ord, nz = 0;
    if ((b & 0x7fffu) > 0x7c00u) ord = 0u;
    else if ((b & 0x7fffu) == 0u) { ord = 0x8000u; nz = b >> 15; }
    else ord = (b & 0x8000u) ? (uint32_t)(unsigned short)~b : (uint32_t)(b | 0x8000u);
    return (ord << 16) | (slot << 1) | nz;
}
__device__ __forceinline__ unsigned short key_bits(uint32_t key) {
    const uint32_t ord = key >> 16;
    if (ord == 0u) return 0x7fffu;
    if (ord == 0x8000u) return (key & 1u) ? 0x8000u : 0u;
    return (ord & 0x8000u) ? (unsigned short)(ord & 0x7fffu) : (unsigned short)~ord;
}

__device__ __forceinline__ void unpack_rec(const TriRec* rec, H3& a, H3& b, H3& c, H3& n) {
    const uint4 q0 = __ldg(reinterpret_cast<const uint4*>(rec));
    const uint2 q1 = __ldg(reinterpret_cast<const uint2*>(rec) + 2);
    a = {h_from_bits(q0.x & 0xffff), h_from_bits(q0.x >> 16), h_from_bits(q0.y & 0xffff)};
    b = {h_from_bits(q0.y >> 16), h_from_bits(q0.z & 0xffff), h_from_bits(q0.z >> 16)};
    c = {h_from_bits(q0.w & 0xffff), h_from_bits(q0.w >> 16), h_from_bits(q1.x & 0xffff)};
    n = {h_from_bits(q1.x >> 16), h_from_bits(q1.y & 0xffff), h_from_bits(q1.y >> 16)};
}

// A ray that holds a hit with k > 11.0 and no nearer one: the first slot whose value is <= 11.0 (a miss, or a hit at
// exactly 11.0) wins torch.min, and that slot is not necessarily 0.  Vanishingly rare (the rover would have to hover
// 11 m above the mesh), so one thread simply walks the K candidates with the literal op sequence.
static __device__ __noinline__ uint32_t literal_ray(const int32_t* row, int K, const TriRec* recs, H3 s, H3 d) {
    uint32_t best = 0xffffffffu;
    for (int j = 0; j < K; ++j) {
        H3 a, b, c, nn;
        unpack_rec(recs + __ldg(row + j), a, b, c, nn);
        best = min(best, make_key(h_bits(pair_test(s, d, a, b, c, nn)), (uint32_t)j));
    }
    return best;
}

// The same two look-ups for a layer whose K-contiguous index was released (rvb_terrain_release_index): the K-list of cell
// (cx, cy) is the set of entries of its 3x3 block's union list whose slot byte for the sub-cell is not 0xFF, and that byte IS the
// slot.  min() over keys that carry the slot does not depend on the order the candidates are visited in.
static __device__ __noinline__ uint32_t literal_ray_blk(const int32_t* ids, const uint4* slots, int n, int sub, const TriRec* recs,
                                                        H3 s, H3 d) {
    uint32_t best = 0xffffffffu;
    for (int e = 0; e < n; ++e) {
        const uint32_t slot = __ldg(reinterpret_cast<const unsigned char*>(slots + e) + sub);
        if (slot == 0xffu) continue;
        H3 a, b, c, nn;
        unpack_rec(recs + __ldg(ids + e), a, b, c, nn);
        best = min(best, make_key(h_bits(pair_test(s, d, a, b, c, nn)), slot));
    }
    return best;
}

static __device__ __noinline__ int32_t tri_of_slot_blk(const int32_t* ids, const uint4* slots, int n, int sub, int slot) {
    for (int e = 0; e < n; ++e)
        if ((int)__ldg(reinterpret_cast<const unsigned char*>(slots + e) + sub) == slot) return __ldg(ids + e);
    return 0;
}

// Epilogue in ray order: coalesced stores of dist / hit slot / hit triangle / pt / sources and the fused sparse+dense
// observation columns (heightmap_distribution.py:126-133, rover.py:324-325).  res[p] = best key of local ray p; a set bit
// in far[] marks a ray that saw a hit beyond the 11.0 miss sentinel (resolved literally here).
__device__ __forceinline__ void epilogue(const TiledParams& q, int64_t n, int p0, int np, const Trig& tr, double tx, double ty,
                                         double tz, __half2 dx2, __half2 dy2, __half2 dz2, const uint32_t* res,
                                         const uint32_t* far, int tid, int nthreads) {
    const H3 dlit = {__low2half(dx2), __low2half(dy2), __low2half(dz2)};
    const bool want_geo = q.hit_tri || q.pt || q.sources;
    // Fast path (the production call: distances + observation columns only, no ray of the tile saw a hit beyond the miss sentinel):
    // every load of the thread's <= 8 rays is issued before the first store -- in the general loop below a ray's column indices,
    // its stores and the next ray's loads form one dependent chain, and the CTA sits in this tail at memory latency (the obs
    // output cost 4.6 % of the kernel)
    {
        bool any_far = false;
        for (int i = tid; i < (np + 31) / 32; i += nthreads) any_far |= far[i] != 0u;
        any_far = __syncthreads_or(any_far ? 1 : 0) != 0;
        if (!any_far && !want_geo && !q.hit_slot && np <= 8 * nthreads) {
            uint32_t key[8];
            int ca[8], cb[8];
            const bool want_cols = q.obs != nullptr || q.obs16 != nullptr;
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int p = tid + u * nthreads;
                key[u] = p < np ? res[p] : 0u;
                ca[u] = (want_cols && p < np) ? __ldg(q.col_a + p0 + p) : -1;
                cb[u] = (want_cols && p < np) ? __ldg(q.col_b + p0 + p) : -1;
            }
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int p = tid + u * nthreads;
                if (p < np) {
                    const __half d = h_from_bits(key_bits(key[u]));
                    q.dist[n * q.P + p0 + p] = d;
                    const __half hv = h_mul(d, __float2half_rn(0.5f));                       // fp16(dist / 2)
                    if (q.obs) {
                        const float v = __half2float(hv);
                        if (ca[u] >= 0) q.obs[n * q.obs_ld + ca[u]] = v;
                        if (cb[u] >= 0) q.obs[n * q.obs_ld + cb[u]] = v;
                    }
                    if (q.obs16) {
                        if (ca[u] >= 0) q.obs16[n * q.obs16_ld + (ca[u] - q.obs16_col0)] = hv;
                        if (cb[u] >= 0) q.obs16[n * q.obs16_ld + (cb[u] - q.obs16_col0)] = hv;
                    }
                }
            }
            return;
        }
    }
    for (int p = tid; p < np; p += nthreads) {
        uint32_t key = res[p];
        const bool far_hit = (far[p >> 5] >> (p & 31)) & 1u;
        if (far_hit && (key >> 16) == ORD_MISS) {
            const double* pp = q.pattern + (int64_t)(p0 + p) * 3;
            double xo, yo, zo;
            body_transform<double>(pp[0], pp[1], pp[2], tr, tx, ty, tz, xo, yo, zo);
            const H3 s = {h_from_double(xo), h_from_double(yo), h_from_double(zo)};
            const int2 c = ray_cell(s.x, s.y, q.shift_x, q.shift_y, q.res, q.inv_res, q.G0, q.G1, q.sem);
            if (q.index) {
                key = literal_ray(q.index + ((int64_t)c.x * q.G1 + c.y) * q.Ks, q.K, q.recs, s, dlit);
            } else {
                const uint32_t bi = (uint32_t)(c.x / RVB_BLK) * (uint32_t)q.nBy + (uint32_t)(c.y / RVB_BLK);
                const uint32_t o0 = __ldg(q.blk_off + bi), o1 = __ldg(q.blk_off + bi + 1);
                key = literal_ray_blk(q.blk_ids + o0, q.blk_slots + o0, (int)(o1 - o0), (c.x % RVB_BLK) * RVB_BLK + c.y % RVB_BLK, q.recs, s, dlit);
            }
        }
        const unsigned short kb = key_bits(key);
        const int slot = (int)((key >> 1) & 0x7fffu);
        const int64_t o = n * q.P + p0 + p;
        q.dist[o] = h_from_bits(kb);
        if (q.hit_slot) q.hit_slot[o] = slot;
        if (want_geo) {
            const double* pp = q.pattern + (int64_t)(p0 + p) * 3;
            double xo, yo, zo;
            body_transform<double>(pp[0], pp[1], pp[2], tr, tx, ty, tz, xo, yo, zo);
            const __half hx = h_from_double(xo), hy = h_from_double(yo), hz = h_from_double(zo);
            if (q.sources) { q.sources[o * 3 + 0] = hx; q.sources[o * 3 + 1] = hy; q.sources[o * 3 + 2] = hz; }
            if (q.hit_tri) {
                const int2 c = ray_cell(hx, hy, q.shift_x, q.shift_y, q.res, q.inv_res, q.G0, q.G1, q.sem);
                if (q.index) {
                    q.hit_tri[o] = __ldg(q.index + ((int64_t)c.x * q.G1 + c.y) * q.Ks + slot);
                } else {
                    const uint32_t bi = (uint32_t)(c.x / RVB_BLK) * (uint32_t)q.nBy + (uint32_t)(c.y / RVB_BLK);
                    const uint32_t o0 = __ldg(q.blk_off + bi), o1 = __ldg(q.blk_off + bi + 1);
                    q.hit_tri[o] = tri_of_slot_blk(q.blk_ids + o0, q.blk_slots + o0, (int)(o1 - o0), (c.x % RVB_BLK) * RVB_BLK + c.y % RVB_BLK, slot);
                }
            }
            if (q.pt) {
                const __half k = h_from_bits(kb);
                q.pt[o * 3 + 0] = h_sub(hx, h_mul(__low2half(dx2), k));     // ray_casting.py:63
                q.pt[o * 3 + 1] = h_sub(hy, h_mul(__low2half(dy2), k));
                q.pt[o * 3 + 2] = h_sub(hz, h_mul(__low2half(dz2), k));
            }
        }
        if (q.obs) {
            const float v = __half2float(h_mul(h_from_bits(kb), __float2half_rn(0.5f)));     // fp16(dist / 2) -> f32
            const int ca = q.col_a[p0 + p], cb = q.col_b[p0 + p];
            if (ca >= 0) q.obs[n * q.obs_ld + ca] = v;
            if (cb >= 0) q.obs[n * q.obs_ld + cb] = v;
        }
        if (q.obs16) {                                                                        // the same value, kept in fp16
            const __half v = h_mul(h_from_bits(kb), __float2half_rn(0.5f));
            const int ca = q.col_a[p0 + p], cb = q.col_b[p0 + p];
            if (ca >= 0) q.obs16[n * q.obs16_ld + (ca - q.obs16_col0)] = v;
            if (cb >= 0) q.obs16[n * q.obs16_ld + (cb - q.obs16_col0)] = v;
        }
    }
}

}  // namespace rc

