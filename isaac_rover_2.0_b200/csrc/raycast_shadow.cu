// Production heightmap ray-cast kernel ("shadow" culling): Camera.get_depths (camera.py:60-145) in one launch.
//
// The reference tests every ray against the K = 200 candidates of its cell; about 1.5 of them are hits.  All rays of
// an env share ONE direction d (camera.py:202-207), so a triangle's pre-image under the test -- the set of sources s
// that can pass `n >= -eps, m >= -eps, n + m <= 1 + eps` -- is a prism parallel to d, and the sources lie on a plane
// (the pattern has constant z).  The kernel therefore enumerates TRIANGLES, not (ray, candidate) pairs:
//
//   classify   (hm_classify_kernel, one thread per env) steep envs go on the tiled kernel's work list, cast concurrently on a
//              second stream; the others are ordered tilted-first (their CTAs are the slow ones);
//   phase 1/2  (as raycast_tiled.cu) fp64 body transform -> fp16 sources, cell lookup, counting sort of the tile's rays
//              into column-major bins of 2x2 cells (shared memory; a cell rectangle is a few contiguous ranges);
//   stage 1    per (superblock, triangle of its list -- the union of the K-lists of 8x8 blocks): a bounding disc of the
//              prism's cross-section on the source plane against the rectangle of the superblock's rays, from the
//              triangle's pre-computed 32-byte stage-1 record (centroid, radius, b x c; terrain.cu);
//   stage 2    survivors: exact corners of the cross-section -> xy box -> bin columns -> ray ranges (tasks);
//   stage 3L   rays of a task (one triangle, <= 20 consecutive sorted rays; one task per lane) against the prism ITSELF: the
//              exact linear forms N* = (s - a) . (c x d), M* = (s - a) . (d x b) in fp32 (three packed FFMA2 per ray) against
//              the thresholds stage 2 derived for the triangle -- the same three half-planes whose corners make the box;
//   stage 3b   the (ray, triangle) pairs left (about 1.2 per hit): LITERAL evaluation of ray_casting.py:34-59 with its
//              three IEEE divisions, membership + slot of the triangle in the ray's own cell list (one byte of the superblock
//              entry's per-cell slot table, sb_slot9), atomicMin on (order-preserving fp16 bits, slot) = torch.min.
// Two instantiations: <= 1664 rays per tile (64 registers, 55 KB shared memory, 4 CTAs per SM) and <= 2048 (3 CTAs per SM).
//
// Bit-exactness rests on stage 3b alone; stages 1-3L only have to be CONSERVATIVE (never drop a pair the literal test
// would accept).  The bound: with g = s - a, the reference's numerators N = fl((g x c) . d), M = fl((b x g) . d) differ
// from the exact N* = n det*, M* = m det* (det* = (b x c) . d, s = a + n b + m c + t d) by at most
//     E = GAMMA * |g|_2 * sum_i aw_i + ALPHA,   aw_i = |c_j||d_k| + |c_k||d_j|,   GAMMA = 2^-8 >= (1 + 2^-11)^6 - 1
// (six fp16 roundings per term, ALPHA for subnormal products), so a passing source satisfies
//     n >= -(tlo + E_N)/|det*|,  m >= -(tlo + E_M)/|det*|,  n + m <= (thi' + E_N + E_M)/|det*|
// with tlo/thi the outward-rounded fp16 thresholds of the packed pre-filter of raycast_tiled.cu (a superset of the
// literal test).  |g| is bounded self-consistently from the disc of stage 1.  Triangles for which no bound holds
// (|det*| within rounding of 0, fp16 overflow possible, NaN) are tested against every ray of the superblock.
// tests/shadow_proto.py re-states stages 1-2 in numpy and checks them against a brute-force fp16 evaluation;
// tests/test_shadow_bound_cpu.py runs it.  Tiles this kernel cannot group (rays spread over more than 6144 bins or
// 64 superblocks, a list longer than the queue encoding, fp16 overflow) are handed to the tiled kernel through a second
// work list.
#include <ctype.h>
#include <errno.h>
#include <stdlib.h>

#include <cub/device/device_radix_sort.cuh>

#include "raycast_common.cuh"
#include "shadow_bounds.cuh"

namespace {

using namespace rc;

constexpr int TT = 256;
constexpr int NW = TT / 32;
constexpr int RT_MAX = 2048;       // rays per tile; must equal raycast_tiled.cu's (shared tiling of the fall-back list)
constexpr int BIN_CAP = 2048;      // bins in the tile's bounding box (2x2-cell bins: a 3.4 m x 6.6 m pattern at 45 degrees of yaw needs ~1300)
constexpr int SB = RVB_SB;          // blocks per superblock side
constexpr int SBC = RVB_SB * RVB_BLK;   // cells per superblock side
constexpr int ITEM_CAP = 64;       // superblocks per tile (7 bits travel in the stage-1 queue)
constexpr int CHUNK = 32;          // list entries per pulled work chunk (one stage-1 batch)
constexpr int CHUNK_CAP = 1024;    // chunks per tile (u8 chunk -> item table)
constexpr int QCAP = 64;           // per-warp queues q1, q2 (each drained below 32 after every push of <= 32)
constexpr int QCAP3 = 128;         // q4 (stage 3L pushes while it holds < 32 entries, stage 3b drains in batches of 32)
constexpr int TASK_RAYS = 20;      // rays per task (<= 32: one mask bit each); sweep with the shipped kernel: 8 +5 %, 12 +1 %, 16 +0.45 %, 20 best, 24 +0.2 %, 32 +1 %
constexpr int MIN_SH = 1;          // finest bins: 2x2 cells, 2 % faster than single cells (fewer tasks)
constexpr float COS_STEEP = 0.7f;  // envs whose ray direction has |d_z| below this go to the tiled kernel (their prisms are long
                                   // slivers); 0.8 until a sweep: -0.6 % at 0.7.  Results do not depend on it
constexpr int REL_BITS = 15;        // queue entries name a triangle as item << 15 | position in the item's list
constexpr int ILL_CAP = 128;        // triangles without a bound ("ill": fp16 determinant within rounding of zero) a tile may meet before it
                                   // is handed to the tiled kernel, whose cost does not depend on them (a 1M-triangle heightfield has ~1
                                   // per tile; a mesh finer than the fp16 grid of its coordinates has hundreds)
constexpr int RT_SMALL = 1664;      // ray capacity of the 4-CTAs-per-SM instantiation (the reference pattern has 1634 rays)

struct Item {
    uint32_t list_off, list_len;
    float rlox, rhix, rloy, rhiy;   // rectangle holding the sources of the superblock's rays
    uint32_t bx;                    // bin columns with rays: lo | hi << 16 (absolute bin coordinates)
    uint32_t by;
};
static_assert(sizeof(Item) == 32, "Item");

struct Smem {
    uint2* rays;         // [RT]  sorted by block: (sx | sy << 16, sz | (p | (cy % 24) << 11) << 16)
    uint32_t* res;       // [RT]  best key per local ray id
    uint32_t* bins;      // [BIN_CAP / 2 + 2]  u16 counters, then exclusive offsets (column-major bins)
    Item* items;         // [ITEM_CAP]
    uint32_t* cum;       // [ITEM_CAP + 1]  chunks before item i
    unsigned char* chunk_item;   // [CHUNK_CAP]  item of the k-th chunk that survived the window cull
    unsigned short* chunk_win;   // [CHUNK_CAP]  its window, relative to the first window of the item's list
    uint2* q1;           // [NW][QCAP]  stage-1 survivors: (superblock-list entry, gball bits | item)
    uint4* q2;           // [NW][QCAP]  tasks: (item << 15 | list position, ray start | count << 16, T1 | T2 << 16, T3 | sign << 15)
    uint32_t* q4;        // [NW][QCAP3]  pairs inside the prism: ray position | (item << 15 | list position) << 11
    int32_t* q1t;        // [NW][QCAP]   triangle id of the q1 / q2 / q4 entry: travels with it, so that no stage has to go back to
    int32_t* q2t;        // [NW][QCAP]   sb_ids (a dependent global load in front of every record fetch)
    int32_t* q4t;        // [NW][QCAP3]
    uint32_t* far;       // [RT / 32]
};

__host__ __device__ inline size_t shadow_smem_bytes(int RT) {       // RT = ray capacity of the instantiation
    return (size_t)RT * 8 + (size_t)((RT + 3) & ~3) * 4 + (size_t)(BIN_CAP / 2 + 4) * 4 + (size_t)ITEM_CAP * 32 +
           (size_t)(ITEM_CAP + 4) * 4 + (size_t)CHUNK_CAP * 3 + (size_t)NW * (QCAP * (8 + 16 + 4 + 4) + QCAP3 * (4 + 4)) + (size_t)(((RT + 31) / 32 + 3) & ~3) * 4;
}

// bins are u16 pairs packed into the u32 words the histogram's atomicAdd works on (little endian: even bin = low half)
__device__ __forceinline__ uint32_t off16(const uint32_t* bins, int bin) { return reinterpret_cast<const unsigned short*>(bins)[bin]; }

// monotone non-decreasing in v (the arithmetic of cell_coord on an fp32 coordinate)
__device__ __forceinline__ int cell_coord_f(float x, float shift, float res, float inv_res, int gmax, int sem) {
    float v = __fsub_rn(x, shift);
    v = (sem == RVB_SEM_TORCH_CPU) ? __fdiv_rn(v, res) : __fmul_rn(v, inv_res);
    v = fminf(fmaxf(v, 0.0f), (float)gmax);
    return (int)rintf(v);
}

struct TriF {
    float ax, ay, az, bx, by, bz, cx, cy, cz;
};
__device__ __forceinline__ TriF tri_f(const uint4& q0, const uint2& q1) {
    TriF t;
    t.ax = hf(q0.x & 0xffff); t.ay = hf(q0.x >> 16); t.az = hf(q0.y & 0xffff);
    t.bx = hf(q0.y >> 16); t.by = hf(q0.z & 0xffff); t.bz = hf(q0.z >> 16);
    t.cx = hf(q0.w & 0xffff); t.cy = hf(q0.w >> 16); t.cz = hf(q1.x & 0xffff);
    return t;
}

// positive fp32 (or +inf) -> its upper 16 bits, rounded up
__device__ __forceinline__ uint32_t bf16_up(float x) { return (__float_as_uint(x) + 0xFFFFu) >> 16; }

// Stage 2 (tests/shadow_proto.py: stage2): xy box of the sources that can pass; full = no bound.  T12 / T3s: the thresholds of
// the three half-planes N' >= -T1, M' >= -T2, N' + M' <= T3 that bound the prism (un-normalised: N' = sgn N*, ...), 16 bits each,
// rounded up, with the sign of the literal det in bit 15 of T3s -- what stage 3L tests every ray of the triangle's tasks against.
__device__ __forceinline__ void stage2(const TriF& t, const uint2& q1, const EnvC& e, H3 d16, float gball, float& x0, float& x1,
                                       float& y0, float& y1, bool& full, uint32_t& T12, uint32_t& T3s) {
    const __half n0 = h_from_bits(q1.x >> 16), n1 = h_from_bits(q1.y & 0xffff), n2 = h_from_bits(q1.y >> 16);
    const __half det_h = h_add(h_add(h_mul(n0, d16.x), h_mul(n1, d16.y)), h_mul(n2, d16.z));           // ray_casting.py:41
    const __half da = __habs(det_h);
    const float tlo = __half2float(__hfma(da, h_from_bits(0x2E68u), h_from_bits(0x0002u)));              // = -tlo of the pre-filter
    const float thi = __half2float(__hfma(da, h_from_bits(0x3C6Bu), h_from_bits(0x0002u)));
    const float wx = t.cy * e.dz - t.cz * e.dy, wy = t.cz * e.dx - t.cx * e.dz, wz = t.cx * e.dy - t.cy * e.dx;    // c x d
    const float dets = fmaf(t.bx, wx, fmaf(t.by, wy, t.bz * wz));
    const float adx = fabsf(e.dx), ady = fabsf(e.dy), adz = fabsf(e.dz);
    const float acx = fabsf(t.cx), acy = fabsf(t.cy), acz = fabsf(t.cz), abx = fabsf(t.bx), aby = fabsf(t.by), abz = fabsf(t.bz);
    const float saw = fmaf(acy + acz, adx, fmaf(acz + acx, ady, (acx + acy) * adz));
    const float sawp = fmaf(aby + abz, adx, fmaf(abz + abx, ady, (abx + aby) * adz));
    const float rdet = __fdividef(1.0f, fabsf(dets)) * 1.001f;
    const float EN = fmaf(GAMMA * gball, saw, ALPHA), EM = fmaf(GAMMA * gball, sawp, ALPHA);
    const float l1 = (tlo + EN) * rdet, l2 = (tlo + EM) * rdet;
    const float t3 = fmaf(thi, 1.0009766f, 5.9604645e-08f) + EN + EM;
    const float l3 = t3 * rdet;
    const bool sign_ok = (__float_as_uint(dets) >> 31) == (uint32_t)(h_bits(det_h) >> 15);
    const bool good = sign_ok && (fmaxf(fmaxf(l1, l2), l3) <= L_CAP) && (l1 == l1) && (l2 == l2) && (l3 == l3);
    x0 = y0 = __int_as_float(0x7f800000);
    x1 = y1 = __int_as_float(0xff800000);
    float ext = 0.0f;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const float cn = (k == 1) ? (l3 + l2) : -l1, cm = (k == 2) ? (l3 + l1) : -l2;       // corners A, B, C in (n, m)
        const float Px = fmaf(cn, t.bx, fmaf(cm, t.cx, t.ax)), Py = fmaf(cn, t.by, fmaf(cm, t.cy, t.ay)),
                    Pz = fmaf(cn, t.bz, fmaf(cm, t.cz, t.az));
        const float nP = fmaf(Px, e.nux, fmaf(Py, e.nuy, Pz * e.nuz));
        const float t0 = (e.hlo - nP) * e.inv_nd, t1 = (e.hhi - nP) * e.inv_nd;
        const float xa = fmaf(t0, e.dx, Px), xb = fmaf(t1, e.dx, Px), ya = fmaf(t0, e.dy, Py), yb = fmaf(t1, e.dy, Py);
        x0 = fminf(x0, fminf(xa, xb)); x1 = fmaxf(x1, fmaxf(xa, xb));
        y0 = fminf(y0, fminf(ya, yb)); y1 = fmaxf(y1, fmaxf(ya, yb));
        ext = fmaxf(ext, fmaxf(fabsf(xa), fabsf(xb)) + fmaxf(fabsf(ya), fabsf(yb)));
    }
    const float sl = fmaf(ext, 7.6293945e-06f, 9.5367432e-07f);       // 2 * 2^-18 (ext is max |x| + |y| of one corner), 2^-20
    x0 -= sl; x1 += sl; y0 -= sl; y1 += sl;
    full = !good || !(x0 <= x1) || !(y0 <= y1);
    T12 = full ? 0x7F807F80u : (bf16_up((tlo + EN) * LIN_SLACK) | (bf16_up((tlo + EM) * LIN_SLACK) << 16));
    T3s = full ? 0x7F80u : (bf16_up(t3 * LIN_SLACK) | ((uint32_t)(h_bits(det_h) >> 15) << 15));
}

__device__ __forceinline__ bool is_steep(const H3& d16, float cos_steep) { return !(fabsf(__half2float(d16.z)) >= cos_steep); }

constexpr int ORDER_SH = 3;          // the env order's map cells: 2^3 x 2^3 index cells (0.8 m at the reference's 0.1 m)

// v's low 16 bits spread to the even bits
__device__ __forceinline__ uint32_t spread_bits(uint32_t v) {
    v &= 0xffffu;
    v = (v | (v << 8)) & 0x00ff00ffu;
    v = (v | (v << 4)) & 0x0f0f0f0fu;
    v = (v | (v << 2)) & 0x33333333u;
    return (v | (v << 1)) & 0x55555555u;
}

// One thread per env: the ray direction as the kernels compute it -> steep envs onto the tiled kernel's work list (every tile,
// with `steep_list`), and (with `keys`) the env's key of the order the shadow and rock kernels cast envs in: tilted envs (long
// shadows = slow CTAs) first, then the rest; within each class the Z-order code of the env's map cell, so that the CTAs resident
// at one time read the candidate lists, records and slot table of one small patch of the map, from L2.
__global__ void hm_classify_kernel(const TiledParams q, int64_t N, int zbits, uint32_t* __restrict__ keys, int32_t* __restrict__ ids,
                                   int* __restrict__ steep_count, int32_t* __restrict__ steep_list) {
    const int64_t n = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (n >= N) return;
    const float px = q.pos[n * 3 + 0], py = q.pos[n * 3 + 1];
    const Trig tr = make_trig(q.euler, q.trig, n);
    const H3 d16 = env_dir16(tr, (double)px, (double)py, (double)q.pos[n * 3 + 2]);
    const bool steep = is_steep(d16, q.cos_steep);
    if (steep && steep_list) {
        const int at = atomicAdd(steep_count, q.tiles);
        for (int t = 0; t < q.tiles; ++t) steep_list[at + t] = (int32_t)(n * q.tiles + t);
    }
    if (keys) {
        const bool tilted = !steep && !(fabsf(__half2float(d16.z)) >= 0.97f);
        const uint32_t cx = (uint32_t)cell_coord_f(px, q.shift_x, q.res, q.inv_res, q.G0 - 1, q.sem) >> ORDER_SH;
        const uint32_t cy = (uint32_t)min(cell_coord_f(py, q.shift_y, q.res, q.inv_res, q.G0 - 1, q.sem), q.G1 - 1) >> ORDER_SH;
        keys[n] = ((tilted ? 0u : 1u) << (2 * zbits)) | spread_bits(cx) << 1 | spread_bits(cy);
        ids[n] = (int32_t)n;
    }
}

template <bool DBGK, int RTC>
__global__ void __launch_bounds__(TT, RTC <= RT_SMALL ? 4 : 3) hm_shadow_kernel(const TiledParams q) {
    extern __shared__ uint4 smem_raw[];
    __shared__ int s_box[4];
    __shared__ float s_red[NW][12];
    __shared__ uint32_t s_warp[NW];
    __shared__ EnvC s_env;
    __shared__ int s_next, s_nitems, s_nchunks, s_bail, s_ill;
    __shared__ int s_bkt[2][8];                        // window cull: windows per cost bucket, then the next free slot of each
    __shared__ unsigned short s_item_rays[ITEM_CAP];   // rays per item (by rank)

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // The envs at the end of the order are cut in two (rays [0, split_at) and [split_at, P), one CTA each): the grid's last wave
    // then consists of CTAs of half the duration, which shortens the tail where SMs wait for the last CTAs (tiles == 1 only).
    int64_t opos = blockIdx.x / q.tiles;
    int tile = blockIdx.x % q.tiles, p0_ = tile * q.tile_size, np_ = min(q.tile_size, q.P - p0_);
    if (q.split_from >= 0 && (int64_t)blockIdx.x >= q.split_from) {
        const int64_t k = (int64_t)blockIdx.x - q.split_from;
        opos = q.split_from + (k >> 1);
        tile = 0;
        p0_ = (k & 1) ? q.split_at : 0;
        np_ = (k & 1) ? q.P - q.split_at : q.split_at;
    }
    const int64_t n = __ldg(q.order + opos);
    const int32_t work_id = (int32_t)(n * q.tiles + tile);
    const int p0 = p0_;
    const int np = np_;
    const int RT = q.tile_size;

    Smem sm;
    // fixed layout (sized for RTC rays): every shared-memory address is base + constant, nothing to keep in registers
    sm.rays = reinterpret_cast<uint2*>(smem_raw);
    sm.res = reinterpret_cast<uint32_t*>(sm.rays + RTC);
    sm.bins = sm.res + RTC;
    sm.items = reinterpret_cast<Item*>(sm.bins + BIN_CAP / 2 + 4);
    sm.cum = reinterpret_cast<uint32_t*>(sm.items + ITEM_CAP);
    sm.chunk_item = reinterpret_cast<unsigned char*>(sm.cum + ITEM_CAP + 4);
    sm.chunk_win = reinterpret_cast<unsigned short*>(sm.chunk_item + CHUNK_CAP);
    sm.q1 = reinterpret_cast<uint2*>(sm.chunk_win + CHUNK_CAP);
    sm.q2 = reinterpret_cast<uint4*>(sm.q1 + NW * QCAP);
    sm.q4 = reinterpret_cast<uint32_t*>(sm.q2 + NW * QCAP);
    sm.q1t = reinterpret_cast<int32_t*>(sm.q4 + NW * QCAP3);
    sm.q2t = sm.q1t + NW * QCAP;
    sm.q4t = sm.q2t + NW * QCAP;
    sm.far = reinterpret_cast<uint32_t*>(sm.q4t + NW * QCAP3);

    // ---- phase 0
    for (int i = tid; i < BIN_CAP / 2 + 4; i += TT) sm.bins[i] = 0u;
    for (int i = tid; i < (RT + 31) / 32; i += TT) sm.far[i] = 0u;
    if (tid == 0) {
        s_box[0] = s_box[1] = 0x7fffffff;
        s_box[2] = s_box[3] = -1;
        s_next = 0;
        s_bail = 0;
        s_ill = 0;
    }
    const Trig tr = make_trig(q.euler, q.trig, n);
    const double tx = (double)q.pos[n * 3 + 0], ty = (double)q.pos[n * 3 + 1], tz = (double)q.pos[n * 3 + 2];
    const H3 d16 = env_dir16(tr, tx, ty, tz);
    const __half2 dx2 = __half2half2(d16.x), dy2 = __half2half2(d16.y), dz2 = __half2half2(d16.z);
    // rays nearly horizontal in the WORLD (steep env): hm_classify_kernel put this env on the tiled kernel's list already
    if (is_steep(d16, q.cos_steep)) return;
    __syncthreads();

    // ---- phase 1: sources, cells, ranges
    constexpr int RPT = (RTC + TT - 1) / TT;
    uint32_t r_sxy[RPT], r_sz[RPT];
    int r_cell[RPT];
    int mnx = 0x7fffffff, mny = 0x7fffffff, mxx = -1, mxy = -1;
    float lo_x = __int_as_float(0x7f800000), lo_y = lo_x, hi_x = -lo_x, hi_y = -lo_x, amax_s = 0.0f;
    float pz_lo = lo_x, pz_hi = -lo_x, pxy = 0.0f;
    bool bad = false;
#pragma unroll
    for (int i = 0; i < RPT; ++i) {
        const int p = tid + i * TT;
        r_cell[i] = -1;
        if (p < np) {
            const double* pp = q.pattern + (int64_t)(p0 + p) * 3;
            const double px = pp[0], py = pp[1], pz = pp[2];
            double xo, yo, zo;
            body_transform<double>(px, py, pz, tr, tx, ty, tz, xo, yo, zo);
            const __half hx = h_from_double(xo), hy = h_from_double(yo), hz = h_from_double(zo);
            r_sxy[i] = (uint32_t)h_bits(hx) | ((uint32_t)h_bits(hy) << 16);
            const int2 c = ray_cell(hx, hy, q.shift_x, q.shift_y, q.res, q.inv_res, q.G0, q.G1, q.sem);
            // (the 5 spare bits next to p: the cell's y within its superblock, half of the slot-table index of stage 3b)
            r_sz[i] = (uint32_t)h_bits(hz) | (((uint32_t)p | ((uint32_t)(c.y % SBC) << 11)) << 16);
            r_cell[i] = (c.x << 16) | c.y;
            mnx = min(mnx, c.x); mxx = max(mxx, c.x); mny = min(mny, c.y); mxy = max(mxy, c.y);
            const float fx = __half2float(hx), fy = __half2float(hy), fz = __half2float(hz);
            lo_x = fminf(lo_x, fx); hi_x = fmaxf(hi_x, fx); lo_y = fminf(lo_y, fy); hi_y = fmaxf(hi_y, fy);
            amax_s = fmaxf(amax_s, fmaxf(fmaxf(fabsf(fx), fabsf(fy)), fabsf(fz)));
            bad |= !(fabsf(fx) <= 65504.0f) || !(fabsf(fy) <= 65504.0f) || !(fabsf(fz) <= 65504.0f);
            pz_lo = fminf(pz_lo, __double2float_rd(pz)); pz_hi = fmaxf(pz_hi, __double2float_ru(pz));
            pxy = fmaxf(pxy, fmaxf(fabsf(__double2float_ru(fabs(px))), fabsf(__double2float_ru(fabs(py)))));
        }
    }
    mnx = __reduce_min_sync(0xffffffffu, mnx); mny = __reduce_min_sync(0xffffffffu, mny);
    mxx = __reduce_max_sync(0xffffffffu, mxx); mxy = __reduce_max_sync(0xffffffffu, mxy);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        lo_x = fminf(lo_x, __shfl_xor_sync(0xffffffffu, lo_x, o)); hi_x = fmaxf(hi_x, __shfl_xor_sync(0xffffffffu, hi_x, o));
        lo_y = fminf(lo_y, __shfl_xor_sync(0xffffffffu, lo_y, o)); hi_y = fmaxf(hi_y, __shfl_xor_sync(0xffffffffu, hi_y, o));
        amax_s = fmaxf(amax_s, __shfl_xor_sync(0xffffffffu, amax_s, o));
        pz_lo = fminf(pz_lo, __shfl_xor_sync(0xffffffffu, pz_lo, o)); pz_hi = fmaxf(pz_hi, __shfl_xor_sync(0xffffffffu, pz_hi, o));
        pxy = fmaxf(pxy, __shfl_xor_sync(0xffffffffu, pxy, o));
    }
    bad = __any_sync(0xffffffffu, bad);
    if (lane == 0) {
        atomicMin(&s_box[0], mnx); atomicMin(&s_box[1], mny);
        atomicMax(&s_box[2], mxx); atomicMax(&s_box[3], mxy);
        float* w = s_red[warp];
        w[0] = lo_x; w[1] = hi_x; w[2] = lo_y; w[3] = hi_y; w[4] = amax_s; w[5] = pz_lo; w[6] = pz_hi; w[7] = pxy;
        if (bad) s_bail = 1;
    }
    __syncthreads();
    // bins: 2^sh x 2^sh cells, the finest that lets the tile's bounding box fit the histogram (sh = 0 for a rover on its wheels);
    // 2^sh divides the superblock side (24 cells), so bins never straddle superblocks
    int sh = q.min_sh;
    while (sh < 3 && (int64_t)((s_box[2] >> sh) - (s_box[0] >> sh) + 1) * ((s_box[3] >> sh) - (s_box[1] >> sh) + 1) > BIN_CAP) ++sh;
    const int bx0 = s_box[0] >> sh, by0 = s_box[1] >> sh;          // (bx0, by0, BW, BH: bounding box of the tile's rays in BINS)
    const int BW = (s_box[2] >> sh) - bx0 + 1, BH = (s_box[3] >> sh) - by0 + 1;
    const int SBB = SBC >> sh;                                       // bins per superblock side
    const int sbx0 = bx0 / SBB, sby0 = by0 / SBB;
    const int nsx = (s_box[2] >> sh) / SBB - sbx0 + 1, nsy = (s_box[3] >> sh) / SBB - sby0 + 1;
    float g_lox = s_red[0][0], g_hix = s_red[0][1], g_loy = s_red[0][2], g_hiy = s_red[0][3];
    {
        float a_s = s_red[0][4], z0 = s_red[0][5], z1 = s_red[0][6], pm = s_red[0][7];
#pragma unroll
        for (int w = 1; w < NW; ++w) {
            g_lox = fminf(g_lox, s_red[w][0]); g_hix = fmaxf(g_hix, s_red[w][1]);
            g_loy = fminf(g_loy, s_red[w][2]); g_hiy = fmaxf(g_hiy, s_red[w][3]);
            a_s = fmaxf(a_s, s_red[w][4]); z0 = fminf(z0, s_red[w][5]); z1 = fmaxf(z1, s_red[w][6]); pm = fmaxf(pm, s_red[w][7]);
        }
        if (tid == 0) {
            // source plane: s = t + x c1 + y c2 + z c3 (columns of camera.py:197-199), nu = c1 x c2 (tests/shadow_proto.py: EnvConsts)
            const double sx = tr.sx, cx = tr.cx, sy = tr.sy, cy = tr.cy, sz = tr.sz, cz = tr.cz;
            const double c1x = cz * cy, c1y = -sz * cy, c1z = sy;
            const double c2x = sz * cx + cz * sy * sx, c2y = cz * cx - sz * sy * sx, c2z = -cy * sx;
            const double c3x = sz * sx - cz * sy * cx, c3y = cz * sx + sz * sy * cx, c3z = cy * cx;
            const float nux = (float)(c1y * c2z - c1z * c2y), nuy = (float)(c1z * c2x - c1x * c2z), nuz = (float)(c1x * c2y - c1y * c2x);
            const double h0 = (double)nux * tx + (double)nuy * ty + (double)nuz * tz;
            const double k1 = (double)nux * c1x + (double)nuy * c1y + (double)nuz * c1z;
            const double k2 = (double)nux * c2x + (double)nuy * c2y + (double)nuz * c2z;
            const double k3 = (double)nux * c3x + (double)nuy * c3y + (double)nuz * c3z;
            const double ha = h0 + (double)z0 * k3, hb = h0 + (double)z1 * k3;
            // half ulp of the largest source coordinate (sources are fp16 values); every coordinate moves by at most that
            const uint32_t ab = __float_as_uint(a_s);
            const int ex = (int)(ab >> 23) - 127;
            const float qh = (ex >= -14) ? __uint_as_float((uint32_t)(ex - 11 + 127) << 23) : 2.9802322e-08f;
            const double an = fabs((double)nux) + fabs((double)nuy) + fabs((double)nuz);
            // tau: rounding of the sources + the fp32 evaluation of nu . P in the stages + pattern x/y leakage
            const double tau = an * (double)qh * 1.01 + (double)pm * (fabs(k1) + fabs(k2)) +
                               1e-6 * (fabs(ha) + fabs(hb) + an * ((double)a_s + 16.0)) + 1e-7;
            EnvC e;
            e.dx = __half2float(d16.x); e.dy = __half2float(d16.y); e.dz = __half2float(d16.z);
            e.nux = nux; e.nuy = nuy; e.nuz = nuz;
            const float nd = fmaf(nux, e.dx, fmaf(nuy, e.dy, nuz * e.dz));
            e.inv_nd = 1.0f / nd;
            e.hlo = __double2float_rd(fmin(ha, hb) - tau);
            e.hhi = __double2float_ru(fmax(ha, hb) + tau);
            e.hmid = 0.5f * (e.hlo + e.hhi);
            const float dn = sqrtf(fmaf(e.dx, e.dx, fmaf(e.dy, e.dy, e.dz * e.dz))) * 1.000001f;
            const float nn = sqrtf(fmaf(nux, nux, fmaf(nuy, nuy, nuz * nuz))) * 1.000001f;
            e.dn = dn;
            e.kappa = dn * nn / fabsf(nd) * 1.00001f;
            e.lam = dn * (0.5f * (e.hhi - e.hlo) + 1e-6f * (fabsf(e.hlo) + fabsf(e.hhi))) / fabsf(nd) * 1.00001f + 1e-7f;
            e.smax = a_s;
            s_env = e;
            // cos of the angle between the rays and the plane normal ~ 1; steep = rays nearly horizontal in the WORLD
            const bool steep = is_steep(d16, q.cos_steep);
            const bool ungrouped = (int64_t)BW * BH > BIN_CAP || (int64_t)nsx * nsy > ITEM_CAP;
            const bool degenerate = !(fabsf(nd) > 0.5f) || !(e.kappa < 2.0f) || !(e.lam < 1e4f) || !(a_s <= 65504.0f);
            if (steep || ungrouped || degenerate) s_bail = 1;
        }
    }
    __syncthreads();
    if (s_bail) {
        // hand this (env, tile) to the tiled kernel
        if (tid == 0) q.fb_list[atomicAdd(q.fb_count, 1)] = work_id;
        return;
    }

    // ---- phase 2: counting sort by cell, column-major bins
    {
        uint32_t r_rank[RPT];
#pragma unroll
        for (int i = 0; i < RPT; ++i) {
            if (r_cell[i] >= 0) {
                const int bin = (((r_cell[i] >> 16) >> sh) - bx0) * BH + (((r_cell[i] & 0xffff) >> sh) - by0);
                const uint32_t old = atomicAdd(&sm.bins[bin >> 1], 1u << ((bin & 1) * 16));
                r_rank[i] = (old >> ((bin & 1) * 16)) & 0xffffu;
            }
        }
        __syncthreads();
        // exclusive scan in bin order: thread t owns the contiguous words [t * wpt, (t + 1) * wpt)
        const int nwords = ((BW * BH) >> 1) + 1;                 // covers bins 0 .. BW*BH (sentinel = total)
        const int wpt = (nwords + TT - 1) / TT;
        const int w0 = tid * wpt, w1 = min(w0 + wpt, nwords);
        uint32_t tot = 0;
        for (int w = w0; w < w1; ++w) {
            const uint32_t v = sm.bins[w];
            tot += (v & 0xffffu) + (v >> 16);
        }
        uint32_t inc = tot;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t v = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += v;
        }
        if (lane == 31) s_warp[warp] = inc;
        __syncthreads();
        uint32_t run = inc - tot;
#pragma unroll
        for (int w = 0; w < NW; ++w)
            if (w < warp) run += s_warp[w];
        for (int w = w0; w < w1; ++w) {
            const uint32_t v = sm.bins[w];
            const uint32_t a = v & 0xffffu, b = v >> 16;
            sm.bins[w] = run | ((run + a) << 16);
            run += a + b;
        }
        __syncthreads();
#pragma unroll
        for (int i = 0; i < RPT; ++i) {
            if (r_cell[i] >= 0) {
                const int p = tid + i * TT;
                const int bin = (((r_cell[i] >> 16) >> sh) - bx0) * BH + (((r_cell[i] & 0xffff) >> sh) - by0);
                sm.rays[off16(sm.bins, bin) + r_rank[i]] = make_uint2(r_sxy[i], r_sz[i]);
                sm.res[p] = KEY_INIT;
            }
        }
    }
    // ---- superblock items: block rectangle with rays, source rectangle, candidate list
    const int nsb = nsx * nsy;
    int* it_red = reinterpret_cast<int*>(sm.q2);          // [5][ITEM_CAP] bx lo, bx hi, by lo, by hi, rays (queues are idle here)
    for (int i = tid; i < nsb; i += TT) {
        it_red[i] = 0x7fffffff; it_red[ITEM_CAP + i] = -1;
        it_red[2 * ITEM_CAP + i] = 0x7fffffff; it_red[3 * ITEM_CAP + i] = -1;
        it_red[4 * ITEM_CAP + i] = 0;
    }
    if (tid == 0) s_nitems = 0;
    __syncthreads();
    for (int i = tid; i < nsb * SBB; i += TT) {
        const int sbi = i / SBB, col = i % SBB;
        const int SX = sbx0 + sbi / nsy, SY = sby0 + sbi % nsy;
        const int bx = SX * SBB + col;
        if (bx < bx0 || bx >= bx0 + BW) continue;
        const int rlo = max(by0, SY * SBB), rhi = min(by0 + BH - 1, SY * SBB + SBB - 1);
        const int base = (bx - bx0) * BH - by0;
        if (off16(sm.bins, base + rhi + 1) == off16(sm.bins, base + rlo)) continue;       // no ray in this cell column
        int ylo = 0x7fffffff, yhi = -1;
        for (int y = rlo; y <= rhi; ++y) {
            if (off16(sm.bins, base + y + 1) > off16(sm.bins, base + y)) {
                ylo = min(ylo, y);
                yhi = y;
            }
        }
        if (yhi >= 0) {
            atomicMin(&it_red[sbi], bx); atomicMax(&it_red[ITEM_CAP + sbi], bx);
            atomicMin(&it_red[2 * ITEM_CAP + sbi], ylo); atomicMax(&it_red[3 * ITEM_CAP + sbi], yhi);
            atomicAdd(&it_red[4 * ITEM_CAP + sbi], (int)(off16(sm.bins, base + rhi + 1) - off16(sm.bins, base + rlo)));
        }
    }
    __syncthreads();
    {
        const float slop = 1e-6f * (fmaxf(fabsf(q.shift_x), fabsf(q.shift_y)) + (float)max(q.G0, q.G1) * q.res) + 1e-4f * q.res;
        const float inf = __int_as_float(0x7f800000);
        for (int i = tid; i < nsb; i += TT) {
            const int bxl = it_red[i], bxh = it_red[ITEM_CAP + i], byl = it_red[2 * ITEM_CAP + i], byh = it_red[3 * ITEM_CAP + i];
            if (bxh < 0) continue;
            // heavy superblocks first: the warps' last chunks are then cheap ones (the CTA ends at its slowest warp)
            const int mine = it_red[4 * ITEM_CAP + i];
            int rank = 0;
            for (int j = 0; j < nsb; ++j) {
                const int cj = it_red[4 * ITEM_CAP + j];
                rank += (cj > mine || (cj == mine && j < i && cj > 0)) ? 1 : 0;
            }
            atomicAdd(&s_nitems, 1);
            const int SX = sbx0 + i / nsy, SY = sby0 + i % nsy;
            const uint32_t sb = (uint32_t)SX * (uint32_t)q.nSBy + (uint32_t)SY;
            Item it;
            it.list_off = __ldg(q.sb_off + sb);
            it.list_len = __ldg(q.sb_off + sb + 1) - it.list_off;
            if (it.list_len > (1u << REL_BITS)) s_bail = 1;          // queue entries keep REL_BITS bits of list position
            const int cxl = bxl << sh, cxh = ((bxh + 1) << sh) - 1, cyl = byl << sh, cyh = ((byh + 1) << sh) - 1;          // cells
            // a source whose cell is >= c lies above shift + (c - 0.5) res (minus slop); clamped border cells hold everything beyond
            it.rlox = fmaxf(g_lox, cxl <= 0 ? -inf : q.shift_x + ((float)cxl - 0.52f) * q.res - slop);
            it.rhix = fminf(g_hix, cxh >= q.G0 - 1 ? inf : q.shift_x + ((float)cxh + 0.52f) * q.res + slop);
            it.rloy = fmaxf(g_loy, cyl <= 0 ? -inf : q.shift_y + ((float)cyl - 0.52f) * q.res - slop);
            it.rhiy = fminf(g_hiy, cyh >= min(q.G0, q.G1) - 1 ? inf : q.shift_y + ((float)cyh + 0.52f) * q.res + slop);
            it.bx = (uint32_t)bxl | ((uint32_t)bxh << 16);
            it.by = (uint32_t)byl | ((uint32_t)byh << 16);
            sm.items[rank] = it;
            s_item_rays[rank] = (unsigned short)min(mine, 65535);
        }
    }
    __syncthreads();
    {
        // chunks = windows of 32 list entries ALIGNED in sb_ids (window w = entries [32 w, 32 w + 32): the lists' ends share windows
        // with their neighbours); windows before each item (warp 0: 4 items per lane), then the chunk -> item table
        const int ni = s_nitems;
        if (warp == 0) {
            uint32_t c[4], tot = 0;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int i = lane * 4 + j;
                c[j] = i < ni ? ((sm.items[i].list_off & (CHUNK - 1)) + sm.items[i].list_len + CHUNK - 1) / CHUNK : 0u;
                tot += c[j];
            }
            uint32_t inc = tot;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t v = __shfl_up_sync(0xffffffffu, inc, o);
                if (lane >= o) inc += v;
            }
            uint32_t run = inc - tot;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int i = lane * 4 + j;
                if (i <= ni) sm.cum[i] = run;
                run += c[j];
            }
            if (lane == 31) s_nchunks = (int)inc;
        }
        __syncthreads();
        if (s_nchunks > CHUNK_CAP || s_bail) {
            if (tid == 0) q.fb_list[atomicAdd(q.fb_count, 1)] = work_id;
            return;
        }
        unsigned char* all_item = reinterpret_cast<unsigned char*>(sm.q1);          // [CHUNK_CAP], the queues are idle here
        unsigned char* all_key = all_item + CHUNK_CAP;                              // [CHUNK_CAP] cost bucket, 0xFF = culled
        for (int i = tid; i < ni; i += TT)
            for (uint32_t c = sm.cum[i]; c < sm.cum[i + 1]; ++c) all_item[c] = (unsigned char)i;
        if (tid < 16) s_bkt[tid >> 3][tid & 7] = 0;
        __syncthreads();
        // window cull: a window none of whose triangles stage 1 could keep for the item's ray rectangle is dropped here, 32
        // entries at a time (one thread per window).  The survivors go into the chunk table the warps pull from, the expensive ones
        // (many rays of the item under the window) first: the warps' last chunks are then cheap and they finish together
        const int total = s_nchunks;
        for (int g = tid; g < total; g += TT) {
            const int item = all_item[g];
            const Item& it = sm.items[item];
            const uint4* rp = reinterpret_cast<const uint4*>(q.sb_chunk + (it.list_off >> 5) + (g - (int)sm.cum[item]));
            union { uint4 u[4]; ChunkRec c; } rec;
            uint4 c0, c1, c2, c3;
            ldg_rec32(rp, c0, c1);
            ldg_rec32(rp + 2, c2, c3);
            rec.u[0] = c0; rec.u[1] = c1; rec.u[2] = c2; rec.u[3] = c3;
            float ov;
            int key;
            if (chunk_cull(rec.c, s_env, it.rlox, it.rhix, it.rloy, it.rhiy, ov)) key = 0xFF;
            else key = 7 - min(7, (int)(sqrtf((float)s_item_rays[item] * ov) * 0.25f));      // bucket 0: >= 784 rays under the window
            all_key[g] = (unsigned char)key;
            if (key != 0xFF) atomicAdd(&s_bkt[0][key], 1);
        }
        __syncthreads();
        if (tid == 0) {
            int run = 0;
            for (int b = 0; b < 8; ++b) {
                s_bkt[1][b] = run;
                run += s_bkt[0][b];
            }
            if (DBGK) {
                atomicAdd(q.dbg + 20, (unsigned long long)total);
                atomicAdd(q.dbg + 21, (unsigned long long)run);
            }
            s_nchunks = run;
        }
        __syncthreads();
        for (int g = tid; g < total; g += TT) {
            const int key = all_key[g];
            if (key != 0xFF) {
                const int item = all_item[g];
                const int at = atomicAdd(&s_bkt[1][key], 1);
                sm.chunk_item[at] = (unsigned char)item;
                sm.chunk_win[at] = (unsigned short)(g - (int)sm.cum[item]);
            }
        }
    }
    __syncthreads();

    // ---- phase 3: warps pull (superblock, 32 list entries); stage 1 -> q1 -> stage 2 -> q2 -> stage 3L -> q4 -> stage 3b.
    // One dispatcher loop per warp; every stage's code exists once (the kernel must stay inside the instruction cache).
    const EnvC& e = s_env;            // read from shared memory where used (stages 1 and 2), not held in registers
    const int nchunks = s_nchunks;
    uint2* q1 = sm.q1 + warp * QCAP;
    uint4* q2 = sm.q2 + warp * QCAP;
    uint32_t* q4 = sm.q4 + warp * QCAP3;
    int32_t* q1t = sm.q1t + warp * QCAP;
    int32_t* q2t = sm.q2t + warp * QCAP;
    int32_t* q4t = sm.q4t + warp * QCAP3;
    uint32_t h1 = 0, t1 = 0, h2 = 0, t2 = 0, h4 = 0, t4 = 0;          // warp-uniform
    const uint32_t lt_mask = (1u << lane) - 1u;
    const uint32_t FULLM = 0xffffffffu;
    enum { A1 = 0, A2_START, A2_EMIT, A3L_START, A3L_RUN, A3B };
#define DBG(i, v) do { if (DBGK) { const unsigned long long v_ = (unsigned long long)(v); if (lane == 0) atomicAdd(q.dbg + (i), v_); } } while (0)

    // stage-1 pipeline: the ids of chunk k+1 are in flight while chunk k is tested (its stage-1 records are loaded on the spot:
    // holding them across the dispatcher loop costs eight registers the 64-register instantiation does not have)
    int32_t idA = -1, idB = -1;
    uint32_t entA = 0, entB = 0;           // superblock-list entry of the lane's triangle
    int itemA = -1, itemB = -1;            // -1: no chunk
    auto pull = [&](int32_t& id, uint32_t& ent, int& item) {
        int g = 0;
        if (lane == 0) g = atomicAdd(&s_next, 1);
        g = __shfl_sync(FULLM, g, 0);
        item = -1;
        id = -1;
        if (g < nchunks) {
            item = sm.chunk_item[g];
            const Item& it = sm.items[item];
            ent = (((it.list_off >> 5) + (uint32_t)sm.chunk_win[g]) << 5) + lane;
            if (ent >= it.list_off && ent - it.list_off < it.list_len) id = __ldg(q.sb_ids + ent);
        }
    };
    pull(idA, entA, itemA);
    pull(idB, entB, itemB);
    bool more = true, in2 = false, in3 = false;
    // stage-2 emission state (per lane)
    uint32_t e_ent = 0, e_T12 = 0, e_T3s = 0, e_cur = 0, e_end = 0;
    int32_t e_tri = 0;
    int e_col = 1, e_cx1 = 0, e_rlo = 0, e_rhi = 0;
    // stage-3L state (per lane): task + bit i set = ray start + i lies inside the prism
    uint32_t a_ent = 0, a_start = 0, a_mask = 0;
    int32_t a_tri = 0;
    const int task_rays = q.task_rays;

    long long c_start = 0, c_dry = 0;
    if (DBGK) c_start = clock64();
    while (true) {
        const uint32_t n1 = t1 - h1, n2 = t2 - h2, n4 = t4 - h4;
        int action;
        uint32_t cnt = 32u;
        if (n4 >= 32u) action = A3B;
        else if (in3) action = A3L_RUN;
        else if (n2 >= 32u) action = A3L_START;
        else if (in2) action = A2_EMIT;
        else if (n1 >= 32u) action = A2_START;
        else if (more) action = A1;
        else if (n1) { action = A2_START; cnt = n1; }
        else if (n2) { action = A3L_START; cnt = n2; }
        else if (n4) { action = A3B; cnt = n4; }
        else break;
        __syncwarp();
        DBG(12, 1);
        switch (action) {
        case A1: {
            do {
                if (itemA < 0) {
                    more = false;
                    if (DBGK) c_dry = clock64();
                    break;
                }
                const int32_t id = idA;
                const uint32_t ent = entA;
                const int item = itemA;
                uint4 r0 = make_uint4(0, 0, 0, 0), r1 = r0;
                if (id >= 0) {
                    ldg_rec32(q.s1 + id, r0, r1);
                }
                idA = idB; itemA = itemB; entA = entB;
                pull(idB, entB, itemB);
                const Item& it = sm.items[item];
                bool keep = false;
                float gball = 0.0f;
                if (id >= 0) keep = stage1(r0, r1, e, it.rlox, it.rhix, it.rloy, it.rhiy, gball);
                const uint32_t m = __ballot_sync(FULLM, keep);
                if (keep) {
                    const uint32_t at = (t1 + __popc(m & lt_mask)) & (QCAP - 1);
                    q1[at] = make_uint2(ent, ((__float_as_uint(gball) + 0x7fu) & ~0x7fu) | (uint32_t)item);
                    q1t[at] = id;
                    // stage 2 will want the triangle's record: start bringing it into L2 now
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(q.recs + id));
                }
                t1 += __popc(m);
                DBG(0, 1); DBG(1, __popc(m));
                const uint32_t mi = __ballot_sync(FULLM, keep && gball == __int_as_float(0x7f800000));
                if (mi) {
                    if (lane == 0) atomicAdd(&s_ill, __popc(mi));
                    if (*reinterpret_cast<volatile int*>(&s_ill) > ILL_CAP) {       // give the tile up: every warp drops what it holds
                        more = false; in2 = false; in3 = false;
                        h1 = t1; h2 = t2; h4 = t4;
                        itemA = -1;
                        break;
                    }
                }
            } while (t1 - h1 < 32u);
            break;
        }
        case A2_START: {
            // up to 32 surviving triangles, one per lane -> box -> block columns
            e_col = 1; e_cx1 = 0; e_cur = 0; e_end = 0;                   // empty column range
            if ((uint32_t)lane < cnt) {
                const uint2 en = q1[(h1 + lane) & (QCAP - 1)];
                e_ent = en.x;
                const int32_t tri = q1t[(h1 + lane) & (QCAP - 1)];
                e_tri = tri;
                const float gball = __uint_as_float(en.y & ~0x7fu);
                const Item& it = sm.items[en.y & 0x7fu];
                e_ent = ((en.y & 0x7fu) << REL_BITS) | (e_ent - it.list_off);
                const uint4 r0 = __ldg(reinterpret_cast<const uint4*>(q.recs + tri));
                const uint2 r1 = __ldg(reinterpret_cast<const uint2*>(q.recs + tri) + 2);
                float x0, x1, y0, y1;
                bool full;
                stage2(tri_f(r0, r1), r1, e, d16, gball, x0, x1, y0, y1, full, e_T12, e_T3s);
                int bxl = (int)(it.bx & 0xffffu), bxh = (int)(it.bx >> 16), byl = (int)(it.by & 0xffffu), byh = (int)(it.by >> 16);
                if (!full) {
                    bxl = max(bxl, cell_coord_f(x0, q.shift_x, q.res, q.inv_res, q.G0 - 1, q.sem) >> sh);
                    bxh = min(bxh, cell_coord_f(x1, q.shift_x, q.res, q.inv_res, q.G0 - 1, q.sem) >> sh);
                    byl = max(byl, min(cell_coord_f(y0, q.shift_y, q.res, q.inv_res, q.G0 - 1, q.sem), q.G1 - 1) >> sh);
                    byh = min(byh, min(cell_coord_f(y1, q.shift_y, q.res, q.inv_res, q.G0 - 1, q.sem), q.G1 - 1) >> sh);
                }
                if (bxl <= bxh && byl <= byh) {
                    e_col = bxl; e_cx1 = bxh;
                    e_rlo = byl - by0; e_rhi = byh - by0 + 1;
                }
            }
            h1 += cnt;
            in2 = true;
            DBG(2, cnt); DBG(13, __popc(__ballot_sync(FULLM, e_T12 == 0x7F807F80u && (uint32_t)lane < cnt)));
        }
        // fall through: nothing of higher priority became ready
        case A2_EMIT: {
            // tasks of <= TASK_RAYS consecutive sorted rays; runs until q2 holds a batch or the lanes are done
            while (true) {
                while (e_cur >= e_end && e_col <= e_cx1) {
                    const int b = (e_col - bx0) * BH;
                    e_cur = off16(sm.bins, b + e_rlo);
                    e_end = off16(sm.bins, b + e_rhi);
                    ++e_col;
                }
                const bool have = e_cur < e_end;
                const uint32_t m = __ballot_sync(FULLM, have);
                if (!m) {
                    in2 = false;
                    break;
                }
                if (have) {
                    const uint32_t c = min(e_end - e_cur, (uint32_t)task_rays);
                    const uint32_t at = (t2 + __popc(m & lt_mask)) & (QCAP - 1);
                    q2[at] = make_uint4(e_ent, e_cur | (c << 16), e_T12, e_T3s);
                    q2t[at] = e_tri;
                    e_cur += c;
                }
                t2 += __popc(m);
                DBG(3, __popc(m)); DBG(10, 1);
                if (t2 - h2 >= 32u) break;
            }
            break;
        }
        case A3L_START: {
            // One task per lane: every ray of the task against the three half-planes of the triangle's prism, N' = g . (c x d'),
            // M' = g . (d' x b) with g = s - a and d' = sgn(det) d -- exact linear forms evaluated in fp32 (FFMA2: N' and M' in one
            // issue slot) -> bit mask of the rays inside.  No warp-level work inside the loop.
            a_mask = 0u;
            if ((uint32_t)lane < cnt) {
                const uint4 tk = q2[(h2 + lane) & (QCAP - 1)];
                a_ent = tk.x;
                a_start = tk.y & 0xffffu;
                const int c = (int)(tk.y >> 16);
                const int32_t tri = q2t[(h2 + lane) & (QCAP - 1)];
                a_tri = tri;
                const uint4 r0 = __ldg(reinterpret_cast<const uint4*>(q.recs + tri));
                const uint32_t r1 = __ldg(reinterpret_cast<const uint32_t*>(q.recs + tri) + 4);
                const float sg = (tk.w & 0x8000u) ? -1.0f : 1.0f;
                const float dx = sg * e.dx, dy = sg * e.dy, dz = sg * e.dz;
                const float ax = hf(r0.x & 0xffff), ay = hf(r0.x >> 16), az = hf(r0.y & 0xffff);
                const float bx = hf(r0.y >> 16), by = hf(r0.z & 0xffff), bz = hf(r0.z >> 16);
                const float cx = hf(r0.w & 0xffff), cy = hf(r0.w >> 16), cz = hf(r1 & 0xffff);
                const float w1x = cy * dz - cz * dy, w1y = cz * dx - cx * dz, w1z = cx * dy - cy * dx;          // c x d'
                const float w2x = dy * bz - dz * by, w2y = dz * bx - dx * bz, w2z = dx * by - dy * bx;          // d' x b
                const float T1 = -__uint_as_float(tk.z << 16), T2 = -__uint_as_float(tk.z & 0xffff0000u);
                const float T3 = __uint_as_float((tk.w & 0x7fffu) << 16);
                for (int i = 0; i < c; ++i) {
                    const uint2 ray = sm.rays[a_start + i];
                    const float gx = hf(ray.x & 0xffff) - ax, gy = hf(ray.x >> 16) - ay, gz = hf(ray.y & 0xffff) - az;
                    float Nn = 0.f, Mn = 0.f;
                    ffma2(Nn, Mn, w1x, w2x, gx);
                    ffma2(Nn, Mn, w1y, w2y, gy);
                    ffma2(Nn, Mn, w1z, w2z, gz);
                    const bool in = (Nn >= T1) && (Mn >= T2) && (Nn + Mn <= T3);
                    a_mask |= (in ? 1u : 0u) << i;
                }
            }
            h2 += cnt;
            in3 = __any_sync(FULLM, a_mask != 0u);
            if (DBGK) {
                const int c = (uint32_t)lane < cnt ? (int)(q2[(h2 - cnt + lane) & (QCAP - 1)].y >> 16) : 0;
                const int cm = __reduce_max_sync(FULLM, c), cs = __reduce_add_sync(FULLM, c), ib = __reduce_add_sync(FULLM, __popc(a_mask));
                DBG(4, cm); DBG(5, cs); DBG(6, ib);
            }
            if (!in3) break;
        }
        // fall through
        case A3L_RUN: {
            // expand the masks into (ray, entry) pairs: a warp scan gives every lane the queue position of its first pair, so the
            // lanes write their pairs without any warp-level work inside the loop; runs until q4 is full or the masks are empty
            while (true) {
                const uint32_t c = (uint32_t)__popc(a_mask);
                uint32_t inc = c;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const uint32_t v = __shfl_up_sync(FULLM, inc, o);
                    if (lane >= o) inc += v;
                }
                const uint32_t total = __shfl_sync(FULLM, inc, 31);
                if (!total) {
                    in3 = false;
                    break;
                }
                const uint32_t room = (uint32_t)QCAP3 - (t4 - h4);        // > 96: this stage only runs while q4 holds < 32 pairs
                uint32_t at = inc - c;                                    // queue position of this lane's next pair, relative to t4
                const uint32_t code = a_ent << 11;
                while (a_mask != 0u && at < room) {
                    const uint32_t bit = (uint32_t)__ffs((int)a_mask) - 1u;
                    a_mask &= a_mask - 1u;
                    q4[(t4 + at) & (QCAP3 - 1)] = (a_start + bit) | code;
                    q4t[(t4 + at) & (QCAP3 - 1)] = a_tri;
                    ++at;
                }
                t4 += min(total, room);
                DBG(11, 1);
                if (total <= room) {            // every mask is empty now
                    in3 = false;
                    break;
                }
                if (t4 - h4 >= 32u) break;
            }
            break;
        }
        case A3B: {
            // literal evaluation + slot lookup of up to 32 queued (ray, triangle) pairs, one per lane
            do {
                if ((uint32_t)lane < cnt) {
                    const uint32_t pc = q4[(h4 + lane) & (QCAP3 - 1)];
                    const uint2 ray = sm.rays[pc & 0x7ffu];
                    const uint32_t ent = sm.items[pc >> (11 + REL_BITS)].list_off + ((pc >> 11) & ((1u << REL_BITS) - 1u));
                    const int32_t tri = q4t[(h4 + lane) & (QCAP3 - 1)];
                    const H3 s = {h_from_bits(ray.x & 0xffff), h_from_bits(ray.x >> 16), h_from_bits(ray.y & 0xffff)};
                    const uint32_t meta = ray.y >> 16, p = meta & 0x7ffu, cym = meta >> 11;
                    // slot of the triangle in the K-list of the ray's own cell (0xFF: not in it): ONE look-up in the superblock entry's
                    // per-cell table, issued before the literal test runs so that its latency hides behind the arithmetic
                    const int cx = cell_coord(s.x, q.shift_x, q.res, q.inv_res, q.G0 - 1, q.sem);
                    const uint32_t slot = __ldg(q.sb_slot9 + (size_t)ent * (SBC * SBC) + (uint32_t)((cx % SBC) * SBC) + cym);
                    H3 a, b, c, nn;
                    unpack_rec(q.recs + tri, a, b, c, nn);
                    const __half k = pair_test(s, d16, a, b, c, nn);
                    const uint32_t key0 = make_key(h_bits(k), 0u), ord = key0 >> 16;
                    // a hit at exactly 11.0 equals the all-miss result (slot 0); a hit farther than a confirmed one cannot win
                    if (DBGK && h_bits(k) != RVB_H_MISS) atomicAdd(q.dbg + 8, 1ull);
                    if (h_bits(k) != RVB_H_MISS && slot != 0xffu && (ord > ORD_MISS || ord <= (sm.res[p] >> 16))) {
                        if (DBGK) atomicAdd(q.dbg + 9, 1ull);
                        const uint32_t key = key0 | (slot << 1);          // the triangle is in the ray's own cell list
                        if (ord > ORD_MISS) atomicOr(&sm.far[p >> 5], 1u << (p & 31));      // k > 11: see epilogue
                        else atomicMin(&sm.res[p], key);
                    }
                }
                h4 += cnt;
                DBG(7, 1);
            } while (cnt == 32u && t4 - h4 >= 32u);
            break;
        }
        }
    }
    if (DBGK) {
        // per warp: cycles until the chunk supply ran dry, cycles of the drain, cycles waited at the barrier below
        const long long c_done = clock64();
        __syncthreads();
        const long long c_all = clock64();
        if (lane == 0) {
            atomicAdd(q.dbg + 16, (unsigned long long)(c_dry - c_start));
            atomicAdd(q.dbg + 17, (unsigned long long)(c_done - c_dry));
            atomicAdd(q.dbg + 18, (unsigned long long)(c_all - c_done));
            atomicAdd(q.dbg + 19, 1ull);
        }
    }
    __syncthreads();
    if (s_ill > ILL_CAP) {          // too many triangles without a bound: the tiled kernel casts this tile (results so far are dropped)
        if (tid == 0) q.fb_list[atomicAdd(q.fb_count, 1)] = work_id;
        return;
    }

    // ---- phase 4
    // pose and trigonometry are re-read here (volatile: no common sub-expression with phase 0) instead of living in twelve
    // registers across phase 3
    {
        const volatile float* vp = q.pos + n * 3;
        const double ex_ = (double)vp[0], ey_ = (double)vp[1], ez_ = (double)vp[2];
        Trig tr2;
        if (q.trig) {
            const volatile float* t6 = q.trig + n * 6;
            tr2 = {t6[0], t6[1], t6[2], t6[3], t6[4], t6[5]};
        } else {
            const volatile float* ve = q.euler + n * 3;
            const float r_ = -ve[0], p_ = -ve[1], y_ = -ve[2];
            tr2 = {sinf(r_), cosf(r_), sinf(p_), cosf(p_), sinf(y_), cosf(y_)};
        }
        epilogue(q, n, p0, np, tr2, ex_, ey_, ez_, dx2, dy2, dz2, sm.res, sm.far, tid, TT);
    }
}

}  // namespace

// The whole of `name`'s value as a number in [lo, hi] (an integer if `integer`) into v; unset leaves v alone.  `range` states
// the accepted values in the error message.
static int read_knob(const char* name, double lo, double hi, bool integer, const char* range, double& v) {
    const char* s = getenv(name);
    if (!s) return RVB_OK;
    char* end = nullptr;
    errno = 0;
    const double x = integer ? (double)strtoll(s, &end, 10) : strtod(s, &end);
    if (*s == '\0' || isspace((unsigned char)*s) || *end != '\0' || errno != 0 || !(x >= lo && x <= hi)) {
        char detail[128];
        snprintf(detail, sizeof(detail), "'%.32s' is not %s", s, range);
        return rvb_set_error(RVB_ERR_INVALID, name, detail);
    }
    v = x;
    return RVB_OK;
}

int read_raycast_knobs(RaycastKnobs& k) {
    double force = -1, cos_steep = COS_STEEP, min_sh = MIN_SH, task_rays = TASK_RAYS, split = -1, dbg = 0;
    int rc_;
    if ((rc_ = read_knob("RVB_SHADOW_FORCE", 0, 1, true, "0 or 1", force))) return rc_;
    if ((rc_ = read_knob("RVB_COS_STEEP", 0, 1, false, "a number in [0, 1]", cos_steep))) return rc_;
    // 2^3 cells, the coarsest bins phase 1 goes up to; bins must divide the superblock side (24 cells)
    if ((rc_ = read_knob("RVB_SHADOW_SH", 0, 3, true, "an integer in 0..3", min_sh))) return rc_;
    if ((rc_ = read_knob("RVB_SHADOW_TASK_RAYS", 1, 32, true, "an integer in 1..32", task_rays))) return rc_;
    if ((rc_ = read_knob("RVB_SHADOW_SPLIT", 0, 9e18, true, "an integer >= 0", split))) return rc_;
    if ((rc_ = read_knob("RVB_SHADOW_DBG", 0, 1, true, "0 or 1", dbg))) return rc_;
    k.force = (int)force;
    k.cos_steep = (float)cos_steep;
    k.min_sh = (int)min_sh;
    k.task_rays = (int)task_rays;
    k.split = (int64_t)split;
    k.dbg = dbg != 0;
    return RVB_OK;
}

// The tiled kernel over the (env, tile) items of a work list on the device; each item is cut into 8 slices, one CTA each.
static int launch_tiled_list(rc::TiledParams q, const int* count, const int32_t* list, int64_t grid, cudaStream_t st) {
    q.work_count = count;
    q.work_list = list;
    q.work_slices = 8;
    return launch_tiled(q, true, grid, st);
}

// The env order of q's N envs into order[N] (hm_classify_kernel's keys, stable radix sort: equal keys keep index order); with
// steep_list, the same launch also puts the steep envs on it.  q needs the poses, the grid and cos_steep.
static int sort_envs(const rc::TiledParams& q, int64_t N, int32_t* order, int* steep_count, int32_t* steep_list, cudaStream_t st) {
    RVB_REQUIRE(N < ((int64_t)1 << 31), "env order: more than 2^31 - 1 envs");
    int zbits = 0;          // bits per axis of the Z-order code: enough for the layer's grid, no more (fewer radix passes)
    while ((((int64_t)max(q.G0, q.G1) - 1) >> ORDER_SH) >> zbits) ++zbits;
    // the class bit and two zbits-bit coordinates in a 32-bit key
    RVB_REQUIRE(zbits <= 15, "env order: grid wider than 2^18 cells");
    const int key_bits = 2 * zbits + 1;
    RvbTemp<uint32_t> keys;           // [2N]  keys, sorted keys
    RvbTemp<int32_t> ids;
    RVB_CUDA(keys.alloc_pool(2 * (size_t)N, st));
    RVB_CUDA(ids.alloc_pool((size_t)N, st));
    hm_classify_kernel<<<(unsigned)ceil_div(N, 256), 256, 0, st>>>(q, N, zbits, keys.p, ids.p, steep_count, steep_list);
    RVB_LAUNCH_CHECK();
    size_t bytes = 0;
    RVB_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, bytes, keys.p, keys.p + N, ids.p, order, (int)N, 0, key_bits, st));
    RvbTemp<unsigned char> tmp;
    RVB_CUDA(tmp.alloc_pool(bytes, st));
    RVB_CUDA(cub::DeviceRadixSort::SortPairs(tmp.p, bytes, keys.p, keys.p + N, ids.p, order, (int)N, 0, key_bits, st));
    return RVB_OK;
}

int build_env_order(const rc::TiledParams& q, int64_t N, float cos_steep, int32_t* order, cudaStream_t st) {
    rc::TiledParams c = q;
    c.cos_steep = cos_steep;
    return sort_envs(c, N, order, nullptr, nullptr, st);
}

int launch_shadow(rc::TiledParams q, int64_t N, const RaycastKnobs& knobs, const int32_t* order, cudaStream_t st) {
    RVB_REQUIRE(q.sb_ids != nullptr && q.sb_slot9 != nullptr && q.sb_chunk != nullptr && q.blk_ids != nullptr && q.s1 != nullptr,
                "heightmap ray-cast (shadow): layer has no block lists");
    RVB_REQUIRE(q.tile_size <= 2048, "heightmap ray-cast (shadow): tile larger than 2048 rays");
    int64_t nblocks = N * q.tiles;
    // the last nsplit envs of the order are cast by two CTAs of half the rays each
    q.split_from = -1;
    {
        int64_t nsplit = N >= 8 * 148 ? 3 * 148 : 0;            // measured at 4096 envs: -2 % (444), -1.2 % (592), -1 % (296)
        if (knobs.split >= 0) nsplit = knobs.split;
        if (q.tiles == 1 && q.P >= 64 && nsplit > 0) {
            if (nsplit > N) nsplit = N;
            q.split_from = N - nsplit;
            q.split_at = q.P / 2;
            nblocks = N + nsplit;
        }
    }
    // scratch: with RVB_SHADOW_DBG=1 the kernel's 24 counters (8 bytes each) first; then [0] steep count, [1] handed-back count,
    // the steep list [nblocks], the hand-back list [nblocks] and, without the caller's, the env order [N]
    const int64_t ndbg = knobs.dbg ? 2 * 24 : 0;          // in ints
    // The scratch is declared BEFORE the join guard: destructors run in reverse order, so st first waits for the side stream's
    // tiled kernel, which reads the steep list and the counters, and only then gives the scratch back to the pool.
    RvbTemp<int> scratch;
    RvbJoinGuard guard(st);
    RVB_CUDA(scratch.alloc_pool((size_t)(ndbg + 2 + 2 * nblocks + (order ? 0 : N)), st));
    RVB_CUDA(cudaMemsetAsync(scratch.p, 0, sizeof(int) * (size_t)(ndbg + 2), st));
    int* const counts = scratch.p + ndbg;
    int32_t* steep_list = counts + 2;
    q.fb_count = counts + 1;
    q.fb_list = counts + 2 + nblocks;
    q.cos_steep = knobs.cos_steep;
    q.min_sh = knobs.min_sh;
    q.task_rays = knobs.task_rays;
    static thread_local int configured_device = -1;
    const int lrc = set_smem_limits(configured_device, {{(const void*)hm_shadow_kernel<false, RT_MAX>, shadow_smem_bytes(RT_MAX)},
                                                        {(const void*)hm_shadow_kernel<true, RT_MAX>, shadow_smem_bytes(RT_MAX)},
                                                        {(const void*)hm_shadow_kernel<false, RT_SMALL>, shadow_smem_bytes(RT_SMALL)},
                                                        {(const void*)hm_shadow_kernel<true, RT_SMALL>, shadow_smem_bytes(RT_SMALL)}});
    if (lrc != RVB_OK) return lrc;
    RvbSide* side = nullptr;
    RVB_CUDA(rvb_side_stream(1, &side));
    if (order) {
        // the caller's order (the fused step builds one for the ray-cast and the rock kernel): this launch only makes the steep
        // list.  The caller's classify launch could make it too, but its count would then need a memset in front of the caller's
        // fork of the rock kernel, on the step's critical path; this launch runs after the fork, while the shadow kernel waits for
        // the rock kernel's CTAs, and costs nothing measurable (profiles/r8_env_plan_check.txt)
        hm_classify_kernel<<<(unsigned)ceil_div(N, 256), 256, 0, st>>>(q, N, 0, nullptr, nullptr, counts, steep_list);
        RVB_LAUNCH_CHECK();
        q.order = order;
    } else {
        int32_t* own = counts + 2 + 2 * nblocks;
        const int orc = sort_envs(q, N, own, counts, steep_list, st);
        if (orc != RVB_OK) return orc;
        q.order = own;
    }
    // steep envs: the tiled kernel on the second stream, concurrently with the shadow kernel
    const int64_t tgrid = nblocks < 148 * 3 ? nblocks : 148 * 3;
    RVB_CUDA(cudaEventRecord(side->fork, st));
    RVB_CUDA(cudaStreamWaitEvent(side->s, side->fork, 0));
    const int rcs = launch_tiled_list(q, counts, steep_list, tgrid, side->s);
    if (rcs != RVB_OK) return rcs;
    RVB_CUDA(cudaEventRecord(side->join, side->s));
    guard.join = side->join;
    const bool dbg = knobs.dbg;
    if (dbg) q.dbg = reinterpret_cast<unsigned long long*>(scratch.p);
    const unsigned grid = (unsigned)nblocks;
    if (q.tile_size <= RT_SMALL) {
        if (dbg) hm_shadow_kernel<true, RT_SMALL><<<grid, TT, shadow_smem_bytes(RT_SMALL), st>>>(q);
        else hm_shadow_kernel<false, RT_SMALL><<<grid, TT, shadow_smem_bytes(RT_SMALL), st>>>(q);
    } else {
        if (dbg) hm_shadow_kernel<true, RT_MAX><<<grid, TT, shadow_smem_bytes(RT_MAX), st>>>(q);
        else hm_shadow_kernel<false, RT_MAX><<<grid, TT, shadow_smem_bytes(RT_MAX), st>>>(q);
    }
    RVB_LAUNCH_CHECK();
    if (dbg) {
        unsigned long long h[24];
        int fb = 0;
        RVB_CUDA(cudaStreamSynchronize(st));
        RVB_CUDA(cudaMemcpy(h, q.dbg, sizeof(h), cudaMemcpyDeviceToHost));
        RVB_CUDA(cudaMemcpy(&fb, q.fb_count, sizeof(int), cudaMemcpyDeviceToHost));
        const double ne = (double)(nblocks - fb);
        fprintf(stderr, "[shadow dbg] tiles %lld, handed back %d; per tile: chunks %.1f, stage-1 keeps %.1f, stage-2 triangles %.1f (no bound: %.2f), "
                        "tasks %.1f (emit iterations %.1f), prism loop iterations %.1f, rays tested %.1f, inside the prism %.1f, "
                        "3b batches %.1f, literal hits %.1f, slot lookups %.1f, dispatches %.1f\n",
                (long long)nblocks, fb, h[0] / ne, h[1] / ne, h[2] / ne, h[13] / ne, h[3] / ne, h[10] / ne, h[4] / ne, h[5] / ne, h[6] / ne,
                h[7] / ne, h[8] / ne, h[9] / ne, h[12] / ne);
        fprintf(stderr, "[shadow dbg] windows of 32 list entries per tile: %.1f, kept by the window cull: %.1f\n", h[20] / ne, h[21] / ne);
        if (h[19])
            fprintf(stderr, "[shadow dbg] phase 3 per warp (cycles): pulling chunks %.0f, draining the queues %.0f, waiting at the final barrier %.0f\n",
                    (double)h[16] / h[19], (double)h[17] / h[19], (double)h[18] / h[19]);
    }
    // (env, tile) items the shadow kernel handed back: the tiled kernel loops over the list (usually empty).
    return launch_tiled_list(q, q.fb_count, q.fb_list, tgrid, st);
}
