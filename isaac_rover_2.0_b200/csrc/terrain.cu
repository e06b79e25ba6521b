// Terrain-layer handle: K-contiguous index copy + pre-resolved triangle records.
#include <memory>
#include <new>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <cub/device/device_select.cuh>

#include "common.cuh"

static thread_local char g_err[512] = "";

int rvb_set_error(int code, const char* what, const char* detail) {
    snprintf(g_err, sizeof(g_err), "rover_b200: %s (%s)", what ? what : "error", detail ? detail : "");
    return code;
}

extern "C" const char* rvb_last_error(void) { return g_err; }

#include <mutex>
cudaError_t rvb_scratch_alloc(void** p, size_t bytes, cudaStream_t st) {
    static std::mutex mu;
    static cudaMemPool_t pools[64] = {};
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev < 0 || dev >= 64) return cudaMallocAsync(p, bytes, st);
    cudaMemPool_t pool;
    {
        std::lock_guard<std::mutex> lk(mu);
        if (!pools[dev]) {
            cudaMemPoolProps props = {};
            props.allocType = cudaMemAllocationTypePinned;
            props.handleTypes = cudaMemHandleTypeNone;
            props.location.type = cudaMemLocationTypeDevice;
            props.location.id = dev;
            if ((e = cudaMemPoolCreate(&pools[dev], &props)) != cudaSuccess) return e;
            uint64_t keep = UINT64_MAX;
            if ((e = cudaMemPoolSetAttribute(pools[dev], cudaMemPoolAttrReleaseThreshold, &keep)) != cudaSuccess) return e;
        }
        pool = pools[dev];
    }
    return cudaMallocFromPoolAsync(p, bytes, pool, st);
}
cudaError_t rvb_side_stream(int slot, RvbSide** out) {
    static thread_local RvbSide table[64][2] = {};
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev < 0 || dev >= 64 || slot < 0 || slot > 1) return cudaErrorInvalidValue;
    RvbSide& sd = table[dev][slot];
    if (!sd.s) {
        cudaStream_t s = nullptr;
        cudaEvent_t f = nullptr, j = nullptr;
        if ((e = cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking)) != cudaSuccess) return e;
        if ((e = cudaEventCreateWithFlags(&f, cudaEventDisableTiming)) != cudaSuccess) { cudaStreamDestroy(s); return e; }
        if ((e = cudaEventCreateWithFlags(&j, cudaEventDisableTiming)) != cudaSuccess) { cudaStreamDestroy(s); cudaEventDestroy(f); return e; }
        sd.s = s; sd.fork = f; sd.join = j;
    }
    *out = &sd;
    return cudaSuccess;
}
extern "C" int rvb_abi_version(void) { return RVB_ABI_VERSION; }

// [G0,G1,K] strided view -> contiguous.  One thread per output element; consecutive threads walk K, so
// the store is coalesced; the load is coalesced along whichever source stride is 1 only for K-major
// inputs -- this runs once per terrain, bandwidth is irrelevant.
__global__ void repack_index_kernel(const int32_t* __restrict__ src, int64_t G0, int64_t G1, int64_t K, int64_t Ks,
                                    int64_t s0, int64_t s1, int64_t sk, int32_t T, int32_t* __restrict__ dst, int* bad) {
    int64_t total = G0 * G1 * Ks;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        int64_t k = i % Ks, c = i / Ks;
        int64_t g1 = c % G1, g0 = c / G1;
        int32_t v = 0;                                  // pad slot: a valid triangle id that is never evaluated
        if (k < K) {
            v = src[g0 * s0 + g1 * s1 + k * sk];
            if (v < 0 || v >= T) {
                atomicExch(bad, 1);
                v = 0;
            }
        }
        dst[i] = v;
    }
}

// a = v[t2], b = v[t1]-a, c = v[t0]-a, n = b x c with fp16 roundings (ray_casting.py:34-40).
__global__ void build_records_kernel(const int32_t* __restrict__ tri, int64_t T, const __half* __restrict__ vert,
                                     int64_t V, TriRec* __restrict__ recs, S1Rec* __restrict__ s1recs, int* bad) {
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= T) return;
    int32_t i0 = tri[i * 3 + 0], i1 = tri[i * 3 + 1], i2 = tri[i * 3 + 2];
    if (i0 < 0 || i0 >= V || i1 < 0 || i1 >= V || i2 < 0 || i2 >= V) {
        atomicExch(bad, 2);
        i0 = i1 = i2 = 0;
    }
    H3 v0 = {vert[i0 * 3], vert[i0 * 3 + 1], vert[i0 * 3 + 2]};
    H3 v1 = {vert[i1 * 3], vert[i1 * 3 + 1], vert[i1 * 3 + 2]};
    H3 a = {vert[i2 * 3], vert[i2 * 3 + 1], vert[i2 * 3 + 2]};
    H3 b = h3_sub(v1, a), c = h3_sub(v0, a);
    H3 n = h3_cross(b, c);
    TriRec r;
    r.a[0] = a.x; r.a[1] = a.y; r.a[2] = a.z;
    r.b[0] = b.x; r.b[1] = b.y; r.b[2] = b.z;
    r.c[0] = c.x; r.c[1] = c.y; r.c[2] = c.z;
    r.n[0] = n.x; r.n[1] = n.y; r.n[2] = n.z;
    r.pad[0] = r.pad[1] = r.pad[2] = r.pad[3] = __ushort_as_half(0);
    recs[i] = r;
    // stage-1 record of the shadow kernel: the same fp32 operations, in the same order, as its per-triangle prologue
    const float ax = __half2float(a.x), ay = __half2float(a.y), az = __half2float(a.z);
    const float bx = __half2float(b.x), by = __half2float(b.y), bz = __half2float(b.z);
    const float cx = __half2float(c.x), cy = __half2float(c.y), cz = __half2float(c.z);
    const float third = 0.33333334f;
    const float mx = __fmul_rn(__fadd_rn(bx, cx), third), my = __fmul_rn(__fadd_rn(by, cy), third), mz = __fmul_rn(__fadd_rn(bz, cz), third);
    const float ex = __fsub_rn(bx, cx), ey = __fsub_rn(by, cy), ez = __fsub_rn(bz, cz);
    const float b2 = fmaf(bx, bx, fmaf(by, by, __fmul_rn(bz, bz))), c2 = fmaf(cx, cx, fmaf(cy, cy, __fmul_rn(cz, cz))),
                e2 = fmaf(ex, ex, fmaf(ey, ey, __fmul_rn(ez, ez)));
    const float amax = fmaxf(fmaxf(fabsf(ax), fabsf(ay)), fabsf(az));
    const float cb = fmaxf(fmaxf(fmaxf(fabsf(bx), fabsf(by)), fabsf(bz)), fmaxf(fmaxf(fabsf(cx), fabsf(cy)), fabsf(cz)));
    S1Rec s;
    s.qx = __fadd_rn(ax, mx); s.qy = __fadd_rn(ay, my); s.qz = __fadd_rn(az, mz);
    s.r = __fadd_rn(__fmul_rn(__fmul_rn(0.6666667f, sqrtf(fmaxf(fmaxf(b2, c2), e2))), 1.00001f), __fmul_rn(1e-6f, amax));
    s.nx = __fsub_rn(__fmul_rn(by, cz), __fmul_rn(bz, cy));
    s.ny = __fsub_rn(__fmul_rn(bz, cx), __fmul_rn(bx, cz));
    s.nz = __fsub_rn(__fmul_rn(bx, cy), __fmul_rn(by, cx));
    // cb, amax are fp16 values already (|difference of fp16| can need one more bit: round up)
    s.cb_amax = (uint32_t)__half_as_ushort(__float2half_ru(cb)) | ((uint32_t)__half_as_ushort(__float2half_ru(amax)) << 16);
    s1recs[i] = s;
    // triangles whose fp16 determinant is rounding noise even for a vertical ray (raycast_shadow.cu stage 1: adet <= 4 e_det):
    // the shadow kernel has no bound for them.  Counted once per layer: a mesh finer than the fp16 grid of its coordinates
    // has many, and the heightmap ray-cast then runs the tiled kernel, whose cost does not depend on them.
    const float e_det = 0.00390625f * 6.1f * cb * cb + 1.9073486328125e-06f;
    // (a triangle whose fp16 normal is exactly zero is not counted: it can never be hit -- det = n . d = 0 makes the reference's
    // quotients inf / NaN, which fail its test -- and is left out of the superblock lists altogether, see sb_keys_kernel)
    const bool dead = ((h_bits(n.x) | h_bits(n.y) | h_bits(n.z)) & 0x7fffu) == 0u;
    const bool ill = !dead && !(fabsf(s.nz) > 4.0f * e_det);
    const unsigned m = __ballot_sync(__activemask(), ill);
    if (m && (threadIdx.x & 31) == (__ffs(__activemask()) - 1)) atomicAdd(bad + 1, __popc(m));
}

// ------------------------------------------------------------------------------------------------
// Block lists: one CTA per RVB_BLK x RVB_BLK block.  Keys (id << 16 | sub-cell << 8 | slot) of the block's cells are
// sorted in shared memory; runs of equal id become one entry.  Run twice: count, then (after a scan) write.
// ------------------------------------------------------------------------------------------------
constexpr int BLK_THREADS = 256;
constexpr int BLK_MAXKEYS = 4096;      // >= RVB_BLK^2 * 255

__global__ void __launch_bounds__(BLK_THREADS)
build_blocks_kernel(const int32_t* __restrict__ index, int G0, int G1, int K, int Ks, int nBy, const uint32_t* __restrict__ off,
                    uint32_t* __restrict__ counts, int32_t* __restrict__ ids, uint4* __restrict__ slots) {
    __shared__ unsigned long long keys[BLK_MAXKEYS];
    __shared__ uint32_t s_warp[BLK_THREADS / 32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int I = blockIdx.x / nBy, J = blockIdx.x % nBy;
    const int nk = RVB_BLK * RVB_BLK * K;
    int n2 = 64;
    while (n2 < nk) n2 <<= 1;
    for (int t = tid; t < n2; t += BLK_THREADS) {
        unsigned long long key = ~0ull;
        if (t < nk) {
            const int sub = t / K, slot = t % K;
            const int ci = I * RVB_BLK + sub / RVB_BLK, cj = J * RVB_BLK + sub % RVB_BLK;
            if (ci < G0 && cj < G1)
                key = ((unsigned long long)(uint32_t)index[((int64_t)ci * G1 + cj) * Ks + slot] << 16) | (unsigned)(sub << 8) | (unsigned)slot;
        }
        keys[t] = key;
    }
    __syncthreads();
    for (int k = 2; k <= n2; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = tid; i < n2; i += BLK_THREADS) {
                const int ixj = i ^ j;
                if (ixj > i) {
                    const unsigned long long a = keys[i], b = keys[ixj];
                    if ((a > b) == ((i & k) == 0)) {
                        keys[i] = b;
                        keys[ixj] = a;
                    }
                }
            }
            __syncthreads();
        }
    }
    // entry number of key i = (number of id changes in [0, i]) - 1; thread t owns the contiguous keys [t*per, (t+1)*per)
    const int per = n2 / BLK_THREADS > 0 ? n2 / BLK_THREADS : 1;
    const int lo = tid * per, hi = min(lo + per, n2);
    uint32_t mine = 0;
    for (int i = lo; i < hi && lo < n2; ++i) {
        const unsigned long long k = keys[i];
        if (k != ~0ull && (i == 0 || (keys[i - 1] >> 16) != (k >> 16))) ++mine;
    }
    uint32_t inc = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t v = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += v;
    }
    if (lane == 31) s_warp[warp] = inc;
    __syncthreads();
    uint32_t base = 0, total = 0;
    for (int w = 0; w < BLK_THREADS / 32; ++w) {
        if (w < warp) base += s_warp[w];
        total += s_warp[w];
    }
    if (!ids) {
        if (tid == 0) counts[blockIdx.x] = (total + 1u) & ~1u;      // even: lanes fetch id pairs with 8-byte loads
        return;
    }
    int32_t* out_id = ids + off[blockIdx.x];
    uint4* out_sl = slots + off[blockIdx.x];
    if (tid == 0 && (total & 1u)) {
        // pad entry of an odd list: the largest id again (keeps the list sorted and the id valid; its slots stay 0xFF)
        const int nci = min(RVB_BLK, G0 - I * RVB_BLK), ncj = min(RVB_BLK, G1 - J * RVB_BLK);
        out_id[total] = (int32_t)(keys[nci * ncj * K - 1] >> 16);
    }
    uint32_t e = base + inc - mine;          // entries started before this thread's first key
    for (int i = lo; i < hi && lo < n2; ++i) {
        const unsigned long long k = keys[i];
        if (k == ~0ull) break;
        const bool first = (i == 0 || (keys[i - 1] >> 16) != (k >> 16));
        if (first) {
            ++e;
            out_id[e - 1] = (int32_t)(k >> 16);
        }
        // e - 1 is this key's entry (a run that started in an earlier thread's range keeps that thread's number).
        // A cell list that repeats a triangle keeps the LOWEST slot (torch.min returns the first index on ties).
        if (i == 0 || (keys[i - 1] >> 8) != (k >> 8))
            reinterpret_cast<unsigned char*>(out_sl + (e - 1))[(k >> 8) & 0xff] = (unsigned char)(k & 0xff);
    }
}

// ------------------------------------------------------------------------------------------------
// Superblock lists: keys (superblock << 32 | id) of every block-list entry, radix-sorted and made unique.
// ------------------------------------------------------------------------------------------------
// Triangles whose fp16 normal n = b x c is exactly zero (collapsed vertices: a mesh finer than the fp16 grid of its coordinates has
// millions) get the all-ones key: they sort behind every superblock and are cut off.  No ray can hit them (det = n . d = 0 ->
// the reference's n, m are inf / NaN and fail ray_casting.py:59), so the kernel that ENUMERATES triangles need not see them; the
// block lists and the index keep them (their slots exist, and the far-hit walk evaluates every slot literally).
__global__ void sb_keys_kernel(const uint32_t* __restrict__ blk_off, const int32_t* __restrict__ blk_ids, const TriRec* __restrict__ recs,
                               int nBy, int nSBy, unsigned long long* __restrict__ keys) {
    const int I = blockIdx.x / nBy, J = blockIdx.x % nBy;
    const unsigned long long sb = (unsigned long long)((I / RVB_SB) * nSBy + (J / RVB_SB)) << 32;
    const uint32_t o0 = blk_off[blockIdx.x], o1 = blk_off[blockIdx.x + 1];
    for (uint32_t e = o0 + threadIdx.x; e < o1; e += blockDim.x) {
        const int32_t id = blk_ids[e];
        const TriRec& r = recs[id];
        const bool dead = ((h_bits(r.n[0]) | h_bits(r.n[1]) | h_bits(r.n[2])) & 0x7fffu) == 0u;
        keys[e] = dead ? ~0ull : (sb | (uint32_t)id);
    }
}

__global__ void sb_offsets_kernel(const unsigned long long* __restrict__ keys, int64_t n, int64_t nsb, uint32_t* __restrict__ off) {
    const int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (s > nsb) return;
    const unsigned long long want = (unsigned long long)s << 32;       // first key >= want
    int64_t lo = 0, hi = n;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (keys[mid] < want) lo = mid + 1; else hi = mid;
    }
    off[s] = (uint32_t)lo;
}

__global__ void sb_ids_kernel(const unsigned long long* __restrict__ keys, int64_t n, int32_t* __restrict__ ids) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) ids[i] = (int32_t)(uint32_t)keys[i];
}

// The slot bytes per (superblock-list entry, block), gathered once from the block lists: the shadow kernel's literal stage then
// needs ONE look-up per (ray, triangle) pair instead of two dependent ones (position in the block list, then the slot byte there):
// 6.23 -> 5.99 ms per 32,768 envs for 576 instead of 128 bytes per entry.  The entry's triangle is found in each of the
// superblock's block lists by binary search (lists sorted by id; the pad entry of an odd list repeats the last id, so the
// search lands on the real entry).
__global__ void sb_slot9_kernel(const uint32_t* __restrict__ sb_off, const int32_t* __restrict__ sb_ids, const uint32_t* __restrict__ blk_off,
                                const int32_t* __restrict__ blk_ids, const uint4* __restrict__ blk_slots, int nBx, int nBy, int nSBy,
                                unsigned char* __restrict__ out) {
    const int SX = blockIdx.x / nSBy, SY = blockIdx.x % nSBy;
    const uint32_t e0 = sb_off[blockIdx.x], e1 = sb_off[blockIdx.x + 1];
    const uint32_t total = (e1 - e0) * (RVB_SB * RVB_SB);
    for (uint32_t w = threadIdx.x; w < total; w += blockDim.x) {
        const uint32_t ent = e0 + w / (RVB_SB * RVB_SB), b = w % (RVB_SB * RVB_SB);
        const int I = SX * RVB_SB + (int)(b / RVB_SB), J = SY * RVB_SB + (int)(b % RVB_SB);
        uint4 sl = make_uint4(0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu);
        if (I < nBx && J < nBy) {
            const int32_t id = sb_ids[ent];
            const uint32_t o1 = blk_off[(uint32_t)I * nBy + J + 1];
            uint32_t lo = blk_off[(uint32_t)I * nBy + J], hi = o1;
            while (lo < hi) {
                const uint32_t mid = (lo + hi) >> 1;
                if (blk_ids[mid] < id) lo = mid + 1; else hi = mid;
            }
            if (lo < o1 && blk_ids[lo] == id) sl = blk_slots[lo];
        }
        // laid out by CELL of the superblock (24 x 24): the kernel indexes it with (cx % 24) * 24 + cy % 24
        const unsigned char* sb = reinterpret_cast<const unsigned char*>(&sl);
        constexpr int SBC = RVB_SB * RVB_BLK;
        unsigned char* o = out + (size_t)ent * (SBC * SBC);
        const int ci0 = (int)(b / RVB_SB) * RVB_BLK, cj0 = (int)(b % RVB_SB) * RVB_BLK;
        for (int i = 0; i < 9; ++i) o[(ci0 + i / RVB_BLK) * SBC + cj0 + i % RVB_BLK] = sb[i];
    }
}

// one warp per window of 32 superblock-list entries: bounds of their stage-1 records
__global__ void sb_chunk_kernel(const int32_t* __restrict__ sb_ids, int64_t n, const S1Rec* __restrict__ s1, ChunkRec* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int64_t w = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    if (w * 32 >= n) return;
    const int64_t ent = w * 32 + lane;
    const float inf = __int_as_float(0x7f800000);
    float lo[3] = {inf, inf, inf}, hi[3] = {-inf, -inf, -inf}, nlo[3] = {inf, inf, inf}, nhi[3] = {-inf, -inf, -inf};
    float rmax = 0.f, cbmax = 0.f, amax = 0.f;
    bool bad = false;
    if (ent < n) {
        const S1Rec r = s1[sb_ids[ent]];
        const float cb = __half2float(__ushort_as_half((unsigned short)(r.cb_amax & 0xffffu)));
        const float am = __half2float(__ushort_as_half((unsigned short)(r.cb_amax >> 16)));
        lo[0] = hi[0] = r.qx; lo[1] = hi[1] = r.qy; lo[2] = hi[2] = r.qz;
        nlo[0] = nhi[0] = r.nx; nlo[1] = nhi[1] = r.ny; nlo[2] = nhi[2] = r.nz;
        rmax = r.r; cbmax = cb; amax = am;
        const float sum = r.qx + r.qy + r.qz + r.r + r.nx + r.ny + r.nz + cb + am;
        bad = !(fabsf(sum) <= 3.0e38f);          // NaN or inf anywhere
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            lo[i] = fminf(lo[i], __shfl_xor_sync(0xffffffffu, lo[i], o)); hi[i] = fmaxf(hi[i], __shfl_xor_sync(0xffffffffu, hi[i], o));
            nlo[i] = fminf(nlo[i], __shfl_xor_sync(0xffffffffu, nlo[i], o)); nhi[i] = fmaxf(nhi[i], __shfl_xor_sync(0xffffffffu, nhi[i], o));
        }
        rmax = fmaxf(rmax, __shfl_xor_sync(0xffffffffu, rmax, o));
        cbmax = fmaxf(cbmax, __shfl_xor_sync(0xffffffffu, cbmax, o));
        amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, o));
    }
    bad = __any_sync(0xffffffffu, bad);
    if (lane == 0) {
        ChunkRec c;
        c.x0 = bad ? __int_as_float(0x7fc00000) : lo[0]; c.x1 = hi[0]; c.y0 = lo[1]; c.y1 = hi[1]; c.z0 = lo[2]; c.z1 = hi[2];
        c.rmax = rmax; c.cbmax = cbmax; c.amax = amax;
        c.nxlo = nlo[0]; c.nxhi = nhi[0]; c.nylo = nlo[1]; c.nyhi = nhi[1]; c.nzlo = nlo[2]; c.nzhi = nhi[2];
        c.pad = 0.f;
        out[w] = c;
    }
}

static int build_superblock_lists(rvb_terrain* t, cudaStream_t st) {
    t->nSBx = (int32_t)ceil_div(t->nBx, RVB_SB);
    t->nSBy = (int32_t)ceil_div(t->nBy, RVB_SB);
    const int64_t nb = (int64_t)t->nBx * t->nBy, nsb = (int64_t)t->nSBx * t->nSBy, n = t->n_ent;
    if (!t->blk_ids || n <= 0 || n >= ((int64_t)1 << 31)) return RVB_OK;
    RvbTemp<unsigned long long> k0, k1;
    RvbTemp<int64_t> d_num;
    RvbTemp<unsigned char> tmp;
    RVB_CUDA(k0.alloc(n));
    RVB_CUDA(k1.alloc(n));
    RVB_CUDA(d_num.alloc(1));
    sb_keys_kernel<<<(unsigned)nb, 128, 0, st>>>(t->blk_off, t->blk_ids, t->recs, t->nBy, t->nSBy, k0.p);
    RVB_LAUNCH_CHECK();
    const int sb_bits = 32;          // all 64 key bits: the all-ones key of the dropped triangles has to sort last
    size_t b0 = 0, b1 = 0;
    RVB_CUDA(cub::DeviceRadixSort::SortKeys(nullptr, b0, k0.p, k1.p, (int)n, 0, 32 + sb_bits, st));
    RVB_CUDA(cub::DeviceSelect::Unique(nullptr, b1, k1.p, k0.p, d_num.p, (int)n, st));
    RVB_CUDA(tmp.alloc(b0 > b1 ? b0 : b1));
    RVB_CUDA(cub::DeviceRadixSort::SortKeys(tmp.p, b0, k0.p, k1.p, (int)n, 0, 32 + sb_bits, st));
    RVB_CUDA(cub::DeviceSelect::Unique(tmp.p, b1, k1.p, k0.p, d_num.p, (int)n, st));
    int64_t n_u = 0;
    unsigned long long last = 0;          // largest sorted key: all ones exactly when dropped triangles exist
    RVB_CUDA(cudaMemcpyAsync(&n_u, d_num.p, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    RVB_CUDA(cudaMemcpyAsync(&last, k1.p + n - 1, sizeof(last), cudaMemcpyDeviceToHost, st));
    RVB_CUDA(cudaStreamSynchronize(st));
    if (n_u > 0 && last == ~0ull) --n_u;          // the dropped triangles' one surviving key
    t->n_sb_ent = n_u;
    const size_t n_alloc = n_u > 0 ? n_u : 1;
    RVB_CUDA(cudaMalloc(&t->sb_off, sizeof(uint32_t) * (nsb + 1)));
    RVB_CUDA(cudaMalloc(&t->sb_ids, sizeof(int32_t) * n_alloc));
    sb_offsets_kernel<<<(unsigned)ceil_div(nsb + 1, 256), 256, 0, st>>>(k0.p, n_u, nsb, t->sb_off);
    sb_ids_kernel<<<(unsigned)ceil_div(n_alloc, 256), 256, 0, st>>>(k0.p, n_u, t->sb_ids);
    RVB_LAUNCH_CHECK();
    RVB_CUDA(cudaMalloc(&t->sb_slot9, (size_t)9 * RVB_SB * RVB_SB * n_alloc));
    sb_slot9_kernel<<<(unsigned)nsb, 256, 0, st>>>(t->sb_off, t->sb_ids, t->blk_off, t->blk_ids, t->blk_slots, t->nBx, t->nBy, t->nSBy,
                                                   t->sb_slot9);
    RVB_LAUNCH_CHECK();
    const int64_t nwin = ceil_div(n_alloc, 32);
    RVB_CUDA(cudaMalloc(&t->sb_chunk, sizeof(ChunkRec) * (size_t)nwin));
    sb_chunk_kernel<<<(unsigned)ceil_div(nwin * 32, 256), 256, 0, st>>>(t->sb_ids, n_u, t->s1recs, t->sb_chunk);
    RVB_LAUNCH_CHECK();
    RVB_CUDA(cudaStreamSynchronize(st));
    return RVB_OK;
}

static int build_block_lists(rvb_terrain* t, cudaStream_t st) {
    t->nBx = (int32_t)ceil_div(t->G0, RVB_BLK);
    t->nBy = (int32_t)ceil_div(t->G1, RVB_BLK);
    const int64_t nb = (int64_t)t->nBx * t->nBy;
    if (t->K > 255 || nb >= ((int64_t)1 << 31)) return RVB_OK;      // per-cell path only
    RvbTemp<uint32_t> counts;
    RvbTemp<unsigned char> tmp;
    RVB_CUDA(cudaMalloc(&t->blk_off, sizeof(uint32_t) * (nb + 1)));
    RVB_CUDA(counts.alloc(nb + 1));
    RVB_CUDA(cudaMemsetAsync(counts.p, 0, sizeof(uint32_t) * (nb + 1), st));
    build_blocks_kernel<<<(unsigned)nb, BLK_THREADS, 0, st>>>(t->index, (int)t->G0, (int)t->G1, (int)t->K, (int)t->Ks, t->nBy, nullptr,
                                                             counts.p, nullptr, nullptr);
    RVB_LAUNCH_CHECK();
    size_t tmp_bytes = 0;
    RVB_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, counts.p, t->blk_off, (int)(nb + 1), st));
    RVB_CUDA(tmp.alloc(tmp_bytes));
    RVB_CUDA(cub::DeviceScan::ExclusiveSum(tmp.p, tmp_bytes, counts.p, t->blk_off, (int)(nb + 1), st));
    uint32_t total = 0;
    RVB_CUDA(cudaMemcpyAsync(&total, t->blk_off + nb, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    RVB_CUDA(cudaStreamSynchronize(st));
    t->n_ent = total;
    RVB_CUDA(cudaMalloc(&t->blk_ids, sizeof(int32_t) * (size_t)(total > 0 ? total : 1)));
    RVB_CUDA(cudaMalloc(&t->blk_slots, sizeof(uint4) * (size_t)(total > 0 ? total : 1)));
    RVB_CUDA(cudaMemsetAsync(t->blk_ids, 0, sizeof(int32_t) * (size_t)total, st));
    RVB_CUDA(cudaMemsetAsync(t->blk_slots, 0xff, sizeof(uint4) * (size_t)total, st));
    build_blocks_kernel<<<(unsigned)nb, BLK_THREADS, 0, st>>>(t->index, (int)t->G0, (int)t->G1, (int)t->K, (int)t->Ks, t->nBy, t->blk_off,
                                                             nullptr, t->blk_ids, t->blk_slots);
    RVB_LAUNCH_CHECK();
    return build_superblock_lists(t, st);
}

extern "C" int rvb_terrain_create(rvb_terrain** out, const int32_t* map_indices, int64_t G0, int64_t G1, int64_t K,
                                  int64_t stride_g0, int64_t stride_g1, int64_t stride_k, const int32_t* triangles,
                                  int64_t T, const uint16_t* vertices, int64_t V, float res, float shift_x,
                                  float shift_y, int sem, int flags, void* stream) {
    RVB_REQUIRE(out != nullptr, "rvb_terrain_create: out is null");
    RVB_REQUIRE((flags & ~RVB_LAYER_INDEX_ONLY) == 0, "rvb_terrain_create: unknown flag");
    *out = nullptr;
    RVB_REQUIRE(map_indices && triangles && vertices, "rvb_terrain_create: null device pointer");
    RVB_REQUIRE(G0 > 0 && G1 > 0 && K > 0 && K <= 4096, "rvb_terrain_create: need G0,G1 > 0 and 0 < K <= 4096");
    RVB_REQUIRE(T > 0 && T < (int64_t)1 << 31 && V > 0 && V < (int64_t)1 << 31, "rvb_terrain_create: bad T or V");
    RVB_REQUIRE(res > 0.0f, "rvb_terrain_create: res must be > 0");
    RVB_REQUIRE(sem == RVB_SEM_TORCH_CUDA || sem == RVB_SEM_TORCH_CPU, "rvb_terrain_create: bad sem");
    cudaStream_t st = as_stream(stream);
    // value-initialised (every array null), so on a failure rvb_terrain_destroy frees exactly what was built
    std::unique_ptr<rvb_terrain, int (*)(rvb_terrain*)> t(new (std::nothrow) rvb_terrain(), rvb_terrain_destroy);
    if (!t) return rvb_set_error(RVB_ERR_NOMEM, "rvb_terrain_create", "host allocation failed");
    t->G0 = G0; t->G1 = G1; t->K = K; t->Ks = (K + 1) & ~(int64_t)1; t->T = T; t->V = V;
    t->res = res; t->shift_x = shift_x; t->shift_y = shift_y; t->sem = sem;
    RVB_CUDA(cudaGetDevice(&t->device));
    RVB_CUDA(cudaMalloc(&t->index, sizeof(int32_t) * G0 * G1 * t->Ks));
    RVB_CUDA(cudaMalloc(&t->recs, sizeof(TriRec) * T));
    RVB_CUDA(cudaMalloc(&t->s1recs, sizeof(S1Rec) * T));
    {
        RvbTemp<int> bad;
        RVB_CUDA(bad.alloc(2));
        RVB_CUDA(cudaMemsetAsync(bad.p, 0, 2 * sizeof(int), st));
        repack_index_kernel<<<148 * 8, 256, 0, st>>>(map_indices, G0, G1, K, t->Ks, stride_g0, stride_g1, stride_k, (int32_t)T,
                                                     t->index, bad.p);
        build_records_kernel<<<(unsigned)ceil_div(T, 256), 256, 0, st>>>(triangles, T, (const __half*)vertices, V,
                                                                         t->recs, t->s1recs, bad.p);
        RVB_LAUNCH_CHECK();
        int hb[2] = {0, 0};
        RVB_CUDA(cudaMemcpyAsync(hb, bad.p, sizeof(hb), cudaMemcpyDeviceToHost, st));
        RVB_CUDA(cudaStreamSynchronize(st));
        if (hb[0])
            return rvb_set_error(RVB_ERR_INVALID, "rvb_terrain_create",
                                 hb[0] == 1 ? "map_indices holds a triangle id outside [0,T)" : "triangles holds a vertex id outside [0,V)");
        t->n_ill = hb[1];
    }
    if (!(flags & RVB_LAYER_INDEX_ONLY)) {
        const int rc = build_block_lists(t.get(), st);
        if (rc != RVB_OK) return rc;
        RVB_CUDA(cudaStreamSynchronize(st));
    }
    *out = t.release();
    return RVB_OK;
}

extern "C" int rvb_terrain_destroy(rvb_terrain* t) {
    if (!t) return RVB_OK;
    cudaFree(t->index);
    cudaFree(t->recs);
    cudaFree(t->s1recs);
    cudaFree(t->blk_off);
    cudaFree(t->blk_ids);
    cudaFree(t->blk_slots);
    cudaFree(t->sb_off);
    cudaFree(t->sb_ids);
    cudaFree(t->sb_slot9);
    cudaFree(t->sb_chunk);
    delete t;
    return RVB_OK;
}

// The K-contiguous copy of the index (G0*G1*Ks int32, 3.2 GB on the benchmark world) is what the per-pair cross-check kernel, the
// rock kernel and rvb_cast_rays read.  The production heightmap ray-cast does not: the shadow and tiled kernels enumerate the block
// / superblock lists, and the two rare look-ups that went through the index (a ray with a hit beyond 11 m, the optional hit-triangle
// output) can be answered from the block lists (raycast_common.cuh).  A heightmap layer can therefore give the copy back.
extern "C" int rvb_terrain_release_index(rvb_terrain* t) {
    RVB_REQUIRE(t != nullptr, "rvb_terrain_release_index: null handle");
    if (!t->index) return RVB_OK;
    RVB_REQUIRE(t->blk_ids != nullptr && t->blk_slots != nullptr,
                "rvb_terrain_release_index: the layer has no block lists (K > 255), its kernels read the index");
    int prev = 0;
    RVB_CUDA(cudaGetDevice(&prev));
    RVB_CUDA(cudaSetDevice(t->device));
    cudaError_t e = cudaDeviceSynchronize();          // launches that still read the copy
    if (e == cudaSuccess) e = cudaFree(t->index);
    cudaSetDevice(prev);
    RVB_CUDA(e);
    t->index = nullptr;
    return RVB_OK;
}

extern "C" int rvb_terrain_has_index(const rvb_terrain* t) { return t && t->index ? 1 : 0; }

extern "C" int64_t rvb_terrain_unbounded_triangles(const rvb_terrain* t) { return t ? (int64_t)t->n_ill : 0; }

extern "C" int64_t rvb_terrain_bytes(const rvb_terrain* t) {
    if (!t) return 0;
    return (t->index ? (int64_t)sizeof(int32_t) * t->G0 * t->G1 * t->Ks : 0) + (int64_t)(sizeof(TriRec) + sizeof(S1Rec)) * t->T +
           (t->blk_ids ? (int64_t)(sizeof(uint4) + sizeof(int32_t)) * t->n_ent + (int64_t)sizeof(uint32_t) * ((int64_t)t->nBx * t->nBy + 1) : 0) +
           (t->sb_ids ? (int64_t)(sizeof(int32_t) + 9 * RVB_SB * RVB_SB) * t->n_sb_ent + (int64_t)sizeof(uint32_t) * ((int64_t)t->nSBx * t->nSBy + 1) +
                         (int64_t)sizeof(ChunkRec) * ceil_div(t->n_sb_ent > 0 ? t->n_sb_ent : 1, 32) : 0);
}
