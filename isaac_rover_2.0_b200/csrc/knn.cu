// Offline K-nearest-centroid index builder (rover_utils.py:52-118 _get_knn_triangles) on the device.
//
// Reference semantics: 2-D triangle centroids rounded to fp16, cell (i,j) at fp16 coordinates
// (cell_x[i], cell_y[j]) (torch.arange(0, G*res, res, dtype=float16), passed in so that torch's own arange
// rounding is used), distance = fp16(sqrt(fp32(dx16)^2 + fp32(dy16)^2)) with dx16 = fp16(cx16 - px16)
// (torch.norm on a Half tensor), K smallest per cell.  torch.topk leaves the order of equal distances
// unspecified; here the order is (distance, triangle id), which makes the asset reproducible.
//
// The reference brute-forces all T triangles for every cell (3600 topk calls).  Here the centroids are
// binned into a uniform bucket grid (CSR) and each cell -- one CTA -- scans a window of buckets that
// provably contains every triangle whose fp16 distance can be <= the K-th smallest one, sorts the
// candidates' 64-bit keys (distance bits << 32 | id) in shared memory and writes the first K ids.
#include <cub/device/device_scan.cuh>
#include <math_constants.h>

#include "common.cuh"

namespace {

struct BucketGrid {
    float x0, y0, inv_b, b;
    int nx, ny;
};

__device__ __forceinline__ unsigned enc_f(float f) {   // order-preserving float -> uint
    unsigned u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__host__ __device__ __forceinline__ float dec_f(unsigned u) {
    unsigned v = (u & 0x80000000u) ? (u & 0x7fffffffu) : ~u;
#ifdef __CUDA_ARCH__
    return __uint_as_float(v);
#else
    float f;
    memcpy(&f, &v, 4);
    return f;
#endif
}

// centroid = fp16(((v0 + v1) + v2) / 3) in fp64 (rover_utils.py:69-73 on the fp16 vertex asset)
__global__ void centroid_kernel(const int32_t* __restrict__ tri, int64_t T, const __half* __restrict__ vert, int64_t V,
                                __half2* __restrict__ cen, unsigned* __restrict__ bbox, int* bad) {
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= T) return;
    int32_t a = tri[i * 3], b = tri[i * 3 + 1], c = tri[i * 3 + 2];
    if (a < 0 || a >= V || b < 0 || b >= V || c < 0 || c >= V) {
        atomicExch(bad, 1);
        a = b = c = 0;
    }
    double x = __ddiv_rn(__dadd_rn(__dadd_rn((double)__half2float(vert[a * 3]), (double)__half2float(vert[b * 3])),
                                   (double)__half2float(vert[c * 3])), 3.0);
    double y = __ddiv_rn(__dadd_rn(__dadd_rn((double)__half2float(vert[a * 3 + 1]), (double)__half2float(vert[b * 3 + 1])),
                                   (double)__half2float(vert[c * 3 + 1])), 3.0);
    __half hx = h_from_double(x), hy = h_from_double(y);
    cen[i] = __halves2half2(hx, hy);
    atomicMin(bbox + 0, enc_f(__half2float(hx)));
    atomicMax(bbox + 1, enc_f(__half2float(hx)));
    atomicMin(bbox + 2, enc_f(__half2float(hy)));
    atomicMax(bbox + 3, enc_f(__half2float(hy)));
}

__device__ __forceinline__ int bucket_coord(float v, float v0, float inv_b, int n) {
    int c = (int)floorf((v - v0) * inv_b);
    return min(max(c, 0), n - 1);
}

__global__ void bucket_count_kernel(const __half2* __restrict__ cen, int64_t T, BucketGrid g, int* __restrict__ counts) {
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= T) return;
    float2 c = __half22float2(cen[i]);
    atomicAdd(counts + bucket_coord(c.x, g.x0, g.inv_b, g.nx) * g.ny + bucket_coord(c.y, g.y0, g.inv_b, g.ny), 1);
}

__global__ void bucket_fill_kernel(const __half2* __restrict__ cen, int64_t T, BucketGrid g, const int* __restrict__ offsets,
                                   int* __restrict__ cursor, int* __restrict__ items) {
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= T) return;
    float2 c = __half22float2(cen[i]);
    int b = bucket_coord(c.x, g.x0, g.inv_b, g.nx) * g.ny + bucket_coord(c.y, g.y0, g.inv_b, g.ny);
    items[offsets[b] + atomicAdd(cursor + b, 1)] = (int)i;
}

constexpr int KNN_THREADS = 128;
constexpr int KNN_CAP = 2048;      // keys sorted at once (16 KB of shared memory)

__device__ __forceinline__ unsigned long long knn_key(__half2 cen, __half px, __half py, int id) {
    __half dx = h_sub(__low2half(cen), px), dy = h_sub(__high2half(cen), py);
    float fx = __half2float(dx), fy = __half2float(dy);
    __half d = __float2half_rn(__fsqrt_rn(__fadd_rn(__fmul_rn(fx, fx), __fmul_rn(fy, fy))));
    return ((unsigned long long)h_bits(d) << 32) | (unsigned)id;     // d >= 0: bit order == value order
}

// in-place bitonic sort of n (power of two) 64-bit keys in shared memory
__device__ void bitonic_sort(unsigned long long* keys, int n) {
    for (int k = 2; k <= n; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = threadIdx.x; i < n; i += KNN_THREADS) {
                int ixj = i ^ j;
                if (ixj > i) {
                    unsigned long long a = keys[i], b = keys[ixj];
                    bool up = (i & k) == 0;
                    if ((a > b) == up) {
                        keys[i] = b;
                        keys[ixj] = a;
                    }
                }
            }
            __syncthreads();
        }
    }
}

__global__ void __launch_bounds__(KNN_THREADS)
knn_cells_kernel(const __half2* __restrict__ cen, BucketGrid g, const int* __restrict__ offsets,
                 const int* __restrict__ items, const __half* __restrict__ cell_x, const __half* __restrict__ cell_y,
                 int G0, int G1, int K, int r0, int32_t* __restrict__ out) {
    __shared__ unsigned long long keys[KNN_CAP];
    __shared__ int s_r;
    const int cell = blockIdx.x;
    const int ci = cell / G1, cj = cell % G1;
    const __half px = cell_x[ci], py = cell_y[cj];
    const float fx = __half2float(px), fy = __half2float(py);
    const int bx = bucket_coord(fx, g.x0, g.inv_b, g.nx), by = bucket_coord(fy, g.y0, g.inv_b, g.ny);
    const int rmax = max(g.nx, g.ny);
    int r = r0;
    const int64_t plane = (int64_t)G0 * G1;
    while (true) {
        // The buckets (x, ya..yb) of one window row are contiguous in the CSR item array, so the window is
        // (xb-xa+1) contiguous item segments.  They are streamed through the key buffer: whenever it fills up
        // it is sorted and cut back to the best K.  Control flow is uniform across the CTA.
        const int xa = max(bx - r, 0), xb = min(bx + r, g.nx - 1), ya = max(by - r, 0), yb = min(by + r, g.ny - 1);
        int fill = 0, kept = 0;
        for (int x = xa; x <= xb; ++x) {
            int beg = offsets[x * g.ny + ya];
            const int end = offsets[x * g.ny + yb + 1];
            while (beg < end) {
                const int n = min(KNN_CAP - fill, end - beg);
                for (int q = threadIdx.x; q < n; q += KNN_THREADS) {
                    const int id = items[beg + q];
                    keys[fill + q] = knn_key(cen[id], px, py, id);
                }
                fill += n;
                beg += n;
                if (fill == KNN_CAP) {
                    __syncthreads();
                    bitonic_sort(keys, KNN_CAP);
                    fill = K;
                }
            }
        }
        {
            int p2 = 2;
            while (p2 < fill) p2 <<= 1;
            for (int i = fill + threadIdx.x; i < p2; i += KNN_THREADS) keys[i] = ~0ull;
            __syncthreads();
            bitonic_sort(keys, p2);
            kept = min(fill, K);
        }
        // ---- is the window provably large enough?
        bool done = false;
        int next_r = r + 1;
        if (xa == 0 && ya == 0 && xb == g.nx - 1 && yb == g.ny - 1) done = true;        // whole grid scanned
        else if (kept >= K) {
            const float dk = __half2float(h_from_bits((unsigned short)(keys[K - 1] >> 32)));
            // every triangle outside the window is farther than r*b from the (bbox-clamped) cell; fp16 evaluation
            // of its distance cannot come out below r*b*(1 - 2^-8)
            const float safe = (float)r * g.b * (1.0f - 1.0f / 256.0f);
            if (dk < safe) done = true;
            else next_r = max(r + 1, (int)ceilf(dk / (g.b * (1.0f - 1.0f / 256.0f))) + 1);
        }
        if (threadIdx.x == 0) s_r = done ? -1 : min(next_r, rmax);
        __syncthreads();
        if (s_r < 0) {
            for (int k = threadIdx.x; k < K; k += KNN_THREADS)
                out[(int64_t)k * plane + cell] = (k < kept) ? (int32_t)(keys[k] & 0xffffffffu) : (int32_t)(keys[kept - 1] & 0xffffffffu);
            return;
        }
        r = s_r;
        __syncthreads();
    }
}

}  // namespace

extern "C" int rvb_build_knn_index(const int32_t* triangles, int64_t T, const uint16_t* vertices, int64_t V,
                                   const uint16_t* cell_x, const uint16_t* cell_y, int64_t G0, int64_t G1, int64_t K,
                                   int32_t* out, void* stream) {
    RVB_REQUIRE(triangles && vertices && cell_x && cell_y && out, "rvb_build_knn_index: null pointer");
    RVB_REQUIRE(T > 0 && T < ((int64_t)1 << 31) && V > 0 && V < ((int64_t)1 << 31), "rvb_build_knn_index: bad T or V");
    RVB_REQUIRE(G0 > 0 && G1 > 0 && G0 * G1 < ((int64_t)1 << 31), "rvb_build_knn_index: bad grid");
    RVB_REQUIRE(K > 0 && K <= 1024 && K <= T, "rvb_build_knn_index: need 0 < K <= min(T, 1024)");
    cudaStream_t st = as_stream(stream);
    RvbTemp<__half2> cen;
    RvbTemp<unsigned> bbox;          // 4 encoded bounds, then the bad-vertex flag
    RvbTemp<int> counts, items;
    RvbTemp<unsigned char> tmp;
    RVB_CUDA(cen.alloc_pool(T, st));
    RVB_CUDA(bbox.alloc_pool(5, st));
    int* bad = reinterpret_cast<int*>(bbox.p + 4);
    const unsigned init[5] = {0xffffffffu, 0u, 0xffffffffu, 0u, 0u};
    RVB_CUDA(cudaMemcpyAsync(bbox.p, init, sizeof(init), cudaMemcpyHostToDevice, st));
    centroid_kernel<<<(unsigned)ceil_div(T, 256), 256, 0, st>>>(triangles, T, (const __half*)vertices, V, cen.p, bbox.p, bad);
    RVB_LAUNCH_CHECK();
    unsigned hb[5];
    RVB_CUDA(cudaMemcpyAsync(hb, bbox.p, sizeof(hb), cudaMemcpyDeviceToHost, st));
    RVB_CUDA(cudaStreamSynchronize(st));
    if (hb[4]) return rvb_set_error(RVB_ERR_INVALID, "rvb_build_knn_index", "triangles holds a vertex id outside [0,V)");
    const float x0 = dec_f(hb[0]), x1 = dec_f(hb[1]), y0 = dec_f(hb[2]), y1 = dec_f(hb[3]);
    const float w = fmaxf(x1 - x0, 1e-3f), h = fmaxf(y1 - y0, 1e-3f);
    // ~12 triangles per bucket on average, at most ~4M buckets
    float b = sqrtf(12.0f * w * h / (float)T);
    b = fmaxf(b, fmaxf(w, h) / 2000.0f);
    BucketGrid g;
    g.x0 = x0; g.y0 = y0; g.b = b; g.inv_b = 1.0f / b;
    g.nx = (int)floorf(w / b) + 1; g.ny = (int)floorf(h / b) + 1;
    const int64_t NB = (int64_t)g.nx * g.ny;
    RVB_CUDA(counts.alloc_pool((NB + 1) * 2, st));
    int* offsets = counts.p + NB + 1;
    RVB_CUDA(items.alloc_pool(T, st));
    RVB_CUDA(cudaMemsetAsync(counts.p, 0, sizeof(int) * (NB + 1), st));
    bucket_count_kernel<<<(unsigned)ceil_div(T, 256), 256, 0, st>>>(cen.p, T, g, counts.p);
    size_t tmp_bytes = 0;
    RVB_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, counts.p, offsets, (int)(NB + 1), st));
    RVB_CUDA(tmp.alloc_pool(tmp_bytes, st));
    RVB_CUDA(cub::DeviceScan::ExclusiveSum(tmp.p, tmp_bytes, counts.p, offsets, (int)(NB + 1), st));
    RVB_CUDA(cudaMemsetAsync(counts.p, 0, sizeof(int) * (NB + 1), st));
    bucket_fill_kernel<<<(unsigned)ceil_div(T, 256), 256, 0, st>>>(cen.p, T, g, offsets, counts.p, items.p);
    // initial window radius: a disc holding K triangles at average density, in buckets
    const float dens = (float)T / (w * h);
    const int r0 = (int)ceilf(sqrtf((float)K / (3.14159f * dens)) / b) + 1;
    knn_cells_kernel<<<(unsigned)(G0 * G1), KNN_THREADS, 0, st>>>(cen.p, g, offsets, items.p, (const __half*)cell_x,
                                                                 (const __half*)cell_y, (int)G0, (int)G1, (int)K, r0, out);
    RVB_LAUNCH_CHECK();
    return RVB_OK;
}
