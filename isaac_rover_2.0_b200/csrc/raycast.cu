// Heightmap ray-cast: Camera.get_depths (camera.py:60-145) and the generic "cast fp16 rays against a
// layer" used by Rock_Detection.get_collisions (rock_detect.py:52-149).
//
// variant 1 ("simple"): one warp per ray, lanes stride over the K candidates of the ray's cell, every
// (ray, candidate) pair evaluated with the literal op sequence of ray_casting.py.  Kept as the on-device
// cross-check for the production kernel (raycast_shadow.cu) and its tiled fall-back (raycast_tiled.cu).
#include "raycast_common.cuh"

// ------------------------------------------------------------------------------------------------
// setup: sources (fp64 transform -> fp16), per-env direction, per-ray cell
// ------------------------------------------------------------------------------------------------
__global__ void hm_setup_kernel(const float* __restrict__ pos, const float* __restrict__ euler,
                                const float* __restrict__ trig, const double* __restrict__ pattern, int P,
                                __half* __restrict__ src16, __half* __restrict__ dneg16) {
    const int64_t n = blockIdx.y;
    __shared__ Trig s_t;
    __shared__ double s_pos[3];
    if (threadIdx.x == 0) {
        s_t = make_trig(euler, trig, n);
        s_pos[0] = (double)pos[n * 3 + 0];
        s_pos[1] = (double)pos[n * 3 + 1];
        s_pos[2] = (double)pos[n * 3 + 2];
    }
    __syncthreads();
    const Trig t = s_t;
    const double tx = s_pos[0], ty = s_pos[1], tz = s_pos[2];
    int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p < P) {
        double xo, yo, zo;
        body_transform<double>(pattern[p * 3 + 0], pattern[p * 3 + 1], pattern[p * 3 + 2], t, tx, ty, tz, xo, yo, zo);
        __half* o = src16 + (n * P + p) * 3;
        o[0] = h_from_double(xo);
        o[1] = h_from_double(yo);
        o[2] = h_from_double(zo);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        const H3 d = rc::env_dir16(t, tx, ty, tz);
        dneg16[n * 3 + 0] = d.x;
        dneg16[n * 3 + 1] = d.y;
        dneg16[n * 3 + 2] = d.z;
    }
}

__global__ void normalize_dirs_kernel(const __half* __restrict__ dirs, int64_t R, __half* __restrict__ dneg16) {
    int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (r >= R) return;
    H3 d = neg_normalize({dirs[r * 3], dirs[r * 3 + 1], dirs[r * 3 + 2]});
    dneg16[r * 3 + 0] = d.x;
    dneg16[r * 3 + 1] = d.y;
    dneg16[r * 3 + 2] = d.z;
}

// ------------------------------------------------------------------------------------------------
// simple cast: warp per ray
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
cast_simple_kernel(const int32_t* __restrict__ index, const TriRec* __restrict__ recs, int G0, int G1, int K, int Ks,
                   float res, float inv_res, float shift_x, float shift_y, int sem,
                   const __half* __restrict__ src16, const __half* __restrict__ dneg16, int64_t R,
                   int64_t rays_per_dir, __half* __restrict__ dist, int32_t* __restrict__ hit_slot,
                   int32_t* __restrict__ hit_tri, __half* __restrict__ pt, float* __restrict__ obs, int64_t obs_ld,
                   const int32_t* __restrict__ col_a, const int32_t* __restrict__ col_b) {
    const int lane = threadIdx.x & 31;
    const int64_t ray = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    if (ray >= R) return;
    const H3 s = {src16[ray * 3], src16[ray * 3 + 1], src16[ray * 3 + 2]};
    const int64_t di = ray / rays_per_dir;
    const H3 d = {dneg16[di * 3], dneg16[di * 3 + 1], dneg16[di * 3 + 2]};
    const int2 cell = rc::ray_cell(s.x, s.y, shift_x, shift_y, res, inv_res, G0, G1, sem);
    const int32_t* row = index + ((int64_t)cell.x * G1 + cell.y) * Ks;
    uint32_t best = 0xffffffffu;
    unsigned short best_bits = RVB_H_MISS;
    for (int j = lane; j < K; j += 32) {
        const int32_t id = __ldg(row + j);
        const uint4* rp = reinterpret_cast<const uint4*>(recs + id);
        uint4 q0 = __ldg(rp), q1 = __ldg(rp + 1);
        const __half* h0 = reinterpret_cast<const __half*>(&q0);
        const __half* h1 = reinterpret_cast<const __half*>(&q1);
        H3 a = {h0[0], h0[1], h0[2]}, b = {h0[3], h0[4], h0[5]}, c = {h0[6], h0[7], h1[0]}, n = {h1[1], h1[2], h1[3]};
        __half k = pair_test(s, d, a, b, c, n);
        uint32_t key = min_key(k, (uint32_t)j);
        if (key < best) {
            best = key;
            best_bits = h_bits(k);
        }
    }
    const uint32_t wbest = __reduce_min_sync(0xffffffffu, best);
    const unsigned owner = __ballot_sync(0xffffffffu, best == wbest);
    const int src_lane = __ffs(owner) - 1;
    const unsigned short kb = (unsigned short)__shfl_sync(0xffffffffu, (int)best_bits, src_lane);
    if (lane == 0) {
        const int slot = (int)(wbest & 0xffffu);
        const __half k = h_from_bits(kb);
        dist[ray] = k;
        if (hit_slot) hit_slot[ray] = slot;
        if (hit_tri) hit_tri[ray] = row[slot];
        if (pt) {
            pt[ray * 3 + 0] = h_sub(s.x, h_mul(d.x, k));     // ray_casting.py:63
            pt[ray * 3 + 1] = h_sub(s.y, h_mul(d.y, k));
            pt[ray * 3 + 2] = h_sub(s.z, h_mul(d.z, k));
        }
        if (obs) {
            const int64_t n = ray / rays_per_dir, p = ray % rays_per_dir;
            const float v = __half2float(h_mul(k, __float2half_rn(0.5f)));   // fp16 (dist / 2), exact either way
            const int ca = col_a[p], cb = col_b[p];
            if (ca >= 0) obs[n * obs_ld + ca] = v;
            if (cb >= 0) obs[n * obs_ld + cb] = v;
        }
    }
}

static int launch_cast_simple(const rvb_terrain* t, const __half* src16, const __half* dneg16, int64_t R,
                              int64_t rays_per_dir, __half* dist, int32_t* hit_slot, int32_t* hit_tri, __half* pt,
                              float* obs, int64_t obs_ld, const int32_t* col_a, const int32_t* col_b, cudaStream_t st) {
    const int64_t blocks = ceil_div(R * 32, 256);
    RVB_REQUIRE(blocks < ((int64_t)1 << 31), "cast: too many rays for one launch");
    cast_simple_kernel<<<(unsigned)blocks, 256, 0, st>>>(t->index, t->recs, (int)t->G0, (int)t->G1, (int)t->K, (int)t->Ks, t->res,
                                                         1.0f / t->res, t->shift_x, t->shift_y, t->sem, src16, dneg16, R,
                                                         rays_per_dir, dist, hit_slot, hit_tri, pt, obs, obs_ld, col_a, col_b);
    RVB_LAUNCH_CHECK();
    return RVB_OK;
}

int heightmap_raycast(const rvb_terrain* t, const rc::TiledParams& q, int64_t N, int variant, const RaycastKnobs& knobs,
                      const int32_t* order, cudaStream_t st) {
    if (variant != 1) {
        // a layer with more than 2 % of triangles the shadow kernel has no bound for (terrain.cu: n_ill): the tiled kernel is the faster one
        const bool shadow_ok = knobs.force >= 0 ? knobs.force == 1 : t->n_ill * 50 <= t->T;
        if (variant == 0 && t->sb_ids != nullptr && shadow_ok) return launch_shadow(q, N, knobs, order, st);
        return launch_tiled(q, t->blk_ids != nullptr && variant != 2, N * q.tiles, st);
    }
    __half* src16 = q.sources;
    RvbTemp<__half> scratch;          // the N directions, then (without `sources`) the N * P sources
    RVB_CUDA(scratch.alloc_pool(3 * (size_t)N + (src16 ? 0 : 3 * (size_t)N * q.P), st));
    __half* dneg = scratch.p;
    if (!src16) src16 = scratch.p + 3 * N;
    dim3 grid((unsigned)ceil_div(q.P, 256), (unsigned)N);
    hm_setup_kernel<<<grid, 256, 0, st>>>(q.pos, q.euler, q.trig, q.pattern, q.P, src16, dneg);
    RVB_LAUNCH_CHECK();
    return launch_cast_simple(t, src16, dneg, N * q.P, q.P, q.dist, q.hit_slot, q.hit_tri, q.pt, q.obs, q.obs_ld, q.col_a, q.col_b, st);
}

extern "C" int rvb_heightmap_raycast(const rvb_terrain* t, const float* pos, const float* euler, const float* trig,
                                     const double* pattern, int64_t P, int64_t N, uint16_t* dist, int32_t* hit_slot,
                                     int32_t* hit_tri, uint16_t* pt, uint16_t* sources, float* obs, int64_t obs_ld,
                                     uint16_t* obs_h16, int64_t obs_h16_ld, int obs_h16_col0, const int32_t* col_a,
                                     const int32_t* col_b, int variant, void* stream) {
    RaycastKnobs knobs;
    const int krc = read_raycast_knobs(knobs);
    if (krc != RVB_OK) return krc;
    rc::TiledParams q{};
    q.pos = pos; q.euler = euler; q.trig = trig; q.pattern = pattern;
    q.dist = (__half*)dist; q.hit_slot = hit_slot; q.hit_tri = hit_tri; q.pt = (__half*)pt; q.sources = (__half*)sources;
    q.obs = obs; q.obs_ld = obs_ld; q.col_a = col_a; q.col_b = col_b;
    q.obs16 = (__half*)obs_h16; q.obs16_ld = obs_h16_ld; q.obs16_col0 = obs_h16_col0;
    const int prc = fill_tiled_params(t, P, N, variant, q);
    if (prc != RVB_OK || N == 0) return prc;
    return heightmap_raycast(t, q, N, variant, knobs, nullptr, as_stream(stream));
}

extern "C" int rvb_cast_rays(const rvb_terrain* t, const uint16_t* sources, const uint16_t* directions, int64_t R,
                             uint16_t* dist, int32_t* hit_slot, int32_t* hit_tri, uint16_t* pt, void* stream) {
    RVB_REQUIRE(R >= 0, "rvb_cast_rays: R < 0");
    if (R == 0) return RVB_OK;
    RVB_REQUIRE(t && sources && directions && dist, "rvb_cast_rays: null pointer");
    RVB_REQUIRE(t->index != nullptr, "rvb_cast_rays: the layer released its index (rvb_terrain_release_index)");
    cudaStream_t st = as_stream(stream);
    RvbTemp<__half> dneg;
    RVB_CUDA(dneg.alloc_pool(3 * (size_t)R, st));
    normalize_dirs_kernel<<<(unsigned)ceil_div(R, 256), 256, 0, st>>>((const __half*)directions, R, dneg.p);
    return launch_cast_simple(t, (const __half*)sources, dneg.p, R, 1, (__half*)dist, hit_slot, hit_tri, (__half*)pt, nullptr, 0, nullptr,
                              nullptr, st);
}

// ------------------------------------------------------------------------------------------------
// ray_distance (ray_casting.py:3-66): n rays vs n raw triangles
// ------------------------------------------------------------------------------------------------
__global__ void ray_distance_kernel(const __half* __restrict__ src, const __half* __restrict__ dirs,
                                    const __half* __restrict__ tri, int64_t n, __half* __restrict__ k_out,
                                    __half* __restrict__ pt) {
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    H3 s = {src[i * 3], src[i * 3 + 1], src[i * 3 + 2]};
    H3 d = neg_normalize({dirs[i * 3], dirs[i * 3 + 1], dirs[i * 3 + 2]});
    const __half* q = tri + i * 9;
    H3 v0 = {q[0], q[1], q[2]}, v1 = {q[3], q[4], q[5]}, a = {q[6], q[7], q[8]};
    H3 b = h3_sub(v1, a), c = h3_sub(v0, a);
    H3 nn = h3_cross(b, c);
    __half k = pair_test(s, d, a, b, c, nn);
    k_out[i] = k;
    if (pt) {
        pt[i * 3 + 0] = h_sub(s.x, h_mul(d.x, k));
        pt[i * 3 + 1] = h_sub(s.y, h_mul(d.y, k));
        pt[i * 3 + 2] = h_sub(s.z, h_mul(d.z, k));
    }
}

extern "C" int rvb_ray_distance(const uint16_t* sources, const uint16_t* directions, const uint16_t* triangles,
                                int64_t n, uint16_t* k, uint16_t* pt, void* stream) {
    RVB_REQUIRE(n >= 0, "rvb_ray_distance: n < 0");
    if (n == 0) return RVB_OK;
    RVB_REQUIRE(sources && directions && triangles && k, "rvb_ray_distance: null pointer");
    ray_distance_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, as_stream(stream)>>>(
        (const __half*)sources, (const __half*)directions, (const __half*)triangles, n, (__half*)k, (__half*)pt);
    RVB_LAUNCH_CHECK();
    return RVB_OK;
}
