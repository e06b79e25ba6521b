// Production heightmap ray-cast kernel: Camera.get_depths (camera.py:60-145) in ONE launch.
//
// One CTA per (env, ray tile).  Phases, all inside the CTA:
//   1. every thread transforms its rays (fp64 body transform -> fp16 sources, camera.py:165-212) and looks up
//      their grid cell (camera.py:233-264);
//   2. the tile's rays are grouped by 3x3-cell BLOCK (terrain.cu builds, per block, the union of its cells' K-lists
//      with the slot each triangle holds in each cell) with a counting sort over the tile's bounding box
//      (shared-memory histogram + scan): ~10 rays share one fetch of every candidate record, while each ray is
//      still answered from exactly its own cell's list (a survivor that is not in the ray's cell is dropped, its
//      slot in that cell's list is the tie-break key).  Layers with K > 255 use the same kernel with 1x1 blocks;
//   3. warps pull (cell, ray-range) items from a shared counter.  A lane owns TWO candidates of the cell's list:
//      it gathers their pre-resolved 32-byte records (L2-resident table), packs them into half2 registers and
//      then loops over the rays of the item.  All fp16 arithmetic of ray_casting.py:34-56 runs as packed
//      HADD2/HMUL2 (.rn, never contracted) on the two candidates at once;
//   4. the three divisions of ray_casting.py:44-56 are NOT executed for candidates that miss: the barycentric
//      test `n >= -eps, m >= -eps, n + m <= 1 + eps` on the rounded quotients is decided exactly from the
//      un-divided numerators (see pair2_keys); only candidates that pass (about 1 in 140) pay for the one
//      IEEE division that produces k.  A candidate whose n+m lies within 2^-9 of the threshold is re-evaluated
//      with the literal op sequence (pair_test), so the result is bit-identical by construction;
//   5. per ray: warp REDUX.MIN over a 32-bit key (order-preserving fp16 bits << 16 | slot) reproduces torch.min
//      (NaN first, ties -> lowest slot), merged across candidate chunks with a shared-memory atomicMin;
//   6. epilogue in ray order: coalesced stores of dist / hit slot / hit triangle / pt / sources and the fused
//      sparse+dense observation columns (heightmap_distribution.py:126-133, rover.py:324-325).
#include "raycast_common.cuh"

namespace {

using namespace rc;

constexpr int TT = 256;            // threads per CTA
constexpr int NW = TT / 32;
constexpr int RT_MAX = 2048;       // rays per tile (<= 8 per thread)
constexpr int RPT = RT_MAX / TT;
constexpr int BIN_CAP = 8192;      // cells in the tile's bounding box that can be histogrammed (u16 counters)
constexpr int MAX_ITEM_RAYS = 32;  // rays per work item (heavier cells / blocks are split)
constexpr int WQ_CAP = 128;        // per-warp survivor ring (<= 31 pending + 64 new per ray)

struct Smem {
    uint4* ray_s;        // [RT]  sorted by cell: (sx2, sy2, sz2 duplicated halves, local ray id)
    uint32_t* res;       // [RT]  best key per local ray id
    uint2* items;        // [RT]  (cell, start | count << 16)
    uint32_t* bins;      // [BIN_CAP / 2]  u16 counters, then exclusive offsets
    uint2* wq;           // [NW][WQ_CAP]  per-warp ring of candidates that survived the pre-filter: (pos << 16 | slot, triangle)
    uint32_t* far;       // [RT / 32]  rays holding a hit beyond the 11.0 miss sentinel (resolved literally in the epilogue)
};

// Literal evaluation of up to 32 queued (ray, candidate) pairs, one per lane (ray_casting.py:34-59).
// Queue entry: B == 1: (pos << 16 | slot, triangle id);  B > 1: (pos << 16, absolute entry of the block list) -- the
// triangle id and the slot it holds in the ray's own cell are looked up here, where 32 lanes overlap the loads;
// a candidate that is not in the ray's cell list (slot 0xFF) is dropped.
template <int B>
__device__ __forceinline__ void drain32(const Smem& sm, const uint2* wq, uint32_t head, uint32_t n, int lane, const TriRec* recs,
                                        const int32_t* blk_ids, const uint4* blk_slots, H3 d) {
    if ((uint32_t)lane < n) {
        const uint2 e = wq[(head + lane) & (WQ_CAP - 1)];
        const uint4 rs = sm.ray_s[e.x >> 16];
        uint32_t slot = e.x & 0xffffu, id = e.y;
        if (B > 1) {
            id = (uint32_t)__ldg(blk_ids + e.y);
            slot = __ldg(reinterpret_cast<const unsigned char*>(blk_slots + e.y) + (rs.w >> 16));
            if (slot == 0xffu) return;
        }
        H3 a, b, c, nn;
        unpack_rec(recs + id, a, b, c, nn);
        const H3 s = {h_from_bits(rs.x & 0xffff), h_from_bits(rs.y & 0xffff), h_from_bits(rs.z & 0xffff)};
        const __half k = pair_test(s, d, a, b, c, nn);
        const uint32_t key = make_key(h_bits(k), slot);
        const uint32_t p = rs.w & 0xffffu;
        if ((key >> 16) > ORD_MISS) atomicOr(&sm.far[p >> 5], 1u << (p & 31));      // k > 11: see epilogue
        else atomicMin(&sm.res[p], key);
    }
}

template <int B>
__device__ __forceinline__ void hm_tiled_body(const TiledParams& q, const int work, const int sub, const int nsub) {
    extern __shared__ uint4 smem_raw[];
    __shared__ int s_box[4];          // min cx, min cy, max cx, max cy
    __shared__ uint32_t s_warp[NW];
    __shared__ int s_nitems, s_next;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t n = work / q.tiles;
    const int tile = work % q.tiles;
    // work-list mode cuts a tile into nsub slices (one CTA each): the few listed envs then finish in a fraction of the time
    const int tile_np = min(q.tile_size, q.P - tile * q.tile_size);
    const int slice = (tile_np + nsub - 1) / nsub;
    const int p0 = tile * q.tile_size + sub * slice;
    const int np = min(slice, tile_np - sub * slice);
    if (np <= 0) return;
    const int RT = q.tile_size;

    Smem sm;
    sm.ray_s = smem_raw;
    sm.res = reinterpret_cast<uint32_t*>(sm.ray_s + RT);
    sm.items = reinterpret_cast<uint2*>(sm.res + ((RT + 3) & ~3));
    sm.bins = reinterpret_cast<uint32_t*>(sm.items + ((RT + 1) & ~1));
    sm.wq = reinterpret_cast<uint2*>(sm.bins + BIN_CAP / 2);
    sm.far = reinterpret_cast<uint32_t*>(sm.wq + NW * WQ_CAP);

    // ---- phase 0: clear histogram, per-env constants
    for (int i = tid; i < BIN_CAP / 8; i += TT) reinterpret_cast<uint4*>(sm.bins)[i] = make_uint4(0, 0, 0, 0);
    for (int i = tid; i < (RT + 31) / 32; i += TT) sm.far[i] = 0u;
    if (tid == 0) {
        s_box[0] = s_box[1] = 0x7fffffff;
        s_box[2] = s_box[3] = -1;
        s_next = NW;
    }
    const Trig tr = make_trig(q.euler, q.trig, n);
    const double tx = (double)q.pos[n * 3 + 0], ty = (double)q.pos[n * 3 + 1], tz = (double)q.pos[n * 3 + 2];
    const H3 d = env_dir16(tr, tx, ty, tz);
    const __half2 dx2 = __half2half2(d.x), dy2 = __half2half2(d.y), dz2 = __half2half2(d.z);
    __syncthreads();

    // ---- phase 1: sources + cells of this thread's rays (kept in registers across the sort)
    uint32_t r_sxy[RPT], r_sz[RPT];
    int r_cell[RPT];                // block (cell when B == 1) x << 16 | y   (G <= 65535 checked on the host)
    int mnx = 0x7fffffff, mny = 0x7fffffff, mxx = -1, mxy = -1;
#pragma unroll
    for (int i = 0; i < RPT; ++i) {
        const int p = tid + i * TT;
        r_cell[i] = -1;
        if (p < np) {
            const double* pp = q.pattern + (int64_t)(p0 + p) * 3;
            double xo, yo, zo;
            body_transform<double>(pp[0], pp[1], pp[2], tr, tx, ty, tz, xo, yo, zo);
            const __half hx = h_from_double(xo), hy = h_from_double(yo), hz = h_from_double(zo);
            r_sxy[i] = (uint32_t)h_bits(hx) | ((uint32_t)h_bits(hy) << 16);
            const int2 c = ray_cell(hx, hy, q.shift_x, q.shift_y, q.res, q.inv_res, q.G0, q.G1, q.sem);
            int cx = c.x, cy = c.y;
            uint32_t sub = 0;
            if (B > 1) {
                const int bx = cx / B, by = cy / B;
                sub = (uint32_t)((cx - bx * B) * B + (cy - by * B));
                cx = bx; cy = by;
            }
            r_sz[i] = (uint32_t)h_bits(hz) | (sub << 16);
            r_cell[i] = (cx << 16) | cy;
            mnx = min(mnx, cx); mxx = max(mxx, cx); mny = min(mny, cy); mxy = max(mxy, cy);
        }
    }
    mnx = __reduce_min_sync(0xffffffffu, mnx); mny = __reduce_min_sync(0xffffffffu, mny);
    mxx = __reduce_max_sync(0xffffffffu, mxx); mxy = __reduce_max_sync(0xffffffffu, mxy);
    if (lane == 0) {
        atomicMin(&s_box[0], mnx); atomicMin(&s_box[1], mny);
        atomicMax(&s_box[2], mxx); atomicMax(&s_box[3], mxy);
    }
    __syncthreads();
    const int bx0 = s_box[0], by0 = s_box[1];
    const int BW = s_box[2] - bx0 + 1, BH = s_box[3] - by0 + 1;
    const bool grouped = (int64_t)BW * BH <= BIN_CAP;

    int nitems;
    if (grouped) {
        // ---- phase 2: counting sort by cell
        uint32_t r_rank[RPT];
#pragma unroll
        for (int i = 0; i < RPT; ++i) {
            if (r_cell[i] >= 0) {
                const int bin = ((r_cell[i] >> 16) - bx0) * BH + ((r_cell[i] & 0xffff) - by0);
                const uint32_t old = atomicAdd(&sm.bins[bin >> 1], 1u << ((bin & 1) * 16));
                r_rank[i] = (old >> ((bin & 1) * 16)) & 0xffffu;
            }
        }
        __syncthreads();
        // exclusive scan over bins; thread t owns words t, t + TT, ...  (order of cells is irrelevant);
        // packed accumulator: rays in the low 16 bits, items in the high 16 bits
        const int nwords = (BW * BH + 1) >> 1;
        uint32_t tot = 0;
        for (int w = tid; w < nwords; w += TT) {
            const uint32_t v = sm.bins[w];
            const uint32_t a = v & 0xffffu, b = v >> 16;
            tot += (a + b) + (((a + MAX_ITEM_RAYS - 1) / MAX_ITEM_RAYS + (b + MAX_ITEM_RAYS - 1) / MAX_ITEM_RAYS) << 16);
        }
        uint32_t inc = tot;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t v = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += v;
        }
        if (lane == 31) s_warp[warp] = inc;
        __syncthreads();
        uint32_t base = 0, total = 0;
#pragma unroll
        for (int w = 0; w < NW; ++w) {
            const uint32_t v = s_warp[w];
            if (w < warp) base += v;
            total += v;
        }
        uint32_t run = base + inc - tot;
        for (int w = tid; w < nwords; w += TT) {
            const uint32_t v = sm.bins[w];
            uint32_t off[2];
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const uint32_t cnt = h ? (v >> 16) : (v & 0xffffu);
                off[h] = run & 0xffffu;
                if (cnt) {
                    const int bin = 2 * w + h;
                    const int cx = bx0 + bin / BH, cy = by0 + bin % BH;
                    const uint32_t cell = (uint32_t)cx * (uint32_t)(B > 1 ? q.nBy : q.G1) + (uint32_t)cy;
                    uint32_t it = run >> 16, start = run & 0xffffu;
                    for (uint32_t done = 0; done < cnt; done += MAX_ITEM_RAYS, ++it)
                        sm.items[it] = make_uint2(cell, (start + done) | (min(cnt - done, (uint32_t)MAX_ITEM_RAYS) << 16));
                    run += cnt + (((cnt + MAX_ITEM_RAYS - 1) / MAX_ITEM_RAYS) << 16);
                }
            }
            sm.bins[w] = off[0] | (off[1] << 16);
        }
        nitems = (int)(total >> 16);
        __syncthreads();
        // scatter into cell order
#pragma unroll
        for (int i = 0; i < RPT; ++i) {
            if (r_cell[i] >= 0) {
                const int p = tid + i * TT;
                const int bin = ((r_cell[i] >> 16) - bx0) * BH + ((r_cell[i] & 0xffff) - by0);
                const uint32_t posn = ((sm.bins[bin >> 1] >> ((bin & 1) * 16)) & 0xffffu) + r_rank[i];
                sm.ray_s[posn] = make_uint4(__byte_perm(r_sxy[i], 0, 0x1010), __byte_perm(r_sxy[i], 0, 0x3232),
                                            __byte_perm(r_sz[i], 0, 0x1010), (uint32_t)p | (r_sz[i] & 0xffff0000u));
                sm.res[p] = KEY_INIT;
            }
        }
    } else {
        // bounding box too large to histogram (rays spread over more than BIN_CAP cells): every ray is its own item
#pragma unroll
        for (int i = 0; i < RPT; ++i) {
            if (r_cell[i] >= 0) {
                const int p = tid + i * TT;
                const uint32_t cell = (uint32_t)(r_cell[i] >> 16) * (uint32_t)(B > 1 ? q.nBy : q.G1) + (uint32_t)(r_cell[i] & 0xffff);
                sm.items[p] = make_uint2(cell, (uint32_t)p | (1u << 16));
                sm.ray_s[p] = make_uint4(__byte_perm(r_sxy[i], 0, 0x1010), __byte_perm(r_sxy[i], 0, 0x3232),
                                         __byte_perm(r_sz[i], 0, 0x1010), (uint32_t)p | (r_sz[i] & 0xffff0000u));
                sm.res[p] = KEY_INIT;
            }
        }
        nitems = np;
    }
    __syncthreads();

    // ---- phase 3: warps pull items; lanes own candidate pairs
    const H3 dlit = {__low2half(dx2), __low2half(dy2), __low2half(dz2)};
    uint2* wq = sm.wq + warp * WQ_CAP;
    uint32_t q_head = 0, q_tail = 0;          // warp-uniform
    const uint32_t lt_mask = (1u << lane) - 1u;
    const uint32_t ray_s_addr = (uint32_t)__cvta_generic_to_shared(sm.ray_s);
    // candidate list of an item: the cell's row of the index (B == 1) or the block's union list
    auto list_of = [&](uint32_t cell, const int32_t*& ids, uint32_t& o0) -> int {
        if (B == 1) {
            ids = q.index + (int64_t)cell * q.Ks;
            o0 = 0;
            return q.K;
        }
        o0 = __ldg(q.blk_off + cell);
        const uint32_t o1 = __ldg(q.blk_off + cell + 1);
        ids = q.blk_ids + o0;
        return (int)(o1 - o0);
    };
    // survivors of one ray -> queue (warp-uniform control flow); returns with fewer than 32 pending
    auto enqueue = [&](uint32_t f, int pos, int j0, int2 ids, uint32_t o0) {
        const bool m0 = (f & 0xffffu) != 0u, m1 = (f >> 16) != 0u;
        const uint32_t b0m = __ballot_sync(0xffffffffu, m0), b1m = __ballot_sync(0xffffffffu, m1);
        const uint32_t x = (uint32_t)pos << 16;
        if (m0) wq[(q_tail + __popc(b0m & lt_mask)) & (WQ_CAP - 1)] = B == 1 ? make_uint2(x | (uint32_t)j0, (uint32_t)ids.x) : make_uint2(x, o0 + (uint32_t)j0);
        q_tail += __popc(b0m);
        if (m1) wq[(q_tail + __popc(b1m & lt_mask)) & (WQ_CAP - 1)] = B == 1 ? make_uint2(x | (uint32_t)(j0 + 1), (uint32_t)ids.y) : make_uint2(x, o0 + (uint32_t)j0 + 1u);
        q_tail += __popc(b1m);
        if (q_tail - q_head >= 32u) {
            __syncwarp();
            do {
                drain32<B>(sm, wq, q_head, 32u, lane, q.recs, q.blk_ids, q.blk_slots, dlit);
                q_head += 32u;
            } while (q_tail - q_head >= 32u);
            __syncwarp();
        }
    };
    int item = warp;
    while (item < nitems) {
        int next = 0;
        if (lane == 0) next = atomicAdd(&s_next, 1);
        next = __shfl_sync(0xffffffffu, next, 0);
        const uint2 it = sm.items[item];
        const int32_t* ids_base;
        uint32_t o0;
        const int U = list_of(it.x, ids_base, o0);
        const int2* rowl = reinterpret_cast<const int2*>(ids_base) + lane;      // this lane's id pairs (lists have even length)
        if (next < nitems) {
            // pull the next item's candidate ids towards L2 while this one is being processed
            const int32_t* nids;
            uint32_t no0;
            const int nU = list_of(sm.items[next].x, nids, no0);
            if (lane * 32 < nU) asm volatile("prefetch.global.L2 [%0];" ::"l"(nids + lane * 32));
        }
        const int cnt = it.y >> 16;
        const uint32_t ray0 = ray_s_addr + (it.y & 0xffffu) * 16u;
        int2 ids = (2 * lane < U) ? __ldg(rowl) : make_int2(0, 0);
        for (int c0 = 0; c0 < U; c0 += 64) {
            const int j0 = c0 + 2 * lane;
            const int2 ids_next = (j0 + 64 < U) ? __ldg(rowl + (c0 >> 1) + 32) : make_int2(0, 0);   // in flight during the ray loop
            uint4 a0, a1w, b0, b1w;
            ldg_rec32(q.recs + ids.x, a0, a1w);
            ldg_rec32(q.recs + ids.y, b0, b1w);
            const uint2 a1 = make_uint2(a1w.x, a1w.y), b1 = make_uint2(b1w.x, b1w.y);
            const Tri2 t = pack_tri2(a0, a1, b0, b1);
            const Cand2 cd = make_cand2(t, dx2, dy2, dz2, j0 < U, j0 + 1 < U);
            uint32_t ra = ray0;
            int r = 0;
            for (; r + 2 <= cnt; r += 2, ra += 32u) {
                uint32_t x0, y0, z0, w0, x1, y1, z1, w1;
                asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(x0), "=r"(y0), "=r"(z0), "=r"(w0) : "r"(ra));
                asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4+16];" : "=r"(x1), "=r"(y1), "=r"(z1), "=r"(w1) : "r"(ra));
                const uint32_t f0 = prefilter2(u2h(x0), u2h(y0), u2h(z0), dx2, dy2, dz2, t, cd);
                const uint32_t f1 = prefilter2(u2h(x1), u2h(y1), u2h(z1), dx2, dy2, dz2, t, cd);
                if (__any_sync(0xffffffffu, (f0 | f1) != 0u)) {      // about 1 candidate in 100 survives
                    const int pos = (int)((ra - ray_s_addr) >> 4);
                    enqueue(f0, pos, j0, ids, o0);
                    enqueue(f1, pos + 1, j0, ids, o0);
                }
            }
            if (r < cnt) {
                uint32_t x0, y0, z0, w0;
                asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(x0), "=r"(y0), "=r"(z0), "=r"(w0) : "r"(ra));
                const uint32_t f0 = prefilter2(u2h(x0), u2h(y0), u2h(z0), dx2, dy2, dz2, t, cd);
                if (__any_sync(0xffffffffu, f0 != 0u)) enqueue(f0, (int)((ra - ray_s_addr) >> 4), j0, ids, o0);
            }
            ids = ids_next;
        }
        item = next;
    }
    __syncwarp();
    if (q_tail != q_head) drain32<B>(sm, wq, q_head, q_tail - q_head, lane, q.recs, q.blk_ids, q.blk_slots, dlit);
    __syncthreads();

    // ---- phase 4: epilogue in ray order
    epilogue(q, n, p0, np, tr, tx, ty, tz, dx2, dy2, dz2, sm.res, sm.far, tid, TT);
}

// One CTA per (env, tile); in work-list mode (the shadow kernel's fall-back list) CTAs loop over the listed items.
template <int B>
__global__ void __launch_bounds__(TT, 3) hm_tiled_kernel(const TiledParams q) {
    if (q.work_list) {
        const int cnt = *q.work_count;
        for (int w = blockIdx.x; w < cnt * q.work_slices; w += gridDim.x) {
            hm_tiled_body<B>(q, q.work_list[w / q.work_slices], w % q.work_slices, q.work_slices);
            __syncthreads();
        }
    } else {
        hm_tiled_body<B>(q, (int)blockIdx.x, 0, 1);
    }
}

size_t tiled_smem_bytes(int RT) {
    return (size_t)RT * 16 + (size_t)((RT + 3) & ~3) * 4 + (size_t)((RT + 1) & ~1) * 8 + (size_t)BIN_CAP * 2 +
           (size_t)NW * WQ_CAP * 8 + (size_t)((RT + 31) / 32) * 4;
}

}  // namespace

int fill_tiled_params(const rvb_terrain* t, int64_t P, int64_t N, int variant, rc::TiledParams& q) {
    RVB_REQUIRE(N >= 0 && P > 0 && P <= 65535, "rvb_heightmap_raycast: need N >= 0, 0 < P <= 65535");
    if (N == 0) return RVB_OK;
    RVB_REQUIRE(t && q.pos && q.euler && q.pattern && q.dist, "rvb_heightmap_raycast: null pointer");
    RVB_REQUIRE(!q.obs || (q.col_a && q.col_b && q.obs_ld > 0), "rvb_heightmap_raycast: obs needs col_a, col_b, obs_ld");
    RVB_REQUIRE(!q.obs16 || (q.col_a && q.col_b && q.obs16_ld > 0 && q.obs16_col0 >= 0), "rvb_heightmap_raycast: obs_h16 needs col_a, col_b, obs_h16_ld");
    RVB_REQUIRE(variant >= 0 && variant <= 3, "rvb_heightmap_raycast: variant must be 0, 1, 2 or 3");
    RVB_REQUIRE(!q.obs16 || variant != 1, "rvb_heightmap_raycast: the per-pair cross-check kernel (variant 1) has no packed output");
    RVB_REQUIRE(variant != 2 || t->index != nullptr, "rvb_heightmap_raycast: variant 2 reads the index the layer released (rvb_terrain_release_index)");
    if (variant == 1) {
        RVB_REQUIRE(t->index != nullptr, "rvb_heightmap_raycast: variant 1 reads the index the layer released (rvb_terrain_release_index)");
        RVB_REQUIRE(N <= 65535, "rvb_heightmap_raycast: variant 1 handles at most 65535 envs per call");
    } else {
        RVB_REQUIRE(t->G0 <= 32767 && t->G1 <= 65535, "heightmap ray-cast: grid larger than 32767 x 65535 cells");
        RVB_REQUIRE(t->K <= 16383, "heightmap ray-cast: K > 16383");
        RVB_REQUIRE(t->G0 * t->G1 < ((int64_t)1 << 32), "heightmap ray-cast: more than 2^32 cells");
    }
    q.index = t->index; q.recs = t->recs; q.s1 = t->s1recs;
    q.blk_off = t->blk_off; q.blk_ids = t->blk_ids; q.blk_slots = t->blk_slots; q.nBy = t->nBy;
    q.sb_off = t->sb_off; q.sb_ids = t->sb_ids; q.sb_slot9 = t->sb_slot9; q.sb_chunk = t->sb_chunk; q.nSBy = t->nSBy;
    q.G0 = (int)t->G0; q.G1 = (int)t->G1; q.K = (int)t->K; q.Ks = (int)t->Ks;
    q.res = t->res; q.inv_res = 1.0f / t->res; q.shift_x = t->shift_x; q.shift_y = t->shift_y; q.sem = t->sem;
    q.P = (int)P;
    q.tiles = (int)ceil_div(P, RT_MAX);
    q.tile_size = (int)ceil_div(P, q.tiles);
    RVB_REQUIRE(N * q.tiles < ((int64_t)1 << 31), "heightmap ray-cast: too many (env, tile) blocks for one launch");
    return RVB_OK;
}

int launch_tiled(const rc::TiledParams& q, bool blocks, int64_t grid, cudaStream_t st) {
    static thread_local int configured_device = -1;
    const int rc_ = set_smem_limits(configured_device, {{(const void*)hm_tiled_kernel<1>, tiled_smem_bytes(RT_MAX)},
                                                        {(const void*)hm_tiled_kernel<RVB_BLK>, tiled_smem_bytes(RT_MAX)}});
    if (rc_ != RVB_OK) return rc_;
    const size_t smem = tiled_smem_bytes(q.tile_size);
    if (blocks) hm_tiled_kernel<RVB_BLK><<<(unsigned)grid, TT, smem, st>>>(q);
    else hm_tiled_kernel<1><<<(unsigned)grid, TT, smem, st>>>(q);
    RVB_LAUNCH_CHECK();
    return RVB_OK;
}
