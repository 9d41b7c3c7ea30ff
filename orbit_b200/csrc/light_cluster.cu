// light_cluster.cu — clustered light assignment (sm_100a).
//
// Stands in for compute_clusters (src/passes/cluster.rs:368-591) and its three compute shaders:
//   mark_active.comp:27-57               -> mark_active_kernel
//   active_cluster_compaction.comp:17-44 -> compact_clusters_kernel
//   light_culling.comp:34-151            -> light_view_kernel + light_culling_kernel
//
// B200 design:
//   * mark_active: 2-3 global atomics per PIXEL in the reference; here lanes of a warp that hit the same
//     cluster are merged with a ballot loop over the distinct keys + full-mask redux (max / or), so one lane per
//     distinct cluster issues the atomics.
//     atomicMax / atomicOr are order-independent, so the result is deterministic; an L2 read first skips the
//     atomic when the stored value already covers ours (same-address atomics serialise, reads do not).
//   * compaction: ballot + CTA scan + decoupled look-back instead of atomicAdd: cluster ids come out ascending.
//   * light culling: the reference recomputes view*light_position for every (cluster, light) pair and walks
//     the light list twice; here light view-space spheres are computed once (16 B each, L2-resident), a 1024-thread
//     CTA owns one active cluster, each of its 32 warps tests a contiguous stripe of the lights 32 at a time and
//     ballot-compacts hits in ascending order into shared memory; stripes are concatenated in order up to the
//     reference's cap of 256, and per-cluster ranges are packed in compacted-list order by a look-back scan
//     instead of atomicAdd.
#include "params.cuh"

namespace orbit {


// ---------------------------------------------------------------------------------------------------------
// Merge, inside one warp, the lanes that hit the same key, with one REDUX per distinct key instead of match.any +
// partial-mask redux (ncu: the partial-mask `__reduce_or_sync` is a ~32-instruction software loop and was the top
// line of this kernel). Lanes with key == kNoKey take no part. fn(leader_lane_is_me, same_mask) is called by the
// lanes of one key at a time.
constexpr uint32_t kNoKey = 0xFFFFFFFFu;

// kImage: depth from p.depth_tex (a depth image, orbit_light_cluster_image) instead of the linear buffer p.depth
template <bool kImage>
__device__ __forceinline__ void mark_active_body(const ClusterParams& p) {
    const OrbitClusterCullInfo& ci = p.info;
    const uint32_t W = ci.screen_size[0], H = ci.screen_size[1];
    const uint32_t cx = ci.cluster_count[0], cy = ci.cluster_count[1], cz = ci.cluster_count[2];
    const uint32_t tile_px = ci.tile_size_px;
    // a warp covers 32 consecutive pixels of kRows consecutive rows per step (kRows independent loads in flight)
    constexpr uint32_t kRows = 4u;
    const uint32_t warps_per_row = (W + 31u) / 32u;
    const uint32_t row_groups = (H + kRows - 1u) / kRows;
    const uint32_t total_warps = warps_per_row * row_groups;   // < 2^32: screen sizes are bounded by the API
    const uint32_t lane = threadIdx.x & 31u;
    for (uint32_t wi = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); wi < total_warps; wi += gridDim.x * (blockDim.x >> 5)) {
        const uint32_t row_group = wi / warps_per_row;           // 32-bit: a 64-bit division here cost ~100 instructions per step
        const uint32_t y0 = row_group * kRows;
        const uint32_t x0 = (wi - row_group * warps_per_row) * 32u;
        const uint32_t x = x0 + lane;
        float dv[kRows];
#pragma unroll
        for (uint32_t k = 0; k < kRows; ++k) {
            if constexpr (kImage) dv[k] = (x < W && y0 + k < H) ? depth_texel(p.depth_tex, (int)x, (int)(y0 + k)) : 0.0f;
            else dv[k] = (x < W && y0 + k < H) ? __ldg(p.depth + (size_t)(y0 + k) * W + x) : 0.0f;
        }
        // tile column of this lane: one (warp-uniform) integer division per step instead of one per pixel
        uint32_t tx = x0 / tile_px;
        {
            uint32_t t = x0 - tx * tile_px + lane;
            if (tile_px >= 8u) { while (t >= tile_px) { t -= tile_px; ++tx; } } else { tx += t / tile_px; }
        }
        const uint32_t ty0 = y0 / tile_px;
        uint32_t ry = y0 - ty0 * tile_px;   // row offset inside the tile row, advanced per k
        uint32_t ty = ty0;
        // ---- per-lane math for the kRows pixels of this lane's column (no warp-level operations yet)
        uint32_t cl[kRows], tl[kRows], mk[kRows], bn[kRows], bx[kRows];
#pragma unroll
        for (uint32_t k = 0; k < kRows; ++k) {
            const uint32_t y = y0 + k;
            cl[k] = kNoKey; tl[k] = kNoKey; mk[k] = 0u; bn[k] = 0u; bx[k] = 0u;
            if (x < W && y < H) {
                const float d = dv[k];
                // sky pixels (d == +0, the clear value of the reverse-Z buffer) would send the IEEE division into its
                // ~50-instruction slow path for the whole warp; z_near / +0 is +inf exactly when z_near > 0
                const float z = (__float_as_uint(d) == 0u && ci.z_near > 0.0f) ? __uint_as_float(0x7F800000u) : fdiv(ci.z_near, d);
                const uint32_t slice = f2u(fma_(orbit_log2f(z), p.z_scale, p.z_bias));
                mk[k] = shl1(slice);
                if (mk[k] != 0u) tl[k] = tx + ty * cx;
                if (slice < cz) {
                    cl[k] = tx + ty * cx + slice * cx * cy;
                    bn[k] = __float_as_uint(sub(1.0f, d));
                    bx[k] = __float_as_uint(d);
                }
            }
            if (++ry == tile_px) { ry = 0u; ++ty; }
        }
        // ---- lane-local merge: vertically adjacent pixels mostly fall into the same cluster / tile, so rows 1..3 are
        //      folded into the first row with the same key and the warp-level merge below usually runs once, not kRows times
#pragma unroll
        for (uint32_t k = 1; k < kRows; ++k) {
#pragma unroll
            for (uint32_t j = 0; j < k; ++j) {
                if (cl[k] != kNoKey && cl[k] == cl[j]) { bn[j] = max(bn[j], bn[k]); bx[j] = max(bx[j], bx[k]); cl[k] = kNoKey; }
                if (tl[k] != kNoKey && tl[k] == tl[j]) { mk[j] |= mk[k]; tl[k] = kNoKey; }
            }
        }
#pragma unroll
        for (uint32_t k = 0; k < kRows; ++k) {
            // ---- cluster depth bounds: one pair of atomics per distinct cluster of the warp
            uint32_t todo = __ballot_sync(0xFFFFFFFFu, cl[k] != kNoKey);
            while (todo) {
                const uint32_t key = __shfl_sync(0xFFFFFFFFu, cl[k], __ffs((int)todo) - 1);
                const bool mine = cl[k] == key;
                const uint32_t same = __ballot_sync(0xFFFFFFFFu, mine);
                const uint32_t mn = __reduce_max_sync(0xFFFFFFFFu, mine ? bn[k] : 0u);
                const uint32_t mx = __reduce_max_sync(0xFFFFFFFFu, mine ? bx[k] : 0u);
                if (lane == (uint32_t)(__ffs((int)same) - 1)) {
                    // values only grow: a (possibly stale) read that is already >= ours makes the atomic a no-op
                    uint32_t* b = p.depth_bounds + 2u * (size_t)key;
                    if (__ldcg(b) < mn) atomicMax(b, mn);
                    if (__ldcg(b + 1) < mx) atomicMax(b + 1, mx);
                }
                todo &= ~same;
            }
            // ---- tile slice masks: one atomicOr per distinct tile of the warp
            todo = __ballot_sync(0xFFFFFFFFu, tl[k] != kNoKey);
            while (todo) {
                const uint32_t key = __shfl_sync(0xFFFFFFFFu, tl[k], __ffs((int)todo) - 1);
                const bool mine = tl[k] == key;
                const uint32_t same = __ballot_sync(0xFFFFFFFFu, mine);
                const uint32_t orm = __reduce_or_sync(0xFFFFFFFFu, mine ? mk[k] : 0u);
                if (lane == (uint32_t)(__ffs((int)same) - 1) && (__ldcg(p.tile_masks + key) & orm) != orm) atomicOr(p.tile_masks + key, orm);
                todo &= ~same;
            }
        }
    }
}

__global__ void __launch_bounds__(256) mark_active_kernel(const __grid_constant__ ClusterParams p) { mark_active_body<false>(p); }
__global__ void __launch_bounds__(256) mark_active_image_kernel(const __grid_constant__ ClusterParams p) { mark_active_body<true>(p); }

struct Aabb3 { float lo[3], hi[3]; };

__device__ __forceinline__ void unproject(const OrbitClusterCullInfo& ci, float px, float py, float* out) {
    const float tx = fdiv(px, (float)ci.screen_size[0]), ty = fdiv(py, (float)ci.screen_size[1]);
    const float clx = sub(mul(tx, 2.0f), 1.0f), cly = sub(mul(sub(1.0f, ty), 2.0f), 1.0f);
    const float* m = &ci.screen_to_view_matrix.m[0][0];
    const float vx = add(add(add(mul(m[0], clx), mul(m[4], cly)), mul(m[8], 1.0f)), mul(m[12], 1.0f));
    const float vy = add(add(add(mul(m[1], clx), mul(m[5], cly)), mul(m[9], 1.0f)), mul(m[13], 1.0f));
    const float vz = add(add(add(mul(m[2], clx), mul(m[6], cly)), mul(m[10], 1.0f)), mul(m[14], 1.0f));
    const float vw = add(add(add(mul(m[3], clx), mul(m[7], cly)), mul(m[11], 1.0f)), mul(m[15], 1.0f));
    out[0] = fdiv(vx, vw); out[1] = fdiv(vy, vw); out[2] = fdiv(vz, vw);
}

__device__ __forceinline__ void z_plane_point(const float* v, float zd, float* out) {
    const float dn = add(add(mul(0.0f, v[0]), mul(0.0f, v[1])), mul(-1.0f, v[2]));  // dot((0,0,-1), v)
    const float t = fdiv(zd, dn);
    out[0] = mul(v[0], t); out[1] = mul(v[1], t); out[2] = mul(v[2], t);
}

__device__ __forceinline__ Aabb3 cluster_volume(const ClusterParams& p, uint32_t idx) {
    const OrbitClusterCullInfo& ci = p.info;
    const uint32_t cx = ci.cluster_count[0], cy = ci.cluster_count[1];
    const uint32_t z = idx / (cx * cy);
    const uint32_t rem = idx - z * cx * cy;
    const uint32_t y = rem / cx, x = rem - y * cx;
    const float minx = (float)(x * ci.tile_size_px), miny = (float)(y * ci.tile_size_px);
    const float maxx = fminf(add(minx, (float)ci.tile_size_px), (float)ci.screen_size[0]);
    const float maxy = fminf(add(miny, (float)ci.tile_size_px), (float)ci.screen_size[1]);
    float vmin[3], vmax[3];
    unproject(ci, minx, miny, vmin);
    unproject(ci, maxx, maxy, vmax);
    const float min_d = sub(1.0f, __uint_as_float(__ldcg(p.depth_bounds + 2u * (size_t)idx)));
    const float max_d = __uint_as_float(__ldcg(p.depth_bounds + 2u * (size_t)idx + 1u));
    const float cnear = fdiv(ci.z_near, max_d), cfar = fdiv(ci.z_near, min_d);
    float p0[3], p1[3], p2[3], p3[3];
    z_plane_point(vmin, cnear, p0); z_plane_point(vmin, cfar, p1);
    z_plane_point(vmax, cnear, p2); z_plane_point(vmax, cfar, p3);
    Aabb3 a;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        a.lo[k] = fminf(fminf(p0[k], p1[k]), fminf(p2[k], p3[k]));
        a.hi[k] = fmaxf(fmaxf(p0[k], p1[k]), fmaxf(p2[k], p3[k]));
    }
    return a;
}

// The offset / count grid as a 3-D R32G32_UINT array (orbit_light_cluster_image_grid): each storing kernel has a kGrid twin
// that writes texel (x, y, z) of p.offset_count_surf where the linear form writes words 2 idx, 2 idx + 1. An array cannot be
// cleared with cudaMemsetAsync, so the compaction kernel's twin writes (0, 0) to every inactive cluster and the list kernels
// write every active one: each call writes every texel once.
__device__ __forceinline__ void grid_store(const ClusterParams& p, uint32_t idx, uint32_t off, uint32_t count) {
    const uint32_t cx = p.info.cluster_count[0], cy = p.info.cluster_count[1];
    const uint32_t z = idx / (cx * cy), t = idx - z * cx * cy, y = t / cx, x = t - y * cx;
    surf3Dwrite(make_uint2(off, count), p.offset_count_surf, (int)(x * 8u), (int)y, (int)z, cudaBoundaryModeZero);
}

// ---------------------------------------------------------------------------------------------------------
template <bool kGrid>
__device__ __forceinline__ void compact_clusters_body(const ClusterParams& p) {
    __shared__ uint32_t s_warp[8];
    __shared__ uint32_t s_tile, s_base;
    const OrbitClusterCullInfo& ci = p.info;
    const uint32_t cx = ci.cluster_count[0], cy = ci.cluster_count[1], cz = ci.cluster_count[2];
    const uint32_t total = cx * cy * cz;
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    const unsigned int epoch = scan_epoch(p.scan);
    if (tid == 0) s_tile = atomicAdd(p.scan.ticket, 1u);
    __syncthreads();
    const uint32_t tile = s_tile;
    const uint32_t idx = tile * 256u + tid;
    bool active = false;
    if (idx < total && p.cluster_totals != nullptr) p.cluster_totals[idx] = 0u;   // hit totals of the light-parallel path (one per possible slot)
    if (idx < total) {
        const uint32_t z = idx / (cx * cy);
        const uint32_t t = idx - z * cx * cy;   // tile index = x + y*cx
        active = (__ldcg(p.tile_masks + t) & shl1(z)) != 0u;
    }
    const uint32_t bal = __ballot_sync(0xFFFFFFFFu, active);
    if (lane == 0u) s_warp[warp] = __popc(bal);
    __syncthreads();
    uint32_t warp_base = 0u, tile_total = 0u;
#pragma unroll
    for (int w = 0; w < 8; ++w) { const uint32_t v = s_warp[w]; if ((uint32_t)w < warp) warp_base += v; tile_total += v; }
    if (warp == 0u) {
        const uint32_t base = lookback_exclusive(p.scan, epoch, tile, tile_total);
        if (lane == 0u) {
            s_base = base;
            if (tile == gridDim.x - 1u) {
                const uint32_t n = base + tile_total;
                p.unique_clusters[0] = (n + 255u) / 256u;   // div_ceil(cluster_count, 256)
                p.unique_clusters[1] = 1u;
                p.unique_clusters[2] = 1u;
                p.unique_clusters[3] = n;
            }
        }
    }
    __syncthreads();
    if (active) {
        const uint32_t slot = s_base + warp_base + __popc(bal & ((1u << lane) - 1u));
        p.unique_clusters[4u + slot] = idx;
        // the light-parallel culling path reads every active cluster's view-space box from many CTAs: computed once, here
        // (ten IEEE divisions per cluster, light_culling.comp:68-119), 32 bytes per compacted-list slot
        if (p.cluster_boxes != nullptr) {
            const Aabb3 b = cluster_volume(p, idx);
            p.cluster_boxes[2u * (size_t)slot] = make_float4(b.lo[0], b.lo[1], b.lo[2], 0.0f);
            p.cluster_boxes[2u * (size_t)slot + 1u] = make_float4(b.hi[0], b.hi[1], b.hi[2], 0.0f);
        }
    }
    if constexpr (kGrid) {
        if (idx < total && !active) grid_store(p, idx, 0u, 0u);
    }
    if (tid == 0) scan_cta_exit(p.scan, epoch);
}

__global__ void __launch_bounds__(256) compact_clusters_kernel(const __grid_constant__ ClusterParams p) { compact_clusters_body<false>(p); }
__global__ void __launch_bounds__(256) compact_clusters_grid_kernel(const __grid_constant__ ClusterParams p) { compact_clusters_body<true>(p); }

// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) light_view_kernel(const __grid_constant__ ClusterParams p) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= p.info.global_light_count) return;
    const uint8_t* l = p.lights + (size_t)j * 64u;
    const uint32_t type = __ldg(reinterpret_cast<const uint32_t*>(l));
    const float4 pos = __ldg(reinterpret_cast<const float4*>(l + 32));      // position xyz, inner_radius
    const float radius = __ldg(reinterpret_cast<const float*>(l + 60));
    const float* m = &p.info.world_to_view_matrix.m[0][0];
    float4 o;
    o.x = add(add(add(mul(m[0], pos.x), mul(m[4], pos.y)), mul(m[8], pos.z)), mul(m[12], 1.0f));
    o.y = add(add(add(mul(m[1], pos.x), mul(m[5], pos.y)), mul(m[9], pos.z)), mul(m[13], 1.0f));
    o.z = add(add(add(mul(m[2], pos.x), mul(m[6], pos.y)), mul(m[10], pos.z)), mul(m[14], 1.0f));
    o.w = (type == ORBIT_LIGHT_POINT) ? radius : __uint_as_float(0x7F800000u);  // non-point lights always hit
    p.light_view[j] = o;
}

constexpr int kLcWarps = 32;

// One CTA of kLcWarps warps per active cluster (persistent over clusters through a ticket). The light list is cut
// into kLcWarps contiguous stripes, one per warp; a warp tests 32 lights per step and ballot-compacts its hits
// in ascending order into its own shared-memory list (at most 256 entries can ever be used). The stripes are then
// concatenated in warp order up to the reference's cap of 256, and the cluster's range in the global list comes
// from a look-back scan over clusters in compacted-list order. With few active clusters (typical: ~100 of 3456)
// this spreads each cluster's L tests over 1024 threads instead of one warp (measured 716 us -> see profiles/).
// The kernel is in light_culling_kernel.cuh, compiled twice: light_culling_kernel (linear offset / count buffer) and
// light_culling_grid_kernel (grid array, see grid_store).
#define ORBIT_LC_KERNEL light_culling_kernel
#define ORBIT_LC_GRID 0
#include "light_culling_kernel.cuh"
#undef ORBIT_LC_KERNEL
#undef ORBIT_LC_GRID
#define ORBIT_LC_KERNEL light_culling_grid_kernel
#define ORBIT_LC_GRID 1
#include "light_culling_kernel.cuh"
#undef ORBIT_LC_KERNEL
#undef ORBIT_LC_GRID

// ---------------------------------------------------------------------------------------------------------
// Light-parallel formulation of light_culling.comp:121-151 (the path taken whenever its bit matrix fits the scratch budget;
// the CTA-per-cluster kernel above remains for grids with ~10^6 clusters). The CTA-per-cluster kernel re-streams the whole
// light array once per active cluster and occupies one SM per cluster (C4: 99 clusters -> 99 of 148 SMs, 232 G tests/s).
// Here the work is cut the other way:
//   1. light_hits_kernel: a CTA owns 512 consecutive lights (two per thread, view-space sphere computed in registers —
//      no light_view pass) and a chunk of 32 active clusters whose view-space boxes sit in shared memory; every
//      (light, cluster) test is one broadcast shared-memory read of the box + ~17 FP32 instructions, a ballot per
//      (warp, cluster) yields 32 hit bits, and the CTA leaves a 16-word row per cluster in a bit matrix
//      [active cluster][light / 32] (coalesced 64-byte stores). Grid = light blocks x cluster chunks: every SM busy.
//   2. light_lists_kernel: a warp per active cluster reads its row of the matrix (2049 words at C4), counts, caps at 256
//      (the reference keeps the FIRST 256 hits in ascending light order: light_culling.comp:121-132), the clusters' ranges
//      are packed in compacted-list order by the look-back scan, and the warp expands its row's first 256 set bits into
//      ascending light indices. Same arithmetic per test as the kernel above, so the lists are bit-identical.
constexpr uint32_t kLhLightsPerCta = 512u, kLhClusterChunk = 32u, kLhWordsPerCta = kLhLightsPerCta / 32u;

// hits:   [active cluster][words_per_cluster]   one bit per light; words_per_cluster = 16 x light blocks (rows are 64-byte aligned)
// counts: [active cluster][light_blocks]        hits of the cluster among the 512 lights of one light block
// totals: [active cluster]                      hits of the cluster among all lights (atomic sums; zeroed by the compaction kernel)
//
// Most lights touch no active cluster at all (C4: 743 hits in 6.5 M tests), so the CTA first tests its 512 lights against the
// UNION of the chunk's 32 boxes — exact as a filter: per axis the distance to the union is <= the distance to a member, and
// rounding (subtract, max, fma accumulate in the same order) is monotonic, so acc(union) > r^2 implies acc(member) > r^2 —
// and only the lights that pass (compacted in ascending order) meet the 32 boxes: a warp takes one light, lane = cluster, the
// ballot is the light's hit mask over the chunk. Same arithmetic per test as the CTA-per-cluster kernel: identical lists.
__global__ void __launch_bounds__(256) light_hits_kernel(const __grid_constant__ ClusterParams p, uint32_t* __restrict__ hits,
                                                         uint32_t* __restrict__ counts, uint32_t words_per_cluster) {
    __shared__ float s_box[kLhClusterChunk][8];                  // lo xyz, hi xyz (padded to 32 bytes)
    __shared__ float s_union[8];
    __shared__ uint32_t s_out[kLhClusterChunk][kLhWordsPerCta];
    __shared__ float4 s_sphere[kLhLightsPerCta];                 // view-space centre, squared radius (-1: no such light)
    __shared__ uint32_t s_list[kLhLightsPerCta];                 // lights that pass the union test, ascending
    __shared__ uint32_t s_wcount[16], s_nlist;
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    const uint32_t nactive = __ldcg(p.unique_clusters + 3);
    if (blockIdx.y * kLhClusterChunk >= nactive) return;        // chunk rows beyond the active clusters: nothing to do, before any load
    const uint32_t L = p.info.global_light_count;
    const uint32_t light0 = blockIdx.x * kLhLightsPerCta;
    // this thread's two lights: light0 + tid and light0 + 256 + tid (bit matrix word = block * 16 + k * 8 + warp, bit = lane)
#pragma unroll
    for (int k = 0; k < 2; ++k) {
        const uint32_t j = light0 + (uint32_t)k * 256u + tid;
        float4 sp = make_float4(0.0f, 0.0f, 0.0f, -1.0f);
        if (j < L) {
            const uint8_t* l = p.lights + (size_t)j * 64u;
            const uint32_t type = __ldg(reinterpret_cast<const uint32_t*>(l));
            const float4 pos = __ldg(reinterpret_cast<const float4*>(l + 32));      // position xyz, inner_radius
            const float radius = __ldg(reinterpret_cast<const float*>(l + 60));
            const float* m = &p.info.world_to_view_matrix.m[0][0];
            sp.x = add(add(add(mul(m[0], pos.x), mul(m[4], pos.y)), mul(m[8], pos.z)), mul(m[12], 1.0f));
            sp.y = add(add(add(mul(m[1], pos.x), mul(m[5], pos.y)), mul(m[9], pos.z)), mul(m[13], 1.0f));
            sp.z = add(add(add(mul(m[2], pos.x), mul(m[6], pos.y)), mul(m[10], pos.z)), mul(m[14], 1.0f));
            const float w = (type == ORBIT_LIGHT_POINT) ? radius : __uint_as_float(0x7F800000u);   // non-point lights always hit
            sp.w = mul(w, w);
        }
        s_sphere[(uint32_t)k * 256u + tid] = sp;
    }
    // squared distance from a sphere centre to a box, per axis: v < lo adds (lo-v)^2, v > hi adds (v-hi)^2
    // (light_culling.comp:52-66); lo <= hi, so at most one applies and d is that term's base (or 0, and fma(0,0,acc) == acc)
    auto dist2 = [](const float4 sp, const float4 lo, const float4 hi) -> float {
        float acc = 0.0f;
        float d = fmaxf(fmaxf(sub(lo.x, sp.x), sub(sp.x, hi.x)), 0.0f); acc = fma_(d, d, acc);
        d = fmaxf(fmaxf(sub(lo.y, sp.y), sub(sp.y, hi.y)), 0.0f); acc = fma_(d, d, acc);
        d = fmaxf(fmaxf(sub(lo.z, sp.z), sub(sp.z, hi.z)), 0.0f); acc = fma_(d, d, acc);
        return acc;
    };
    for (uint32_t chunk0 = blockIdx.y * kLhClusterChunk; chunk0 < nactive; chunk0 += gridDim.y * kLhClusterChunk) {
        const uint32_t nc = min(kLhClusterChunk, nactive - chunk0);
        __syncthreads();                                         // previous chunk's boxes, rows and list are no longer read
        if (tid < 2u * nc) *reinterpret_cast<float4*>(&s_box[tid >> 1][(tid & 1u) * 4u]) = __ldcg(p.cluster_boxes + 2u * (size_t)chunk0 + tid);
        s_out[tid >> 4][tid & 15u] = 0u; s_out[16u + (tid >> 4)][tid & 15u] = 0u;
        __syncthreads();
        if (warp == 0u) {                                        // union of the chunk's boxes (lanes beyond nc: neutral)
            float lo[3], hi[3];
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                lo[a] = lane < nc ? s_box[lane][a] : __uint_as_float(0x7F800000u);
                hi[a] = lane < nc ? s_box[lane][4 + a] : __uint_as_float(0xFF800000u);
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    lo[a] = fminf(lo[a], __shfl_xor_sync(0xFFFFFFFFu, lo[a], o));
                    hi[a] = fmaxf(hi[a], __shfl_xor_sync(0xFFFFFFFFu, hi[a], o));
                }
            }
            if (lane == 0u) { s_union[0] = lo[0]; s_union[1] = lo[1]; s_union[2] = lo[2]; s_union[3] = 0.0f;
                              s_union[4] = hi[0]; s_union[5] = hi[1]; s_union[6] = hi[2]; s_union[7] = 0.0f; }
        }
        __syncthreads();
        // ---- lights that reach the union, in ascending order (thread's light k has local index k * 256 + tid)
        const float4 ulo = *reinterpret_cast<const float4*>(&s_union[0]), uhi = *reinterpret_cast<const float4*>(&s_union[4]);
        uint32_t bal[2];
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const float4 sp = s_sphere[(uint32_t)k * 256u + tid];
            bal[k] = __ballot_sync(0xFFFFFFFFu, sp.w >= 0.0f && dist2(sp, ulo, uhi) <= sp.w);
            if (lane == 0u) s_wcount[(uint32_t)k * 8u + warp] = (uint32_t)__popc(bal[k]);
        }
        __syncthreads();
        {
            uint32_t before[2] = {0u, 0u}, total = 0u;
#pragma unroll
            for (uint32_t w = 0; w < 16u; ++w) {
                const uint32_t v = s_wcount[w];
                if (w < warp) before[0] += v;
                if (w < 8u + warp) before[1] += v;
                total += v;
            }
#pragma unroll
            for (int k = 0; k < 2; ++k)
                if ((bal[k] >> lane) & 1u) s_list[before[k] + (uint32_t)__popc(bal[k] & ((1u << lane) - 1u))] = (uint32_t)k * 256u + tid;
            if (tid == 0) s_nlist = total;
        }
        __syncthreads();
        // ---- a warp per listed light, lane = cluster of the chunk: the ballot is the light's hit mask over the chunk
        const uint32_t nlist = s_nlist;
        const float4 lo = lane < nc ? *reinterpret_cast<const float4*>(&s_box[lane][0]) : make_float4(0.f, 0.f, 0.f, 0.f);
        const float4 hi = lane < nc ? *reinterpret_cast<const float4*>(&s_box[lane][4]) : make_float4(0.f, 0.f, 0.f, 0.f);
        for (uint32_t i = warp; i < nlist; i += 8u) {
            const uint32_t li = s_list[i];
            const float4 sp = s_sphere[li];
            const bool hit = lane < nc && dist2(sp, lo, hi) <= sp.w;
            if (hit) atomicOr(&s_out[lane][li >> 5], 1u << (li & 31u));
        }
        __syncthreads();
        // rows out: 16 consecutive words per cluster + their popcount (16 lanes per cluster: half-warp reduction)
        for (uint32_t i0 = 0; i0 < kLhClusterChunk * kLhWordsPerCta; i0 += 256u) {
            const uint32_t i = i0 + tid, c = i >> 4, w = i & 15u;
            const uint32_t v = c < nc ? s_out[c][w] : 0u;
            const uint32_t word = blockIdx.x * kLhWordsPerCta + w;
            if (c < nc) hits[(size_t)(chunk0 + c) * words_per_cluster + word] = v;
            uint32_t n = (uint32_t)__popc(v);
            n += __shfl_xor_sync(0xFFFFFFFFu, n, 1); n += __shfl_xor_sync(0xFFFFFFFFu, n, 2);
            n += __shfl_xor_sync(0xFFFFFFFFu, n, 4); n += __shfl_xor_sync(0xFFFFFFFFu, n, 8);
            if (c < nc && w == 0u) {
                counts[(size_t)(chunk0 + c) * gridDim.x + blockIdx.x] = n;
                if (n != 0u) atomicAdd(p.cluster_totals + chunk0 + c, n);
            }
        }
    }
}

// One warp per active cluster, 32 clusters per CTA, no dependency between CTAs: a tile's first index in the global list is
// the sum of the capped totals of all clusters before it (the totals are a few hundred words: every CTA adds them up itself,
// one round of loads, instead of a look-back chain over tiles). The cluster's hit BLOCKS (light blocks with a hit: at most
// 256) are compacted into shared memory in ascending order with their ranks, and lanes expand them in parallel — one
// round of 64-byte row reads for up to 32 hit blocks, wherever in the light range they lie (block by block in 32-block steps
// took one dependent round trip per step).
constexpr int kLlWarps = 32;
template <bool kGrid>
__device__ __forceinline__ void light_lists_body(const ClusterParams& p, const uint32_t* __restrict__ hits, const uint32_t* __restrict__ counts,
                                                 uint32_t words_per_cluster, uint32_t light_blocks) {
    __shared__ uint32_t s_cnt[kLlWarps], s_part[kLlWarps];
    __shared__ uint32_t s_base;
    __shared__ uint32_t s_blocks[kLlWarps][ORBIT_MAX_LIGHTS_PER_CLUSTER];   // block << 9 | rank of its first hit (< 256), per hit block of the warp's cluster
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    const uint32_t nactive = __ldcg(p.unique_clusters + 3);
    if (nactive == 0u) {
        if (blockIdx.x == 0 && tid == 0) p.light_index_words[0] = 0u;
        return;
    }
    const uint32_t ntiles = (nactive + kLlWarps - 1u) / kLlWarps;
    for (uint32_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const uint32_t t = tile * kLlWarps + warp;                         // this warp's active cluster (compacted-list position)
        const bool have = t < nactive;
        const uint32_t* crow = counts + (size_t)t * light_blocks;
        // ---- loads of this round, all independent: the totals below the tile, the cluster's total, index and block counts
        uint32_t below = 0u;
        for (uint32_t c = tid; c < tile * kLlWarps; c += kLlWarps * 32u) below += min(__ldcg(p.cluster_totals + c), (uint32_t)ORBIT_MAX_LIGHTS_PER_CLUSTER);
        const uint32_t count = have ? min(__ldcg(p.cluster_totals + t), (uint32_t)ORBIT_MAX_LIGHTS_PER_CLUSTER) : 0u;
        const uint32_t idx = have ? __ldcg(p.unique_clusters + 4u + t) : 0u;
        constexpr int kKeep = 8;
        uint32_t kept[kKeep];
#pragma unroll
        for (int k = 0; k < kKeep; ++k) kept[k] = (have && (uint32_t)k * 32u + lane < light_blocks) ? __ldcg(crow + (uint32_t)k * 32u + lane) : 0u;
        below = __reduce_add_sync(0xFFFFFFFFu, below);
        __syncthreads();                                                   // previous round's s_cnt / s_part / s_base are no longer read
        if (lane == 0u) { s_cnt[warp] = count; s_part[warp] = below; }
        __syncthreads();
        uint32_t before = 0u, total = 0u, base = 0u;
#pragma unroll
        for (int w = 0; w < kLlWarps; ++w) { const uint32_t v = s_cnt[w]; if ((uint32_t)w < warp) before += v; total += v; base += s_part[w]; }
        if (tile == ntiles - 1u && tid == 0) {
            p.light_index_words[0] = base + total;
            if ((uint64_t)base + total > p.capacity_indices) *p.overflow_flag = 1u;
        }
        if (!have) continue;
        const uint32_t off = base + before;
        if (lane == 0u) {
            if constexpr (kGrid) grid_store(p, idx, off, count);
            else { p.offset_count_image[2u * (size_t)idx] = off; p.offset_count_image[2u * (size_t)idx + 1u] = count; }
        }
        if (count == 0u) continue;
        // ---- hit blocks of the cluster in ascending order, with the rank of their first hit. The block counts were requested
        // with the round's other loads (kept[]: 8 x 32 blocks = 131 072 lights in registers, indexed by compile-time constants
        // only); lights beyond that are walked 32 blocks per dependent load.
        uint32_t* const blk = &s_blocks[warp][0];
        uint32_t nblk = 0u, running = 0u;
        auto step = [&](const uint32_t b0, const uint32_t n) {
            uint32_t inc = n;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const uint32_t v = __shfl_up_sync(0xFFFFFFFFu, inc, d);
                if (lane >= (uint32_t)d) inc += v;
            }
            const uint32_t pos = running + inc - n;
            const bool keep = n != 0u && pos < count;
            const uint32_t km = __ballot_sync(0xFFFFFFFFu, keep);
            if (keep) blk[nblk + (uint32_t)__popc(km & ((1u << lane) - 1u))] = ((b0 + lane) << 9) | pos;
            nblk += (uint32_t)__popc(km);
            running += __shfl_sync(0xFFFFFFFFu, inc, 31);
        };
#pragma unroll
        for (int k = 0; k < kKeep; ++k)
            if ((uint32_t)k * 32u < light_blocks && running < count) step((uint32_t)k * 32u, kept[k]);
#pragma unroll 1
        for (uint32_t b0 = (uint32_t)kKeep * 32u; b0 < light_blocks && running < count; b0 += 32u)
            step(b0, b0 + lane < light_blocks ? __ldcg(crow + b0 + lane) : 0u);
        __syncwarp();
        // ---- expansion: a lane per hit block, the block's 16 words in four 16-byte loads
        const uint32_t* row = hits + (size_t)t * words_per_cluster;
        for (uint32_t i = lane; i < nblk; i += 32u) {
            const uint32_t e = blk[i], eb = e >> 9;
            uint32_t pos = e & 511u;
            const uint4* r4 = reinterpret_cast<const uint4*>(row + (size_t)eb * kLhWordsPerCta);
            const uint4 v0 = __ldcg(r4), v1 = __ldcg(r4 + 1), v2 = __ldcg(r4 + 2), v3 = __ldcg(r4 + 3);
            const uint32_t words[kLhWordsPerCta] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w, v2.x, v2.y, v2.z, v2.w, v3.x, v3.y, v3.z, v3.w};
#pragma unroll
            for (uint32_t w = 0; w < kLhWordsPerCta; ++w) {
                uint32_t word = words[w];
                while (word != 0u && pos < count) {
                    const uint32_t bit = (uint32_t)__ffs((int)word) - 1u;
                    if ((uint64_t)off + pos < p.capacity_indices) p.light_index_words[1u + off + pos] = (eb * kLhWordsPerCta + w) * 32u + bit;
                    word &= word - 1u;
                    ++pos;
                }
            }
        }
    }
}

__global__ void __launch_bounds__(kLlWarps * 32) light_lists_kernel(const __grid_constant__ ClusterParams p, const uint32_t* __restrict__ hits,
                                                                    const uint32_t* __restrict__ counts, uint32_t words_per_cluster, uint32_t light_blocks) {
    light_lists_body<false>(p, hits, counts, words_per_cluster, light_blocks);
}
__global__ void __launch_bounds__(kLlWarps * 32) light_lists_grid_kernel(const __grid_constant__ ClusterParams p, const uint32_t* __restrict__ hits,
                                                                         const uint32_t* __restrict__ counts, uint32_t words_per_cluster, uint32_t light_blocks) {
    light_lists_body<true>(p, hits, counts, words_per_cluster, light_blocks);
}

uint32_t light_hits_blocks(uint32_t n_lights) { return (n_lights + kLhLightsPerCta - 1u) / kLhLightsPerCta; }

cudaError_t launch_light_hits(const ClusterParams& p, uint32_t* hits, uint32_t* counts, uint32_t words_per_cluster, uint32_t max_clusters, cudaStream_t s) {
    const uint32_t gx = light_hits_blocks(p.info.global_light_count);
    uint32_t gy = (max_clusters + kLhClusterChunk - 1u) / kLhClusterChunk;
    if (gy > 16u) gy = 16u;                                      // chunks beyond that are strided over by the same CTAs
    if (gx == 0u) return cudaSuccess;
    light_hits_kernel<<<dim3(gx, gy ? gy : 1u), 256, 0, s>>>(p, hits, counts, words_per_cluster);
    return cudaGetLastError();
}
// to_grid: the offset / count grid goes to p.offset_count_surf (the same for the compaction and CTA-per-cluster launchers)
cudaError_t launch_light_lists(const ClusterParams& p, const uint32_t* hits, const uint32_t* counts, uint32_t words_per_cluster, int grid, cudaStream_t s,
                               bool to_grid) {
    (to_grid ? light_lists_grid_kernel : light_lists_kernel)<<<grid, kLlWarps * 32, 0, s>>>(p, hits, counts, words_per_cluster,
                                                                                           light_hits_blocks(p.info.global_light_count));
    return cudaGetLastError();
}

cudaError_t launch_mark_active(const ClusterParams& p, int grid, cudaStream_t s, bool image) {
    if (image) mark_active_image_kernel<<<grid, 256, 0, s>>>(p);
    else mark_active_kernel<<<grid, 256, 0, s>>>(p);
    return cudaGetLastError();
}
cudaError_t launch_compact_clusters(const ClusterParams& p, cudaStream_t s, bool grid) {
    const uint32_t total = p.info.cluster_count[0] * p.info.cluster_count[1] * p.info.cluster_count[2];
    (grid ? compact_clusters_grid_kernel : compact_clusters_kernel)<<<(total + 255u) / 256u, 256, 0, s>>>(p);
    return cudaGetLastError();
}
cudaError_t launch_light_view(const ClusterParams& p, cudaStream_t s) {
    const uint32_t L = p.info.global_light_count;
    if (L == 0) return cudaSuccess;
    light_view_kernel<<<(L + 255u) / 256u, 256, 0, s>>>(p);
    return cudaGetLastError();
}
static constexpr size_t light_culling_smem_bytes() { return (size_t)kLcWarps * ORBIT_MAX_LIGHTS_PER_CLUSTER * sizeof(uint32_t); }

// More than 48 KB of dynamic shared memory: opt in once per DEVICE (called from orbit_ctx_create with the context's device current).
cudaError_t light_cluster_configure_device() {
    const cudaError_t e = cudaFuncSetAttribute(light_culling_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)light_culling_smem_bytes());
    if (e != cudaSuccess) return e;
    return cudaFuncSetAttribute(light_culling_grid_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)light_culling_smem_bytes());
}

cudaError_t launch_light_culling(const ClusterParams& p, int grid, cudaStream_t s, bool to_grid) {
    (to_grid ? light_culling_grid_kernel : light_culling_kernel)<<<grid, kLcWarps * 32, light_culling_smem_bytes(), s>>>(p);
    return cudaGetLastError();
}

}  // namespace orbit
