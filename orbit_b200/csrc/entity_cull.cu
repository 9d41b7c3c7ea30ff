// entity_cull.cu — per-entity frustum + two-pass occlusion cull, LOD select, ordered dispatch-record emission.
//
// Stands in for shaders/entity_cull.comp:104-245 driven by create_meshlet_dispatch_command
// (src/passes/draw_gen.rs:327-380).
//
// B200 design: one thread per entity draw as in the reference (256 per CTA), but the reference's
// `atomicAdd(workgroup_count_x, n)` + per-thread serial record loop (entity_cull.comp:211-223) becomes a CTA
// scan + an ordered prefix over CTAs followed by load-balanced emission: the CTA's records form one contiguous
// span, thread j writes record j of the span after a binary search for its owning draw, so stores are dense and
// the record order is (entity-draw index, chunk) regardless of scheduling. The kernel is latency-bound (10^4..
// 2.5*10^5 threads), so dependent memory round trips are what is minimised: the whole 128-byte MeshInfo (sphere
// + LOD table) is fetched up front instead of after the LOD is known, and when the grid is co-resident
// (kFlat) tiles are block indices and the prefix is a flat gather of all lower CTAs' aggregates — no ticket
// atomic, no hop-by-hop look-back; larger grids fall back to ticket + decoupled look-back (scan.cuh).
// The pass-2 visibility word is the warp ballot (reference: subgroupBallot with 32-wide subgroups).
#include "params.cuh"

namespace orbit {

#ifndef ORBIT_EC_THREADS
#define ORBIT_EC_THREADS 256
#endif
constexpr int kEcThreads = ORBIT_EC_THREADS;   // entity draws per CTA (tuning experiments: -DORBIT_EC_THREADS=128)
constexpr uint32_t kEcBatch = 2048u;           // records staged in shared memory per round of the emission (32 KB)


template <bool kFlat>
__global__ void __launch_bounds__(kEcThreads) entity_cull_kernel(const __grid_constant__ EntityCullParams p) {
    __shared__ uint4 s_recs[kEcBatch];            // the tile's records, staged for coalesced stores
    __shared__ uint32_t s_warp[kEcThreads / 32];
    __shared__ uint32_t s_tile, s_base;

    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    const OrbitCullInfo& ci = p.cull;
    pdl_wait();
    ORBIT_TRACE_STAMP(p.scan.trace, 0, 0);
    const unsigned int epoch = scan_epoch(p.scan);
    // Tiles are handed out by an atomic ticket in BOTH variants, so the CTAs that own a tile's predecessors are always running
    // or finished and the waits below (look-back, flat gather) cannot deadlock, whatever else shares the GPU and in whatever
    // order CTAs are dispatched. The look-back variant waits for its ticket; the flat variant (small, latency-bound grids) does
    // not: it requests the draw words of tile blockIdx.x while the ticket is in flight — CTAs are dispatched in index order in
    // practice, so the guess is right and the atomic costs no dependent round trip — and re-requests them in the rare case
    // that the ticket disagrees.
    if (tid == 0) s_tile = atomicAdd(p.scan.ticket, 1u);
    uint32_t tile = blockIdx.x;
    if (!kFlat) {
        __syncthreads();
        tile = s_tile;
    }
    const uint32_t ntiles = gridDim.x;

    // The draw words are requested before the device-side count is known (gid < draw_end <= the host's
    // entity_draw_count, which sized the buffer): one dependent round trip less on a latency-bound kernel.
    uint32_t gid = p.draw_begin + tile * kEcThreads + tid;
    uint32_t entity_index = 0u, mesh_index = 0u, vis_offset = 0u;
    if (gid < p.draw_end) {
        entity_index = __ldg(p.entity_draw_words + 1u + 3u * (size_t)gid + 0u);
        mesh_index = __ldg(p.entity_draw_words + 1u + 3u * (size_t)gid + 1u);
        vis_offset = __ldg(p.entity_draw_words + 1u + 3u * (size_t)gid + 2u);
    }
    if (kFlat) {
        __syncthreads();
        if (s_tile != tile) {                                    // out-of-order dispatch: take the ticket's tile instead
            tile = s_tile;
            gid = p.draw_begin + tile * kEcThreads + tid;
            entity_index = mesh_index = vis_offset = 0u;
            if (gid < p.draw_end) {
                entity_index = __ldg(p.entity_draw_words + 1u + 3u * (size_t)gid + 0u);
                mesh_index = __ldg(p.entity_draw_words + 1u + 3u * (size_t)gid + 1u);
                vis_offset = __ldg(p.entity_draw_words + 1u + 3u * (size_t)gid + 2u);
            }
        }
    }
    const uint32_t count = min(__ldg(p.entity_draw_words), p.draw_end);
    ORBIT_TRACE_STAMP(p.scan.trace, 0, 1 + 0 * (count + epoch));
    const uint32_t pass = ci.occlusion_pass;
    const bool mocc = ci.meshlet_visibility_buffer != ORBIT_NO_BUFFER;

    uint32_t chunks = 0u, lod_off = 0u, lod_cnt = 0u;
    bool visible = false;
    const bool in_range = gid < count;
    if (in_range) {
        // every load that depends only on the draw words, issued back to back (ordered loads, orbit_device.cuh): what
        // is needed last goes first, the model matrix — consumed by the very next instructions — last
        const uint8_t* mi = p.mesh_infos + (size_t)mesh_index * 128u;
        uint4 lods[4];                                                            // 8 x (meshlet_offset, meshlet_count)
#pragma unroll
        for (int k = 0; k < 4; ++k) lods[k] = ld_v4_ordered(mi + 64 + 16 * k);
        const uint4 mi_hdr = ld_v4_ordered(mi + 48);                              // vertex_offset, data_offset, lod_count, pad
        uint32_t vword = 0xFFFFFFFFu;
        if (pass == 1u || pass == 2u) vword = ld_u32_ordered(p.entity_visibility + (gid >> 5));
        const float4 sph = as_float4(ld_v4_ordered(mi));
        float4 mcol[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) mcol[k] = as_float4(ld_v4_ordered(p.entities + (size_t)entity_index * 8u + k));
        const bool vib = ((vword >> (gid & 31u)) & 1u) != 0u;
        visible = (pass == 1u) ? vib : true;
        ORBIT_TRACE_STAMP(p.scan.trace, 0, 2 + 0 * (uint32_t)(mcol[3].w != 0.0f) + 0 * (lods[0].x & sph.x != 0.0f));

        // view * model (entity_cull.comp:131-133)
        ModelView mv;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const float4 b = mcol[k];
#pragma unroll
            for (int row = 0; row < 4; ++row)
                mv.m[k * 4 + row] = add(add(add(mul(ci.view_matrix.m[0][row], b.x), mul(ci.view_matrix.m[1][row], b.y)),
                                            mul(ci.view_matrix.m[2][row], b.z)), mul(ci.view_matrix.m[3][row], b.w));
        }
        mv.scale = largest_scale(mv.m);
        Sphere s = transform_sphere(mv, sph.x, sph.y, sph.z, sph.w);
        if (visible) visible = frustum_test(ci, s);
        if (pass == 2u && visible) visible = occlusion_test(ci, s, p.hiz);
        bool should_draw = visible;
        if (pass == 2u) should_draw = visible && (!vib || mocc);
        if (should_draw) {
            const float dx = sub(ci.lod_target_pos_view_space[0], s.x);
            const float dy = sub(ci.lod_target_pos_view_space[1], s.y);
            const float dz = sub(ci.lod_target_pos_view_space[2], s.z);
            const float lod_distance = sub(fsqrt(dot3(dx, dy, dz, dx, dy, dz)), s.r);
            const float f = fdiv(orbit_log2f(fdiv(fmaxf(lod_distance, 0.0f), ci.lod_base)), orbit_log2f(ci.lod_step));
            uint32_t lod = f2u(fmaxf(add(f, 1.0f), 0.0f));
            lod = min(max(lod, ci.min_mesh_lod), ci.max_mesh_lod);
            const uint32_t lod_count = mi_hdr.z;
            const uint32_t li = min(lod, lod_count - 1u) & 7u;
            uint2 L = make_uint2(lods[0].x, lods[0].y);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                if (li == 2u * k) L = make_uint2(lods[k].x, lods[k].y);
                if (li == 2u * k + 1u) L = make_uint2(lods[k].z, lods[k].w);
            }
            chunks = (L.y + 31u) >> 5;
            lod_off = L.x; lod_cnt = L.y;
        }
    }
    // pass 2: visibility word of these 32 draws (lanes past `count` contribute 0)
    const uint32_t vis_mask = __ballot_sync(0xFFFFFFFFu, visible);
    ORBIT_TRACE_STAMP(p.scan.trace, 0, 3 + 0 * (vis_mask & 1u));
    if (pass == 2u && lane == 0u && gid < count) p.entity_visibility[gid >> 5] = vis_mask;

    // ---- CTA exclusive scan of chunk counts
    uint32_t incl = chunks;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, d);
        if (lane >= (uint32_t)d) incl += t;
    }
    if (lane == 31u) s_warp[warp] = incl;
    __syncthreads();
    uint32_t warp_base = 0u, tile_total = 0u;
#pragma unroll
    for (int w = 0; w < kEcThreads / 32; ++w) {
        const uint32_t v = s_warp[w];
        if ((uint32_t)w < warp) warp_base += v;
        tile_total += v;
    }
    const uint32_t my_excl = warp_base + incl - chunks;     // first record of this draw inside the tile's span
    ORBIT_TRACE_STAMP(p.scan.trace, 0, 4 + 0 * (tile_total & 1u));
    if (warp == 0u) {
        uint32_t base;
        if (kFlat) {
            if (lane == 0u) publish(p.scan.status + tile, pack_status(epoch, kFlagAggregate, tile_total));
            base = gather_lower_aggregates(p.scan, epoch, tile);
        } else {
            base = lookback_exclusive(p.scan, epoch, tile, tile_total);
        }
        ORBIT_TRACE_STAMP(p.scan.trace, 0, 5 + 0 * (base & 1u));
        if (lane == 0u) {
            s_base = base;
            if (tile == ntiles - 1u) {
                p.dispatch_words[0] = base + tile_total;   // workgroup_count_x
                p.dispatch_words[1] = 1u;                  // fill_buffer {.,1,1}: draw_gen.rs:356-363
                p.dispatch_words[2] = 1u;
                if (p.dispatch_mirror != nullptr) { p.dispatch_mirror[0] = base + tile_total; p.dispatch_mirror[1] = 1u; p.dispatch_mirror[2] = 1u; }
                if ((uint64_t)base + tile_total > p.capacity_records) *p.overflow_flag = 1u;
            }
        }
    }
    __syncthreads();
    pdl_launch_dependents();
    // ---- emission: the tile's records form one contiguous span of the buffer. Every draw writes its own records into the
    // shared-memory image of the span (no search for the owner of a record), then the CTA copies the image out word by word:
    // consecutive threads store consecutive words (the records start 12 bytes into the buffer, so 16-byte stores would be
    // misaligned; per-record scalar stores touched 16 sectors per instruction and made this phase 2 us of a 9 us kernel).
    const uint64_t base = s_base;
    for (uint32_t batch0 = 0u; batch0 < tile_total; batch0 += kEcBatch) {
        // every earlier chunk of a draw is full, so visibility_offset += count/32 adds exactly 1 per chunk
        for (uint32_t k = my_excl < batch0 ? batch0 - my_excl : 0u; k < chunks && my_excl + k < batch0 + kEcBatch; ++k) {
            const uint32_t n = min(lod_cnt - 32u * k, 32u);
            s_recs[my_excl + k - batch0] = make_uint4(entity_index, lod_off + 32u * k, n, vis_offset + k);
            // (An L2 prefetch of the records' meshlets from here — one cp.async.bulk.prefetch per record, for the test kernel
            // that follows — was measured: 880 bulk prefetches per CTA queue up in the SM's copy unit and the C2 frame got
            // 11 us SLOWER.)
        }
        __syncthreads();
        const uint64_t first = base + batch0;                                     // record index of the image's first record
        uint64_t n = min(kEcBatch, tile_total - batch0);
        if (first >= p.capacity_records) n = 0u; else if (first + n > p.capacity_records) n = p.capacity_records - first;
        const uint32_t* const img = reinterpret_cast<const uint32_t*>(s_recs);
        uint32_t* const dst = p.dispatch_words + 3u + first * 4u;
        for (uint32_t w = tid; w < (uint32_t)n * 4u; w += kEcThreads) dst[w] = img[w];
        if (p.dispatch_mirror != nullptr) {
            uint32_t* const dst2 = p.dispatch_mirror + 3u + first * 4u;
            for (uint32_t w = tid; w < (uint32_t)n * 4u; w += kEcThreads) dst2[w] = img[w];
        }
        __syncthreads();
    }
    ORBIT_TRACE_STAMP(p.scan.trace, 0, 6);
    if (tid == 0) scan_cta_exit(p.scan, epoch);
    ORBIT_TRACE_STAMP(p.scan.trace, 0, 7);
}

// orbit_entity_cull_views (kPass 0) and orbit_entity_cull_views_occlusion (kPass 1, 2): entity_cull_kernel for views[0..n_views)
// of one scene, in one launch (no mirror buffer). kPass 1 reads each view's entity visibility bit, kPass 2 runs the Hi-Z test
// against each view's pyramid and writes each view's visibility words; every view of a launch has that pass (the host refuses
// mixed passes). It is a kernel of its own rather than a template parameter of entity_cull_kernel because the single-view
// kernel's SASS must stay as it is, and every folded form tried reordered it. The scene fields (draw words, mesh infos, entities, draw range, scan state) are read from views[0]. Tickets are handed out
// tile-major, view-minor: ticket t covers draw tile t / n_views for view t % n_views, so the lower draw tiles of a view always
// hold lower tickets and the waits below keep their no-deadlock argument. The scan descriptors of view v are the block
// [v * draw tiles, (v + 1) * draw tiles): each view's prefix (flat gather or look-back) sees only its own tiles.
template <bool kFlat, int kPass>
__global__ void __launch_bounds__(kEcThreads) entity_cull_views_kernel(const __grid_constant__ EntityViewsParams params) {
    const EntityCullParams* const views = params.view;
    __shared__ uint4 s_recs[kEcBatch];            // the tile's records, staged for coalesced stores
    __shared__ uint32_t s_warp[kEcThreads / 32];
    __shared__ uint32_t s_tile, s_base;

    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    const uint32_t n_views = params.n_views;
    const EntityCullParams& p0 = views[0];
    pdl_wait();
    ORBIT_TRACE_STAMP(p0.scan.trace, 0, 0);
    const unsigned int epoch = scan_epoch(p0.scan);
    // Tiles are handed out by an atomic ticket in BOTH variants, so the CTAs that own a tile's predecessors are always running
    // or finished and the waits below (look-back, flat gather) cannot deadlock, whatever else shares the GPU and in whatever
    // order CTAs are dispatched. The look-back variant waits for its ticket; the flat variant (small, latency-bound grids) does
    // not: it requests the draw words of tile blockIdx.x while the ticket is in flight — CTAs are dispatched in index order in
    // practice, so the guess is right and the atomic costs no dependent round trip — and re-requests them in the rare case
    // that the ticket disagrees.
    if (tid == 0) s_tile = atomicAdd(p0.scan.ticket, 1u);
    uint32_t tile = blockIdx.x;
    if (!kFlat) {
        __syncthreads();
        tile = s_tile;
    }
    const uint32_t ntiles = gridDim.x / n_views;                 // draw tiles per view

    // The draw words are requested before the device-side count is known (gid < draw_end <= the host's
    // entity_draw_count, which sized the buffer): one dependent round trip less on a latency-bound kernel.
    uint32_t gid = p0.draw_begin + (tile / n_views) * kEcThreads + tid;
    uint32_t entity_index = 0u, mesh_index = 0u, vis_offset = 0u;
    if (gid < p0.draw_end) {
        entity_index = __ldg(p0.entity_draw_words + 1u + 3u * (size_t)gid + 0u);
        mesh_index = __ldg(p0.entity_draw_words + 1u + 3u * (size_t)gid + 1u);
        vis_offset = __ldg(p0.entity_draw_words + 1u + 3u * (size_t)gid + 2u);
    }
    if (kFlat) {
        __syncthreads();
        if (s_tile != tile) {                                    // out-of-order dispatch: take the ticket's tile instead
            tile = s_tile;
            gid = p0.draw_begin + (tile / n_views) * kEcThreads + tid;
            entity_index = mesh_index = vis_offset = 0u;
            if (gid < p0.draw_end) {
                entity_index = __ldg(p0.entity_draw_words + 1u + 3u * (size_t)gid + 0u);
                mesh_index = __ldg(p0.entity_draw_words + 1u + 3u * (size_t)gid + 1u);
                vis_offset = __ldg(p0.entity_draw_words + 1u + 3u * (size_t)gid + 2u);
            }
        }
    }
    const uint32_t view = tile % n_views;
    tile /= n_views;                                             // from here on: the draw tile of this view
    ScanState scan = p0.scan;
    scan.status += (size_t)view * ntiles;
    const EntityCullParams& p = views[view];
    const OrbitCullInfo& ci = p.cull;
    const uint32_t count = min(__ldg(p0.entity_draw_words), p0.draw_end);
    ORBIT_TRACE_STAMP(p0.scan.trace, 0, 1 + 0 * (count + epoch));

    uint32_t chunks = 0u, lod_off = 0u, lod_cnt = 0u;
    bool visible = false;                                        // kPass 2: this view's new visibility bit of the draw
    const bool in_range = gid < count;
    if (in_range) {
        // every load that depends only on the draw words, issued back to back (ordered loads, orbit_device.cuh): what
        // is needed last goes first, the model matrix — consumed by the very next instructions — last
        const uint8_t* mi = p.mesh_infos + (size_t)mesh_index * 128u;
        uint4 lods[4];                                                            // 8 x (meshlet_offset, meshlet_count)
#pragma unroll
        for (int k = 0; k < 4; ++k) lods[k] = ld_v4_ordered(mi + 64 + 16 * k);
        const uint4 mi_hdr = ld_v4_ordered(mi + 48);                              // vertex_offset, data_offset, lod_count, pad
        uint32_t vword = 0xFFFFFFFFu;
        if constexpr (kPass != 0) vword = ld_u32_ordered(p.entity_visibility + (gid >> 5));
        const float4 sph = as_float4(ld_v4_ordered(mi));
        float4 mcol[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) mcol[k] = as_float4(ld_v4_ordered(p.entities + (size_t)entity_index * 8u + k));
        const bool vib = ((vword >> (gid & 31u)) & 1u) != 0u;
        ORBIT_TRACE_STAMP(p.scan.trace, 0, 2 + 0 * (uint32_t)(mcol[3].w != 0.0f) + 0 * (lods[0].x & sph.x != 0.0f));

        // view * model (entity_cull.comp:131-133)
        ModelView mv;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const float4 b = mcol[k];
#pragma unroll
            for (int row = 0; row < 4; ++row)
                mv.m[k * 4 + row] = add(add(add(mul(ci.view_matrix.m[0][row], b.x), mul(ci.view_matrix.m[1][row], b.y)),
                                            mul(ci.view_matrix.m[2][row], b.z)), mul(ci.view_matrix.m[3][row], b.w));
        }
        mv.scale = largest_scale(mv.m);
        Sphere s = transform_sphere(mv, sph.x, sph.y, sph.z, sph.w);
        bool should_draw;                                            // entity_cull.comp:137-189, as in entity_cull_kernel
        if constexpr (kPass == 0) {
            should_draw = frustum_test(ci, s);                       // pass 0: should_draw = visible
        } else {
            const bool mocc = ci.meshlet_visibility_buffer != ORBIT_NO_BUFFER;
            visible = (kPass == 1) ? vib : true;
            if (visible) visible = frustum_test(ci, s);
            if (kPass == 2 && visible) visible = occlusion_test(ci, s, p.hiz);
            should_draw = (kPass == 2) ? visible && (!vib || mocc) : visible;
        }
        if (should_draw) {
            const float dx = sub(ci.lod_target_pos_view_space[0], s.x);
            const float dy = sub(ci.lod_target_pos_view_space[1], s.y);
            const float dz = sub(ci.lod_target_pos_view_space[2], s.z);
            const float lod_distance = sub(fsqrt(dot3(dx, dy, dz, dx, dy, dz)), s.r);
            const float f = fdiv(orbit_log2f(fdiv(fmaxf(lod_distance, 0.0f), ci.lod_base)), orbit_log2f(ci.lod_step));
            uint32_t lod = f2u(fmaxf(add(f, 1.0f), 0.0f));
            lod = min(max(lod, ci.min_mesh_lod), ci.max_mesh_lod);
            const uint32_t lod_count = mi_hdr.z;
            const uint32_t li = min(lod, lod_count - 1u) & 7u;
            uint2 L = make_uint2(lods[0].x, lods[0].y);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                if (li == 2u * k) L = make_uint2(lods[k].x, lods[k].y);
                if (li == 2u * k + 1u) L = make_uint2(lods[k].z, lods[k].w);
            }
            chunks = (L.y + 31u) >> 5;
            lod_off = L.x; lod_cnt = L.y;
        }
    }
    if constexpr (kPass == 2) {   // this view's visibility word of these 32 draws (lanes past `count` contribute 0)
        const uint32_t vis_mask = __ballot_sync(0xFFFFFFFFu, visible);
        if (lane == 0u && gid < count) p.entity_visibility[gid >> 5] = vis_mask;
    }

    // ---- CTA exclusive scan of chunk counts
    uint32_t incl = chunks;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, d);
        if (lane >= (uint32_t)d) incl += t;
    }
    if (lane == 31u) s_warp[warp] = incl;
    __syncthreads();
    uint32_t warp_base = 0u, tile_total = 0u;
#pragma unroll
    for (int w = 0; w < kEcThreads / 32; ++w) {
        const uint32_t v = s_warp[w];
        if ((uint32_t)w < warp) warp_base += v;
        tile_total += v;
    }
    const uint32_t my_excl = warp_base + incl - chunks;     // first record of this draw inside the tile's span
    ORBIT_TRACE_STAMP(p.scan.trace, 0, 4 + 0 * (tile_total & 1u));
    if (warp == 0u) {
        uint32_t base;
        if (kFlat) {
            if (lane == 0u) publish(scan.status + tile, pack_status(epoch, kFlagAggregate, tile_total));
            base = gather_lower_aggregates(scan, epoch, tile);
        } else {
            base = lookback_exclusive(scan, epoch, tile, tile_total);
        }
        ORBIT_TRACE_STAMP(p.scan.trace, 0, 5 + 0 * (base & 1u));
        if (lane == 0u) {
            s_base = base;
            if (tile == ntiles - 1u) {
                p.dispatch_words[0] = base + tile_total;   // workgroup_count_x
                p.dispatch_words[1] = 1u;                  // fill_buffer {.,1,1}: draw_gen.rs:356-363
                p.dispatch_words[2] = 1u;
                if ((uint64_t)base + tile_total > p.capacity_records) *p.overflow_flag = 1u;
            }
        }
    }
    __syncthreads();
    pdl_launch_dependents();
    // ---- emission: the tile's records form one contiguous span of the buffer. Every draw writes its own records into the
    // shared-memory image of the span (no search for the owner of a record), then the CTA copies the image out word by word:
    // consecutive threads store consecutive words (the records start 12 bytes into the buffer, so 16-byte stores would be
    // misaligned; per-record scalar stores touched 16 sectors per instruction and made this phase 2 us of a 9 us kernel).
    const uint64_t base = s_base;
    for (uint32_t batch0 = 0u; batch0 < tile_total; batch0 += kEcBatch) {
        // every earlier chunk of a draw is full, so visibility_offset += count/32 adds exactly 1 per chunk
        for (uint32_t k = my_excl < batch0 ? batch0 - my_excl : 0u; k < chunks && my_excl + k < batch0 + kEcBatch; ++k) {
            const uint32_t n = min(lod_cnt - 32u * k, 32u);
            s_recs[my_excl + k - batch0] = make_uint4(entity_index, lod_off + 32u * k, n, vis_offset + k);
            // (An L2 prefetch of the records' meshlets from here — one cp.async.bulk.prefetch per record, for the test kernel
            // that follows — was measured: 880 bulk prefetches per CTA queue up in the SM's copy unit and the C2 frame got
            // 11 us SLOWER.)
        }
        __syncthreads();
        const uint64_t first = base + batch0;                                     // record index of the image's first record
        uint64_t n = min(kEcBatch, tile_total - batch0);
        if (first >= p.capacity_records) n = 0u; else if (first + n > p.capacity_records) n = p.capacity_records - first;
        const uint32_t* const img = reinterpret_cast<const uint32_t*>(s_recs);
        uint32_t* const dst = p.dispatch_words + 3u + first * 4u;
        for (uint32_t w = tid; w < (uint32_t)n * 4u; w += kEcThreads) dst[w] = img[w];
        __syncthreads();
    }
    ORBIT_TRACE_STAMP(p.scan.trace, 0, 6);
    if (tid == 0) scan_cta_exit(p0.scan, epoch);
    ORBIT_TRACE_STAMP(p.scan.trace, 0, 7);
}

cudaError_t launch_entity_cull(const EntityCullParams& p, uint32_t n_draws, uint32_t coresident_ctas, cudaStream_t stream) {
    uint32_t grid = (n_draws + kEcThreads - 1) / kEcThreads;
    if (grid == 0) grid = 1;
    if (grid <= coresident_ctas) return launch_kernel(entity_cull_kernel<true>, dim3(grid), dim3(kEcThreads), 0, stream, p);
    return launch_kernel(entity_cull_kernel<false>, dim3(grid), dim3(kEcThreads), 0, stream, p);
}

template <int kPass>
static cudaError_t launch_entity_views_pass(const EntityViewsParams& pv, uint32_t grid, uint32_t coresident_ctas, cudaStream_t stream) {
    if (grid <= coresident_ctas) return launch_kernel(entity_cull_views_kernel<true, kPass>, dim3(grid), dim3(kEcThreads), 0, stream, pv);
    return launch_kernel(entity_cull_views_kernel<false, kPass>, dim3(grid), dim3(kEcThreads), 0, stream, pv);
}

// coresident_ctas: from entity_cull_views_max_ctas_per_sm of the same pass
cudaError_t launch_entity_cull_views(const EntityViewsParams& pv, uint32_t n_draws, uint32_t coresident_ctas, cudaStream_t stream) {
    uint32_t tiles = (n_draws + kEcThreads - 1) / kEcThreads;
    if (tiles == 0) tiles = 1;
    const uint32_t grid = tiles * pv.n_views;
    const uint32_t pass = pv.view[0].cull.occlusion_pass;
    if (pass == 1u) return launch_entity_views_pass<1>(pv, grid, coresident_ctas, stream);
    if (pass == 2u) return launch_entity_views_pass<2>(pv, grid, coresident_ctas, stream);
    return launch_entity_views_pass<0>(pv, grid, coresident_ctas, stream);
}

int entity_cull_max_ctas_per_sm() {
    int n = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, entity_cull_kernel<true>, kEcThreads, 0);
    return n;
}

int entity_cull_views_max_ctas_per_sm(uint32_t occlusion_pass) {
    int n = 0;
    if (occlusion_pass == 1u) cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, entity_cull_views_kernel<true, 1>, kEcThreads, 0);
    else if (occlusion_pass == 2u) cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, entity_cull_views_kernel<true, 2>, kEcThreads, 0);
    else cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, entity_cull_views_kernel<true, 0>, kEcThreads, 0);
    return n;
}

}  // namespace orbit
