// light_culling_kernel.cuh — the CTA-per-cluster light culling kernel of light_cluster.cu (the comment above its inclusion
// there describes it), included twice: ORBIT_LC_KERNEL names the kernel, and ORBIT_LC_GRID = 1 stores each cluster's offset and
// count into the grid surface (ClusterParams::offset_count_surf) instead of the linear buffer. The kernel is spelled out once
// and compiled as two kernels rather than a template body inlined into two wrappers: inlined, the linear kernel's light loop
// came out of the compiler with different instructions than the kernel written directly.
// No include guard: meant to be included more than once.

__global__ void __launch_bounds__(kLcWarps * 32) ORBIT_LC_KERNEL(const __grid_constant__ ClusterParams p) {
    extern __shared__ uint32_t s_dyn[];                       // kLcWarps x 256 hit lists
    __shared__ uint32_t s_warp[kLcWarps];
    __shared__ uint32_t s_tile, s_off;
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    uint32_t* const my_list = s_dyn + warp * ORBIT_MAX_LIGHTS_PER_CLUSTER;
    const unsigned int epoch = scan_epoch(p.scan);
    const uint32_t nactive = __ldcg(p.unique_clusters + 3);
    const uint32_t L = p.info.global_light_count;
    const uint32_t per = (L + kLcWarps - 1) / kLcWarps;
    const uint32_t j_begin = min(warp * per, L), j_end = min(j_begin + per, L);
    while (true) {
        __syncthreads();
        if (tid == 0) s_tile = atomicAdd(p.scan.ticket, 1u);
        __syncthreads();
        const uint32_t tile = s_tile;
        if (tile >= nactive) {
            if (tile == 0u && tid == 0) p.light_index_words[0] = 0u;
            break;
        }
        const uint32_t idx = __ldcg(p.unique_clusters + 4u + tile);
        const Aabb3 box = cluster_volume(p, idx);
        uint32_t count = 0u;   // hits of this warp's stripe (uncapped)
        for (uint32_t j0 = j_begin; j0 < j_end; j0 += 128u) {
            float4 sv[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {   // four independent 512-byte loads in flight per warp
                const uint32_t j = j0 + (uint32_t)u * 32u + lane;
                sv[u] = j < j_end ? __ldg(p.light_view + j) : make_float4(0.f, 0.f, 0.f, -1.f);
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const uint32_t j = j0 + (uint32_t)u * 32u + lane;
                bool hit = false;
                if (j < j_end) {
                    const float4 s = sv[u];
                    float acc = 0.0f;
                    const float c[3] = {s.x, s.y, s.z};
#pragma unroll
                    for (int k = 0; k < 3; ++k) {
                        // lo <= hi, so at most one of the reference's two branches adds a term; d is that term's
                        // base (or 0, and fma(0,0,acc) == acc): same value, no divergence
                        const float v = c[k];
                        const float d = fmaxf(fmaxf(sub(box.lo[k], v), sub(v, box.hi[k])), 0.0f);
                        acc = fma_(d, d, acc);
                    }
                    hit = acc <= mul(s.w, s.w);
                }
                const uint32_t bal = __ballot_sync(0xFFFFFFFFu, hit);
                if (hit) {
                    const uint32_t r = count + __popc(bal & ((1u << lane) - 1u));
                    if (r < ORBIT_MAX_LIGHTS_PER_CLUSTER) my_list[r] = j;
                }
                count += __popc(bal);
            }
        }
        if (lane == 0u) s_warp[warp] = min(count, ORBIT_MAX_LIGHTS_PER_CLUSTER);
        __syncthreads();
        // exclusive prefix of the (capped) stripe counts in warp order; everything past 256 is dropped
        uint32_t before = 0u, total = 0u;
#pragma unroll
        for (int w = 0; w < kLcWarps; ++w) { const uint32_t v = s_warp[w]; if ((uint32_t)w < warp) before += v; total += v; }
        total = min(total, ORBIT_MAX_LIGHTS_PER_CLUSTER);
        if (warp == 0u) {
            const uint32_t off = lookback_exclusive(p.scan, epoch, tile, total);
            if (lane == 0u) {
                s_off = off;
#if ORBIT_LC_GRID
                grid_store(p, idx, off, total);
#else
                p.offset_count_image[2u * (size_t)idx] = off;
                p.offset_count_image[2u * (size_t)idx + 1u] = total;
#endif
                if (tile == nactive - 1u) {
                    p.light_index_words[0] = off + total;
                    if ((uint64_t)off + total > p.capacity_indices) *p.overflow_flag = 1u;
                }
            }
        }
        __syncthreads();
        const uint32_t off = s_off;
        const uint32_t mine = min(count, ORBIT_MAX_LIGHTS_PER_CLUSTER);
        for (uint32_t k = lane; k < mine; k += 32u) {
            const uint32_t r = before + k;
            if (r < ORBIT_MAX_LIGHTS_PER_CLUSTER && (uint64_t)off + r < p.capacity_indices) p.light_index_words[1u + off + r] = my_list[k];
        }
    }
    if (tid == 0) scan_cta_exit(p.scan, epoch);
}
