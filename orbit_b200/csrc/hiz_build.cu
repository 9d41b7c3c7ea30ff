// hiz_build.cu — the whole depth pyramid in ONE launch (sm_100a).
//
// Stands in for DepthPyramid::update (src/passes/draw_gen.rs:510-566): 11-12 serialized dispatches of
// shaders/depth_reduce.comp with a full barrier between mips, each texel = ReduceMin-sampler fetch
// (src/graphics/device.rs:1404-1420) at the texel-centre UV of the previous level.
//
// CUDA has no min-reduction texture filter, so the 2x2 footprint is computed explicitly (which also makes it
// exact): level 0 takes the footprint of ((x+.5)/w0, (y+.5)/h0) in the W x H depth buffer (ratio in (1,2], the
// reference's non-conservative 2-texel footprint is reproduced, not "fixed"); level l>=1 is the exact 2x2
// block of level l-1, clamped when a dimension has collapsed to 1.
//
// Structure (FidelityFX-SPD-like): a CTA of 8 warps owns a 64x64 tile of level 0. A warp owns 8 rows; a lane
// owns two adjacent columns of each, so levels 1..3 are reduced in registers + warp shuffles, levels 4..6 by
// one warp through a 8x8 shared-memory tile. The last CTA to finish (atomic ticket) reduces the remaining
// small levels out of L2. Pyramids smaller than 64 in a dimension take the generic tail path only.
#include "params.cuh"

namespace orbit {


__device__ __forceinline__ float ld_cg(const float* p) { return __ldcg(p); }

// Generic level-by-level reduction of levels [first, levels) by ONE CTA (reads level first-1 from global / L2).
__device__ void hiz_tail(const HizBuildParams& p, uint32_t first) {
    for (uint32_t l = first; l < p.levels; ++l) {
        const uint32_t w = max(p.width >> l, 1u), h = max(p.height >> l, 1u);
        float* dst = p.texels + p.level_offset[l];
        if (l == 0u) {
            for (uint32_t i = threadIdx.x; i < w * h; i += blockDim.x) {
                const uint32_t x = i % w, y = i / w;
                int x0, x1, y0, y1;
                footprint(fdiv(add((float)x, 0.5f), (float)w), p.depth_w, x0, x1);
                footprint(fdiv(add((float)y, 0.5f), (float)h), p.depth_h, y0, y1);
                const float* r0 = p.depth + (size_t)y0 * p.depth_w;
                const float* r1 = p.depth + (size_t)y1 * p.depth_w;
                dst[i] = fminf(fminf(__ldg(r0 + x0), __ldg(r0 + x1)), fminf(__ldg(r1 + x0), __ldg(r1 + x1)));
            }
        } else {
            const uint32_t sw = max(p.width >> (l - 1u), 1u), sh = max(p.height >> (l - 1u), 1u);
            const float* src = p.texels + p.level_offset[l - 1u];
            for (uint32_t i = threadIdx.x; i < w * h; i += blockDim.x) {
                const uint32_t x = i % w, y = i / w;
                const uint32_t x0 = min(2u * x, sw - 1u), x1 = min(2u * x + 1u, sw - 1u);
                const uint32_t y0 = min(2u * y, sh - 1u), y1 = min(2u * y + 1u, sh - 1u);
                dst[i] = fminf(fminf(ld_cg(src + (size_t)y0 * sw + x0), ld_cg(src + (size_t)y0 * sw + x1)),
                               fminf(ld_cg(src + (size_t)y1 * sw + x0), ld_cg(src + (size_t)y1 * sw + x1)));
            }
        }
        __threadfence_block();
        __syncthreads();
    }
}

// Top of the pyramid by the last CTA: level `first-1` (at most 4096 texels) is pulled into shared memory with one
// round of L2 loads, then every remaining level is reduced out of shared memory (no global round trip per level).
__device__ void hiz_tail_smem(const HizBuildParams& p, uint32_t first, float* s_a, float* s_b) {
    uint32_t sw = max(p.width >> (first - 1u), 1u), sh = max(p.height >> (first - 1u), 1u);
    const float* src_g = p.texels + p.level_offset[first - 1u];
    for (uint32_t i = threadIdx.x; i < sw * sh; i += blockDim.x) s_a[i] = ld_cg(src_g + i);
    __syncthreads();
    float* src = s_a;
    float* dst = s_b;
    for (uint32_t l = first; l < p.levels; ++l) {
        const uint32_t w = max(p.width >> l, 1u), h = max(p.height >> l, 1u);
        float* out = p.texels + p.level_offset[l];
        for (uint32_t i = threadIdx.x; i < w * h; i += blockDim.x) {
            const uint32_t x = i % w, y = i / w;
            const uint32_t x0 = min(2u * x, sw - 1u), x1 = min(2u * x + 1u, sw - 1u);
            const uint32_t y0 = min(2u * y, sh - 1u), y1 = min(2u * y + 1u, sh - 1u);
            const float v = fminf(fminf(src[y0 * sw + x0], src[y0 * sw + x1]), fminf(src[y1 * sw + x0], src[y1 * sw + x1]));
            dst[i] = v;
            out[i] = v;
        }
        __syncthreads();
        float* t = src; src = dst; dst = t;
        sw = w; sh = h;
    }
}

__global__ void __launch_bounds__(256) hiz_small_kernel(const __grid_constant__ HizBuildParams p) {
    pdl_wait();
    hiz_tail(p, 0u);
}

// One pyramid, one CTA per 64x64 tile of level 0 (blockIdx.x); the batched kernel runs one row of the grid per pyramid.
__device__ __forceinline__ void hiz_build_body(const HizBuildParams& p) {
    __shared__ float s_l3[8][8];
    __shared__ bool s_last;
    __shared__ float s_top_a[4096], s_top_b[1024];
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    const uint32_t tiles_x = p.width >> 6;
    const uint32_t tx = blockIdx.x % tiles_x, ty = blockIdx.x / tiles_x;
    pdl_wait();
    ORBIT_TRACE_STAMP(p.trace, 4, 0);

    // ---- level 0: lane owns columns 2*lane, 2*lane+1 of rows warp*8 .. warp*8+7 of the tile
    const uint32_t x_a = tx * 64u + 2u * lane;
    int xa0, xa1, xb0, xb1;
    footprint(fdiv(add((float)x_a, 0.5f), (float)p.width), p.depth_w, xa0, xa1);
    footprint(fdiv(add((float)(x_a + 1u), 0.5f), (float)p.width), p.depth_w, xb0, xb1);
    const uint32_t y_base = ty * 64u + warp * 8u;
    float va[8], vb[8];
    {
        // All 64 texel loads of the thread leave back to back, before any of them is consumed: left to the compiler, the loads of
        // a row were issued only when the row before had been reduced (two rows in flight: four to five dependent DRAM round
        // trips for the tile, "level0 loaded" 4.9 us into an 8 us kernel). `asm volatile` keeps the loads in program order.
        const float* r0[8];
        const float* r1[8];
#pragma unroll
        for (int r = 0; r < 8; ++r) {
            int y0, y1;
            footprint(fdiv(add((float)(y_base + r), 0.5f), (float)p.height), p.depth_h, y0, y1);
            r0[r] = p.depth + (size_t)y0 * p.depth_w;
            r1[r] = p.depth + (size_t)y1 * p.depth_w;
        }
        float t[8][8];
        auto ld_nc = [](const float* q) -> float { float v; asm volatile("ld.global.nc.f32 %0, [%1];" : "=f"(v) : "l"(q)); return v; };
#pragma unroll
        for (int r = 0; r < 8; ++r) {
            t[r][0] = ld_nc(r0[r] + xa0); t[r][1] = ld_nc(r0[r] + xa1); t[r][2] = ld_nc(r1[r] + xa0); t[r][3] = ld_nc(r1[r] + xa1);
            t[r][4] = ld_nc(r0[r] + xb0); t[r][5] = ld_nc(r0[r] + xb1); t[r][6] = ld_nc(r1[r] + xb0); t[r][7] = ld_nc(r1[r] + xb1);
        }
#pragma unroll
        for (int r = 0; r < 8; ++r) {
            va[r] = fminf(fminf(t[r][0], t[r][1]), fminf(t[r][2], t[r][3]));
            vb[r] = fminf(fminf(t[r][4], t[r][5]), fminf(t[r][6], t[r][7]));
        }
    }
    ORBIT_TRACE_STAMP(p.trace, 4, 1 + 0 * (uint32_t)(va[7] + vb[7] > 2.0f));
    {
        float* l0 = p.texels + p.level_offset[0];
#pragma unroll
        for (int r = 0; r < 8; ++r)
            *reinterpret_cast<float2*>(l0 + (size_t)(y_base + r) * p.width + x_a) = make_float2(va[r], vb[r]);
    }
    // ---- level 1: 4 rows x 32 columns per warp, one texel per lane per row
    float l1[4];
    {
        const uint32_t w1 = p.width >> 1;
        float* d = p.texels + p.level_offset[1];
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            l1[r] = fminf(fminf(va[2 * r], vb[2 * r]), fminf(va[2 * r + 1], vb[2 * r + 1]));
            d[(size_t)((y_base >> 1) + r) * w1 + (tx * 32u + lane)] = l1[r];
        }
    }
    // ---- level 2: 2 rows x 16 columns per warp (even lanes hold the result)
    float l2[2];
    {
        const uint32_t w2 = p.width >> 2;
        float* d = p.texels + p.level_offset[2];
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            float v = fminf(l1[2 * r], l1[2 * r + 1]);
            l2[r] = fminf(v, __shfl_xor_sync(0xFFFFFFFFu, v, 1));
            if ((lane & 1u) == 0u) d[(size_t)((y_base >> 2) + r) * w2 + (tx * 16u + (lane >> 1))] = l2[r];
        }
    }
    // ---- level 3: 1 row x 8 columns per warp (lanes 0,4,8,.. hold the result)
    float l3;
    {
        const uint32_t w3 = p.width >> 3;
        float v = fminf(l2[0], l2[1]);
        l3 = fminf(v, __shfl_xor_sync(0xFFFFFFFFu, v, 2));
        if ((lane & 3u) == 0u) {
            p.texels[p.level_offset[3] + (size_t)(y_base >> 3) * w3 + (tx * 8u + (lane >> 2))] = l3;
            s_l3[warp][lane >> 2] = l3;
        }
    }
    __syncthreads();
    // ---- levels 4..6 of the tile by warp 0: 4x4, 2x2, 1x1
    if (warp == 0u) {
        const uint32_t x4 = lane & 3u, y4 = (lane >> 2) & 3u;  // lanes 0..15 meaningful
        float v4 = fminf(fminf(s_l3[2 * y4][2 * x4], s_l3[2 * y4][2 * x4 + 1]), fminf(s_l3[2 * y4 + 1][2 * x4], s_l3[2 * y4 + 1][2 * x4 + 1]));
        if (lane < 16u) p.texels[p.level_offset[4] + (size_t)(ty * 4u + y4) * (p.width >> 4) + (tx * 4u + x4)] = v4;
        // level 5: combine x pairs (xor 1) and y pairs (xor 4)
        float v5 = fminf(v4, __shfl_xor_sync(0xFFFFFFFFu, v4, 1));
        v5 = fminf(v5, __shfl_xor_sync(0xFFFFFFFFu, v5, 4));
        if (lane < 16u && (lane & 5u) == 0u)
            p.texels[p.level_offset[5] + (size_t)(ty * 2u + (y4 >> 1)) * (p.width >> 5) + (tx * 2u + (x4 >> 1))] = v5;
        float v6 = fminf(v5, __shfl_xor_sync(0xFFFFFFFFu, v5, 2));
        v6 = fminf(v6, __shfl_xor_sync(0xFFFFFFFFu, v6, 8));
        if (lane == 0u) p.texels[p.level_offset[6] + (size_t)ty * (p.width >> 6) + tx] = v6;
    }
    ORBIT_TRACE_STAMP(p.trace, 4, 2);
    pdl_launch_dependents();
    if (p.levels <= 7u) return;
    // ---- remaining small levels: last CTA to arrive
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned int prev = atomicAdd(p.ticket, 1u);
        s_last = (prev + 1u == gridDim.x);
        if (s_last) *p.ticket = 0u;
    }
    __syncthreads();
    ORBIT_TRACE_STAMP(p.trace, 4, 3);
    if (!s_last) return;
    __threadfence();
    if ((p.width >> 6) * (p.height >> 6) <= 4096u) hiz_tail_smem(p, 7u, s_top_a, s_top_b);
    else hiz_tail(p, 7u);
    ORBIT_TRACE_STAMP(p.trace, 4, 4);
}

__global__ void __launch_bounds__(256) hiz_build_kernel(const __grid_constant__ HizBuildParams p) { hiz_build_body(p); }

// orbit_hiz_build_views: pyramid blockIdx.y; each has its own ticket, so each row's last CTA reduces that pyramid's top levels
__global__ void __launch_bounds__(256) hiz_build_views_kernel(const __grid_constant__ HizBuildViewsParams pv) { hiz_build_body(pv.view[blockIdx.y]); }
__global__ void __launch_bounds__(256) hiz_small_views_kernel(const __grid_constant__ HizBuildViewsParams pv) {
    pdl_wait();
    hiz_tail(pv.view[blockIdx.y], 0u);
}

cudaError_t launch_hiz_build(const HizBuildParams& p, cudaStream_t stream) {
    if (p.width >= 64u && p.height >= 64u && p.levels >= 7u) {
        const uint32_t grid = (p.width >> 6) * (p.height >> 6);
        return launch_kernel(hiz_build_kernel, dim3(grid), dim3(256), 0, stream, p);
    } else {
        return launch_kernel(hiz_small_kernel, dim3(1), dim3(256), 0, stream, p);
    }
    return cudaGetLastError();
}

cudaError_t launch_hiz_build_views(const HizBuildViewsParams& pv, cudaStream_t stream) {
    const HizBuildParams& p = pv.view[0];   // every pyramid of the call has this geometry
    if (p.width >= 64u && p.height >= 64u && p.levels >= 7u)
        return launch_kernel(hiz_build_views_kernel, dim3((p.width >> 6) * (p.height >> 6), pv.n_views), dim3(256), 0, stream, pv);
    return launch_kernel(hiz_small_views_kernel, dim3(1, pv.n_views), dim3(256), 0, stream, pv);
}

}  // namespace orbit
