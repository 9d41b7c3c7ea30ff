// orbit_device.cuh — device-side leaf arithmetic of the visibility pipeline (sm_100a).
//
// Implements the pinned arithmetic contract of DESIGN.md §3 with explicit round-to-nearest intrinsics, so the
// result does not depend on -fmad / -prec-div / -prec-sqrt: every product and sum is individually rounded
// (__fmul_rn/__fadd_rn are never contracted by ptxas), fused multiply-add appears only where the reference's
// shipped SPIR-V has GLSL.std.450 Fma, division and square root are IEEE (__fdiv_rn/__fsqrt_rn).
// Reference sources restated here: shaders/entity_cull.comp:28-43,83-102,146-191 and
// shaders/meshlet_cull.comp:28-43,83-106,160-205 (sphere transform, Mara/McGuire projection, occlusion block),
// shaders/light_cluster/cluster_common.glsl:18-20 (depth slice).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/orbit_cuda.h"

namespace orbit {

#define ORBIT_DEV __device__ __forceinline__

#ifndef ORBIT_EXPERIMENT_FAST_MATH
ORBIT_DEV float mul(float a, float b) { return __fmul_rn(a, b); }
ORBIT_DEV float add(float a, float b) { return __fadd_rn(a, b); }
ORBIT_DEV float sub(float a, float b) { return __fsub_rn(a, b); }
ORBIT_DEV float fdiv(float a, float b) { return __fdiv_rn(a, b); }
ORBIT_DEV float fsqrt(float a) { return __fsqrt_rn(a); }
ORBIT_DEV float fma_(float a, float b, float c) { return __fmaf_rn(a, b, c); }
#else
// EXPERIMENT ONLY (never shipped, results are NOT bit-exact): contraction allowed, approximate division and square
// root — used once to measure what the pinned arithmetic contract costs (profiles/r1_contract_cost.txt).
ORBIT_DEV float mul(float a, float b) { return a * b; }
ORBIT_DEV float add(float a, float b) { return a + b; }
ORBIT_DEV float sub(float a, float b) { return a - b; }
ORBIT_DEV float fdiv(float a, float b) { return __fdividef(a, b); }
ORBIT_DEV float fsqrt(float a) { return __frsqrt_rn(a) * a; }
ORBIT_DEV float fma_(float a, float b, float c) { return fmaf(a, b, c); }
#endif

ORBIT_DEV float dot3(float ax, float ay, float az, float bx, float by, float bz) {
    return add(add(mul(ax, bx), mul(ay, by)), mul(az, bz));
}

// Model-view matrix of one dispatch record / entity draw, column-major m[col*4+row], plus the largest column
// scale (largest_scale_from_matrix, meshlet_cull.comp:28-35).
struct ModelView {
    float m[16];
    float scale;
};

ORBIT_DEV float largest_scale(const float* m) {
    float xx = dot3(m[0], m[1], m[2], m[0], m[1], m[2]);
    float yy = dot3(m[4], m[5], m[6], m[4], m[5], m[6]);
    float zz = dot3(m[8], m[9], m[10], m[8], m[9], m[10]);
    return fsqrt(fmaxf(xx, fmaxf(yy, zz)));
}

// (M * (x,y,z,w))[row]
ORBIT_DEV float mat_row(const float* m, int row, float x, float y, float z, float w) {
    return add(add(add(mul(m[0 + row], x), mul(m[4 + row], y)), mul(m[8 + row], z)), mul(m[12 + row], w));
}

struct Sphere {
    float x, y, z;   // view-space centre
    float r;         // rounded r_model * scale
    float r_model;   // model-space radius (three later uses take the unrounded product through Fma)
    float s;         // scale
};

ORBIT_DEV Sphere transform_sphere(const ModelView& mv, float cx, float cy, float cz, float r_model) {
    Sphere o;
    float px = mat_row(mv.m, 0, cx, cy, cz, 1.0f);
    float py = mat_row(mv.m, 1, cx, cy, cz, 1.0f);
    float pz = mat_row(mv.m, 2, cx, cy, cz, 1.0f);
    float pw = mat_row(mv.m, 3, cx, cy, cz, 1.0f);
    if (pw != 1.0f) {  // x/1 == x exactly, so skipping the IEEE division is bit-identical (affine matrices)
        px = fdiv(px, pw); py = fdiv(py, pw); pz = fdiv(pz, pw);
    }
    o.x = px; o.y = py; o.z = pz;
    o.r_model = r_model; o.s = mv.scale;
    o.r = mul(r_model, mv.scale);
    return o;
}

ORBIT_DEV bool frustum_test(const OrbitCullInfo& ci, const Sphere& s) {
    bool visible = true;
    const float nr = -s.r;
    const uint32_t n = ci.cull_plane_count;
#pragma unroll 1
    for (uint32_t i = 0; i < n; ++i) {
        float d = add(dot3(ci.cull_planes[i][0], ci.cull_planes[i][1], ci.cull_planes[i][2], s.x, s.y, s.z),
                      ci.cull_planes[i][3]);
        visible = visible && (d > nr);
    }
    return visible;
}

// Nearest-mip level of lod = log2(x), exact on exponent / mantissa (no log2 evaluation), clamped to [0, levels-1].
// Branch-free: x <= 0 / NaN / denormal -> 0, +inf -> levels-1; for a normal x = m * 2^e the level is e + (m > fl(sqrt 2)),
// and adding (0x800000 - 0x3504F4) to the bit pattern carries into the exponent exactly when the 23 mantissa bits exceed
// those of fl(sqrt 2) = 0x3FB504F3. (Was ~20 instructions with three branches; the oracle keeps the branching form.)
ORBIT_DEV uint32_t hiz_level(float x, uint32_t levels) {
    const float xc = fmaxf(x, 0.0f);                                  // NaN, negatives, -0 -> +-0
    const int k = ((int)(__float_as_uint(xc) + 0x004AFB0Cu) >> 23) - 127;
    return (uint32_t)min(max(k, 0), (int)levels - 1);
}

// Depth pyramid as the kernels see it: one linear allocation, levels back to back. Level sizes are powers of two
// (orbit_hiz_geometry: npot(depth)/2), which the sampling code below relies on.
struct HizDevice {
    const float* texels;
    uint32_t width, height, levels;
    uint32_t level_offset[ORBIT_HIZ_MAX_LEVELS];
};

// Texel indices i0, i1 of the bilinear footprint along one axis of a level whose size is 2^lw (as float: wf):
//   fx = u*w - 0.5; i0 = floor(fx); i1 = i0 + 1, both clamped to [0, w-1]   (NaN -> the pair (0, 0))
// fmaxf(fx, -1) maps NaN and everything below -1 to -1, fminf(., w) everything above w to w, so the conversion cannot
// overflow and the clamps are two integer min/max.
ORBIT_DEV void footprint(float u, float wf, int hi, int& i0, int& i1) {
    const float fx = sub(mul(u, wf), 0.5f);
    const int a = __float2int_rd(fminf(fmaxf(fx, -1.0f), wf));      // in [-1, w]
    i0 = min(max(a, 0), hi);
    i1 = min(a + 1, hi);
}

ORBIT_DEV void footprint(float u, uint32_t w, int& i0, int& i1) { footprint(u, (float)w, (int)w - 1, i0, i1); }   // any size (depth buffer)

// Depth texel (x, y) of a depth image (orbit_depth_image_wrap's texture: unnormalised, point, clamp, element type): an
// unfiltered integer-coordinate load (TLD.LZ, the texelFetch analogue). tex2D<float> at texel centres would be a filtered
// TEX instead. `volatile` keeps a run of these fetches in program order, like the level-0 loads of the linear source.
ORBIT_DEV float depth_texel(cudaTextureObject_t t, int x, int y) {
    float4 v;   // one channel: .y .z .w are not read
    asm volatile("tex.2d.v4.f32.s32 {%0, %1, %2, %3}, [%4, {%5, %6}];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(t), "r"(x), "r"(y));
    return v.x;
}
// depth_texel when `fetch` is set (a predicated load), else 0
ORBIT_DEV float depth_texel_if(cudaTextureObject_t t, int x, int y, bool fetch) {
    float4 v = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    asm volatile("{ .reg .pred q; setp.ne.b32 q, %7, 0; @q tex.2d.v4.f32.s32 {%0, %1, %2, %3}, [%4, {%5, %6}]; }"
                 : "+f"(v.x), "+f"(v.y), "+f"(v.z), "+f"(v.w) : "l"(t), "r"(x), "r"(y), "r"((int)fetch));
    return v.x;
}

// ReduceMin sampler (device.rs:1404-1420) on level `lvl`: min of the 2x2 bilinear footprint, read through the
// non-coherent (texture / L1) path with 32-bit texel indices.
ORBIT_DEV float hiz_sample(const HizDevice& hz, uint32_t lw0, uint32_t lh0, uint32_t lvl, float u, float v) {
    const uint32_t lw = lw0 > lvl ? lw0 - lvl : 0u, lh = lh0 > lvl ? lh0 - lvl : 0u;   // log2 of the level's size
    const float wf = __uint_as_float((127u + lw) << 23), hf = __uint_as_float((127u + lh) << 23);
    int x0, x1, y0, y1;
    footprint(u, wf, (int)((1u << lw) - 1u), x0, x1);
    footprint(v, hf, (int)((1u << lh) - 1u), y0, y1);
    const uint32_t base = hz.level_offset[lvl];
    const uint32_t r0 = base + ((uint32_t)y0 << lw), r1 = base + ((uint32_t)y1 << lw);
    const float a = __ldg(hz.texels + (r0 + (uint32_t)x0)), b = __ldg(hz.texels + (r0 + (uint32_t)x1));
    const float c = __ldg(hz.texels + (r1 + (uint32_t)x0)), d = __ldg(hz.texels + (r1 + (uint32_t)x1));
    return fminf(fminf(a, b), fminf(c, d));
}

// Occlusion block of the entity stage, in two halves: occlusion_project computes everything up to the pyramid level and
// the footprint's centre (no pyramid texel is read), occlusion_sample samples the level (hiz_sample) and compares. occlusion_test is the two
// in a row. In the perspective case s.z is negated in place (the entity stage's LOD distance later reads the negated
// value, as in the reference).
struct HizProbe {
    bool sample;     // false: visible without a texel (sphere not entirely beyond the near plane, unknown projection type)
    float depth;     // the sphere's nearest depth
    uint32_t lvl;    // pyramid level to sample
    float u, v;      // footprint centre
};

// kProj: 0 perspective, 1 orthographic, -1 decided at run time from ci.projection_type.
template <int kProj = -1>
ORBIT_DEV HizProbe occlusion_project(const OrbitCullInfo& ci, Sphere& s, const HizDevice& hz, const uint32_t hiz_lw, const uint32_t hiz_lh) {
    HizProbe q;
    q.sample = false;
    float ax, ay, az, aw, depth;
    const uint32_t proj = kProj >= 0 ? (uint32_t)kProj : ci.projection_type;
    if (proj == 0u) {
        float zp = -s.z;
        s.z = zp;
        bool cullable = zp >= fma_(s.r_model, s.s, ci.z_near);
        if (!cullable) return q;  // visible stays true; nothing below has side effects
        float P00 = ci.p00_or_width_recip_x2, P11 = ci.p11_or_height_recip_x2;
        float r = s.r, nr = -s.r;
        float c0 = -s.x, c1 = -zp;
        float zz = mul(c1, c1);
        float sx = fsqrt(fma_(nr, r, add(mul(c0, c0), zz)));
        float minx0 = add(mul(sx, c0), mul(nr, c1)), minx1 = add(mul(r, c0), mul(sx, c1));
        float maxx0 = add(mul(sx, c0), mul(r, c1)), maxx1 = add(mul(nr, c0), mul(sx, c1));
        float d0 = -s.y;
        float sy = fsqrt(fma_(nr, r, add(mul(d0, d0), zz)));
        float miny0 = add(mul(sy, d0), mul(nr, c1)), miny1 = add(mul(r, d0), mul(sy, c1));
        float maxy0 = add(mul(sy, d0), mul(r, c1)), maxy1 = add(mul(nr, d0), mul(sy, c1));
        float a0 = mul(fdiv(minx0, minx1), P00), a1 = mul(fdiv(miny0, miny1), P11);
        float a2 = mul(fdiv(maxx0, maxx1), P00), a3 = mul(fdiv(maxy0, maxy1), P11);
        ax = fma_(a0, 0.5f, 0.5f); ay = fma_(a3, -0.5f, 0.5f);
        az = fma_(a2, 0.5f, 0.5f); aw = fma_(a1, -0.5f, 0.5f);
        depth = fdiv(ci.z_near, fma_(-s.r_model, s.s, zp));
    } else if (proj == 1u) {
        float sr = ci.p00_or_width_recip_x2;
        float ctrx = mul(s.x, sr), ctry = mul(s.y, sr);
        float box = mul(sr, s.r);
        float b0 = fma_(box, -1.0f, ctrx), b1 = fma_(box, -1.0f, ctry);
        float b2 = fma_(box, 1.0f, ctrx), b3 = fma_(box, 1.0f, ctry);
        b0 = fminf(fmaxf(b0, -1.0f), 1.0f); b1 = fminf(fmaxf(b1, -1.0f), 1.0f);
        b2 = fminf(fmaxf(b2, -1.0f), 1.0f); b3 = fminf(fmaxf(b3, -1.0f), 1.0f);
        ax = fma_(b0, 0.5f, 0.5f); ay = fma_(b1, -0.5f, 0.5f);
        az = fma_(b2, 0.5f, 0.5f); aw = fma_(b3, -0.5f, 0.5f);
        float k = fdiv(1.0f, sub(ci.z_far, ci.z_near));
        depth = mul(k, add(fma_(s.r_model, s.s, s.z), ci.z_far));
    } else {
        return q;
    }
    float W = mul(sub(az, ax), (float)hz.width);
    float H = mul(sub(aw, ay), (float)hz.height);
    float u = mul(add(ax, az), 0.5f), v = mul(add(ay, aw), 0.5f);
    uint32_t lvl = hiz_level(fmaxf(W, H), hz.levels);
    q.sample = true;
    q.depth = depth; q.lvl = lvl; q.u = u; q.v = v;
    return q;
}
ORBIT_DEV bool occlusion_sample(const HizProbe& q, const HizDevice& hz, const uint32_t hiz_lw, const uint32_t hiz_lh) {
    if (!q.sample) return true;
    float sampled = hiz_sample(hz, hiz_lw, hiz_lh, q.lvl, q.u, q.v);
    return q.depth >= sampled;
}
template <int kProj = -1>
ORBIT_DEV bool occlusion_test(const OrbitCullInfo& ci, Sphere& s, const HizDevice& hz, const uint32_t hiz_lw, const uint32_t hiz_lh) {
    return occlusion_sample(occlusion_project<kProj>(ci, s, hz, hiz_lw, hiz_lh), hz, hiz_lw, hiz_lh);
}
ORBIT_DEV uint32_t hiz_log2(uint32_t n) { return 31u - (uint32_t)__clz((int)max(n, 1u)); }   // of a level-0 side (a power of two)
template <int kProj = -1>
ORBIT_DEV bool occlusion_test(const OrbitCullInfo& ci, Sphere& s, const HizDevice& hz) {
    return occlusion_test<kProj>(ci, s, hz, hiz_log2(hz.width), hiz_log2(hz.height));
}

// Loads that are issued where they are written. In the latency-bound kernels the order of the independent loads is
// the schedule: left alone, nvcc AND ptxas sink a prefetch below arithmetic that waits on an earlier load (register
// pressure heuristic), turning two overlapped round trips into two dependent ones. PTX `ld.volatile` operations keep
// their program order among themselves, so a chain "prefetches first, the load the next instruction needs last" pins
// all of them before the first use. (Volatile loads are served by L2, which is where this single-use data lives.)
ORBIT_DEV uint4 ld_v4_ordered(const void* p) {
    uint4 v;
    asm volatile("ld.volatile.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
    return v;
}
ORBIT_DEV uint32_t ld_u32_ordered(const void* p) {
    uint32_t v;
    asm volatile("ld.volatile.global.u32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}
ORBIT_DEV float4 as_float4(uint4 v) { return make_float4(__uint_as_float(v.x), __uint_as_float(v.y), __uint_as_float(v.z), __uint_as_float(v.w)); }

// ConvertFToU pinned: NaN/negative -> 0, >= 2^32 -> 0xFFFFFFFF (cvt.rzi.u32.f32 saturates exactly like this).
ORBIT_DEV uint32_t f2u(float f) { return __float2uint_rz(f); }
ORBIT_DEV uint32_t shl1(uint32_t s) { return s >= 32u ? 0u : (1u << s); }

// Contract log2 (DESIGN.md §3): identical algorithm to the oracle's, restated.
ORBIT_DEV float orbit_log2f(float x) {
    uint32_t u = __float_as_uint(x);
    if ((u << 1) == 0u) return __uint_as_float(0xFF800000u);
    if (u >> 31) return __uint_as_float(0x7FC00000u);
    if (u >= 0x7F800000u) return x;
    int e = 0;
    if (u < 0x00800000u) { x = mul(x, 8388608.0f); u = __float_as_uint(x); e = -23; }
    e += (int)(u >> 23) - 127;
    float m = __uint_as_float((u & 0x007FFFFFu) | 0x3F800000u);
    if (m > 1.41421354f) { m = mul(m, 0.5f); e += 1; }
    float t = fdiv(sub(m, 1.0f), add(m, 1.0f));
    float s = mul(t, t);
    float p = 0.3205986261f;
    p = fma_(s, p, 0.4121982336f);
    p = fma_(s, p, 0.5770775080f);
    p = fma_(s, p, 0.9617958665f);
    p = fma_(s, p, 2.8853900433f);
    return add((float)e, mul(t, p));
}

}  // namespace orbit
