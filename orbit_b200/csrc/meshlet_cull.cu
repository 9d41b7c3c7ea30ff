// meshlet_cull.cu — per-meshlet frustum / normal-cone / two-pass Hi-Z culling + ordered compaction (sm_100a).
//
// Stands in for shaders/meshlet_cull.comp:108-255 driven by create_meshlet_draw_commands
// (src/passes/draw_gen.rs:382-435) and, for the optional task payload output, the task-shader twins
// (shaders/forward/forward_depth_prepass.task:224-256).
//
// B200 design (not the reference's one-workgroup-per-record + atomicAdd). Measured on C2 the stage is bound by
// instruction issue before HBM (IEEE-exact division / square root of the projection math), so the design
// minimises executed warp-instructions and never blocks a CTA:
//   * TWO launches. `meshlet_test_kernel` is embarrassingly parallel: persistent warps take tiles of R records
//     CYCLICALLY (tile = global warp id + k * total warps), test every lane and leave one draw mask per record in
//     an L2-resident scratch array — no inter-CTA ordering at all, so hot regions of the scene are spread over
//     all SMs (a contiguous static split measured 2-3x slower: the CTAs owning the visible part of the city made
//     everyone wait). `meshlet_emit_kernel` then orders and writes the survivors: contiguous record ranges per
//     CTA, popcount sums, ONE published aggregate per CTA, a flat gather of all lower aggregates (no hop-by-hop
//     look-back: that propagates only 32 tiles per L2 round trip and dominated v1/v2), and the commands are
//     rebuilt from 16 B of each surviving meshlet (L2 hits). The record count is read on the device (the
//     reference's dispatch_indirect) — no host round trip;
//   * lane = meshlet of a record, exactly the reference's 32-lane group, so ballots are the reference's
//     visibility words; the meshlets of a tile (R records x 1 KB contiguous) are staged into shared memory by
//     TMA bulk copies (cp.async.bulk + mbarrier, one copy per record issued by R lanes), so R KB per warp are in
//     flight without holding registers, and the next tile's copy is issued as soon as the current one is consumed;
//   * view*model is computed once per record by 16 lanes (two records per step) and broadcast through shared
//     memory — the reference recomputes the 4x4 product in every lane;
//   * pass 1: only lanes whose visibility bit is set can be visible, so they are PACKED across the tile's
//     records before any meshlet is loaded or tested (the early pass touches only last frame's survivors);
//   * pass 2: lanes surviving frustum + cone are PACKED into a per-warp queue and the expensive Hi-Z projection
//     runs on full warps of survivors instead of once per record at ~17% lane occupancy;
//   * survivors are ranked by ballot + popc; draw order = (record index, lane), independent of scheduling.
#include "params.cuh"

namespace orbit {

constexpr int kMcWarps = 8;
constexpr int kMcThreads = kMcWarps * 32;
constexpr int kMvStride = 20;   // 16 matrix entries + scale, padded
constexpr uint32_t kNone = 0xFFFFFFFFu;

struct ItemTest {
    Sphere s;
    bool pre_visible;   // passed frustum + cone
};

// frustum + cone for one meshlet against the model-view matrix (columns c0..c3, largest column scale `scale`)
// kProj: 0 perspective, 1 orthographic, -1 decided at run time from ci.projection_type. CI: OrbitCullInfo, or ViewCull (the
// fields this test reads, staged in shared memory by the batched packed kernel)
template <int kProj, typename CI>
__device__ __forceinline__ ItemTest test_item(const CI& ci, const float4 c0, const float4 c1, const float4 c2, const float4 c3,
                                              const float scale, const float cx, const float cy, const float cz, const float r_model,
                                              const uint32_t cone) {
    ItemTest out;
    // (M * (c,1))[row]; m3*1.0f == m3 exactly
    float px = add(add(add(mul(c0.x, cx), mul(c1.x, cy)), mul(c2.x, cz)), c3.x);
    float py = add(add(add(mul(c0.y, cx), mul(c1.y, cy)), mul(c2.y, cz)), c3.y);
    float pz = add(add(add(mul(c0.z, cx), mul(c1.z, cy)), mul(c2.z, cz)), c3.z);
    const float pw = add(add(add(mul(c0.w, cx), mul(c1.w, cy)), mul(c2.w, cz)), c3.w);
    if (pw != 1.0f) { px = fdiv(px, pw); py = fdiv(py, pw); pz = fdiv(pz, pw); }   // x/1 == x exactly
    Sphere& s = out.s;
    s.x = px; s.y = py; s.z = pz;
    s.r_model = r_model; s.s = scale;
    s.r = mul(s.r_model, scale);
    const float nr = -s.r;
    bool visible = true;
    const uint32_t n = ci.cull_plane_count;
    if (n == 5u) {
        // the main-view case (forward.rs:268 passes planes[0..5]): straight-line code, plane coefficients as constant-bank
        // operands, no loop control
#pragma unroll
        for (uint32_t i = 0; i < 5u; ++i) {
            const float d = add(dot3(ci.cull_planes[i][0], ci.cull_planes[i][1], ci.cull_planes[i][2], px, py, pz), ci.cull_planes[i][3]);
            visible = visible && (d > nr);
        }
    } else {
#pragma unroll 1
        for (uint32_t i = 0; i < n; ++i) {
            const float d = add(dot3(ci.cull_planes[i][0], ci.cull_planes[i][1], ci.cull_planes[i][2], px, py, pz), ci.cull_planes[i][3]);
            visible = visible && (d > nr);
        }
    }
    {
        // cone test: computed for every lane (no branch on `visible`: a warp nearly always has a visible lane, and the
        // branch + reconvergence cost more than the predicated-off work saved)
        const float K = 0.007874015718698502f;
        const float kx = mul((float)(int)(int8_t)(cone & 0xFFu), K);
        const float ky = mul((float)(int)(int8_t)((cone >> 8) & 0xFFu), K);
        const float kz = mul((float)(int)(int8_t)((cone >> 16) & 0xFFu), K);
        const float cutoff = mul((float)((int)cone >> 24), K);
        // (M * (k,0)).xyz: the w column contributes m3*0.0f (kept: +-0 / NaN propagate as in the oracle)
        const float axx = add(add(add(mul(c0.x, kx), mul(c1.x, ky)), mul(c2.x, kz)), mul(c3.x, 0.0f));
        const float axy = add(add(add(mul(c0.y, kx), mul(c1.y, ky)), mul(c2.y, kz)), mul(c3.y, 0.0f));
        const float axz = add(add(add(mul(c0.z, kx), mul(c1.z, ky)), mul(c2.z, kz)), mul(c3.z, 0.0f));
        const uint32_t proj = kProj >= 0 ? (uint32_t)kProj : ci.projection_type;
        if (proj == 0u) {
            const float lhs = dot3(px, py, pz, axx, axy, axz);
            const float len = fsqrt(dot3(px, py, pz, px, py, pz));
            visible = visible && !(lhs >= fma_(cutoff, len, s.r));
        } else if (proj == 1u) {
            const float camx = sub(px, 0.0f), camy = sub(py, 0.0f), camz = sub(pz, -1.0f);
            const float qx = sub(px, camx), qy = sub(py, camy), qz = sub(pz, camz);
            const float lhs = dot3(qx, qy, qz, axx, axy, axz);
            const float len = fsqrt(dot3(qx, qy, qz, qx, qy, qz));
            visible = visible && !(lhs >= fma_(cutoff, len, s.r));
        }
    }
    out.pre_visible = visible;
    return out;
}

__device__ __forceinline__ bool draw_rule(const OrbitCullInfo& ci, const MeshletCullParams& p, bool visible, bool vib, bool pass2,
                                          uint32_t packed) {
    if (!visible) return false;
    const uint32_t material_index = packed & 0xFFFFu;
    const uint32_t alpha = __ldg(reinterpret_cast<const uint32_t*>(
        p.materials + (size_t)material_index * ORBIT_MATERIAL_STRIDE_BYTES + ORBIT_MATERIAL_ALPHA_MODE_OFFSET));
    bool should_draw = (shl1(alpha) & ci.alpha_mode_flags) != 0u;
    if (pass2 && (shl1(alpha) & ci.noskip_alpha_mode) == 0u) should_draw = !vib;   // overrides the alpha filter (meshlet_cull.comp:210-213)
    return should_draw;
}

__device__ __forceinline__ void store_command(uint32_t* __restrict__ dst, uint32_t vertex_offset, uint32_t data_offset, uint32_t packed,
                                              uint32_t entity, uint32_t meshlet_index) {
    dst[0] = (packed >> 24) * 3u;                              // triangle_count * 3
    dst[1] = 1u;
    dst[2] = (data_offset + ((packed >> 16) & 0xFFu)) * 4u;    // (data_offset + vertex_count) * 4
    dst[3] = data_offset;
    dst[4] = entity;
    dst[5] = vertex_offset;
    dst[6] = meshlet_index;
}

// Survivor counts are accumulated per CHUNK of consecutive records by the test kernel (integer atomics: the sums are
// order-independent) so that the emit kernel can order its output with a shared-memory scan instead of an
// inter-CTA exchange. Chunk size: a power of two >= 32 records such that there are at most kMaxChunks chunks.
constexpr uint32_t kMaxChunks = 2048u;
__device__ __forceinline__ uint32_t chunk_shift_of(uint32_t nrec) {
    const uint32_t per = (nrec + kMaxChunks - 1u) / kMaxChunks;            // records per chunk needed, >= 0
    const uint32_t sh = per <= 1u ? 0u : 32u - (uint32_t)__clz((int)(per - 1u));   // ceil(log2(per))
    return max(5u, sh);
}

// ---- asynchronous global -> shared copies (cp.async, SASS: LDGSTS + LDGDEPBAR / DEPBAR) -----------------------------
// The stream kernel prefetches through shared memory, NOT through registers: a register prefetch carried around the
// loop ties the data to one of the six SASS scoreboards, and ptxas put a wait on that scoreboard ~100 instructions
// after the loads were issued (measured: 12 % of all warp time in one FMUL, profiles/r2_meshlet_test_history.txt) —
// a warp then exposes a full DRAM latency per record. cp.async completion is tracked by its own group counter.
__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void cp_async_16_stream(uint32_t dst, const void* src, uint64_t policy) {
    asm volatile("cp.async.cg.shared.global.L2::cache_hint [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "l"(policy) : "memory");
}
__device__ __forceinline__ void cp_async_16(uint32_t dst, const void* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_4(uint32_t dst, const void* src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ uint64_t l2_evict_first_policy() {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ void sts32(uint32_t addr, uint32_t v) { asm volatile("st.shared.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory"); }
__device__ __forceinline__ uint32_t lds32(uint32_t addr) { uint32_t v; asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory"); return v; }
__device__ __forceinline__ uint4 lds128(uint32_t addr) {
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr) : "memory");
    return v;
}

// ---- packed binary32 pairs (sm_100: FMUL2 / FFMA2, PTX mul.rn.f32x2 / fma.rn.f32x2) ------------------------------------
// Instruction issue, not HBM, bounds the meshlet test, so the multiplies / adds / fmas of the pinned arithmetic contract
// are issued two at a time wherever two independent values go through the same operation. Each half is rounded exactly
// like the scalar operation (IEEE round-to-nearest per component), so results stay bit-identical to the
// scalar oracle — PROVIDED nothing is contracted: ptxas 12.9 fuses mul.rn.f32x2 + add.rn.f32x2 into FFMA2 even under
// -fmad=false (it does not do that to the scalar .rn forms). The packed ADD is therefore never emitted: a + b is issued
// as fma(a, ONE, b) and a - b as fma(b, MINUS_ONE, a) with ONE / MINUS_ONE read from the kernel parameters (the compiler
// cannot know their values, so there is no multiply-add pair left to contract; the single rounding of the fma equals the
// rounding of the sum). tests/test_gpu_packed_math.py compares the packed leaf functions with the scalar ones bit for bit.
struct PkConsts { float2 one, mone; };
ORBIT_DEV float2 pk(float a, float b) { return make_float2(a, b); }
ORBIT_DEV float2 pmul(float2 a, float2 b) { return __fmul2_rn(a, b); }
ORBIT_DEV float2 pmuls(float2 a, float s) { return __fmul2_rn(a, make_float2(s, s)); }
ORBIT_DEV float2 pfma(float2 a, float2 b, float2 c) { return __ffma2_rn(a, b, c); }
ORBIT_DEV float2 padd(const PkConsts& k, float2 a, float2 b) { return __ffma2_rn(a, k.one, b); }
ORBIT_DEV float2 psub(const PkConsts& k, float2 a, float2 b) { return __ffma2_rn(b, k.mone, a); }
ORBIT_DEV float2 pneg(const PkConsts& k, float2 a) { return __fmul2_rn(a, k.mone); }
ORBIT_DEV float2 pdot3(const PkConsts& k, float2 ax, float2 ay, float2 az, float2 bx, float2 by, float2 bz) {
    return padd(k, padd(k, pmul(ax, bx), pmul(ay, by)), pmul(az, bz));
}
ORBIT_DEV float2 psqrt(float2 a) { return make_float2(fsqrt(a.x), fsqrt(a.y)); }
ORBIT_DEV float2 pdiv(float2 a, float2 b) { return make_float2(fdiv(a.x, b.x), fdiv(a.y, b.y)); }

// test_item with the arithmetic packed two-wide ACROSS COMPONENTS of one meshlet: the (x, y) and (z, w) rows of the
// transform, two cull planes at a time (coefficients pre-paired on the host: MeshletCullParams::planes_t), the (x, y)
// rows of the cone axis. The matrix columns come out of shared memory as natural (x, y) / (z, w) pairs and the meshlet's
// scalars are broadcast operands, so no register pairs have to be assembled. Same operations, same order, same rounding
// per component as test_item (pinned by tests/test_gpu_packed_math.py and by the parity suite).
struct ItemXY { float2 pxy; float pz, r; bool pre_visible; };
ORBIT_DEV float2 lo2(const float4 v) { return make_float2(v.x, v.y); }
ORBIT_DEV float2 hi2(const float4 v) { return make_float2(v.z, v.w); }

template <int kProj>
__device__ __forceinline__ ItemXY test_item_xy(const OrbitCullInfo& ci, const MeshletCullParams& p, const PkConsts& k, const float4 c0, const float4 c1,
                                              const float4 c2, const float4 c3, const float scale, const float cx, const float cy, const float cz,
                                              const float r_model, const uint32_t cone) {
    ItemXY out;
    // (M * (c,1)) rows (x,y) and (z,w); m3*1.0f == m3 exactly
    float2 pxy = padd(k, padd(k, padd(k, pmuls(lo2(c0), cx), pmuls(lo2(c1), cy)), pmuls(lo2(c2), cz)), lo2(c3));
    const float2 pzw = padd(k, padd(k, padd(k, pmuls(hi2(c0), cx), pmuls(hi2(c1), cy)), pmuls(hi2(c2), cz)), hi2(c3));
    float pz = pzw.x;
    if (pzw.y != 1.0f) { pxy.x = fdiv(pxy.x, pzw.y); pxy.y = fdiv(pxy.y, pzw.y); pz = fdiv(pz, pzw.y); }   // x/1 == x exactly
    const float r = mul(r_model, scale);
    out.pxy = pxy; out.pz = pz; out.r = r;
    bool visible = true;
    const uint32_t n = ci.cull_plane_count;
    if (n == 5u) {
        // the main-view case (forward.rs:268 passes planes[0..5]): straight-line code; the sixth slot repeats plane 4
#pragma unroll
        for (uint32_t j = 0; j < 3u; ++j) {
            const float2 d = padd(k, padd(k, padd(k, pmuls(p.planes_t[j][0], pxy.x), pmuls(p.planes_t[j][1], pxy.y)), pmuls(p.planes_t[j][2], pz)), p.planes_t[j][3]);
            visible = visible && (d.x > -r) && (d.y > -r);
        }
    } else {
        const uint32_t np = (n + 1u) >> 1;
#pragma unroll 1
        for (uint32_t j = 0; j < np; ++j) {
            const float2 d = padd(k, padd(k, padd(k, pmuls(p.planes_t[j][0], pxy.x), pmuls(p.planes_t[j][1], pxy.y)), pmuls(p.planes_t[j][2], pz)), p.planes_t[j][3]);
            visible = visible && (d.x > -r) && (d.y > -r);
        }
    }
    {
        const float K = 0.007874015718698502f;
        const float kx = mul((float)(int)(int8_t)(cone & 0xFFu), K);
        const float ky = mul((float)(int)(int8_t)((cone >> 8) & 0xFFu), K);
        const float kz = mul((float)(int)(int8_t)((cone >> 16) & 0xFFu), K);
        const float cutoff = mul((float)((int)cone >> 24), K);
        // (M * (k,0)).xyz: the w column contributes m3*0.0f (kept: +-0 / NaN propagate as in the oracle)
        const float2 axy = padd(k, padd(k, padd(k, pmuls(lo2(c0), kx), pmuls(lo2(c1), ky)), pmuls(lo2(c2), kz)), pmuls(lo2(c3), 0.0f));
        const float az = add(add(add(mul(c0.z, kx), mul(c1.z, ky)), mul(c2.z, kz)), mul(c3.z, 0.0f));
        const uint32_t proj = kProj >= 0 ? (uint32_t)kProj : ci.projection_type;
        if (proj == 0u) {
            const float2 t = pmul(pxy, axy), u = pmul(pxy, pxy);
            const float lhs = add(add(t.x, t.y), mul(pz, az));
            const float len = fsqrt(add(add(u.x, u.y), mul(pz, pz)));
            visible = visible && !(lhs >= fma_(cutoff, len, r));
        } else if (proj == 1u) {
            // camera = c - (0,0,-1); q = c - camera (two subtractions, not simplified: meshlet_cull.comp:150-156)
            const float2 camxy = psub(k, pxy, pk(0.0f, 0.0f));
            const float camz = sub(pz, -1.0f);
            const float2 qxy = psub(k, pxy, camxy);
            const float qz = sub(pz, camz);
            const float2 t = pmul(qxy, axy), u = pmul(qxy, qxy);
            const float lhs = add(add(t.x, t.y), mul(qz, az));
            const float len = fsqrt(add(add(u.x, u.y), mul(qz, qz)));
            visible = visible && !(lhs >= fma_(cutoff, len, r));
        }
    }
    out.pre_visible = visible;
    return out;
}

// occlusion_test (orbit_device.cuh) for two candidates at once: component .x = first, .y = second candidate.
// Returns bit 0 / bit 1 = candidate visible.
template <int kProj>
__device__ __forceinline__ uint32_t occlusion_pair(const OrbitCullInfo& ci, const PkConsts& k, const float2 x, const float2 y, const float2 z,
                                                  const float2 r_model, const float2 s, const HizDevice& hz, const uint32_t hiz_lw,
                                                  const uint32_t hiz_lh) {
    float2 ax, ay, az, aw, depth;
    bool cull_a = true, cull_b = true;        // cullable (perspective only)
    const float2 r = pmul(r_model, s);
    const uint32_t proj = kProj >= 0 ? (uint32_t)kProj : ci.projection_type;
    if (proj == 0u) {
        const float2 zp = pneg(k, z);
        const float2 lim = pfma(r_model, s, pk(ci.z_near, ci.z_near));
        cull_a = zp.x >= lim.x; cull_b = zp.y >= lim.y;
        const float P00 = ci.p00_or_width_recip_x2, P11 = ci.p11_or_height_recip_x2;
        const float2 nr = pneg(k, r);
        const float2 c0 = pneg(k, x), c1 = pneg(k, zp), d0 = pneg(k, y);
        const float2 zz = pmul(c1, c1);
        const float2 sx = psqrt(pfma(nr, r, padd(k, pmul(c0, c0), zz)));
        const float2 sy = psqrt(pfma(nr, r, padd(k, pmul(d0, d0), zz)));
        const float2 nrc1 = pmul(nr, c1), rc1 = pmul(r, c1);
        const float2 sxc0 = pmul(sx, c0), sxc1 = pmul(sx, c1), syd0 = pmul(sy, d0), syc1 = pmul(sy, c1);
        const float2 minx0 = padd(k, sxc0, nrc1), minx1 = padd(k, pmul(r, c0), sxc1);
        const float2 maxx0 = padd(k, sxc0, rc1), maxx1 = padd(k, pmul(nr, c0), sxc1);
        const float2 miny0 = padd(k, syd0, nrc1), miny1 = padd(k, pmul(r, d0), syc1);
        const float2 maxy0 = padd(k, syd0, rc1), maxy1 = padd(k, pmul(nr, d0), syc1);
        const float2 a0 = pmuls(pdiv(minx0, minx1), P00), a1 = pmuls(pdiv(miny0, miny1), P11);
        const float2 a2 = pmuls(pdiv(maxx0, maxx1), P00), a3 = pmuls(pdiv(maxy0, maxy1), P11);
        const float2 h = pk(0.5f, 0.5f), nh = pk(-0.5f, -0.5f);
        ax = pfma(a0, h, h); ay = pfma(a3, nh, h);
        az = pfma(a2, h, h); aw = pfma(a1, nh, h);
        depth = pdiv(pk(ci.z_near, ci.z_near), pfma(pneg(k, r_model), s, zp));
    } else if (proj == 1u) {
        const float sr = ci.p00_or_width_recip_x2;
        const float2 ctrx = pmuls(x, sr), ctry = pmuls(y, sr);
        const float2 box = pmuls(r, sr);
        const float2 one = pk(1.0f, 1.0f), mone = pk(-1.0f, -1.0f);
        float2 b0 = pfma(box, mone, ctrx), b1 = pfma(box, mone, ctry);
        float2 b2 = pfma(box, one, ctrx), b3 = pfma(box, one, ctry);
        b0 = pk(fminf(fmaxf(b0.x, -1.0f), 1.0f), fminf(fmaxf(b0.y, -1.0f), 1.0f));
        b1 = pk(fminf(fmaxf(b1.x, -1.0f), 1.0f), fminf(fmaxf(b1.y, -1.0f), 1.0f));
        b2 = pk(fminf(fmaxf(b2.x, -1.0f), 1.0f), fminf(fmaxf(b2.y, -1.0f), 1.0f));
        b3 = pk(fminf(fmaxf(b3.x, -1.0f), 1.0f), fminf(fmaxf(b3.y, -1.0f), 1.0f));
        const float2 h = pk(0.5f, 0.5f), nh = pk(-0.5f, -0.5f);
        ax = pfma(b0, h, h); ay = pfma(b1, nh, h);
        az = pfma(b2, h, h); aw = pfma(b3, nh, h);
        const float kk = fdiv(1.0f, sub(ci.z_far, ci.z_near));
        depth = pmuls(padd(k, pfma(r_model, s, z), pk(ci.z_far, ci.z_far)), kk);
    } else {
        return 3u;
    }
    const float2 W = pmuls(psub(k, az, ax), (float)hz.width);
    const float2 H = pmuls(psub(k, aw, ay), (float)hz.height);
    const float2 u = pmuls(padd(k, ax, az), 0.5f), v = pmuls(padd(k, ay, aw), 0.5f);
    uint32_t vis = 0u;
    {
        const uint32_t lvl = hiz_level(fmaxf(W.x, H.x), hz.levels);
        const float sampled = hiz_sample(hz, hiz_lw, hiz_lh, lvl, u.x, v.x);
        if (!cull_a || depth.x >= sampled) vis |= 1u;
    }
    {
        const uint32_t lvl = hiz_level(fmaxf(W.y, H.y), hz.levels);
        const float sampled = hiz_sample(hz, hiz_lw, hiz_lh, lvl, u.y, v.y);
        if (!cull_b || depth.y >= sampled) vis |= 2u;
    }
    return vis;
}
struct RecordWords { uint32_t ent, moff, cnt, vo; };

// Hi-Z test of `n` (<= 64) queued candidates starting at ring position qhead (even), two per lane; publishes the
// results (see the kernel comment) and returns the number of draws found by the warp. Inlined at its single call site (between tiles).
template <int kProj>
__device__ __forceinline__ uint32_t drain_candidates(const MeshletCullParams& p, const PkConsts& k, const uint32_t qbase, const uint32_t ring_mask, const uint32_t qhead,
                                                  const uint32_t n, uint32_t* const chunk_counts, const uint32_t chunk_shift,
                                                  const uint32_t hiz_lw, const uint32_t hiz_lh, const uint32_t lane,
                                                  uint32_t* const main_chunk_counts, uint32_t& main_drawn_out) {
    const OrbitCullInfo& ci = p.cull;
    const uint32_t cs4 = (ring_mask + 1u) * 4u;      // bytes between the component arrays of the ring
    // per lane: the record of its first visible candidate with the bits the lane contributes to that record's visibility word
    // / LATE entry / MAIN entry, and — when the lane's two candidates belong to different records — the second one apart
    uint32_t rec0 = 0xFFFFFFFFu, vo0 = 0u, vbits = 0u, lbits = 0u, mbits = 0u;
    uint32_t rec1 = 0xFFFFFFFFu, vo1 = 0u, vbit1 = 0u, lbit1 = 0u, mbit1 = 0u;
    if (2u * lane < n) {
        // candidates 2*lane and 2*lane+1 sit in adjacent slots (qhead is even: the ring advances by 64 or empties)
        const uint32_t qa = qbase + ((qhead + 2u * lane) & ring_mask) * 4u;
        float2 cx, cy, cz, crm, cs;
        asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(cx.x), "=f"(cx.y) : "r"(qa) : "memory");
        asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(cy.x), "=f"(cy.y) : "r"(qa + 1u * cs4) : "memory");
        asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(cz.x), "=f"(cz.y) : "r"(qa + 2u * cs4) : "memory");
        asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(crm.x), "=f"(crm.y) : "r"(qa + 3u * cs4) : "memory");
        asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(cs.x), "=f"(cs.y) : "r"(qa + 4u * cs4) : "memory");
        uint32_t vis = occlusion_pair<kProj>(ci, k, cx, cy, cz, crm, cs, p.hiz, hiz_lw, hiz_lh);
        if (2u * lane + 1u >= n) vis &= 1u;                               // odd tail: the second slot is stale
#pragma unroll
        for (uint32_t c = 0; c < 2u; ++c) {
            if ((vis >> c) & 1u) {
                const uint32_t rec = lds32(qa + 5u * cs4 + c * 4u), vo = lds32(qa + 6u * cs4 + c * 4u), id = lds32(qa + 7u * cs4 + c * 4u);
                const uint32_t bit = 1u << (id & 31u);
                // should_draw = visible && alpha passes the filter; in pass 2, unless the alpha mode is "noskip",
                // should_draw = visible && !visible_last_frame (this overrides the alpha filter, meshlet_cull.comp:207-213)
                const uint32_t abit = shl1(id >> 6);
                const bool draw = (abit & ci.noskip_alpha_mode) ? (abit & ci.alpha_mode_flags) != 0u : (id & 32u) == 0u;
                // fused MAIN pass: pass 1 over the bit being written, same camera — visible there is this `visible`, and
                // should_draw = visible && alpha passes the MAIN pass's filter (meshlet_cull.comp:137,207)
                const bool mdraw = main_chunk_counts != nullptr && (abit & p.main_alpha_mode_flags) != 0u;
                if (rec0 == 0xFFFFFFFFu || rec == rec0) {
                    rec0 = rec; vo0 = vo; vbits |= bit; if (draw) lbits |= bit; if (mdraw) mbits |= bit;
                } else {
                    rec1 = rec; vo1 = vo; vbit1 = bit; if (draw) lbit1 = bit; if (mdraw) mbit1 = bit;
                }
            }
        }
    }
    __syncwarp();
    // Publication, once per RECORD instead of once per candidate: the candidates of a drain are in record order, so the lanes
    // that found something mostly share two or three records. The lanes of a record OR their bits together (redux.or) and
    // the lowest of them issues one RED.OR per word — visibility word, LATE entry, MAIN entry — and one RED.ADD of the
    // popcount per list to the record's chunk counter (the bits of a record are distinct, so the popcount of the OR is the
    // number of survivors). Per-candidate atomics on the few dozen chunk counters of the visible part of the scene cost the
    // fused late pass of C2 10 us. A lane whose two candidates straddle a record boundary publishes the second one itself.
    uint32_t drawn = 0u;
    uint32_t todo = __ballot_sync(0xFFFFFFFFu, vbits != 0u);
    if (todo != 0u) {
        const bool any_late = __any_sync(0xFFFFFFFFu, (lbits | lbit1) != 0u);
        // one record at a time with FULL-mask reductions (a partial-mask redux is a ~32-instruction software loop, and so is
        // match.any; a drain's visible candidates belong to two or three records)
        while (todo != 0u) {
            const uint32_t key = __shfl_sync(0xFFFFFFFFu, rec0, __ffs((int)todo) - 1);
            const bool mine = vbits != 0u && rec0 == key;
            const uint32_t same = __ballot_sync(0xFFFFFFFFu, mine);
            const uint32_t v = __reduce_or_sync(0xFFFFFFFFu, mine ? vbits : 0u);
            const uint32_t l = any_late ? __reduce_or_sync(0xFFFFFFFFu, mine ? lbits : 0u) : 0u;
            const uint32_t m = main_chunk_counts != nullptr ? __reduce_or_sync(0xFFFFFFFFu, mine ? mbits : 0u) : 0u;
            if (lane == (uint32_t)(__ffs((int)same) - 1)) {
                atomicOr(p.meshlet_visibility + vo0, v);
                if (l != 0u) { atomicOr(reinterpret_cast<uint32_t*>(p.draw_masks + rec0), l); atomicAdd(chunk_counts + (rec0 >> chunk_shift), (uint32_t)__popc(l)); }
                if (m != 0u) { atomicOr(reinterpret_cast<uint32_t*>(p.main_masks + rec0), m); atomicAdd(main_chunk_counts + (rec0 >> chunk_shift), (uint32_t)__popc(m)); }
            }
            todo &= ~same;
        }
        if (vbit1 != 0u) {
            atomicOr(p.meshlet_visibility + vo1, vbit1);
            if (lbit1 != 0u) { atomicOr(reinterpret_cast<uint32_t*>(p.draw_masks + rec1), lbit1); atomicAdd(chunk_counts + (rec1 >> chunk_shift), 1u); }
            if (mbit1 != 0u) { atomicOr(reinterpret_cast<uint32_t*>(p.main_masks + rec1), mbit1); atomicAdd(main_chunk_counts + (rec1 >> chunk_shift), 1u); }
        }
        __syncwarp();
        if (any_late) drawn = __reduce_add_sync(0xFFFFFFFFu, (uint32_t)__popc(lbits) + (lbit1 != 0u ? 1u : 0u));
        if (main_chunk_counts != nullptr) main_drawn_out += __reduce_add_sync(0xFFFFFFFFu, (uint32_t)__popc(mbits) + (mbit1 != 0u ? 1u : 0u));
    }
    return drawn;
}

// ---- TMA bulk copy + mbarrier plumbing (PTX; SASS: UBLKCP / SYNCS) --------------------------------------------
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "LAB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra DONE;\n"
        "bra LAB_WAIT;\n"
        "DONE:\n"
        "}" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_1d(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}

template <int R>
struct __align__(128) WarpSmem {
    uint4 meshlets[R * 64];        // R records x 32 meshlets x 2 x 16 B, filled by TMA
    float mv[R][kMvStride];        // view*model + scale per record
    float4 rows[R][4];             // model matrices of the NEXT tile's entities (cp.async, issued with the TMA copy)
    uint32_t vis[4 * ((R + 3) / 4)];   // last frame's visibility words of the NEXT tile's records (pass 2)
    uint32_t q[8][128];            // Hi-Z candidate ring (pass 2): x, y, z, r_model, scale, record, visibility offset, id
    unsigned long long bar;        // mbarrier of the TMA copies
};
constexpr uint32_t kRing = 128u;
#ifndef ORBIT_DIRECT_MIN_CTAS
#define ORBIT_DIRECT_MIN_CTAS 3
#endif
#ifndef ORBIT_DIRECT_WARPS
#define ORBIT_DIRECT_WARPS 8
#endif
constexpr int kDwWarps = ORBIT_DIRECT_WARPS;     // warps per CTA of the direct test kernel (they share the CTA's tile counter)
constexpr int kDwThreads = kDwWarps * 32;

// view * model (+ largest column scale) for every record of a tile: 16 lanes per record, two records per step
template <int R>
__device__ __forceinline__ void tile_model_view(const float4* rows, float* mv_base, uint32_t my_word, uint32_t lane,
                                                float v0, float v1, float v2, float v3) {
#pragma unroll
    for (int st = 0; st < R / 2; ++st) {
        const uint32_t half = lane >> 4, e = lane & 15u;
        const uint32_t cnt = __shfl_sync(0xFFFFFFFFu, my_word, (2 * st + half) * 4 + 2);
        if (cnt != 0u) {
            const float4 b = rows[(2 * st + half) * 4 + (e >> 2)];
            mv_base[(2 * st + half) * kMvStride + e] = add(add(add(mul(v0, b.x), mul(v1, b.y)), mul(v2, b.z)), mul(v3, b.w));
        }
    }
    __syncwarp();
    if (lane < (uint32_t)R) mv_base[lane * kMvStride + 16] = largest_scale(mv_base + lane * kMvStride);
    __syncwarp();
}

// ---------------------------------------------------------------------------------------------------------
// Direct mode: pass 0, pass 2, and pass 1 without a meshlet visibility buffer — every lane of every record is
// tested. kPass2 = (occlusion_pass == 2 && meshlet occlusion culling on); kProj as in test_item.
//
// Persistent warps; a TILE is R consecutive records, tested one after the other with lane j = meshlet j of the record
// (the reference's 32-lane group, so a ballot is the reference's visibility word). Tile t belongs to CTA t % gridDim.x
// (static, cyclic: every CTA gets the same mix of cheap and expensive stretches of the record list); inside the CTA the
// warps take their CTA's tiles from a SHARED-MEMORY counter (first tile: the warp's index, the next two requested
// ahead), because the cost of a record varies 3x between one whose meshlets all fail the frustum and one that queues 30
// Hi-Z tests — with a static split the 2.5 tiles per warp of C2 quantise to 3, and a device-wide atomic ticket
// (measured) serialises 13 k same-address atomics in L2 for as long as the math takes.
// The tile's meshlets (R x 1 KB contiguous) are staged into shared memory by TMA bulk copies (cp.async.bulk + mbarrier,
// one copy per record issued by R lanes): R KB per warp in flight without holding registers or scoreboards, the next
// tile's copy issued as soon as the current one has been consumed; the record words are prefetched two tiles ahead.
// (A per-lane register prefetch and per-lane cp.async staging were both measured and lost: profiles/r2_meshlet_test_history.txt.)
// view*model is computed once per record by 16 lanes (two records per step) and broadcast through shared memory —
// the reference recomputes the 4x4 product in every lane.
//
// Instruction issue, not HBM, bounds this stage, so the arithmetic of the pinned contract is issued two-wide (FMUL2 /
// FFMA2, see PkConsts): across the components of a meshlet in the frustum / cone test (test_item_xy) and across two
// candidates per lane in the Hi-Z test (occlusion_pair).
//
// Pass 2: lanes surviving frustum + cone are packed into a per-warp ring (8 words per candidate) and the Hi-Z
// projection (5 IEEE divisions, 2 square roots) runs on 64 candidates at a time, two per lane, across record and tile
// boundaries; only the very last drain of a warp is partial. Results leave per candidate: the records' visibility
// words are stored as 0 when their tile starts and visible candidates OR their bit in afterwards (RED.OR; a __syncwarp
// between the stores and the first drain orders the two), likewise the draw masks and the chunks' survivor counts — so
// a record never waits for its candidates and there are no per-record result masks to carry.
//
// kBatch (orbit_meshlet_cull_views, pass 0; orbit_meshlet_cull_views_occlusion, pass 1 without and pass 2 with or without
// meshlet occlusion): the tiles are those of the CONCATENATION of views[0..n_views)'s record lists, each view's list cut into
// tiles of its own (a tile never straddles two views). Every CTA reads the views' record counts once (one round trip; lane v
// of every warp holds view v's count and one past its last tile); a tile takes view matrix, paired planes and alpha filter from
// its view's block, and its draw masks, side words and survivor counts go to that view's scratch. The scene fields (meshlets,
// entities, materials) are read from views[0]. Pass 2: a tile's last-frame visibility words come from its view's buffer, and
// the Hi-Z ring holds the candidates of ONE view at a time — when a warp's next tile belongs to another view, an extra empty
// iteration drains what is left against the old view's pyramid, CullInfo and buffers first (a warp's tiles ascend through
// the concatenation, so that is at most n_views - 1 partial drains per warp). All pyramids of a call have the same geometry.
template <int R, bool kPass2, int kProj, bool kBatch>
__device__ __forceinline__ void meshlet_test_direct_body(const MeshletCullParams* views, uint32_t n_views) {
    static_assert(R == 2 || R == 4 || R == 8, "records per warp tile");
    const MeshletCullParams& p = views[0];
    extern __shared__ __align__(128) unsigned char s_raw[];
    WarpSmem<R>* const all = reinterpret_cast<WarpSmem<R>*>(s_raw + 128);
    uint32_t* const s_next_tile = reinterpret_cast<uint32_t*>(s_raw);

    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    const uint32_t lt = (1u << lane) - 1u;
    WarpSmem<R>& ws = all[warp];
    const OrbitCullInfo& ci = p.cull;
    const PkConsts k = {p.pk_one, p.pk_mone};
    pdl_wait();
    ORBIT_TRACE_STAMP(p.scan.trace, 1, 0);
    if (threadIdx.x == 0) *s_next_tile = kDwWarps;
    __syncthreads();
    // ---- this CTA's tiles: local index j -> tile blockIdx.x + j * gridDim.x; j = warp first, then from the counter.
    // (Device-wide dynamic hand-out was measured twice and lost twice: a ticket per tile serialises ~13 k same-address atomics
    // in one L2 slice; batches of 8 tiles claimed per CTA need only ~1.5 k, but the claiming warp then sits out one L2 atomic
    // round trip per batch with its next tile's loads not yet issued — late pass 34.4 us vs 27.7 us; profiles/r2_meshlet_test_history.txt.)
    auto fetch_tile = [&]() -> uint32_t {
        uint32_t j = 0u;
        if (lane == 0u) j = atomicAdd(s_next_tile, 1u);
        j = __shfl_sync(0xFFFFFFFFu, j, 0);
        const uint64_t t = (uint64_t)blockIdx.x + (uint64_t)j * gridDim.x;
        return t < 0x7FFFFFFFull ? (uint32_t)t : 0x7FFFFFFFu;
    };
    uint32_t t_cur = blockIdx.x + warp * gridDim.x, t_next = fetch_tile(), t_next2 = fetch_tile();
    // The record words of this warp's first two tiles are requested BEFORE the record count is known (bounded by the
    // dispatch buffer's capacity, masked by the count afterwards): one dependent round trip less in the prologue.
    // record words of a tile: lane l < 4R holds word l (entity, meshlet_offset, meshlet_count, visibility_offset per record)
    auto load_words = [&](uint32_t tile, uint64_t bound) -> uint32_t {
        uint32_t w = 0u;
        if (lane < 4u * R && (uint64_t)tile * R + (lane >> 2) < bound) w = __ldcg(p.dispatch_words + 3u + (size_t)tile * R * 4u + lane);
        return w;
    };
    // batched views: lane v < n_views holds view v's record count, its survivor-counter parity and one past its last tile
    uint32_t v_nrec = 0u, v_half = 0u, v_tile_end = 0u;
    if constexpr (kBatch) {
        if (lane < n_views) {
            v_nrec = (uint32_t)min((uint64_t)__ldcg(views[lane].dispatch_words), views[lane].capacity_records);
            v_half = __ldcg(views[lane].chunk_parity) & 1u;                   // see below: one parity per view
            if (blockIdx.x == 0 && warp == 0u) views[lane].chunk_parity[1] = v_half;
        }
        v_tile_end = (v_nrec + R - 1) / R;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, v_tile_end, d);
            if (lane >= (uint32_t)d) v_tile_end += t;
        }
    }
    // tile t of the concatenation (warp-uniform, t < tiles_total) -> view, first record inside the view, the view's record count
    struct ViewTile { uint32_t view, rec0, nrec; };
    auto locate = [&](uint32_t t) -> ViewTile {
        const uint32_t v = (uint32_t)__popc(__ballot_sync(0xFFFFFFFFu, lane < n_views && v_tile_end <= t));
        const uint32_t first = __shfl_sync(0xFFFFFFFFu, v_tile_end, (v - 1u) & 31u);
        return ViewTile{v, (t - (v ? first : 0u)) * R, __shfl_sync(0xFFFFFFFFu, v_nrec, v & 31u)};
    };
    auto load_view_words = [&](uint32_t tile) -> uint32_t {
        const ViewTile w = locate(tile);
        uint32_t x = 0u;
        if (lane < 4u * R && w.rec0 + (lane >> 2) < w.nrec) x = __ldcg(views[w.view].dispatch_words + 3u + (size_t)w.rec0 * 4u + lane);
        return x;
    };
    uint32_t cur_word = 0u, next_word = 0u, nrec = 0u;
    if constexpr (!kBatch) {
        cur_word = load_words(t_cur, p.capacity_records); next_word = load_words(t_next, p.capacity_records);
        nrec = __ldcg(p.dispatch_words);  // workgroup_count_x written by the entity stage
        if ((uint64_t)nrec > p.capacity_records) nrec = (uint32_t)p.capacity_records;
    }
    ORBIT_TRACE_STAMP(p.scan.trace, 1, 1 + 0 * (nrec & 1u));
    uint32_t chunk_shift = chunk_shift_of(nrec);     // batched views: those of the current tile's view (set per tile below)
    // Scratch is double-buffered by a parity that lives in device memory (CUDA-graph replays must see fresh state).
    // Word A is read by test kernels and written by emit kernels; word B the other way round: a kernel never writes
    // a word that CTAs of the same launch read, so the stream order of the launches is the only synchronisation.
    uint32_t half = 0u;
    if constexpr (!kBatch) {
        half = __ldcg(p.chunk_parity) & 1u;
        if (blockIdx.x == 0 && threadIdx.x == 0) p.chunk_parity[1] = half;
    }
    uint32_t* chunk_counts = p.chunk_counts + half * kMaxChunks;
    uint32_t* draw_total = p.draw_total + half;
    uint32_t* main_chunk_counts = nullptr;            // fused MAIN pass (pass 2 only): its own double-buffered scratch
    uint32_t main_total = 0u, mhalf = 0u;
    if (kPass2 && p.main_masks != nullptr) {
        mhalf = __ldcg(p.main_chunk_parity) & 1u;
        if (blockIdx.x == 0 && threadIdx.x == 0) p.main_chunk_parity[1] = mhalf;
        main_chunk_counts = p.main_chunk_counts + mhalf * kMaxChunks;
    }
    const uint32_t tiles_total = kBatch ? __shfl_sync(0xFFFFFFFFu, v_tile_end, 31) : (nrec + R - 1) / R;
    if constexpr (kBatch) {
        if (t_cur < tiles_total) cur_word = load_view_words(t_cur);
        if (t_next < tiles_total) next_word = load_view_words(t_next);
    }
    // row `lane&3` of the view matrix, for the 16-lane view*model product (batched views: the current tile's view)
    const uint32_t vrow_i = lane & 3u;
    float v0 = ci.view_matrix.m[0][vrow_i], v1 = ci.view_matrix.m[1][vrow_i];
    float v2 = ci.view_matrix.m[2][vrow_i], v3 = ci.view_matrix.m[3][vrow_i];
    uint32_t cur_view = kBatch ? 0xFFFFFFFFu : 0u;    // no view yet: the first tile loads its view's state
    const uint32_t hiz_lw = 31u - (uint32_t)__clz((int)max(p.hiz.width, 1u)), hiz_lh = 31u - (uint32_t)__clz((int)max(p.hiz.height, 1u));
    float* const mv_base = &ws.mv[0][0];
    const uint32_t bar = smem_addr(&ws.bar);
    const uint32_t buf = smem_addr(&ws.meshlets[0]);
    const uint32_t qbase = smem_addr(&ws.q[0][0]);
    const uint32_t rows_s = smem_addr(&ws.rows[0][0]), vis_s = smem_addr(&ws.vis[0]);
    if (lane == 0u) { mbar_init(bar, R); mbar_fence_init(); }
    __syncwarp();
    uint32_t parity = 0u;

    // lane r < R issues the bulk copy of record r (count x 32 B) and arrives on the barrier
    // ... and the tile's model matrices (lane l < 4R: column l&3 of record l>>2) and, in pass 2, last frame's visibility
    // words (lane 16+r... of record r) go through cp.async into their staging slots: none of the three waits for a load
    auto issue_tma = [&](uint32_t words, uint32_t tile) {
        const uint32_t off = __shfl_sync(0xFFFFFFFFu, words, (lane * 4u + 1u) & 31u);
        const uint32_t cnt = __shfl_sync(0xFFFFFFFFu, words, (lane * 4u + 2u) & 31u);
        {
            const uint32_t rr = (lane >> 2) & (uint32_t)(R - 1);
            const uint32_t ent_r = __shfl_sync(0xFFFFFFFFu, words, rr * 4u + 0u), cnt_r = __shfl_sync(0xFFFFFFFFu, words, rr * 4u + 2u);
            if (lane < 4u * R && cnt_r != 0u) cp_async_16(rows_s + lane * 16u, p.entities + (size_t)ent_r * 8u + (lane & 3u));
            if (kPass2) {
                const uint32_t* mvis = p.meshlet_visibility;                  // batched: the visibility words of the tile's view
                if constexpr (kBatch) mvis = views[locate(tile).view].meshlet_visibility;
                const uint32_t rv = lane & (uint32_t)(R - 1);
                const uint32_t vo_r = __shfl_sync(0xFFFFFFFFu, words, rv * 4u + 3u), cnt_v = __shfl_sync(0xFFFFFFFFu, words, rv * 4u + 2u);
                if (lane >= 16u && lane < 16u + (uint32_t)R && cnt_v != 0u) cp_async_4(vis_s + rv * 4u, mvis + vo_r);
            }
            cp_async_commit();
        }
        if (lane < (uint32_t)R) {
            if (cnt != 0u) {
                const uint32_t bytes = min(cnt, 32u) * 32u;
                mbar_arrive_expect_tx(bar, bytes);
                tma_load_1d(buf + lane * 1024u, p.meshlets + 2u * (size_t)off, bytes, bar);
            } else {
                mbar_arrive(bar);
            }
        }
    };
    if constexpr (!kBatch) {   // the two speculative loads were bounded by the buffer capacity; now apply the real record count
        if (!(lane < 4u * R && (uint64_t)t_cur * R + (lane >> 2) < (uint64_t)nrec)) cur_word = 0u;
        if (!(lane < 4u * R && (uint64_t)t_next * R + (lane >> 2) < (uint64_t)nrec)) next_word = 0u;
    }
    uint32_t warp_total = 0u;   // survivors found by this warp (lets the emit kernel skip everything when zero)
#ifdef ORBIT_TRACE
    bool trace_first = true;
#endif
    uint32_t qhead = 0u, qn = 0u;   // ring-buffer read position and fill (entries [qhead, qhead+qn) mod 128 are pending)
    if (t_cur < tiles_total) issue_tma(cur_word, t_cur);
    // One extra, empty iteration after the last tile flushes what is left in the ring through the same drain code.
    bool final_pass = t_cur >= tiles_total;
    while (true) {
        uint32_t rec0 = t_cur * R;
        bool view_flush = false;   // batched pass 2: this iteration only drains the ring, the tile waits for the next one
        if constexpr (kBatch) {
            if (!final_pass) {
                const ViewTile w = locate(t_cur);
                rec0 = w.rec0; nrec = w.nrec;
                if constexpr (kPass2) view_flush = w.view != cur_view && qn != 0u;   // the ring holds the previous view's candidates
                if (w.view != cur_view && !view_flush) {                      // warp-uniform; a warp's tiles ascend, so do their views
                    if (lane == 0u && warp_total != 0u) atomicAdd(draw_total, warp_total);
                    warp_total = 0u;
                    cur_view = w.view;
                    const uint32_t h = __shfl_sync(0xFFFFFFFFu, v_half, cur_view);
                    chunk_shift = chunk_shift_of(nrec);
                    chunk_counts = views[cur_view].chunk_counts + h * kMaxChunks;
                    draw_total = views[cur_view].draw_total + h;
                    const OrbitCullInfo& cv = views[cur_view].cull;
                    v0 = cv.view_matrix.m[0][vrow_i]; v1 = cv.view_matrix.m[1][vrow_i];
                    v2 = cv.view_matrix.m[2][vrow_i]; v3 = cv.view_matrix.m[3][vrow_i];
                }
            }
        }
        const bool flush = final_pass || view_flush;   // an iteration without a tile: only the drain below runs
        const MeshletCullParams& pt = kBatch ? views[cur_view & (ORBIT_MAX_BATCH_VIEWS - 1)] : p;   // the tile's view
        const uint32_t my_word = flush ? 0u : cur_word;
        uint32_t my_mask = 0u;       // lane r < R: draw mask of record r (passes without Hi-Z)
        uint32_t vw = 0u;            // lane r < R, pass 2: last frame's visibility word of record r (decides should_draw)
        if (!flush) {
            cur_word = next_word;
            if constexpr (kBatch) next_word = t_next2 < tiles_total ? load_view_words(t_next2) : 0u;
            else next_word = t_next2 < tiles_total ? load_words(t_next2, nrec) : 0u;
            if (kPass2) {
                // lane r: the record's visibility word is read, then stored as 0 — visible candidates OR their bits in
                // afterwards (meshlet_cull.comp:235-242); likewise the draw mask
                const uint32_t ent = __shfl_sync(0xFFFFFFFFu, my_word, (lane * 4u + 0u) & 31u);
                const uint32_t mof = __shfl_sync(0xFFFFFFFFu, my_word, (lane * 4u + 1u) & 31u);
                const uint32_t my_cnt = __shfl_sync(0xFFFFFFFFu, my_word, (lane * 4u + 2u) & 31u);
                const uint32_t my_vo = __shfl_sync(0xFFFFFFFFu, my_word, (lane * 4u + 3u) & 31u);
                cp_async_wait_all();
                __syncwarp();
                if (lane < (uint32_t)R && my_cnt != 0u) {
                    vw = ws.vis[lane];
                    pt.meshlet_visibility[my_vo] = 0u;
                }
                if (lane < (uint32_t)R && rec0 + lane < nrec) {
                    pt.draw_masks[rec0 + lane] = make_uint4(0u, ent, mof, 1u);   // .w = 1: no side-array entries, the emit kernel reads the meshlet
                    if (main_chunk_counts != nullptr) p.main_masks[rec0 + lane] = make_uint4(0u, ent, mof, 1u);
                }
            } else {
                cp_async_wait_all();
                __syncwarp();
            }
            tile_model_view<R>(&ws.rows[0][0], mv_base, my_word, lane, v0, v1, v2, v3);
            mbar_wait(bar, parity);
            parity ^= 1u;
#ifdef ORBIT_TRACE
            if (p.scan.trace != nullptr && threadIdx.x == 0 && trace_first) { trace_first = false; ORBIT_TRACE_STAMP(p.scan.trace, 1, 2); }
#endif
        }
        // The record loop is deliberately NOT unrolled (instruction cache). The extra, empty iterations after a warp's last
        // tile (final_pass) and before a batched warp's first tile of another view (view_flush) only run the drain below, on
        // whatever is left in the ring.
#pragma unroll 1
        for (uint32_t r = 0; r < (uint32_t)R; ++r) {
            const uint32_t cnt = __shfl_sync(0xFFFFFFFFu, my_word, r * 4u + 2u);   // 0 for records past the end
            if (cnt != 0u) {                                                        // warp-uniform
                const float* mvr = mv_base + r * kMvStride;
                const float4 c0 = *reinterpret_cast<const float4*>(mvr), c1 = *reinterpret_cast<const float4*>(mvr + 4);
                const float4 c2 = *reinterpret_cast<const float4*>(mvr + 8), c3 = *reinterpret_cast<const float4*>(mvr + 12);
                const float scale = mvr[16];
                const bool in_rec = lane < cnt;
                const uint4 a = ws.meshlets[r * 64u + lane * 2u];
                const uint4 b = ws.meshlets[r * 64u + lane * 2u + 1u];
                uint32_t alpha = 32u;                                               // out-of-record lanes: no alpha bit
                if (in_rec) alpha = __ldg(reinterpret_cast<const uint32_t*>(      // L1-resident table; issued here, used after the test
                    p.materials + (size_t)(b.w & 0xFFFFu) * ORBIT_MATERIAL_STRIDE_BYTES + ORBIT_MATERIAL_ALPHA_MODE_OFFSET));
                const ItemXY t = test_item_xy<kProj>(pt.cull, pt, k, c0, c1, c2, c3, scale, __uint_as_float(a.x), __uint_as_float(a.y),
                                                     __uint_as_float(a.z), __uint_as_float(a.w), b.x);
                const bool pre = in_rec && t.pre_visible;
                if (!kPass2) {
                    // should_draw = visible && alpha passes the filter (meshlet_cull.comp:207)
                    const bool draw = pre && (shl1(alpha) & pt.cull.alpha_mode_flags) != 0u;
                    const uint32_t mask = __ballot_sync(0xFFFFFFFFu, draw);
                    if (lane == r) my_mask = mask;
                    // the command words of a survivor travel to the emit kernel through a side array (L2-resident at the sizes
                    // where the emit kernel is latency-bound; at C5 scale it replaces a second 32-byte read of every surviving meshlet)
                    const uint32_t ent_r = __shfl_sync(0xFFFFFFFFu, my_word, r * 4u);
                    if (draw && pt.cmd_side != nullptr) pt.cmd_side[(size_t)(rec0 + r) * 32u + lane] = make_uint4(b.y, b.z, b.w, ent_r);
                } else {
                    // queue the survivors for the Hi-Z test
                    const uint32_t pre_mask = __ballot_sync(0xFFFFFFFFu, pre);
                    const uint32_t vwr = __shfl_sync(0xFFFFFFFFu, vw, r);
                    const uint32_t vo = __shfl_sync(0xFFFFFFFFu, my_word, r * 4u + 3u);
                    if (pre) {
                        // id word: lane | visible-last-frame << 5 | min(alpha mode, 32) << 6 (alpha modes >= 32 select no bit)
                        const uint32_t id = lane | (((vwr >> lane) & 1u) << 5) | (min(alpha, 32u) << 6);
                        const uint32_t qa = qbase + ((qhead + qn + (uint32_t)__popc(pre_mask & lt)) & (kRing - 1u)) * 4u;
                        constexpr uint32_t cs4 = kRing * 4u;
                        sts32(qa, __float_as_uint(t.pxy.x)); sts32(qa + cs4, __float_as_uint(t.pxy.y)); sts32(qa + 2u * cs4, __float_as_uint(t.pz));
                        sts32(qa + 3u * cs4, a.w); sts32(qa + 4u * cs4, __float_as_uint(scale));
                        sts32(qa + 5u * cs4, rec0 + r); sts32(qa + 6u * cs4, vo); sts32(qa + 7u * cs4, id);
                    }
                    qn += (uint32_t)__popc(pre_mask);
                }
            }
            // ---- Hi-Z test of 64 queued candidates (the ring holds the < 64 left over plus a record's 32); the warp's
            // very last drain takes whatever is left
            if (kPass2 && (qn >= 64u || (flush && qn != 0u))) {
                const uint32_t n = min(qn, 64u);
                __syncwarp();
                warp_total += drain_candidates<kProj>(pt, k, qbase, kRing - 1u, qhead, n, chunk_counts, chunk_shift, hiz_lw, hiz_lh, lane,
                                                      main_chunk_counts, main_total);
                qhead = (qhead + n) & (kRing - 1u);
                qn -= n;
            }
        }
        if constexpr (kBatch && kPass2) {
            // the same tile again, now with an empty ring; its head back at 0: drain_candidates reads candidate pairs with 8-byte
            // loads and needs an even head, which the odd-sized flush may have left behind
            if (view_flush) { qhead = 0u; continue; }
        }
        if (final_pass) break;
        // every lane has read its meshlets: the staging buffer is free -> start the next tile's copy now
        __syncwarp();
        if (t_next < tiles_total) issue_tma(cur_word, t_next);
        if (!kPass2) {
            // one {draw mask, entity, meshlet offset} per record, kept L2-resident for the emit kernel (so it needs one
            // load per record and never touches the dispatch buffer); survivors counted per chunk
            const uint32_t ent = __shfl_sync(0xFFFFFFFFu, my_word, (lane * 4u + 0u) & 31u);
            const uint32_t mof = __shfl_sync(0xFFFFFFFFu, my_word, (lane * 4u + 1u) & 31u);
            if (lane < (uint32_t)R && rec0 + lane < nrec) pt.draw_masks[rec0 + lane] = make_uint4(my_mask, ent, mof, pt.cmd_side != nullptr ? 0u : 1u);
            const uint32_t tile_total = __reduce_add_sync(0xFFFFFFFFu, __popc(my_mask));
            if (lane == 0u && tile_total != 0u) atomicAdd(chunk_counts + (rec0 >> chunk_shift), tile_total);   // a tile never straddles a chunk
            warp_total += tile_total;
        }
        t_cur = t_next; t_next = t_next2;
        t_next2 = t_next2 < tiles_total ? fetch_tile() : 0x7FFFFFFFu;
        final_pass = t_cur >= tiles_total;
    }
    ORBIT_TRACE_STAMP(p.scan.trace, 1, 3);
    pdl_launch_dependents();
    if (lane == 0u && warp_total != 0u) atomicAdd(draw_total, warp_total);
    if (kPass2 && lane == 0u && main_total != 0u) atomicAdd(p.main_draw_total + mhalf, main_total);
#ifdef ORBIT_TRACE
    __syncthreads();
    ORBIT_TRACE_STAMP(p.scan.trace, 1, 4);
#endif
}

template <int R, bool kPass2, int kProj>
__global__ void __launch_bounds__(kDwThreads, ORBIT_DIRECT_MIN_CTAS) meshlet_test_direct_kernel(const __grid_constant__ MeshletCullParams p) {
    meshlet_test_direct_body<R, kPass2, kProj, false>(&p, 1u);
}

// orbit_meshlet_cull_views (pass 0) and orbit_meshlet_cull_views_occlusion (kPass2: pass 2 with meshlet occlusion; else pass 1
// or 2 without it) over the concatenation of up to 16 views' record lists
template <int R, bool kPass2, int kProj>
__global__ void __launch_bounds__(kDwThreads, ORBIT_DIRECT_MIN_CTAS) meshlet_test_views_kernel(const __grid_constant__ MeshletViewsParams pv) {
    meshlet_test_direct_body<R, kPass2, kProj, true>(pv.view, pv.n_views);
}

// ---------------------------------------------------------------------------------------------------------
// Packed mode: pass 1 with a meshlet visibility buffer. Only lanes whose visibility bit is set can be visible
// (visible = visible_in_buffer, meshlet_cull.comp:137), so only those meshlets are loaded and tested.
//
// The kernel is latency-bound, and the candidates are badly distributed: most tiles of R records hold none (occluded
// entities), a tile inside the visible part of the scene up to 32 R. A warp that tests its own tile's candidates 32 at a
// time sets the kernel's duration by the heaviest tile (measured on C2: warps without candidates done after 2.6 us, the
// heaviest after 9.7 us; profiles/r2_frame_timeline.txt). So the candidates of a CTA's eight tiles go into ONE
// shared-memory queue and all eight warps drain it, two batches of 32 per step with both batches' meshlet gathers in
// flight and their arithmetic interleaved; and the tiles of a CTA are taken gridDim.x apart (tile = (round * 8 + warp) *
// gridDim.x + blockIdx.x), so every CTA gets the same mix of empty and full tiles. The dependent loads of a tile (record
// words -> visibility word + model matrix -> meshlets) are software-pipelined across rounds: round k+1's chain is started
// before round k's queue is drained, and the first two rounds' record words are requested before the record count is known.
template <int R>
struct __align__(16) PackedCtaSmem {
    float mv[kMcWarps][R][kMvStride];      // view*model + scale per record of the round's tiles
    uint32_t words[kMcWarps][R * 4];       // the tiles' record words
    uint32_t mask[kMcWarps][R];            // draw masks being accumulated
    uint32_t queue[kMcWarps * R * 32];     // candidates: warp << 8 | record << 5 | lane
    uint32_t qcount[2];                    // queue fill, double-buffered by round parity
};

// Loads of one tile that depend only on its record words, kept in registers until the tile's turn comes:
// model-matrix rows (16 lanes per record, two records per step) and last frame's visibility word (lane r < R).
template <int R>
struct PackedPrefetch {
    float4 b[R / 2];
    uint32_t vw;
};

template <int R>
__device__ __forceinline__ PackedPrefetch<R> packed_issue_loads(const MeshletCullParams& p, uint32_t words, uint32_t lane) {
    PackedPrefetch<R> f;
    const uint32_t my_cnt = __shfl_sync(0xFFFFFFFFu, words, (lane * 4u + 2u) & 31u);
    const uint32_t my_vo = __shfl_sync(0xFFFFFFFFu, words, (lane * 4u + 3u) & 31u);
    f.vw = 0u;
    if (lane < (uint32_t)R && my_cnt != 0u) f.vw = __ldcg(p.meshlet_visibility + my_vo) & (my_cnt >= 32u ? 0xFFFFFFFFu : ((1u << my_cnt) - 1u));
#pragma unroll
    for (int st = 0; st < R / 2; ++st) {
        const uint32_t half = lane >> 4, e = lane & 15u;
        const uint32_t ent = __shfl_sync(0xFFFFFFFFu, words, (2 * st + half) * 4 + 0);
        const uint32_t cnt = __shfl_sync(0xFFFFFFFFu, words, (2 * st + half) * 4 + 2);
        f.b[st] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (cnt != 0u) f.b[st] = __ldg(p.entities + (size_t)ent * 8u + (e >> 2));
    }
    return f;
}

// view * model (+ largest column scale) of the tile's records from the prefetched rows (same arithmetic as tile_model_view)
template <int R>
__device__ __forceinline__ void packed_finish_model_view(const PackedPrefetch<R>& f, float* mv_base, uint32_t lane,
                                                         float v0, float v1, float v2, float v3) {
#pragma unroll
    for (int st = 0; st < R / 2; ++st) {
        const uint32_t half = lane >> 4, e = lane & 15u;
        const float4 b = f.b[st];
        mv_base[(2 * st + half) * kMvStride + e] = add(add(add(mul(v0, b.x), mul(v1, b.y)), mul(v2, b.z)), mul(v3, b.w));
    }
    __syncwarp();
    if (lane < (uint32_t)R) mv_base[lane * kMvStride + 16] = largest_scale(mv_base + lane * kMvStride);
    __syncwarp();
}

#ifndef ORBIT_PACKED_MIN_CTAS
#define ORBIT_PACKED_MIN_CTAS 4
#endif
template <int R>
__global__ void __launch_bounds__(kMcThreads, ORBIT_PACKED_MIN_CTAS) meshlet_test_packed_kernel(const __grid_constant__ MeshletCullParams p) {
    static_assert(R == 2 || R == 4 || R == 8, "records per warp tile");
    __shared__ PackedCtaSmem<R> sm;
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    const uint32_t lt = (1u << lane) - 1u;
    const OrbitCullInfo& ci = p.cull;
    pdl_wait();
    ORBIT_TRACE_STAMP(p.scan.trace, 2, 0);
    if (threadIdx.x < 2u) sm.qcount[threadIdx.x] = 0u;
    // tile of (round, warp): CTAs interleave at tile granularity, a CTA's own tiles lie gridDim.x apart
    const uint64_t round_stride = (uint64_t)kMcWarps * gridDim.x;
    const uint64_t tile_first = (uint64_t)warp * gridDim.x + blockIdx.x;
    auto spec_words = [&](uint64_t tile, uint64_t bound) -> uint32_t {
        const uint64_t rec = tile * R + (lane >> 2);
        return (lane < 4u * R && rec < bound) ? __ldcg(p.dispatch_words + 3u + (size_t)tile * R * 4u + lane) : 0u;
    };
    uint32_t cur_word = spec_words(tile_first, p.capacity_records), next_word = spec_words(tile_first + round_stride, p.capacity_records);
    uint32_t nrec = __ldcg(p.dispatch_words);
    if ((uint64_t)nrec > p.capacity_records) nrec = (uint32_t)p.capacity_records;
    ORBIT_TRACE_STAMP_AFTER(p.scan.trace, 2, 1, nrec + cur_word);
    const uint32_t chunk_rec = 1u << chunk_shift_of(nrec);
    const uint32_t half = __ldcg(p.chunk_parity) & 1u;   // see meshlet_test_direct_kernel
    if (blockIdx.x == 0 && threadIdx.x == 0) p.chunk_parity[1] = half;
    uint32_t* const chunk_counts = p.chunk_counts + half * kMaxChunks;
    uint32_t* const draw_total = p.draw_total + half;
    const uint64_t tiles_total = ((uint64_t)nrec + R - 1) / R;
    if (!(lane < 4u * R && tile_first * R + (lane >> 2) < nrec)) cur_word = 0u;
    if (!(lane < 4u * R && (tile_first + round_stride) * R + (lane >> 2) < nrec)) next_word = 0u;
    const uint32_t vrow_i = lane & 3u;
    const float v0 = ci.view_matrix.m[0][vrow_i], v1 = ci.view_matrix.m[1][vrow_i];
    const float v2 = ci.view_matrix.m[2][vrow_i], v3 = ci.view_matrix.m[3][vrow_i];
    uint32_t warp_total = 0u;
    PackedPrefetch<R> cur = packed_issue_loads<R>(p, cur_word, lane);
    __syncthreads();                                                        // qcount zeroed
    for (uint32_t round = 0; (uint64_t)round * round_stride + blockIdx.x < tiles_total; ++round) {   // CTA-uniform
        const uint64_t tile = tile_first + (uint64_t)round * round_stride;
        const uint32_t rec0 = (uint32_t)min(tile * R, (uint64_t)0xFFFFFFFFu);
        const uint32_t my_word = cur_word;
        const uint32_t vw = cur.vw;
        const uint32_t qpar = round & 1u;
        // ---- A. this warp's tile: record words and matrices into shared memory, candidates into the CTA's queue
        if (lane < 4u * R) sm.words[warp][lane] = my_word;
        if (lane < (uint32_t)R) sm.mask[warp][lane] = 0u;
        const uint32_t any_vw = __ballot_sync(0xFFFFFFFFu, vw != 0u);
#ifdef ORBIT_TRACE
        if (round == 0u) ORBIT_TRACE_STAMP_AFTER(p.scan.trace, 2, 5, any_vw);
#endif
        if (any_vw != 0u) {                                                 // warp-uniform: tiles without candidates skip the matrix math
            packed_finish_model_view<R>(cur, &sm.mv[warp][0][0], lane, v0, v1, v2, v3);
            uint32_t n_items = 0u;
#pragma unroll
            for (int r = 0; r < R; ++r) n_items += __popc(__shfl_sync(0xFFFFFFFFu, vw, r));
            uint32_t base = 0u;
            if (lane == 0u) base = atomicAdd(&sm.qcount[qpar], n_items);
            base = __shfl_sync(0xFFFFFFFFu, base, 0);
#pragma unroll
            for (int r = 0; r < R; ++r) {
                const uint32_t m = __shfl_sync(0xFFFFFFFFu, vw, r);
                if ((m >> lane) & 1u) sm.queue[base + __popc(m & lt)] = (warp << 8) | ((uint32_t)r << 5) | lane;
                base += __popc(m);
            }
        }
        // ---- start the next round's chain (its record words arrived while the previous round was tested)
        PackedPrefetch<R> nxt = packed_issue_loads<R>(p, next_word, lane);
        uint32_t next2_word = 0u;
        {
            const uint64_t t2 = tile + 2u * round_stride;
            if (t2 < tiles_total && lane < 4u * R && t2 * R + (lane >> 2) < nrec) next2_word = __ldcg(p.dispatch_words + 3u + (size_t)t2 * R * 4u + lane);
        }
        __syncthreads();
        // ---- C. all warps drain the queue: batches warp, warp + 8, ...; two batches per step
        const uint32_t total = sm.qcount[qpar];
        if (threadIdx.x == 0) sm.qcount[qpar ^ 1u] = 0u;                    // the next round's counter (last read two barriers ago)
#ifdef ORBIT_TRACE
        if (round == 0u) { ORBIT_TRACE_STAMP(p.scan.trace, 2, 6); ORBIT_TRACE_VALUE(p.scan.trace, 8, total); }
#endif
        for (uint32_t b0 = warp * 32u; b0 < total; b0 += 2u * kMcWarps * 32u) {
            uint32_t id[2]; uint4 ma[2], mb[2]; bool live[2]; uint32_t alpha[2];
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                const uint32_t i = b0 + (uint32_t)u * kMcWarps * 32u + lane;
                live[u] = i < total;
                id[u] = sm.queue[live[u] ? i : 0u];                         // dead lanes redo candidate 0 and drop the result
                const uint32_t moff = sm.words[id[u] >> 8][((id[u] >> 5) & 7u) * 4u + 1u];
                const uint4* m = p.meshlets + 2u * ((size_t)moff + (id[u] & 31u));
                ma[u] = __ldg(m); mb[u] = __ldg(m + 1);
            }
#pragma unroll
            for (int u = 0; u < 2; ++u)
                alpha[u] = __ldg(reinterpret_cast<const uint32_t*>(p.materials + (size_t)(mb[u].w & 0xFFFFu) * ORBIT_MATERIAL_STRIDE_BYTES + ORBIT_MATERIAL_ALPHA_MODE_OFFSET));
#ifdef ORBIT_TRACE
            if (round == 0u && b0 == warp * 32u) { ORBIT_TRACE_STAMP_AFTER(p.scan.trace, 2, 7, ma[0].x + ma[1].x); ORBIT_TRACE_STAMP_AFTER(p.scan.trace, 2, 9, alpha[0] + alpha[1]); }
#endif
            bool pre[2];
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                const float* mvr = &sm.mv[id[u] >> 8][(id[u] >> 5) & 7u][0];
                const ItemTest t = test_item<-1>(ci, *reinterpret_cast<const float4*>(mvr), *reinterpret_cast<const float4*>(mvr + 4),
                                                 *reinterpret_cast<const float4*>(mvr + 8), *reinterpret_cast<const float4*>(mvr + 12), mvr[16],
                                                 __uint_as_float(ma[u].x), __uint_as_float(ma[u].y), __uint_as_float(ma[u].z), __uint_as_float(ma[u].w), mb[u].x);
                pre[u] = t.pre_visible;
            }
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                // should_draw = visible && alpha passes the filter (meshlet_cull.comp:207); pass 1: visible_last_frame holds for every candidate
                if (live[u] && pre[u] && (shl1(alpha[u]) & ci.alpha_mode_flags) != 0u) {
                    const uint32_t w = id[u] >> 8, r = (id[u] >> 5) & 7u, j = id[u] & 31u;
                    atomicOr(&sm.mask[w][r], 1u << j);
                    // the command words of a survivor travel to the emit kernel through an L2-resident side array
                    const uint64_t rec = ((uint64_t)w * gridDim.x + blockIdx.x + (uint64_t)round * round_stride) * R + r;
                    if (p.cmd_side != nullptr) p.cmd_side[rec * 32u + j] = make_uint4(mb[u].y, mb[u].z, mb[u].w, sm.words[w][r * 4u]);
                }
            }
        }
#ifdef ORBIT_TRACE
        if (round == 0u) ORBIT_TRACE_STAMP(p.scan.trace, 2, 10);
#endif
        __syncthreads();
#ifdef ORBIT_TRACE
        if (round == 0u) ORBIT_TRACE_STAMP(p.scan.trace, 2, 11);
#endif
        // ---- E. this warp's tile: draw masks out, survivors counted per chunk
        uint32_t my_draw_mask = 0u;
        if (lane < (uint32_t)R) my_draw_mask = sm.mask[warp][lane];
        {
            const uint32_t ent = __shfl_sync(0xFFFFFFFFu, my_word, (lane * 4u + 0u) & 31u);
            const uint32_t mof = __shfl_sync(0xFFFFFFFFu, my_word, (lane * 4u + 1u) & 31u);
            if (lane < (uint32_t)R && (uint64_t)rec0 + lane < nrec) p.draw_masks[rec0 + lane] = make_uint4(my_draw_mask, ent, mof, p.cmd_side != nullptr ? 0u : 1u);
        }
        const uint32_t tile_total = __reduce_add_sync(0xFFFFFFFFu, __popc(my_draw_mask));
        if (lane == 0u && tile_total != 0u) atomicAdd(chunk_counts + rec0 / chunk_rec, tile_total);
        warp_total += tile_total;
        cur = nxt;
        cur_word = next_word;
        next_word = next2_word;
    }
    ORBIT_TRACE_STAMP(p.scan.trace, 2, 3);
    pdl_launch_dependents();
    if (lane == 0u && warp_total != 0u) atomicAdd(draw_total, warp_total);
#ifdef ORBIT_TRACE
    __syncthreads();
    ORBIT_TRACE_STAMP(p.scan.trace, 2, 4);
#endif
}

// orbit_meshlet_cull_views_occlusion, pass 1 with meshlet visibility buffers: meshlet_test_packed_kernel over the concatenation
// of the views' record lists (each view's list cut into tiles of its own, located as in meshlet_test_direct_body). A CTA's
// queue mixes the candidates of several views: every warp notes the view and first record of its tile of the round in shared
// memory, and the fields of each view's CullInfo that the test reads — paired with nothing, the plain test_item arithmetic —
// are staged once per CTA (16 x 208 bytes), so a candidate is tested against its own view's planes and alpha filter. A warp's
// tile takes view matrix, visibility words, draw masks, side words and survivor counters from its view.
struct ViewCull {
    float cull_planes[ORBIT_MAX_CULL_PLANES][4];
    uint32_t cull_plane_count, projection_type, alpha_mode_flags, pad;
};
template <int R>
__global__ void __launch_bounds__(kMcThreads, ORBIT_PACKED_MIN_CTAS) meshlet_test_packed_views_kernel(const __grid_constant__ MeshletViewsParams pv) {
    static_assert(R == 2 || R == 4 || R == 8, "records per warp tile");
    __shared__ PackedCtaSmem<R> sm;
    __shared__ ViewCull s_cull[ORBIT_MAX_BATCH_VIEWS];
    __shared__ uint32_t s_view[kMcWarps], s_rec0[kMcWarps];   // view and first record (inside the view) of each warp's tile
    const MeshletCullParams* const views = pv.view;
    const MeshletCullParams& p = views[0];                     // scene fields
    const uint32_t n_views = pv.n_views;
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    const uint32_t lt = (1u << lane) - 1u;
    pdl_wait();
    ORBIT_TRACE_STAMP(p.scan.trace, 2, 0);
    if (threadIdx.x < 2u) sm.qcount[threadIdx.x] = 0u;
    for (uint32_t v = warp; v < n_views; v += kMcWarps) {      // warp-uniform view, lane = word
        const OrbitCullInfo& cv = views[v].cull;
        for (uint32_t i = lane; i < 4u * ORBIT_MAX_CULL_PLANES; i += 32u) (&s_cull[v].cull_planes[0][0])[i] = (&cv.cull_planes[0][0])[i];
        if (lane == 0u) { s_cull[v].cull_plane_count = cv.cull_plane_count; s_cull[v].projection_type = cv.projection_type; s_cull[v].alpha_mode_flags = cv.alpha_mode_flags; }
    }
    // lane v < n_views: view v's record count, its survivor-counter parity and one past its last tile (meshlet_test_direct_body)
    uint32_t v_nrec = 0u, v_half = 0u, v_tile_end = 0u;
    if (lane < n_views) {
        v_nrec = (uint32_t)min((uint64_t)__ldcg(views[lane].dispatch_words), views[lane].capacity_records);
        v_half = __ldcg(views[lane].chunk_parity) & 1u;
        if (blockIdx.x == 0 && warp == 0u) views[lane].chunk_parity[1] = v_half;
    }
    v_tile_end = (v_nrec + R - 1) / R;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, v_tile_end, d);
        if (lane >= (uint32_t)d) v_tile_end += t;
    }
    const uint64_t tiles_total = __shfl_sync(0xFFFFFFFFu, v_tile_end, 31);
    struct ViewTile { uint32_t view, rec0, nrec; };
    auto locate = [&](uint64_t t) -> ViewTile {                 // t < tiles_total, warp-uniform
        const uint32_t v = (uint32_t)__popc(__ballot_sync(0xFFFFFFFFu, lane < n_views && v_tile_end <= t));
        const uint32_t first = __shfl_sync(0xFFFFFFFFu, v_tile_end, (v - 1u) & 31u);
        return ViewTile{v, ((uint32_t)t - (v ? first : 0u)) * R, __shfl_sync(0xFFFFFFFFu, v_nrec, v & 31u)};
    };
    auto tile_words = [&](uint64_t t) -> uint32_t {             // record words of tile t (0 past the end)
        if (t >= tiles_total) return 0u;
        const ViewTile w = locate(t);
        return (lane < 4u * R && w.rec0 + (lane >> 2) < w.nrec) ? __ldcg(views[w.view].dispatch_words + 3u + (size_t)w.rec0 * 4u + lane) : 0u;
    };
    auto view_of = [&](uint64_t t) -> uint32_t { return t < tiles_total ? locate(t).view : 0u; };
    const uint64_t round_stride = (uint64_t)kMcWarps * gridDim.x;
    const uint64_t tile_first = (uint64_t)warp * gridDim.x + blockIdx.x;
    uint32_t cur_word = tile_words(tile_first), next_word = tile_words(tile_first + round_stride);
    ORBIT_TRACE_STAMP_AFTER(p.scan.trace, 2, 1, cur_word);
    uint32_t cur_view = kNone;                                  // the view whose counters warp_total belongs to
    uint32_t chunk_rec = 1u;
    uint32_t* chunk_counts = nullptr;
    uint32_t* draw_total = nullptr;
    float v0 = 0.f, v1 = 0.f, v2 = 0.f, v3 = 0.f;
    const uint32_t vrow_i = lane & 3u;
    uint32_t warp_total = 0u;
    PackedPrefetch<R> cur = packed_issue_loads<R>(views[view_of(tile_first)], cur_word, lane);
    __syncthreads();                                                        // qcount zeroed, CullInfos staged
    for (uint32_t round = 0; (uint64_t)round * round_stride + blockIdx.x < tiles_total; ++round) {   // CTA-uniform
        const uint64_t tile = tile_first + (uint64_t)round * round_stride;
        ViewTile w{0u, 0u, 0u};
        if (tile < tiles_total) {
            w = locate(tile);
            if (w.view != cur_view) {                           // warp-uniform; a warp's tiles ascend, so do their views
                if (lane == 0u && warp_total != 0u) atomicAdd(draw_total, warp_total);
                warp_total = 0u;
                cur_view = w.view;
                const MeshletCullParams& pv_ = views[cur_view];
                chunk_rec = 1u << chunk_shift_of(w.nrec);
                const uint32_t h = __shfl_sync(0xFFFFFFFFu, v_half, cur_view);
                chunk_counts = pv_.chunk_counts + h * kMaxChunks;
                draw_total = pv_.draw_total + h;
                v0 = pv_.cull.view_matrix.m[0][vrow_i]; v1 = pv_.cull.view_matrix.m[1][vrow_i];
                v2 = pv_.cull.view_matrix.m[2][vrow_i]; v3 = pv_.cull.view_matrix.m[3][vrow_i];
            }
        }
        const uint32_t rec0 = w.rec0;
        const uint32_t my_word = cur_word;
        const uint32_t vw = cur.vw;
        const uint32_t qpar = round & 1u;
        // ---- A. this warp's tile: record words and matrices into shared memory, candidates into the CTA's queue
        if (lane < 4u * R) sm.words[warp][lane] = my_word;
        if (lane < (uint32_t)R) sm.mask[warp][lane] = 0u;
        if (lane == 0u) { s_view[warp] = w.view; s_rec0[warp] = rec0; }
        const uint32_t any_vw = __ballot_sync(0xFFFFFFFFu, vw != 0u);
        if (any_vw != 0u) {                                                 // warp-uniform: tiles without candidates skip the matrix math
            packed_finish_model_view<R>(cur, &sm.mv[warp][0][0], lane, v0, v1, v2, v3);
            uint32_t n_items = 0u;
#pragma unroll
            for (int r = 0; r < R; ++r) n_items += __popc(__shfl_sync(0xFFFFFFFFu, vw, r));
            uint32_t base = 0u;
            if (lane == 0u) base = atomicAdd(&sm.qcount[qpar], n_items);
            base = __shfl_sync(0xFFFFFFFFu, base, 0);
#pragma unroll
            for (int r = 0; r < R; ++r) {
                const uint32_t m = __shfl_sync(0xFFFFFFFFu, vw, r);
                if ((m >> lane) & 1u) sm.queue[base + __popc(m & lt)] = (warp << 8) | ((uint32_t)r << 5) | lane;
                base += __popc(m);
            }
        }
        // ---- start the next round's chain (its record words arrived while the previous round was tested)
        PackedPrefetch<R> nxt = packed_issue_loads<R>(views[view_of(tile + round_stride)], next_word, lane);
        const uint32_t next2_word = tile_words(tile + 2u * round_stride);
        __syncthreads();
        // ---- C. all warps drain the queue: batches warp, warp + 8, ...; two batches per step
        const uint32_t total = sm.qcount[qpar];
        if (threadIdx.x == 0) sm.qcount[qpar ^ 1u] = 0u;                    // the next round's counter (last read two barriers ago)
        for (uint32_t b0 = warp * 32u; b0 < total; b0 += 2u * kMcWarps * 32u) {
            uint32_t id[2]; uint4 ma[2], mb[2]; bool live[2]; uint32_t alpha[2];
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                const uint32_t i = b0 + (uint32_t)u * kMcWarps * 32u + lane;
                live[u] = i < total;
                id[u] = sm.queue[live[u] ? i : 0u];                         // dead lanes redo candidate 0 and drop the result
                const uint32_t moff = sm.words[id[u] >> 8][((id[u] >> 5) & 7u) * 4u + 1u];
                const uint4* m = p.meshlets + 2u * ((size_t)moff + (id[u] & 31u));
                ma[u] = __ldg(m); mb[u] = __ldg(m + 1);
            }
#pragma unroll
            for (int u = 0; u < 2; ++u)
                alpha[u] = __ldg(reinterpret_cast<const uint32_t*>(p.materials + (size_t)(mb[u].w & 0xFFFFu) * ORBIT_MATERIAL_STRIDE_BYTES + ORBIT_MATERIAL_ALPHA_MODE_OFFSET));
            bool pre[2];
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                const float* mvr = &sm.mv[id[u] >> 8][(id[u] >> 5) & 7u][0];
                const ItemTest t = test_item<-1>(s_cull[s_view[id[u] >> 8]], *reinterpret_cast<const float4*>(mvr), *reinterpret_cast<const float4*>(mvr + 4),
                                                 *reinterpret_cast<const float4*>(mvr + 8), *reinterpret_cast<const float4*>(mvr + 12), mvr[16],
                                                 __uint_as_float(ma[u].x), __uint_as_float(ma[u].y), __uint_as_float(ma[u].z), __uint_as_float(ma[u].w), mb[u].x);
                pre[u] = t.pre_visible;
            }
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                // should_draw = visible && alpha passes the view's filter (meshlet_cull.comp:207); pass 1: visible_last_frame holds for every candidate
                const uint32_t w_ = id[u] >> 8, vv = s_view[w_];
                if (live[u] && pre[u] && (shl1(alpha[u]) & s_cull[vv].alpha_mode_flags) != 0u) {
                    const uint32_t r = (id[u] >> 5) & 7u, j = id[u] & 31u;
                    atomicOr(&sm.mask[w_][r], 1u << j);
                    // the command words of a survivor travel to the emit kernel through its view's side array
                    uint4* const side = views[vv].cmd_side;
                    if (side != nullptr) side[((size_t)s_rec0[w_] + r) * 32u + j] = make_uint4(mb[u].y, mb[u].z, mb[u].w, sm.words[w_][r * 4u]);
                }
            }
        }
        __syncthreads();
        // ---- E. this warp's tile: draw masks out, survivors counted per chunk of its view
        uint32_t my_draw_mask = 0u;
        if (lane < (uint32_t)R) my_draw_mask = sm.mask[warp][lane];
        if (tile < tiles_total) {
            const MeshletCullParams& pt = views[w.view];
            const uint32_t ent = __shfl_sync(0xFFFFFFFFu, my_word, (lane * 4u + 0u) & 31u);
            const uint32_t mof = __shfl_sync(0xFFFFFFFFu, my_word, (lane * 4u + 1u) & 31u);
            if (lane < (uint32_t)R && rec0 + lane < w.nrec) pt.draw_masks[rec0 + lane] = make_uint4(my_draw_mask, ent, mof, pt.cmd_side != nullptr ? 0u : 1u);
            const uint32_t tile_total = __reduce_add_sync(0xFFFFFFFFu, __popc(my_draw_mask));
            if (lane == 0u && tile_total != 0u) atomicAdd(chunk_counts + rec0 / chunk_rec, tile_total);
            warp_total += tile_total;
        }
        cur = nxt;
        cur_word = next_word;
        next_word = next2_word;
    }
    ORBIT_TRACE_STAMP(p.scan.trace, 2, 3);
    pdl_launch_dependents();
    if (lane == 0u && warp_total != 0u) atomicAdd(draw_total, warp_total);
}

// Position of the n-th (0-based) set bit of m (n < popc(m)): branch-free binary search on popcounts of halves.
__device__ __forceinline__ uint32_t select_set_bit(uint32_t m, uint32_t n) {
    uint32_t pos = 0u;
#pragma unroll
    for (uint32_t w = 16u; w != 0u; w >>= 1) {
        const uint32_t c = __popc(m & ((1u << w) - 1u));
        const bool hi = n >= c;
        n -= hi ? c : 0u;
        pos += hi ? w : 0u;
        m = hi ? (m >> w) : m;
    }
    return pos;
}

// ---------------------------------------------------------------------------------------------------------
// Second launch: ordered, OUTPUT-BALANCED emission with no inter-CTA exchange.
//   1. every CTA loads the (at most 2048) per-chunk survivor counts the test kernel accumulated and scans them in
//      shared memory: chunk prefix P. (Earlier versions published per-CTA aggregates and gathered them — three
//      more dependent global round trips in a kernel whose whole runtime is a handful of round trips.)
//   2. the T outputs are split evenly over all warps of the grid; a warp binary-searches P for the chunk holding
//      its first output, walks that chunk's draw masks 32 records at a time, and writes its outputs. Survivors
//      cluster in the visible part of the scene, so splitting by RECORDS leaves a few CTAs with 10-16x the average
//      work; splitting by OUTPUTS gives every warp the same number.
//   3. the counts of the OTHER parity are zeroed for the next call and the parity word the next test kernel reads is
//      flipped — no done-counter, fence or atomic on the way out (that exit chain was ~1/3 of this kernel's samples).
constexpr int kEmitWarps = 8;
constexpr uint32_t kEmitBulkSurvivors = 1u << 18;   // lists at least this long are emitted by every launched CTA
constexpr uint32_t kMaxRegions = 16u;   // ranks of a sharded view (orbit_draws_from_masks)
__device__ __forceinline__ void meshlet_emit_body(const MeshletCullParams& p) {
    __shared__ uint32_t s_prefix[kMaxChunks];            // inclusive survivor count up to chunk c
    __shared__ uint32_t s_warp_total[kEmitWarps];
    __shared__ uint32_t s_rec[kEmitWarps][4][32];
    __shared__ uint32_t s_payload[kEmitWarps][32 * 11];   // task-payload staging (only used when requested)
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    __shared__ uint32_t s_region[kMaxRegions + 1];        // sharded view: first record of every rank's region of the entry array
    const bool want_payload = p.task_payloads != nullptr;
    pdl_wait();
    if (p.n_regions != 0u && tid == 0) {
        uint32_t acc = 0u;
        for (uint32_t k = 0; k < p.n_regions; ++k) { s_region[k] = acc; acc += (uint32_t)min((uint64_t)__ldcg(p.region_counts + k), p.region_stride); }
        s_region[p.n_regions] = acc;
    }
    if (p.n_regions != 0u) __syncthreads();
    // record index -> entry index: identity, or (sharded view) rank k's records lie at k * region_stride
    auto entry_of = [&](uint32_t rec) -> size_t {
        if (p.n_regions == 0u) return rec;
        uint32_t k = 0u;
        while (k + 1u < p.n_regions && rec >= s_region[k + 1u]) ++k;
        return (size_t)k * p.region_stride + (rec - s_region[k]);
    };
    ORBIT_TRACE_STAMP(p.trace_emit, 3, 0);
    // Long lists want every CTA the SM can hold (their walk is bound by the loads in flight: C5, 10 M survivors: 274 / 212 /
    // 185 us per view with 1 / 2 / 3 CTAs per SM); for short ones more CTAs only repeat the chunk scan and thin out the shares
    // (C2 frame: +2.4 us with 3 instead of 2 per SM). The launch is sized for the long case; a SURPLUS CTA first looks at the
    // survivor count alone (12 bytes) and leaves at once when the list is short.
    const bool surplus = p.emit_small_grid != 0u && blockIdx.x >= p.emit_small_grid;
    if (surplus) {
        const uint2 tt = __ldcg(reinterpret_cast<const uint2*>(p.draw_total));
        const uint32_t par = __ldcg(p.chunk_parity + 1) & 1u;
        if ((par ? tt.y : tt.x) < kEmitBulkSurvivors) {
            // its share of the other parity's counters still has to be zeroed for the next call
            for (uint32_t i = blockIdx.x * blockDim.x + tid; i < kMaxChunks; i += gridDim.x * blockDim.x) p.chunk_counts[(par ^ 1u) * kMaxChunks + i] = 0u;
            return;
        }
    }
    // both halves of the chunk counts are requested before the parity is known: one round trip instead of two
    uint32_t v0[8], v1[8];
    {
        const uint4* c0 = reinterpret_cast<const uint4*>(p.chunk_counts) + tid * 2u;
        const uint4* c1 = reinterpret_cast<const uint4*>(p.chunk_counts + kMaxChunks) + tid * 2u;
        const uint4 a0 = __ldcg(c0), a1 = __ldcg(c0 + 1), b0 = __ldcg(c1), b1 = __ldcg(c1 + 1);
        v0[0] = a0.x; v0[1] = a0.y; v0[2] = a0.z; v0[3] = a0.w; v0[4] = a1.x; v0[5] = a1.y; v0[6] = a1.z; v0[7] = a1.w;
        v1[0] = b0.x; v1[1] = b0.y; v1[2] = b0.z; v1[3] = b0.w; v1[4] = b1.x; v1[5] = b1.y; v1[6] = b1.z; v1[7] = b1.w;
    }
    // both parities' totals in ONE 8-byte load (two 4-byte loads get the second one predicated on the parity by ptxas,
    // even as volatile asm: a dependent round trip in a kernel that is only a handful of round trips long)
    const uint2 t01 = __ldcg(reinterpret_cast<const uint2*>(p.draw_total));
    const uint32_t t0 = t01.x, t1 = t01.y;
    uint32_t nrec = __ldcg(p.dispatch_words);
    const uint32_t parity = __ldcg(p.chunk_parity + 1) & 1u;   // word B: the half the test kernel of this call used
    const uint32_t grand_total = parity ? t1 : t0;
    ORBIT_TRACE_STAMP_AFTER(p.trace_emit, 3, 1, grand_total + v0[0] + v1[7]);
    if ((uint64_t)nrec > p.capacity_records) nrec = (uint32_t)p.capacity_records;
    // zero the other parity's counters for the next call (it runs after this kernel in stream order)
    for (uint32_t i = blockIdx.x * blockDim.x + tid; i < kMaxChunks; i += gridDim.x * blockDim.x) p.chunk_counts[(parity ^ 1u) * kMaxChunks + i] = 0u;
    if (blockIdx.x == 0 && tid == 0) { p.draw_total[parity ^ 1u] = 0u; p.chunk_parity[0] = parity ^ 1u; }   // word A for the next call
    const uint32_t eff_grid = (grand_total >= kEmitBulkSurvivors || p.emit_small_grid == 0u) ? gridDim.x : min(gridDim.x, p.emit_small_grid);
    const uint32_t gw = blockIdx.x * kEmitWarps + warp, GW = eff_grid * kEmitWarps;
    if (grand_total != 0u) {
        const uint32_t chunk_rec = 1u << chunk_shift_of(nrec);
        const uint32_t nchunks = (nrec + chunk_rec - 1u) / chunk_rec;
        // ---- 1. chunk counts -> inclusive prefix in shared memory (8 consecutive chunks per thread)
        uint32_t v[8], local = 0u;
#pragma unroll
        for (int k = 0; k < 8; ++k) { v[k] = parity ? v1[k] : v0[k]; local += v[k]; }
        uint32_t incl = local;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, d);
            if (lane >= (uint32_t)d) incl += t;
        }
        if (lane == 31u) s_warp_total[warp] = incl;
        __syncthreads();
        uint32_t run = incl - local;
#pragma unroll
        for (int w = 0; w < kEmitWarps; ++w) if ((uint32_t)w < warp) run += s_warp_total[w];
#pragma unroll
        for (int k = 0; k < 8; ++k) { run += v[k]; s_prefix[tid * 8u + (uint32_t)k] = run; }
        __syncthreads();
        const uint32_t total = s_prefix[kMaxChunks - 1u];
        ORBIT_TRACE_STAMP(p.trace_emit, 3, 2 + 0 * (total & 1u));
        if (blockIdx.x == 0 && tid == 0) {
            p.draw_words[0] = total;   // exact count even when it exceeds capacity
            if ((uint64_t)total > p.capacity_draws) *p.overflow_flag = 1u;
        }
        // ---- 2. my share of the outputs
        const uint32_t o_begin = (uint32_t)(((uint64_t)total * gw) / GW);
        const uint32_t o_end = (uint32_t)(((uint64_t)total * (gw + 1u)) / GW);
        uint32_t* const sr = &s_rec[warp][0][0];
        uint32_t* const stage = &s_payload[warp][0];          // command staging (the task-payload pass below runs after the emission)
        if (o_begin < o_end && chunk_rec == 32u) {
            // ---- 2a. lists of at most 65 536 records (a chunk IS one 32-record group): every LANE locates its own output.
            // The prefix gives the group of output o and its rank k inside it; the lane reads the group's 32 mask words (32
            // independent 4-byte loads: lanes of the same group hit the same sectors), finds the record holding the k-th survivor,
            // then fetches the record's entry and the command words together. Two dependent round trips however sparse the
            // survivors are — the group walk below pays one per 4 groups, and a share of ~30 outputs in a sparse stretch of the
            // C2 lists took up to seven (profiles/r2_frame_timeline_before.txt: emitted after 3.3 .. 7.9 us).
            const bool side_possible = p.cmd_side != nullptr && p.cull.occlusion_pass != 2u;   // pass-2 entries never have side words
            for (uint32_t ob = o_begin; ob < o_end; ob += 32u) {
                const bool act = ob + lane < o_end;
                const uint32_t o = act ? ob + lane : o_end - 1u;                // idle lanes shadow the share's last output
                uint32_t lo = 0u, hi = nchunks - 1u;
#pragma unroll 1
                while (__any_sync(0xFFFFFFFFu, lo < hi)) {
                    if (lo < hi) {
                        const uint32_t mid = (lo + hi) >> 1;
                        if (s_prefix[mid] > o) hi = mid; else lo = mid + 1u;
                    }
                }
                const uint32_t k = o - (lo ? s_prefix[lo - 1u] : 0u);
                const uint32_t rec0 = lo * 32u;
                uint32_t m[32];
                if (p.n_regions == 0u) {            // entries in record order: 32 plain loads, nothing between them
                    const uint32_t* const mw = reinterpret_cast<const uint32_t*>(p.draw_masks + rec0);
#pragma unroll
                    for (uint32_t r = 0; r < 32u; ++r) m[r] = rec0 + r < nrec ? __ldcg(mw + 4u * r) : 0u;
                } else {                            // sharded view: a group may straddle two ranks' regions
#pragma unroll 1
                    for (uint32_t r = 0; r < 32u; ++r) {
                        const uint32_t v = rec0 + r < nrec ? __ldcg(reinterpret_cast<const uint32_t*>(p.draw_masks + entry_of(rec0 + r))) : 0u;
#pragma unroll
                        for (uint32_t q = 0; q < 32u; ++q) if (q == r) m[q] = v;
                    }
                }
                uint32_t acc = 0u, rsel = 0u, ksel = 0u, msel = 1u;
#pragma unroll
                for (uint32_t r = 0; r < 32u; ++r) {
                    const uint32_t pc = (uint32_t)__popc(m[r]);
                    if (k >= acc && k < acc + pc) { rsel = r; ksel = k - acc; msel = m[r]; }
                    acc += pc;
                }
                const uint32_t j = select_set_bit(msel, ksel);
                const uint32_t rec = rec0 + rsel;
                const uint4 e = __ldcg(p.draw_masks + entry_of(rec));
                uint4 cw = make_uint4(0u, 0u, 0u, 0u);
                if (side_possible) cw = __ldcg(p.cmd_side + (size_t)rec * 32u + j);
                const uint32_t midx = e.z + j;
                if (e.w & 1u) { const uint4 mb = __ldg(p.meshlets + 2u * (size_t)midx + 1); cw = make_uint4(mb.y, mb.z, mb.w, 0u); }
                else if (!side_possible) cw = __ldcg(p.cmd_side + (size_t)rec * 32u + j);
                __syncwarp();
                if (act) store_command(stage + lane * 7u, cw.x, cw.y, cw.z, e.y, midx);
                __syncwarp();
                const uint64_t first = ob;
                uint64_t n_out = min(32u, o_end - ob);
                if (first >= p.capacity_draws) n_out = 0u; else if (first + n_out > p.capacity_draws) n_out = p.capacity_draws - first;
                uint32_t* const dst = p.draw_words + 1u + first * 7u;
                for (uint32_t w = lane; w < (uint32_t)n_out * 7u; w += 32u) dst[w] = stage[w];
            }
            ORBIT_TRACE_STAMP(p.trace_emit, 3, 6);
        } else if (o_begin < o_end) {
            // ---- 2b. longer lists: walk the groups of the share
            // chunk holding output o_begin: first c with P[c] > o_begin
            uint32_t lo = 0u, hi = nchunks - 1u;
            while (lo < hi) {
                const uint32_t mid = (lo + hi) >> 1;
                if (s_prefix[mid] > o_begin) hi = mid; else lo = mid + 1u;
            }
            ORBIT_TRACE_STAMP_AFTER(p.trace_emit, 3, 4, lo);
            uint32_t running = lo ? s_prefix[lo - 1u] : 0u;               // outputs before record `rec`
            uint32_t rec = lo * chunk_rec;
            // At a chunk boundary the prefix tells whether the chunk holds any survivor: empty chunks are stepped over
            // without touching memory (a warp whose share of the outputs straddles an invisible stretch of the record
            // list would otherwise pay one dependent load per 32 records of it), and the masks of the next group are
            // requested before the current group is processed.
            uint32_t cur_chunk = lo, in_chunk = 0u;                        // rec == cur_chunk * chunk_rec + in_chunk
            auto advance = [&]() -> uint32_t {                               // next group of 32 records worth loading
                in_chunk += 32u;
                if (in_chunk >= chunk_rec) {
                    in_chunk = 0u;
                    ++cur_chunk;
                    while (cur_chunk < nchunks && s_prefix[cur_chunk] == s_prefix[cur_chunk - 1u]) ++cur_chunk;
                }
                return cur_chunk < nchunks ? cur_chunk * chunk_rec + in_chunk : nrec;
            };
            auto load_masks = [&](uint32_t r) -> uint4 {
                const uint32_t my = r + lane;
                return my < nrec ? __ldcg(p.draw_masks + entry_of(my)) : make_uint4(0u, 0u, 0u, 0u);
            };
            // Four groups of 32 records in flight: a warp whose share of the outputs lies in a sparsely surviving stretch
            // walks many groups for its ~30 outputs, one dependent L2 round trip each (that tail was half of this kernel's
            // time on the C2 early pass; profiles/r2_frame_timeline.txt).
            constexpr int kDepth = 4;
            uint32_t recs[kDepth]; uint4 es[kDepth];
            recs[0] = rec; es[0] = load_masks(rec);
#pragma unroll
            for (int u = 1; u < kDepth; ++u) { recs[u] = advance(); es[u] = load_masks(recs[u]); }
#ifdef ORBIT_TRACE
            bool trace_first_group = false; uint32_t trace_groups = 0u;
#endif
            bool more = true;
            while (more) {
#pragma unroll
                for (int u = 0; u < kDepth; ++u) {
                    if (!(running < o_end && recs[u] < nrec)) { more = false; break; }
                    const uint4 e = es[u];
                    const uint32_t group_rec = recs[u];
                    recs[u] = advance();
                    es[u] = load_masks(recs[u]);                             // speculative: unused when the share ends first
                    const uint32_t dm = e.x, entity = e.y, moff = e.z;
                    const uint32_t pc = __popc(dm);
                    uint32_t inc = pc;
#pragma unroll
                    for (int d = 1; d < 32; d <<= 1) {
                        const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, inc, d);
                        if (lane >= (uint32_t)d) inc += t;
                    }
                    const uint32_t step_total = __shfl_sync(0xFFFFFFFFu, inc, 31);
#ifdef ORBIT_TRACE
                    if (!trace_first_group) { trace_first_group = true; ORBIT_TRACE_STAMP_AFTER(p.trace_emit, 3, 5, step_total); }
                    ++trace_groups;
#endif
                    if (running + step_total > o_begin) {
                        __syncwarp();
                        sr[lane] = inc; sr[32 + lane] = dm; sr[64 + lane] = entity; sr[96 + lane] = moff | (e.w << 31);
                        __syncwarp();
                        const uint32_t l0 = o_begin > running ? o_begin - running : 0u;            // first local output of mine
                        const uint32_t l1 = min(step_total, o_end - running);                      // one past my last local output
                        // 32 outputs per step: every lane builds its command (7 words) in shared memory, then the warp writes the
                        // step's commands — contiguous in the output — as consecutive words (seven 128-byte stores instead of seven
                        // 28-byte-strided ones that touch 28 sectors each; the emit kernel writes 28 B per survivor and was store-bound
                        // at C5 scale)
                        // Two batches of 32 outputs per iteration: both batches' command words are requested before the first is
                        // staged, so a warp has two dependent L2 / DRAM round trips in flight instead of one (the walk of a long
                        // list is one such round trip per 32 outputs per warp: at C5 scale — 10 M survivors, 130 batches per warp —
                        // that chain, not bandwidth, set the kernel's 223 us).
                        for (uint32_t ol0 = l0; ol0 < l1; ol0 += 64u) {
                            uint4 cw[2]; uint32_t ent[2], midx[2]; bool act[2];
#pragma unroll
                            for (uint32_t k = 0; k < 2u; ++k) {
                                const uint32_t ol = ol0 + 32u * k + lane;
                                act[k] = ol < l1;
                                cw[k] = make_uint4(0u, 0u, 0u, 0u); ent[k] = 0u; midx[k] = 0u;
                                if (act[k]) {
                                    uint32_t a = 0u, b = 31u;
#pragma unroll
                                    for (int it = 0; it < 5; ++it) {
                                        const uint32_t mid = (a + b) >> 1;
                                        if (sr[mid] > ol) b = mid; else a = mid + 1u;
                                    }
                                    const uint32_t r = a;
                                    const uint32_t excl = r ? sr[r - 1u] : 0u;
                                    const uint32_t j = select_set_bit(sr[32 + r], ol - excl);   // (ol-excl)-th survivor of the record
                                    const uint32_t mo = sr[96 + r];
                                    midx[k] = (mo & 0x7FFFFFFFu) + j;
                                    ent[k] = sr[64 + r];
                                    // command words: from the side array the test kernel filled (x,y,z = vertex_offset, data_offset, packed
                                    // counts), or — pass 2, whose candidates do not carry them — from the meshlet itself
                                    if (mo >> 31) { const uint4 mb = __ldg(p.meshlets + 2u * (size_t)midx[k] + 1); cw[k] = make_uint4(mb.y, mb.z, mb.w, 0u); }
                                    else cw[k] = __ldcg(p.cmd_side + (size_t)(group_rec + r) * 32u + j);
                                }
                            }
#pragma unroll
                            for (uint32_t k = 0; k < 2u; ++k) {
                                const uint32_t ob = ol0 + 32u * k;                               // first local output of this batch
                                if (ob < l1) {                                                   // warp-uniform
                                    // every lane builds its command (7 words) in shared memory, then the warp writes the batch's
                                    // commands — contiguous in the output — as consecutive words (seven 128-byte stores instead of
                                    // seven 28-byte-strided ones that touch 28 sectors each)
                                    __syncwarp();
                                    if (act[k]) store_command(stage + lane * 7u, cw[k].x, cw[k].y, cw[k].z, ent[k], midx[k]);
                                    __syncwarp();
                                    const uint64_t first = (uint64_t)running + ob;               // index of the batch's first command
                                    uint64_t n_out = min(32u, l1 - ob);
                                    if (first >= p.capacity_draws) n_out = 0u; else if (first + n_out > p.capacity_draws) n_out = p.capacity_draws - first;
                                    uint32_t* const dst = p.draw_words + 1u + first * 7u;
                                    for (uint32_t w = lane; w < (uint32_t)n_out * 7u; w += 32u) dst[w] = stage[w];
                                }
                            }
                        }
                    }
                    running += step_total;
                }
            }
            ORBIT_TRACE_STAMP(p.trace_emit, 3, 6);
            ORBIT_TRACE_VALUE(p.trace_emit, 8, trace_groups);
            ORBIT_TRACE_VALUE(p.trace_emit, 9, o_end - o_begin);
        }
    } else if (blockIdx.x == 0 && tid == 0) {
        p.draw_words[0] = 0u;   // nothing survived (the steady-state late pass)
    }
#ifdef ORBIT_TRACE
    __syncthreads();
    ORBIT_TRACE_STAMP(p.trace_emit, 3, 3);
#endif
    pdl_launch_dependents();   // after the emission: an early trigger measured 20% slower when there is a lot to emit
    if (want_payload) {
        // MeshTaskPayload + emitted task count per record (indices ascending by lane — the task shader's atomicAdd
        // order is arbitrary). One LANE per record packs the 11 words; the warp stages its 32 consecutive records
        // (1408 contiguous bytes of the payload array) in shared memory and writes them out coalesced.
        uint32_t* const st = &s_payload[warp][0];
        for (uint32_t base = gw * 32u; base < nrec; base += GW * 32u) {
            const uint32_t r = base + lane;
            uint4 e = make_uint4(0u, 0u, 0u, 0u);
            if (r < nrec) e = __ldcg(p.draw_masks + entry_of(r));
            uint32_t m = e.x;
            __syncwarp();
            st[lane * 11u] = __popc(m); st[lane * 11u + 1u] = e.y; st[lane * 11u + 2u] = e.z;
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                uint32_t packed_idx = 0u;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const uint32_t b = (uint32_t)__ffs((int)m);          // 0 when m is empty
                    packed_idx |= (b ? b - 1u : 0u) << (8 * k);
                    m &= m - 1u;                                         // 0 & 0xFFFFFFFF stays 0
                }
                st[lane * 11u + 3u + (uint32_t)q] = packed_idx;
            }
            __syncwarp();
            const uint32_t nwords = min(32u, nrec - base) * 11u;
            uint32_t* const tp = p.task_payloads + (size_t)base * 11u;
            for (uint32_t i = lane; i < nwords; i += 32u) tp[i] = st[i];
        }
    }
}

__global__ void __launch_bounds__(kEmitWarps * 32) meshlet_emit_kernel(const __grid_constant__ MeshletCullParams p) { meshlet_emit_body(p); }

// Two lists in one launch (fused LATE + MAIN: blockIdx.y = 0 emits the LATE list, 1 the MAIN list; each list's CTAs only ever
// look at blockIdx.x / gridDim.x): the LATE list of a steady frame is empty, and its emit kernel was 3 us of launch + look.
struct EmitPair { MeshletCullParams list[2]; };
__global__ void __launch_bounds__(kEmitWarps * 32) meshlet_emit_pair_kernel(const __grid_constant__ EmitPair pp) { meshlet_emit_body(pp.list[blockIdx.y]); }
// The same for up to 16 lists (orbit_meshlet_cull_views): blockIdx.y = view.
__global__ void __launch_bounds__(kEmitWarps * 32) meshlet_emit_views_kernel(const __grid_constant__ MeshletViewsParams pv) { meshlet_emit_body(pv.view[blockIdx.y]); }

// ---------------------------------------------------------------------------------------------------------
// Multi-GPU (SURVEY §8e, meshlet ranges of one view): a rank that only TESTS its records ships the 16-byte
// {draw mask, entity, meshlet offset, 1} entries instead of 28-byte draw commands (C3: 28 MB instead of 229 MB to the
// rank that submits the draws) into its own region of that rank's entry array; the receiving rank reads the regions in rank
// order — rank-major = canonical record order —, recounts the survivors per chunk and runs the ordinary emit kernel.
//
// Stores this rank's entries [0, own count) into its region of the receiving rank's entry array (dst_region: usually
// peer-mapped, so these are NVLink stores) and its record count into dst_count — no rank needs another rank's count, so the
// exchange has no collective besides the closing fence. The count comes from the dispatch buffer's header on the device.
__global__ void __launch_bounds__(256) record_masks_put_kernel(const uint4* __restrict__ src, const uint32_t* __restrict__ dispatch_words,
                                                               uint4* __restrict__ dst_region, uint32_t* __restrict__ dst_count, uint64_t capacity) {
    const uint64_t n = min((uint64_t)__ldcg(dispatch_words), capacity);
    if (blockIdx.x == 0 && threadIdx.x == 0) *dst_count = (uint32_t)n;
    const uint64_t gsize = (uint64_t)gridDim.x * blockDim.x;
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (; i + 3u * gsize < n; i += 4u * gsize) {                          // four independent 16-byte stores in flight (NVLink)
        uint4 v[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) v[k] = __ldcg(src + i + (uint64_t)k * gsize);
#pragma unroll
        for (int k = 0; k < 4; ++k) __stcg(dst_region + i + (uint64_t)k * gsize, v[k]);
    }
    for (; i < n; i += gsize) __stcg(dst_region + i, __ldcg(src + i));
}

// Survivors per chunk of the combined list (same double-buffered scratch protocol as the test kernels, so the emit kernel
// that follows cannot tell the difference) and the combined record count as a dispatch-buffer header for it.
__global__ void __launch_bounds__(256) record_masks_recount_kernel(const __grid_constant__ MeshletCullParams p, uint32_t* __restrict__ header_out) {
    __shared__ uint32_t s_region[kMaxRegions + 1];
    if (threadIdx.x == 0) {
        uint32_t acc = 0u;
        for (uint32_t k = 0; k < p.n_regions; ++k) { s_region[k] = acc; acc += (uint32_t)min((uint64_t)__ldcg(p.region_counts + k), p.region_stride); }
        s_region[p.n_regions] = acc;
    }
    __syncthreads();
    const uint32_t nrec = (uint32_t)min((uint64_t)s_region[p.n_regions], p.capacity_records);
    const uint32_t chunk_shift = chunk_shift_of(nrec);
    const uint32_t half = __ldcg(p.chunk_parity) & 1u;
    if (blockIdx.x == 0 && threadIdx.x == 0) { p.chunk_parity[1] = half; header_out[0] = nrec; header_out[1] = 1u; header_out[2] = 1u; }
    uint32_t* const chunk_counts = p.chunk_counts + half * kMaxChunks;
    const uint32_t lane = threadIdx.x & 31u;
    uint32_t mine = 0u;
    // a warp covers 32 consecutive records = at most one chunk (chunks are >= 32 records and 32-aligned)
    for (uint64_t base = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) & ~31ull; base < nrec; base += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t r = (uint32_t)base + lane;
        uint32_t pc = 0u;
        if (r < nrec) {
            uint32_t k = 0u;
            while (k + 1u < p.n_regions && r >= s_region[k + 1u]) ++k;
            pc = (uint32_t)__popc(__ldcg(reinterpret_cast<const uint32_t*>(p.draw_masks + (size_t)k * p.region_stride + (r - s_region[k]))));
        }
        const uint32_t s = __reduce_add_sync(0xFFFFFFFFu, pc);
        if (lane == 0u && s != 0u) { atomicAdd(chunk_counts + (uint32_t)(base >> chunk_shift), s); mine += s; }
    }
    if (mine != 0u) atomicAdd(p.draw_total + half, mine);
}

cudaError_t launch_record_masks_put(const uint4* src, const uint32_t* dispatch_words, uint4* dst_region, uint32_t* dst_count, uint64_t capacity,
                                    int grid, cudaStream_t s) {
    record_masks_put_kernel<<<grid, 256, 0, s>>>(src, dispatch_words, dst_region, dst_count, capacity);
    return cudaGetLastError();
}

cudaError_t launch_draws_from_masks(const MeshletCullParams& p, uint32_t* header, int grid, int emit_grid, cudaStream_t s) {
    record_masks_recount_kernel<<<grid, 256, 0, s>>>(p, header);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    return launch_kernel(meshlet_emit_kernel, dim3(emit_grid), dim3(kEmitWarps * 32), 0, s, p);
}

// ---- launch plumbing ---------------------------------------------------------------------------------------
struct TestVariant { bool packed; bool pass2; int proj; };
static TestVariant variant_of(const OrbitCullInfo& ci) {
    const bool mocc = ci.meshlet_visibility_buffer != ORBIT_NO_BUFFER;
    TestVariant v;
    v.packed = ci.occlusion_pass == 1u && mocc;
    v.pass2 = ci.occlusion_pass == 2u && mocc;
    v.proj = ci.projection_type <= 1u ? (int)ci.projection_type : -1;
    return v;
}

#ifndef ORBIT_TILE_RECORDS
#define ORBIT_TILE_RECORDS 4
#endif
constexpr int kTileR = ORBIT_TILE_RECORDS;   // records per warp tile of the direct test kernel
#ifndef ORBIT_PACKED_RECORDS
#define ORBIT_PACKED_RECORDS 8
#endif
constexpr int kPackedR = ORBIT_PACKED_RECORDS;   // records per warp tile of the packed (pass 1) test kernel
static constexpr size_t direct_smem_bytes() { return 128u + sizeof(WarpSmem<kTileR>) * kDwWarps; }

template <bool kPass2, int kProj>
static cudaError_t launch_stream(const MeshletCullParams& p, int grid, cudaStream_t stream, int* occupancy) {
    if (occupancy) {
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(occupancy, meshlet_test_direct_kernel<kTileR, kPass2, kProj>, kDwThreads, direct_smem_bytes());
        return cudaSuccess;
    }
    return launch_kernel(meshlet_test_direct_kernel<kTileR, kPass2, kProj>, dim3(grid), dim3(kDwThreads), direct_smem_bytes(), stream, p);
}

// The direct test kernels use more than 48 KB of dynamic shared memory: opt in once per DEVICE (the attribute is per device,
// so this is called from orbit_ctx_create with the context's device current).
cudaError_t meshlet_cull_configure_device() {
    cudaError_t e;
#define ORBIT_SET(kp2, proj) \
    e = cudaFuncSetAttribute(meshlet_test_direct_kernel<kTileR, kp2, proj>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)direct_smem_bytes()); \
    if (e != cudaSuccess) return e;
    ORBIT_SET(false, 0) ORBIT_SET(false, 1) ORBIT_SET(false, -1) ORBIT_SET(true, 0) ORBIT_SET(true, 1) ORBIT_SET(true, -1)
#undef ORBIT_SET
#define ORBIT_SET(kp2, proj) \
    e = cudaFuncSetAttribute(meshlet_test_views_kernel<kTileR, kp2, proj>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)direct_smem_bytes()); \
    if (e != cudaSuccess) return e;
    ORBIT_SET(false, 0) ORBIT_SET(false, 1) ORBIT_SET(false, -1)
    return cudaSuccess;
}

// The same for the batched pass-2 test kernels, called by the first orbit_meshlet_cull_views_occlusion call that needs them
// rather than by orbit_ctx_create: setting the attribute loads the kernel, and what orbit_ctx_create loads or allocates shifts
// the device memory allocated after it, to which the single-view stages are sensitive (DESIGN.md §4, batched views).
cudaError_t meshlet_cull_configure_views_pass2() {
    cudaError_t e;
    ORBIT_SET(true, 0) ORBIT_SET(true, 1) ORBIT_SET(true, -1)
#undef ORBIT_SET
    return cudaSuccess;
}

static cudaError_t launch_test(const MeshletCullParams& p, int grid, cudaStream_t stream, int* occupancy) {
    const TestVariant v = variant_of(p.cull);
    if (v.packed) {
        // the packed kernel fills its 32-lane test batches from a whole tile of 8 records (a 4-record tile's batch is 44 % full on C2)
        if (occupancy) { cudaOccupancyMaxActiveBlocksPerMultiprocessor(occupancy, meshlet_test_packed_kernel<kPackedR>, kMcThreads, 0); return cudaSuccess; }
        return launch_kernel(meshlet_test_packed_kernel<kPackedR>, dim3(grid), dim3(kMcThreads), 0, stream, p);
    }
    if (v.pass2) {
        if (v.proj == 0) return launch_stream<true, 0>(p, grid, stream, occupancy);
        if (v.proj == 1) return launch_stream<true, 1>(p, grid, stream, occupancy);
        return launch_stream<true, -1>(p, grid, stream, occupancy);
    }
    if (v.proj == 0) return launch_stream<false, 0>(p, grid, stream, occupancy);
    if (v.proj == 1) return launch_stream<false, 1>(p, grid, stream, occupancy);
    return launch_stream<false, -1>(p, grid, stream, occupancy);
}

// Index of the kernel variant a CullInfo selects (api.cu caches one occupancy per variant).
int meshlet_cull_variant_index(const OrbitCullInfo& ci) {
    const TestVariant v = variant_of(ci);
    return v.packed ? 0 : 1 + (v.pass2 ? 3 : 0) + (v.proj + 1);
}

int meshlet_cull_max_ctas_per_sm(const MeshletCullParams& p) {
    int n = 0;
    launch_test(p, 0, nullptr, &n);
    return n;
}

cudaError_t launch_meshlet_emit(const MeshletCullParams& p, int emit_grid, cudaStream_t stream) {
    return launch_kernel(meshlet_emit_kernel, dim3(emit_grid), dim3(kEmitWarps * 32), 0, stream, p);
}
cudaError_t launch_meshlet_emit_pair(const MeshletCullParams& a, const MeshletCullParams& b, int emit_grid, cudaStream_t stream) {
    EmitPair pp;
    pp.list[0] = a; pp.list[1] = b;
    return launch_kernel(meshlet_emit_pair_kernel, dim3(emit_grid, 2), dim3(kEmitWarps * 32), 0, stream, pp);
}

cudaError_t launch_meshlet_cull(const MeshletCullParams& p, int grid, int emit_grid, cudaStream_t stream) {
    if (grid > 0) {
        cudaError_t e = launch_test(p, grid, stream, nullptr);
        if (e != cudaSuccess) return e;
    }
    if (emit_grid > 0) return launch_kernel(meshlet_emit_kernel, dim3(emit_grid), dim3(kEmitWarps * 32), 0, stream, p);
    return cudaSuccess;
}

template <bool kPass2, int kProj>
static cudaError_t launch_views_test(const MeshletViewsParams& pv, int grid, cudaStream_t stream, int* occupancy) {
    if (occupancy) {
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(occupancy, meshlet_test_views_kernel<kTileR, kPass2, kProj>, kDwThreads, direct_smem_bytes());
        return cudaSuccess;
    }
    return launch_kernel(meshlet_test_views_kernel<kTileR, kPass2, kProj>, dim3(grid), dim3(kDwThreads), direct_smem_bytes(), stream, pv);
}

// the batched test kernel of the variant the views' CullInfo selects (all views of a call select the same one): as for a single view
static cudaError_t launch_views_test_any(const MeshletViewsParams& pv, const OrbitCullInfo& ci, int grid, cudaStream_t stream, int* occupancy) {
    const TestVariant v = variant_of(ci);
    if (v.packed) {
        if (occupancy) { cudaOccupancyMaxActiveBlocksPerMultiprocessor(occupancy, meshlet_test_packed_views_kernel<kPackedR>, kMcThreads, 0); return cudaSuccess; }
        return launch_kernel(meshlet_test_packed_views_kernel<kPackedR>, dim3(grid), dim3(kMcThreads), 0, stream, pv);
    }
    if (v.pass2) {
        if (v.proj == 0) return launch_views_test<true, 0>(pv, grid, stream, occupancy);
        if (v.proj == 1) return launch_views_test<true, 1>(pv, grid, stream, occupancy);
        return launch_views_test<true, -1>(pv, grid, stream, occupancy);
    }
    if (v.proj == 0) return launch_views_test<false, 0>(pv, grid, stream, occupancy);
    if (v.proj == 1) return launch_views_test<false, 1>(pv, grid, stream, occupancy);
    return launch_views_test<false, -1>(pv, grid, stream, occupancy);
}

int meshlet_cull_views_max_ctas_per_sm(const OrbitCullInfo& ci) {
    int n = 0;
    launch_views_test_any(MeshletViewsParams{}, ci, 0, nullptr, &n);
    return n;
}

// test kernel over the concatenated lists (one persistent wave), then one emit launch with a row of emit_grid_per_view CTAs per view
cudaError_t launch_meshlet_cull_views(const MeshletViewsParams& pv, int grid, int emit_grid_per_view, cudaStream_t stream) {
    cudaError_t e = launch_views_test_any(pv, pv.view[0].cull, grid, stream, nullptr);
    if (e != cudaSuccess) return e;
    return launch_kernel(meshlet_emit_views_kernel, dim3(emit_grid_per_view, pv.n_views), dim3(kEmitWarps * 32), 0, stream, pv);
}

int meshlet_emit_max_ctas_per_sm() {
    int n = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, meshlet_emit_kernel, kEmitWarps * 32, 0);
    return n;
}

}  // namespace orbit
