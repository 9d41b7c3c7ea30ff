// orbit_passes.hpp — header-only C++ mirror of the reference's culling-pass interface over the C ABI.
//
// The reference's host is Rust (no toolchain in the build image); this is the compiled-language host side the
// parity tests can build here. Names and argument meaning follow src/passes/draw_gen.rs and src/passes/cluster.rs:
//   CullInfo / OcclusionCullInfo / Projection / AlphaModeFlags   draw_gen.rs:24-203,630-641; camera.rs:66-98
//   CullInfo::to_gpu                                             draw_gen.rs:121-203
//   create_meshlet_dispatch_command                              draw_gen.rs:327-380
//   create_meshlet_draw_commands                                 draw_gen.rs:382-435
//   DepthPyramid::{new,resize,update}                            draw_gen.rs:451-567
//   ClusterSettings::{tile_counts,cluster_grid_info}             cluster.rs:35-72
// Failure behaviour: the reference asserts / unwraps; here a failed call throws std::runtime_error.
#pragma once
#include <cmath>
#include <cstring>
#include <stdexcept>
#include <string>
#include <vector>
#include "orbit_cuda.h"

namespace orbit_host {

inline void check(int rc, const char* what) {
    if (rc != ORBIT_OK) throw std::runtime_error(std::string(what) + ": " + orbit_error_string(rc));
}

struct AlphaModeFlags { enum : uint32_t { OPAQUE = 1, MASKED = 2, TRANSPARENT = 4, ALL = 7 }; };

struct Projection {
    enum Kind { Perspective, Orthographic } kind = Perspective;
    float fov = 0, near_clip = 0.01f, far_clip = 0, half_width = 0;
    static Projection perspective(float fov, float near_clip) { Projection p; p.kind = Perspective; p.fov = fov; p.near_clip = near_clip; return p; }
    static Projection orthographic(float half_width, float near_clip, float far_clip) {
        Projection p; p.kind = Orthographic; p.half_width = half_width; p.near_clip = near_clip; p.far_clip = far_clip; return p;
    }
};

struct OcclusionCullInfo {
    enum Kind { None = 0, VisibilityRead = 1, VisibilityWrite = 2 } kind = None;
    uint32_t* visibility_buffer = nullptr;          // device
    uint32_t* meshlet_visibility_buffer = nullptr;  // device; nullptr disables meshlet occlusion culling
    orbit_hiz* depth_pyramid = nullptr;
    uint32_t noskip_alphamode = 0;
    float aspect_ratio = 1.0f;
    uint32_t pass_index() const { return (uint32_t)kind; }
};

struct CullInfo {
    float view_matrix[16];                       // column-major (glam Mat4 memory order)
    std::vector<float> view_space_cull_planes;   // 4 floats per plane, at most 12 planes
    Projection projection;
    OcclusionCullInfo occlusion_culling;
    uint32_t alpha_mode_filter = AlphaModeFlags::OPAQUE | AlphaModeFlags::MASKED;
    uint32_t lod_range_start = 0, lod_range_end = 8;
    float lod_base = 16.0f, lod_step = 2.0f;
    float lod_target_pos_view_space[3] = {0, 0, 0};

    OrbitCullInfo to_gpu() const {  // draw_gen.rs:121-203
        const size_t n = view_space_cull_planes.size() / 4;
        if (n > ORBIT_MAX_CULL_PLANES) throw std::runtime_error("assert!(cull_planes.len() <= MAX_CULL_PLANES)");
        OrbitCullInfo g;
        std::memset(&g, 0, sizeof(g));
        std::memcpy(&g.view_matrix, view_matrix, 64);
        if (n) std::memcpy(g.cull_planes, view_space_cull_planes.data(), n * 16);
        g.cull_plane_count = (uint32_t)n;
        g.alpha_mode_flags = alpha_mode_filter;
        const OcclusionCullInfo& oc = occlusion_culling;
        g.occlusion_pass = oc.pass_index();
        g.visibility_buffer = oc.visibility_buffer ? 0u : ORBIT_NO_BUFFER;
        g.meshlet_visibility_buffer = oc.meshlet_visibility_buffer ? 0u : ORBIT_NO_BUFFER;
        g.depth_pyramid = oc.depth_pyramid ? 0u : ORBIT_NO_BUFFER;
        g.min_mesh_lod = lod_range_start;
        g.max_mesh_lod = lod_range_end - 1u;
        g.lod_base = lod_base; g.lod_step = lod_step;
        std::memcpy(g.lod_target_pos_view_space, lod_target_pos_view_space, 12);
        g.projection_type = projection.kind == Projection::Perspective ? 0u : 1u;
        if (oc.kind == OcclusionCullInfo::VisibilityWrite) {
            g.noskip_alpha_mode = oc.noskip_alphamode;
            if (projection.kind == Projection::Perspective) {
                const float f = 1.0f / std::tan(0.5f * projection.fov);
                g.p00_or_width_recip_x2 = f / oc.aspect_ratio;
                g.p11_or_height_recip_x2 = f;
                g.z_near = projection.near_clip;
            } else {
                const float width = projection.half_width * 2.0f;
                const float height = width * (1.0f / oc.aspect_ratio);
                g.p00_or_width_recip_x2 = (1.0f / width) * 2.0f;
                g.p11_or_height_recip_x2 = (1.0f / height) * 2.0f;
                g.z_near = projection.near_clip;
                g.z_far = projection.far_clip;
            }
        }
        return g;
    }
};

// Device buffers owned by GpuAssets (assets/mod.rs:230-239) and SceneData (scene.rs:358-369).
struct AssetGraphData { const void* mesh_info_buffer; const void* meshlet_buffer; const void* materials_buffer; };
struct SceneGraphData { uint32_t entity_draw_count; const void* entity_draw_buffer; const void* entity_buffer; };

inline OrbitSceneBuffers scene_buffers(const AssetGraphData& a, const SceneGraphData& s, const CullInfo& c) {
    OrbitSceneBuffers sb;
    std::memset(&sb, 0, sizeof(sb));
    sb.entity_draws = s.entity_draw_buffer; sb.mesh_infos = a.mesh_info_buffer; sb.entities = s.entity_buffer;
    sb.meshlets = a.meshlet_buffer; sb.materials = a.materials_buffer;
    sb.entity_visibility = c.occlusion_culling.visibility_buffer;
    sb.meshlet_visibility = c.occlusion_culling.meshlet_visibility_buffer;
    sb.entity_draw_count = s.entity_draw_count;
    return sb;
}

// draw_gen.rs:327-380. `meshlet_dispatch_buffer` = device memory of 12 + 16*capacity_records bytes.
inline void create_meshlet_dispatch_command(orbit_ctx* ctx, const AssetGraphData& assets, const SceneGraphData& scene, const CullInfo& cull,
                                            void* meshlet_dispatch_buffer, uint64_t capacity_records, void* stream) {
    const OrbitCullInfo g = cull.to_gpu();
    const OrbitSceneBuffers sb = scene_buffers(assets, scene, cull);
    check(orbit_entity_cull(ctx, &g, &sb, cull.occlusion_culling.depth_pyramid, meshlet_dispatch_buffer, capacity_records, stream),
          "create_meshlet_dispatch_command");
}

// draw_gen.rs:382-435. `draw_command_buffer` = device memory of 4 + 28*capacity_draws bytes.
inline void create_meshlet_draw_commands(orbit_ctx* ctx, const AssetGraphData& assets, const SceneGraphData& scene, const CullInfo& cull,
                                         const void* meshlet_dispatch_buffer, uint64_t capacity_records, void* draw_command_buffer,
                                         uint64_t capacity_draws, void* stream, void* task_payloads = nullptr) {
    const OrbitCullInfo g = cull.to_gpu();
    const OrbitSceneBuffers sb = scene_buffers(assets, scene, cull);
    check(orbit_meshlet_cull(ctx, &g, &sb, cull.occlusion_culling.depth_pyramid, meshlet_dispatch_buffer, capacity_records,
                             draw_command_buffer, capacity_draws, task_payloads, stream),
          "create_meshlet_draw_commands");
}

// The LATE cull of the depth prepass (forward.rs:266-403) and the MAIN pass's cull (forward.rs:518-548) in their fused form
// (orbit_cuda.h): both passes' dispatch buffers and draw lists from one entity kernel and one test kernel, byte for byte what the
// four separate create_* calls write. Returns false — nothing launched — when the two CullInfos are not a compatible pair
// (another camera, planes or LOD parameters, or no meshlet visibility buffer): the caller then issues the separate calls.
inline bool create_late_and_main_commands(orbit_ctx* ctx, const AssetGraphData& assets, const SceneGraphData& scene, const CullInfo& late,
                                          const CullInfo& main_pass, void* late_dispatch_buffer, void* main_dispatch_buffer,
                                          uint64_t capacity_records, void* late_draw_command_buffer, void* main_draw_command_buffer,
                                          uint64_t capacity_draws, void* stream, void* late_task_payloads = nullptr,
                                          void* main_task_payloads = nullptr) {
    const OrbitCullInfo gl = late.to_gpu(), gm = main_pass.to_gpu();
    if (!orbit_cull_pair_compatible(&gl, &gm)) return false;
    const OrbitSceneBuffers sb = scene_buffers(assets, scene, late);
    check(orbit_entity_cull_late_main(ctx, &gl, &gm, &sb, late.occlusion_culling.depth_pyramid, late_dispatch_buffer, main_dispatch_buffer,
                                      capacity_records, stream), "create_late_and_main_commands (entity stage)");
    check(orbit_meshlet_cull_late_main(ctx, &gl, &gm, &sb, late.occlusion_culling.depth_pyramid, late_dispatch_buffer, capacity_records,
                                       late_draw_command_buffer, main_draw_command_buffer, capacity_draws, late_task_payloads,
                                       main_task_payloads, stream), "create_late_and_main_commands (meshlet stage)");
    return true;
}

// draw_gen.rs:451-567
class DepthPyramid {
public:
    DepthPyramid(orbit_ctx* ctx, uint32_t width, uint32_t height) : ctx_(ctx) { check(orbit_hiz_create(ctx, width, height, &hiz_), "DepthPyramid::new"); w_ = width; h_ = height; }
    ~DepthPyramid() { orbit_hiz_destroy(hiz_); }
    DepthPyramid(const DepthPyramid&) = delete;
    DepthPyramid& operator=(const DepthPyramid&) = delete;
    void resize(uint32_t width, uint32_t height) {
        if (width == w_ && height == h_) return;
        orbit_hiz_destroy(hiz_); hiz_ = nullptr; usable = false;
        check(orbit_hiz_create(ctx_, width, height, &hiz_), "DepthPyramid::resize"); w_ = width; h_ = height;
    }
    void update(const float* depth_buffer, void* stream) { check(orbit_hiz_build(ctx_, hiz_, depth_buffer, w_, h_, stream), "DepthPyramid::update"); usable = true; }
    // the depth attachment as a wrapped CUDA array (orbit_depth_image_wrap), e.g. imported from Vulkan
    void update(const orbit_depth_image* depth_image, void* stream) { check(orbit_hiz_build_image(ctx_, hiz_, depth_image, stream), "DepthPyramid::update"); usable = true; }
    // mirror every later build into a caller-owned cudaMipmappedArray_t (orbit_hiz_attach_image), e.g. the renderer's pyramid
    // image imported from Vulkan; resize() creates a new pyramid without one (attach the new size's array then)
    void attach_image(void* cuda_mipmapped_array) { check(orbit_hiz_attach_image(ctx_, hiz_, cuda_mipmapped_array), "DepthPyramid::attach_image"); }
    orbit_hiz* get_current() const { return hiz_; }
    bool usable = false;
private:
    orbit_ctx* ctx_; orbit_hiz* hiz_ = nullptr; uint32_t w_ = 0, h_ = 0;
};

// SceneData::update_scene, scene.rs:404-492 (mesh part): the caller owns the device arrays (transforms, mesh slots, visibility
// offsets, the allocator's cursor word) and the two output buffers; `import_to_graph` hands them to the culling passes.
struct SceneData {
    OrbitSceneUpdate buffers;   // device pointers + n_entities + visibility_capacity_words (see orbit_cuda.h)
    void update_scene(orbit_ctx* ctx, const AssetGraphData& assets, void* stream) {
        OrbitSceneUpdate u = buffers;
        u.mesh_infos = assets.mesh_info_buffer;
        check(orbit_scene_update(ctx, &u, stream), "SceneData::update_scene");
    }
    // scene.rs:494-502. entity_draw_count is the host's upper bound; the kernels clamp to the device-side count.
    SceneGraphData import_to_graph() const { return SceneGraphData{buffers.n_entities, buffers.entity_draws, buffers.entity_data}; }
};

// cluster.rs:15-72
struct ClusterSettings {
    uint32_t px_size_power = 3, screen_resolution[2] = {0, 0}, z_slice_count = 32, tile_size_px_override = 0;
    float far_plane = 200.0f, luminance_cutoff = 0.25f;
    uint32_t tile_px_size() const { return tile_size_px_override ? tile_size_px_override : (1u << px_size_power); }
    void tile_counts(uint32_t out[2]) const { for (int i = 0; i < 2; ++i) out[i] = (screen_resolution[i] + tile_px_size() - 1) / tile_px_size(); }
    void cluster_grid_info(float near_, float& z_scale, float& z_bias) const {
        const float log_f_n = std::log2(far_plane / near_);
        z_scale = (float)z_slice_count / log_f_n;
        z_bias = -(((float)z_slice_count * std::log2(near_)) / log_f_n);
    }
};

// compute_clusters, cluster.rs:368-397, with the depth attachment and the cluster offset/count image as wrapped CUDA arrays
// (orbit_depth_image_wrap, orbit_cluster_grid_wrap), e.g. both imported from Vulkan: orbit_light_cluster_image_grid
inline void compute_clusters(orbit_ctx* ctx, const OrbitClusterParams& params, const orbit_depth_image* depth_image, const void* lights,
                             void* tile_masks, void* depth_bounds, void* unique_clusters, const orbit_cluster_grid* light_offset_image,
                             void* light_index_list, uint64_t capacity_indices, void* stream) {
    check(orbit_light_cluster_image_grid(ctx, &params, depth_image, lights, tile_masks, depth_bounds, unique_clusters, light_offset_image,
                                         light_index_list, capacity_indices, stream), "compute_clusters");
}

}  // namespace orbit_host
