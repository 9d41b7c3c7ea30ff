// params.cuh — kernel parameter blocks (passed by value as __grid_constant__) and launcher prototypes shared by
// api.cu and the kernel translation units.
#pragma once
#include "orbit_device.cuh"
#include "scan.cuh"

namespace orbit {

// Launch helper; adds programmatic stream serialization (PDL) when ORBIT_PDL is set (opt-in, see api.cu).
bool pdl_enabled();
template <typename P>
inline cudaError_t launch_kernel(void (*kernel)(const P), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, const P& params) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl_enabled() ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, params);
}

struct MeshletCullParams {
    OrbitCullInfo cull;
    HizDevice hiz;
    const uint32_t* dispatch_words;   // MeshletDispatchBuffer as u32[]: x,y,z then 4 words per record
    const uint4* meshlets;            // 2 x uint4 per meshlet
    const float4* entities;           // 8 x float4 per entity (model matrix = first 4)
    const uint8_t* materials;
    uint32_t* meshlet_visibility;
    uint32_t* draw_words;             // MeshletDrawCommandBuffer as u32[]: count then 7 words per command
    uint32_t* task_payloads;          // nullable, 11 words per record
    uint32_t* overflow_flag;          // host-mapped status word
    uint4* draw_masks;                // scratch: {draw mask, entity, meshlet offset, flag} per dispatch record (test -> emit kernel); flag 1 = no side entries
    uint4* cmd_side;                  // scratch: {vertex_offset, data_offset, packed counts, entity} per (record, lane) of a survivor (test -> emit kernel)
    uint32_t* draw_total;             // scratch[2]: survivors counted by the test kernel, per parity (re-zeroed by the emit kernel)
    uint32_t* chunk_counts;           // scratch: 2 x 2048 per-chunk survivor counts (double-buffered by parity)
    uint32_t* chunk_parity;           // scratch[2]: word A (read by test, written by emit), word B (written by test, read by emit)
    uint64_t capacity_records;
    uint64_t capacity_draws;
    float2 pk_one, pk_mone;           // (1, 1) and (-1, -1): operands of the packed add / subtract (see PkConsts in meshlet_cull.cu)
    float2 planes_t[6][4];            // cull planes paired for the packed test: [j][c] = (planes[2j][c], planes[2j+1][c]); an odd last plane is repeated
    ScanState scan;                   // only .trace is used (development timeline of the test kernel)
    unsigned long long* trace_emit;   // development timeline of the emit kernel
    // sharded view on the receiving rank (orbit_draws_from_masks), else n_regions == 0: draw_masks holds one region of
    // region_stride entries per rank, rank k's first region_counts[k] entries are its records
    const uint32_t* region_counts;
    uint64_t region_stride;
    uint32_t n_regions;
    // fused LATE + MAIN (orbit_meshlet_cull_late_main), else main_masks == nullptr: the pass-2 test kernel also fills the MAIN
    // pass's record entries (pass 1 over the bits it is writing: should_draw = visible && alpha filter) and survivor counts
    uint4* main_masks;
    uint32_t* main_chunk_counts;      // 2 x 2048, double-buffered like chunk_counts
    uint32_t* main_chunk_parity;      // [2], like chunk_parity
    uint32_t* main_draw_total;        // [2], like draw_total
    uint32_t main_alpha_mode_flags;
    // emit kernel: CTAs that take part when the list is short (< kEmitBulkSurvivors); the launch is sized for long lists
    // (occupancy: the walk of a long list is bound by the loads in flight), the surplus CTAs of a short one leave at once
    uint32_t emit_small_grid;
};

struct EntityCullParams {
    OrbitCullInfo cull;
    HizDevice hiz;
    const uint32_t* entity_draw_words;   // EntityDrawBuffer as u32[]: count then 3 words per draw
    const uint8_t* mesh_infos;           // 128 B each
    const float4* entities;              // 8 x float4 each
    uint32_t* entity_visibility;
    uint32_t* dispatch_words;            // MeshletDispatchBuffer as u32[]: x,y,z then 4 words per record
    uint32_t* dispatch_mirror;           // nullable: a second buffer that receives the same header and records (fused LATE + MAIN)
    uint32_t* overflow_flag;
    uint64_t capacity_records;
    uint32_t draw_begin, draw_end;       // sub-range of draws covered by this launch (begin % 32 == 0)
    ScanState scan;
};

// Batched pass-0 views of one scene (orbit_entity_cull_views / orbit_meshlet_cull_views): one full parameter block per view,
// passed by value like the single-view blocks, so everything a replayed CUDA graph needs travels in the kernel parameters.
struct EntityViewsParams {
    EntityCullParams view[ORBIT_MAX_BATCH_VIEWS];   // scene fields and scan state are read from view[0]
    uint32_t n_views;
};
struct MeshletViewsParams {
    MeshletCullParams view[ORBIT_MAX_BATCH_VIEWS];  // scene fields are read from view[0]; per view: CullInfo, planes_t, buffers, scratch
    uint32_t n_views;
};
static_assert(sizeof(EntityViewsParams) <= 32764 && sizeof(MeshletViewsParams) <= 32764, "kernel parameter space is 32 764 bytes");

struct SceneUpdateParams {
    const uint8_t* transforms;           // OrbitTransform[], 48 B each
    const uint32_t* mesh_slots;
    uint32_t* visibility_offsets;
    const uint8_t* mesh_infos;           // 128 B each
    uint32_t* visibility_cursor;
    uint32_t* cursor_snapshot;           // scratch word: cursor value at the start of the update
    unsigned long long* tile_sums;       // scratch: per 256-entity tile, meshed count | visibility words << 32
    float4* entity_data;                 // out, 8 x float4 per instance
    uint32_t* entity_draw_words;         // out, EntityDrawBuffer as u32[]
    uint32_t* overflow_flag;             // host-mapped status word
    uint32_t n_entities, visibility_capacity_words;
};

struct MeshletBoundsParams {
    const uint8_t* vertices;             // vertex array, position = 3 x f32 at the start of each element
    uint32_t vertex_stride;              // bytes (GpuMeshVertex: 32)
    const uint32_t* meshlet_data;        // per meshlet at data_offset: vertex_count indices, then triangle_count x 3 bytes
    uint8_t* meshlets;                   // OrbitMeshlet[]: counts / offsets in, bounding_sphere + cone out
    uint32_t n_meshlets;
    uint32_t* error_flag;                // host-mapped status word (a meshlet with more triangles than the kernel stages)
};

struct MeshBoundsParams {
    const uint8_t* vertices;
    uint32_t vertex_stride;
    const uint32_t* vertex_ranges;       // per mesh: first vertex, vertex count
    uint8_t* mesh_infos;                 // OrbitMeshInfo[]: bounding_sphere @0, aabb.min @16, aabb.max @32 written
    uint32_t n_meshes;
};

struct HizBuildParams {
    const float* depth;
    float* texels;
    uint32_t depth_w, depth_h;
    uint32_t width, height, levels;
    uint32_t level_offset[ORBIT_HIZ_MAX_LEVELS];
    unsigned int* ticket;  // zero on entry, re-zeroed by the last CTA
    unsigned long long* trace;
};
// orbit_hiz_build_views: one block per pyramid (same geometry, own depth buffer, texels and ticket); row blockIdx.y of the grid
struct HizBuildViewsParams {
    HizBuildParams view[ORBIT_MAX_BATCH_VIEWS];
    uint32_t n_views;
};

struct ClusterParams {
    OrbitClusterCullInfo info;
    float z_scale, z_bias;
    const float* depth;
    const uint8_t* lights;            // OrbitLightData[]
    float4* light_view;               // scratch: (view xyz, outer_radius or +inf for non-point lights)
    float4* cluster_boxes;            // scratch (light-parallel path, else nullptr): view-space box lo / hi per compacted-list slot
    uint32_t* cluster_totals;         // scratch (light-parallel path): hits per compacted-list slot, zeroed by the compaction kernel
    uint32_t* tile_masks;
    uint32_t* depth_bounds;           // 2 words per cluster
    uint32_t* unique_clusters;        // 4-word header + indices
    uint32_t* offset_count_image;     // 2 words per cluster
    uint32_t* light_index_words;      // count + indices
    uint32_t* overflow_flag;
    uint64_t capacity_indices;
    ScanState scan;
};

cudaError_t launch_meshlet_cull(const MeshletCullParams&, int grid, int emit_grid, cudaStream_t);
int meshlet_emit_max_ctas_per_sm();
int meshlet_cull_max_ctas_per_sm(const MeshletCullParams&);
int meshlet_cull_variant_index(const OrbitCullInfo&);
cudaError_t meshlet_cull_configure_device();
cudaError_t meshlet_cull_configure_views_pass2();
cudaError_t light_cluster_configure_device();
cudaError_t launch_record_masks_put(const uint4* src, const uint32_t* dispatch_words, uint4* dst_region, uint32_t* dst_count, uint64_t capacity,
                                    int grid, cudaStream_t s);
cudaError_t launch_meshlet_emit(const MeshletCullParams& p, int emit_grid, cudaStream_t s);
cudaError_t launch_meshlet_emit_pair(const MeshletCullParams& a, const MeshletCullParams& b, int emit_grid, cudaStream_t s);
cudaError_t launch_draws_from_masks(const MeshletCullParams& p, uint32_t* header, int grid, int emit_grid, cudaStream_t s);
cudaError_t launch_entity_cull(const EntityCullParams&, uint32_t n_draws, uint32_t coresident_ctas, cudaStream_t);
cudaError_t launch_entity_cull_views(const EntityViewsParams&, uint32_t n_draws, uint32_t coresident_ctas, cudaStream_t);
cudaError_t launch_meshlet_cull_views(const MeshletViewsParams&, int grid, int emit_grid_per_view, cudaStream_t);
int meshlet_cull_views_max_ctas_per_sm(const OrbitCullInfo&);
int entity_cull_max_ctas_per_sm();
int entity_cull_views_max_ctas_per_sm(uint32_t occlusion_pass);
cudaError_t launch_hiz_build(const HizBuildParams&, cudaStream_t);
cudaError_t launch_hiz_build_views(const HizBuildViewsParams&, cudaStream_t);
cudaError_t launch_meshlet_bounds(const MeshletBoundsParams&, int grid, cudaStream_t);
cudaError_t launch_mesh_bounds(const MeshBoundsParams&, int grid, cudaStream_t);
cudaError_t launch_scene_update(const SceneUpdateParams&, cudaStream_t);
cudaError_t launch_mark_active(const ClusterParams&, int grid, cudaStream_t);
cudaError_t launch_compact_clusters(const ClusterParams&, cudaStream_t);
cudaError_t launch_light_view(const ClusterParams&, cudaStream_t);
cudaError_t launch_light_culling(const ClusterParams&, int grid, cudaStream_t);
uint32_t light_hits_blocks(uint32_t n_lights);
cudaError_t launch_light_hits(const ClusterParams&, uint32_t* hits, uint32_t* counts, uint32_t words_per_cluster, uint32_t max_clusters, cudaStream_t);
cudaError_t launch_light_lists(const ClusterParams&, const uint32_t* hits, const uint32_t* counts, uint32_t words_per_cluster, int grid, cudaStream_t);
cudaError_t launch_draws_scatter(const uint32_t* src, uint64_t src_capacity, uint32_t* dst, uint32_t dst_first, uint32_t total_count,
                                 uint64_t dst_capacity, int grid, cudaStream_t s, const uint32_t* rank_counts, uint32_t rank, uint32_t world);

}  // namespace orbit
