/*
 * orbit_cuda.h — C ABI of liborbit_b200.so: the B200 (sm_100a) visibility pipeline behind Orbit's
 * culling-pass interface.
 *
 * The reference (Thefefe/orbit) has no FFI layer; the seam this library replaces is the set of pass
 * creation functions in src/passes/draw_gen.rs and src/passes/cluster.rs.  Each entry point below names
 * the reference function + GPU program it stands in for.  All buffers are raw device pointers in exactly
 * the reference byte layout (include/orbit_layouts.h), so the Vulkan indirect draws of
 * src/graphics/context.rs:1092-1111 can consume the outputs unchanged (memory shared through
 * cudaImportExternalMemory when interop is on; allocated by the caller when headless).
 *
 * Conventions
 *   - return value: 0 = ORBIT_OK, negative = error (orbit_error_string).  The reference has no error
 *     convention (assert!/unwrap: draw_gen.rs:334,390,123-133); argument errors it would have panicked on
 *     are reported as ORBIT_ERR_INVALID_ARGUMENT here.
 *   - every stage call is asynchronous on `stream` (a cudaStream_t passed as void*; NULL = default stream)
 *     and never synchronises with the host.  Nothing is read back (draw_gen.rs never reads back either).
 *   - OrbitCullInfo / OrbitClusterParams / OrbitSceneBuffers are HOST structs, copied into kernel parameter
 *     space at launch; the pointers inside OrbitSceneBuffers are DEVICE pointers.
 *   - a context owns the small device scratch used by the scan-based compaction (tile descriptors, tickets).
 *     Calls of the SAME stage on one context must not run concurrently (two streams), but the stages own disjoint
 *     scratch: one orbit_entity_cull, one orbit_meshlet_cull, one orbit_hiz_build, one orbit_scene_update and one
 *     orbit_light_cluster call may overlap on different streams of one context (orbit_light_cluster shares the scan
 *     descriptors with orbit_entity_cull: those two must not overlap); the orbit_draws_scatter* / orbit_device_copy /
 *     orbit_peer_* helpers touch no context scratch at all. Contexts are independent of each other and of the calling
 *     thread: every entry point makes the context's device current for the duration of the call and restores the caller's
 *     (the reference records passes from rayon workers: context.rs:1392-1423).
 *   - output order is deterministic: dispatch records are ordered by (entity-draw index, chunk), draw
 *     commands by (dispatch record index, lane), compacted clusters and light indices ascending.  The
 *     reference appends with atomicAdd (entity_cull.comp:211, meshlet_cull.comp:228), i.e. in arbitrary
 *     order; any order is valid for its consumers, so a fixed one is a drop-in.
 *   - latency hiding reads ahead: the meshlet stage may LOAD (and then ignore) dispatch-buffer bytes between the
 *     device-side record count and `capacity_records`, and the entity stage entity-draw words up to
 *     `entity_draw_count`; the buffers must be allocated to the stated capacities (contents beyond the counts are
 *     never used; zero them once if a tool such as compute-sanitizer initcheck is to stay quiet).
 *   - scratch grows on the first call that needs more than the context has seen so far (larger capacity_records,
 *     more clusters, more lights): one cudaMalloc inside that call, no synchronisation (orbit_ctx_reserve pre-sizes it);
 *     size a context (reserve or warm-up) before capturing calls into a CUDA graph. Captured calls are replay-safe:
 *     scan epochs, tickets and scratch parities live in device memory, never in kernel parameters.
 *   - there is no CPU fallback: without a CUDA device every entry point that needs one fails.
 */
#ifndef ORBIT_CUDA_H
#define ORBIT_CUDA_H

#include <stdint.h>
#include "orbit_layouts.h"

#ifdef __cplusplus
extern "C" {
#endif

/* 3: orbit_entity_cull_views / orbit_meshlet_cull_views (batched pass-0 views; additive, no layout changed),
 *    orbit_*_late_main + orbit_cull_pair_compatible, orbit_peer_put / orbit_peer_wait, OrbitStatus::peer_timeout (was reserved[0]),
 *    orbit_record_masks_put / region form of orbit_draws_from_masks (replace orbit_record_masks_scatter_ranked).
 * 2: device guards on every entry point, orbit_ctx_reserve, orbit_meshlet_test, scatter sources clamped to their capacity. */
#define ORBIT_ABI_VERSION 3

enum {
    ORBIT_OK = 0,
    ORBIT_ERR_INVALID_ARGUMENT = -1,
    ORBIT_ERR_CUDA = -2,           /* a CUDA runtime call failed; orbit_last_cuda_error() has the code */
    ORBIT_ERR_OUT_OF_MEMORY = -3,
    ORBIT_ERR_NO_DEVICE = -4,
    ORBIT_ERR_CAPACITY = -5        /* reported by orbit_ctx_poll_status only */
};

typedef struct orbit_ctx orbit_ctx;
typedef struct orbit_hiz orbit_hiz;

/* Device-written status, readable after the stream has been synchronised. */
typedef struct OrbitStatus {
    uint32_t dispatch_overflow;   /* entity stage produced more records than capacity_records (extra dropped) */
    uint32_t draw_overflow;       /* meshlet stage produced more draws than capacity_draws (extra dropped)    */
    uint32_t light_index_overflow;/* light lists exceeded capacity_indices (extra dropped)                    */
    uint32_t visibility_overflow; /* scene update needed more visibility words than the buffer holds (the reference
                                     panics here: scene.rs:427 `.unwrap()`)                                   */
    uint32_t asset_error;         /* orbit_meshlet_bounds met a meshlet with more than 128 triangles (left untouched);
                                     orbit_ctx_poll_status then returns ORBIT_ERR_INVALID_ARGUMENT              */
    uint32_t peer_timeout;        /* orbit_peer_wait gave up (~2 s) waiting for a flag: a peer never delivered;
                                     orbit_ctx_poll_status then returns ORBIT_ERR_CUDA                           */
    uint32_t reserved[2];
} OrbitStatus;

/* Device pointers to the long-lived scene / asset arrays the culling path reads.
 * Reference owners: GpuAssets (assets/mod.rs:230-239) and SceneData (scene.rs:358-369). */
typedef struct OrbitSceneBuffers {
    const void* entity_draws;       /* EntityDrawBuffer: u32 count @0, OrbitEntityDraw[] @4             */
    const void* mesh_infos;         /* OrbitMeshInfo[]                                                   */
    const void* entities;           /* OrbitEntityData[]                                                 */
    const void* meshlets;           /* OrbitMeshlet[] (32-byte aligned)                                  */
    const void* materials;          /* GpuMaterialData[] (80-byte stride)                                */
    uint32_t*   entity_visibility;  /* one bit per entity draw, word = draw_index/32 (forward.rs:150-157) */
    uint32_t*   meshlet_visibility; /* one word per dispatch record (scene.rs:354,375-382); may be NULL  */
    uint32_t    entity_draw_count;  /* host copy of the count used to size the launch (draw_gen.rs:377)  */
    uint32_t    draw_begin;         /* first entity-draw index this call covers (multiple of 32);        */
    uint32_t    draw_end;           /* one past the last; 0,0 = all. Used to shard one view over GPUs.   */
    uint32_t    reserved;
} OrbitSceneBuffers;

/* Geometry of a depth pyramid: DepthPyramid::new, draw_gen.rs:456-459 + math.rs:18-20. Level l is
 * max(width>>l,1) x max(height>>l,1) texels of f32 starting at texel offset level_offset[l] of one linear
 * allocation (levels are stored back to back so the whole pyramid is one contiguous broadcastable block). */
#define ORBIT_HIZ_MAX_LEVELS 16
typedef struct OrbitHizInfo {
    uint32_t width, height;       /* level-0 size = [npot(w)/2, npot(h)/2] */
    uint32_t levels;
    uint32_t total_texels;
    uint32_t level_offset[ORBIT_HIZ_MAX_LEVELS];
    float*   texels;              /* device pointer (NULL from orbit_hiz_geometry) */
} OrbitHizInfo;

/* Parameters of clustered light assignment = ClusterCullInfo (cluster.rs:186-207) + the mark_active push
 * block (mark_active.comp:8-23, z_scale/z_bias from ClusterSettings::cluster_grid_info, cluster.rs:63-72). */
typedef struct OrbitClusterParams {
    OrbitClusterCullInfo info;
    float    z_scale;
    float    z_bias;
    uint32_t reserved[2];
} OrbitClusterParams;

/* ---- context ------------------------------------------------------------------------------------------ */
int         orbit_abi_version(void);
const char* orbit_error_string(int code);
int         orbit_last_cuda_error(void);
int         orbit_ctx_create(int device, orbit_ctx** out);
void        orbit_ctx_destroy(orbit_ctx* ctx);
/* Copies the device-written status words (pinned, host-mapped) and clears them. Caller syncs the stream first. */
int         orbit_ctx_poll_status(orbit_ctx* ctx, OrbitStatus* out);
/* Number of kernels this context has launched so far (bench.py reports it as gpu_launches). */
uint64_t    orbit_ctx_launch_count(const orbit_ctx* ctx);
/* Pre-sizes the context's scratch for the largest calls it will see (entity draws per launch, dispatch-buffer capacity in
 * records, lights, clusters, scene-update entities; 0 = leave as is), so that no later stage call allocates. This is the one
 * call that may synchronise the device. Without it scratch grows on demand inside the stage call (cudaMalloc, never a
 * synchronisation or a free: outgrown scratch is parked until orbit_ctx_destroy) — not capturable into a CUDA graph, so
 * reserve, or warm up, before capturing. */
int         orbit_ctx_reserve(orbit_ctx* ctx, uint64_t entity_draws, uint64_t capacity_records, uint64_t n_lights,
                              uint64_t n_clusters, uint64_t n_entities);

/* ---- depth pyramid: DepthPyramid::{new,resize,update,get_current}, draw_gen.rs:451-567 ------------------ */
int  orbit_hiz_geometry(uint32_t depth_width, uint32_t depth_height, OrbitHizInfo* out);  /* host only */
int  orbit_hiz_create(orbit_ctx* ctx, uint32_t depth_width, uint32_t depth_height, orbit_hiz** out);
/* Wrap caller-owned device memory of orbit_hiz_geometry().total_texels floats (interop / torch allocations). */
int  orbit_hiz_wrap(orbit_ctx* ctx, uint32_t depth_width, uint32_t depth_height, float* texels, orbit_hiz** out);
void orbit_hiz_destroy(orbit_hiz* hiz);
int  orbit_hiz_info(const orbit_hiz* hiz, OrbitHizInfo* out);
/* DepthPyramid::update (draw_gen.rs:510-566) + depth_reduce.comp: builds ALL levels from `depth`
 * (depth_width x depth_height f32, row-major, reverse-Z) in one launch. */
int  orbit_hiz_build(orbit_ctx* ctx, orbit_hiz* hiz, const float* depth,
                     uint32_t depth_width, uint32_t depth_height, void* stream);

/* ---- create_meshlet_dispatch_command (draw_gen.rs:327-380) + entity_cull.comp --------------------------- */
/* Writes MeshletDispatchBuffer {x,1,1; records[]} and, in pass 2, the entity visibility words.
 * `hiz` may be NULL unless cull->occlusion_pass == 2. */
int orbit_entity_cull(orbit_ctx* ctx, const OrbitCullInfo* cull, const OrbitSceneBuffers* scene,
                      const orbit_hiz* hiz, void* meshlet_dispatch_buffer, uint64_t capacity_records,
                      void* stream);

/* ---- create_meshlet_draw_commands (draw_gen.rs:382-435) + meshlet_cull.comp ------------------------------ */
/* Reads the dispatch buffer produced above (its record count is read on the device — the reference's
 * dispatch_indirect, draw_gen.rs:432), writes MeshletDrawCommandBuffer {count; draws[]} and, in pass 2 with
 * meshlet occlusion culling on, the meshlet visibility words.
 * `task_payloads` (nullable): additionally emits, per dispatch record, the MeshTaskPayload the task-shader
 * twins build (forward_depth_prepass.task:224-256) plus its emitted mesh-task count:
 * element r = {u32 task_count; OrbitMeshTaskPayload} (44 bytes) for record r.
 * `capacity_records` is the size of the dispatch buffer in records; the device-side count is clamped to it. */
int orbit_meshlet_cull(orbit_ctx* ctx, const OrbitCullInfo* cull, const OrbitSceneBuffers* scene,
                       const orbit_hiz* hiz, const void* meshlet_dispatch_buffer, uint64_t capacity_records,
                       void* draw_command_buffer, uint64_t capacity_draws,
                       void* task_payloads, void* stream);

/* ---- fused LATE + MAIN passes (forward.rs:266-403 followed by forward.rs:518-548) --------------------------------
 * The MAIN pass is pass 1 over the visibility bits the LATE pass (pass 2) has just written. When both passes use the same
 * camera, planes, LOD parameters and visibility buffers and meshlet occlusion culling is on (orbit_cull_pair_compatible
 * returns 1: view matrix, planes, projection type, LOD parameters and visibility buffers are equal; alpha_mode_flags and the
 * fields only pass 2 reads may differ), the
 * MAIN pass's tests repeat the LATE pass's: its dispatch list is the LATE list, and its draw list holds the meshlets the
 * LATE pass finds visible, filtered by the MAIN pass's alpha_mode_flags. The two calls below produce, in one entity
 * kernel and one test kernel (+ one emit kernel per list), byte for byte what
 *   orbit_entity_cull(late) ; orbit_meshlet_cull(late) ; orbit_entity_cull(main) ; orbit_meshlet_cull(main)
 * produce. They return ORBIT_ERR_INVALID_ARGUMENT for an incompatible pair (call the four stages separately then). */
int orbit_cull_pair_compatible(const OrbitCullInfo* late, const OrbitCullInfo* main_pass);
int orbit_entity_cull_late_main(orbit_ctx* ctx, const OrbitCullInfo* late, const OrbitCullInfo* main_pass,
                                const OrbitSceneBuffers* scene, const orbit_hiz* hiz, void* late_dispatch_buffer,
                                void* main_dispatch_buffer, uint64_t capacity_records, void* stream);
int orbit_meshlet_cull_late_main(orbit_ctx* ctx, const OrbitCullInfo* late, const OrbitCullInfo* main_pass,
                                 const OrbitSceneBuffers* scene, const orbit_hiz* hiz, const void* late_dispatch_buffer,
                                 uint64_t capacity_records, void* late_draw_command_buffer, void* main_draw_command_buffer,
                                 uint64_t capacity_draws, void* late_task_payloads /* nullable */,
                                 void* main_task_payloads /* nullable */, void* stream);

/* ---- Hi-Z build + LATE entity cull in one call ------------------------------------------------------------------------------
 * Byte for byte what
 *   orbit_hiz_build(ctx, hiz, depth, depth_width, depth_height) ; orbit_entity_cull(ctx, late, scene, hiz, late_dispatch_buffer)
 * write when main_pass is NULL (main_dispatch_buffer must then be NULL too), and what
 *   orbit_hiz_build(...) ; orbit_entity_cull_late_main(ctx, late, main_pass, scene, hiz, late_dispatch_buffer, main_dispatch_buffer)
 * write otherwise: every pyramid texel, the entity visibility words, the dispatch buffers and the status words. Two launches,
 * as the separate calls, but the entity kernel does everything that does not read the pyramid while the build is still
 * running. Every argument rule of the two calls applies, and late->occlusion_pass must be 2; a refused call
 * (ORBIT_ERR_INVALID_ARGUMENT) launches nothing. Counts as an orbit_hiz_build call and an orbit_entity_cull call (concurrency rules at the top).
 * Only sound because the call enqueues the build itself: the entity stage after any other predecessor is orbit_entity_cull. */
int orbit_hiz_build_entity_cull_late(orbit_ctx* ctx, orbit_hiz* hiz, const float* depth, uint32_t depth_width,
                                     uint32_t depth_height, const OrbitCullInfo* late, const OrbitCullInfo* main_pass /* nullable */,
                                     const OrbitSceneBuffers* scene, void* late_dispatch_buffer,
                                     void* main_dispatch_buffer /* nullable */, uint64_t capacity_records, void* stream);

/* ---- batched pass-0 views (the cascades of ShadowRenderer::render_cascaded_shadow, shadow_renderer.rs:466-712; many cameras
 *      over one scene) ---------------------------------------------------------------------------------------------------
 * n_views (1..ORBIT_MAX_BATCH_VIEWS) pass-0 views of ONE scene. View v's buffers are byte for byte what
 *   orbit_entity_cull(&culls[v], ...) ; orbit_meshlet_cull(&culls[v], ...)
 * write: header, records / commands in canonical order, and task payloads. 3 kernel launches per call pair, whatever n_views
 * is: one entity kernel over n_views x ceil(draws / 256) tiles, one test kernel over the concatenation of the views' record
 * lists, one emit kernel with a row of CTAs per view.
 *   - every view has its own OrbitCullInfo (view matrix, 0..12 planes, LOD target / base / step / range, alpha filter), but
 *     all views of a call have the same projection_type and occlusion_pass == 0;
 *   - `scene` (draw_begin / draw_end included) is shared by all views; dispatch_buffers[v] / draw_command_buffers[v] are view
 *     v's outputs (no two views may share one), all of `capacity_records` / `capacity_draws`; task_payloads may be NULL, and
 *     so may any of its entries;
 *   - ORBIT_ERR_INVALID_ARGUMENT, with nothing launched, for: n_views 0 or above the maximum, a view with occlusion_pass != 0,
 *     mixed projection types, more than 12 planes, a NULL or misaligned buffer, two views sharing a buffer, and everything
 *     orbit_entity_cull / orbit_meshlet_cull refuse;
 *   - overflow as in the single-view calls: each view's header stays exact, records / commands beyond capacity are dropped,
 *     OrbitStatus.dispatch_overflow / draw_overflow are set if any view overflowed;
 *   - concurrency: orbit_entity_cull_views counts as an orbit_entity_cull call and orbit_meshlet_cull_views as an
 *     orbit_meshlet_cull call; calls of both forms may be interleaved on one stream in any order (the batched meshlet stage
 *     keeps its survivor counters apart from the single-view ones). Replay-safe under CUDA-graph capture.
 *   - scratch: the per-record scratch of the meshlet stage grows to n_views x capacity_records records, 528 bytes per record
 *     (C4's four cascades: ~0.74 GB; C5, 16 views: ~5.9 GB); orbit_ctx_reserve(ctx, .., n_views * capacity_records, ..)
 *     pre-sizes it. The first orbit_meshlet_cull_views call of a context also allocates the batched stage's survivor counters
 *     (256 KB): make one batched call before capturing batched calls into a CUDA graph. */
#define ORBIT_MAX_BATCH_VIEWS 16
int orbit_entity_cull_views(orbit_ctx* ctx, const OrbitCullInfo* culls, uint32_t n_views, const OrbitSceneBuffers* scene,
                            void* const* dispatch_buffers, uint64_t capacity_records, void* stream);
int orbit_meshlet_cull_views(orbit_ctx* ctx, const OrbitCullInfo* culls, uint32_t n_views, const OrbitSceneBuffers* scene,
                             const void* const* dispatch_buffers, uint64_t capacity_records, void* const* draw_command_buffers,
                             uint64_t capacity_draws, void* const* task_payloads /* NULL, or entries may be NULL */, void* stream);

/* ---- batched two-pass occlusion views (split-screen, stereo, probe cameras: several cameras with EARLY -> Hi-Z -> LATE -> MAIN
 *      over one scene, forward.rs:213-548 per camera) ------------------------------------------------------------------------
 * orbit_hiz_build_views: DepthPyramid::update for n_views (1..ORBIT_MAX_BATCH_VIEWS) pyramids of the same geometry in ONE launch
 * (the reference's update_multiple_depth_pyramids, draw_gen.rs). Pyramid v is byte for byte what
 * orbit_hiz_build(ctx, hizs[v], depths[v], depth_width, depth_height) writes. Refused (ORBIT_ERR_INVALID_ARGUMENT, nothing
 * launched): n_views 0 or above the maximum, a NULL pyramid or depth buffer, a pyramid not created for depth_width x
 * depth_height, two pyramids on the same texels. Counts as an orbit_hiz_build call; needs no scratch of its own.
 *
 * orbit_entity_cull_views_occlusion / orbit_meshlet_cull_views_occlusion: two-pass occlusion culling of n_views cameras over
 * ONE scene, 3 kernel launches per call pair whatever n_views is. View v's outputs are byte for byte what
 *   orbit_entity_cull(&culls[v], &scenes[v], hizs ? hizs[v] : NULL, ...) ; orbit_meshlet_cull(&culls[v], &scenes[v], ...)
 * write: dispatch header and records, draw count and commands, task payloads, and (pass 2) the view's entity and meshlet
 * visibility words. A frame of N cameras is EARLY (pass 1), orbit_hiz_build_views, LATE (pass 2), MAIN (pass 1): 10 launches.
 *   - views: n_views is 1..ORBIT_MAX_BATCH_VIEWS;
 *   - same pass: every view has the same occlusion_pass, and it is 1 or 2 (pass 0 is orbit_*_cull_views);
 *   - same projection: every view has the same projection_type;
 *   - same meshlet-occlusion setting: either every view has a meshlet visibility buffer (meshlet_visibility_buffer !=
 *     ORBIT_NO_BUFFER) or none does;
 *   - one scene: scenes[v] equals scenes[0] in every field except entity_visibility and meshlet_visibility (draw_begin /
 *     draw_end included);
 *   - no shared buffers: no two views share a visibility buffer (the entity call: entity_visibility; the meshlet call with
 *     meshlet occlusion: meshlet_visibility), a dispatch buffer, a draw buffer or a task payload buffer;
 *   - pyramids: hizs is required for pass 2 and ignored for pass 1; it holds one distinct pyramid per view, all of the same
 *     geometry;
 *   - everything orbit_entity_cull / orbit_meshlet_cull refuse for one view is refused here too;
 *   every refusal returns ORBIT_ERR_INVALID_ARGUMENT with nothing launched.
 *   - overflow, status flags and CUDA-graph replay follow the single-view rules;
 *   - concurrency: the entity call counts as an orbit_entity_cull call and the meshlet call as an orbit_meshlet_cull call;
 *   - scratch: as orbit_meshlet_cull_views (n_views x capacity_records records; the batched survivor counters are allocated
 *     by the first batched meshlet call of either form: make one before capturing batched calls into a CUDA graph). */
int orbit_hiz_build_views(orbit_ctx* ctx, orbit_hiz* const* hizs, const float* const* depths, uint32_t n_views,
                          uint32_t depth_width, uint32_t depth_height, void* stream);
int orbit_entity_cull_views_occlusion(orbit_ctx* ctx, const OrbitCullInfo* culls, uint32_t n_views,
                                      const OrbitSceneBuffers* scenes, const orbit_hiz* const* hizs,
                                      void* const* dispatch_buffers, uint64_t capacity_records, void* stream);
int orbit_meshlet_cull_views_occlusion(orbit_ctx* ctx, const OrbitCullInfo* culls, uint32_t n_views,
                                       const OrbitSceneBuffers* scenes, const orbit_hiz* const* hizs,
                                       const void* const* dispatch_buffers, uint64_t capacity_records,
                                       void* const* draw_command_buffers, uint64_t capacity_draws,
                                       void* const* task_payloads /* NULL, or entries NULL */, void* stream);

/* ---- compute_clusters (cluster.rs:368-591) + light_cluster/{mark_active,active_cluster_compaction,
 *      light_culling}.comp --------------------------------------------------------------------------------- */
/* tile_masks: u32[cx*cy]; depth_bounds: OrbitClusterDepthBounds[cx*cy*cz]; unique_clusters:
 * CompactedClusterIndexList (16 + 4*cx*cy*cz bytes); offset_count_image: uint2[cx*cy*cz] (inactive texels are
 * zeroed); light_index_list: ClusterLightIndices (4 + 4*capacity_indices bytes). */
int orbit_light_cluster(orbit_ctx* ctx, const OrbitClusterParams* params, const float* depth,
                        const void* lights, void* tile_masks, void* depth_bounds, void* unique_clusters,
                        void* offset_count_image, void* light_index_list, uint64_t capacity_indices,
                        void* stream);

/* ---- depth from an image (a depth attachment imported from Vulkan) ------------------------------------------------------
 * An optimally tiled VkImage imported with cudaImportExternalMemory can only be mapped as a CUDA (mipmapped) array, not as a
 * linear pointer. orbit_depth_image wraps such an array, so the depth-reading stages take it directly: no image-to-buffer
 * copy pass per frame and camera. Each *_image call writes byte for byte what its linear twin writes for the same depth values.
 *
 * orbit_depth_image_wrap: `cuda_array` is a caller-owned cudaArray_t (passed as void*), e.g. level 0 of a mipmapped array
 * mapped from an imported VkImage (cudaGetMipmappedArrayLevel(&a, mm, 0)), or one from cudaMallocArray. It must be 2-D
 * (extent depth 0, not layered, not a cubemap), at least 1 x 1, with one 32-bit cudaChannelFormatKindFloat channel; the
 * handle records its width and height. The call creates its own texture object on the array (unnormalised coordinates,
 * point filtering, clamp addressing, element read mode) and allocates nothing on the device. Anything else, a NULL array
 * included, and an array the context's device cannot query, is ORBIT_ERR_INVALID_ARGUMENT. The array stays the caller's.
 * orbit_depth_image_destroy releases the texture object, never the array. Destroying an image, or freeing its array, while
 * enqueued work or a captured CUDA graph still reads it is the caller's error (as with orbit_hiz_destroy).
 *
 * Stage calls: every argument rule of the linear twin applies, and the image's size must equal the depth size the pyramid was
 * created for (orbit_light_cluster_image: params->info.screen_size). A refused call (ORBIT_ERR_INVALID_ARGUMENT) launches
 * nothing. Concurrency and CUDA-graph rules are the twin's; the texture handle travels in the kernel parameters, so a
 * replayed graph reads the array's contents at replay time, for as long as the image lives.
 * Synchronisation: the calls read the array on `stream`. Ordering the renderer's writes of the image before them (an
 * imported Vulkan semaphore waited on `stream` with cudaWaitExternalSemaphoresAsync) is the caller's job. */
typedef struct orbit_depth_image orbit_depth_image;
int  orbit_depth_image_wrap(orbit_ctx* ctx, void* cuda_array, orbit_depth_image** out);
void orbit_depth_image_destroy(orbit_depth_image* image);
/* The wrapped array's width and height in texels. */
int  orbit_depth_image_size(const orbit_depth_image* image, uint32_t* width, uint32_t* height);
/* orbit_hiz_build with the depth read from `image`. */
int  orbit_hiz_build_image(orbit_ctx* ctx, orbit_hiz* hiz, const orbit_depth_image* image, void* stream);
/* orbit_hiz_build_views with depths[v] read from images[v] (all of the pyramids' depth size; a NULL entry is refused). */
int  orbit_hiz_build_views_image(orbit_ctx* ctx, orbit_hiz* const* hizs, const orbit_depth_image* const* images,
                                 uint32_t n_views, void* stream);
/* orbit_hiz_build_entity_cull_late with (depth, depth_width, depth_height) replaced by `image`. */
int  orbit_hiz_build_image_entity_cull_late(orbit_ctx* ctx, orbit_hiz* hiz, const orbit_depth_image* image,
                                            const OrbitCullInfo* late, const OrbitCullInfo* main_pass /* nullable */,
                                            const OrbitSceneBuffers* scene, void* late_dispatch_buffer,
                                            void* main_dispatch_buffer /* nullable */, uint64_t capacity_records, void* stream);
/* orbit_light_cluster with `depth` replaced by `image`. */
int  orbit_light_cluster_image(orbit_ctx* ctx, const OrbitClusterParams* params, const orbit_depth_image* image,
                               const void* lights, void* tile_masks, void* depth_bounds, void* unique_clusters,
                               void* offset_count_image, void* light_index_list, uint64_t capacity_indices,
                               void* stream);

/* ---- outputs into images (the depth pyramid and the cluster grid imported from Vulkan) -------------------------------------
 * The reference keeps the depth pyramid in an R32_SFLOAT image with one mip per level (draw_gen.rs:451-567), which its task
 * shaders and Hi-Z viewer sample, and the cluster offset/count grid in a 3-D R32G32_UINT image (cluster.rs:532-544), which
 * forward.frag reads. Imported into CUDA they are (mipmapped) arrays; these calls write them directly, so no buffer-to-image
 * copy pass per frame and camera is needed.
 *
 * orbit_hiz_attach_image: `cuda_mipmapped_array` is a caller-owned cudaMipmappedArray_t (passed as void*), e.g. one mapped from
 * an imported VkImage with cudaExternalMemoryGetMappedMipmappedArray. From then on every build of `hiz` also stores each level
 * l into level l of the array, byte for byte the linear level: orbit_hiz_build, orbit_hiz_build_image, orbit_hiz_build_views
 * (_image) and orbit_hiz_build(_image)_entity_cull_late. The linear pyramid is still written and stays what every culling
 * call reads (and what orbit_peer_put moves); the array is a write-only mirror that no call reads back.
 *   - refused with ORBIT_ERR_INVALID_ARGUMENT, leaving no CUDA error behind: a NULL argument, a pyramid of another device, a
 *     second attach to the same pyramid (there is no detach: the mirror lives as long as the pyramid), and an array that is
 *     not exactly the pyramid: level l < info.levels must exist with extent max(width>>l,1) x max(height>>l,1) (depth 0), one
 *     32-bit cudaChannelFormatKindFloat channel, created with cudaArraySurfaceLoadStore, neither layered nor a cubemap;
 *   - the call creates one surface object per level and allocates nothing on the device. orbit_hiz_destroy releases them,
 *     never the array. Destroying the pyramid, or freeing the array, while enqueued work or a captured CUDA graph still
 *     writes it is the caller's error;
 *   - batched builds: each pyramid mirrors only if it has an array of its own (mixed batches are fine); two pyramids of one
 *     call with the same array are refused;
 *   - calls enqueued before the attach do not write the mirror. The surface handles travel in the kernel parameters: a
 *     captured graph writes the array that was attached at capture time;
 *   - a pyramid that arrives by orbit_peer_put (the ranks of a sharded view) is not rebuilt there, so its mirror is not written;
 *   - synchronisation: the mirror is written on the build's stream; ordering the renderer's reads after it (an imported
 *     Vulkan semaphore signalled on that stream with cudaSignalExternalSemaphoresAsync) is the caller's job.
 *
 * orbit_cluster_grid_wrap: `cuda_array` is a caller-owned 3-D cudaArray_t (extent depth >= 1) with two 32-bit
 * cudaChannelFormatKindUnsigned channels (x = y = 32, z = w = 0), created with cudaArraySurfaceLoadStore, neither layered nor
 * a cubemap; anything else, NULL included, is ORBIT_ERR_INVALID_ARGUMENT. The call creates one surface object and allocates
 * nothing on the device; orbit_cluster_grid_destroy releases it, never the array (lifetime rules as above).
 * orbit_light_cluster_image_grid: orbit_light_cluster_image with the offset/count grid written into `grid` instead of a
 * linear buffer. Texel (x, y, z), idx = (z*cy + y)*cx + x, holds exactly the two words orbit_light_cluster_image writes at
 * idx; inactive clusters hold (0, 0). Every texel is written by every call, so nothing of a previous frame survives. Every
 * argument rule of orbit_light_cluster_image applies, and the grid's extent must equal params->info.cluster_count; a refused
 * call launches nothing. Counts as an orbit_light_cluster call (concurrency rules at the top). */
int  orbit_hiz_attach_image(orbit_ctx* ctx, orbit_hiz* hiz, void* cuda_mipmapped_array);
typedef struct orbit_cluster_grid orbit_cluster_grid;
int  orbit_cluster_grid_wrap(orbit_ctx* ctx, void* cuda_array, orbit_cluster_grid** out);
void orbit_cluster_grid_destroy(orbit_cluster_grid* grid);
int  orbit_light_cluster_image_grid(orbit_ctx* ctx, const OrbitClusterParams* params, const orbit_depth_image* image,
                                    const void* lights, void* tile_masks, void* depth_bounds, void* unique_clusters,
                                    const orbit_cluster_grid* grid, void* light_index_list, uint64_t capacity_indices,
                                    void* stream);

/* ---- SceneData::update_scene (scene.rs:404-492), the per-frame producer of the entity buffers the culling path
 *      reads (SURVEY §8f item 3). For every entity with a mesh, in entity order: instance_index = running count,
 *      GpuEntityData {model_matrix = Mat4::from_scale_rotation_translation(scale, orientation, position),
 *      normal_matrix = Mat4::from_mat3(Mat3::from_mat4(model.inverse().transpose()))} (scene.rs:69-76),
 *      GpuEntityDraw {instance_index, mesh.slot(), visibility_offset}; an entity without a visibility range gets
 *      ceil(lod0 meshlet_count / 32) words from the allocator (scene.rs:422-431). The reference's
 *      FreeListAllocator hands out consecutive ranges as long as nothing was freed (collections/freelist_alloc.rs:
 *      40-72), which is what this entry point implements: an exclusive prefix sum over the entities that need a
 *      range, starting at *visibility_cursor. Lights and deallocation stay host bookkeeping. ---------------------- */
typedef struct OrbitSceneUpdate {
    const OrbitTransform* transforms;        /* [n_entities] device                                              */
    const uint32_t* mesh_slots;              /* [n_entities] device; ORBIT_NO_MESH = no mesh                     */
    uint32_t*       visibility_offsets;      /* [n_entities] device, in/out; ORBIT_NO_VISIBILITY_RANGE = none yet */
    const void*     mesh_infos;              /* OrbitMeshInfo[] device                                           */
    uint32_t*       visibility_cursor;       /* device word, in/out: first unallocated visibility word           */
    uint32_t        n_entities;
    uint32_t        visibility_capacity_words; /* MESHLET_VISIBILITY_BUFFER_CHUNK_COUNT (scene.rs:392)           */
    void*           entity_data;             /* out: OrbitEntityData[>= n_entities] device                       */
    void*           entity_draws;            /* out: EntityDrawBuffer (u32 count @0, OrbitEntityDraw[] @4)       */
} OrbitSceneUpdate;
int orbit_scene_update(orbit_ctx* ctx, const OrbitSceneUpdate* update, void* stream);

/* ---- asset-side producers of the culling path's inputs (SURVEY §8f item 4) --------------------------------- */
/* The bounds part of compute_meshlets (assets/mesh.rs:292-338): for every OrbitMeshlet m of `meshlets` (vertex_offset,
 * data_offset, vertex_count, triangle_count filled in by the meshlet builder) computes what meshopt::compute_meshlet_bounds
 * returns — bounding_sphere, cone_axis (snorm8 x 3), cone_cutoff (snorm8) — and stores it into the meshlet in place.
 * Geometry: vertex v of the meshlet = vertices[vertex_offset + meshlet_data[data_offset + v]] (position = 3 x f32 at the start
 * of a `vertex_stride`-byte element: GpuMeshVertex, assets/mesh.rs:12-20, stride 32); triangle t = the three bytes at
 * ((u8*)&meshlet_data[data_offset + vertex_count])[3t..3t+3] (the layout compute_meshlets writes, mesh.rs:308-316).
 * Meshlets with more than 128 triangles are left untouched and flagged (OrbitStatus.asset_error). */
int orbit_meshlet_bounds(orbit_ctx* ctx, const void* vertices, uint32_t vertex_stride, const uint32_t* meshlet_data,
                         void* meshlets, uint32_t n_meshlets, void* stream);
/* MeshData::compute_bounds (assets/mesh.rs:192-215) for n_meshes meshes: vertex_ranges[2m] = first vertex, [2m+1] = vertex
 * count; writes OrbitMeshInfo[m].bounding_sphere (centre = AABB middle, radius = largest vertex distance) and .aabb. */
int orbit_mesh_bounds(orbit_ctx* ctx, const void* vertices, uint32_t vertex_stride, const uint32_t* vertex_ranges,
                      void* mesh_infos, uint32_t n_meshes, void* stream);

/* ---- multi-GPU helper (no reference counterpart; SURVEY §8e) --------------------------------------------- */
/* Appends `count` draw commands read from src (a MeshletDrawCommandBuffer, device-side count honoured) into
 * dst (possibly a peer-mapped MeshletDrawCommandBuffer) starting at draw index `dst_first`; when
 * `total_count` != UINT32_MAX also stores it as dst's header. One coalesced copy kernel; used to assemble the
 * rank-major survivor list of a meshlet-range-sharded view through NVLink peer stores. A source count above
 * `src_capacity_draws` (the source overflowed: its header is exact, the excess commands were dropped) is clamped to it. */
int orbit_draws_scatter(orbit_ctx* ctx, const void* src_draw_buffer, uint64_t src_capacity_draws, void* dst_draw_buffer,
                        uint32_t dst_first, uint32_t total_count, uint64_t dst_capacity_draws, void* stream);
/* Same, with the placement taken from the DEVICE: rank_counts[world] = every rank's survivor count (e.g. the result
 * of an all-gather enqueued on the same stream); dst_first = sum of rank_counts[0..rank), header = their total.
 * Nothing is read back to the host, so a whole sharded frame stays asynchronous. Every rank's count is clamped to
 * `src_capacity_draws` (the ranks of one sharded view use equal capacities), so an overflowing rank leaves no gap. */
int orbit_draws_scatter_ranked(orbit_ctx* ctx, const void* src_draw_buffer, uint64_t src_capacity_draws, void* dst_draw_buffer,
                               const uint32_t* rank_counts, uint32_t rank, uint32_t world,
                               uint64_t dst_capacity_draws, void* stream);

/* The same exchange with 16-byte record entries instead of 28-byte commands (config C3: 28 MB instead of 229 MB to the rank
 * that submits the draws). orbit_meshlet_test = the test half of orbit_meshlet_cull: visibility words are written as usual,
 * and for every dispatch record r < count one entry {u32 draw mask, u32 entity, u32 meshlet offset, u32 1} goes to
 * record_masks[r] (16-byte aligned, capacity_records entries); no draw commands are produced.
 * orbit_record_masks_put stores this rank's entries (count = the dispatch buffer's header, read on the device, clamped to
 * capacity_records) into dst_region and the count into *dst_count — both usually peer-mapped memory of the receiving rank,
 * which keeps one region of `region_stride_records` entries and one count word per rank; no rank needs another rank's count,
 * so the exchange needs no collective besides a closing fence.
 * orbit_draws_from_masks runs on the receiving rank: reads the regions in rank order (rank-major = canonical record order),
 * recounts the survivors and emits the MeshletDrawCommandBuffer (command words are read from scene->meshlets). */
int orbit_meshlet_test(orbit_ctx* ctx, const OrbitCullInfo* cull, const OrbitSceneBuffers* scene, const orbit_hiz* hiz,
                       const void* meshlet_dispatch_buffer, uint64_t capacity_records, void* record_masks, void* stream);
int orbit_record_masks_put(orbit_ctx* ctx, const void* src_record_masks, const void* meshlet_dispatch_buffer, uint64_t capacity_records,
                           void* dst_region, uint32_t* dst_count, void* stream);
int orbit_draws_from_masks(orbit_ctx* ctx, const OrbitSceneBuffers* scene, const void* record_masks, uint64_t region_stride_records,
                           const uint32_t* region_counts, uint32_t n_regions /* <= 16 */,
                           void* draw_command_buffer, uint64_t capacity_draws, void* stream);

/* Peer-visible device memory for that assembly: one process per GPU, so a rank's output buffer is shared with the
 * other ranks through CUDA IPC. `orbit_peer_alloc` returns cudaMalloc'd memory plus its 64-byte IPC handle;
 * `orbit_peer_open` maps another rank's buffer into this process (NVLink peer access); stores through the mapped
 * pointer go over NVLink. `orbit_device_copy` is an asynchronous device-to-device copy (reading results back into
 * caller-owned tensors). */
#define ORBIT_IPC_HANDLE_BYTES 64
int  orbit_peer_alloc(orbit_ctx* ctx, uint64_t bytes, void** out_ptr, void* out_handle /* 64 bytes */);
int  orbit_peer_open(orbit_ctx* ctx, const void* handle /* 64 bytes */, void** out_ptr);
int  orbit_peer_close(orbit_ctx* ctx, void* mapped_ptr);
void orbit_peer_free(orbit_ctx* ctx, void* ptr);
int  orbit_device_copy(void* dst, const void* src, uint64_t bytes, void* stream);

/* One-sided transfers with completion flags — what the sharded view uses instead of a collective to get the depth pyramid
 * from the GPU that built it to the others (scatter its chunks, then every GPU forwards its chunk: orbit_b200/multi_gpu.py
 * PyramidBroadcast). orbit_peer_put: up to 16 transfers in ONE launch; a transfer copies `bytes` (a multiple of 16; src and
 * dst 16-byte aligned) from local memory to `dst` (usually peer-mapped: NVLink stores) and then — after all of its stores
 * have been issued and fenced at system scope — writes `flag_value` to `dst_flag` (nullable; usually a word on the receiving
 * GPU). orbit_peer_wait: the stream waits until `n_flags` (<= 32) LOCAL words, `stride_words` apart, all hold `flag_value`
 * (device-side polling, bounded at ~2 s: a flag that never arrives sets OrbitStatus::peer_timeout instead of hanging the
 * GPU). Use a value that increases with every use (a frame counter): no flag is ever reset. Put calls of one context
 * must not overlap each other (they share 16 completion counters). */
typedef struct OrbitPeerPut { const void* src; void* dst; uint64_t bytes; uint32_t* dst_flag; } OrbitPeerPut;
int  orbit_peer_put(orbit_ctx* ctx, const OrbitPeerPut* puts, uint32_t n_puts /* <= 16 */, uint32_t flag_value, void* stream);
int  orbit_peer_wait(orbit_ctx* ctx, const uint32_t* flags, uint32_t n_flags /* <= 32 */, uint32_t stride_words, uint32_t flag_value,
                     void* stream);

#ifdef __cplusplus
}
#endif
#endif /* ORBIT_CUDA_H */
