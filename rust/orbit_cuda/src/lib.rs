//! Rust binding of liborbit_b200.so (include/orbit_cuda.h) — the module a fork of Thefefe/orbit would add next to
//! `src/passes/draw_gen.rs` to route the culling passes through CUDA. SOURCE ONLY: never compiled (no Rust
//! toolchain in the build image). Layouts are the reference's own `#[repr(C)]` structs, so `GpuCullInfo`,
//! `GpuEntityDraw`, `GpuMeshlet`, … from `src/passes/draw_gen.rs:208-237`, `src/scene.rs:120-133`,
//! `src/assets/mod.rs:18-122` can be passed as they are.
#![allow(non_camel_case_types)]
use std::ffi::c_void;

pub const ORBIT_OK: i32 = 0;
pub const ORBIT_ERR_INVALID_ARGUMENT: i32 = -1;
pub const ORBIT_MAX_BATCH_VIEWS: u32 = 16;
pub const ORBIT_NO_BUFFER: u32 = 0xFFFF_FFFF;
pub const ORBIT_HIZ_MAX_LEVELS: usize = 16;

#[repr(C)] pub struct orbit_ctx { _p: [u8; 0] }
#[repr(C)] pub struct orbit_hiz { _p: [u8; 0] }
#[repr(C)] pub struct orbit_depth_image { _p: [u8; 0] }
#[repr(C)] pub struct orbit_cluster_grid { _p: [u8; 0] }

/// = `GpuCullInfo` (draw_gen.rs:208-237), 400 bytes.
#[repr(C)]
#[derive(Clone, Copy)]
pub struct OrbitCullInfo {
    pub view_matrix: [f32; 16],
    pub reprojection_matrix: [f32; 16],
    pub cull_planes: [[f32; 4]; 12],
    pub cull_plane_count: u32,
    pub alpha_mode_flags: u32,
    pub noskip_alpha_mode: u32,
    pub occlusion_pass: u32,
    pub visibility_buffer: u32,
    pub meshlet_visibility_buffer: u32,
    pub depth_pyramid: u32,
    pub secondary_depth_pyramid: u32,
    pub projection_type: u32,
    pub p00_or_width_recip_x2: f32,
    pub p11_or_height_recip_x2: f32,
    pub z_near: f32,
    pub z_far: f32,
    pub lod_base: f32,
    pub lod_step: f32,
    pub min_mesh_lod: u32,
    pub lod_target_pos_view_space: [f32; 3],
    pub max_mesh_lod: u32,
}
const _: () = assert!(std::mem::size_of::<OrbitCullInfo>() == 400);

/// Transform in the 48-byte row layout orbit_scene_update reads (include/orbit_layouts.h; scene.rs:18-23).
#[repr(C)]
#[derive(Clone, Copy)]
pub struct OrbitTransform { pub position: [f32; 3], pub _pad0: f32, pub orientation: [f32; 4], pub scale: [f32; 3], pub _pad1: f32 }

/// Arguments of orbit_scene_update (SceneData::update_scene, scene.rs:404-492). Device pointers.
#[repr(C)]
#[derive(Clone, Copy)]
pub struct OrbitSceneUpdate {
    pub transforms: *const OrbitTransform,
    pub mesh_slots: *const u32,
    pub visibility_offsets: *mut u32,
    pub mesh_infos: *const c_void,
    pub visibility_cursor: *mut u32,
    pub n_entities: u32,
    pub visibility_capacity_words: u32,
    pub entity_data: *mut c_void,
    pub entity_draws: *mut c_void,
}

#[repr(C)]
#[derive(Clone, Copy)]
pub struct OrbitSceneBuffers {
    pub entity_draws: *const c_void,
    pub mesh_infos: *const c_void,
    pub entities: *const c_void,
    pub meshlets: *const c_void,
    pub materials: *const c_void,
    pub entity_visibility: *mut u32,
    pub meshlet_visibility: *mut u32,
    pub entity_draw_count: u32,
    pub draw_begin: u32,
    pub draw_end: u32,
    pub reserved: u32,
}

#[repr(C)]
#[derive(Clone, Copy)]
pub struct OrbitHizInfo {
    pub width: u32, pub height: u32, pub levels: u32, pub total_texels: u32,
    pub level_offset: [u32; ORBIT_HIZ_MAX_LEVELS],
    pub texels: *mut f32,
}

#[repr(C)]
#[derive(Clone, Copy)]
pub struct OrbitClusterCullInfo {
    pub world_to_view_matrix: [f32; 16],
    pub screen_to_view_matrix: [f32; 16],
    pub cluster_count: [u32; 3],
    pub tile_size_px: u32,
    pub screen_size: [u32; 2],
    pub z_near: f32,
    pub z_far: f32,
    pub unique_cluster_buffer: u32, pub cluster_offset_image: u32, pub light_index_buffer: u32, pub depth_bounds_buffer: u32,
    pub global_light_count: u32, pub global_light_list: u32, pub _padding: [u32; 2],
}
const _: () = assert!(std::mem::size_of::<OrbitClusterCullInfo>() == 192);

#[repr(C)]
#[derive(Clone, Copy)]
pub struct OrbitClusterParams { pub info: OrbitClusterCullInfo, pub z_scale: f32, pub z_bias: f32, pub reserved: [u32; 2] }

#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct OrbitStatus { pub dispatch_overflow: u32, pub draw_overflow: u32, pub light_index_overflow: u32, pub visibility_overflow: u32, pub asset_error: u32, pub peer_timeout: u32, pub reserved: [u32; 2] }

#[repr(C)]
#[derive(Clone, Copy)]
pub struct OrbitPeerPut { pub src: *const c_void, pub dst: *mut c_void, pub bytes: u64, pub dst_flag: *mut u32 }

extern "C" {
    pub fn orbit_abi_version() -> i32;
    pub fn orbit_error_string(code: i32) -> *const std::os::raw::c_char;
    pub fn orbit_last_cuda_error() -> i32;
    pub fn orbit_ctx_create(device: i32, out: *mut *mut orbit_ctx) -> i32;
    pub fn orbit_ctx_destroy(ctx: *mut orbit_ctx);
    pub fn orbit_ctx_poll_status(ctx: *mut orbit_ctx, out: *mut OrbitStatus) -> i32;
    pub fn orbit_ctx_launch_count(ctx: *const orbit_ctx) -> u64;
    pub fn orbit_ctx_reserve(ctx: *mut orbit_ctx, entity_draws: u64, capacity_records: u64, n_lights: u64, n_clusters: u64, n_entities: u64) -> i32;
    pub fn orbit_hiz_geometry(depth_width: u32, depth_height: u32, out: *mut OrbitHizInfo) -> i32;
    pub fn orbit_hiz_create(ctx: *mut orbit_ctx, depth_width: u32, depth_height: u32, out: *mut *mut orbit_hiz) -> i32;
    pub fn orbit_hiz_wrap(ctx: *mut orbit_ctx, depth_width: u32, depth_height: u32, texels: *mut f32, out: *mut *mut orbit_hiz) -> i32;
    pub fn orbit_hiz_destroy(hiz: *mut orbit_hiz);
    pub fn orbit_hiz_info(hiz: *const orbit_hiz, out: *mut OrbitHizInfo) -> i32;
    pub fn orbit_hiz_build(ctx: *mut orbit_ctx, hiz: *mut orbit_hiz, depth: *const f32, depth_width: u32, depth_height: u32, stream: *mut c_void) -> i32;
    pub fn orbit_entity_cull(ctx: *mut orbit_ctx, cull: *const OrbitCullInfo, scene: *const OrbitSceneBuffers, hiz: *const orbit_hiz,
                             meshlet_dispatch_buffer: *mut c_void, capacity_records: u64, stream: *mut c_void) -> i32;
    pub fn orbit_meshlet_cull(ctx: *mut orbit_ctx, cull: *const OrbitCullInfo, scene: *const OrbitSceneBuffers, hiz: *const orbit_hiz,
                              meshlet_dispatch_buffer: *const c_void, capacity_records: u64, draw_command_buffer: *mut c_void,
                              capacity_draws: u64, task_payloads: *mut c_void, stream: *mut c_void) -> i32;
    pub fn orbit_light_cluster(ctx: *mut orbit_ctx, params: *const OrbitClusterParams, depth: *const f32, lights: *const c_void,
                               tile_masks: *mut c_void, depth_bounds: *mut c_void, unique_clusters: *mut c_void,
                               offset_count_image: *mut c_void, light_index_list: *mut c_void, capacity_indices: u64, stream: *mut c_void) -> i32;
    pub fn orbit_peer_put(ctx: *mut orbit_ctx, puts: *const OrbitPeerPut, n_puts: u32, flag_value: u32, stream: *mut c_void) -> c_int;
    pub fn orbit_peer_wait(ctx: *mut orbit_ctx, flags: *const u32, n_flags: u32, stride_words: u32, flag_value: u32, stream: *mut c_void) -> c_int;
    pub fn orbit_cull_pair_compatible(late: *const OrbitCullInfo, main_pass: *const OrbitCullInfo) -> c_int;
    pub fn orbit_entity_cull_late_main(ctx: *mut orbit_ctx, late: *const OrbitCullInfo, main_pass: *const OrbitCullInfo, scene: *const OrbitSceneBuffers,
                                       hiz: *const orbit_hiz, late_dispatch_buffer: *mut c_void, main_dispatch_buffer: *mut c_void,
                                       capacity_records: u64, stream: *mut c_void) -> c_int;
    pub fn orbit_meshlet_cull_late_main(ctx: *mut orbit_ctx, late: *const OrbitCullInfo, main_pass: *const OrbitCullInfo, scene: *const OrbitSceneBuffers,
                                        hiz: *const orbit_hiz, late_dispatch_buffer: *const c_void, capacity_records: u64,
                                        late_draw_command_buffer: *mut c_void, main_draw_command_buffer: *mut c_void, capacity_draws: u64,
                                        late_task_payloads: *mut c_void, main_task_payloads: *mut c_void, stream: *mut c_void) -> c_int;
    pub fn orbit_hiz_build_entity_cull_late(ctx: *mut orbit_ctx, hiz: *mut orbit_hiz, depth: *const f32, depth_width: u32, depth_height: u32,
                                            late: *const OrbitCullInfo, main_pass: *const OrbitCullInfo, scene: *const OrbitSceneBuffers,
                                            late_dispatch_buffer: *mut c_void, main_dispatch_buffer: *mut c_void, capacity_records: u64,
                                            stream: *mut c_void) -> c_int;
    pub fn orbit_entity_cull_views(ctx: *mut orbit_ctx, culls: *const OrbitCullInfo, n_views: u32, scene: *const OrbitSceneBuffers,
                                   dispatch_buffers: *const *mut c_void, capacity_records: u64, stream: *mut c_void) -> c_int;
    pub fn orbit_meshlet_cull_views(ctx: *mut orbit_ctx, culls: *const OrbitCullInfo, n_views: u32, scene: *const OrbitSceneBuffers,
                                    dispatch_buffers: *const *const c_void, capacity_records: u64, draw_command_buffers: *const *mut c_void,
                                    capacity_draws: u64, task_payloads: *const *mut c_void, stream: *mut c_void) -> c_int;
    pub fn orbit_hiz_build_views(ctx: *mut orbit_ctx, hizs: *const *mut orbit_hiz, depths: *const *const f32, n_views: u32,
                                 depth_width: u32, depth_height: u32, stream: *mut c_void) -> c_int;
    pub fn orbit_entity_cull_views_occlusion(ctx: *mut orbit_ctx, culls: *const OrbitCullInfo, n_views: u32, scenes: *const OrbitSceneBuffers,
                                             hizs: *const *const orbit_hiz, dispatch_buffers: *const *mut c_void, capacity_records: u64,
                                             stream: *mut c_void) -> c_int;
    pub fn orbit_meshlet_cull_views_occlusion(ctx: *mut orbit_ctx, culls: *const OrbitCullInfo, n_views: u32, scenes: *const OrbitSceneBuffers,
                                              hizs: *const *const orbit_hiz, dispatch_buffers: *const *const c_void, capacity_records: u64,
                                              draw_command_buffers: *const *mut c_void, capacity_draws: u64, task_payloads: *const *mut c_void,
                                              stream: *mut c_void) -> c_int;
    pub fn orbit_draws_scatter_ranked(ctx: *mut orbit_ctx, src_draw_buffer: *const c_void, src_capacity_draws: u64, dst_draw_buffer: *mut c_void,
                                      rank_counts: *const u32, rank: u32, world: u32, dst_capacity_draws: u64, stream: *mut c_void) -> i32;
    pub fn orbit_meshlet_test(ctx: *mut orbit_ctx, cull: *const OrbitCullInfo, scene: *const OrbitSceneBuffers, hiz: *const orbit_hiz,
                              meshlet_dispatch_buffer: *const c_void, capacity_records: u64, record_masks: *mut c_void, stream: *mut c_void) -> i32;
    pub fn orbit_record_masks_put(ctx: *mut orbit_ctx, src_record_masks: *const c_void, meshlet_dispatch_buffer: *const c_void, capacity_records: u64,
                                  dst_region: *mut c_void, dst_count: *mut u32, stream: *mut c_void) -> i32;
    pub fn orbit_draws_from_masks(ctx: *mut orbit_ctx, scene: *const OrbitSceneBuffers, record_masks: *const c_void, region_stride_records: u64,
                                  region_counts: *const u32, n_regions: u32, draw_command_buffer: *mut c_void, capacity_draws: u64,
                                  stream: *mut c_void) -> i32;
    pub fn orbit_scene_update(ctx: *mut orbit_ctx, update: *const OrbitSceneUpdate, stream: *mut c_void) -> i32;
    pub fn orbit_meshlet_bounds(ctx: *mut orbit_ctx, vertices: *const c_void, vertex_stride: u32, meshlet_data: *const u32, meshlets: *mut c_void,
                                n_meshlets: u32, stream: *mut c_void) -> i32;
    pub fn orbit_mesh_bounds(ctx: *mut orbit_ctx, vertices: *const c_void, vertex_stride: u32, vertex_ranges: *const u32, mesh_infos: *mut c_void,
                             n_meshes: u32, stream: *mut c_void) -> i32;
    pub fn orbit_draws_scatter(ctx: *mut orbit_ctx, src_draw_buffer: *const c_void, src_capacity_draws: u64, dst_draw_buffer: *mut c_void,
                               dst_first: u32, total_count: u32, dst_capacity_draws: u64, stream: *mut c_void) -> i32;
    pub fn orbit_depth_image_wrap(ctx: *mut orbit_ctx, cuda_array: *mut c_void, out: *mut *mut orbit_depth_image) -> c_int;
    pub fn orbit_depth_image_destroy(image: *mut orbit_depth_image);
    pub fn orbit_depth_image_size(image: *const orbit_depth_image, width: *mut u32, height: *mut u32) -> c_int;
    pub fn orbit_hiz_build_image(ctx: *mut orbit_ctx, hiz: *mut orbit_hiz, image: *const orbit_depth_image, stream: *mut c_void) -> c_int;
    pub fn orbit_hiz_build_views_image(ctx: *mut orbit_ctx, hizs: *const *mut orbit_hiz, images: *const *const orbit_depth_image, n_views: u32,
                                       stream: *mut c_void) -> c_int;
    pub fn orbit_hiz_build_image_entity_cull_late(ctx: *mut orbit_ctx, hiz: *mut orbit_hiz, image: *const orbit_depth_image,
                                                  late: *const OrbitCullInfo, main_pass: *const OrbitCullInfo, scene: *const OrbitSceneBuffers,
                                                  late_dispatch_buffer: *mut c_void, main_dispatch_buffer: *mut c_void, capacity_records: u64,
                                                  stream: *mut c_void) -> c_int;
    pub fn orbit_light_cluster_image(ctx: *mut orbit_ctx, params: *const OrbitClusterParams, image: *const orbit_depth_image, lights: *const c_void,
                                     tile_masks: *mut c_void, depth_bounds: *mut c_void, unique_clusters: *mut c_void,
                                     offset_count_image: *mut c_void, light_index_list: *mut c_void, capacity_indices: u64,
                                     stream: *mut c_void) -> c_int;
    pub fn orbit_hiz_attach_image(ctx: *mut orbit_ctx, hiz: *mut orbit_hiz, cuda_mipmapped_array: *mut c_void) -> c_int;
    pub fn orbit_cluster_grid_wrap(ctx: *mut orbit_ctx, cuda_array: *mut c_void, out: *mut *mut orbit_cluster_grid) -> c_int;
    pub fn orbit_cluster_grid_destroy(grid: *mut orbit_cluster_grid);
    pub fn orbit_light_cluster_image_grid(ctx: *mut orbit_ctx, params: *const OrbitClusterParams, image: *const orbit_depth_image,
                                          lights: *const c_void, tile_masks: *mut c_void, depth_bounds: *mut c_void,
                                          unique_clusters: *mut c_void, grid: *const orbit_cluster_grid, light_index_list: *mut c_void,
                                          capacity_indices: u64, stream: *mut c_void) -> c_int;
}

/// Safe-ish wrappers shaped like the reference entry points (draw_gen.rs:327-389, 456-566).
pub struct Context(*mut orbit_ctx);
unsafe impl Send for Context {}

#[derive(Debug)]
pub struct Error(pub i32);
fn check(rc: i32) -> Result<(), Error> { if rc == ORBIT_OK { Ok(()) } else { Err(Error(rc)) } }

impl Context {
    pub fn new(device: i32) -> Result<Self, Error> {
        let mut p = std::ptr::null_mut();
        check(unsafe { orbit_ctx_create(device, &mut p) })?;
        Ok(Self(p))
    }
    /// create_meshlet_dispatch_command (draw_gen.rs:327-380): `cull` is `CullInfo::to_gpu()` reinterpreted.
    pub unsafe fn create_meshlet_dispatch_command(&self, cull: &OrbitCullInfo, scene: &OrbitSceneBuffers, hiz: *const orbit_hiz,
                                                  meshlet_dispatch_buffer: *mut c_void, capacity_records: u64, stream: *mut c_void) -> Result<(), Error> {
        check(orbit_entity_cull(self.0, cull, scene, hiz, meshlet_dispatch_buffer, capacity_records, stream))
    }
    /// create_meshlet_draw_commands (draw_gen.rs:382-435).
    pub unsafe fn create_meshlet_draw_commands(&self, cull: &OrbitCullInfo, scene: &OrbitSceneBuffers, hiz: *const orbit_hiz,
                                               meshlet_dispatch_buffer: *const c_void, capacity_records: u64,
                                               draw_command_buffer: *mut c_void, capacity_draws: u64, stream: *mut c_void) -> Result<(), Error> {
        check(orbit_meshlet_cull(self.0, cull, scene, hiz, meshlet_dispatch_buffer, capacity_records, draw_command_buffer,
                                 capacity_draws, std::ptr::null_mut(), stream))
    }
    /// The LATE cull of the depth prepass (forward.rs:266-403) + the MAIN pass's cull (forward.rs:518-548), fused. Ok(false):
    /// the two CullInfos are not a compatible pair and nothing was launched — issue the four separate calls instead.
    pub unsafe fn create_late_and_main_commands(&self, late: &OrbitCullInfo, main_pass: &OrbitCullInfo, scene: &OrbitSceneBuffers,
                                                hiz: *const orbit_hiz, late_dispatch_buffer: *mut c_void, main_dispatch_buffer: *mut c_void,
                                                capacity_records: u64, late_draw_command_buffer: *mut c_void,
                                                main_draw_command_buffer: *mut c_void, capacity_draws: u64, stream: *mut c_void) -> Result<bool, Error> {
        if orbit_cull_pair_compatible(late, main_pass) == 0 { return Ok(false); }
        check(orbit_entity_cull_late_main(self.0, late, main_pass, scene, hiz, late_dispatch_buffer, main_dispatch_buffer, capacity_records, stream))?;
        check(orbit_meshlet_cull_late_main(self.0, late, main_pass, scene, hiz, late_dispatch_buffer, capacity_records, late_draw_command_buffer,
                                           main_draw_command_buffer, capacity_draws, std::ptr::null_mut(), std::ptr::null_mut(), stream))?;
        Ok(true)
    }
    /// Pass-0 culling of up to ORBIT_MAX_BATCH_VIEWS views of one scene (the cascades of render_cascaded_shadow,
    /// shadow_renderer.rs:466-712): buffer v receives what create_meshlet_dispatch_command / create_meshlet_draw_commands
    /// write for `culls[v]`, from 3 kernel launches in all. The three slices have one entry per view.
    pub unsafe fn create_views_commands(&self, culls: &[OrbitCullInfo], scene: &OrbitSceneBuffers, dispatch_buffers: &[*mut c_void],
                                        capacity_records: u64, draw_command_buffers: &[*mut c_void], capacity_draws: u64,
                                        stream: *mut c_void) -> Result<(), Error> {
        if culls.len() > ORBIT_MAX_BATCH_VIEWS as usize || dispatch_buffers.len() != culls.len() || draw_command_buffers.len() != culls.len() {
            return Err(Error(ORBIT_ERR_INVALID_ARGUMENT));
        }
        let n = culls.len() as u32;
        check(orbit_entity_cull_views(self.0, culls.as_ptr(), n, scene, dispatch_buffers.as_ptr(), capacity_records, stream))?;
        check(orbit_meshlet_cull_views(self.0, culls.as_ptr(), n, scene, dispatch_buffers.as_ptr() as *const *const c_void, capacity_records,
                                       draw_command_buffers.as_ptr(), capacity_draws, std::ptr::null(), stream))
    }
    /// One occlusion pass (EARLY or MAIN: pass 1; LATE: pass 2) of up to ORBIT_MAX_BATCH_VIEWS cameras over one scene: buffer v
    /// receives what create_meshlet_dispatch_command / create_meshlet_draw_commands write for `culls[v]` with `scenes[v]` (the
    /// scene with camera v's visibility buffers) and, for pass 2, `pyramids[v]`; 3 kernel launches in all. Every slice has one
    /// entry per camera (`pyramids` is empty for pass 1).
    pub unsafe fn create_views_occlusion_commands(&self, culls: &[OrbitCullInfo], scenes: &[OrbitSceneBuffers], pyramids: &[DepthPyramid],
                                                  dispatch_buffers: &[*mut c_void], capacity_records: u64,
                                                  draw_command_buffers: &[*mut c_void], capacity_draws: u64,
                                                  stream: *mut c_void) -> Result<(), Error> {
        let n = culls.len();
        if n > ORBIT_MAX_BATCH_VIEWS as usize || scenes.len() != n || dispatch_buffers.len() != n || draw_command_buffers.len() != n
            || !(pyramids.is_empty() || pyramids.len() == n) {
            return Err(Error(ORBIT_ERR_INVALID_ARGUMENT));
        }
        let hizs: Vec<*const orbit_hiz> = pyramids.iter().map(|p| p.hiz as *const orbit_hiz).collect();
        let hz = if hizs.is_empty() { std::ptr::null() } else { hizs.as_ptr() };
        check(orbit_entity_cull_views_occlusion(self.0, culls.as_ptr(), n as u32, scenes.as_ptr(), hz, dispatch_buffers.as_ptr(),
                                                capacity_records, stream))?;
        check(orbit_meshlet_cull_views_occlusion(self.0, culls.as_ptr(), n as u32, scenes.as_ptr(), hz,
                                                 dispatch_buffers.as_ptr() as *const *const c_void, capacity_records,
                                                 draw_command_buffers.as_ptr(), capacity_draws, std::ptr::null(), stream))
    }
    /// update_multiple_depth_pyramids (draw_gen.rs): DepthPyramid::update for up to ORBIT_MAX_BATCH_VIEWS pyramids of one size in
    /// one launch; depth buffer v feeds pyramid v.
    pub unsafe fn update_depth_pyramids(&self, pyramids: &mut [DepthPyramid], depths: &[*const f32], stream: *mut c_void) -> Result<(), Error> {
        if pyramids.is_empty() || pyramids.len() > ORBIT_MAX_BATCH_VIEWS as usize || depths.len() != pyramids.len() {
            return Err(Error(ORBIT_ERR_INVALID_ARGUMENT));
        }
        let size = pyramids[0].size;
        let hizs: Vec<*mut orbit_hiz> = pyramids.iter().map(|p| p.hiz).collect();
        check(orbit_hiz_build_views(self.0, hizs.as_ptr(), depths.as_ptr(), pyramids.len() as u32, size[0], size[1], stream))?;
        for p in pyramids.iter_mut() { p.usable = true; }
        Ok(())
    }
}
impl Drop for Context { fn drop(&mut self) { unsafe { orbit_ctx_destroy(self.0) } } }

/// DepthPyramid (draw_gen.rs:451-567) over orbit_hiz.
pub struct DepthPyramid { hiz: *mut orbit_hiz, size: [u32; 2], pub usable: bool }
impl DepthPyramid {
    pub fn new(ctx: &Context, [width, height]: [u32; 2]) -> Result<Self, Error> {
        let mut h = std::ptr::null_mut();
        check(unsafe { orbit_hiz_create(ctx.0, width, height, &mut h) })?;
        Ok(Self { hiz: h, size: [width, height], usable: false })
    }
    pub unsafe fn update(&mut self, ctx: &Context, depth_buffer: *const f32, stream: *mut c_void) -> Result<(), Error> {
        check(orbit_hiz_build(ctx.0, self.hiz, depth_buffer, self.size[0], self.size[1], stream))?;
        self.usable = true;
        Ok(())
    }
    pub fn get_current(&self) -> *const orbit_hiz { self.hiz }
    /// update() followed by the LATE cull's create_meshlet_dispatch_command (`late`: pass 2 against this pyramid) or, with
    /// `main_pass`, by the entity half of create_late_and_main_commands, in one call: the same buffers, with the entity kernel's
    /// pyramid-independent work under the build (orbit_hiz_build_entity_cull_late). `main_dispatch_buffer` is null without `main_pass`.
    pub unsafe fn update_and_cull_late(&mut self, ctx: &Context, depth_buffer: *const f32, late: &OrbitCullInfo, main_pass: Option<&OrbitCullInfo>,
                                       scene: &OrbitSceneBuffers, late_dispatch_buffer: *mut c_void, main_dispatch_buffer: *mut c_void,
                                       capacity_records: u64, stream: *mut c_void) -> Result<(), Error> {
        let main_ptr = main_pass.map_or(std::ptr::null(), |m| m as *const OrbitCullInfo);
        check(orbit_hiz_build_entity_cull_late(ctx.0, self.hiz, depth_buffer, self.size[0], self.size[1], late, main_ptr, scene,
                                               late_dispatch_buffer, main_dispatch_buffer, capacity_records, stream))?;
        self.usable = true;
        Ok(())
    }
}
impl Drop for DepthPyramid { fn drop(&mut self) { unsafe { orbit_hiz_destroy(self.hiz) } } }

/// The depth attachment as a CUDA array (orbit_depth_image_wrap): level 0 of the mipmapped array that
/// cudaExternalMemoryGetMappedMipmappedArray maps from an imported VkImage, with one 32-bit float channel. The array stays the
/// caller's; it, and this handle, must outlive every enqueued call and captured graph that reads them. Ordering the renderer's
/// writes of the image before the calls (an imported semaphore waited on the stream) is the caller's job.
pub struct DepthImage { image: *mut orbit_depth_image, size: [u32; 2] }
impl DepthImage {
    pub unsafe fn wrap(ctx: &Context, cuda_array: *mut c_void) -> Result<Self, Error> {
        let mut p = std::ptr::null_mut();
        check(orbit_depth_image_wrap(ctx.0, cuda_array, &mut p))?;
        let (mut w, mut h) = (0u32, 0u32);
        check(orbit_depth_image_size(p, &mut w, &mut h))?;
        Ok(Self { image: p, size: [w, h] })
    }
    pub fn size(&self) -> [u32; 2] { self.size }
    pub fn as_ptr(&self) -> *const orbit_depth_image { self.image }
}
impl Drop for DepthImage { fn drop(&mut self) { unsafe { orbit_depth_image_destroy(self.image) } } }

impl DepthPyramid {
    /// update() with the depth read from `image` (orbit_hiz_build_image): the same texels.
    pub unsafe fn update_from_image(&mut self, ctx: &Context, image: &DepthImage, stream: *mut c_void) -> Result<(), Error> {
        check(orbit_hiz_build_image(ctx.0, self.hiz, image.image, stream))?;
        self.usable = true;
        Ok(())
    }
    /// update_and_cull_late() with the depth read from `image` (orbit_hiz_build_image_entity_cull_late).
    pub unsafe fn update_from_image_and_cull_late(&mut self, ctx: &Context, image: &DepthImage, late: &OrbitCullInfo,
                                                  main_pass: Option<&OrbitCullInfo>, scene: &OrbitSceneBuffers, late_dispatch_buffer: *mut c_void,
                                                  main_dispatch_buffer: *mut c_void, capacity_records: u64, stream: *mut c_void) -> Result<(), Error> {
        let main_ptr = main_pass.map_or(std::ptr::null(), |m| m as *const OrbitCullInfo);
        check(orbit_hiz_build_image_entity_cull_late(ctx.0, self.hiz, image.image, late, main_ptr, scene, late_dispatch_buffer,
                                                     main_dispatch_buffer, capacity_records, stream))?;
        self.usable = true;
        Ok(())
    }
}

impl Context {
    /// update_depth_pyramids() with depth v read from images[v] (orbit_hiz_build_views_image).
    pub unsafe fn update_depth_pyramids_from_images(&self, pyramids: &mut [DepthPyramid], images: &[&DepthImage], stream: *mut c_void) -> Result<(), Error> {
        if pyramids.is_empty() || pyramids.len() > ORBIT_MAX_BATCH_VIEWS as usize || images.len() != pyramids.len() {
            return Err(Error(ORBIT_ERR_INVALID_ARGUMENT));
        }
        let hizs: Vec<*mut orbit_hiz> = pyramids.iter().map(|p| p.hiz).collect();
        let imgs: Vec<*const orbit_depth_image> = images.iter().map(|i| i.image as *const orbit_depth_image).collect();
        check(orbit_hiz_build_views_image(self.0, hizs.as_ptr(), imgs.as_ptr(), pyramids.len() as u32, stream))?;
        for p in pyramids.iter_mut() { p.usable = true; }
        Ok(())
    }
    /// compute_clusters (cluster.rs:368-591) with the depth read from `image` (orbit_light_cluster_image).
    pub unsafe fn compute_clusters_from_image(&self, params: &OrbitClusterParams, image: &DepthImage, lights: *const c_void,
                                              tile_masks: *mut c_void, depth_bounds: *mut c_void, unique_clusters: *mut c_void,
                                              offset_count_image: *mut c_void, light_index_list: *mut c_void, capacity_indices: u64,
                                              stream: *mut c_void) -> Result<(), Error> {
        check(orbit_light_cluster_image(self.0, params, image.image, lights, tile_masks, depth_bounds, unique_clusters, offset_count_image,
                                        light_index_list, capacity_indices, stream))
    }
}

/// The cluster offset/count grid as a CUDA array (orbit_cluster_grid_wrap): the 3-D R32G32_UINT cluster image
/// (cluster.rs:532-544) mapped from an imported VkImage (cudaExternalMemoryGetMappedMipmappedArray, level 0), created with
/// surface load/store. The array stays the caller's; it, and this handle, must outlive every enqueued call and captured graph
/// that writes them.
pub struct ClusterGrid { grid: *mut orbit_cluster_grid }
impl ClusterGrid {
    pub unsafe fn wrap(ctx: &Context, cuda_array: *mut c_void) -> Result<Self, Error> {
        let mut p = std::ptr::null_mut();
        check(orbit_cluster_grid_wrap(ctx.0, cuda_array, &mut p))?;
        Ok(Self { grid: p })
    }
    pub fn as_ptr(&self) -> *const orbit_cluster_grid { self.grid }
}
impl Drop for ClusterGrid { fn drop(&mut self) { unsafe { orbit_cluster_grid_destroy(self.grid) } } }

impl DepthPyramid {
    /// Mirrors every later build of this pyramid into `cuda_mipmapped_array` (a cudaMipmappedArray_t with exactly this
    /// pyramid's levels, one f32 channel, surface load/store), e.g. the renderer's pyramid image imported from Vulkan
    /// (orbit_hiz_attach_image). The culling calls keep reading the linear pyramid; the array must outlive the pyramid.
    pub unsafe fn attach_image(&mut self, ctx: &Context, cuda_mipmapped_array: *mut c_void) -> Result<(), Error> {
        check(orbit_hiz_attach_image(ctx.0, self.hiz, cuda_mipmapped_array))
    }
}

impl Context {
    /// compute_clusters_from_image() with the offset/count grid written into `grid` (orbit_light_cluster_image_grid).
    pub unsafe fn compute_clusters_into_grid(&self, params: &OrbitClusterParams, image: &DepthImage, lights: *const c_void,
                                             tile_masks: *mut c_void, depth_bounds: *mut c_void, unique_clusters: *mut c_void,
                                             grid: &ClusterGrid, light_index_list: *mut c_void, capacity_indices: u64,
                                             stream: *mut c_void) -> Result<(), Error> {
        check(orbit_light_cluster_image_grid(self.0, params, image.image, lights, tile_masks, depth_bounds, unique_clusters, grid.grid,
                                             light_index_list, capacity_indices, stream))
    }
}
