"""Python mirrors of include/orbit_layouts.h + the ABI structs of include/orbit_cuda.h.

numpy structured dtypes describe the arrays the scene generator writes (reference layouts: src/assets/mod.rs:18-43,
98-122,171-191; src/scene.rs:120-133,278-291; shaders/include/types.glsl:75-228,246-276); ctypes Structures
describe what crosses the C ABI by value.
"""
import ctypes as C

import numpy as np

MAX_CULL_PLANES = 12
MAX_BATCH_VIEWS = 16          # ORBIT_MAX_BATCH_VIEWS: views per orbit_entity_cull_views / orbit_meshlet_cull_views call
MESHLET_DISPATCH_SIZE = 32
MAX_MESH_LODS = 8
NO_BUFFER = 0xFFFFFFFF
MAX_LIGHTS_PER_CLUSTER = 256
HIZ_MAX_LEVELS = 16

PASS_NONE, PASS_VISIBILITY_READ, PASS_VISIBILITY_WRITE = 0, 1, 2
PROJ_PERSPECTIVE, PROJ_ORTHOGRAPHIC = 0, 1
ALPHA_OPAQUE, ALPHA_MASKED, ALPHA_TRANSPARENT = 0, 1, 2
LIGHT_SKY, LIGHT_DIRECTIONAL, LIGHT_POINT = 0, 1, 2

MATERIAL_STRIDE = 80
MATERIAL_ALPHA_OFFSET = 64
ENTITY_DRAW_HEADER = 4
DISPATCH_HEADER = 12
DRAW_HEADER = 4
TASK_PAYLOAD_STRIDE = 44

meshlet_dtype = np.dtype([
    ("bounding_sphere", "<f4", (4,)), ("cone_axis", "i1", (3,)), ("cone_cutoff", "i1"),
    ("vertex_offset", "<u4"), ("data_offset", "<u4"), ("material_index", "<u2"),
    ("vertex_count", "u1"), ("triangle_count", "u1")])
mesh_info_dtype = np.dtype([
    ("bounding_sphere", "<f4", (4,)), ("aabb_min", "<f4", (4,)), ("aabb_max", "<f4", (4,)),
    ("vertex_offset", "<u4"), ("meshlet_data_offset", "<u4"), ("lod_count", "<u4"), ("_padding", "<u4"),
    ("mesh_lods", "<u4", (MAX_MESH_LODS, 2))])   # [lod] = (meshlet_offset, meshlet_count)
entity_dtype = np.dtype([("model_matrix", "<f4", (4, 4)), ("normal_matrix", "<f4", (4, 4))])  # [col][row]
entity_draw_dtype = np.dtype([("entity_index", "<u4"), ("mesh_index", "<u4"), ("visibility_offset", "<u4")])
dispatch_dtype = np.dtype([("entity_index", "<u4"), ("meshlet_offset", "<u4"), ("meshlet_count", "<u4"),
                           ("visibility_offset", "<u4")])
draw_command_dtype = np.dtype([
    ("cmd_index_count", "<u4"), ("cmd_instance_count", "<u4"), ("cmd_first_index", "<u4"),
    ("cmd_vertex_offset", "<i4"), ("cmd_first_instance", "<u4"), ("meshlet_vertex_offset", "<u4"),
    ("meshlet_index", "<u4")])
task_payload_dtype = np.dtype([("task_count", "<u4"), ("entity_index", "<u4"), ("meshlet_offset", "<u4"),
                               ("meshlet_indices", "u1", (32,))])
light_dtype = np.dtype([
    ("light_type", "<u4"), ("shadow_data_index", "<u4"), ("irradiance_map", "<u4"), ("prefiltered_map", "<u4"),
    ("color", "<f4", (3,)), ("intensity", "<f4"), ("position", "<f4", (3,)), ("inner_radius", "<f4"),
    ("direction", "<f4", (3,)), ("outer_radius", "<f4")])
# Transform (scene.rs:18-23) in the 48-byte layout orbit_scene_update reads (include/orbit_layouts.h OrbitTransform)
transform_dtype = np.dtype([("position", "<f4", (3,)), ("_pad0", "<f4"), ("orientation", "<f4", (4,)),
                            ("scale", "<f4", (3,)), ("_pad1", "<f4")])
NO_MESH = 0xFFFFFFFF
NO_VISIBILITY_RANGE = 0xFFFFFFFF
assert transform_dtype.itemsize == 48
assert meshlet_dtype.itemsize == 32 and mesh_info_dtype.itemsize == 128 and entity_dtype.itemsize == 128
assert entity_draw_dtype.itemsize == 12 and dispatch_dtype.itemsize == 16 and draw_command_dtype.itemsize == 28
assert task_payload_dtype.itemsize == 44 and light_dtype.itemsize == 64


class Mat4(C.Structure):
    _fields_ = [("m", (C.c_float * 4) * 4)]  # m[col][row]

    def set(self, a):
        """a: 4x4 array in MATH convention a[row][col]."""
        a = np.asarray(a, dtype=np.float32)
        for col in range(4):
            for row in range(4):
                self.m[col][row] = float(a[row, col])

    def get(self):
        out = np.zeros((4, 4), np.float32)
        for col in range(4):
            for row in range(4):
                out[row, col] = self.m[col][row]
        return out


class CullInfo(C.Structure):
    """GpuCullInfo, 400 bytes (src/passes/draw_gen.rs:208-237)."""
    _fields_ = [
        ("view_matrix", Mat4), ("reprojection_matrix", Mat4),
        ("cull_planes", (C.c_float * 4) * MAX_CULL_PLANES),
        ("cull_plane_count", C.c_uint32), ("alpha_mode_flags", C.c_uint32), ("noskip_alpha_mode", C.c_uint32),
        ("occlusion_pass", C.c_uint32),
        ("visibility_buffer", C.c_uint32), ("meshlet_visibility_buffer", C.c_uint32), ("depth_pyramid", C.c_uint32),
        ("secondary_depth_pyramid", C.c_uint32),
        ("projection_type", C.c_uint32), ("p00_or_width_recip_x2", C.c_float), ("p11_or_height_recip_x2", C.c_float),
        ("z_near", C.c_float),
        ("z_far", C.c_float), ("lod_base", C.c_float), ("lod_step", C.c_float), ("min_mesh_lod", C.c_uint32),
        ("lod_target_pos_view_space", C.c_float * 3), ("max_mesh_lod", C.c_uint32)]


class SceneBuffers(C.Structure):
    _fields_ = [
        ("entity_draws", C.c_void_p), ("mesh_infos", C.c_void_p), ("entities", C.c_void_p), ("meshlets", C.c_void_p),
        ("materials", C.c_void_p), ("entity_visibility", C.c_void_p), ("meshlet_visibility", C.c_void_p),
        ("entity_draw_count", C.c_uint32), ("draw_begin", C.c_uint32), ("draw_end", C.c_uint32), ("reserved", C.c_uint32)]


class HizInfo(C.Structure):
    _fields_ = [("width", C.c_uint32), ("height", C.c_uint32), ("levels", C.c_uint32), ("total_texels", C.c_uint32),
                ("level_offset", C.c_uint32 * HIZ_MAX_LEVELS), ("texels", C.c_void_p)]


class ClusterCullInfo(C.Structure):
    """ClusterCullInfo, 192 bytes (src/passes/cluster.rs:186-207)."""
    _fields_ = [
        ("world_to_view_matrix", Mat4), ("screen_to_view_matrix", Mat4),
        ("cluster_count", C.c_uint32 * 3), ("tile_size_px", C.c_uint32),
        ("screen_size", C.c_uint32 * 2), ("z_near", C.c_float), ("z_far", C.c_float),
        ("unique_cluster_buffer", C.c_uint32), ("cluster_offset_image", C.c_uint32), ("light_index_buffer", C.c_uint32),
        ("depth_bounds_buffer", C.c_uint32),
        ("global_light_count", C.c_uint32), ("global_light_list", C.c_uint32), ("_padding", C.c_uint32 * 2)]


class ClusterParams(C.Structure):
    _fields_ = [("info", ClusterCullInfo), ("z_scale", C.c_float), ("z_bias", C.c_float), ("reserved", C.c_uint32 * 2)]


class Status(C.Structure):
    _fields_ = [("dispatch_overflow", C.c_uint32), ("draw_overflow", C.c_uint32), ("light_index_overflow", C.c_uint32),
                ("visibility_overflow", C.c_uint32), ("asset_error", C.c_uint32), ("peer_timeout", C.c_uint32), ("reserved", C.c_uint32 * 2)]


class PeerPut(C.Structure):
    """OrbitPeerPut (include/orbit_cuda.h): one transfer of orbit_peer_put."""
    _fields_ = [("src", C.c_void_p), ("dst", C.c_void_p), ("bytes", C.c_uint64), ("dst_flag", C.c_void_p)]


class SceneUpdate(C.Structure):
    """OrbitSceneUpdate (include/orbit_cuda.h): arguments of orbit_scene_update (scene.rs:404-492)."""
    _fields_ = [("transforms", C.c_void_p), ("mesh_slots", C.c_void_p), ("visibility_offsets", C.c_void_p),
                ("mesh_infos", C.c_void_p), ("visibility_cursor", C.c_void_p), ("n_entities", C.c_uint32),
                ("visibility_capacity_words", C.c_uint32), ("entity_data", C.c_void_p), ("entity_draws", C.c_void_p)]


assert C.sizeof(SceneUpdate) == 64


class HostFrame(C.Structure):
    """OrbitHostFrame (orbit_b200/host/frame_driver.cpp): one in-flight step of the compiled host frame loop."""
    _fields_ = [("update", SceneUpdate), ("cull_early", CullInfo), ("cull_late", CullInfo),
                ("scene_early", SceneBuffers), ("scene_late", SceneBuffers), ("hiz", C.c_void_p), ("depth", C.c_void_p),
                ("early_dispatch", C.c_void_p), ("early_draws", C.c_void_p), ("late_dispatch", C.c_void_p),
                ("late_draws", C.c_void_p), ("main_dispatch", C.c_void_p), ("main_draws", C.c_void_p),
                ("capacity_records", C.c_uint64), ("capacity_draws", C.c_uint64),
                ("width", C.c_uint32), ("height", C.c_uint32)]


class HostFrameIO(C.Structure):
    _fields_ = [("h_transforms", C.c_void_p), ("h_depth", C.c_void_p), ("h_counts", C.c_void_p),
                ("h_early_draws", C.c_void_p), ("h_late_draws", C.c_void_p), ("h_main_draws", C.c_void_p),
                ("depth_resident", C.c_uint32), ("reserved", C.c_uint32), ("h2d_bytes_per_step", C.c_uint64),
                ("d2h_bytes_last_step", C.c_uint64), ("ms_per_step", C.c_double)]
assert C.sizeof(CullInfo) == 400 and C.sizeof(ClusterCullInfo) == 192 and C.sizeof(ClusterParams) == 208
assert C.sizeof(SceneBuffers) == 72
