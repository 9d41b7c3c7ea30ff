"""Host-side mirror of the reference's culling-pass interface over the C ABI.

Same names, argument meaning and failure behaviour as src/passes/draw_gen.rs and src/passes/cluster.rs:

    CullInfo / OcclusionCullInfo / AlphaModeFlags / Projection        draw_gen.rs:24-203,630-641; camera.rs:66-98
    create_meshlet_dispatch_command(ctx, name, assets, scene, cull)   draw_gen.rs:327-380
    create_meshlet_draw_commands(ctx, name, assets, scene, cull, buf) draw_gen.rs:382-435
    DepthPyramid.{new, resize, update, get_current}                   draw_gen.rs:451-567
    ClusterSettings, compute_clusters                                 cluster.rs:15-72,368-591

torch is used for device memory and streams only; every stage runs in liborbit_b200.so (hand-written CUDA for
sm_100a). There is no CPU path: constructing a Context without a GPU or without the built library raises.
"""
import ctypes as C
from dataclasses import dataclass, field
from typing import Optional, Sequence

import numpy as np
import torch

from . import _lib
from . import layouts as L

MAX_DRAW_COUNT = 1_000_000              # draw_gen.rs:15 (reference capacity; ours is a parameter)
MAX_MESHLET_DISPATCH_COUNT = 1_000_000  # draw_gen.rs:16


class AlphaModeFlags(int):
    """draw_gen.rs:630-641"""
    OPAQUE = 1
    MASKED = 2
    TRANSPARENT = 4
    ALL = 7


@dataclass
class Projection:
    """camera.rs:66-98. kind: 'perspective' (fov, near_clip) or 'orthographic' (half_width, near_clip, far_clip)."""
    kind: str
    fov: float = 0.0
    near_clip: float = 0.01
    far_clip: float = 0.0
    half_width: float = 0.0

    @staticmethod
    def perspective(fov, near_clip):
        return Projection("perspective", fov=fov, near_clip=near_clip)

    @staticmethod
    def orthographic(half_width, near_clip, far_clip):
        return Projection("orthographic", half_width=half_width, near_clip=near_clip, far_clip=far_clip)


@dataclass
class OcclusionCullInfo:
    """draw_gen.rs:24-103. kind: 'none' | 'read' (VisibilityRead) | 'write' (VisibilityWrite)."""
    kind: str = "none"
    visibility_buffer: Optional[torch.Tensor] = None            # int32/uint8 device tensor, one bit per entity draw
    meshlet_visibility_buffer: Optional[torch.Tensor] = None    # None disables meshlet occlusion culling
    depth_pyramid: Optional["DepthPyramid"] = None
    noskip_alphamode: int = 0
    aspect_ratio: float = 1.0

    def pass_index(self):
        return {"none": 0, "read": 1, "write": 2}[self.kind]


@dataclass
class CullInfo:
    """draw_gen.rs:105-119"""
    view_matrix: np.ndarray                          # 4x4, math convention [row, col]
    view_space_cull_planes: Sequence[Sequence[float]]
    projection: Projection
    occlusion_culling: OcclusionCullInfo = field(default_factory=OcclusionCullInfo)
    alpha_mode_filter: int = AlphaModeFlags.OPAQUE | AlphaModeFlags.MASKED
    lod_range: tuple = (0, 8)
    lod_base: float = 16.0
    lod_step: float = 2.0
    lod_target_pos_view_space: tuple = (0.0, 0.0, 0.0)

    def to_gpu(self) -> L.CullInfo:
        """CullInfo::to_gpu, draw_gen.rs:121-203 (f32 arithmetic like the Rust host code)."""
        planes = np.asarray(self.view_space_cull_planes, dtype=np.float32).reshape(-1, 4)
        assert len(planes) <= L.MAX_CULL_PLANES, "assert!(cull_planes.len() <= MAX_CULL_PLANES)"  # draw_gen.rs:334
        g = L.CullInfo()
        g.view_matrix.set(self.view_matrix)
        for i, p in enumerate(planes):
            for k in range(4):
                g.cull_planes[i][k] = float(p[k])
        g.cull_plane_count = len(planes)
        g.alpha_mode_flags = int(self.alpha_mode_filter)
        oc = self.occlusion_culling
        g.occlusion_pass = oc.pass_index()
        # descriptor indices in the reference; here only "present or not" matters (pointers travel in SceneBuffers)
        g.visibility_buffer = 0 if oc.visibility_buffer is not None else L.NO_BUFFER
        g.meshlet_visibility_buffer = 0 if oc.meshlet_visibility_buffer is not None else L.NO_BUFFER
        g.depth_pyramid = 0 if oc.depth_pyramid is not None else L.NO_BUFFER
        g.min_mesh_lod = int(self.lod_range[0])
        g.max_mesh_lod = int(self.lod_range[1]) - 1
        g.lod_base = float(self.lod_base)
        g.lod_step = float(self.lod_step)
        for k in range(3):
            g.lod_target_pos_view_space[k] = float(self.lod_target_pos_view_space[k])
        g.projection_type = 0 if self.projection.kind == "perspective" else 1
        if oc.kind == "write":
            g.noskip_alpha_mode = int(oc.noskip_alphamode)
            f32 = np.float32
            if self.projection.kind == "perspective":
                f = f32(1.0) / np.tan(f32(0.5) * f32(self.projection.fov), dtype=np.float32)
                g.p00_or_width_recip_x2 = float(f32(f) / f32(oc.aspect_ratio))
                g.p11_or_height_recip_x2 = float(f32(f))
                g.z_near = float(self.projection.near_clip)
            else:
                width = f32(self.projection.half_width) * f32(2.0)
                height = f32(width * (f32(1.0) / f32(oc.aspect_ratio)))
                g.p00_or_width_recip_x2 = float((f32(1.0) / width) * f32(2.0))
                g.p11_or_height_recip_x2 = float((f32(1.0) / height) * f32(2.0))
                g.z_near = float(self.projection.near_clip)
                g.z_far = float(self.projection.far_clip)
        return g


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _stream(context=None):
    """torch's current stream ON THE CONTEXT'S DEVICE (the thread's current device may be another one)."""
    return C.c_void_p(torch.cuda.current_stream(context.device if context is not None else None).cuda_stream)


class Context:
    """Stands in for graphics::Context as far as this path needs it: owns the orbit_ctx (scan scratch, status
    words) and the cache of transient output buffers keyed by name (context.rs:1275-1334)."""

    def __init__(self, device=0):
        if not torch.cuda.is_available():
            raise RuntimeError("orbit_b200 needs a CUDA device (no CPU fallback)")
        self.device = torch.device("cuda", device)     # the caller's current device is left alone: the C ABI switches per call
        self._h = C.c_void_p()
        _lib.check(_lib.lib().orbit_ctx_create(device, C.byref(self._h)), "orbit_ctx_create")
        self._transients = {}

    def close(self):
        if self._h:
            _lib.lib().orbit_ctx_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def create_transient(self, name, nbytes):
        t = self._transients.get(name)
        if t is None or t.numel() < nbytes:
            # zero-filled once at creation: the stages read ahead of the device-side counts (orbit_cuda.h, conventions) and
            # never use what they find there, but tools like compute-sanitizer initcheck would flag the loads
            t = torch.zeros(int(nbytes), dtype=torch.uint8, device=self.device)
            self._transients[name] = t
        return t

    def upload(self, array):
        a = np.ascontiguousarray(array)
        return torch.from_numpy(a.view(np.uint8).reshape(-1)).to(self.device)

    def poll_status(self):
        st = L.Status()
        code = _lib.lib().orbit_ctx_poll_status(self._h, C.byref(st))
        return code, st

    @property
    def launch_count(self):
        return int(_lib.lib().orbit_ctx_launch_count(self._h))


@dataclass
class AssetGraphData:
    """Device buffers owned by GpuAssets (assets/mod.rs:230-239)."""
    mesh_info_buffer: torch.Tensor
    meshlet_buffer: torch.Tensor
    materials_buffer: torch.Tensor


@dataclass
class SceneGraphData:
    """Device buffers owned by SceneData (scene.rs:358-369)."""
    entity_draw_count: int
    entity_draw_buffer: torch.Tensor
    entity_buffer: torch.Tensor
    meshlet_visibility_buffer: Optional[torch.Tensor] = None
    light_count: int = 0
    light_data_buffer: Optional[torch.Tensor] = None
    # sharding of one view across GPUs (SURVEY §8e): sub-range of entity draws handled by this process
    draw_begin: int = 0
    draw_end: int = 0
    record_capacity: int = 0     # dispatch records the scene can produce (sum of ceil(lod0/32)); 0 = reference cap
    draw_capacity: int = 0       # meshlet instances (worst-case draws); 0 = reference cap


def _scene_buffers(assets, scene, cull):
    sb = L.SceneBuffers()
    sb.entity_draws = scene.entity_draw_buffer.data_ptr()
    sb.mesh_infos = assets.mesh_info_buffer.data_ptr()
    sb.entities = scene.entity_buffer.data_ptr()
    sb.meshlets = assets.meshlet_buffer.data_ptr()
    sb.materials = assets.materials_buffer.data_ptr()
    oc = cull.occlusion_culling
    sb.entity_visibility = oc.visibility_buffer.data_ptr() if oc.visibility_buffer is not None else 0
    sb.meshlet_visibility = oc.meshlet_visibility_buffer.data_ptr() if oc.meshlet_visibility_buffer is not None else 0
    sb.entity_draw_count = int(scene.entity_draw_count)
    sb.draw_begin, sb.draw_end = int(scene.draw_begin), int(scene.draw_end)
    return sb


class DepthImage:
    """A depth buffer held in a 2-D single-channel float32 CUDA array (orbit_depth_image_wrap): the form a depth attachment
    imported from Vulkan takes (cudaExternalMemoryGetMappedMipmappedArray, level 0). `cuda_array` is the cudaArray_t as an
    integer; the array stays the caller's and must outlive this object and every enqueued or captured call that reads it.
    DepthPyramid.update, compute_clusters and the frame classes take one wherever they take a depth tensor."""

    def __init__(self, context, cuda_array):
        self.context = context
        self._h = C.c_void_p()
        _lib.check(_lib.lib().orbit_depth_image_wrap(context._h, C.c_void_p(int(cuda_array)), C.byref(self._h)), "orbit_depth_image_wrap")
        self.cuda_array = int(cuda_array)
        w, h = C.c_uint32(), C.c_uint32()
        _lib.check(_lib.lib().orbit_depth_image_size(self._h, C.byref(w), C.byref(h)), "orbit_depth_image_size")
        self.size = (w.value, h.value)

    def close(self):
        if self._h:
            _lib.lib().orbit_depth_image_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class ClusterGridImage:
    """The cluster offset/count grid held in a 3-D CUDA array with two 32-bit unsigned channels and surface load/store
    (orbit_cluster_grid_wrap): the form the reference's R32G32_UINT cluster image takes when imported from Vulkan.
    `cuda_array` is the cudaArray_t as an integer; the array stays the caller's and must outlive this object and every
    enqueued or captured call that writes it. compute_clusters(..., light_offset_image=grid) writes the grid into it."""

    def __init__(self, context, cuda_array):
        self.context = context
        self._h = C.c_void_p()
        _lib.check(_lib.lib().orbit_cluster_grid_wrap(context._h, C.c_void_p(int(cuda_array)), C.byref(self._h)), "orbit_cluster_grid_wrap")
        self.cuda_array = int(cuda_array)

    def close(self):
        if self._h:
            _lib.lib().orbit_cluster_grid_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class DepthPyramid:
    """draw_gen.rs:451-567. One linear f32 allocation holding all mips back to back. With `image` (a cudaMipmappedArray_t
    as an integer, e.g. mapped from the renderer's imported pyramid VkImage) every build also stores level l into level l of
    that array (orbit_hiz_attach_image); the linear texels stay what the culling stages read."""

    def __init__(self, context, name, size, image=None):
        self.context, self.name = context, name
        self._h = C.c_void_p()
        self.usable = False
        self.texels = None
        self.size = None
        self.image = int(image) if image is not None else None
        self._make(size)

    new = classmethod(lambda cls, context, name, size, image=None: cls(context, name, size, image))

    def _attach(self):
        if self.image is not None:
            _lib.check(_lib.lib().orbit_hiz_attach_image(self.context._h, self._h, C.c_void_p(self.image)), "orbit_hiz_attach_image")

    def _make(self, size):
        w, h = int(size[0]), int(size[1])
        info = L.HizInfo()
        _lib.check(_lib.lib().orbit_hiz_geometry(w, h, C.byref(info)), "orbit_hiz_geometry")
        self.info = info
        self.texels = torch.zeros(info.total_texels, dtype=torch.float32, device=self.context.device)
        if self._h:
            _lib.lib().orbit_hiz_destroy(self._h)
            self._h = C.c_void_p()
        _lib.check(_lib.lib().orbit_hiz_wrap(self.context._h, w, h, _ptr(self.texels), C.byref(self._h)), "orbit_hiz_wrap")
        self.size = (w, h)
        self.usable = False
        self._attach()

    def resize(self, size, image=None):
        """A mirrored pyramid needs `image`: the array for the new size (the old one no longer fits)."""
        if (int(size[0]), int(size[1])) != self.size:
            if self.image is not None and image is None:
                raise ValueError("DepthPyramid.resize: the pyramid has an image; pass the array for the new size")
            if image is not None:
                self.image = int(image)
            self._make(size)

    def attach_image(self, image):
        """Mirrors every later build into `image` (a cudaMipmappedArray_t as an integer; see the class comment)."""
        if self.image is not None:
            raise ValueError("DepthPyramid.attach_image: the pyramid already has an image")
        self.image = int(image)
        try:
            self._attach()
        except Exception:
            self.image = None
            raise

    def rebind_external(self, device_ptr):
        """Moves the pyramid onto caller-owned device memory of info.total_texels floats (orbit_hiz_wrap): peer-shareable
        memory for the sharded view (multi_gpu.PyramidBroadcast), or an imported Vulkan allocation. Contents start undefined."""
        class _Mem:     # torch.as_tensor understands __cuda_array_interface__
            def __init__(self, ptr, n):
                self.__cuda_array_interface__ = {"shape": (n,), "typestr": "<f4", "data": (int(ptr), False), "version": 2}
        w, h = self.size
        self._external = _Mem(device_ptr, int(self.info.total_texels))
        self.texels = torch.as_tensor(self._external, device=self.context.device)
        if self._h:
            _lib.lib().orbit_hiz_destroy(self._h)
            self._h = C.c_void_p()
        _lib.check(_lib.lib().orbit_hiz_wrap(self.context._h, w, h, C.c_void_p(int(device_ptr)), C.byref(self._h)), "orbit_hiz_wrap")
        self.usable = False
        self._attach()

    def update(self, depth_buffer):
        """depth_buffer: float32 device tensor [H, W] (reverse-Z), or a DepthImage of the same size."""
        if isinstance(depth_buffer, DepthImage):
            assert depth_buffer.size == self.size
            _lib.check(_lib.lib().orbit_hiz_build_image(self.context._h, self._h, depth_buffer._h, _stream(self.context)),
                       "orbit_hiz_build_image")
            self.usable = True
            return
        h, w = depth_buffer.shape
        assert (w, h) == self.size and depth_buffer.dtype == torch.float32 and depth_buffer.is_contiguous()
        _lib.check(_lib.lib().orbit_hiz_build(self.context._h, self._h, _ptr(depth_buffer), w, h, _stream(self.context)), "orbit_hiz_build")
        self.usable = True

    def get_current(self):
        return self

    def level(self, l):
        w, h = max(self.info.width >> l, 1), max(self.info.height >> l, 1)
        o = self.info.level_offset[l]
        return self.texels[o:o + w * h].view(h, w)

    def __del__(self):
        try:
            if self._h:
                _lib.lib().orbit_hiz_destroy(self._h)
        except Exception:
            pass


def create_meshlet_dispatch_command(context, name, assets, scene, cull_info):
    """draw_gen.rs:327-380: returns (cull_info_gpu, meshlet_dispatch_buffer)."""
    assert len(cull_info.view_space_cull_planes) <= L.MAX_CULL_PLANES
    cap = int(scene.record_capacity) or MAX_MESHLET_DISPATCH_COUNT
    buf = context.create_transient(name + "_meshlet_dispatch_buffer", L.DISPATCH_HEADER + 16 * cap)
    g = cull_info.to_gpu()
    sb = _scene_buffers(assets, scene, cull_info)
    pyr = cull_info.occlusion_culling.depth_pyramid
    _lib.check(_lib.lib().orbit_entity_cull(context._h, C.byref(g), C.byref(sb), pyr._h if pyr is not None else None,
                                            _ptr(buf), cap, _stream(context)), "orbit_entity_cull")
    return g, buf


def create_meshlet_draw_commands(context, name, assets, scene, cull_info, meshlet_dispatch_buffer, task_payloads=None):
    """draw_gen.rs:382-435: returns meshlet_draw_command_buffer."""
    assert len(cull_info.view_space_cull_planes) <= L.MAX_CULL_PLANES
    rcap = int(scene.record_capacity) or MAX_MESHLET_DISPATCH_COUNT
    dcap = int(scene.draw_capacity) or MAX_DRAW_COUNT
    buf = context.create_transient(name + "_meshlet_draw_command_buffer", L.DRAW_HEADER + 28 * dcap)
    g = cull_info.to_gpu()
    sb = _scene_buffers(assets, scene, cull_info)
    pyr = cull_info.occlusion_culling.depth_pyramid
    _lib.check(_lib.lib().orbit_meshlet_cull(context._h, C.byref(g), C.byref(sb), pyr._h if pyr is not None else None,
                                             _ptr(meshlet_dispatch_buffer), rcap, _ptr(buf), dcap,
                                             _ptr(task_payloads), _stream(context)), "orbit_meshlet_cull")
    return buf


@dataclass
class ClusterSettings:
    """cluster.rs:15-72. tile_size_px overrides 2**px_size_power when set (BASELINE C4 uses 120 px tiles)."""
    px_size_power: int = 3
    screen_resolution: tuple = (0, 0)
    z_slice_count: int = 32
    far_plane: float = 200.0
    luminance_cutoff: float = 0.25
    tile_size_px: Optional[int] = None

    def tile_px_size(self):
        return self.tile_size_px if self.tile_size_px else 2 ** self.px_size_power

    def set_resolution(self, res):
        self.screen_resolution = (int(res[0]), int(res[1]))

    def tile_counts(self):
        t = self.tile_px_size()
        return [-(-n // t) for n in self.screen_resolution]

    def cluster_counts(self):
        tc = self.tile_counts()
        return [tc[0], tc[1], self.z_slice_count]

    def linear_cluster_count(self):
        c = self.cluster_counts()
        return c[0] * c[1] * c[2]

    def cluster_grid_info(self, near):
        from .scenes import cluster_grid_info
        return cluster_grid_info(near, self.far_plane, self.z_slice_count)


@dataclass
class GraphClusterInfo:
    """cluster.rs:352-366"""
    light_offset_image: object            # uint8 tensor view of uint2[cz][cy][cx], or the ClusterGridImage it was written to
    light_index_buffer: torch.Tensor      # ClusterLightIndices
    tile_depth_slice_mask: torch.Tensor
    cluster_depth_bounds: torch.Tensor
    unique_cluster_buffer: torch.Tensor
    tile_counts: tuple
    z_slice_count: int
    z_scale: float
    z_bias: float
    tile_size_px: int


def compute_clusters(context, settings, view_matrix, projection_matrix, near, depth_buffer, scene, name="clusters",
                     light_offset_image=None):
    """cluster.rs:368-397 = mark_active_clusters + compact_active_clusters + cluster_light_assignment.
    view_matrix / projection_matrix: 4x4 math convention (Camera in the reference).
    depth_buffer: float32 device tensor [H, W], or a DepthImage.
    light_offset_image: a ClusterGridImage of extent cluster_counts() to write the offset/count grid into (orbit_light_cluster
    _image_grid) instead of a buffer; needs a DepthImage depth. The returned info's light_offset_image is then that object."""
    image = isinstance(depth_buffer, DepthImage)
    if light_offset_image is not None and not image:
        raise TypeError("compute_clusters: light_offset_image needs a DepthImage depth buffer")
    w, h = depth_buffer.size if image else (depth_buffer.shape[1], depth_buffer.shape[0])
    assert (w, h) == tuple(settings.screen_resolution)
    cx, cy, cz = settings.cluster_counts()
    n = cx * cy * cz
    p = L.ClusterParams()
    p.info.world_to_view_matrix.set(view_matrix)
    p.info.screen_to_view_matrix.set(np.linalg.inv(np.asarray(projection_matrix, np.float64)))
    p.info.cluster_count[0], p.info.cluster_count[1], p.info.cluster_count[2] = cx, cy, cz
    p.info.tile_size_px = settings.tile_px_size()
    p.info.screen_size[0], p.info.screen_size[1] = w, h
    p.info.z_near, p.info.z_far = float(near), float(settings.far_plane)
    p.info.global_light_count = int(scene.light_count)
    p.z_scale, p.z_bias = settings.cluster_grid_info(near)
    masks = context.create_transient(name + "_tile_depth_slice_mask", 4 * cx * cy)
    bounds = context.create_transient(name + "_cluster_depth_bounds", 8 * n)
    unique = context.create_transient(name + "_unique_cluster_buffer", 16 + 4 * n)
    cap = L.MAX_LIGHTS_PER_CLUSTER * n          # MAX_LIGHT_INDEX_COUNT in the reference is a fixed constant
    index = context.create_transient(name + "_light_index_buffer", 4 + 4 * cap)
    if light_offset_image is not None:
        offsets = light_offset_image
        _lib.check(_lib.lib().orbit_light_cluster_image_grid(context._h, C.byref(p), depth_buffer._h, _ptr(scene.light_data_buffer),
                                                             _ptr(masks), _ptr(bounds), _ptr(unique), light_offset_image._h, _ptr(index),
                                                             cap, _stream(context)), "orbit_light_cluster_image_grid")
    else:
        offsets = context.create_transient(name + "_cluster_offset_image", 8 * n)
        fn, name_ = ((_lib.lib().orbit_light_cluster_image, "orbit_light_cluster_image") if image
                     else (_lib.lib().orbit_light_cluster, "orbit_light_cluster"))
        _lib.check(fn(context._h, C.byref(p), depth_buffer._h if image else _ptr(depth_buffer), _ptr(scene.light_data_buffer),
                      _ptr(masks), _ptr(bounds), _ptr(unique), _ptr(offsets), _ptr(index), cap, _stream(context)), name_)
    return GraphClusterInfo(offsets, index, masks, bounds, unique, (cx, cy), cz, p.z_scale, p.z_bias, settings.tile_px_size()), p
