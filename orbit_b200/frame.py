"""The caller protocol of the culling passes, as ForwardRenderer / ShadowRenderer drive them.

    ForwardRenderer::render_depth_prepass   src/passes/forward.rs:213-430
        EARLY (pass 1, VisibilityRead) -> Hi-Z update -> LATE (pass 2, VisibilityWrite)
    ForwardRenderer::render                 src/passes/forward.rs:518-548   MAIN (pass 1 again, updated bits)
    ShadowRenderer::render_shadow_map       src/passes/shadow_renderer.rs:391-403,693-707   pass 0, orthographic

The reference rasterises between the passes; here the depth buffer that feeds the Hi-Z build is an input
(bench / tests generate it procedurally, a real host would share its depth attachment through
cudaImportExternalMemory).
"""
from dataclasses import dataclass
from typing import Optional

import numpy as np
import torch

from . import layouts as L
from .passes import (AssetGraphData, Context, CullInfo, DepthImage, DepthPyramid, OcclusionCullInfo, Projection, SceneGraphData,
                     _stream, create_meshlet_dispatch_command, create_meshlet_draw_commands)


@dataclass
class DeviceScene:
    assets: AssetGraphData
    scene: SceneGraphData
    n_visibility_words: int
    n_entities: int

    @staticmethod
    def upload(context: Context, s, draw_begin=0, draw_end=0, lights=None):
        assets = AssetGraphData(context.upload(s.mesh_infos), context.upload(s.meshlets), context.upload(s.materials))
        scene = SceneGraphData(entity_draw_count=s.n_entities, entity_draw_buffer=context.upload(s.entity_draws),
                               entity_buffer=context.upload(s.entities), draw_begin=draw_begin, draw_end=draw_end,
                               record_capacity=s.n_records_lod0, draw_capacity=s.n_meshlet_instances)
        if lights is not None:
            scene.light_count = len(lights)
            scene.light_data_buffer = context.upload(lights)
        return DeviceScene(assets, scene, s.n_visibility_words, s.n_entities)


class ViewState:
    """Cross-frame state of one view: the two visibility bitmasks (forward.rs:104-106,150-157; scene.rs:364) and
    the depth pyramid. The reference never clears the bitmasks; the harness defines frame 0 as all zeros."""

    def __init__(self, context, dscene, size, name="view", pyramid_image=None):
        """pyramid_image: a cudaMipmappedArray_t (integer) the pyramid is mirrored into on every build (DepthPyramid)."""
        self.entity_visibility = torch.zeros((dscene.n_entities + 31) // 32 + 1, dtype=torch.int32, device=context.device)
        self.meshlet_visibility = torch.zeros(max(dscene.n_visibility_words, 1), dtype=torch.int32, device=context.device)
        self.depth_pyramid = DepthPyramid(context, name + "_depth_pyramid", size, image=pyramid_image)


def projection_of(view):
    if view.projection_type == L.PROJ_PERSPECTIVE:
        return Projection.perspective(view.fov, view.near)
    return Projection.orthographic(view.half_width, view.near, view.far)


def cull_info_for(view, occlusion: OcclusionCullInfo, frustum_culling=True):
    return CullInfo(view_matrix=view.view, view_space_cull_planes=view.planes if frustum_culling else [],
                    projection=projection_of(view), occlusion_culling=occlusion,
                    lod_range=view.lod_range, lod_base=view.lod_base, lod_step=view.lod_step,
                    lod_target_pos_view_space=view.lod_target_view)


def cull_pass(context, name, dscene, cull_info, task_payloads=None):
    """create_meshlet_dispatch_command + create_meshlet_draw_commands for one CullInfo."""
    _, dispatch = create_meshlet_dispatch_command(context, name, dscene.assets, dscene.scene, cull_info)
    draws = create_meshlet_draw_commands(context, name, dscene.assets, dscene.scene, cull_info, dispatch, task_payloads)
    return dispatch, draws


def depth_prepass_culling(context, dscene, vstate, view, depth_buffer, meshlet_occlusion=True, name="forward_depth_prepass"):
    """EARLY -> Hi-Z -> LATE (forward.rs:266-403). Returns {(stage): (dispatch_buffer, draw_buffer)}."""
    mvis = vstate.meshlet_visibility if meshlet_occlusion else None
    early = cull_info_for(view, OcclusionCullInfo("read", vstate.entity_visibility, mvis))
    out = {"early": cull_pass(context, "early_" + name, dscene, early)}
    vstate.depth_pyramid.update(depth_buffer)
    late = cull_info_for(view, OcclusionCullInfo("write", vstate.entity_visibility, mvis, vstate.depth_pyramid,
                                                 noskip_alphamode=0, aspect_ratio=view.aspect))
    out["late"] = cull_pass(context, "late_" + name, dscene, late)
    return out


def main_pass_culling(context, dscene, vstate, view, meshlet_occlusion=True, name="forward"):
    """MAIN pass (forward.rs:518-548): pass 1 with the bits the late pass just wrote."""
    mvis = vstate.meshlet_visibility if meshlet_occlusion else None
    info = cull_info_for(view, OcclusionCullInfo("read", vstate.entity_visibility, mvis))
    return cull_pass(context, name, dscene, info)


def late_and_main_culling(context, dscene, vstate, view, meshlet_occlusion=True, name="forward_depth_prepass", main_name="forward"):
    """LATE + MAIN in their fused form (orbit_entity_cull_late_main / orbit_meshlet_cull_late_main): byte for byte the buffers of
    the LATE half of depth_prepass_culling followed by main_pass_culling, from one entity kernel and one test kernel. Expects the
    pyramid to be up to date. Raises if the two CullInfos are not a compatible pair (see orbit_cuda.h)."""
    import ctypes as C
    from . import _lib
    from .passes import _ptr, _scene_buffers, _stream
    mvis = vstate.meshlet_visibility if meshlet_occlusion else None
    late = cull_info_for(view, OcclusionCullInfo("write", vstate.entity_visibility, mvis, vstate.depth_pyramid,
                                                 noskip_alphamode=0, aspect_ratio=view.aspect))
    main = cull_info_for(view, OcclusionCullInfo("read", vstate.entity_visibility, mvis))
    gl, gm = late.to_gpu(), main.to_gpu()
    lib = _lib.lib()
    if not lib.orbit_cull_pair_compatible(C.byref(gl), C.byref(gm)):
        raise ValueError("LATE and MAIN CullInfos are not a compatible pair: call the passes separately")
    sc = dscene.scene
    rcap, dcap = int(sc.record_capacity) or 1_000_000, int(sc.draw_capacity) or 1_000_000
    mk = context.create_transient
    out = {}
    for k, n in (("late", "late_" + name), ("main", main_name)):
        out[k] = (mk(n + "_meshlet_dispatch_buffer", L.DISPATCH_HEADER + 16 * rcap), mk(n + "_meshlet_draw_command_buffer", L.DRAW_HEADER + 28 * dcap))
    sb = _scene_buffers(dscene.assets, sc, late)
    _lib.check(lib.orbit_entity_cull_late_main(context._h, C.byref(gl), C.byref(gm), C.byref(sb), vstate.depth_pyramid._h,
                                               _ptr(out["late"][0]), _ptr(out["main"][0]), rcap, _stream(context)), "orbit_entity_cull_late_main")
    _lib.check(lib.orbit_meshlet_cull_late_main(context._h, C.byref(gl), C.byref(gm), C.byref(sb), vstate.depth_pyramid._h,
                                                _ptr(out["late"][0]), rcap, _ptr(out["late"][1]), _ptr(out["main"][1]), dcap, None, None,
                                                _stream(context)), "orbit_meshlet_cull_late_main")
    return out


def cull_views(context, dscene, cull_infos, name="views", task_payloads=None):
    """Pass-0 culling of several views of one scene (the cascades of ShadowRenderer::render_cascaded_shadow,
    shadow_renderer.rs:466-712, or many cameras) through orbit_entity_cull_views / orbit_meshlet_cull_views: 3 kernel launches
    per group of up to MAX_BATCH_VIEWS views. Returns one (dispatch_buffer, draw_buffer) pair per CullInfo, byte for byte what
    cull_pass returns for it. `task_payloads`: None, or one flag per view (a payload buffer is returned as a third element of
    the views whose flag is set). Every view must be pass 0 with the same projection type."""
    import ctypes as C
    from . import _lib
    from .passes import _scene_buffers, _stream
    lib = _lib.lib()
    sc = dscene.scene
    rcap, dcap = int(sc.record_capacity) or 1_000_000, int(sc.draw_capacity) or 1_000_000
    mk = context.create_transient
    infos = list(cull_infos)
    want = list(task_payloads) if task_payloads is not None else [False] * len(infos)
    out = []
    for g0 in range(0, len(infos), L.MAX_BATCH_VIEWS):
        group = infos[g0:g0 + L.MAX_BATCH_VIEWS]
        n = len(group)
        gs = (L.CullInfo * n)(*[ci.to_gpu() for ci in group])
        bufs = []
        for v in range(g0, g0 + n):
            tag = "%s%d" % (name, v)
            pay = mk(tag + "_task_payloads", 44 * rcap) if want[v] else None
            bufs.append((mk(tag + "_meshlet_dispatch_buffer", L.DISPATCH_HEADER + 16 * rcap),
                         mk(tag + "_meshlet_draw_command_buffer", L.DRAW_HEADER + 28 * dcap), pay))
        ptrs = lambda k: (C.c_void_p * n)(*[b[k].data_ptr() if b[k] is not None else None for b in bufs])
        sb = _scene_buffers(dscene.assets, sc, group[0])
        _lib.check(lib.orbit_entity_cull_views(context._h, gs, n, C.byref(sb), ptrs(0), rcap, _stream(context)), "orbit_entity_cull_views")
        _lib.check(lib.orbit_meshlet_cull_views(context._h, gs, n, C.byref(sb), ptrs(0), rcap, ptrs(1), dcap,
                                                ptrs(2) if any(b[2] is not None for b in bufs) else None, _stream(context)),
                   "orbit_meshlet_cull_views")
        out.extend((d, w) if p is None else (d, w, p) for d, w, p in bufs)
    return out


class _ViewsPass:
    """One batched occlusion pass (EARLY, LATE or MAIN) of up to MAX_BATCH_VIEWS views, every argument packed once:
    orbit_entity_cull_views_occlusion + orbit_meshlet_cull_views_occlusion, 3 launches. `infos`: one CullInfo per view (one
    pass, one projection type); `pyramids`: the views' DepthPyramids (pass 2) or None; `task_payloads`: None or one flag per view."""

    def __init__(self, context, dscene, infos, pyramids, tags, task_payloads=None):
        import ctypes as C
        from . import _lib
        from .passes import _scene_buffers
        self.context, self._lib, self._C = context, _lib.lib(), C
        n = self.n = len(infos)
        sc = dscene.scene
        self.rcap, self.dcap = int(sc.record_capacity) or 1_000_000, int(sc.draw_capacity) or 1_000_000
        mk = context.create_transient
        self.gs = (L.CullInfo * n)(*[ci.to_gpu() for ci in infos])
        self.sbs = (L.SceneBuffers * n)(*[_scene_buffers(dscene.assets, sc, ci) for ci in infos])
        self.hizs = (C.c_void_p * n)(*[p._h.value for p in pyramids]) if pyramids is not None else None
        want = list(task_payloads) if task_payloads is not None else [False] * n
        self.outputs = [(mk(t + "_meshlet_dispatch_buffer", L.DISPATCH_HEADER + 16 * self.rcap),
                         mk(t + "_meshlet_draw_command_buffer", L.DRAW_HEADER + 28 * self.dcap),
                         mk(t + "_task_payloads", 44 * self.rcap) if w else None) for t, w in zip(tags, want)]
        ptrs = lambda k: (C.c_void_p * n)(*[o[k].data_ptr() if o[k] is not None else None for o in self.outputs])
        self.dispatch, self.draws = ptrs(0), ptrs(1)
        self.payloads = ptrs(2) if any(want) else None

    def launch(self, s):
        from . import _lib
        h = self.context._h
        _lib.check(self._lib.orbit_entity_cull_views_occlusion(h, self.gs, self.n, self.sbs, self.hizs, self.dispatch, self.rcap, s),
                   "orbit_entity_cull_views_occlusion")
        _lib.check(self._lib.orbit_meshlet_cull_views_occlusion(h, self.gs, self.n, self.sbs, self.hizs, self.dispatch, self.rcap,
                                                                self.draws, self.dcap, self.payloads, s), "orbit_meshlet_cull_views_occlusion")

    def results(self):
        return [(d, w) if p is None else (d, w, p) for d, w, p in self.outputs]


class _HizViews:
    """orbit_hiz_build_views for the pyramids of up to MAX_BATCH_VIEWS views (one depth buffer each, all of one size), or
    orbit_hiz_build_views_image when the depth buffers are DepthImages."""

    def __init__(self, context, pyramids, depth_buffers):
        import ctypes as C
        from . import _lib
        self.context, self._lib, self.pyramids = context, _lib.lib(), list(pyramids)
        n = self.n = len(self.pyramids)
        self.depths = list(depth_buffers)
        self.hizs = (C.c_void_p * n)(*[p._h.value for p in self.pyramids])
        self.image = all(isinstance(d, DepthImage) for d in self.depths)
        if self.image:
            assert len({d.size for d in self.depths}) == 1, "every depth image of a batch has the same size"
            self.dptrs = (C.c_void_p * n)(*[d._h.value for d in self.depths])
            return
        shapes = {tuple(d.shape) for d in depth_buffers}
        assert len(shapes) == 1, "every depth buffer of a batch has the same size"
        self.h, self.w = shapes.pop()
        assert all(d.dtype == torch.float32 and d.is_contiguous() for d in depth_buffers)
        self.dptrs = (C.c_void_p * n)(*[d.data_ptr() for d in self.depths])

    def launch(self, s):
        from . import _lib
        if self.image:
            _lib.check(self._lib.orbit_hiz_build_views_image(self.context._h, self.hizs, self.dptrs, self.n, s), "orbit_hiz_build_views_image")
        else:
            _lib.check(self._lib.orbit_hiz_build_views(self.context._h, self.hizs, self.dptrs, self.n, self.w, self.h, s), "orbit_hiz_build_views")
        for p in self.pyramids:
            p.usable = True


def _groups(n):
    return [range(g0, min(g0 + L.MAX_BATCH_VIEWS, n)) for g0 in range(0, n, L.MAX_BATCH_VIEWS)]


def _early_info(vstate, view, meshlet_occlusion):
    return cull_info_for(view, OcclusionCullInfo("read", vstate.entity_visibility, vstate.meshlet_visibility if meshlet_occlusion else None))


def _late_info(vstate, view, meshlet_occlusion):
    mvis = vstate.meshlet_visibility if meshlet_occlusion else None
    return cull_info_for(view, OcclusionCullInfo("write", vstate.entity_visibility, mvis, vstate.depth_pyramid, noskip_alphamode=0,
                                                 aspect_ratio=view.aspect))


def depth_prepass_views(context, dscene, vstates, views, depth_buffers, meshlet_occlusion=True, name="forward_depth_prepass"):
    """depth_prepass_culling for several cameras over one scene: EARLY, Hi-Z and LATE of every group of up to MAX_BATCH_VIEWS
    cameras in 3 + 1 + 3 launches (orbit_*_cull_views_occlusion, orbit_hiz_build_views). `vstates`, `views`, `depth_buffers`:
    one per camera (one projection type, depth buffers of one size). Returns one {"early": .., "late": ..} per camera, each
    (dispatch_buffer, draw_buffer), byte for byte what depth_prepass_culling returns for that camera alone."""
    s = _stream(context)
    out = []
    for g in _groups(len(views)):
        early = _ViewsPass(context, dscene, [_early_info(vstates[v], views[v], meshlet_occlusion) for v in g], None,
                           ["early_%s%d" % (name, v) for v in g])
        early.launch(s)
        _HizViews(context, [vstates[v].depth_pyramid for v in g], [depth_buffers[v] for v in g]).launch(s)
        late = _ViewsPass(context, dscene, [_late_info(vstates[v], views[v], meshlet_occlusion) for v in g],
                          [vstates[v].depth_pyramid for v in g], ["late_%s%d" % (name, v) for v in g])
        late.launch(s)
        out.extend({"early": e, "late": l} for e, l in zip(early.results(), late.results()))
    return out


def main_pass_views(context, dscene, vstates, views, meshlet_occlusion=True, name="forward"):
    """main_pass_culling for several cameras: MAIN (pass 1 over the bits the LATE pass wrote) of every group of up to
    MAX_BATCH_VIEWS cameras in 3 launches. Returns one (dispatch_buffer, draw_buffer) per camera."""
    s = _stream(context)
    out = []
    for g in _groups(len(views)):
        main = _ViewsPass(context, dscene, [_early_info(vstates[v], views[v], meshlet_occlusion) for v in g], None,
                          ["%s%d" % (name, v) for v in g])
        main.launch(s)
        out.extend(main.results())
    return out


class PreparedViews:
    """PreparedFrame for several cameras over one scene: EARLY -> Hi-Z -> LATE (and, with `main_pass`, MAIN) of every camera,
    every argument packed once, 3 + 1 + 3 (+ 3) launches per group of up to MAX_BATCH_VIEWS cameras instead of 7 (10) per
    camera. `capture()` / `replay()` put the whole multi-camera frame into one CUDA graph. `outputs[v]`: camera v's
    {"early", "late"[, "main"]} -> (dispatch_buffer, draw_buffer). `depth_buffers`: tensors, or DepthImages (all of one kind)."""

    def __init__(self, context, dscene, vstates, views, depth_buffers, meshlet_occlusion=True, name="views", main_pass=True):
        self.context = context
        self.stages = []
        self.outputs = [dict() for _ in views]
        for g in _groups(len(views)):
            pyr = [vstates[v].depth_pyramid for v in g]
            early_infos = [_early_info(vstates[v], views[v], meshlet_occlusion) for v in g]
            passes = [("early", _ViewsPass(context, dscene, early_infos, None, ["early_%s%d" % (name, v) for v in g])),
                      ("hiz", _HizViews(context, pyr, [depth_buffers[v] for v in g])),
                      ("late", _ViewsPass(context, dscene, [_late_info(vstates[v], views[v], meshlet_occlusion) for v in g], pyr,
                                          ["late_%s%d" % (name, v) for v in g]))]
            if main_pass:
                passes.append(("main", _ViewsPass(context, dscene, early_infos, None, ["main_%s%d" % (name, v) for v in g])))
            for k, st in passes:
                if k != "hiz":
                    for v, r in zip(g, st.results()):
                        self.outputs[v][k] = r
            self.stages.extend(st for _, st in passes)
        self.graph = None

    def launch(self):
        s = _stream(self.context)
        for st in self.stages:
            st.launch(s)

    def capture(self):
        self.launch()  # warm: scratch growth / occupancy queries must not happen during capture
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            self.launch()
        self.graph = g
        return g

    def replay(self):
        self.graph.replay()


def shadow_pass_culling(context, dscene, view, name="shadow"):
    """One cascade (shadow_renderer.rs:693-707): pass 0, no occlusion."""
    return cull_pass(context, name, dscene, cull_info_for(view, OcclusionCullInfo("none")))


def read_dispatch(buf):
    """Device MeshletDispatchBuffer -> (count, records ndarray)."""
    hdr = buf[:12].cpu().numpy().view(np.uint32)
    n = int(hdr[0])
    recs = buf[12:12 + 16 * n].cpu().numpy().view(L.dispatch_dtype)
    return hdr.copy(), recs


def read_draws(buf, capacity=None):
    n = int(buf[:4].cpu().numpy().view(np.uint32)[0])
    m = n if capacity is None else min(n, capacity)
    return n, buf[4:4 + 28 * m].cpu().numpy().view(L.draw_command_dtype)


class PreparedFrame:
    """One view's culling for a frame with every argument packed once: the depth prepass EARLY -> Hi-Z -> LATE
    (forward.rs:266-403) and, with `main_pass`, the MAIN pass after it (forward.rs:518-548: pass 1 again, reading the
    visibility bits the late pass just wrote — the same CullInfo as EARLY, other output buffers).

    The reference re-declares the passes each frame on its render graph; the packed form is the CUDA analogue:
    asynchronous stage calls on one stream, optionally captured into a CUDA graph (`capture()` / `replay()`) so
    a frame costs one graph launch. Safe to replay: the scan epoch and tickets live in device memory.

    `depth_buffer` is a float32 device tensor [H, W] or a DepthImage; with an image, hiz() and hiz_entity_late() (so launch())
    call the *_image entry points, which write the same bytes."""

    def __init__(self, context, dscene, vstate, view, depth_buffer, meshlet_occlusion=True, name="forward_depth_prepass", main_pass=False,
                 fuse_late_main=True):
        import ctypes as C
        from . import _lib
        from .passes import _ptr, _scene_buffers
        self.image = isinstance(depth_buffer, DepthImage)
        self.context, self.dscene, self.vstate, self.view, self.depth = context, dscene, vstate, view, depth_buffer
        self._lib, self._C, self._ptr = _lib.lib(), C, _ptr
        mvis = vstate.meshlet_visibility if meshlet_occlusion else None
        early = cull_info_for(view, OcclusionCullInfo("read", vstate.entity_visibility, mvis))
        late = cull_info_for(view, OcclusionCullInfo("write", vstate.entity_visibility, mvis, vstate.depth_pyramid,
                                                     noskip_alphamode=0, aspect_ratio=view.aspect))
        self.g_early, self.g_late = early.to_gpu(), late.to_gpu()
        self.sb_early = _scene_buffers(dscene.assets, dscene.scene, early)
        self.sb_late = _scene_buffers(dscene.assets, dscene.scene, late)
        sc = dscene.scene
        self.rcap = int(sc.record_capacity) or 1_000_000
        self.dcap = int(sc.draw_capacity) or 1_000_000
        mk = context.create_transient
        self.early_dispatch = mk("early_" + name + "_meshlet_dispatch_buffer", L.DISPATCH_HEADER + 16 * self.rcap)
        self.early_draws = mk("early_" + name + "_meshlet_draw_command_buffer", L.DRAW_HEADER + 28 * self.dcap)
        self.late_dispatch = mk("late_" + name + "_meshlet_dispatch_buffer", L.DISPATCH_HEADER + 16 * self.rcap)
        self.late_draws = mk("late_" + name + "_meshlet_draw_command_buffer", L.DRAW_HEADER + 28 * self.dcap)
        self.main_pass = main_pass
        self.main_dispatch = self.main_draws = None
        if main_pass:
            self.main_dispatch = mk("main_" + name + "_meshlet_dispatch_buffer", L.DISPATCH_HEADER + 16 * self.rcap)
            self.main_draws = mk("main_" + name + "_meshlet_draw_command_buffer", L.DRAW_HEADER + 28 * self.dcap)
        # LATE + MAIN fused (one entity kernel, one test kernel, an emit kernel per list) whenever the pair allows it
        self.fused = bool(main_pass and fuse_late_main and self._lib.orbit_cull_pair_compatible(C.byref(self.g_late), C.byref(self.g_early)))
        self.graph = None
        if self.image:
            self._hw = depth_buffer.size
            self._hiz_build, self._hiz_entity_late = self._lib.orbit_hiz_build_image, self._lib.orbit_hiz_build_image_entity_cull_late
        else:
            h, w = depth_buffer.shape
            self._hw = (w, h)
            self._hiz_build, self._hiz_entity_late = self._lib.orbit_hiz_build, self._lib.orbit_hiz_build_entity_cull_late

    def _stream(self):
        return self._C.c_void_p(torch.cuda.current_stream(self.context.device).cuda_stream)

    def _depth_args(self):
        """The depth arguments of the build calls chosen at construction: (image) or (depth, width, height)."""
        return (self.depth._h,) if self.image else (self._ptr(self.depth), self._hw[0], self._hw[1])

    def entity(self, late, s=None):
        C, lib, p = self._C, self._lib, self._ptr
        s = s or self._stream()
        if late == "main":
            late, g, sb, out = False, self.g_early, self.sb_early, self.main_dispatch
        else:
            g, sb, out = (self.g_late, self.sb_late, self.late_dispatch) if late else (self.g_early, self.sb_early, self.early_dispatch)
        rc = lib.orbit_entity_cull(self.context._h, C.byref(g), C.byref(sb), self.vstate.depth_pyramid._h if late else None,
                                   p(out), self.rcap, s)
        if rc:
            raise RuntimeError("orbit_entity_cull: %d" % rc)

    def meshlet(self, late, s=None, context=None):
        """`context`: run the stage on another Context's scratch (bench.py times the test kernel alone that way)."""
        C, lib, p = self._C, self._lib, self._ptr
        s = s or self._stream()
        if late == "main":
            late, g, sb, disp, out = False, self.g_early, self.sb_early, self.main_dispatch, self.main_draws
        else:
            g, sb, disp, out = ((self.g_late, self.sb_late, self.late_dispatch, self.late_draws) if late
                                else (self.g_early, self.sb_early, self.early_dispatch, self.early_draws))
        rc = lib.orbit_meshlet_cull((context or self.context)._h, C.byref(g), C.byref(sb), self.vstate.depth_pyramid._h if late else None,
                                    p(disp), self.rcap, p(out), self.dcap, None, s)
        if rc:
            raise RuntimeError("orbit_meshlet_cull: %d" % rc)

    def entity_late_main(self, s=None):
        C, lib, p = self._C, self._lib, self._ptr
        rc = lib.orbit_entity_cull_late_main(self.context._h, C.byref(self.g_late), C.byref(self.g_early), C.byref(self.sb_late),
                                             self.vstate.depth_pyramid._h, p(self.late_dispatch), p(self.main_dispatch), self.rcap, s or self._stream())
        if rc:
            raise RuntimeError("orbit_entity_cull_late_main: %d" % rc)

    def meshlet_late_main(self, s=None, context=None):
        C, lib, p = self._C, self._lib, self._ptr
        rc = lib.orbit_meshlet_cull_late_main((context or self.context)._h, C.byref(self.g_late), C.byref(self.g_early), C.byref(self.sb_late),
                                              self.vstate.depth_pyramid._h, p(self.late_dispatch), self.rcap, p(self.late_draws), p(self.main_draws),
                                              self.dcap, None, None, s or self._stream())
        if rc:
            raise RuntimeError("orbit_meshlet_cull_late_main: %d" % rc)

    def meshlet_test(self, late, record_masks, s=None):
        """The test half of the meshlet stage (orbit_meshlet_test): visibility words + one 16-byte entry per dispatch record into
        `record_masks`; used by the sharded view, whose draw commands are emitted on the rank that submits them."""
        C, lib, p = self._C, self._lib, self._ptr
        s = s or self._stream()
        g, sb, disp = (self.g_late, self.sb_late, self.late_dispatch) if late else (self.g_early, self.sb_early, self.early_dispatch)
        rc = lib.orbit_meshlet_test(self.context._h, C.byref(g), C.byref(sb), self.vstate.depth_pyramid._h if late else None,
                                    p(disp), self.rcap, p(record_masks), s)
        if rc:
            raise RuntimeError("orbit_meshlet_test: %d" % rc)

    def hiz(self, s=None):
        s = s or self._stream()
        rc = self._hiz_build(self.context._h, self.vstate.depth_pyramid._h, *self._depth_args(), s)
        if rc:
            raise RuntimeError("%s: %d" % (self._hiz_build.__name__, rc))

    def hiz_entity_late(self, s=None):
        """hiz() followed by entity(True) — with a fused frame, by entity_late_main() — as ONE call
        (orbit_hiz_build_entity_cull_late): the same buffers, but the entity kernel's work that does not read the pyramid runs
        under the build."""
        C, lib, p = self._C, self._lib, self._ptr
        g_main, main_dispatch = (C.byref(self.g_early), p(self.main_dispatch)) if self.fused else (None, None)
        rc = self._hiz_entity_late(self.context._h, self.vstate.depth_pyramid._h, *self._depth_args(),
                                   C.byref(self.g_late), g_main, C.byref(self.sb_late), p(self.late_dispatch), main_dispatch,
                                   self.rcap, s or self._stream())
        if rc:
            raise RuntimeError("%s: %d" % (self._hiz_entity_late.__name__, rc))

    def launch(self, overlap_main_entity=False):
        """The frame's stage calls in dependency order. `overlap_main_entity`: the MAIN pass's entity stage depends only on the
        entity visibility bits the LATE entity stage wrote, not on the late MESHLET stage, so it may be forked onto a side stream
        beside the late meshlet test (the entity and meshlet stages use disjoint context scratch: orbit_cuda.h, "Threading").
        Measured on C2 (profiles/r2_frame_timeline.txt): the entity kernel is hidden, but the late test kernel — persistent CTAs
        with a static tile split — ends 7 us later when 40 SMs start a third of their CTAs late, so the frame gains nothing
        (104.5 vs 104.2 us); off by default, kept because it is bit-identical and pays off when the late pass is small."""
        s = self._stream()
        self.entity(False, s); self.meshlet(False, s)
        self.hiz_entity_late(s)
        if self.fused:
            self.meshlet_late_main(s)
            return
        if not self.main_pass:
            self.meshlet(True, s)
            return
        if not overlap_main_entity:
            self.meshlet(True, s); self.entity("main", s); self.meshlet("main", s)
            return
        main = torch.cuda.current_stream(self.context.device)
        if getattr(self, "_side", None) is None:
            self._side = torch.cuda.Stream(device=self.context.device, priority=-1)   # high priority: its 40 CTAs must get their SM
            # slots before the persistent CTAs of the late meshlet test fill every SM (kernel-node priority is captured with the stream's)
        fork = torch.cuda.Event(); fork.record(main)
        self._side.wait_event(fork)
        self.entity("main", self._C.c_void_p(self._side.cuda_stream))
        join = torch.cuda.Event(); join.record(self._side)
        self.meshlet(True, s)
        main.wait_event(join)
        self.meshlet("main", s)

    def capture(self):
        self.launch()  # warm: scratch growth / occupancy queries must not happen during capture
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            self.launch()
        self.graph = g
        return g

    def replay(self):
        self.graph.replay()


def host_frame_loop(context, prepared, scene_datas, h_transforms, h_depth, h_counts, h_early_draws, h_late_draws, h_main_draws, steps,
                    lookahead=2, depth_resident=False):
    """End-to-end frame loop with HOST inputs/outputs run by the compiled host driver (orbit_b200/host/frame_driver.cpp):
    per step, pinned-host Transforms + depth -> device (`depth_resident`: the depth buffer stays on the device, as with
    Vulkan interop), orbit_scene_update, the stage calls of EARLY / Hi-Z / LATE / MAIN, the three survivor lists -> pinned host; `lookahead` steps in flight ahead of the one being read back, rotating over `prepared`
    (PreparedFrame) / `scene_datas` (scene.SceneData) copies. Returns the driver's report."""
    import ctypes as C
    from . import _lib
    n = len(prepared)
    assert not any(pf.image for pf in prepared), "the host frame driver reads depth from a linear buffer"
    frames = (L.HostFrame * n)()
    for f, pf, sd in zip(frames, prepared, scene_datas):
        sd.update_scene(pf.dscene.assets)       # packs sd._packed (and keeps the ranges allocated)
        f.update = sd._packed
        f.cull_early, f.cull_late, f.scene_early, f.scene_late = pf.g_early, pf.g_late, pf.sb_early, pf.sb_late
        f.hiz = pf.vstate.depth_pyramid._h.value
        f.depth = pf.depth.data_ptr()
        f.early_dispatch, f.early_draws = pf.early_dispatch.data_ptr(), pf.early_draws.data_ptr()
        f.late_dispatch, f.late_draws = pf.late_dispatch.data_ptr(), pf.late_draws.data_ptr()
        f.main_dispatch, f.main_draws = pf.main_dispatch.data_ptr(), pf.main_draws.data_ptr()
        f.capacity_records, f.capacity_draws = pf.rcap, pf.dcap
        f.width, f.height = pf._hw
    torch.cuda.synchronize()
    io = L.HostFrameIO()
    io.h_transforms, io.h_depth, io.h_counts = h_transforms.data_ptr(), h_depth.data_ptr(), h_counts.data_ptr()
    io.h_early_draws, io.h_late_draws, io.h_main_draws = h_early_draws.data_ptr(), h_late_draws.data_ptr(), h_main_draws.data_ptr()
    io.depth_resident = 1 if depth_resident else 0
    _lib.check(_lib.host_lib().orbit_host_frame_loop(context._h, frames, n, C.byref(io), int(steps), int(lookahead)), "orbit_host_frame_loop")
    return {"ms_per_step": io.ms_per_step, "h2d_bytes_per_step": int(io.h2d_bytes_per_step), "d2h_bytes_per_step": int(io.d2h_bytes_last_step)}
