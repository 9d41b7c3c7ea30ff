"""GPU parity of the batched pass-0 views (orbit_entity_cull_views / orbit_meshlet_cull_views, orbit_cuda.h): one entity kernel,
one test kernel and one emit kernel for up to 16 views must leave in every view's buffers, byte for byte, what
orbit_entity_cull + orbit_meshlet_cull (and the oracle's cull_pass) leave for that view alone: dispatch header + records, draw
count + commands, task payloads. Cases: the shadow cascades of C4 (reduced scale against the oracle, full size against separate
calls), 16 C5 cameras with an empty view, a view without planes and per-view alpha filters, a multi-LOD scene with per-view LOD
parameters, one view, task payloads for some views, overflow in one view, CUDA-graph replay interleaved with single-view calls,
a draw sub-range, and every refusal of the contract."""
import ctypes as C

import numpy as np
import pytest
import torch

from orbit_b200 import scenes

pytestmark = pytest.mark.gpu


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _batched(ctx, ds, infos, rcap, dcap, tag, payloads=None):
    """orbit_entity_cull_views + orbit_meshlet_cull_views over `infos` (CullInfo objects); returns [(dispatch, draws, payload)]."""
    from orbit_b200 import _lib, layouts as L
    from orbit_b200.passes import _scene_buffers
    lib, n, mk = _lib.lib(), len(infos), ctx.create_transient
    gs = (L.CullInfo * n)(*[ci.to_gpu() for ci in infos])
    bufs = [(mk("%s%d_d" % (tag, v), L.DISPATCH_HEADER + 16 * rcap), mk("%s%d_w" % (tag, v), L.DRAW_HEADER + 28 * dcap),
             mk("%s%d_p" % (tag, v), 44 * rcap) if payloads and payloads[v] else None) for v in range(n)]
    ptrs = lambda k: (C.c_void_p * n)(*[b[k].data_ptr() if b[k] is not None else None for b in bufs])
    sb = _scene_buffers(ds.assets, ds.scene, infos[0])
    assert lib.orbit_entity_cull_views(ctx._h, gs, n, C.byref(sb), ptrs(0), rcap, _stream()) == 0
    assert lib.orbit_meshlet_cull_views(ctx._h, gs, n, C.byref(sb), ptrs(0), rcap, ptrs(1), dcap, ptrs(2) if payloads else None, _stream()) == 0
    return bufs


def _single(ctx, ds, info, rcap, dcap, tag, payload=False):
    """orbit_entity_cull + orbit_meshlet_cull for one view, same capacities."""
    from orbit_b200 import _lib, layouts as L
    from orbit_b200.passes import _scene_buffers
    lib, mk = _lib.lib(), ctx.create_transient
    g = info.to_gpu()
    d, w = mk(tag + "_d", L.DISPATCH_HEADER + 16 * rcap), mk(tag + "_w", L.DRAW_HEADER + 28 * dcap)
    pay = mk(tag + "_p", 44 * rcap) if payload else None
    sb = _scene_buffers(ds.assets, ds.scene, info)
    assert lib.orbit_entity_cull(ctx._h, C.byref(g), C.byref(sb), None, _p(d), rcap, _stream()) == 0
    assert lib.orbit_meshlet_cull(ctx._h, C.byref(g), C.byref(sb), None, _p(d), rcap, _p(w), dcap, _p(pay), _stream()) == 0
    return d, w, pay


def _bytes(buf):
    return buf.cpu().numpy() if isinstance(buf, torch.Tensor) else buf


def _same(a, b, rcap, dcap, what):
    """Dispatch header + the records kept, draw count + the commands kept, byte for byte; returns (records, draws)."""
    da, db = _bytes(a[0]), _bytes(b[0])
    n = int(da[:4].view(np.uint32)[0])
    assert np.array_equal(da[:12], db[:12]), (what, "dispatch header", da[:12].view(np.uint32), db[:12].view(np.uint32))
    assert np.array_equal(da[12:12 + 16 * min(n, rcap)], db[12:12 + 16 * min(n, rcap)]), (what, "records")
    wa, wb = _bytes(a[1]), _bytes(b[1])
    m = int(wa[:4].view(np.uint32)[0])
    assert m == int(wb[:4].view(np.uint32)[0]), (what, "draw count", m, int(wb[:4].view(np.uint32)[0]))
    assert np.array_equal(wa[4:4 + 28 * min(m, dcap)], wb[4:4 + 28 * min(m, dcap)]), (what, "draws")
    return n, m


def _none(view, **kw):
    from orbit_b200 import frame
    from orbit_b200.passes import OcclusionCullInfo
    return frame.cull_info_for(view, OcclusionCullInfo("none"), **kw)


def _caps(ds):
    return int(ds.scene.record_capacity), int(ds.scene.draw_capacity)


def test_cascades_follow_the_oracle_in_three_launches(gpu_context, oracle):
    """The four cascades of ShadowRenderer::render_cascaded_shadow (6-11 planes each, LOD range 2.. for cascades 2-3) over a
    reduced C4 scene, through frame.cull_views: three launches, every buffer equal to the oracle's cull_pass of that view."""
    from orbit_b200 import frame
    ctx = gpu_context
    sc, view = scenes.config_c4(scale=0.03)
    casc = scenes.cascade_views(view)
    ds = frame.DeviceScene.upload(ctx, sc)
    hs = oracle.HostScene(sc)
    infos = [_none(cv) for cv in casc]
    frame.cull_views(ctx, ds, infos, name="casc_warm"); torch.cuda.synchronize()
    before = ctx.launch_count
    out = frame.cull_views(ctx, ds, infos, name="casc")
    assert ctx.launch_count - before == 3
    torch.cuda.synchronize()
    rcap, dcap = _caps(ds)
    seen = [_same(g, oracle.cull_pass(hs, ci.to_gpu()), rcap, dcap, ("cascade", v)) for v, (g, ci) in enumerate(zip(out, infos))]
    assert all(m > 0 for _, m in seen), seen


def test_cascades_at_full_size_match_separate_calls(gpu_context):
    """Full-size C4 (10 M meshlets): the batched cascades against four separate orbit_entity_cull + orbit_meshlet_cull calls."""
    from orbit_b200 import frame
    ctx = gpu_context
    sc, view = scenes.config_c4()
    ds = frame.DeviceScene.upload(ctx, sc)
    infos = [_none(cv) for cv in scenes.cascade_views(view)]
    rcap, dcap = _caps(ds)
    out = _batched(ctx, ds, infos, rcap, dcap, "cfull")
    ref = [_single(ctx, ds, ci, rcap, dcap, "cfull_s%d" % v) for v, ci in enumerate(infos)]
    torch.cuda.synchronize()
    seen = [_same(a, b, rcap, dcap, ("full cascade", v)) for v, (a, b) in enumerate(zip(out, ref))]
    assert all(m > 0 for _, m in seen), seen


def test_sixteen_cameras_with_an_empty_view_no_planes_and_alpha_filters(gpu_context, oracle):
    """16 C5 cameras in one call: one looks at the sky (empty lists), one has no cull planes, every view its own alpha filter."""
    from orbit_b200 import frame
    ctx = gpu_context
    sc, views = scenes.config_c5(scale=0.01, n_views=16)
    views[3] = scenes.perspective_view((0.0, 1.0e4, 0.0), (0.0, 1.0, 0.0), 1920, 1080, up=(0.0, 0.0, 1.0))
    infos = [_none(v, frustum_culling=(i != 5)) for i, v in enumerate(views)]
    for i, ci in enumerate(infos):
        ci.alpha_mode_filter = [0b011, 0b001, 0b010, 0b111, 0b000][i % 5]
    assert infos[5].to_gpu().cull_plane_count == 0
    ds = frame.DeviceScene.upload(ctx, sc)
    hs = oracle.HostScene(sc)
    out = frame.cull_views(ctx, ds, infos, name="c5v")
    torch.cuda.synchronize()
    rcap, dcap = _caps(ds)
    seen = [_same(g, oracle.cull_pass(hs, ci.to_gpu()), rcap, dcap, ("camera", v)) for v, (g, ci) in enumerate(zip(out, infos))]
    assert seen[3] == (0, 0)
    assert sum(1 for n, m in seen if m > 0) >= 8, seen


def test_multi_lod_scene_with_per_view_lod_parameters(gpu_context, oracle):
    """A three-LOD lattice seen by 16 cameras with their own LOD base, step, range and target: the records (LOD choice) of
    every view equal the oracle's."""
    from orbit_b200 import frame
    ctx = gpu_context
    sc, view = scenes.config_c1(scale=0.3, lods=(100, 40, 12))
    rng = np.random.default_rng(20261020)
    lo, hi = np.asarray(sc.aabb_min, np.float64), np.asarray(sc.aabb_max, np.float64)
    infos = []
    for i in range(16):
        eye = lo + (hi - lo) * rng.uniform(0.0, 1.0, 3)
        d = rng.normal(size=3); d /= np.linalg.norm(d)
        v = scenes.perspective_view(tuple(eye), tuple(d), 1280, 720, fov_deg=float(rng.uniform(50.0, 100.0)))
        v.lod_base = float(rng.choice([2.0, 8.0, 30.0]))
        v.lod_step = float(rng.choice([1.5, 2.0, 3.0]))
        v.lod_range = [(0, 8), (1, 8), (2, 8), (0, 1), (1, 2)][i % 5]
        v.lod_target_view = tuple(float(x) for x in rng.uniform(-5.0, 5.0, 3))
        infos.append(_none(v))
    ds = frame.DeviceScene.upload(ctx, sc)
    hs = oracle.HostScene(sc)
    out = frame.cull_views(ctx, ds, infos, name="lodv")
    torch.cuda.synchronize()
    rcap, dcap = _caps(ds)
    for v, (g, ci) in enumerate(zip(out, infos)):
        _same(g, oracle.cull_pass(hs, ci.to_gpu()), rcap, dcap, ("lod view", v))


def test_one_view_equals_the_single_view_calls(gpu_context):
    from orbit_b200 import frame
    ctx = gpu_context
    sc, view = scenes.config_c2(scale=0.05)
    ds = frame.DeviceScene.upload(ctx, sc)
    info = _none(view)
    g = frame.cull_views(ctx, ds, [info], name="one")[0]
    ref = frame.cull_pass(ctx, "one_ref", ds, info)
    torch.cuda.synchronize()
    rcap, dcap = _caps(ds)
    assert _same(g, ref, rcap, dcap, "one view")[1] > 0


def test_task_payloads_for_some_views(gpu_context, oracle):
    from orbit_b200 import frame
    ctx = gpu_context
    sc, views = scenes.config_c5(scale=0.01, n_views=6)
    infos = [_none(v) for v in views]
    flags = [True, False, True, True, False, True]
    ds = frame.DeviceScene.upload(ctx, sc)
    hs = oracle.HostScene(sc)
    out = frame.cull_views(ctx, ds, infos, name="payv", task_payloads=flags)
    torch.cuda.synchronize()
    rcap, dcap = _caps(ds)
    for v, (g, ci) in enumerate(zip(out, infos)):
        assert len(g) == (3 if flags[v] else 2)
        o = oracle.cull_pass(hs, ci.to_gpu(), task_payloads=True)
        n, _ = _same(g, o, rcap, dcap, ("payload view", v))
        if flags[v]:
            assert np.array_equal(g[2][:44 * n].cpu().numpy(), o[2][:44 * n]), ("payloads", v)


def test_overflow_in_one_view_only(gpu_context):
    """A record capacity, then a draw capacity, between the longest and the second-longest list: the long view's header stays
    exact and its excess is dropped as in the single-view calls, the status flag is set, the other views are complete."""
    from orbit_b200 import frame
    ctx = gpu_context
    sc, view = scenes.config_c4(scale=0.03)
    ds = frame.DeviceScene.upload(ctx, sc)
    infos = [_none(cv) for cv in scenes.cascade_views(view)]
    rcap, dcap = _caps(ds)
    full = _batched(ctx, ds, infos, rcap, dcap, "ovf_full")
    torch.cuda.synchronize()
    counts = [_same(g, g, rcap, dcap, "self") for g in full]
    ctx.poll_status()
    for k, flag in ((0, "dispatch_overflow"), (1, "draw_overflow")):
        lens = [c[k] for c in counts]
        big = int(np.argmax(lens))
        second = max(x for v, x in enumerate(lens) if v != big)
        assert lens[big] > second + 1, counts
        cap = (lens[big] + second) // 2
        r2, d2 = (cap, dcap) if k == 0 else (rcap, cap)
        out = _batched(ctx, ds, infos, r2, d2, "ovf%d" % k)
        torch.cuda.synchronize()
        code, st = ctx.poll_status()
        assert code == -5 and getattr(st, flag) == 1, flag
        ref = [_single(ctx, ds, ci, r2, d2, "ovf%d_s%d" % (k, v)) for v, ci in enumerate(infos)]
        torch.cuda.synchronize()
        ctx.poll_status()
        for v in range(len(infos)):
            got = _same(out[v], ref[v], r2, d2, (flag, v))
            assert got[k] == counts[v][k], (flag, v)                           # the header is exact
            if v != big:
                _same(out[v], full[v], rcap, dcap, (flag, "unaffected", v))


def test_graph_replay_interleaved_with_single_view_calls(gpu_context):
    """Batched calls and single-view calls on one context and stream, interleaved, captured once into a CUDA graph and replayed
    over frames whose entity matrices move; after every replay each list equals separate single-view calls made afterwards."""
    from orbit_b200 import frame
    ctx = gpu_context
    sc, views = scenes.config_c5(scale=0.02, n_views=6)
    ds = frame.DeviceScene.upload(ctx, sc)
    rcap, dcap = _caps(ds)
    infos = [_none(v) for v in views]

    def work():
        from orbit_b200 import _lib, layouts as L
        from orbit_b200.passes import _scene_buffers
        lib, mk = _lib.lib(), ctx.create_transient
        n = 4
        gs = (L.CullInfo * n)(*[ci.to_gpu() for ci in infos[:4]])
        bufs = [(mk("gr%d_d" % v, L.DISPATCH_HEADER + 16 * rcap), mk("gr%d_w" % v, L.DRAW_HEADER + 28 * dcap)) for v in range(n)]
        sb = _scene_buffers(ds.assets, ds.scene, infos[0])
        ptrs = lambda k: (C.c_void_p * n)(*[b[k].data_ptr() for b in bufs])
        g4 = infos[4].to_gpu()
        d4, w4 = mk("gr4_d", L.DISPATCH_HEADER + 16 * rcap), mk("gr4_w", L.DRAW_HEADER + 28 * dcap)
        w4b = mk("gr4_wb", L.DRAW_HEADER + 28 * dcap)
        s = _stream()
        assert lib.orbit_entity_cull_views(ctx._h, gs, n, C.byref(sb), ptrs(0), rcap, s) == 0
        assert lib.orbit_entity_cull(ctx._h, C.byref(g4), C.byref(sb), None, _p(d4), rcap, s) == 0
        assert lib.orbit_meshlet_cull(ctx._h, C.byref(g4), C.byref(sb), None, _p(d4), rcap, _p(w4), dcap, None, s) == 0
        assert lib.orbit_meshlet_cull_views(ctx._h, gs, n, C.byref(sb), ptrs(0), rcap, ptrs(1), dcap, None, s) == 0
        assert lib.orbit_meshlet_cull(ctx._h, C.byref(g4), C.byref(sb), None, _p(d4), rcap, _p(w4b), dcap, None, s) == 0
        return bufs + [(d4, w4), (d4, w4b)]

    outs = work(); torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        outs = work()
    ents = ds.scene.entity_buffer.view(torch.float32).view(-1, 32)
    for f in range(3):
        ents[f::5, 12] += 3.0                      # x translation of every fifth entity (model matrix column 3)
        ents[f::7, 14] -= 2.0
        graph.replay()
        torch.cuda.synchronize()
        got = [(o[0].cpu().numpy().copy(), o[1].cpu().numpy().copy()) for o in outs]
        ref = [_single(ctx, ds, ci, rcap, dcap, "gr_ref%d" % v) for v, ci in enumerate(infos[:5])]
        torch.cuda.synchronize()
        for v in range(4):
            _same(got[v], ref[v], rcap, dcap, (f, "batched", v))
        _same(got[4], ref[4], rcap, dcap, (f, "single"))
        _same(got[5], ref[4], rcap, dcap, (f, "single again"))


def test_draw_sub_range(gpu_context):
    from orbit_b200 import frame
    ctx = gpu_context
    sc, view = scenes.config_c4(scale=0.03)
    infos = [_none(cv) for cv in scenes.cascade_views(view)]
    n = sc.n_entities
    ds = frame.DeviceScene.upload(ctx, sc, draw_begin=32 * (n // 96), draw_end=2 * n // 3)
    out = frame.cull_views(ctx, ds, infos, name="rng")
    ref = [frame.cull_pass(ctx, "rng_ref%d" % v, ds, ci) for v, ci in enumerate(infos)]
    torch.cuda.synchronize()
    rcap, dcap = _caps(ds)
    seen = [_same(a, b, rcap, dcap, ("range", v)) for v, (a, b) in enumerate(zip(out, ref))]
    assert any(m > 0 for _, m in seen)


def test_refusals_launch_nothing(gpu_context):
    from orbit_b200 import _lib, frame, layouts as L
    from orbit_b200.passes import _scene_buffers
    ctx, lib = gpu_context, _lib.lib()
    sc, view = scenes.config_c4(scale=0.01)
    casc = scenes.cascade_views(view)
    ds = frame.DeviceScene.upload(ctx, sc)
    rcap, dcap = _caps(ds)
    mk = ctx.create_transient
    infos = [_none(cv) for cv in casc]
    sb = _scene_buffers(ds.assets, ds.scene, infos[0])
    d = [mk("ref_d%d" % v, L.DISPATCH_HEADER + 16 * rcap) for v in range(17)]
    w = [mk("ref_w%d" % v, L.DRAW_HEADER + 28 * dcap) for v in range(17)]
    INVALID = _lib.ERR_INVALID_ARGUMENT

    def call(gs, n, dp, wp, scene=sb, pay=None):
        arr = lambda ps: (C.c_void_p * max(len(ps), 1))(*ps)
        before = ctx.launch_count
        a = lib.orbit_entity_cull_views(ctx._h, gs, n, C.byref(scene), arr(dp), rcap, _stream())
        b = lib.orbit_meshlet_cull_views(ctx._h, gs, n, C.byref(scene), arr(dp), rcap, arr(wp), dcap, pay, _stream())
        assert ctx.launch_count == before
        return a, b

    def gpu(n, edit=None):
        gs = (L.CullInfo * max(n, 1))(*[infos[v % 4].to_gpu() for v in range(max(n, 1))])
        if edit:
            edit(gs)
        return gs

    ptr = lambda ts, off=0: [t.data_ptr() + off for t in ts]
    cases = {
        "zero views": (gpu(0), 0, ptr(d[:1]), ptr(w[:1])),
        "17 views": (gpu(17), 17, ptr(d), ptr(w)),
        "pass 1": (gpu(4, lambda g: setattr(g[2], "occlusion_pass", 1)), 4, ptr(d[:4]), ptr(w[:4])),
        "mixed projection": (gpu(4, lambda g: setattr(g[1], "projection_type", L.PROJ_PERSPECTIVE)), 4, ptr(d[:4]), ptr(w[:4])),
        "13 planes": (gpu(4, lambda g: setattr(g[3], "cull_plane_count", 13)), 4, ptr(d[:4]), ptr(w[:4])),
        "NULL buffer": (gpu(4), 4, ptr(d[:3]) + [None], ptr(w[:3]) + [None]),
        "misaligned": (gpu(4), 4, ptr(d[:3]) + ptr(d[3:4], 2), ptr(w[:3]) + ptr(w[3:4], 2)),
        "shared buffer": (gpu(4), 4, ptr(d[:3]) + ptr(d[:1]), ptr(w[:3]) + ptr(w[:1])),
    }
    for what, (gs, n, dp, wp) in cases.items():
        assert call(gs, n, dp, wp) == (INVALID, INVALID), what
    # a draw buffer shared by two views (dispatch buffers distinct): the meshlet stage refuses
    before = ctx.launch_count
    arr = lambda ps: (C.c_void_p * len(ps))(*ps)
    assert lib.orbit_meshlet_cull_views(ctx._h, gpu(4), 4, C.byref(sb), arr(ptr(d[:4])), rcap, arr(ptr(w[:3]) + ptr(w[:1])), dcap, None,
                                        _stream()) == INVALID
    # what check_cull refuses for the single-view calls: a draw range that does not start on a multiple of 32, no meshlets
    bad = L.SceneBuffers.from_buffer_copy(sb); bad.draw_begin = 5
    assert lib.orbit_entity_cull_views(ctx._h, gpu(4), 4, C.byref(bad), arr(ptr(d[:4])), rcap, _stream()) == INVALID
    bad = L.SceneBuffers.from_buffer_copy(sb); bad.meshlets = 0
    assert lib.orbit_meshlet_cull_views(ctx._h, gpu(4), 4, C.byref(bad), arr(ptr(d[:4])), rcap, arr(ptr(w[:4])), dcap, None, _stream()) == INVALID
    assert ctx.launch_count == before
