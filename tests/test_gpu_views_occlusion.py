"""GPU parity of the batched two-pass occlusion cameras (orbit_hiz_build_views, orbit_entity_cull_views_occlusion,
orbit_meshlet_cull_views_occlusion; orbit_cuda.h): EARLY, Hi-Z, LATE and MAIN of up to 16 cameras in one launch per kernel must
leave in every camera's buffers, byte for byte, what the single-view calls (and the oracle) leave for that camera alone: dispatch
header + records, draw count + commands, task payloads, both visibility bitmasks and every pyramid texel. Cases: reduced C5
cameras over three frames against the oracle (10 launches per frame), full-size C2 against separate calls, 16 cameras with an
empty view, a view without planes, per-view alpha filters and LOD parameters, an orthographic batch, a batch without meshlet
occlusion, task payloads for some views, overflow in one view, CUDA-graph replay of PreparedViews interleaved with single-view
and pass-0 batched calls, a draw sub-range, warps whose tiles cross a view boundary (the Hi-Z ring flush), the batched pyramid
build at three sizes, and every refusal of the contract."""
import ctypes as C

import numpy as np
import pytest
import torch

from orbit_b200 import scenes

pytestmark = pytest.mark.gpu


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _np(t):
    return t.cpu().numpy() if isinstance(t, torch.Tensor) else t


def _u32(t):
    return np.ascontiguousarray(_np(t)).view(np.uint32)


def _same(a, b, rcap, dcap, what):
    """Dispatch header + the records kept, draw count + the commands kept, byte for byte; returns (records, draws)."""
    da, db = _np(a[0]), _np(b[0])
    n = int(da[:4].view(np.uint32)[0])
    assert np.array_equal(da[:12], db[:12]), (what, "dispatch header", da[:12].view(np.uint32), db[:12].view(np.uint32))
    assert np.array_equal(da[12:12 + 16 * min(n, rcap)], db[12:12 + 16 * min(n, rcap)]), (what, "records")
    wa, wb = _np(a[1]), _np(b[1])
    m = int(wa[:4].view(np.uint32)[0])
    assert m == int(wb[:4].view(np.uint32)[0]), (what, "draw count", m, int(wb[:4].view(np.uint32)[0]))
    assert np.array_equal(wa[4:4 + 28 * min(m, dcap)], wb[4:4 + 28 * min(m, dcap)]), (what, "draws")
    return n, m


def _caps(ds):
    return int(ds.scene.record_capacity), int(ds.scene.draw_capacity)


def _info(vs, view, kind, mocc=True, alpha=None, frustum=True):
    from orbit_b200 import frame
    from orbit_b200.passes import OcclusionCullInfo
    mvis = vs.meshlet_visibility if mocc else None
    if kind == "write":
        oc = OcclusionCullInfo("write", vs.entity_visibility, mvis, vs.depth_pyramid, noskip_alphamode=0, aspect_ratio=view.aspect)
    else:
        oc = OcclusionCullInfo("read", vs.entity_visibility, mvis)
    ci = frame.cull_info_for(view, oc, frustum_culling=frustum)
    if alpha is not None:
        ci.alpha_mode_filter = alpha
    return ci


class _Cams:
    """Cameras over one scene, each with a batched ViewState and a single-view twin; one frame = EARLY, Hi-Z, LATE, MAIN."""

    def __init__(self, ctx, ds, views, depths, tag, mocc=True, alphas=None, frustum=None, payloads=None):
        from orbit_b200 import frame
        self.ctx, self.ds, self.views, self.tag, self.mocc = ctx, ds, views, tag, mocc
        self.depths = [d if isinstance(d, torch.Tensor) else torch.from_numpy(d).to(ctx.device) for d in depths]
        n = len(views)
        self.alphas = alphas or [None] * n
        self.frustum = frustum or [True] * n
        self.payloads = payloads
        self.vb = [frame.ViewState(ctx, ds, (v.width, v.height), name="%s_b%d" % (tag, i)) for i, v in enumerate(views)]
        self.vs = [frame.ViewState(ctx, ds, (v.width, v.height), name="%s_s%d" % (tag, i)) for i, v in enumerate(views)]

    def infos(self, states, kind):
        return [_info(s, v, kind, self.mocc, a, f) for s, v, a, f in zip(states, self.views, self.alphas, self.frustum)]

    def batched(self):
        from orbit_b200 import frame
        s, n, out = _stream(), len(self.views), {}
        early = frame._ViewsPass(self.ctx, self.ds, self.infos(self.vb, "read"), None, ["%s_e%d" % (self.tag, v) for v in range(n)], self.payloads)
        early.launch(s)
        frame._HizViews(self.ctx, [b.depth_pyramid for b in self.vb], self.depths).launch(s)
        late = frame._ViewsPass(self.ctx, self.ds, self.infos(self.vb, "write"), [b.depth_pyramid for b in self.vb],
                                ["%s_l%d" % (self.tag, v) for v in range(n)], self.payloads)
        late.launch(s)
        main = frame._ViewsPass(self.ctx, self.ds, self.infos(self.vb, "read"), None, ["%s_m%d" % (self.tag, v) for v in range(n)], self.payloads)
        main.launch(s)
        return {"early": early.results(), "late": late.results(), "main": main.results()}

    def single(self):
        from orbit_b200 import frame
        out = {"early": [], "late": [], "main": []}
        pay = self.payloads or [False] * len(self.views)
        rcap = _caps(self.ds)[0]

        def one(k, v, info):
            t = self.ctx.create_transient("%s_s%s%d_p" % (self.tag, k, v), 44 * rcap) if pay[v] else None
            d, w = frame.cull_pass(self.ctx, "%s_s%s%d" % (self.tag, k, v), self.ds, info, task_payloads=t)
            out[k].append((d, w) if t is None else (d, w, t))

        for v, vs in enumerate(self.vs):
            one("early", v, self.infos(self.vs, "read")[v])
            vs.depth_pyramid.update(self.depths[v])
            one("late", v, self.infos(self.vs, "write")[v])
            one("main", v, self.infos(self.vs, "read")[v])
        return out

    def compare(self, got, ref, what, rcap=None, dcap=None):
        r0, d0 = _caps(self.ds)
        rcap, dcap = rcap or r0, dcap or d0
        seen = {}
        for k in ("early", "late", "main"):
            seen[k] = [_same(g, r, rcap, dcap, (what, k, v)) for v, (g, r) in enumerate(zip(got[k], ref[k]))]
        for v, (b, s) in enumerate(zip(self.vb, self.vs)):
            assert np.array_equal(_u32(b.entity_visibility), _u32(s.entity_visibility)), (what, "entity visibility", v)
            assert np.array_equal(_u32(b.meshlet_visibility), _u32(s.meshlet_visibility)), (what, "meshlet visibility", v)
            assert np.array_equal(_u32(b.depth_pyramid.texels), _u32(s.depth_pyramid.texels)), (what, "pyramid", v)
        return seen


def _c5(scale, n_views, ctx):
    from orbit_b200 import frame
    sc, views = scenes.config_c5(scale=scale, n_views=n_views)
    return sc, views, frame.DeviceScene.upload(ctx, sc)


def test_c5_cameras_follow_the_oracle_over_three_frames_in_ten_launches(gpu_context, oracle):
    """4 perspective C5 cameras (reduced scale) over three frames, the cameras moving between frames: EARLY ->
    orbit_hiz_build_views -> LATE -> MAIN through depth_prepass_views / main_pass_views, 1 + 3 x 3 launches per frame, every
    list, visibility bitmask and pyramid texel equal to the oracle's for that camera (one HostScene per camera)."""
    from orbit_b200 import frame
    ctx = gpu_context
    sc, views, ds = _c5(0.01, 4, ctx)
    hss = [oracle.HostScene(sc) for _ in views]
    vss = [frame.ViewState(ctx, ds, (v.width, v.height), name="c5o%d" % i) for i, v in enumerate(views)]
    for f in range(3):
        if f:
            views = [scenes.perspective_view(tuple(np.linalg.inv(v.view)[:3, 3] + np.array([0.7 * f, 0.0, -0.5 * f])),
                                             tuple(-np.linalg.inv(v.view)[:3, 2]), v.width, v.height) for v in views]
        depths = [scenes.make_depth(sc, v) for v in views]
        d_depths = [torch.from_numpy(d).to(ctx.device) for d in depths]
        torch.cuda.synchronize()
        before = ctx.launch_count
        g = frame.depth_prepass_views(ctx, ds, vss, views, d_depths, name="c5o")
        main = frame.main_pass_views(ctx, ds, vss, views, name="c5o_main")
        assert ctx.launch_count - before == 1 + 3 * 3
        torch.cuda.synchronize()
        for v, (view, hs, vs) in enumerate(zip(views, hss, vss)):
            o = oracle.depth_prepass_culling(hs, view, depths[v])
            o["main"] = oracle.main_pass_culling(hs, view)
            rcap, dcap = _caps(ds)
            for k in ("early", "late"):
                _same(g[v][k], o[k], rcap, dcap, (f, v, k))
            _same(main[v], o["main"], rcap, dcap, (f, v, "main"))
            assert np.array_equal(_u32(vs.entity_visibility), hs.entity_visibility), (f, v)
            assert np.array_equal(_u32(vs.meshlet_visibility), hs.meshlet_visibility), (f, v)
            assert np.array_equal(_u32(vs.depth_pyramid.texels), hs.hiz_texels.view(np.uint32)), (f, v)
    assert sum(int(_np(m[1])[:4].view(np.uint32)[0]) > 0 for m in main) >= 2


def test_full_size_c2_four_cameras_match_separate_calls(gpu_context):
    ctx = gpu_context
    from orbit_b200 import frame
    sc, view = scenes.config_c2()
    ds = frame.DeviceScene.upload(ctx, sc)
    eye = np.linalg.inv(view.view)[:3, 3]
    fwd = -np.linalg.inv(view.view)[:3, 2]
    views = [view] + [scenes.perspective_view(tuple(eye + off), tuple(fwd), view.width, view.height)
                      for off in ((4.0, 0.0, 0.0), (-6.0, 1.0, 3.0), (0.0, 3.0, -8.0))]
    cams = _Cams(ctx, ds, views, [scenes.make_depth(sc, v) for v in views], "c2f")
    for f in range(2):
        got = cams.batched(); ref = cams.single()
        torch.cuda.synchronize()
        seen = cams.compare(got, ref, ("c2", f))
        assert all(m > 0 for _, m in seen["main"]), seen


def test_sixteen_cameras_with_an_empty_view_no_planes_alpha_filters_and_lod_parameters(gpu_context):
    """16 C5 cameras: one looks at the sky (empty lists), one has no cull planes, every camera its own alpha filter and LOD
    base / step / range / target; two frames against the single-view calls."""
    ctx = gpu_context
    sc, views, ds = _c5(0.01, 16, ctx)
    views[3] = scenes.perspective_view((0.0, 1.0e4, 0.0), (0.0, 1.0, 0.0), 1920, 1080, up=(0.0, 0.0, 1.0))
    rng = np.random.default_rng(20261020)
    for i, v in enumerate(views):
        v.lod_base = float(rng.choice([2.0, 8.0, 30.0])); v.lod_step = float(rng.choice([1.5, 2.0, 3.0]))
        v.lod_range = [(0, 8), (1, 8), (0, 1)][i % 3]
        v.lod_target_view = tuple(float(x) for x in rng.uniform(-5.0, 5.0, 3))
    depths = [scenes.make_depth(sc, v) for v in views[:4]]
    alphas = [[0b011, 0b001, 0b010, 0b111, 0b000][i % 5] for i in range(16)]
    cams = _Cams(ctx, ds, views, [depths[i % 4] for i in range(16)], "c16", alphas=alphas, frustum=[i != 5 for i in range(16)])
    assert cams.infos(cams.vb, "read")[5].to_gpu().cull_plane_count == 0
    for f in range(2):
        got = cams.batched(); ref = cams.single()
        torch.cuda.synchronize()
        seen = cams.compare(got, ref, ("16 cameras", f))
        assert seen["late"][3] == (0, 0) and seen["main"][3] == (0, 0)
        assert sum(1 for _, m in seen["late"] + seen["main"] if m > 0) >= 8, seen


def test_orthographic_batch(gpu_context):
    ctx = gpu_context
    from orbit_b200 import frame
    sc, view = scenes.config_c4(scale=0.03)
    ds = frame.DeviceScene.upload(ctx, sc)
    views = scenes.cascade_views(view)      # the four orthographic shadow cascades, here with two-pass occlusion
    cams = _Cams(ctx, ds, views, [scenes.make_depth(sc, v) for v in views], "orth")
    for f in range(2):
        got = cams.batched(); ref = cams.single()
        torch.cuda.synchronize()
        seen = cams.compare(got, ref, ("ortho", f))
        assert any(m > 0 for _, m in seen["late"] + seen["main"]), seen


def test_batch_without_meshlet_occlusion(gpu_context):
    ctx = gpu_context
    sc, views, ds = _c5(0.01, 5, ctx)
    cams = _Cams(ctx, ds, views, [scenes.make_depth(sc, v) for v in views], "nomocc", mocc=False)
    for f in range(2):
        got = cams.batched(); ref = cams.single()
        torch.cuda.synchronize()
        seen = cams.compare(got, ref, ("no meshlet occlusion", f))
        assert any(m > 0 for _, m in seen["main"]), seen


def test_task_payloads_for_some_views(gpu_context):
    ctx = gpu_context
    sc, views, ds = _c5(0.01, 4, ctx)
    flags = [True, False, True, False]
    cams = _Cams(ctx, ds, views, [scenes.make_depth(sc, v) for v in views], "pay", payloads=flags)
    for f in range(2):
        got = cams.batched(); ref = cams.single()
        torch.cuda.synchronize()
        seen = cams.compare(got, ref, ("payloads", f))
        for k in ("early", "late", "main"):
            for v in range(4):
                assert len(got[k][v]) == (3 if flags[v] else 2)
                if flags[v]:
                    n = seen[k][v][0]
                    assert np.array_equal(_np(got[k][v][2])[:44 * n], _np(ref[k][v][2])[:44 * n]), (k, v)


def test_overflow_in_one_view_only(gpu_context):
    """A record capacity, then a draw capacity, between the longest and the second-longest EARLY list of the second frame: the
    long view's header stays exact and its excess is dropped as in the single-view calls, the status flag is set, and every
    view's buffers and bitmasks equal the single-view calls with the same capacities."""
    ctx = gpu_context
    sc, views, ds = _c5(0.01, 4, ctx)
    depths = [scenes.make_depth(sc, v) for v in views]
    probe = _Cams(ctx, ds, views, depths, "ovp")
    probe.batched(); probe.single(); torch.cuda.synchronize()
    got = probe.batched(); torch.cuda.synchronize()
    counts = [_same(g, g, *_caps(ds), "self") for g in got["early"]]
    ctx.poll_status()
    for k, flag in ((0, "dispatch_overflow"), (1, "draw_overflow")):
        lens = [c[k] for c in counts]
        big = int(np.argmax(lens))
        second = max(x for v, x in enumerate(lens) if v != big)
        assert lens[big] > second + 1, counts
        cap = (lens[big] + second) // 2
        cams = _Cams(ctx, ds, views, depths, "ov%d" % k)
        cams.batched(); cams.single(); torch.cuda.synchronize(); ctx.poll_status()   # frame 0: every list fits
        scene = ds.scene
        saved = (scene.record_capacity, scene.draw_capacity)
        try:
            if k == 0:
                scene.record_capacity = cap
            else:
                scene.draw_capacity = cap
            got = cams.batched(); torch.cuda.synchronize()
            code, st = ctx.poll_status()
            assert code == -5 and getattr(st, flag) == 1, flag
            ref = cams.single(); torch.cuda.synchronize(); ctx.poll_status()
            r2, d2 = int(scene.record_capacity), int(scene.draw_capacity)
            for v in range(4):
                n = _same(got["early"][v], ref["early"][v], r2, d2, (flag, v))
                assert n[k] == counts[v][k], (flag, v)                          # the header is exact
        finally:
            scene.record_capacity, scene.draw_capacity = saved


def test_prepared_views_graph_replay_interleaved_with_single_view_and_pass0_calls(gpu_context):
    """PreparedViews (4 cameras, EARLY -> Hi-Z -> LATE -> MAIN) captured into one CUDA graph together with a single-view frame and
    a pass-0 batched call on the same context and stream, replayed over frames whose entity matrices move; after every replay
    each camera's lists, bitmasks and pyramid equal a single-view twin run alongside."""
    from orbit_b200 import frame
    from orbit_b200.passes import OcclusionCullInfo
    ctx = gpu_context
    sc, views, ds = _c5(0.02, 6, ctx)
    depths = [torch.from_numpy(scenes.make_depth(sc, v)).to(ctx.device) for v in views[:5]]
    vb = [frame.ViewState(ctx, ds, (v.width, v.height), name="pv_b%d" % i) for i, v in enumerate(views[:4])]
    vsingle = frame.ViewState(ctx, ds, (views[4].width, views[4].height), name="pv_single")
    prep = frame.PreparedViews(ctx, ds, vb, views[:4], depths[:4], name="pv")
    one = frame.PreparedFrame(ctx, ds, vsingle, views[4], depths[4], name="pv_one", main_pass=True)
    p0 = [frame.cull_info_for(views[5], OcclusionCullInfo("none"))]

    def work():
        prep.launch(); one.launch(); out = frame.cull_views(ctx, ds, p0, name="pv_p0")
        return out

    work(); torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        p0_out = work()
    twins = _Cams(ctx, ds, views[:4], depths[:4], "pv_t")
    for b, t in zip(vb, twins.vs):   # the twins start from the state the warm-up frame left
        t.entity_visibility.copy_(b.entity_visibility); t.meshlet_visibility.copy_(b.meshlet_visibility)
    ents = ds.scene.entity_buffer.view(torch.float32).view(-1, 32)
    rcap, dcap = _caps(ds)
    for f in range(3):
        ents[f::5, 12] += 3.0
        ents[f::7, 14] -= 2.0
        graph.replay()
        ref = twins.single()
        torch.cuda.synchronize()
        for k in ("early", "late", "main"):
            for v in range(4):
                _same(prep.outputs[v][k], ref[k][v], rcap, dcap, (f, k, v))
        for v, (b, t) in enumerate(zip(vb, twins.vs)):
            assert np.array_equal(_u32(b.entity_visibility), _u32(t.entity_visibility)), (f, v)
            assert np.array_equal(_u32(b.meshlet_visibility), _u32(t.meshlet_visibility)), (f, v)
            assert np.array_equal(_u32(b.depth_pyramid.texels), _u32(t.depth_pyramid.texels)), (f, v)
        _same(p0_out[0], frame.cull_pass(ctx, "pv_p0_ref", ds, p0[0]), rcap, dcap, (f, "pass 0"))
        torch.cuda.synchronize()


def test_draw_sub_range(gpu_context):
    from orbit_b200 import frame
    ctx = gpu_context
    sc, views = scenes.config_c5(scale=0.01, n_views=6)
    n = sc.n_entities
    ds = frame.DeviceScene.upload(ctx, sc, draw_begin=32 * (n // 96), draw_end=2 * n // 3)
    cams = _Cams(ctx, ds, views, [scenes.make_depth(sc, v) for v in views], "rng")
    drawn = 0
    for f in range(2):
        got = cams.batched(); ref = cams.single()
        torch.cuda.synchronize()
        seen = cams.compare(got, ref, ("range", f))
        drawn += sum(m for _, m in seen["early"] + seen["late"] + seen["main"])
    assert drawn > 0


def test_view_changes_inside_a_warp_flush_the_hiz_ring():
    """The pass-2 test kernel's Hi-Z candidate ring holds one view at a time: a warp whose next tile belongs to the next view
    drains what is queued first (an extra, empty iteration) and restarts the ring at slot 0. With one test CTA per SM
    (ORBIT_MC_CTAS_PER_SM=1, read at context creation) the 8 cameras' LATE lists hold more than twice as many tiles as there are
    warps, so every warp takes several tiles and the warps whose tiles straddle a view boundary go through that flush; every
    list, bitmask and pyramid must still equal the single-view calls."""
    import os
    from orbit_b200.passes import Context
    os.environ["ORBIT_MC_CTAS_PER_SM"] = "1"
    try:
        ctx = Context(0)
    finally:
        del os.environ["ORBIT_MC_CTAS_PER_SM"]
    try:
        sc, views, ds = _c5(0.02, 8, ctx)
        cams = _Cams(ctx, ds, views, [scenes.make_depth(sc, v) for v in views], "flush")
        warps = 8 * torch.cuda.get_device_properties(0).multi_processor_count   # 8 warps per test CTA, one CTA per SM
        late_tiles = []
        for f in range(2):
            got = cams.batched(); ref = cams.single()
            torch.cuda.synchronize()
            seen = cams.compare(got, ref, ("flush", f))
            late_tiles.append(sum((n + 3) // 4 for n, _ in seen["late"]))           # 4 records per tile
        assert max(late_tiles) > 2 * warps, (late_tiles, warps)
    finally:
        ctx.close()


@pytest.mark.parametrize("size", [(1920, 1080), (3840, 2160), (1000, 37)])
def test_hiz_build_views_equals_hiz_build(gpu_context, size):
    from orbit_b200 import _lib
    from orbit_b200.passes import DepthPyramid
    ctx, lib = gpu_context, _lib.lib()
    w, h = size
    g = torch.Generator(device="cpu").manual_seed(w * 7 + h)
    depths = [torch.rand((h, w), generator=g).to(ctx.device) for _ in range(16)]
    for n in (1, 4, 16):
        a = [DepthPyramid(ctx, "hzb%d" % v, (w, h)) for v in range(n)]
        b = [DepthPyramid(ctx, "hzs%d" % v, (w, h)) for v in range(n)]
        before = ctx.launch_count
        assert lib.orbit_hiz_build_views(ctx._h, (C.c_void_p * n)(*[p._h.value for p in a]),
                                         (C.c_void_p * n)(*[d.data_ptr() for d in depths[:n]]), n, w, h, _stream()) == 0
        assert ctx.launch_count - before == 1
        for p, d in zip(b, depths):
            p.update(d)
        torch.cuda.synchronize()
        for v in range(n):
            assert np.array_equal(_u32(a[v].texels), _u32(b[v].texels)), (size, n, v)
        # a second batched build over the same pyramids: the tickets were re-armed
        assert lib.orbit_hiz_build_views(ctx._h, (C.c_void_p * n)(*[p._h.value for p in a]),
                                         (C.c_void_p * n)(*[d.data_ptr() for d in depths[:n][::-1]]), n, w, h, _stream()) == 0
        for p, d in zip(b, depths[:n][::-1]):
            p.update(d)
        torch.cuda.synchronize()
        for v in range(n):
            assert np.array_equal(_u32(a[v].texels), _u32(b[v].texels)), (size, n, v, "again")


def test_refusals_launch_nothing(gpu_context):
    from orbit_b200 import _lib, frame, layouts as L
    from orbit_b200.passes import DepthPyramid, _scene_buffers
    ctx, lib = gpu_context, _lib.lib()
    sc, views, ds = _c5(0.005, 17, ctx)
    rcap, dcap = _caps(ds)
    mk = ctx.create_transient
    vss = [frame.ViewState(ctx, ds, (v.width, v.height), name="rf%d" % i) for i, v in enumerate(views)]
    d = [mk("rf_d%d" % v, L.DISPATCH_HEADER + 16 * rcap) for v in range(17)]
    w = [mk("rf_w%d" % v, L.DRAW_HEADER + 28 * dcap) for v in range(17)]
    pay = [mk("rf_p%d" % v, 44 * rcap) for v in range(17)]
    INVALID = _lib.ERR_INVALID_ARGUMENT
    arr = lambda ps: (C.c_void_p * max(len(ps), 1))(*ps)

    def pack(kind, n=4, mocc=True):
        infos = [_info(vss[v], views[v], kind, mocc) for v in range(n)]
        gs = (L.CullInfo * max(n, 1))(*[ci.to_gpu() for ci in infos])
        sbs = (L.SceneBuffers * max(n, 1))(*[_scene_buffers(ds.assets, ds.scene, ci) for ci in infos])
        hz = [vss[v].depth_pyramid._h.value for v in range(n)]
        return gs, sbs, hz

    def call(gs, sbs, n, hz, dp, wp, pp=None):
        before = ctx.launch_count
        a = lib.orbit_entity_cull_views_occlusion(ctx._h, gs, n, sbs, arr(hz) if hz is not None else None, arr(dp), rcap, _stream())
        b = lib.orbit_meshlet_cull_views_occlusion(ctx._h, gs, n, sbs, arr(hz) if hz is not None else None, arr(dp), rcap, arr(wp), dcap,
                                                   arr(pp) if pp is not None else None, _stream())
        assert ctx.launch_count == before
        return a, b

    ptr = lambda ts, off=0: [t.data_ptr() + off for t in ts]
    cases = {}
    gs, sbs, hz = pack("write"); cases["zero views"] = (gs, sbs, 0, hz, ptr(d[:1]), ptr(w[:1]))
    gs, sbs, hz = pack("write", 17); cases["17 views"] = (gs, sbs, 17, hz, ptr(d), ptr(w))
    gs, sbs, hz = pack("read"); gs[0].occlusion_pass = 0; gs[1].occlusion_pass = 0; gs[2].occlusion_pass = 0; gs[3].occlusion_pass = 0
    cases["pass 0"] = (gs, sbs, 4, hz, ptr(d[:4]), ptr(w[:4]))
    gs, sbs, hz = pack("read"); gs[2].occlusion_pass = 2; cases["mixed passes"] = (gs, sbs, 4, hz, ptr(d[:4]), ptr(w[:4]))
    gs, sbs, hz = pack("write"); gs[1].projection_type = L.PROJ_ORTHOGRAPHIC; cases["mixed projection"] = (gs, sbs, 4, hz, ptr(d[:4]), ptr(w[:4]))
    gs, sbs, hz = pack("write"); gs[2].meshlet_visibility_buffer = L.NO_BUFFER; cases["mixed meshlet occlusion"] = (gs, sbs, 4, hz, ptr(d[:4]), ptr(w[:4]))
    gs, sbs, hz = pack("write"); sbs[3].entities = sbs[3].entities + 16; cases["another scene"] = (gs, sbs, 4, hz, ptr(d[:4]), ptr(w[:4]))
    gs, sbs, hz = pack("write"); sbs[3].draw_end = 32; cases["another draw range"] = (gs, sbs, 4, hz, ptr(d[:4]), ptr(w[:4]))
    gs, sbs, hz = pack("write"); sbs[2].entity_visibility = sbs[0].entity_visibility; sbs[2].meshlet_visibility = sbs[0].meshlet_visibility
    cases["shared visibility"] = (gs, sbs, 4, hz, ptr(d[:4]), ptr(w[:4]))
    gs, sbs, hz = pack("write"); cases["shared dispatch / draw buffer"] = (gs, sbs, 4, hz, ptr(d[:3]) + ptr(d[:1]), ptr(w[:3]) + ptr(w[:1]))
    gs, sbs, hz = pack("write"); cases["NULL buffer"] = (gs, sbs, 4, hz, ptr(d[:3]) + [None], ptr(w[:3]) + [None])
    gs, sbs, hz = pack("write"); cases["misaligned"] = (gs, sbs, 4, hz, ptr(d[:3]) + ptr(d[3:4], 2), ptr(w[:3]) + ptr(w[3:4], 2))
    gs, sbs, hz = pack("write"); cases["no pyramids in pass 2"] = (gs, sbs, 4, None, ptr(d[:4]), ptr(w[:4]))
    gs, sbs, hz = pack("write"); cases["NULL pyramid"] = (gs, sbs, 4, hz[:3] + [None], ptr(d[:4]), ptr(w[:4]))
    gs, sbs, hz = pack("write"); cases["shared pyramid"] = (gs, sbs, 4, hz[:3] + hz[:1], ptr(d[:4]), ptr(w[:4]))
    odd = DepthPyramid(ctx, "rf_odd", (640, 480))
    gs, sbs, hz = pack("write"); cases["pyramids of two geometries"] = (gs, sbs, 4, hz[:3] + [odd._h.value], ptr(d[:4]), ptr(w[:4]))
    gs, sbs, hz = pack("write"); gs[3].cull_plane_count = 13; cases["13 planes"] = (gs, sbs, 4, hz, ptr(d[:4]), ptr(w[:4]))
    for what, (gs, sbs, n, hz, dp, wp) in cases.items():
        assert call(gs, sbs, n, hz, dp, wp) == (INVALID, INVALID), what
    # what only one stage refuses: a draw range that does not start on a multiple of 32 (entity stage); a shared task
    # payload buffer and no meshlets (meshlet stage)
    before = ctx.launch_count
    gs, sbs, hz = pack("write")
    for v in range(4):
        sbs[v].draw_begin = 5
    assert lib.orbit_entity_cull_views_occlusion(ctx._h, gs, 4, sbs, arr(hz), arr(ptr(d[:4])), rcap, _stream()) == INVALID
    gs, sbs, hz = pack("write")
    assert lib.orbit_meshlet_cull_views_occlusion(ctx._h, gs, 4, sbs, arr(hz), arr(ptr(d[:4])), rcap, arr(ptr(w[:4])), dcap,
                                                  arr(ptr(pay[:3]) + ptr(pay[:1])), _stream()) == INVALID
    for v in range(4):
        sbs[v].meshlets = 0
    assert lib.orbit_meshlet_cull_views_occlusion(ctx._h, gs, 4, sbs, arr(hz), arr(ptr(d[:4])), rcap, arr(ptr(w[:4])), dcap, None,
                                                  _stream()) == INVALID
    assert ctx.launch_count == before
    # the pyramid build: zero / 17 pyramids, a wrong depth size, a shared pyramid, a NULL depth buffer
    depth = torch.zeros((1080, 1920), dtype=torch.float32, device=ctx.device)
    hz = [vss[v].depth_pyramid._h.value for v in range(17)]
    dps = [depth.data_ptr()] * 17
    before = ctx.launch_count
    for what, (h, dp, n, wh) in {"zero": (hz, dps, 0, (1920, 1080)), "17": (hz, dps, 17, (1920, 1080)), "size": (hz, dps, 4, (1920, 1088)),
                                 "shared": (hz[:3] + hz[:1], dps, 4, (1920, 1080)), "NULL depth": (hz, dps[:3] + [None], 4, (1920, 1080))}.items():
        assert lib.orbit_hiz_build_views(ctx._h, arr(h), arr(dp), n, wh[0], wh[1], _stream()) == INVALID, what
    assert ctx.launch_count == before
