"""GPU parity of orbit_hiz_build_entity_cull_late (orbit_cuda.h): the Hi-Z build and the LATE entity stage in one call, whose
entity kernel runs its pyramid-independent work before griddepcontrol.wait. Every case runs two copies of one frame side by
side: one with the separate calls (orbit_hiz_build, then orbit_entity_cull or orbit_entity_cull_late_main), one through
PreparedFrame.launch, which uses the new call. After every frame both copies must hold the same bytes: pyramid texels, entity
and meshlet visibility words, every dispatch buffer (header and records) and every draw list. Cases: the C2 steady-state frame,
a moving camera (A, A, B as in bench.py), an orthographic camera, MAIN present (fused LATE + MAIN) and absent, a CUDA graph
replayed over alternating scene copies, the same frames with ORBIT_NO_PDL=1 (the wait is a no-op, stream order alone
orders the kernels), and every refused argument combination on a real context."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from orbit_b200 import scenes

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _ortho_views(sc):
    lo, hi = np.asarray(sc.aabb_min), np.asarray(sc.aabb_max)
    c = 0.5 * (lo + hi)
    return (scenes.orthographic_view((c[0] - 60.0, c[1] + 40.0, c[2] - 60.0), (0.6, -0.45, 0.66), 1024, 1024, 80.0, 0.5, 400.0),
            scenes.orthographic_view((c[0] - 40.0, c[1] + 40.0, c[2] - 70.0), (0.5, -0.45, 0.74), 1024, 1024, 80.0, 0.5, 400.0))


def _separate(pf):
    """pf's frame with orbit_hiz_build and the separate LATE entity call (the form PreparedFrame.launch had before)."""
    pf.entity(False); pf.meshlet(False); pf.hiz()
    if pf.fused:
        pf.entity_late_main(); pf.meshlet_late_main()
        return
    pf.entity(True); pf.meshlet(True)
    if pf.main_pass:
        pf.entity("main"); pf.meshlet("main")


def _bytes(pf):
    from orbit_b200.frame import read_dispatch, read_draws
    out = {"texels": pf.vstate.depth_pyramid.texels.cpu().numpy().view(np.uint32).copy(),
           "entity_visibility": pf.vstate.entity_visibility.cpu().numpy().view(np.uint32).copy(),
           "meshlet_visibility": pf.vstate.meshlet_visibility.cpu().numpy().view(np.uint32).copy()}
    stages = ("early", "late", "main") if pf.main_pass else ("early", "late")
    for k in stages:
        hdr, recs = read_dispatch(getattr(pf, k + "_dispatch"))
        n, draws = read_draws(getattr(pf, k + "_draws"))
        out[k + "_dispatch"] = np.concatenate([hdr, recs.view(np.uint32).ravel()])
        out[k + "_draws"] = np.concatenate([np.array([n], np.uint32), draws.view(np.uint32).ravel()])
    return out


def _assert_same(a, b, what):
    assert a.keys() == b.keys()
    for k in a:
        assert np.array_equal(a[k], b[k]), (what, k)


def _pair(ctx, ds, view, d_depth, tag, main_pass):
    """Two PreparedFrames of one view and scene, each with its own bitmasks, pyramid and output buffers."""
    from orbit_b200 import frame
    out = []
    for form in ("sep", "new"):
        vs = frame.ViewState(ctx, ds, (view.width, view.height), name="hef_%s_%s" % (tag, form))
        out.append(frame.PreparedFrame(ctx, ds, vs, view, d_depth, name="hef_%s_%s" % (tag, form), main_pass=main_pass))
    return out


def _retarget(ctx, pf, view, d_depth, main_pass):
    """The same buffers and bitmasks, another camera and depth buffer (the moving-camera frame of bench.py)."""
    from orbit_b200 import frame
    q = frame.PreparedFrame(ctx, pf.dscene, pf.vstate, view, d_depth, name="moved", main_pass=main_pass)
    for k in ("early", "late", "main") if main_pass else ("early", "late"):
        for b in ("_dispatch", "_draws"):
            setattr(q, k + b, getattr(pf, k + b))
    return q


def run_frames(ctx, case, main_pass):
    """Frames A, A, B, A of `case` through both forms, compared after each; returns the LATE record count of every frame."""
    from orbit_b200 import frame
    if case == "c2":
        sc, _ = scenes.config_c2()
        import bench
        view_a, view_b = bench.c2_view(scenes, sc, 0), bench.c2_view(scenes, sc, 4)
    elif case == "ortho":
        sc, _ = scenes.config_c2(scale=0.08)
        view_a, view_b = _ortho_views(sc)
    else:
        raise ValueError(case)
    ds = frame.DeviceScene.upload(ctx, sc)
    d_a = torch.from_numpy(scenes.make_depth(sc, view_a)).to(ctx.device)
    d_b = torch.from_numpy(scenes.make_depth(sc, view_b)).to(ctx.device)
    sep, new = _pair(ctx, ds, view_a, d_a, case + str(int(main_pass)), main_pass)
    assert sep.fused == new.fused == main_pass
    sep_b, new_b = _retarget(ctx, sep, view_b, d_b, main_pass), _retarget(ctx, new, view_b, d_b, main_pass)
    late_records = []
    # A, A: first frame and steady state; B: the camera moved (the LATE pass finds survivors); A again
    for i, (s, n) in enumerate([(sep, new), (sep, new), (sep_b, new_b), (sep, new)]):
        _separate(s)
        n.launch()
        torch.cuda.synchronize()
        a, b = _bytes(s), _bytes(n)
        _assert_same(a, b, (case, main_pass, i))
        late_records.append(int(a["late_dispatch"][0]))
    return late_records


@pytest.mark.parametrize("main_pass", [True, False], ids=["main", "no_main"])
@pytest.mark.parametrize("case", ["c2", "ortho"])
def test_same_bytes_as_the_separate_calls(gpu_context, case, main_pass):
    late = run_frames(gpu_context, case, main_pass)
    assert late[0] > 0, late        # first frame (all bits zero): the LATE pass draws what the pyramid does not hide


def test_graph_replays_over_alternating_scene_copies(gpu_context):
    """Two scene copies, each a PreparedFrame pair captured into CUDA graphs; 24 replays alternate between the copies (tickets,
    scan epochs and the Hi-Z ticket live in device memory), every one compared with the separate calls' graph."""
    from orbit_b200 import frame
    ctx = gpu_context
    sc, view = scenes.config_c2(scale=0.25)
    d = torch.from_numpy(scenes.make_depth(sc, view)).to(ctx.device)
    pairs = [_pair(ctx, frame.DeviceScene.upload(ctx, sc), view, d, "graph%d" % i, True) for i in range(2)]
    graphs = []
    for sep, new in pairs:
        _separate(sep); torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            _separate(sep)
        new.capture()                 # one warm frame, then the capture
        graphs.append((g, new))
    for r in range(24):
        k = r % 2
        graphs[k][0].replay(); graphs[k][1].replay()
        torch.cuda.synchronize()
        _assert_same(_bytes(pairs[k][0]), _bytes(pairs[k][1]), ("replay", r))


def test_without_pdl_in_a_subprocess(gpu_context):
    """ORBIT_NO_PDL=1: launches without programmatic serialization, griddepcontrol.wait is a no-op and the entity kernel
    starts only when the build has finished. Same frames as the C2 case, MAIN present and absent."""
    env = dict(os.environ, ORBIT_NO_PDL="1")
    code = ("import sys; sys.path.insert(0, %r); sys.path.insert(0, %r)\n"
            "import test_gpu_hiz_entity_fused as t\n"
            "from orbit_b200.passes import Context\n"
            "ctx = Context(0)\n"
            "for m in (True, False): print(t.run_frames(ctx, 'c2', m))\n"
            "ctx.close()\n" % (ROOT, os.path.join(ROOT, "tests")))
    res = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stdout + res.stderr


def test_refused_calls_launch_nothing(gpu_context):
    """Every rule of orbit_hiz_build + orbit_entity_cull(_late_main), plus late pass 2 and a MAIN dispatch buffer only with a
    MAIN CullInfo: each refused combination returns ORBIT_ERR_INVALID_ARGUMENT, launches nothing and leaves every buffer as
    it was."""
    from orbit_b200 import _lib, frame, layouts as L
    from orbit_b200.passes import _ptr
    ctx, lib = gpu_context, _lib.lib()
    sc, view = scenes.config_c1(scale=0.2)
    d = torch.from_numpy(scenes.make_depth(sc, view)).to(ctx.device)
    ds = frame.DeviceScene.upload(ctx, sc)
    vs = frame.ViewState(ctx, ds, (view.width, view.height), name="hef_bad")
    pf = frame.PreparedFrame(ctx, ds, vs, view, d, name="hef_bad", main_pass=True)
    assert pf.fused
    pf.launch(); torch.cuda.synchronize()
    before = _bytes(pf)
    n0 = lib.orbit_ctx_launch_count(ctx._h)
    w, h = pf._hw
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    late_d, main_d = _ptr(pf.late_dispatch), _ptr(pf.main_dispatch)

    def call(ctx_h=ctx._h, hiz=vs.depth_pyramid._h, depth=_ptr(d), dw=w, dh=h, late=None, main=None, sb=None, ld=late_d, md=main_d):
        gl = late if late is not None else L.CullInfo.from_buffer_copy(pf.g_late)
        gm = main if main is not None else L.CullInfo.from_buffer_copy(pf.g_early)
        b = sb if sb is not None else L.SceneBuffers.from_buffer_copy(pf.sb_late)
        return lib.orbit_hiz_build_entity_cull_late(ctx_h, hiz, depth, dw, dh, None if late is False else C.byref(gl),
                                                    None if main is False else C.byref(gm), C.byref(b), ld, md, pf.rcap, s)

    def edited(src, **kw):
        g = type(src).from_buffer_copy(src)
        for k, v in kw.items():
            setattr(g, k, v)
        return g
    bad = {
        "no context": dict(ctx_h=None), "no pyramid": dict(hiz=None), "no depth": dict(depth=None),
        "depth width": dict(dw=w + 1), "depth height": dict(dh=h - 1), "no late CullInfo": dict(late=False),
        "late pass 0": dict(late=edited(pf.g_late, occlusion_pass=0)), "late pass 1": dict(late=edited(pf.g_late, occlusion_pass=1)),
        "MAIN without its buffer": dict(md=None), "MAIN buffer without MAIN": dict(main=False),
        "MAIN buffer = LATE buffer": dict(md=late_d), "MAIN buffer misaligned": dict(md=C.c_void_p(pf.main_dispatch.data_ptr() + 2)),
        "incompatible pair": dict(main=edited(pf.g_early, lod_base=pf.g_early.lod_base * 2.0)),
        "MAIN pass 2": dict(main=edited(pf.g_early, occlusion_pass=2)),
        "no LATE buffer": dict(ld=None, main=False, md=None), "LATE buffer misaligned": dict(ld=C.c_void_p(pf.late_dispatch.data_ptr() + 1)),
        "too many planes": dict(late=edited(pf.g_late, cull_plane_count=L.MAX_CULL_PLANES + 1)),
        "no entity visibility": dict(sb=edited(pf.sb_late, entity_visibility=None)),
        "no entities": dict(sb=edited(pf.sb_late, entities=None)),
        "mesh infos misaligned": dict(sb=edited(pf.sb_late, mesh_infos=pf.sb_late.mesh_infos + 4)),
        "draw_begin % 32": dict(sb=edited(pf.sb_late, draw_begin=3, draw_end=50)),
        "draw_begin > draw_end": dict(sb=edited(pf.sb_late, draw_begin=64, draw_end=32)),
    }
    for what, kw in bad.items():
        assert call(**kw) == _lib.ERR_INVALID_ARGUMENT, what
    torch.cuda.synchronize()
    assert lib.orbit_ctx_launch_count(ctx._h) == n0
    _assert_same(before, _bytes(pf), "after the refused calls")
    assert call() == 0 and lib.orbit_ctx_launch_count(ctx._h) == n0 + 2     # the valid call: two launches
    torch.cuda.synchronize()
