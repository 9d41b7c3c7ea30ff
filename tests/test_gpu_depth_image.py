"""GPU parity of the depth-image entry points (orbit_depth_image_wrap and the *_image stage calls, orbit_cuda.h): depth read
from a 2-D float CUDA array, the form a Vulkan depth attachment takes once imported, must give byte for byte what the linear
calls give for the same depth values. The arrays are made here through cudart (cudaMallocArray, cudaMallocMipmappedArray +
cudaGetMipmappedArrayLevel), filled with cudaMemcpy2DToArrayAsync. Cases: pyramids at the sizes of test_hiz_bit_exact (plain
arrays and level 0 of a mipmapped array) against orbit_hiz_build and the oracle, the batched build with 1, 4 and 16 images,
the C2 frame through PreparedFrame (moving camera, orthographic camera, MAIN present and absent, a CUDA graph replayed over
alternating scene copies with the arrays re-filled between replays, ORBIT_NO_PDL=1 in a subprocess), four batched cameras
through PreparedViews, clustered light assignment, and every refused argument on a real context."""
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

# cudaChannelFormatKind, cudaMemcpyKind and array flags of cuda_runtime_api.h
KIND_SIGNED, KIND_UNSIGNED, KIND_FLOAT = 0, 1, 2
MEMCPY_D2D = 3
ARRAY_LAYERED = 0x01


class _Desc(C.Structure):
    _fields_ = [("x", C.c_int), ("y", C.c_int), ("z", C.c_int), ("w", C.c_int), ("f", C.c_int)]


class _Extent(C.Structure):
    _fields_ = [("width", C.c_size_t), ("height", C.c_size_t), ("depth", C.c_size_t)]


def _load_cudart():
    """libcudart.so.12 of the CUDA toolkit (as test_gpu_cpp_host.py links it), else the one torch's wheel ships."""
    cands = ["/usr/local/cuda/lib64/libcudart.so.12",
             os.path.join(os.path.dirname(os.path.dirname(torch.__file__)), "nvidia", "cuda_runtime", "lib", "libcudart.so.12")]
    for p in cands:
        if os.path.exists(p):
            return C.CDLL(p)
    pytest.fail("libcudart.so.12 not found in %s" % cands)


class Arrays:
    """CUDA arrays made through cudart and freed at teardown. Arrays and streams are driver objects shared by every cudart
    in the process (cudaArray_t and CUarray are interchangeable), so the library's texture objects can read them."""

    def __init__(self, device):
        self.rt = _load_cudart()
        self.rt.cudaSetDevice(device.index or 0)
        self.arrays, self.mipmaps = [], []

    def _ck(self, rc, what):
        assert rc == 0, "%s failed: cudaError %d" % (what, rc)

    def array(self, w, h, bits=(32, 0, 0, 0), kind=KIND_FLOAT):
        a = C.c_void_p()
        self._ck(self.rt.cudaMallocArray(C.byref(a), C.byref(_Desc(*bits, kind)), C.c_size_t(w), C.c_size_t(h), C.c_uint(0)), "cudaMallocArray")
        self.arrays.append(a.value)
        return a.value

    def array3d(self, w, h, d, flags):
        a = C.c_void_p()
        self._ck(self.rt.cudaMalloc3DArray(C.byref(a), C.byref(_Desc(32, 0, 0, 0, KIND_FLOAT)), _Extent(w, h, d), C.c_uint(flags)),
                 "cudaMalloc3DArray")
        self.arrays.append(a.value)
        return a.value

    def mip_level0(self, w, h, levels=3):
        mm, a = C.c_void_p(), C.c_void_p()
        self._ck(self.rt.cudaMallocMipmappedArray(C.byref(mm), C.byref(_Desc(32, 0, 0, 0, KIND_FLOAT)), _Extent(w, h, 0), C.c_uint(levels),
                                                  C.c_uint(0)), "cudaMallocMipmappedArray")
        self.mipmaps.append(mm.value)
        self._ck(self.rt.cudaGetMipmappedArrayLevel(C.byref(a), mm, C.c_uint(0)), "cudaGetMipmappedArrayLevel")
        return a.value

    def fill(self, arr, depth):
        """Copies `depth` (a float32 device tensor [H, W]) into `arr` on torch's current stream."""
        h, w = depth.shape
        s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        self._ck(self.rt.cudaMemcpy2DToArrayAsync(C.c_void_p(arr), C.c_size_t(0), C.c_size_t(0), C.c_void_p(depth.data_ptr()),
                                                  C.c_size_t(4 * w), C.c_size_t(4 * w), C.c_size_t(h), C.c_int(MEMCPY_D2D), s),
                 "cudaMemcpy2DToArrayAsync")

    def free(self):
        torch.cuda.synchronize()
        for a in self.arrays:
            self.rt.cudaFreeArray(C.c_void_p(a))
        for m in self.mipmaps:
            self.rt.cudaFreeMipmappedArray(C.c_void_p(m))
        self.arrays, self.mipmaps = [], []


@pytest.fixture(scope="module")
def arrays(gpu_context):
    a = Arrays(gpu_context.device)
    yield a
    a.free()


def _image(ctx, arrays, depth, mip=False):
    """A DepthImage holding the values of `depth` (float32 device tensor [H, W])."""
    from orbit_b200.passes import DepthImage
    h, w = depth.shape
    arr = arrays.mip_level0(w, h) if mip else arrays.array(w, h)
    arrays.fill(arr, depth)
    img = DepthImage(ctx, arr)
    assert img.size == (w, h)
    return img


def _u32(t):
    return t.cpu().numpy().view(np.uint32)


def _random_depth(w, h):
    rng = np.random.default_rng(w * 7919 + h)
    depth = rng.random((h, w), dtype=np.float32)
    depth[rng.random((h, w)) < 0.3] = 0.0
    return depth


# ---- pyramids ------------------------------------------------------------------------------------------------------------
SIZES = [(1920, 1080), (3840, 2160), (1280, 720), (100, 60), (64, 64), (129, 257), (2, 2), (4096, 33)]
MIP_SIZES = [(1920, 1080), (129, 257)]


@pytest.mark.parametrize("size,mip", [(s, False) for s in SIZES] + [(s, True) for s in MIP_SIZES],
                         ids=["%dx%d" % s for s in SIZES] + ["%dx%d_mip_level0" % s for s in MIP_SIZES])
def test_pyramid_same_as_linear_and_oracle(gpu_context, arrays, oracle, size, mip):
    from orbit_b200.passes import DepthPyramid
    ctx = gpu_context
    w, h = size
    depth = _random_depth(w, h)
    d = torch.from_numpy(depth).to(ctx.device)
    img = _image(ctx, arrays, d, mip)
    lin, tex = DepthPyramid(ctx, "dimg_lin", (w, h)), DepthPyramid(ctx, "dimg_tex", (w, h))
    tex.texels.fill_(-1.0)
    lin.update(d)
    tex.update(img)
    torch.cuda.synchronize()
    _, ref = oracle.hiz_build(depth)
    assert np.array_equal(_u32(tex.texels), _u32(lin.texels))
    assert np.array_equal(_u32(tex.texels), ref.view(np.uint32))
    img.close()


@pytest.mark.parametrize("n", [1, 4, 16])
@pytest.mark.parametrize("size", [(1920, 1080), (100, 60)], ids=["1920x1080", "100x60"])
def test_batched_build_same_as_linear(gpu_context, arrays, size, n):
    from orbit_b200 import frame
    from orbit_b200.passes import DepthPyramid
    ctx = gpu_context
    w, h = size
    ds = [torch.from_numpy(np.roll(_random_depth(w, h), 7 * v, axis=1)).to(ctx.device) for v in range(n)]
    imgs = [_image(ctx, arrays, d) for d in ds]
    lin = [DepthPyramid(ctx, "dimgv_lin%d" % v, (w, h)) for v in range(n)]
    tex = [DepthPyramid(ctx, "dimgv_tex%d" % v, (w, h)) for v in range(n)]
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    frame._HizViews(ctx, lin, ds).launch(s)
    hv = frame._HizViews(ctx, tex, imgs)
    assert hv.image
    hv.launch(s)
    torch.cuda.synchronize()
    for v in range(n):
        assert np.array_equal(_u32(tex[v].texels), _u32(lin[v].texels)), v
    for i in imgs:
        i.close()


# ---- frames --------------------------------------------------------------------------------------------------------------
def _fused():
    import test_gpu_hiz_entity_fused as F      # the comparison helpers of the fused call's parity test
    return F


def _pair(ctx, ds, view, d_depth, image, tag, main_pass):
    """Two PreparedFrames of one view and scene with their own bitmasks, pyramid and buffers: depth from the tensor / the image."""
    from orbit_b200 import frame
    out = []
    for form, src in (("lin", d_depth), ("img", image)):
        vs = frame.ViewState(ctx, ds, (view.width, view.height), name="dimg_%s_%s" % (tag, form))
        out.append(frame.PreparedFrame(ctx, ds, vs, view, src, name="dimg_%s_%s" % (tag, form), main_pass=main_pass))
    assert not out[0].image and out[1].image
    return out


def run_frames(ctx, arrays, case, main_pass):
    """Frames A, A, B, A of `case`, depth from a tensor and from an image, both through PreparedFrame.launch (so
    orbit_hiz_build_entity_cull_late and orbit_hiz_build_image_entity_cull_late), compared after each frame."""
    from orbit_b200 import frame
    F = _fused()
    if case == "c2":
        sc, _ = scenes.config_c2()
        import bench
        view_a, view_b = bench.c2_view(scenes, sc, 0), bench.c2_view(scenes, sc, 4)
    elif case == "ortho":
        sc, _ = scenes.config_c2(scale=0.08)
        view_a, view_b = F._ortho_views(sc)
    else:
        raise ValueError(case)
    ds = frame.DeviceScene.upload(ctx, sc)
    d_a = torch.from_numpy(scenes.make_depth(sc, view_a)).to(ctx.device)
    d_b = torch.from_numpy(scenes.make_depth(sc, view_b)).to(ctx.device)
    i_a, i_b = _image(ctx, arrays, d_a), _image(ctx, arrays, d_b)
    lin, img = _pair(ctx, ds, view_a, d_a, i_a, case + str(int(main_pass)), main_pass)
    assert lin.fused == img.fused == main_pass
    lin_b, img_b = F._retarget(ctx, lin, view_b, d_b, main_pass), F._retarget(ctx, img, view_b, i_b, main_pass)
    late_records = []
    for i, (a, b) in enumerate([(lin, img), (lin, img), (lin_b, img_b), (lin, img)]):
        a.launch()
        b.launch()
        torch.cuda.synchronize()
        x, y = F._bytes(a), F._bytes(b)
        F._assert_same(x, y, (case, main_pass, i))
        late_records.append(int(x["late_dispatch"][0]))
    return late_records


@pytest.mark.parametrize("main_pass", [True, False], ids=["main", "no_main"])
@pytest.mark.parametrize("case", ["c2", "ortho"])
def test_frame_same_bytes_as_linear(gpu_context, arrays, case, main_pass):
    late = run_frames(gpu_context, arrays, case, main_pass)
    assert late[0] > 0, late


def test_graph_replays_refilling_the_arrays(gpu_context, arrays):
    """Two scene copies, each a (tensor, image) PreparedFrame pair captured into CUDA graphs; 24 replays alternate between the
    copies, and before every replay the depth tensors and arrays are re-filled with one of two depth buffers (the graph reads
    the array at replay time)."""
    from orbit_b200 import frame
    F = _fused()
    ctx = gpu_context
    sc, view = scenes.config_c2(scale=0.25)
    import bench
    srcs = [torch.from_numpy(scenes.make_depth(sc, v)).to(ctx.device) for v in (view, bench.c2_view(scenes, sc, 1))]
    pairs = []
    for i in range(2):
        d = srcs[0].clone()
        img = _image(ctx, arrays, d)
        arr = arrays.arrays[-1]
        lin, tex = _pair(ctx, frame.DeviceScene.upload(ctx, sc), view, d, img, "graph%d" % i, True)
        lin.capture(); tex.capture()
        pairs.append((lin, tex, d, arr))
    for r in range(24):
        lin, tex, d, arr = pairs[r % 2]
        src = srcs[(r // 2) % 2]
        d.copy_(src)
        arrays.fill(arr, src)
        lin.replay(); tex.replay()
        torch.cuda.synchronize()
        F._assert_same(F._bytes(lin), F._bytes(tex), ("replay", r))


def test_without_pdl_in_a_subprocess(gpu_context):
    env = dict(os.environ, ORBIT_NO_PDL="1")
    code = ("import sys; sys.path.insert(0, %r); sys.path.insert(0, %r)\n"
            "import test_gpu_depth_image as t\n"
            "from orbit_b200.passes import Context\n"
            "ctx = Context(0)\n"
            "arrays = t.Arrays(ctx.device)\n"
            "for m in (True, False): print(t.run_frames(ctx, arrays, 'c2', m))\n"
            "arrays.free()\n"
            "ctx.close()\n" % (ROOT, os.path.join(ROOT, "tests")))
    res = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stdout + res.stderr


def test_batched_cameras_same_as_linear(gpu_context, arrays):
    """PreparedViews of four C2 cameras (EARLY, batched Hi-Z, LATE, MAIN) fed by four images equals the same frame fed by tensors."""
    from orbit_b200 import frame
    import bench
    ctx = gpu_context
    sc, _ = scenes.config_c2()
    views = [bench.c2_view(scenes, sc, i) for i in range(4)]
    ds = frame.DeviceScene.upload(ctx, sc)
    depths = [torch.from_numpy(scenes.make_depth(sc, v)).to(ctx.device) for v in views]
    imgs = [_image(ctx, arrays, d) for d in depths]
    out = []
    for form, srcs in (("lin", depths), ("img", imgs)):
        vs = [frame.ViewState(ctx, ds, (v.width, v.height), name="dimg_pv_%s%d" % (form, i)) for i, v in enumerate(views)]
        pv = frame.PreparedViews(ctx, ds, vs, views, srcs, name="dimg_pv_" + form)
        out.append((pv, vs))
    for f in range(2):
        for pv, _ in out:
            pv.launch()
        torch.cuda.synchronize()
        (pa, va), (pb, vb) = out
        for v in range(4):
            for k in ("early", "late", "main"):
                (da, wa), (db, wb) = pa.outputs[v][k], pb.outputs[v][k]
                (ha, ra), (hb, rb) = frame.read_dispatch(da), frame.read_dispatch(db)
                assert np.array_equal(ha, hb) and np.array_equal(ra.view(np.uint32), rb.view(np.uint32)), (f, v, k, "dispatch")
                (na, xa), (nb, xb) = frame.read_draws(wa), frame.read_draws(wb)
                assert na == nb and np.array_equal(xa.view(np.uint32), xb.view(np.uint32)), (f, v, k, "draws")
            for t in ("entity_visibility", "meshlet_visibility"):
                assert np.array_equal(_u32(getattr(va[v], t)), _u32(getattr(vb[v], t))), (f, v, t)
            assert np.array_equal(_u32(va[v].depth_pyramid.texels), _u32(vb[v].depth_pyramid.texels)), (f, v)


# ---- clusters ------------------------------------------------------------------------------------------------------------
def _clusters_both(ctx, arrays, sc, view, depth, lights, settings):
    from orbit_b200 import frame
    from orbit_b200.passes import compute_clusters
    ds = frame.DeviceScene.upload(ctx, sc, lights=lights)
    d = torch.from_numpy(depth).to(ctx.device)
    img = _image(ctx, arrays, d)
    res = []
    for tag, src in (("lin", d), ("img", img)):
        info, _ = compute_clusters(ctx, settings, view.view, view.projection_matrix, view.near, src, ds.scene, name="dimg_cl_" + tag)
        torch.cuda.synchronize()
        res.append({k: getattr(info, k).cpu().numpy().copy() for k in ("tile_depth_slice_mask", "cluster_depth_bounds",
                                                                       "unique_cluster_buffer", "light_offset_image", "light_index_buffer")})
    for k in res[0]:
        assert np.array_equal(res[0][k], res[1][k]), k
    img.close()
    return res[0]


def test_clusters_c4_reduced(gpu_context, arrays):
    from orbit_b200.passes import ClusterSettings
    sc, view = scenes.config_c4(scale=0.02)
    depth = scenes.make_depth(sc, view)
    lights = scenes.make_lights(scenes.SEEDS["C4"], 4096, sc.aabb_min, sc.aabb_max)
    r = _clusters_both(gpu_context, arrays, sc, view, depth, lights, ClusterSettings(screen_resolution=(1920, 1080), z_slice_count=24,
                                                                                      tile_size_px=120))
    assert r["unique_cluster_buffer"].view(np.uint32)[3] > 0 and r["light_index_buffer"].view(np.uint32)[0] > 0


def test_clusters_default_settings(gpu_context, arrays):
    from orbit_b200.passes import ClusterSettings
    sc, _ = scenes.config_c4(scale=0.005)
    view = scenes.perspective_view((-6.0, 3.0, -6.0), (0.6, 0.0, 0.8), 320, 180)
    depth = scenes.make_depth(sc, view)
    lights = scenes.make_lights(scenes.SEEDS["C4"] + 1, 3000, sc.aabb_min * 0.3, sc.aabb_max * 0.3, intensity=(20.0, 60.0))
    r = _clusters_both(gpu_context, arrays, sc, view, depth, lights, ClusterSettings(screen_resolution=(320, 180)))
    assert r["light_index_buffer"].view(np.uint32)[0] > 0


def test_clusters_no_lights_and_sky_only(gpu_context, arrays):
    from orbit_b200.passes import ClusterSettings
    sc, _ = scenes.config_c4(scale=0.005)
    view = scenes.perspective_view((-6.0, 3.0, -6.0), (0.6, 0.0, 0.8), 256, 128)
    depth = np.zeros((128, 256), np.float32)
    lights = scenes.make_lights(1, 16, sc.aabb_min, sc.aabb_max)
    r = _clusters_both(gpu_context, arrays, sc, view, depth, lights, ClusterSettings(screen_resolution=(256, 128)))
    assert r["unique_cluster_buffer"].view(np.uint32)[3] == 0 and r["light_index_buffer"].view(np.uint32)[0] == 0


# ---- refusals ------------------------------------------------------------------------------------------------------------
def test_wrap_refuses_every_array_but_2d_float32(gpu_context, arrays):
    from orbit_b200 import _lib
    ctx, lib = gpu_context, _lib.lib()
    n0 = lib.orbit_ctx_launch_count(ctx._h)
    bad = {
        "float2": arrays.array(64, 32, (32, 32, 0, 0)), "half": arrays.array(64, 32, (16, 0, 0, 0)),
        "uint32": arrays.array(64, 32, (32, 0, 0, 0), KIND_UNSIGNED), "int32": arrays.array(64, 32, (32, 0, 0, 0), KIND_SIGNED),
        "8-bit": arrays.array(64, 32, (8, 0, 0, 0), KIND_UNSIGNED), "1-D": arrays.array(64, 0),
        "layered": arrays.array3d(64, 32, 2, ARRAY_LAYERED), "3-D": arrays.array3d(64, 32, 4, 0), "NULL": None,
    }
    for what, arr in bad.items():
        out = C.c_void_p(1234)
        assert lib.orbit_depth_image_wrap(ctx._h, C.c_void_p(arr), C.byref(out)) == _lib.ERR_INVALID_ARGUMENT, what
        assert out.value is None, what
    good = C.c_void_p()
    assert lib.orbit_depth_image_wrap(ctx._h, C.c_void_p(arrays.array(64, 32)), C.byref(good)) == _lib.OK
    w, h = C.c_uint32(), C.c_uint32()
    assert lib.orbit_depth_image_size(good, C.byref(w), C.byref(h)) == _lib.OK and (w.value, h.value) == (64, 32)
    lib.orbit_depth_image_destroy(good)
    assert lib.orbit_ctx_launch_count(ctx._h) == n0


def test_refused_stage_calls_launch_nothing(gpu_context, arrays):
    """Size mismatches for every stage variant, NULL handles, and every rule the fused call inherits from
    orbit_hiz_build_entity_cull_late: ORBIT_ERR_INVALID_ARGUMENT, nothing launched, every buffer as it was."""
    from orbit_b200 import _lib, frame, layouts as L
    from orbit_b200.passes import ClusterSettings, DepthPyramid, _ptr, compute_clusters
    F = _fused()
    ctx, lib = gpu_context, _lib.lib()
    sc, view = scenes.config_c1(scale=0.2)
    d = torch.from_numpy(scenes.make_depth(sc, view)).to(ctx.device)
    img = _image(ctx, arrays, d)
    small = _image(ctx, arrays, d[:, :-1].contiguous())      # one column narrower
    short = _image(ctx, arrays, d[:-1].contiguous())         # one row shorter
    ds = frame.DeviceScene.upload(ctx, sc, lights=scenes.make_lights(1, 16, sc.aabb_min, sc.aabb_max))
    vs = frame.ViewState(ctx, ds, (view.width, view.height), name="dimg_bad")
    pf = frame.PreparedFrame(ctx, ds, vs, view, img, name="dimg_bad", main_pass=True)
    assert pf.fused and pf.image
    pf.launch(); torch.cuda.synchronize()
    st = ClusterSettings(screen_resolution=(view.width, view.height))
    info, params = compute_clusters(ctx, st, view.view, view.projection_matrix, view.near, img, ds.scene, name="dimg_bad_cl")
    torch.cuda.synchronize()
    before = F._bytes(pf)
    before_cl = [t.cpu().numpy().copy() for t in (info.tile_depth_slice_mask, info.cluster_depth_bounds, info.unique_cluster_buffer,
                                                    info.light_offset_image, info.light_index_buffer)]
    n0 = lib.orbit_ctx_launch_count(ctx._h)
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    hiz = vs.depth_pyramid._h
    other = DepthPyramid(ctx, "dimg_bad_other", (view.width, view.height))
    late_d, main_d = _ptr(pf.late_dispatch), _ptr(pf.main_dispatch)

    # orbit_hiz_build_image
    for what, args in {"no context": (None, hiz, img._h), "no pyramid": (ctx._h, None, img._h), "no image": (ctx._h, hiz, None),
                       "narrower image": (ctx._h, hiz, small._h), "shorter image": (ctx._h, hiz, short._h)}.items():
        assert lib.orbit_hiz_build_image(*args, s) == _lib.ERR_INVALID_ARGUMENT, what

    # orbit_hiz_build_views_image
    def views(hs, ims, n=None):
        n = len(hs) if n is None else n
        return lib.orbit_hiz_build_views_image(ctx._h, (C.c_void_p * len(hs))(*[h.value if h else None for h in hs]),
                                               (C.c_void_p * len(ims))(*[i._h.value if i else None for i in ims]), n, s)
    for what, (hs, ims, n) in {"no views": ([hiz], [img], 0), "too many": ([hiz], [img], L.MAX_BATCH_VIEWS + 1),
                               "NULL image slot": ([hiz, other._h], [img, None], None), "NULL first image": ([hiz, other._h], [None, img], None),
                               "NULL pyramid slot": ([hiz, None], [img, img], None), "shared pyramid": ([hiz, hiz], [img, img], None),
                               "narrower image": ([hiz, other._h], [img, small], None), "shorter image": ([hiz, other._h], [short, short], None)}.items():
        if n is not None and n > len(hs):
            hs, ims = hs * n, ims * n
        assert views(hs, ims, n) == _lib.ERR_INVALID_ARGUMENT, what
    assert lib.orbit_hiz_build_views_image(ctx._h, None, None, 1, s) == _lib.ERR_INVALID_ARGUMENT

    # orbit_hiz_build_image_entity_cull_late: the image rules and every rule of the linear fused call
    def fused(ctx_h=ctx._h, hiz=hiz, image=img._h, late=None, main=None, sb=None, ld=late_d, md=main_d):
        gl = late if late is not None else L.CullInfo.from_buffer_copy(pf.g_late)
        gm = main if main is not None else L.CullInfo.from_buffer_copy(pf.g_early)
        b = sb if sb is not None else L.SceneBuffers.from_buffer_copy(pf.sb_late)
        return lib.orbit_hiz_build_image_entity_cull_late(ctx_h, hiz, image, None if late is False else C.byref(gl),
                                                          None if main is False else C.byref(gm), C.byref(b), ld, md, pf.rcap, s)

    def edited(src, **kw):
        g = type(src).from_buffer_copy(src)
        for k, v in kw.items():
            setattr(g, k, v)
        return g
    bad = {
        "no context": dict(ctx_h=None), "no pyramid": dict(hiz=None), "no image": dict(image=None),
        "narrower image": dict(image=small._h), "shorter image": dict(image=short._h), "no late CullInfo": dict(late=False),
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
        assert fused(**kw) == _lib.ERR_INVALID_ARGUMENT, what

    # orbit_light_cluster_image: screen_size must be the image's size
    bufs = [_ptr(t) for t in (info.tile_depth_slice_mask, info.cluster_depth_bounds, info.unique_cluster_buffer, info.light_offset_image,
                              info.light_index_buffer)]
    cap = (info.light_index_buffer.numel() - 4) // 4
    lights = _ptr(ds.scene.light_data_buffer)
    for what, image in {"no image": None, "narrower image": small._h, "shorter image": short._h}.items():
        assert lib.orbit_light_cluster_image(ctx._h, C.byref(params), image, lights, *bufs, cap, s) == _lib.ERR_INVALID_ARGUMENT, what
    assert lib.orbit_light_cluster_image(None, C.byref(params), img._h, lights, *bufs, cap, s) == _lib.ERR_INVALID_ARGUMENT

    torch.cuda.synchronize()
    assert lib.orbit_ctx_launch_count(ctx._h) == n0
    F._assert_same(before, F._bytes(pf), "after the refused calls")
    after_cl = [t.cpu().numpy() for t in (info.tile_depth_slice_mask, info.cluster_depth_bounds, info.unique_cluster_buffer,
                                          info.light_offset_image, info.light_index_buffer)]
    for a, b in zip(before_cl, after_cl):
        assert np.array_equal(a, b)
    assert fused() == 0 and lib.orbit_ctx_launch_count(ctx._h) == n0 + 2     # the valid call: two launches
    assert lib.orbit_hiz_build_image(ctx._h, hiz, img._h, s) == 0 and lib.orbit_ctx_launch_count(ctx._h) == n0 + 3
    torch.cuda.synchronize()
    for i in (img, small, short):
        i.close()
