"""GPU: outputs written into CUDA arrays, the form the renderer's Vulkan images take once imported (orbit_cuda.h, "outputs into
images"). A pyramid with a mirror (orbit_hiz_attach_image) stores every level into its mipmapped array byte for byte as the
linear level, and its linear pyramid stays what an unmirrored pyramid's is; orbit_light_cluster_image_grid writes the cluster
offset/count grid into a 3-D R32G32_UINT array byte for byte as orbit_light_cluster_image writes its buffer.

The arrays are made through cudart (cudaMallocMipmappedArray / cudaMalloc3DArray with cudaArraySurfaceLoadStore), pre-filled
with 0xFFFFFFFF so that a texel nobody wrote shows, and read back with cudaMemcpy2DFromArrayAsync per level and cudaMemcpy3DAsync.
Cases: pyramids at the sizes of test_hiz_bit_exact from a depth tensor and from a DepthImage (against an unmirrored pyramid and
the oracle); the batched build with 1, 4 and 16 pyramids, mirrored and not, in both depth forms; the fused Hi-Z + LATE entity
call and the C2 frame through PreparedFrame (moving camera, MAIN present and absent, a CUDA graph replayed over alternating scene
copies, ORBIT_NO_PDL=1 in a subprocess); four cameras through PreparedViews; the cluster grid on both light-culling paths, run
three times over different depths; and every refusal on a real context."""
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
sys.path.insert(0, os.path.join(ROOT, "tests"))

from test_gpu_depth_image import KIND_FLOAT, KIND_UNSIGNED, MEMCPY_D2D, Arrays, _Desc, _Extent, _image, _random_depth  # noqa: E402

ARRAY_LAYERED, ARRAY_SURFACE_LDST = 0x01, 0x02      # cudaArrayLayered, cudaArraySurfaceLoadStore
GARBAGE = -1                                         # as int32: 0xFFFFFFFF, a texel nobody wrote


class _Pos(C.Structure):
    _fields_ = [("x", C.c_size_t), ("y", C.c_size_t), ("z", C.c_size_t)]


class _PitchedPtr(C.Structure):
    _fields_ = [("ptr", C.c_void_p), ("pitch", C.c_size_t), ("xsize", C.c_size_t), ("ysize", C.c_size_t)]


class _Memcpy3DParms(C.Structure):
    _fields_ = [("srcArray", C.c_void_p), ("srcPos", _Pos), ("srcPtr", _PitchedPtr),
                ("dstArray", C.c_void_p), ("dstPos", _Pos), ("dstPtr", _PitchedPtr), ("extent", _Extent), ("kind", C.c_int)]


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


class Images(Arrays):
    """Arrays of test_gpu_depth_image plus the output images: mipmapped pyramid arrays and 3-D cluster grids."""

    def mipmapped(self, w, h, levels, flags=ARRAY_SURFACE_LDST, bits=(32, 0, 0, 0), kind=KIND_FLOAT, layers=0):
        mm = C.c_void_p()
        self._ck(self.rt.cudaMallocMipmappedArray(C.byref(mm), C.byref(_Desc(*bits, kind)), _Extent(w, h, layers), C.c_uint(levels),
                                                  C.c_uint(flags)), "cudaMallocMipmappedArray")
        self.mipmaps.append(mm.value)
        return mm.value

    def pyramid_array(self, info):
        """A mipmapped array with exactly the pyramid's levels, one float channel, surface load/store, filled with garbage."""
        mm = self.mipmapped(info.width, info.height, info.levels)
        self.spoil(mm, info)
        return mm

    def spoil(self, mm, info):
        """Every level of the pyramid array to 0xFFFFFFFF."""
        for l in range(info.levels):
            self.fill_level(mm, l, torch.full((max(info.height >> l, 1), max(info.width >> l, 1)), GARBAGE, dtype=torch.int32, device="cuda"))

    def level(self, mm, l):
        a = C.c_void_p()
        self._ck(self.rt.cudaGetMipmappedArrayLevel(C.byref(a), C.c_void_p(mm), C.c_uint(l)), "cudaGetMipmappedArrayLevel")
        return a.value

    def fill_level(self, mm, l, values):
        self.fill(self.level(mm, l), values)

    def read_level(self, mm, l, w, h):
        """Level l (w x h texels of 4 bytes) as a uint32 numpy array [h, w]."""
        out = torch.empty((h, w), dtype=torch.int32, device="cuda")
        self._ck(self.rt.cudaMemcpy2DFromArrayAsync(C.c_void_p(out.data_ptr()), C.c_size_t(4 * w), C.c_void_p(self.level(mm, l)),
                                                    C.c_size_t(0), C.c_size_t(0), C.c_size_t(4 * w), C.c_size_t(h), C.c_int(MEMCPY_D2D),
                                                    _stream()), "cudaMemcpy2DFromArrayAsync")
        torch.cuda.synchronize()
        return out.cpu().numpy().view(np.uint32)

    def grid(self, cx, cy, cz, flags=ARRAY_SURFACE_LDST, bits=(32, 32, 0, 0), kind=KIND_UNSIGNED):
        a = C.c_void_p()
        self._ck(self.rt.cudaMalloc3DArray(C.byref(a), C.byref(_Desc(*bits, kind)), _Extent(cx, cy, cz), C.c_uint(flags)), "cudaMalloc3DArray")
        self.arrays.append(a.value)
        return a.value

    def _copy3d(self, arr, t, cx, cy, cz, to_array):
        p = _Memcpy3DParms()
        lin = _PitchedPtr(t.data_ptr(), 8 * cx, 8 * cx, cy)
        if to_array:
            p.srcPtr, p.dstArray = lin, arr
        else:
            p.srcArray, p.dstPtr = arr, lin
        p.extent = _Extent(cx, cy, cz)
        p.kind = MEMCPY_D2D
        self._ck(self.rt.cudaMemcpy3DAsync(C.byref(p), _stream()), "cudaMemcpy3DAsync")

    def fill_grid(self, arr, cx, cy, cz, word=GARBAGE):
        self._copy3d(arr, torch.full((cz, cy, cx, 2), word, dtype=torch.int32, device="cuda"), cx, cy, cz, True)

    def read_grid(self, arr, cx, cy, cz):
        """The grid as uint32 words in the linear buffer's order: texel (x, y, z) at words 2 idx, 2 idx + 1, idx = (z cy + y) cx + x."""
        out = torch.empty(2 * cx * cy * cz, dtype=torch.int32, device="cuda")
        self._copy3d(arr, out, cx, cy, cz, False)
        torch.cuda.synchronize()
        return out.cpu().numpy().view(np.uint32)


@pytest.fixture(scope="module")
def images(gpu_context):
    a = Images(gpu_context.device)
    yield a
    a.free()


def _u32(t):
    return t.cpu().numpy().view(np.uint32)


def _geometry(w, h):
    from orbit_b200 import _lib, layouts as L
    info = L.HizInfo()
    _lib.check(_lib.lib().orbit_hiz_geometry(w, h, C.byref(info)), "orbit_hiz_geometry")
    return info


def assert_mirror(images, pyramid, mm, what=""):
    """Every level of the array equals the pyramid's linear level, byte for byte."""
    info = pyramid.info
    for l in range(info.levels):
        w, h = max(info.width >> l, 1), max(info.height >> l, 1)
        assert np.array_equal(images.read_level(mm, l, w, h), _u32(pyramid.level(l))), (what, "level", l)


# ---- pyramids ------------------------------------------------------------------------------------------------------------
SIZES = [(1920, 1080), (3840, 2160), (1280, 720), (100, 60), (64, 64), (129, 257), (2, 2), (4096, 33)]


@pytest.mark.parametrize("form", ["tensor", "image"])
@pytest.mark.parametrize("size", SIZES, ids=["%dx%d" % s for s in SIZES])
def test_mirror_equals_linear_and_oracle(gpu_context, images, oracle, size, form):
    from orbit_b200.passes import DepthPyramid
    ctx = gpu_context
    w, h = size
    depth = _random_depth(w, h)
    d = torch.from_numpy(depth).to(ctx.device)
    src = _image(ctx, images, d) if form == "image" else d
    plain = DepthPyramid(ctx, "oimg_plain", (w, h))
    mm = images.pyramid_array(plain.info)
    mirrored = DepthPyramid(ctx, "oimg_mirrored", (w, h), image=mm)
    mirrored.texels.fill_(-1.0)
    plain.update(src)
    mirrored.update(src)
    torch.cuda.synchronize()
    _, ref = oracle.hiz_build(depth)
    assert np.array_equal(_u32(mirrored.texels), _u32(plain.texels))
    assert np.array_equal(_u32(mirrored.texels), ref.view(np.uint32))
    assert_mirror(images, mirrored, mm, size)


@pytest.mark.parametrize("form", ["tensor", "image"])
@pytest.mark.parametrize("n", [1, 4, 16])
@pytest.mark.parametrize("size", [(1920, 1080), (100, 60)], ids=["1920x1080", "100x60"])
def test_batched_build_mixed_mirrors(gpu_context, images, size, n, form):
    """Pyramids 0, 2, 4, .. have a mirror, the others not; the mirrored ones' arrays equal their linear levels and every linear
    pyramid equals the unmirrored batch's."""
    from orbit_b200 import frame
    from orbit_b200.passes import DepthPyramid
    ctx = gpu_context
    w, h = size
    ds = [torch.from_numpy(np.roll(_random_depth(w, h), 7 * v, axis=1)).to(ctx.device) for v in range(n)]
    srcs = [_image(ctx, images, d) for d in ds] if form == "image" else ds
    plain = [DepthPyramid(ctx, "oimgv_plain%d" % v, (w, h)) for v in range(n)]
    mms = {v: images.pyramid_array(plain[0].info) for v in range(0, n, 2)}
    mixed = [DepthPyramid(ctx, "oimgv_mixed%d" % v, (w, h), image=mms.get(v)) for v in range(n)]
    s = _stream()
    frame._HizViews(ctx, plain, srcs).launch(s)
    frame._HizViews(ctx, mixed, srcs).launch(s)
    torch.cuda.synchronize()
    for v in range(n):
        assert np.array_equal(_u32(mixed[v].texels), _u32(plain[v].texels)), v
        if v in mms:
            assert_mirror(images, mixed[v], mms[v], ("view", v))


# ---- the fused call and frames -------------------------------------------------------------------------------------------
def _fused():
    import test_gpu_hiz_entity_fused as F      # the comparison helpers of the fused call's parity test
    return F


def _frames(ctx, images, ds, view, src, tag, main_pass):
    """Two PreparedFrames of one view and scene with their own bitmasks and buffers: pyramid unmirrored / mirrored."""
    from orbit_b200 import frame
    mm = images.pyramid_array(_geometry(view.width, view.height))
    out = []
    for form, image in (("plain", None), ("mirrored", mm)):
        vs = frame.ViewState(ctx, ds, (view.width, view.height), name="oimg_%s_%s" % (tag, form), pyramid_image=image)
        out.append(frame.PreparedFrame(ctx, ds, vs, view, src, name="oimg_%s_%s" % (tag, form), main_pass=main_pass))
    return out[0], out[1], mm


def _status(ctx):
    code, st = ctx.poll_status()
    return code, bytes(st)


def run_frames(ctx, images, main_pass, form):
    """Frames A, A, B, A of C2 through PreparedFrame.launch (the fused orbit_hiz_build(_image)_entity_cull_late), unmirrored and
    mirrored: dispatch and draw buffers, bitmasks, pyramid and status equal after each frame, and the mirror equals the pyramid."""
    from orbit_b200 import frame
    import bench
    F = _fused()
    sc, _ = scenes.config_c2()
    view_a, view_b = bench.c2_view(scenes, sc, 0), bench.c2_view(scenes, sc, 4)
    ds = frame.DeviceScene.upload(ctx, sc)
    d_a = torch.from_numpy(scenes.make_depth(sc, view_a)).to(ctx.device)
    d_b = torch.from_numpy(scenes.make_depth(sc, view_b)).to(ctx.device)
    s_a, s_b = (_image(ctx, images, d_a), _image(ctx, images, d_b)) if form == "image" else (d_a, d_b)
    plain, mirrored, mm = _frames(ctx, images, ds, view_a, s_a, "f%d%s" % (main_pass, form), main_pass)
    assert plain.fused == mirrored.fused == main_pass
    plain_b, mirrored_b = F._retarget(ctx, plain, view_b, s_b, main_pass), F._retarget(ctx, mirrored, view_b, s_b, main_pass)
    late_records = []
    _status(ctx)
    for i, (a, b) in enumerate([(plain, mirrored), (plain, mirrored), (plain_b, mirrored_b), (plain, mirrored)]):
        a.launch()
        torch.cuda.synchronize()
        st_a = _status(ctx)
        b.launch()
        torch.cuda.synchronize()
        assert _status(ctx) == st_a, (main_pass, form, i, "status")
        x, y = F._bytes(a), F._bytes(b)
        F._assert_same(x, y, (main_pass, form, i))
        assert_mirror(images, b.vstate.depth_pyramid, mm, (main_pass, form, i))
        late_records.append(int(x["late_dispatch"][0]))
    return late_records


@pytest.mark.parametrize("form", ["tensor", "image"])
@pytest.mark.parametrize("main_pass", [True, False], ids=["main", "no_main"])
def test_frame_with_mirrored_pyramid(gpu_context, images, main_pass, form):
    late = run_frames(gpu_context, images, main_pass, form)
    assert late[0] > 0, late


def test_graph_replays_write_the_mirror(gpu_context, images):
    """Two scene copies, each an (unmirrored, mirrored) PreparedFrame pair captured into CUDA graphs; 24 replays alternate between
    the copies and between two depth buffers. Before every replay the mirror is overwritten with garbage: the replay writes it."""
    from orbit_b200 import frame
    import bench
    F = _fused()
    ctx = gpu_context
    sc, view = scenes.config_c2(scale=0.25)
    srcs = [torch.from_numpy(scenes.make_depth(sc, v)).to(ctx.device) for v in (view, bench.c2_view(scenes, sc, 1))]
    pairs = []
    for i in range(2):
        d = srcs[0].clone()
        plain, mirrored, mm = _frames(ctx, images, frame.DeviceScene.upload(ctx, sc), view, d, "graph%d" % i, True)
        plain.capture(); mirrored.capture()
        pairs.append((plain, mirrored, d, mm))
    info = pairs[0][1].vstate.depth_pyramid.info
    for r in range(24):
        plain, mirrored, d, mm = pairs[r % 2]
        d.copy_(srcs[(r // 2) % 2])
        images.spoil(mm, info)
        plain.replay(); mirrored.replay()
        torch.cuda.synchronize()
        F._assert_same(F._bytes(plain), F._bytes(mirrored), ("replay", r))
        assert_mirror(images, mirrored.vstate.depth_pyramid, mm, ("replay", r))


def test_without_pdl_in_a_subprocess(gpu_context):
    env = dict(os.environ, ORBIT_NO_PDL="1")
    code = ("import sys; sys.path.insert(0, %r); sys.path.insert(0, %r)\n"
            "import test_gpu_output_images as t\n"
            "from orbit_b200.passes import Context\n"
            "ctx = Context(0)\n"
            "images = t.Images(ctx.device)\n"
            "for m in (True, False): print(t.run_frames(ctx, images, m, 'tensor'))\n"
            "images.free()\n"
            "ctx.close()\n" % (ROOT, os.path.join(ROOT, "tests")))
    res = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stdout + res.stderr


def test_batched_cameras_with_mirrors(gpu_context, images):
    """PreparedViews of four C2 cameras (EARLY, batched Hi-Z, LATE, MAIN) with mirrored pyramids equals the same frame without."""
    from orbit_b200 import frame
    import bench
    ctx = gpu_context
    sc, _ = scenes.config_c2()
    views = [bench.c2_view(scenes, sc, i) for i in range(4)]
    ds = frame.DeviceScene.upload(ctx, sc)
    depths = [torch.from_numpy(scenes.make_depth(sc, v)).to(ctx.device) for v in views]
    out, mms = [], []
    for form in ("plain", "mirrored"):
        vs = []
        for i, v in enumerate(views):
            mm = None
            if form == "mirrored":
                mm = images.pyramid_array(_geometry(v.width, v.height))
                mms.append(mm)
            vs.append(frame.ViewState(ctx, ds, (v.width, v.height), name="oimg_pv_%s%d" % (form, i), pyramid_image=mm))
        out.append((frame.PreparedViews(ctx, ds, vs, views, depths, name="oimg_pv_" + form), vs))
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
            assert_mirror(images, vb[v].depth_pyramid, mms[v], (f, v))


# ---- cluster grid --------------------------------------------------------------------------------------------------------
KEYS = ("tile_depth_slice_mask", "cluster_depth_bounds", "unique_cluster_buffer", "light_index_buffer")


def _cluster_case(case):
    """(scene, view, depth, lights, settings) of a cluster case."""
    from orbit_b200.passes import ClusterSettings
    if case in ("c4_reduced", "no_lights"):
        sc, view = scenes.config_c4(scale=0.02)
        lights = scenes.make_lights(scenes.SEEDS["C4"], 4096, sc.aabb_min, sc.aabb_max) if case == "c4_reduced" else None
        return sc, view, scenes.make_depth(sc, view), lights, ClusterSettings(screen_resolution=(1920, 1080), z_slice_count=24, tile_size_px=120)
    sc, _ = scenes.config_c4(scale=0.005)
    if case == "default_cap":         # reference defaults: 8 px tiles, 32 slices; hits the 256 cap
        view = scenes.perspective_view((-6.0, 3.0, -6.0), (0.6, 0.0, 0.8), 320, 180)
        lights = scenes.make_lights(scenes.SEEDS["C4"] + 1, 3000, sc.aabb_min * 0.3, sc.aabb_max * 0.3, intensity=(20.0, 60.0))
        return sc, view, scenes.make_depth(sc, view), lights, ClusterSettings(screen_resolution=(320, 180))
    if case == "sky":                 # all sky: no active cluster
        view = scenes.perspective_view((-6.0, 3.0, -6.0), (0.6, 0.0, 0.8), 256, 128)
        return sc, view, np.zeros((128, 256), np.float32), scenes.make_lights(1, 16, sc.aabb_min, sc.aabb_max), ClusterSettings(screen_resolution=(256, 128))
    raise ValueError(case)


def run_grid_case(ctx, images, case):
    """The case's depth, then its rows flipped, then all sky, into one DepthImage and one grid (filled with garbage once, before
    the first run): after every run the grid equals orbit_light_cluster_image's buffer and every other output is the same.
    Returns (active clusters, light indices, largest per-cluster count) of each run."""
    from orbit_b200 import frame
    from orbit_b200.passes import ClusterGridImage, DepthImage, compute_clusters
    sc, view, depth, lights, st = _cluster_case(case)
    ds = frame.DeviceScene.upload(ctx, sc, lights=lights)
    assert ds.scene.light_count == (0 if lights is None else len(lights))
    cx, cy, cz = st.cluster_counts()
    h, w = depth.shape
    arr = images.array(w, h)
    img = DepthImage(ctx, arr)
    garr = images.grid(cx, cy, cz)
    images.fill_grid(garr, cx, cy, cz)
    grid = ClusterGridImage(ctx, garr)
    stats = []
    for run, dv in enumerate((depth, np.ascontiguousarray(depth[::-1]), np.zeros_like(depth))):
        images.fill(arr, torch.from_numpy(dv).to(ctx.device))
        lin, _ = compute_clusters(ctx, st, view.view, view.projection_matrix, view.near, img, ds.scene, name="oimg_cl_lin")
        out, _ = compute_clusters(ctx, st, view.view, view.projection_matrix, view.near, img, ds.scene, name="oimg_cl_grid",
                                  light_offset_image=grid)
        torch.cuda.synchronize()
        assert out.light_offset_image is grid
        for k in KEYS:
            assert np.array_equal(getattr(lin, k).cpu().numpy(), getattr(out, k).cpu().numpy()), (case, run, k)
        want = lin.light_offset_image[:8 * cx * cy * cz].cpu().numpy().view(np.uint32)
        got = images.read_grid(garr, cx, cy, cz)
        assert np.array_equal(got, want), (case, run, "grid")
        stats.append((int(_u32(lin.unique_cluster_buffer)[3]), int(_u32(lin.light_index_buffer)[0]), int(want[1::2].max())))
    img.close(); grid.close()
    return stats


CASES = ["c4_reduced", "default_cap", "sky", "no_lights"]


def _check_stats(case, stats):
    first = stats[0]
    if case == "c4_reduced":
        assert first[0] > 0 and first[1] > 0, stats
    elif case == "default_cap":
        assert first[2] == 256, stats
    elif case == "sky":
        assert first[0] == 0 and first[1] == 0, stats
    elif case == "no_lights":
        assert first[0] > 0 and first[1] == 0, stats
    assert stats[2][0] == 0, stats      # the all-sky run leaves no active cluster: every texel went back to (0, 0)


@pytest.mark.parametrize("case", CASES)
def test_grid_light_parallel_path(gpu_context, images, case):
    _check_stats(case, run_grid_case(gpu_context, images, case))


@pytest.mark.parametrize("case", CASES)
def test_grid_cta_per_cluster_path(case):
    """The same on the CTA-per-cluster kernel, forced with a zero bit-matrix budget in a process of its own."""
    env = dict(os.environ, ORBIT_LIGHT_HITS_BUDGET_MB="0")
    code = ("import sys; sys.path.insert(0, %r); sys.path.insert(0, %r)\n"
            "import test_gpu_output_images as t\n"
            "from orbit_b200.passes import Context\n"
            "ctx = Context(0)\n"
            "images = t.Images(ctx.device)\n"
            "t._check_stats(%r, t.run_grid_case(ctx, images, %r))\n"
            "images.free()\n"
            "ctx.close()\n" % (ROOT, os.path.join(ROOT, "tests"), case, case))
    res = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stdout + res.stderr


# ---- refusals ------------------------------------------------------------------------------------------------------------
def test_refusals_launch_nothing(gpu_context, images):
    """Every refused attach, batched build, grid wrap and grid call: ORBIT_ERR_INVALID_ARGUMENT and no launch. A refused attach
    leaves no CUDA error behind (the next stage calls, which check cudaGetLastError after their launches, succeed)."""
    from orbit_b200 import _lib, frame
    from orbit_b200.passes import ClusterGridImage, ClusterSettings, DepthImage, DepthPyramid, compute_clusters
    ctx, lib = gpu_context, _lib.lib()
    w, h = 640, 360
    pyr = DepthPyramid(ctx, "oimg_bad", (w, h))
    info = pyr.info                                           # 512 x 256, 10 levels
    n0 = lib.orbit_ctx_launch_count(ctx._h)
    bad = {
        "wider level 0": images.mipmapped(2 * info.width, info.height, info.levels),
        "taller level 0": images.mipmapped(info.width, 2 * info.height, info.levels),
        "too few levels": images.mipmapped(info.width, info.height, info.levels - 1),
        "float2 format": images.mipmapped(info.width, info.height, info.levels, bits=(32, 32, 0, 0)),
        "half format": images.mipmapped(info.width, info.height, info.levels, bits=(16, 0, 0, 0)),
        "uint32 kind": images.mipmapped(info.width, info.height, info.levels, kind=KIND_UNSIGNED),
        "no surface flag": images.mipmapped(info.width, info.height, info.levels, flags=0),
        "layered": images.mipmapped(info.width, info.height, info.levels, flags=ARRAY_LAYERED | ARRAY_SURFACE_LDST, layers=2),
    }
    for what, mm in bad.items():
        assert lib.orbit_hiz_attach_image(ctx._h, pyr._h, C.c_void_p(mm)) == _lib.ERR_INVALID_ARGUMENT, what
    good = images.pyramid_array(info)
    assert lib.orbit_hiz_attach_image(ctx._h, pyr._h, C.c_void_p(good)) == _lib.OK
    assert lib.orbit_hiz_attach_image(ctx._h, pyr._h, C.c_void_p(images.pyramid_array(info))) == _lib.ERR_INVALID_ARGUMENT, "second attach"
    assert lib.orbit_hiz_attach_image(ctx._h, pyr._h, C.c_void_p(good)) == _lib.ERR_INVALID_ARGUMENT, "second attach, same array"

    # the same array on two pyramids of one batched call (each attach alone is fine)
    other = DepthPyramid(ctx, "oimg_bad_other", (w, h))
    assert lib.orbit_hiz_attach_image(ctx._h, other._h, C.c_void_p(good)) == _lib.OK
    d = torch.zeros((h, w), dtype=torch.float32, device=ctx.device)
    hizs = (C.c_void_p * 2)(pyr._h.value, other._h.value)
    depths = (C.c_void_p * 2)(d.data_ptr(), d.data_ptr())
    s = _stream()
    assert lib.orbit_hiz_build_views(ctx._h, hizs, depths, 2, w, h, s) == _lib.ERR_INVALID_ARGUMENT, "shared mirror"
    depth_arr = images.array(w, h)
    images.fill(depth_arr, d)
    img = DepthImage(ctx, depth_arr)
    imgs = (C.c_void_p * 2)(img._h.value, img._h.value)
    assert lib.orbit_hiz_build_views_image(ctx._h, hizs, imgs, 2, s) == _lib.ERR_INVALID_ARGUMENT, "shared mirror, image"

    # grids: the wrap takes only 3-D two-channel uint32 arrays with surface load/store
    st = ClusterSettings(screen_resolution=(w, h))
    cx, cy, cz = st.cluster_counts()
    bad_grids = {
        "2-D": images.grid(cx, cy, 0), "one channel": images.grid(cx, cy, cz, bits=(32, 0, 0, 0)),
        "four channels": images.grid(cx, cy, cz, bits=(32, 32, 32, 32)), "float kind": images.grid(cx, cy, cz, kind=KIND_FLOAT),
        "16-bit channels": images.grid(cx, cy, cz, bits=(16, 16, 0, 0)), "no surface flag": images.grid(cx, cy, cz, flags=0),
        "layered": images.grid(cx, cy, cz, flags=ARRAY_LAYERED | ARRAY_SURFACE_LDST),
    }
    for what, arr in bad_grids.items():
        out = C.c_void_p(1234)
        assert lib.orbit_cluster_grid_wrap(ctx._h, C.c_void_p(arr), C.byref(out)) == _lib.ERR_INVALID_ARGUMENT, what
        assert out.value is None, what
    # a grid whose extent differs from cluster_count, on a valid call otherwise
    sc, _ = scenes.config_c4(scale=0.005)
    ds = frame.DeviceScene.upload(ctx, sc, lights=scenes.make_lights(1, 16, sc.aabb_min, sc.aabb_max))
    view = scenes.perspective_view((-6.0, 3.0, -6.0), (0.6, 0.0, 0.8), w, h)
    for what, ext in {"narrower": (cx - 1, cy, cz), "shorter": (cx, cy - 1, cz), "fewer slices": (cx, cy, cz - 1),
                      "more slices": (cx, cy, cz + 1)}.items():
        g = ClusterGridImage(ctx, images.grid(*ext))
        with pytest.raises(_lib.OrbitError):
            compute_clusters(ctx, st, view.view, view.projection_matrix, view.near, img, ds.scene, name="oimg_bad_cl", light_offset_image=g)
        g.close()
    with pytest.raises(TypeError):
        compute_clusters(ctx, st, view.view, view.projection_matrix, view.near, d, ds.scene, name="oimg_bad_cl",
                         light_offset_image=ClusterGridImage(ctx, images.grid(cx, cy, cz)))
    torch.cuda.synchronize()
    assert lib.orbit_ctx_launch_count(ctx._h) == n0

    # the valid calls after all of that: no CUDA error was left behind
    g = ClusterGridImage(ctx, images.grid(cx, cy, cz))
    compute_clusters(ctx, st, view.view, view.projection_matrix, view.near, img, ds.scene, name="oimg_bad_cl", light_offset_image=g)
    pyr.update(d)
    torch.cuda.synchronize()
    assert lib.orbit_ctx_launch_count(ctx._h) > n0
    assert_mirror(images, pyr, good, "after the refusals")
    g.close(); img.close()
