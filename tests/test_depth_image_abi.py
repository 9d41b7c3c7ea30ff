"""CPU: the depth-image entry points (orbit_depth_image_* and the *_image stage variants) are declared in the C header,
exported with the prototypes of _lib.py, and refuse a NULL context, pyramid or image (and a NULL slot of the batched call's
image array) before they use the context or a device. Handles here are zero-filled stand-ins: refused calls must return
before touching them, and orbit_hiz_wrap only reads the context's device number."""
import ctypes as C
import os
import re

import pytest

from orbit_b200 import _lib
from orbit_b200 import layouts as L

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = ["orbit_depth_image_wrap", "orbit_depth_image_destroy", "orbit_depth_image_size", "orbit_hiz_build_image",
         "orbit_hiz_build_views_image", "orbit_hiz_build_image_entity_cull_late", "orbit_light_cluster_image"]


@pytest.mark.parametrize("name", NAMES)
def test_declared_in_the_header_and_exported(name):
    hdr = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "orbit_cuda.h")).read(), flags=re.S)
    m = re.search(r"\b(?:int|void)\s+%s\s*\(([^;]*)\)\s*;" % name, hdr)
    assert m, name
    assert getattr(_lib.lib(), name) is not None
    assert len(m.group(1).split(",")) == len(_lib.PROTOTYPES[name][1])


@pytest.fixture
def handles():
    lib = _lib.lib()
    fake_ctx = C.create_string_buffer(1 << 16)                 # zero-filled: device 0
    fake_img = C.create_string_buffer(64)
    ctx, img = C.c_void_p(C.addressof(fake_ctx)), C.c_void_p(C.addressof(fake_img))
    hiz = C.c_void_p()
    assert lib.orbit_hiz_wrap(ctx, 640, 360, C.c_void_p(1 << 20), C.byref(hiz)) == _lib.OK
    yield lib, ctx, hiz, img
    lib.orbit_hiz_destroy(hiz)
    del fake_ctx, fake_img


def test_wrap_refuses_null_arguments(handles):
    lib, ctx, _, _ = handles
    out = C.c_void_p(1234)
    assert lib.orbit_depth_image_wrap(None, C.c_void_p(1 << 20), C.byref(out)) == _lib.ERR_INVALID_ARGUMENT
    assert out.value is None                                    # *out is cleared on refusal
    assert lib.orbit_depth_image_wrap(ctx, None, C.byref(out)) == _lib.ERR_INVALID_ARGUMENT
    assert lib.orbit_depth_image_wrap(ctx, C.c_void_p(1 << 20), None) == _lib.ERR_INVALID_ARGUMENT
    w, h = C.c_uint32(), C.c_uint32()
    assert lib.orbit_depth_image_size(None, C.byref(w), C.byref(h)) == _lib.ERR_INVALID_ARGUMENT
    lib.orbit_depth_image_destroy(None)


def test_hiz_build_image_refuses_null_handles(handles):
    lib, ctx, hiz, img = handles
    assert lib.orbit_hiz_build_image(None, hiz, img, None) == _lib.ERR_INVALID_ARGUMENT
    assert lib.orbit_hiz_build_image(ctx, None, img, None) == _lib.ERR_INVALID_ARGUMENT
    assert lib.orbit_hiz_build_image(ctx, hiz, None, None) == _lib.ERR_INVALID_ARGUMENT


def test_hiz_build_views_image_refuses_null_handles(handles):
    lib, ctx, hiz, img = handles
    hizs = (C.c_void_p * 2)(hiz.value, hiz.value)
    imgs = (C.c_void_p * 2)(img.value, img.value)
    assert lib.orbit_hiz_build_views_image(None, hizs, imgs, 2, None) == _lib.ERR_INVALID_ARGUMENT
    assert lib.orbit_hiz_build_views_image(ctx, None, imgs, 2, None) == _lib.ERR_INVALID_ARGUMENT
    assert lib.orbit_hiz_build_views_image(ctx, hizs, None, 2, None) == _lib.ERR_INVALID_ARGUMENT
    assert lib.orbit_hiz_build_views_image(ctx, hizs, imgs, 0, None) == _lib.ERR_INVALID_ARGUMENT
    assert lib.orbit_hiz_build_views_image(ctx, hizs, imgs, L.MAX_BATCH_VIEWS + 1, None) == _lib.ERR_INVALID_ARGUMENT
    for slot in range(2):
        bad = (C.c_void_p * 2)(img.value, img.value)
        bad[slot] = None
        assert lib.orbit_hiz_build_views_image(ctx, hizs, bad, 2, None) == _lib.ERR_INVALID_ARGUMENT, slot
        bad_hiz = (C.c_void_p * 2)(hiz.value, hiz.value)
        bad_hiz[slot] = None
        assert lib.orbit_hiz_build_views_image(ctx, bad_hiz, imgs, 2, None) == _lib.ERR_INVALID_ARGUMENT, slot


def test_hiz_build_image_entity_cull_late_refuses_null_handles(handles):
    lib, ctx, hiz, img = handles
    late = L.CullInfo()
    late.occlusion_pass = 2
    late.visibility_buffer = late.meshlet_visibility_buffer = 0
    sb = L.SceneBuffers()
    sb.entity_draws, sb.mesh_infos, sb.entities, sb.entity_visibility = 1 << 20, 2 << 20, 3 << 20, 4 << 20
    sb.entity_draw_count = 1000

    def call(c=ctx, h=hiz, i=img):
        return lib.orbit_hiz_build_image_entity_cull_late(c, h, i, C.byref(late), None, C.byref(sb), C.c_void_p(5 << 20), None, 1000, None)
    assert call(c=None) == _lib.ERR_INVALID_ARGUMENT
    assert call(h=None) == _lib.ERR_INVALID_ARGUMENT
    assert call(i=None) == _lib.ERR_INVALID_ARGUMENT


def test_light_cluster_image_refuses_null_handles(handles):
    lib, ctx, _, img = handles
    p = L.ClusterParams()
    p.info.cluster_count[0], p.info.cluster_count[1], p.info.cluster_count[2] = 16, 9, 32
    p.info.tile_size_px = 120
    p.info.screen_size[0], p.info.screen_size[1] = 1920, 1080
    bufs = [C.c_void_p(k << 20) for k in range(1, 6)]

    def call(c=ctx, i=img, params=p):
        return lib.orbit_light_cluster_image(c, None if params is None else C.byref(params), i, None, *bufs, 1000, None)
    assert call(c=None) == _lib.ERR_INVALID_ARGUMENT
    assert call(i=None) == _lib.ERR_INVALID_ARGUMENT
    assert call(params=None) == _lib.ERR_INVALID_ARGUMENT
