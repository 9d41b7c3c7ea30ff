"""CPU: the output-image entry points (orbit_hiz_attach_image, orbit_cluster_grid_*, orbit_light_cluster_image_grid) are
declared in the C header, exported with the prototypes of _lib.py, and refuse a NULL context, pyramid, array, grid, image or
params before they use the context or a device. Handles here are zero-filled stand-ins: refused calls must return before
touching them, and orbit_hiz_wrap only reads the context's device number. The C++ host mirror's new members compile."""
import ctypes as C
import os
import re
import subprocess

import pytest

from orbit_b200 import _lib
from orbit_b200 import layouts as L

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = ["orbit_hiz_attach_image", "orbit_cluster_grid_wrap", "orbit_cluster_grid_destroy", "orbit_light_cluster_image_grid"]


@pytest.mark.parametrize("name", NAMES)
def test_declared_in_the_header_and_exported(name):
    hdr = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "orbit_cuda.h")).read(), flags=re.S)
    m = re.search(r"\b(?:int|void)\s+%s\s*\(([^;]*)\)\s*;" % name, hdr)
    assert m, name
    assert getattr(_lib.lib(), name) is not None
    assert len(m.group(1).split(",")) == len(_lib.PROTOTYPES[name][1])


def test_abi_version_unchanged():
    assert _lib.lib().orbit_abi_version() == 3


@pytest.fixture
def handles():
    lib = _lib.lib()
    fake_ctx = C.create_string_buffer(1 << 16)                 # zero-filled: device 0
    fake_obj = C.create_string_buffer(64)                       # stands in for a depth image, a grid or an array
    ctx, obj = C.c_void_p(C.addressof(fake_ctx)), C.c_void_p(C.addressof(fake_obj))
    hiz = C.c_void_p()
    assert lib.orbit_hiz_wrap(ctx, 640, 360, C.c_void_p(1 << 20), C.byref(hiz)) == _lib.OK
    yield lib, ctx, hiz, obj
    lib.orbit_hiz_destroy(hiz)
    del fake_ctx, fake_obj


def test_attach_refuses_null_arguments(handles):
    lib, ctx, hiz, arr = handles
    assert lib.orbit_hiz_attach_image(None, hiz, arr) == _lib.ERR_INVALID_ARGUMENT
    assert lib.orbit_hiz_attach_image(ctx, None, arr) == _lib.ERR_INVALID_ARGUMENT
    assert lib.orbit_hiz_attach_image(ctx, hiz, None) == _lib.ERR_INVALID_ARGUMENT


def test_attach_refuses_a_pyramid_of_another_device(handles):
    lib, _, hiz, arr = handles
    other = C.create_string_buffer(1 << 16)
    C.c_int.from_buffer(other).value = 1                        # orbit_ctx::device is its first member
    assert lib.orbit_hiz_attach_image(C.c_void_p(C.addressof(other)), hiz, arr) == _lib.ERR_INVALID_ARGUMENT


def test_grid_wrap_refuses_null_arguments(handles):
    lib, ctx, _, arr = handles
    out = C.c_void_p(1234)
    assert lib.orbit_cluster_grid_wrap(None, arr, C.byref(out)) == _lib.ERR_INVALID_ARGUMENT
    assert out.value is None                                    # *out is cleared on refusal
    assert lib.orbit_cluster_grid_wrap(ctx, None, C.byref(out)) == _lib.ERR_INVALID_ARGUMENT
    assert lib.orbit_cluster_grid_wrap(ctx, arr, None) == _lib.ERR_INVALID_ARGUMENT
    lib.orbit_cluster_grid_destroy(None)


def test_light_cluster_image_grid_refuses_null_handles(handles):
    lib, ctx, _, obj = handles
    p = L.ClusterParams()
    p.info.cluster_count[0], p.info.cluster_count[1], p.info.cluster_count[2] = 16, 9, 32
    p.info.tile_size_px = 120
    p.info.screen_size[0], p.info.screen_size[1] = 1920, 1080
    masks, bounds, unique, index = (C.c_void_p(k << 20) for k in range(1, 5))

    def call(c=ctx, i=obj, g=obj, params=p, m=masks, b=bounds, u=unique, x=index):
        return lib.orbit_light_cluster_image_grid(c, None if params is None else C.byref(params), i, None, m, b, u, g, x, 1000, None)
    assert call(c=None) == _lib.ERR_INVALID_ARGUMENT
    assert call(i=None) == _lib.ERR_INVALID_ARGUMENT
    assert call(g=None) == _lib.ERR_INVALID_ARGUMENT
    assert call(params=None) == _lib.ERR_INVALID_ARGUMENT
    assert call(m=None) == _lib.ERR_INVALID_ARGUMENT
    assert call(b=None) == _lib.ERR_INVALID_ARGUMENT
    assert call(u=None) == _lib.ERR_INVALID_ARGUMENT
    assert call(x=None) == _lib.ERR_INVALID_ARGUMENT


def test_cpp_host_members_compile(tmp_path):
    src = tmp_path / "output_images.cpp"
    src.write_text(r'''
#include "orbit_passes.hpp"
void mirrored(orbit_ctx* ctx, void* pyramid_array, const orbit_depth_image* depth, const orbit_cluster_grid* grid, void* stream) {
    orbit_host::DepthPyramid pyramid(ctx, 1920, 1080);
    pyramid.attach_image(pyramid_array);
    pyramid.update(depth, stream);
    OrbitClusterParams params{};
    orbit_host::compute_clusters(ctx, params, depth, nullptr, nullptr, nullptr, nullptr, grid, nullptr, 0, stream);
}
''')
    subprocess.check_call(["/usr/bin/g++", "-std=c++17", "-fsyntax-only", "-I", os.path.join(ROOT, "include"), str(src)])
