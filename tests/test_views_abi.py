"""CPU: the batched-view limit is the same number in the C header and in layouts.py, and the batched entry points refuse a
missing context or an empty view list without touching a device."""
import ctypes as C
import os
import re

from orbit_b200 import _lib
from orbit_b200 import layouts as L

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_max_batch_views_matches_the_header():
    hdr = open(os.path.join(ROOT, "include", "orbit_cuda.h")).read()
    m = re.search(r"#define\s+ORBIT_MAX_BATCH_VIEWS\s+(\d+)", hdr)
    assert m and int(m.group(1)) == L.MAX_BATCH_VIEWS


def test_views_calls_refuse_without_a_context():
    lib = _lib.lib()
    gs = (L.CullInfo * 1)()
    sb = L.SceneBuffers()
    bufs = (C.c_void_p * 1)(None)
    assert lib.orbit_entity_cull_views(None, gs, 1, C.byref(sb), bufs, 1, None) == _lib.ERR_INVALID_ARGUMENT
    assert lib.orbit_meshlet_cull_views(None, gs, 1, C.byref(sb), bufs, 1, bufs, 1, None, None) == _lib.ERR_INVALID_ARGUMENT
