"""CPU: the batched two-pass occlusion entry points are declared in the C header, exported by the built library with the
prototypes of _lib.py, and refuse a missing context or an empty view list without touching a device."""
import ctypes as C
import os
import re

from orbit_b200 import _lib
from orbit_b200 import layouts as L

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = ("orbit_hiz_build_views", "orbit_entity_cull_views_occlusion", "orbit_meshlet_cull_views_occlusion")


def test_declared_in_the_header_and_exported():
    hdr = open(os.path.join(ROOT, "include", "orbit_cuda.h")).read()
    lib = _lib.lib()
    for name in NAMES:
        assert re.search(r"\bint\s+%s\s*\(" % name, hdr), name
        assert name in _lib.PROTOTYPES, name
        assert getattr(lib, name) is not None


def test_header_arguments_match_the_prototypes():
    """Argument count of each declaration equals the ctypes prototype's (the header is the ABI's source of truth)."""
    hdr = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "orbit_cuda.h")).read(), flags=re.S)
    for name in NAMES:
        m = re.search(r"\bint\s+%s\s*\(([^;]*)\)\s*;" % name, hdr)
        assert m, name
        assert len(m.group(1).split(",")) == len(_lib.PROTOTYPES[name][1]), name


def test_refuse_without_a_context_or_views():
    lib = _lib.lib()
    gs = (L.CullInfo * 1)()
    gs[0].occlusion_pass = 1
    sb = (L.SceneBuffers * 1)()
    bufs = (C.c_void_p * 1)(None)
    bad = _lib.ERR_INVALID_ARGUMENT
    assert lib.orbit_hiz_build_views(None, bufs, bufs, 1, 64, 64, None) == bad
    assert lib.orbit_entity_cull_views_occlusion(None, gs, 1, sb, None, bufs, 1, None) == bad
    assert lib.orbit_meshlet_cull_views_occlusion(None, gs, 1, sb, None, bufs, 1, bufs, 1, None, None) == bad
