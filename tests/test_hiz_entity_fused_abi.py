"""CPU: orbit_hiz_build_entity_cull_late (Hi-Z build + LATE entity stage in one call) is declared in the C header, exported
with the prototype of _lib.py, and refuses every bad argument combination before it uses the context or a device. The
context handle here is a zero-filled stand-in: refused calls must return before touching it (a refused call launches
nothing), and orbit_hiz_wrap only reads its device number."""
import ctypes as C
import os
import re

from orbit_b200 import _lib
from orbit_b200 import layouts as L

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAME = "orbit_hiz_build_entity_cull_late"


def test_declared_in_the_header_and_exported():
    hdr = open(os.path.join(ROOT, "include", "orbit_cuda.h")).read()
    assert re.search(r"\bint\s+%s\s*\(" % NAME, hdr)
    assert getattr(_lib.lib(), NAME) is not None
    m = re.search(r"\bint\s+%s\s*\(([^;]*)\)\s*;" % NAME, re.sub(r"/\*.*?\*/", "", hdr, flags=re.S))
    assert m and len(m.group(1).split(",")) == len(_lib.PROTOTYPES[NAME][1])


def _valid_late():
    g = L.CullInfo()
    g.occlusion_pass = 2
    g.visibility_buffer = g.meshlet_visibility_buffer = 0
    g.lod_base, g.lod_step = 10.0, 2.0
    return g


def _main_of(late):
    g = L.CullInfo.from_buffer_copy(late)
    g.occlusion_pass = 1
    return g


def test_refuses_every_bad_combination():
    lib = _lib.lib()
    fake_ctx = C.create_string_buffer(1 << 16)                 # zero-filled: device 0
    ctx = C.c_void_p(C.addressof(fake_ctx))
    hiz = C.c_void_p()
    assert lib.orbit_hiz_wrap(ctx, 640, 360, C.c_void_p(1 << 20), C.byref(hiz)) == _lib.OK
    late = _valid_late()
    main = _main_of(late)
    assert lib.orbit_cull_pair_compatible(C.byref(late), C.byref(main)) == 1
    sb = L.SceneBuffers()
    sb.entity_draws, sb.mesh_infos, sb.entities, sb.entity_visibility = 1 << 20, 2 << 20, 3 << 20, 4 << 20
    sb.entity_draw_count = 1000
    late_d, main_d, depth = C.c_void_p(5 << 20), C.c_void_p(6 << 20), C.c_void_p(7 << 20)

    def call(ctx=ctx, hiz=hiz, depth=depth, dw=640, dh=360, late=late, main=main, sb=sb, ld=late_d, md=main_d):
        return lib.orbit_hiz_build_entity_cull_late(ctx, hiz, depth, dw, dh, None if late is None else C.byref(late),
                                                    None if main is None else C.byref(main), C.byref(sb), ld, md, 1000, None)

    def edit(src, **kw):
        g = type(src).from_buffer_copy(src)
        for k, v in kw.items():
            setattr(g, k, v)
        return g
    cases = {
        "no context": dict(ctx=None), "no pyramid": dict(hiz=None), "no depth": dict(depth=None),
        "depth width": dict(dw=641), "depth height": dict(dh=359), "no late CullInfo": dict(late=None),
        "late pass 0": dict(late=edit(late, occlusion_pass=0), main=None, md=None),
        "late pass 1": dict(late=edit(late, occlusion_pass=1), main=None, md=None),
        "MAIN without its buffer": dict(md=None), "MAIN buffer without MAIN": dict(main=None),
        "MAIN buffer = LATE buffer": dict(md=late_d), "MAIN buffer misaligned": dict(md=C.c_void_p((6 << 20) + 2)),
        "incompatible pair": dict(main=edit(main, lod_base=20.0)), "MAIN pass 2": dict(main=edit(main, occlusion_pass=2)),
        "MAIN without meshlet occlusion": dict(late=edit(late, meshlet_visibility_buffer=L.NO_BUFFER),
                                               main=edit(main, meshlet_visibility_buffer=L.NO_BUFFER)),
        "no LATE buffer": dict(ld=None, main=None, md=None), "LATE buffer misaligned": dict(ld=C.c_void_p((5 << 20) + 1)),
        "too many planes": dict(late=edit(late, cull_plane_count=L.MAX_CULL_PLANES + 1), main=None, md=None),
        "pass above 2": dict(late=edit(late, occlusion_pass=3), main=None, md=None),
        "no entity visibility": dict(sb=edit(sb, entity_visibility=None)), "no entities": dict(sb=edit(sb, entities=None)),
        "no draw words": dict(sb=edit(sb, entity_draws=None)), "no mesh infos": dict(sb=edit(sb, mesh_infos=None)),
        "mesh infos misaligned": dict(sb=edit(sb, mesh_infos=(2 << 20) + 4)), "entities misaligned": dict(sb=edit(sb, entities=(3 << 20) + 8)),
        "draw words misaligned": dict(sb=edit(sb, entity_draws=(1 << 20) + 2)),
        "draw_begin % 32": dict(sb=edit(sb, draw_begin=3, draw_end=50)), "draw_begin > draw_end": dict(sb=edit(sb, draw_begin=64, draw_end=32)),
    }
    try:
        for what, kw in cases.items():
            assert call(**kw) == _lib.ERR_INVALID_ARGUMENT, what
            if "main" not in kw and "md" not in kw:     # the same rule holds without the MAIN pass
                assert call(main=None, md=None, **kw) == _lib.ERR_INVALID_ARGUMENT, (what, "no MAIN")
    finally:
        lib.orbit_hiz_destroy(hiz)
