"""CPU: the C-ABI library loads, exports every symbol include/orbit_cuda.h declares, refuses to run without a
GPU (no CPU fallback), and the Python / C views of every layout agree byte for byte."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np

from orbit_b200 import _lib
from orbit_b200 import layouts as L

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_loads_and_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "orbit_cuda.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(orbit_[a-z0-9_]+)\s*\(", hdr))
    assert declared, "no declarations parsed"
    assert declared == set(_lib.PROTOTYPES), (declared ^ set(_lib.PROTOTYPES))
    lib = _lib.lib()
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.orbit_abi_version() == 3
    assert lib.orbit_error_string(0) == b"ok"


NO_DEVICE_PROBE = r'''
import ctypes as C
from orbit_b200 import _lib
from orbit_b200.passes import Context
h = C.c_void_p()
assert _lib.lib().orbit_ctx_create(0, C.byref(h)) == _lib.ERR_NO_DEVICE
try:
    Context(0)
except RuntimeError:
    pass
else:
    raise AssertionError("Context(0) succeeded without a device")
'''


def test_no_cpu_fallback():
    # every device hidden, so the check runs on a machine with a GPU too
    out = subprocess.run([sys.executable, "-c", NO_DEVICE_PROBE], cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "orbit_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert "oracle_ref" not in text and "liborbit_oracle" not in text and "oracle/" not in text, f


def test_layouts_match_c_header(tmp_path):
    src = tmp_path / "layout_probe.c"
    src.write_text(r'''
#include <stdio.h>
#include "orbit_cuda.h"
#define P(T) printf(#T " %zu\n", sizeof(T))
#define O(T, f) printf(#T "." #f " %zu\n", offsetof(T, f))
int main(void) {
  P(OrbitCullInfo); P(OrbitEntityData); P(OrbitEntityDraw); P(OrbitMeshInfo); P(OrbitMeshlet); P(OrbitMeshletDispatch);
  P(OrbitMeshletDrawCommand); P(OrbitMeshTaskPayload); P(OrbitLightData); P(OrbitClusterCullInfo); P(OrbitClusterParams);
  P(OrbitSceneBuffers); P(OrbitHizInfo); P(OrbitStatus); P(OrbitTransform); P(OrbitSceneUpdate);
  O(OrbitTransform, orientation); O(OrbitTransform, scale); O(OrbitSceneUpdate, n_entities); O(OrbitSceneUpdate, entity_data); O(OrbitStatus, visibility_overflow);
  O(OrbitCullInfo, cull_planes); O(OrbitCullInfo, occlusion_pass); O(OrbitCullInfo, p00_or_width_recip_x2); O(OrbitCullInfo, lod_base);
  O(OrbitCullInfo, lod_target_pos_view_space); O(OrbitCullInfo, max_mesh_lod);
  O(OrbitClusterCullInfo, tile_size_px); O(OrbitClusterCullInfo, z_near); O(OrbitClusterCullInfo, global_light_count);
  O(OrbitClusterParams, z_scale); O(OrbitSceneBuffers, entity_draw_count); O(OrbitHizInfo, level_offset); O(OrbitHizInfo, texels);
  O(OrbitMeshlet, cone_axis); O(OrbitMeshlet, material_index); O(OrbitMeshInfo, mesh_lods); O(OrbitLightData, outer_radius);
  return 0; }''')
    exe = tmp_path / "probe"
    subprocess.check_call(["/usr/bin/gcc", "-std=c11", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = dict(line.rsplit(" ", 1) for line in subprocess.check_output([str(exe)], text=True).splitlines())
    got = {k: int(v) for k, v in got.items()}
    py_sizes = {"OrbitCullInfo": C.sizeof(L.CullInfo), "OrbitEntityData": L.entity_dtype.itemsize, "OrbitEntityDraw": L.entity_draw_dtype.itemsize,
                "OrbitMeshInfo": L.mesh_info_dtype.itemsize, "OrbitMeshlet": L.meshlet_dtype.itemsize, "OrbitMeshletDispatch": L.dispatch_dtype.itemsize,
                "OrbitMeshletDrawCommand": L.draw_command_dtype.itemsize, "OrbitMeshTaskPayload": 40, "OrbitLightData": L.light_dtype.itemsize,
                "OrbitClusterCullInfo": C.sizeof(L.ClusterCullInfo), "OrbitClusterParams": C.sizeof(L.ClusterParams),
                "OrbitSceneBuffers": C.sizeof(L.SceneBuffers), "OrbitHizInfo": C.sizeof(L.HizInfo), "OrbitStatus": C.sizeof(L.Status),
                "OrbitTransform": L.transform_dtype.itemsize, "OrbitSceneUpdate": C.sizeof(L.SceneUpdate)}
    for k, v in py_sizes.items():
        assert got[k] == v, (k, got[k], v)
    offs = {"OrbitCullInfo.cull_planes": L.CullInfo.cull_planes.offset, "OrbitCullInfo.occlusion_pass": L.CullInfo.occlusion_pass.offset,
            "OrbitCullInfo.p00_or_width_recip_x2": L.CullInfo.p00_or_width_recip_x2.offset, "OrbitCullInfo.lod_base": L.CullInfo.lod_base.offset,
            "OrbitCullInfo.lod_target_pos_view_space": L.CullInfo.lod_target_pos_view_space.offset, "OrbitCullInfo.max_mesh_lod": L.CullInfo.max_mesh_lod.offset,
            "OrbitClusterCullInfo.tile_size_px": L.ClusterCullInfo.tile_size_px.offset, "OrbitClusterCullInfo.z_near": L.ClusterCullInfo.z_near.offset,
            "OrbitClusterCullInfo.global_light_count": L.ClusterCullInfo.global_light_count.offset, "OrbitClusterParams.z_scale": L.ClusterParams.z_scale.offset,
            "OrbitSceneBuffers.entity_draw_count": L.SceneBuffers.entity_draw_count.offset, "OrbitHizInfo.level_offset": L.HizInfo.level_offset.offset,
            "OrbitHizInfo.texels": L.HizInfo.texels.offset,
            "OrbitTransform.orientation": L.transform_dtype.fields["orientation"][1], "OrbitTransform.scale": L.transform_dtype.fields["scale"][1],
            "OrbitSceneUpdate.n_entities": L.SceneUpdate.n_entities.offset, "OrbitSceneUpdate.entity_data": L.SceneUpdate.entity_data.offset,
            "OrbitStatus.visibility_overflow": L.Status.visibility_overflow.offset,
            "OrbitMeshlet.cone_axis": L.meshlet_dtype.fields["cone_axis"][1], "OrbitMeshlet.material_index": L.meshlet_dtype.fields["material_index"][1],
            "OrbitMeshInfo.mesh_lods": L.mesh_info_dtype.fields["mesh_lods"][1], "OrbitLightData.outer_radius": L.light_dtype.fields["outer_radius"][1]}
    for k, v in offs.items():
        assert got[k] == v, (k, got[k], v)
    # reference numbers (SURVEY Appendix A.1)
    assert got["OrbitCullInfo"] == 400 and got["OrbitClusterCullInfo"] == 192 and got["OrbitMeshlet"] == 32 and got["OrbitMeshletDrawCommand"] == 28


def test_hiz_geometry_matches_reference_sizing():
    """DepthPyramid::new (draw_gen.rs:456-459) + mip_levels_from_size (math.rs:18-20): 1080p -> 1024^2, 11 mips,
    1 398 101 texels; 4K -> 2048^2, 12 mips."""
    from orbit_b200 import scenes
    for (w, h), (pw, ph, lv, tot) in {(1920, 1080): (1024, 1024, 11, 1398101), (3840, 2160): (2048, 2048, 12, 5592405),
                                      (1280, 720): (1024, 512, 11, None), (100, 60): (64, 32, 7, None), (2, 2): (1, 1, 1, 1)}.items():
        info = L.HizInfo()
        assert _lib.lib().orbit_hiz_geometry(w, h, C.byref(info)) == 0
        assert (info.width, info.height, info.levels) == (pw, ph, lv)
        if tot:
            assert info.total_texels == tot
        pw2, ph2, lv2, offs, tot2 = scenes.hiz_geometry(w, h)
        assert (pw2, ph2, lv2, tot2) == (pw, ph, lv, info.total_texels)
        assert list(info.level_offset[:lv]) == offs
    assert _lib.lib().orbit_hiz_geometry(0, 5, C.byref(L.HizInfo())) == _lib.ERR_INVALID_ARGUMENT


def test_argument_errors_without_gpu():
    lib = _lib.lib()
    assert lib.orbit_entity_cull(None, None, None, None, None, 0, None) == _lib.ERR_INVALID_ARGUMENT
    assert lib.orbit_meshlet_cull(None, None, None, None, None, 0, None, 0, None, None) == _lib.ERR_INVALID_ARGUMENT
    assert lib.orbit_hiz_build(None, None, None, 1, 1, None) == _lib.ERR_INVALID_ARGUMENT
    assert lib.orbit_scene_update(None, None, None) == _lib.ERR_INVALID_ARGUMENT


def test_host_driver_library_loads():
    """liborbit_host.so (compiled host frame loop above the C ABI) loads, resolves against liborbit_b200.so, and its
    struct mirrors have the sizes the C++ side sees."""
    h = _lib.host_lib()
    assert h.orbit_host_frame_loop(None, None, 0, None, 0, 0) == _lib.ERR_INVALID_ARGUMENT
    assert h.orbit_host_sizeof_frame() == C.sizeof(L.HostFrame) and h.orbit_host_sizeof_io() == C.sizeof(L.HostFrameIO)


def test_cull_pair_compatibility_is_a_host_predicate():
    """orbit_cull_pair_compatible needs no GPU: it decides from the two 400-byte structs whether the MAIN pass may be fused into
    the LATE pass (same camera, planes, projection type and LOD parameters, both visibility buffers, pass 2 then pass 1)."""
    import ctypes as C
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from orbit_b200 import _lib, layouts as L, scenes
    import oracle_ref as O
    lib = _lib.lib()
    _, view = scenes.config_c1(scale=0.2)
    late, main = O.gpu_cull_info(view, "write"), O.gpu_cull_info(view, "read")
    ok = lambda a, b: lib.orbit_cull_pair_compatible(C.byref(a), C.byref(b))
    assert ok(late, main) == 1 and ok(main, late) == 0 and ok(late, late) == 0 and ok(main, main) == 0
    assert lib.orbit_cull_pair_compatible(None, C.byref(main)) == 0
    assert ok(late, O.gpu_cull_info(view, "none")) == 0                                   # pass 0 is not pass 1
    assert ok(late, O.gpu_cull_info(view, "read", meshlet_occlusion=False)) == 0          # needs the meshlet visibility buffer
    assert ok(O.gpu_cull_info(view, "write", meshlet_occlusion=False), main) == 0
    g = O.gpu_cull_info(view, "read"); g.alpha_mode_flags = 0b100
    assert ok(late, g) == 1                                                                # another alpha filter is fine
    for field, delta in (("lod_base", 1.0), ("lod_step", 0.5), ("min_mesh_lod", 1), ("max_mesh_lod", -1), ("cull_plane_count", -1), ("projection_type", 1)):
        g = O.gpu_cull_info(view, "read")
        setattr(g, field, getattr(g, field) + delta)
        assert ok(late, g) == 0, field
    g = O.gpu_cull_info(view, "read"); g.cull_planes[0][3] += 1e-3
    assert ok(late, g) == 0
    g = O.gpu_cull_info(view, "read"); g.lod_target_pos_view_space[1] += 1.0
    assert ok(late, g) == 0
    # fields only pass 2 reads (projection scale, near / far) are zero in a pass-1 struct and do not matter
    g = O.gpu_cull_info(view, "read"); g.z_near = 123.0; g.p00_or_width_recip_x2 = 7.0
    assert ok(late, g) == 1
