"""ctypes binding of liborbit_b200.so (the C ABI of include/orbit_cuda.h).

There is no fallback of any kind: if the shared library is missing or a symbol is absent, loading raises.
"""
import ctypes as C
import os

from . import layouts as L

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("ORBIT_B200_LIB") or os.path.join(HERE, "lib", "liborbit_b200.so")   # override: experiments only

OK, ERR_INVALID_ARGUMENT, ERR_CUDA, ERR_OUT_OF_MEMORY, ERR_NO_DEVICE, ERR_CAPACITY = 0, -1, -2, -3, -4, -5

# name -> (restype, argtypes); the single source of truth for tests that check every declared symbol is exported
PROTOTYPES = {
    "orbit_abi_version": (C.c_int, []),
    "orbit_error_string": (C.c_char_p, [C.c_int]),
    "orbit_last_cuda_error": (C.c_int, []),
    "orbit_ctx_create": (C.c_int, [C.c_int, C.POINTER(C.c_void_p)]),
    "orbit_ctx_destroy": (None, [C.c_void_p]),
    "orbit_ctx_poll_status": (C.c_int, [C.c_void_p, C.POINTER(L.Status)]),
    "orbit_ctx_launch_count": (C.c_uint64, [C.c_void_p]),
    "orbit_ctx_reserve": (C.c_int, [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64]),
    "orbit_hiz_geometry": (C.c_int, [C.c_uint32, C.c_uint32, C.POINTER(L.HizInfo)]),
    "orbit_hiz_create": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.POINTER(C.c_void_p)]),
    "orbit_hiz_wrap": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.POINTER(C.c_void_p)]),
    "orbit_hiz_destroy": (None, [C.c_void_p]),
    "orbit_hiz_info": (C.c_int, [C.c_void_p, C.POINTER(L.HizInfo)]),
    "orbit_hiz_build": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p]),
    "orbit_entity_cull": (C.c_int, [C.c_void_p, C.POINTER(L.CullInfo), C.POINTER(L.SceneBuffers), C.c_void_p,
                                    C.c_void_p, C.c_uint64, C.c_void_p]),
    "orbit_meshlet_cull": (C.c_int, [C.c_void_p, C.POINTER(L.CullInfo), C.POINTER(L.SceneBuffers), C.c_void_p,
                                     C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p]),
    "orbit_light_cluster": (C.c_int, [C.c_void_p, C.POINTER(L.ClusterParams), C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]),
    "orbit_scene_update": (C.c_int, [C.c_void_p, C.POINTER(L.SceneUpdate), C.c_void_p]),
    "orbit_draws_scatter": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint64,
                                      C.c_void_p]),
    "orbit_draws_scatter_ranked": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint64,
                                             C.c_void_p]),
    "orbit_cull_pair_compatible": (C.c_int, [C.POINTER(L.CullInfo), C.POINTER(L.CullInfo)]),
    "orbit_entity_cull_late_main": (C.c_int, [C.c_void_p, C.POINTER(L.CullInfo), C.POINTER(L.CullInfo), C.POINTER(L.SceneBuffers), C.c_void_p,
                                              C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]),
    "orbit_meshlet_cull_late_main": (C.c_int, [C.c_void_p, C.POINTER(L.CullInfo), C.POINTER(L.CullInfo), C.POINTER(L.SceneBuffers), C.c_void_p,
                                               C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "orbit_entity_cull_views": (C.c_int, [C.c_void_p, C.POINTER(L.CullInfo), C.c_uint32, C.POINTER(L.SceneBuffers), C.POINTER(C.c_void_p),
                                          C.c_uint64, C.c_void_p]),
    "orbit_meshlet_cull_views": (C.c_int, [C.c_void_p, C.POINTER(L.CullInfo), C.c_uint32, C.POINTER(L.SceneBuffers), C.POINTER(C.c_void_p),
                                           C.c_uint64, C.POINTER(C.c_void_p), C.c_uint64, C.POINTER(C.c_void_p), C.c_void_p]),
    "orbit_hiz_build_views": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_uint32, C.c_uint32, C.c_uint32,
                                        C.c_void_p]),
    "orbit_entity_cull_views_occlusion": (C.c_int, [C.c_void_p, C.POINTER(L.CullInfo), C.c_uint32, C.POINTER(L.SceneBuffers),
                                                    C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_uint64, C.c_void_p]),
    "orbit_meshlet_cull_views_occlusion": (C.c_int, [C.c_void_p, C.POINTER(L.CullInfo), C.c_uint32, C.POINTER(L.SceneBuffers),
                                                     C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_uint64, C.POINTER(C.c_void_p),
                                                     C.c_uint64, C.POINTER(C.c_void_p), C.c_void_p]),
    "orbit_meshlet_test": (C.c_int, [C.c_void_p, C.POINTER(L.CullInfo), C.POINTER(L.SceneBuffers), C.c_void_p, C.c_void_p, C.c_uint64,
                                     C.c_void_p, C.c_void_p]),
    "orbit_record_masks_put": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "orbit_draws_from_masks": (C.c_int, [C.c_void_p, C.POINTER(L.SceneBuffers), C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint32,
                                         C.c_void_p, C.c_uint64, C.c_void_p]),
    "orbit_peer_put": (C.c_int, [C.c_void_p, C.POINTER(L.PeerPut), C.c_uint32, C.c_uint32, C.c_void_p]),
    "orbit_peer_wait": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p]),
    "orbit_meshlet_bounds": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p]),
    "orbit_mesh_bounds": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p]),
    "orbit_peer_alloc": (C.c_int, [C.c_void_p, C.c_uint64, C.POINTER(C.c_void_p), C.c_void_p]),
    "orbit_peer_open": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p)]),
    "orbit_peer_close": (C.c_int, [C.c_void_p, C.c_void_p]),
    "orbit_peer_free": (None, [C.c_void_p, C.c_void_p]),
    "orbit_device_copy": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]),
}

_lib = None


class OrbitError(RuntimeError):
    def __init__(self, code, what):
        self.code = code
        super().__init__("%s failed: %s (code %d, cuda error %d)" % (
            what, lib().orbit_error_string(code).decode(), code, lib().orbit_last_cuda_error()))


def lib():
    """Loads liborbit_b200.so (once). Raises if it is not built — the product never degrades to a CPU path."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                "liborbit_b200.so is not built (%s). Run `python -m orbit_b200.build` (needs nvcc); "
                "orbit_b200 has no CPU fallback." % LIB_PATH)
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(handle, name)  # AttributeError if the symbol is missing
            fn.restype = res
            fn.argtypes = args
        if handle.orbit_abi_version() != 3:
            raise ImportError("liborbit_b200.so ABI version mismatch")
        _lib = handle
    return _lib


_host = None


def host_lib():
    """Loads liborbit_host.so: the compiled host-side frame driver above the C ABI (orbit_b200/host/frame_driver.cpp)."""
    global _host
    if _host is None:
        lib()   # liborbit_b200.so first: the driver links against it
        path = os.path.join(os.path.dirname(LIB_PATH), "liborbit_host.so")
        if not os.path.exists(path):
            raise ImportError("liborbit_host.so is not built (%s). Run `python -m orbit_b200.build`." % path)
        h = C.CDLL(path)
        h.orbit_host_frame_loop.restype = C.c_int
        h.orbit_host_frame_loop.argtypes = [C.c_void_p, C.POINTER(L.HostFrame), C.c_uint32, C.POINTER(L.HostFrameIO), C.c_uint32, C.c_uint32]
        h.orbit_host_pinned_alloc.restype = C.c_void_p
        h.orbit_host_pinned_alloc.argtypes = [C.c_uint64, C.c_int]
        h.orbit_host_pinned_free.restype = None
        h.orbit_host_pinned_free.argtypes = [C.c_void_p]
        _host = h
    return _host


class PinnedBuffer:
    """Pinned host memory from the host driver library (optionally write-combined), viewed as a numpy uint8 array."""

    def __init__(self, nbytes, write_combined=False):
        import numpy as np
        self.nbytes = int(nbytes)
        self.ptr = host_lib().orbit_host_pinned_alloc(self.nbytes, 1 if write_combined else 0)
        if not self.ptr:
            raise MemoryError("cudaHostAlloc(%d bytes) failed" % self.nbytes)
        self.array = np.ctypeslib.as_array((C.c_uint8 * self.nbytes).from_address(self.ptr))

    def data_ptr(self):
        return self.ptr

    def numel(self):
        return self.nbytes

    def close(self):
        if self.ptr:
            self.array = None
            host_lib().orbit_host_pinned_free(self.ptr)
            self.ptr = None


def check(code, what):
    if code != OK:
        raise OrbitError(code, what)
