"""ctypes binding of libecho_b200.so — the C ABI a C# host would bind with [DllImport("echo_b200")] (INTEGRATION.md).

The library is mandatory: there is no CPU fallback. A missing .so or a missing CUDA device raises EchoNativeError.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIBRARY_PATH = os.environ.get("ECHO_B200_LIBRARY", os.path.join(_HERE, "libecho_b200.so"))  # override: A/B builds of the same ABI

OK, ERR_INVALID, ERR_NO_DEVICE, ERR_CUDA, ERR_UNSUPPORTED = range(5)


class EchoNativeError(RuntimeError):
    """Raised like OidnDenoise.ThrowOnNativeError does (Processes/Composition/OidnDenoise.cs:201-206): the status code
    of the failed call plus the message pulled from echo_b200_last_error()."""

    def __init__(self, status, message):
        super().__init__(f"libecho_b200 error {status}: {message}")
        self.status = status


_lib = None

# every symbol include/echo_b200.h and include/echo_b200_debug.h declare
EXPORTS = [
    "echo_b200_device_count", "echo_b200_scene_create", "echo_b200_scene_set_qbvh", "echo_b200_scene_set_triangles",
    "echo_b200_scene_set_spheres", "echo_b200_scene_set_materials", "echo_b200_scene_set_light_tree", "echo_b200_scene_set_infinite",
    "echo_b200_scene_set_camera", "echo_b200_scene_commit", "echo_b200_scene_destroy", "echo_b200_trace_batch", "echo_b200_occlude_batch",
    "echo_b200_trace_batch_device", "echo_b200_occlude_batch_device", "echo_b200_render_tiles", "echo_b200_render_frame_device",
    "echo_b200_frame_resolve_device", "echo_b200_last_error", "echo_b200_version",
    "echo_b200_scene_set_packs", "echo_b200_trace_batch_hierarchy", "echo_b200_occlude_batch_hierarchy", "echo_b200_scene_set_bound_radius", "echo_b200_scene_set_textures", "echo_b200_scene_set_distributions", "echo_b200_build_qbvh", "echo_b200_build_qbvh_instanced", "echo_b200_scene_build_qbvh",
    "echo_b200_debug_evaluate_samples4", "echo_b200_debug_bounds_violations",
    "echo_b200_trace_batch_device_counted", "echo_b200_occlude_batch_device_counted", "echo_b200_debug_bxdf_batch", "echo_b200_debug_math",
    "echo_b200_debug_evaluate_samples",
    "echo_b200_host_alloc", "echo_b200_host_free", "echo_b200_host_register", "echo_b200_host_unregister", "echo_b200_debug_set_option", "echo_b200_debug_measure_peaks", "echo_b200_debug_last_build", "echo_b200_debug_last_light_build", "echo_b200_build_light_tree", "echo_b200_scene_build_light_tree",
    "echo_b200_scene_create_multi", "echo_b200_scene_gpu_count", "echo_b200_build_packs", "echo_b200_scene_build_packs", "echo_b200_debug_last_pack_build",
]


def library():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIBRARY_PATH):
        raise EchoNativeError(-1, f"{LIBRARY_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'`")

    lib = ctypes.CDLL(LIBRARY_PATH)
    p, u32, u64, i32, f32 = ctypes.c_void_p, ctypes.c_uint32, ctypes.c_uint64, ctypes.c_int32, ctypes.c_float

    signatures = {
        "echo_b200_device_count": [ctypes.POINTER(i32)],
        "echo_b200_scene_create": [ctypes.POINTER(p), i32],
        "echo_b200_scene_set_qbvh": [p, p, u32, u32],
        "echo_b200_scene_set_triangles": [p, p, u32],
        "echo_b200_scene_set_spheres": [p, p, u32],
        "echo_b200_scene_set_materials": [p, p, u32],
        "echo_b200_scene_set_light_tree": [p, p, u32, p, p, u32, p, u32],
        "echo_b200_scene_set_infinite": [p, p, u32, f32, f32],
        "echo_b200_scene_set_camera": [p, p],
        "echo_b200_scene_set_packs": [p, p, u32, p, u32],
        "echo_b200_trace_batch_hierarchy": [p, p, p, u64, p, p],
        "echo_b200_occlude_batch_hierarchy": [p, p, p, u64, p],
        "echo_b200_scene_set_bound_radius": [p, f32],
        "echo_b200_scene_set_textures": [p, p, u32, p, u64, p, u32],
        "echo_b200_scene_set_distributions": [p, p, u64],
        "echo_b200_build_qbvh": [i32, p, u32, p, u32, p, ctypes.POINTER(u32), ctypes.POINTER(u32)],
        "echo_b200_scene_build_qbvh": [p, ctypes.POINTER(u32), ctypes.POINTER(u32)],
        "echo_b200_build_qbvh_instanced": [i32, p, u32, p, u32, p, u32, p, ctypes.POINTER(u32), ctypes.POINTER(u32)],
        "echo_b200_debug_evaluate_samples4": [p, p, p, p, u64, p],
        "echo_b200_debug_bounds_violations": [p, ctypes.POINTER(u32)],
        "echo_b200_scene_commit": [p],
        "echo_b200_scene_destroy": [p],
        "echo_b200_trace_batch": [p, p, u64, p],
        "echo_b200_occlude_batch": [p, p, u64, p],
        "echo_b200_trace_batch_device": [p, p, u64, p, p],
        "echo_b200_occlude_batch_device": [p, p, u64, p, p],
        "echo_b200_render_tiles": [p, p, p, u32, p, p],
        "echo_b200_render_frame_device": [p, p, p, u32, p, p, p],
        "echo_b200_frame_resolve_device": [p, p, i32, i32, p],
        "echo_b200_trace_batch_device_counted": [p, p, u64, p, p, p],
        "echo_b200_occlude_batch_device_counted": [p, p, u64, p, p, p],
        "echo_b200_debug_bxdf_batch": [i32, i32, p, p, p, u64, p, p, p],
        "echo_b200_debug_math": [i32, i32, p, p, p, u64, p],
        "echo_b200_debug_evaluate_samples": [p, p, p, p, u64, p],
        "echo_b200_host_alloc": [ctypes.POINTER(p), u64],
        "echo_b200_host_free": [p],
        "echo_b200_host_register": [p, u64],
        "echo_b200_host_unregister": [p],
        "echo_b200_debug_set_option": [ctypes.c_char_p, ctypes.c_int64],
        "echo_b200_debug_measure_peaks": [i32, p],
        "echo_b200_debug_last_build": [p],
        "echo_b200_debug_last_light_build": [p],
        "echo_b200_build_light_tree": [i32, p, u32, p, u32, p, u32, p, u32, p, u32, p, u32, ctypes.POINTER(u32), p, p, u32, ctypes.POINTER(u32), ctypes.POINTER(f32)],
        "echo_b200_scene_build_light_tree": [p, p, u32, ctypes.POINTER(u32), ctypes.POINTER(u32), ctypes.POINTER(f32)],
        "echo_b200_scene_create_multi": [ctypes.POINTER(p), u64],
        "echo_b200_scene_gpu_count": [p, ctypes.POINTER(i32)],
        "echo_b200_build_packs": [i32, p, u32, p, u32, p, u32, p, u32, p, u32, p, u32, p, u32, ctypes.POINTER(u32), p, u32, ctypes.POINTER(u32), p, p, u32,
                                  ctypes.POINTER(u32), ctypes.POINTER(f32)],
        "echo_b200_scene_build_packs": [p, p, u32, ctypes.POINTER(u32), ctypes.POINTER(u32), ctypes.POINTER(u32), ctypes.POINTER(f32)],
        "echo_b200_debug_last_pack_build": [p],
    }

    for name, argtypes in signatures.items():
        function = getattr(lib, name)
        function.argtypes = argtypes
        function.restype = i32

    lib.echo_b200_last_error.restype = ctypes.c_char_p
    lib.echo_b200_version.restype = ctypes.c_char_p
    _lib = lib
    return lib


def check(status):
    if status != OK:
        raise EchoNativeError(status, library().echo_b200_last_error().decode("utf-8", "replace"))


def pointer(array):
    """Raw address of a numpy array (or None / empty -> NULL)."""
    if array is None or array.size == 0:
        return ctypes.c_void_p(0)
    return ctypes.c_void_p(array.ctypes.data)


def device_count():
    count = ctypes.c_int32()
    check(library().echo_b200_device_count(ctypes.byref(count)))
    return count.value


class HostBuffer:
    """Page-locked host memory from echo_b200_host_alloc, viewed as a numpy array: what a host hands to the host-buffer entry
    points so that their copies run asynchronously at the link's rate (a `fixed`-pinned managed array is pageable for CUDA)."""

    def __init__(self, count, dtype):
        import numpy as np
        self.dtype = np.dtype(dtype)
        self.count = int(count)
        self._pointer = ctypes.c_void_p()
        check(library().echo_b200_host_alloc(ctypes.byref(self._pointer), self.count * self.dtype.itemsize))
        buffer = (ctypes.c_uint8 * max(self.count * self.dtype.itemsize, 1)).from_address(self._pointer.value)
        self.array = np.frombuffer(buffer, dtype=self.dtype, count=self.count)

    @property
    def address(self):
        return self._pointer.value

    def free(self):
        if self._pointer is not None and self._pointer.value:
            self.array = None
            library().echo_b200_host_free(self._pointer)
            self._pointer = ctypes.c_void_p()

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def set_option(name, value):
    """echo_b200_debug_set_option: one tuning switch of the wavefront (the ECHO_B200_<name> environment variables), at run time."""
    check(library().echo_b200_debug_set_option(name.encode(), int(value)))


def measure_peaks(device=0):
    """echo_b200_debug_measure_peaks: the on-chip ceilings of `device` in GB/s, measured now (csrc/peaks.cu)."""
    import numpy as np
    out = np.zeros(3, dtype=np.float32)
    check(library().echo_b200_debug_measure_peaks(int(device), pointer(out)))
    return {"l2_read_gbs": float(out[0]), "l2_sector_gbs": float(out[1]), "l1_sector_gbs": float(out[2]),
            "how": "library microbenchmarks: coalesced ld.global.cg over 32 MB in L2; one random 32-byte sector per lane (ld.global.nc.v8.f32) over 64 MB in L2; the same over 8 KB per CTA in L1"}


def last_build():
    """echo_b200_debug_last_build: phases of this thread's last SweepBuilder device build (host wall time around synchronised phases)."""
    import numpy as np
    out = np.zeros(4, dtype=np.float32)
    check(library().echo_b200_debug_last_build(pointer(out)))
    return {"upload_ms": float(out[0]), "device_build_ms": float(out[1]), "download_ms": float(out[2]), "binary_levels": int(out[3])}


def last_light_build():
    """echo_b200_debug_last_light_build: phases of this thread's last device light-tree build (host wall time around synchronised phases)."""
    import numpy as np
    out = np.zeros(4, dtype=np.float32)
    check(library().echo_b200_debug_last_light_build(pointer(out)))
    return {"upload_ms": float(out[0]), "device_build_ms": float(out[1]), "download_ms": float(out[2]), "levels": int(out[3])}


def last_pack_build():
    """echo_b200_debug_last_pack_build: rounds, levels and read-backs of this thread's last build of every pack (echo_b200_build_packs)."""
    import numpy as np
    out = np.zeros(8, dtype=np.float32)
    check(library().echo_b200_debug_last_pack_build(pointer(out)))
    return {"rounds": int(out[0]), "qbvh_levels": int(out[1]), "light_levels": int(out[2]), "read_backs": int(out[3]), "launches": int(out[4]),
            "build_ms": float(out[5]), "rebuilt_packs": int(out[6])}


def host_register(array):
    """cudaHostRegister of a caller-owned numpy array (echo_b200_host_register); pair with host_unregister before it is freed."""
    check(library().echo_b200_host_register(ctypes.c_void_p(array.ctypes.data), array.nbytes))


def host_unregister(array):
    check(library().echo_b200_host_unregister(ctypes.c_void_p(array.ctypes.data)))
