"""ctypes binding of the C ABI declared in include/pixsht.h.  No compute happens in Python."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
DEFAULT_LIB = os.path.join(os.path.dirname(_HERE), "lib", "libpixsht.so")

PIXSHT_OK, ERR_ARG, ERR_CUDA, ERR_UNSUPPORTED, ERR_NOMEM, ERR_NODEVICE = range(6)
F64, F32 = 0, 1
MAP2ALM, ALM2MAP = 0, 1
HOST, DEVICE = 0, 1


class PixshtError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("pixsht error %d: %s" % (code, msg))
        self.code = code


class Geom(ctypes.Structure):
    _fields_ = [("nphi", ctypes.c_int32), ("nrings_total", ctypes.c_int32), ("ring_first", ctypes.c_int32),
                ("nrings", ctypes.c_int32), ("nx", ctypes.c_int32), ("flipx", ctypes.c_int32), ("flipy", ctypes.c_int32),
                ("ring_scheme", ctypes.c_int32), ("phi0", ctypes.c_double)]


# every symbol include/pixsht.h and include/pixsht_sharp_shim.h declare
EXPORTS = ["pixsht_plan_create", "pixsht_plan_create_rings", "pixsht_plan_create_multi", "pixsht_multi_shard", "pixsht_execute_sharded",
           "pixsht_host_alloc", "pixsht_host_free", "pixsht_host_register", "pixsht_host_unregister", "pixsht_plan_destroy", "pixsht_execute", "pixsht_map2alm_iter", "pixsht_execute_batch", "pixsht_get_timings", "pixsht_plan_set_stream",
           "pixsht_plan_set_stage_families", "pixsht_plan_set_polconv", "pixsht_ring_pixarea", "pixsht_stage_alm2phase", "pixsht_stage_phase2alm", "pixsht_stage_phase2map", "pixsht_stage_map2phase",
           "pixsht_phase_row_len", "pixsht_shared_alloc", "pixsht_shared_open", "pixsht_shared_close", "pixsht_shared_free",
           "pixsht_nalm", "pixsht_alm2cl", "pixsht_plan_info", "pixsht_plan_weights", "pixsht_plan_work", "pixsht_plan_work_per_m", "pixsht_last_error", "pixsht_version",
           "pixsht_device_count", "pixsht_measure_fma_peak",
           "sharp_make_geom_info", "sharp_destroy_geom_info", "sharp_map_size", "sharp_make_triangular_alm_info",
           "sharp_destroy_alm_info", "sharp_alm_count", "sharp_execute", "pixsht_shim_status"]


class PixshtLib:
    """Loads a libpixsht shared object.  The product always uses DEFAULT_LIB (the nvcc-built sm_100a library);
    an explicit path exists only so that tests can point the same binding at the host-emulation build."""

    def __init__(self, path=None):
        path = DEFAULT_LIB if path is None else path
        if not os.path.exists(path):
            raise PixshtError(ERR_NODEVICE, "CUDA library %s is missing: run `python -c 'import __graft_entry__ as g; "
                              "g.build()'` (there is no CPU fallback)" % path)
        self.path = path
        L = self.lib = ctypes.CDLL(path)
        vp, i32, dbl = ctypes.c_void_p, ctypes.c_int, ctypes.c_double
        pvp = ctypes.POINTER(ctypes.c_void_p)
        L.pixsht_plan_create.argtypes = [pvp, ctypes.POINTER(Geom), i32, i32, i32, i32]
        L.pixsht_plan_create_rings.argtypes = [pvp, i32, ctypes.POINTER(dbl), ctypes.POINTER(dbl), i32, dbl, i32, i32, i32, i32]
        L.pixsht_plan_create_multi.argtypes = [pvp, ctypes.POINTER(Geom), i32, i32, i32, i32, ctypes.POINTER(ctypes.c_int)]
        L.pixsht_multi_shard.argtypes = [vp, i32, ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_int32)]
        L.pixsht_execute_sharded.argtypes = [vp, i32, i32, pvp, pvp]
        L.pixsht_host_alloc.argtypes = [pvp, ctypes.c_size_t]
        L.pixsht_host_free.argtypes = [vp]
        L.pixsht_host_register.argtypes = [vp, ctypes.c_size_t]
        L.pixsht_host_unregister.argtypes = [vp]
        L.pixsht_plan_destroy.argtypes = [vp]
        L.pixsht_plan_destroy.restype = None
        L.pixsht_execute.argtypes = [vp, i32, i32, pvp, pvp, i32]
        L.pixsht_map2alm_iter.argtypes = [vp, i32, pvp, pvp, i32, i32]
        L.pixsht_execute_batch.argtypes = [vp, i32, i32, pvp, pvp, i32]
        L.pixsht_plan_set_stream.argtypes = [vp, vp, i32]
        L.pixsht_get_timings.argtypes = [vp, ctypes.POINTER(dbl)]
        L.pixsht_plan_set_stage_families.argtypes = [vp, i32, i32]
        L.pixsht_plan_set_polconv.argtypes = [vp, i32]
        L.pixsht_ring_pixarea.argtypes = [ctypes.POINTER(Geom), ctypes.POINTER(dbl)]
        L.pixsht_stage_alm2phase.argtypes = [vp, i32, pvp, i32, vp, vp, ctypes.c_int64, vp]
        L.pixsht_stage_phase2alm.argtypes = [vp, i32, vp, ctypes.c_int64, i32, vp, pvp, vp]
        L.pixsht_stage_phase2map.argtypes = [vp, i32, vp, i32, i32, pvp, vp]
        L.pixsht_stage_map2phase.argtypes = [vp, i32, pvp, i32, i32, vp, vp]
        L.pixsht_alm2cl.argtypes = [i32, i32, vp, vp, ctypes.POINTER(dbl), i32, i32, i32]
        L.pixsht_plan_work.argtypes = [vp, i32, ctypes.POINTER(dbl)]
        L.pixsht_plan_work_per_m.argtypes = [vp, i32, ctypes.POINTER(dbl)]
        L.pixsht_phase_row_len.argtypes = [vp]
        L.pixsht_phase_row_len.restype = ctypes.c_int64
        L.pixsht_shared_alloc.argtypes = [i32, ctypes.c_size_t, pvp, ctypes.c_char_p]
        L.pixsht_shared_open.argtypes = [i32, ctypes.c_char_p, pvp]
        L.pixsht_shared_close.argtypes = [vp]
        L.pixsht_shared_free.argtypes = [vp]
        L.pixsht_nalm.argtypes = [i32, i32]
        L.pixsht_nalm.restype = ctypes.c_int64
        L.pixsht_plan_info.argtypes = [vp, ctypes.POINTER(ctypes.c_int32)]
        L.pixsht_plan_weights.argtypes = [vp, ctypes.POINTER(dbl), ctypes.POINTER(dbl)]
        L.pixsht_last_error.restype = ctypes.c_char_p
        L.pixsht_version.restype = ctypes.c_char_p
        L.pixsht_measure_fma_peak.argtypes = [i32, ctypes.POINTER(dbl), ctypes.POINTER(dbl)]
        # libsharp2-compatible shim
        L.sharp_make_geom_info.argtypes = [i32, ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_ssize_t),
                                           ctypes.POINTER(ctypes.c_int), ctypes.POINTER(dbl), ctypes.POINTER(dbl),
                                           ctypes.POINTER(dbl), pvp]
        L.sharp_make_geom_info.restype = None
        L.sharp_destroy_geom_info.argtypes = [vp]
        L.sharp_destroy_geom_info.restype = None
        L.sharp_map_size.argtypes = [vp]
        L.sharp_map_size.restype = ctypes.c_ssize_t
        L.sharp_make_triangular_alm_info.argtypes = [i32, i32, i32, pvp]
        L.sharp_make_triangular_alm_info.restype = None
        L.sharp_destroy_alm_info.argtypes = [vp]
        L.sharp_destroy_alm_info.restype = None
        L.sharp_alm_count.argtypes = [vp]
        L.sharp_alm_count.restype = ctypes.c_ssize_t
        L.sharp_execute.argtypes = [i32, i32, pvp, pvp, vp, vp, i32, ctypes.POINTER(dbl), ctypes.POINTER(ctypes.c_ulonglong)]
        L.sharp_execute.restype = None

    def check(self, rc):
        if rc != PIXSHT_OK:
            raise PixshtError(rc, self.lib.pixsht_last_error().decode())

    def version(self):
        return self.lib.pixsht_version().decode()

    def device_count(self):
        return int(self.lib.pixsht_device_count())

    def measure_fma_peak(self, device=0):
        a, b = ctypes.c_double(0), ctypes.c_double(0)
        self.check(self.lib.pixsht_measure_fma_peak(device, ctypes.byref(a), ctypes.byref(b)))
        return a.value, b.value


_DEFAULT = None


def get_lib():
    """The product library.  Raises PixshtError if it has not been built -- there is no fallback."""
    global _DEFAULT
    if _DEFAULT is None:
        _DEFAULT = PixshtLib()
    return _DEFAULT
