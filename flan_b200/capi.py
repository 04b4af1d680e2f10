"""ctypes binding of the C ABI in include/flan_b200.h (libflan_b200.so).

There is no fallback: if the CUDA library is missing or no device is usable this raises.
"""
import ctypes
import os

from . import build

_i64 = ctypes.c_int64
_vp = ctypes.c_void_p
_int = ctypes.c_int
_f = ctypes.c_float

OK, INVALID, UNSUPPORTED, CUDA, CANCELLED, NOMEM = range(6)

MAX_DEVICES = 16


class ShardedAudio(ctypes.Structure):
    _fields_ = [("channels", _int), ("n", _i64), ("shards", _int),
                ("lo", _i64 * MAX_DEVICES), ("hi", _i64 * MAX_DEVICES),
                ("own_lo", _i64 * MAX_DEVICES), ("own_hi", _i64 * MAX_DEVICES),
                ("d", _vp * MAX_DEVICES)]


class ShardedPV(ctypes.Structure):
    _fields_ = [("channels", _int), ("frames", _i64), ("bins", _int),
                ("sample_rate", _f), ("analysis_rate", _f), ("window_size", _int), ("shards", _int),
                ("frame_begin", _i64 * (MAX_DEVICES + 1)), ("d", _vp * MAX_DEVICES)]


_pa, _pp = ctypes.POINTER(ShardedAudio), ctypes.POINTER(ShardedPV)

# every symbol include/flan_b200.h declares: (name, restype, argtypes)
SYMBOLS = [
    ("flan_b200_device_count", _int, []),
    ("flan_b200_create", _int, [_int, ctypes.POINTER(_vp)]),
    ("flan_b200_destroy", None, [_vp]),
    ("flan_b200_last_error", ctypes.c_char_p, [_vp]),
    ("flan_b200_set_stream", _int, [_vp, _vp]),
    ("flan_b200_synchronize", _int, [_vp]),
    ("flan_b200_wait", _int, [_vp, _vp]),
    ("flan_b200_wait_copies", _int, [_vp, _vp]),
    ("flan_b200_trim", _int, [_vp]),
    ("flan_b200_host_register", _int, [_vp, _vp, ctypes.c_size_t]),
    ("flan_b200_host_unregister", _int, [_vp, _vp]),
    ("flan_b200_convert_to_pv_h2d", _int, [_vp, _vp, _vp, _int, _i64, _f, _int, _int, _int, _vp, _vp]),
    ("flan_b200_convert_to_audio_d2h", _int, [_vp, _vp, _int, _i64, _int, _f, _f, _int, _vp, _vp, _vp, ctypes.POINTER(_vp)]),
    ("flan_b200_sm_count", _int, [_vp]),
    ("flan_b200_launch_count", _i64, [_vp]),
    ("flan_b200_set_timing", _int, [_vp, _int]),
    ("flan_b200_kernel_time", _int, [_vp, _int, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(_i64)]),
    ("flan_b200_trace", _int, [_vp, ctypes.POINTER(_int), ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double), _int, ctypes.POINTER(_int)]),
    ("flan_b200_malloc", _int, [_vp, ctypes.c_size_t, ctypes.POINTER(_vp)]),
    ("flan_b200_free", _int, [_vp, _vp]),
    ("flan_b200_upload", _int, [_vp, _vp, _vp, ctypes.c_size_t]),
    ("flan_b200_download", _int, [_vp, _vp, _vp, ctypes.c_size_t]),
    ("flan_b200_num_frames", _i64, [_i64, _int]),
    ("flan_b200_hop_from_rates", _int, [_f, _f]),
    ("flan_b200_analysis_rate", _f, [_f, _int]),
    ("flan_b200_convert_to_pv", _int, [_vp, _vp, _int, _i64, _f, _int, _int, _int, _vp, _vp]),
    ("flan_b200_convert_to_pv_range", _int, [_vp, _vp, _i64, _i64, _i64, _int, _i64, _f, _int, _int, _int, _i64, _i64, _vp, _i64]),
    ("flan_b200_convert_to_audio", _int, [_vp, _vp, _int, _i64, _int, _f, _f, _int, _vp, _vp, ctypes.POINTER(_int)]),
    ("flan_b200_phase_summary", _int, [_vp, _vp, _i64, _int, _i64, _i64, _int, _f, _f, _int, _vp]),
    ("flan_b200_phase_carry", _int, [_vp, _vp, _int, _int, _int, _vp]),
    ("flan_b200_convert_to_audio_range", _int, [_vp, _vp, _i64, _int, _i64, _i64, _i64, _int, _f, _f, _int, _vp, _int, _vp, _i64, _i64, _i64]),
    ("flan_b200_convert_to_audio_range_head", _int, [_vp, _vp, _i64, _int, _i64, _i64, _i64, _int, _f, _f, _int, _vp, _int, _vp, _i64, _i64, _i64, _vp]),
    ("flan_b200_exchange_create", _int, [_vp, _int, _int, _int, _int, _i64, ctypes.POINTER(_vp)]),
    ("flan_b200_exchange_destroy", None, [_vp]),
    ("flan_b200_exchange_handle", _int, [_vp, _vp]),
    ("flan_b200_exchange_connect", _int, [_vp, _vp]),
    ("flan_b200_exchange_state_slot", _int, [_vp, ctypes.POINTER(_vp)]),
    ("flan_b200_exchange_put_state", _int, [_vp, _vp]),
    ("flan_b200_exchange_get_states", _int, [_vp, ctypes.POINTER(_vp)]),
    ("flan_b200_exchange_release_states", _int, [_vp]),
    ("flan_b200_exchange_put_halo", _int, [_vp, _vp, _i64, _int, _i64, _vp]),
    ("flan_b200_exchange_add_halo", _int, [_vp, _vp, _i64, _int, _i64]),
    ("flan_b200_add", _int, [_vp, _vp, _vp, _i64]),
    ("flan_b200_mid_side", _int, [_vp, _vp, _vp, _i64]),
    ("flan_b200_repitch", _int, [_vp, _vp, _int, _i64, _int, _f, _vp, _i64, _int, _int, _vp]),
    ("flan_b200_modify_frequency", _int, [_vp, _vp, _int, _i64, _int, _f, _vp, _i64, _int, _vp, _int, _vp]),
    ("flan_b200_stretch_map", _int, [_vp, _vp, _i64, _int, _i64, _int, _f, _f, _vp]),
    ("flan_b200_modify_time_frames", _int, [_vp, _vp, _i64, _int, _i64, _int, _f, _f, ctypes.POINTER(_i64)]),
    ("flan_b200_modify_time", _int, [_vp, _vp, _int, _i64, _int, _f, _f, _vp, _i64, _int, _int, _i64, _vp, _int]),
    ("flan_b200_promise_unchanged", _int, [_vp, _vp]),
    ("flan_b200_hint_resynthesis", _int, [_vp]),
    ("flan_b200_flan_encode", _int, [_vp, _vp, _i64, _f, _f, _vp]),
    ("flan_b200_flan_decode", _int, [_vp, _vp, _i64, _f, _f, _vp]),
    ("flan_b200_save_flan", _int, [_vp, ctypes.c_char_p, _vp, _int, _i64, _int, _f, _f, _int]),
    ("flan_b200_flan_info", _int, [_vp, ctypes.c_char_p, ctypes.POINTER(_int), ctypes.POINTER(_i64), ctypes.POINTER(_int),
                                   ctypes.POINTER(_f), ctypes.POINTER(_f), ctypes.POINTER(_int)]),
    ("flan_b200_load_flan", _int, [_vp, ctypes.c_char_p, _vp, _i64]),
    ("flan_b200_pcm24_encode", _int, [_vp, _vp, _int, _i64, _vp]),
    ("flan_b200_pcm24_decode", _int, [_vp, _vp, _int, _i64, _vp]),
    ("flan_b200_save_wav", _int, [_vp, ctypes.c_char_p, _vp, _int, _i64, _f]),
    ("flan_b200_wav_info", _int, [_vp, ctypes.c_char_p, ctypes.POINTER(_int), ctypes.POINTER(_i64), ctypes.POINTER(_f)]),
    ("flan_b200_load_wav", _int, [_vp, ctypes.c_char_p, _vp, _i64]),
    ("flan_b200_multi_create", _int, [ctypes.POINTER(_int), _int, ctypes.POINTER(_vp)]),
    ("flan_b200_multi_destroy", None, [_vp]),
    ("flan_b200_multi_last_error", ctypes.c_char_p, [_vp]),
    ("flan_b200_multi_device_count", _int, [_vp]),
    ("flan_b200_multi_ctx", _vp, [_vp, _int]),
    ("flan_b200_multi_synchronize", _int, [_vp]),
    ("flan_b200_multi_time_begin", _int, [_vp]),
    ("flan_b200_multi_time_end", _int, [_vp, ctypes.POINTER(ctypes.c_double)]),
    ("flan_b200_multi_plan", _int, [_vp, _int, _i64, _int, _int, _int, ctypes.POINTER(_int), ctypes.POINTER(_i64)]),
    ("flan_b200_multi_scatter_audio", _int, [_vp, _vp, _int, _i64, _int, _int, _int, _pa]),
    ("flan_b200_multi_convert_to_pv", _int, [_vp, _pa, _f, _int, _int, _int, _pp]),
    ("flan_b200_multi_convert_to_audio", _int, [_vp, _pp, _pa]),
    ("flan_b200_multi_hint_resynthesis", _int, [_vp]),
    ("flan_b200_multi_promise_unchanged", _int, [_vp, _pp]),
    ("flan_b200_multi_gather_audio", _int, [_vp, _pa, _vp]),
    ("flan_b200_multi_gather_pv", _int, [_vp, _pp, _vp, _int, _vp]),
    ("flan_b200_multi_repitch", _int, [_vp, _pp, _vp, _i64, _int, _int, _pp]),
    ("flan_b200_multi_stretch", _int, [_vp, _pp, _vp, _i64, _int, _int, _pp]),
    ("flan_b200_multi_modify_time", _int, [_vp, _pp, _vp, _i64, _int, _int, _pp]),
    ("flan_b200_multi_free_audio", _int, [_vp, _pa]),
    ("flan_b200_multi_free_pv", _int, [_vp, _pp]),
    ("flan_b200_multi_convert_to_pv_host", _int, [_vp, _vp, _int, _i64, _f, _int, _int, _int, _pp]),
    ("flan_b200_multi_convert_to_audio_host", _int, [_vp, _pp, _vp, ctypes.POINTER(_int)]),
    ("flan_b200_convert_to_pv_host", _int, [_vp, _vp, _int, _i64, _f, _int, _int, _int, _int, _vp, _vp]),
    ("flan_b200_convert_to_audio_host", _int, [_vp, _vp, _int, _i64, _int, _f, _f, _int, _int, _vp, _vp, ctypes.POINTER(_int)]),
]

_libs = {}


class FlanB200Error(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("flan_b200 error %d: %s" % (code, msg))
        self.code = code


def load(path=None):
    """Load libflan_b200.so (built in-tree by flan_b200.build). Raises if it cannot be loaded.
    path: another build of the same library (the FLAN_B200_DEBUG development build of tools/experiments)."""
    path = path or os.environ.get("FLAN_B200_LIB") or build.lib_path()
    if path in _libs:
        return _libs[path]
    if not os.path.exists(path):
        raise FileNotFoundError(
            "%s is missing: run `python -m flan_b200.build` (nvcc). flan_b200 has no CPU fallback." % path)
    lib = ctypes.CDLL(path)
    for name, res, args in SYMBOLS:
        fn = getattr(lib, name)          # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _libs[path] = lib
    return lib


class Context:
    """Owns a flan_b200_ctx bound to one CUDA device."""

    def __init__(self, device=0, lib_path=None):
        self.lib = load(lib_path)
        h = _vp()
        rc = self.lib.flan_b200_create(device, ctypes.byref(h))
        if rc != OK:
            raise FlanB200Error(rc, self.lib.flan_b200_last_error(None).decode())
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            self.lib.flan_b200_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def check(self, rc):
        if rc != OK:
            raise FlanB200Error(rc, self.lib.flan_b200_last_error(self.h).decode())

    def call(self, name, *args):
        self.check(getattr(self.lib, name)(self.h, *args))
