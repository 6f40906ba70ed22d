"""ctypes binding of the C ABI in include/msdr.h (csrc/libmsdr.so).  No computation happens here."""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
BLOCK = 128
MAX_TAPS = 256
MODE_SYNCAM, MODE_AM, MODE_LSB, MODE_USB, MODE_CW = 0, 1, 2, 3, 4  # stations.h:4
FLAG_AM_Q31 = 1
SNAPSHOT_FRONTEND, SNAPSHOT_ANR = 1 << 16, 1 << 17  # msdr_snapshot_info flags: sections the snapshot has
OK, ERR_ARGUMENT, ERR_LENGTH, ERR_CUDA, ERR_UNSUPPORTED, ERR_NOMEM, ERR_NOT_INITIALISED = 0, -1, -2, -100, -101, -102, -103


class MsdrError(RuntimeError):
    def __init__(self, status, msg=""):
        super().__init__(f"msdr status {status}: {msg}")
        self.status = status


class ChannelState(C.Structure):
    _fields_ = [
        ("mode", C.c_int32),
        ("num_taps", C.c_uint32),
        ("fir_set", C.c_int32),
        ("fir_history", C.c_int16 * MAX_TAPS),
        ("biquad_definition", (C.c_int32 * 32) * 2),
        ("syncam_pll", C.c_float * 3),
    ]


class FrontendState(C.Structure):  # msdr_frontend_state
    _fields_ = [
        ("hpf_x1", C.c_int32),
        ("hpf_y1", C.c_int32),
        ("multiplier", C.c_int32),
        ("agc_idx", C.c_int32),
        ("agc_val", C.c_float),
        ("agc_buffer", C.c_int16 * 25),
        ("reserved", C.c_int16),
    ]


class AnrState(C.Structure):  # msdr_anr_state
    _fields_ = [("d", C.c_float * 512), ("w", C.c_float * 64), ("lidx", C.c_float), ("ngamma", C.c_float), ("in_idx", C.c_int32)]


def lib_path():
    # MSDR_LIBMSDR: developer aid, another build of the same library (kernel tuning experiments: tools/build_variant.sh)
    return os.environ.get("MSDR_LIBMSDR") or os.path.join(_HERE, "csrc", "libmsdr.so")


_lib = None

# every symbol include/msdr.h declares: (restype, argtypes)
_i16p, _i32p = C.POINTER(C.c_int16), C.POINTER(C.c_int32)
SYMBOLS = {
    "msdr_chain_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_uint32, C.c_uint32, C.c_uint32]),
    "msdr_chain_destroy": (None, [C.c_void_p]),
    "msdr_chain_set_stream": (C.c_int, [C.c_void_p, C.c_void_p]),
    "msdr_chain_synchronize": (C.c_int, [C.c_void_p]),
    "msdr_last_error": (C.c_char_p, [C.c_void_p]),
    "msdr_chain_channels": (C.c_uint32, [C.c_void_p]),
    "msdr_chain_set_mode": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_int]),
    "msdr_fir_init_q15": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint16, C.c_void_p, C.c_void_p]),
    "msdr_fir_set_coefficients": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p]),
    "msdr_chain_set_mode_list": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_int]),
    "msdr_fir_init_q15_list": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint16, C.c_void_p, C.c_void_p]),
    "msdr_chain_fir_taps": (C.c_int, [C.c_void_p, C.c_uint32]),
    "msdr_chain_processor_usage": (C.c_int, [C.c_void_p, C.c_double, C.POINTER(C.c_float), C.POINTER(C.c_float)]),
    "msdr_chain_processor_usage_max_reset": (C.c_int, [C.c_void_p]),
    "msdr_biquad_set_coefficients": (C.c_int, [C.c_void_p, C.c_int, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p]),
    "msdr_chain_update": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_size_t]),
    "msdr_chain_update_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_size_t]),
    "msdr_chain_update_range_device": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint32, C.c_size_t]),
    "msdr_chain_update_list_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint32, C.c_size_t]),
    "msdr_chain_update_list": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint32, C.c_size_t]),
    "msdr_chain_last_update_ms": (C.c_int, [C.c_void_p, C.POINTER(C.c_float)]),
    "msdr_chain_launch_count": (C.c_uint64, [C.c_void_p]),
    "msdr_chain_plan_build_count": (C.c_uint64, [C.c_void_p]),
    "msdr_chain_last_kernel": (C.c_char_p, [C.c_void_p]),
    "msdr_chain_get_state": (C.c_int, [C.c_void_p, C.c_uint32, C.POINTER(ChannelState)]),
    "msdr_chain_set_state": (C.c_int, [C.c_void_p, C.c_uint32, C.POINTER(ChannelState)]),
    "msdr_chain_set_option": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int]),
    "msdr_host_alloc": (C.c_void_p, [C.c_size_t]),
    "msdr_host_free": (None, [C.c_void_p]),
    "msdr_op_mix_fs4": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_size_t]),
    "msdr_op_fir_fast_q15": (C.c_int, [C.c_int, C.c_uint16, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_size_t]),
    "msdr_op_demod": (C.c_int, [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_size_t]),
    "msdr_op_biquad": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_size_t]),
    "msdr_op_freq_conv": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_size_t]),
    "msdr_op_sqrt_q31": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32]),
    "msdr_op_fir_demod_tc": (C.c_int, [C.c_int, C.c_uint16, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_size_t]),
    "msdr_study_fir_demod_tc_time": (C.c_int, [C.c_int, C.c_uint16, C.c_uint32, C.c_uint32, C.c_int, C.c_int, C.POINTER(C.c_float)]),
    "msdr_study_sqrt_check": (C.c_int, [C.c_int, C.POINTER(C.c_uint64)]),
    "msdr_frontend_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_uint32, C.c_float, C.c_float, C.c_int]),
    "msdr_frontend_destroy": (None, [C.c_void_p]),
    "msdr_frontend_set_stream": (C.c_int, [C.c_void_p, C.c_void_p]),
    "msdr_frontend_synchronize": (C.c_int, [C.c_void_p]),
    "msdr_frontend_last_error": (C.c_char_p, [C.c_void_p]),
    "msdr_frontend_preset": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint16]),
    "msdr_frontend_update": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_size_t]),
    "msdr_frontend_update_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_size_t]),
    "msdr_frontend_get_state": (C.c_int, [C.c_void_p, C.c_uint32, C.POINTER(FrontendState)]),
    "msdr_frontend_set_state": (C.c_int, [C.c_void_p, C.c_uint32, C.POINTER(FrontendState)]),
    "msdr_frontend_launch_count": (C.c_uint64, [C.c_void_p]),
    "msdr_frontend_set_option": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int]),
    "msdr_chain_enable_frontend": (C.c_int, [C.c_void_p, C.c_float, C.c_float, C.c_int]),
    "msdr_chain_frontend_preset": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint16]),
    "msdr_chain_update_adc": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_size_t]),
    "msdr_chain_update_adc_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_size_t]),
    "msdr_chain_update_adc_range_device": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint32, C.c_size_t]),
    "msdr_chain_update_adc_list_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint32, C.c_size_t]),
    "msdr_chain_update_adc_list": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint32, C.c_size_t]),
    "msdr_chain_frontend_preset_list": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint16]),
    "msdr_chain_get_frontend_state": (C.c_int, [C.c_void_p, C.c_uint32, C.POINTER(FrontendState)]),
    "msdr_chain_set_frontend_state": (C.c_int, [C.c_void_p, C.c_uint32, C.POINTER(FrontendState)]),
    "msdr_amp_gain_multiplier": (C.c_int32, [C.c_float]),
    "msdr_op_dac_codes": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_size_t]),
    "msdr_op_amplifier": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_size_t]),
    "msdr_anr_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_uint32]),
    "msdr_anr_destroy": (None, [C.c_void_p]),
    "msdr_anr_set_stream": (C.c_int, [C.c_void_p, C.c_void_p]),
    "msdr_anr_synchronize": (C.c_int, [C.c_void_p]),
    "msdr_anr_last_error": (C.c_char_p, [C.c_void_p]),
    "msdr_anr_update": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_uint32, C.c_size_t]),
    "msdr_anr_update_device": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_uint32, C.c_size_t]),
    "msdr_anr_get_state": (C.c_int, [C.c_void_p, C.c_uint32, C.POINTER(AnrState)]),
    "msdr_anr_set_state": (C.c_int, [C.c_void_p, C.c_uint32, C.POINTER(AnrState)]),
    "msdr_anr_launch_count": (C.c_uint64, [C.c_void_p]),
    "msdr_chain_set_anr": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_int]),
    "msdr_chain_get_anr_state": (C.c_int, [C.c_void_p, C.c_uint32, C.POINTER(AnrState)]),
    "msdr_chain_set_anr_state": (C.c_int, [C.c_void_p, C.c_uint32, C.POINTER(AnrState)]),
    "msdr_syncam_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_uint32]),
    "msdr_syncam_destroy": (None, [C.c_void_p]),
    "msdr_syncam_set_stream": (C.c_int, [C.c_void_p, C.c_void_p]),
    "msdr_syncam_last_error": (C.c_char_p, [C.c_void_p]),
    "msdr_syncam_update": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_size_t]),
    "msdr_syncam_update_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_size_t]),
    "msdr_syncam_get_state": (C.c_int, [C.c_void_p, C.c_uint32, C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(C.c_float)]),
    "msdr_syncam_set_state": (C.c_int, [C.c_void_p, C.c_uint32, C.c_float, C.c_float, C.c_float]),
    "msdr_syncam_constants": (C.c_int, [C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(C.c_float)]),
    "msdr_syncam_launch_count": (C.c_uint64, [C.c_void_p]),
    "msdr_chain_snapshot_bytes": (C.c_size_t, [C.c_void_p, C.c_uint32]),
    "msdr_chain_snapshot": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_size_t]),
    "msdr_chain_snapshot_device": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_size_t]),
    "msdr_chain_restore": (C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p, C.c_size_t, C.c_uint32, C.c_uint32]),
    "msdr_chain_restore_device": (C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p, C.c_size_t, C.c_uint32, C.c_uint32]),
    "msdr_snapshot_info": (C.c_int, [C.c_void_p, C.c_size_t, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]),
    "msdr_version": (C.c_char_p, []),
}


def lib():
    """Load csrc/libmsdr.so (built by __graft_entry__.build() / `make -C minimal-sdr_b200/csrc`)."""
    global _lib
    if _lib is None:
        path = lib_path()
        if not os.path.exists(path):
            raise ImportError(f"{path} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                              "(nvcc, sm_100a). There is no CPU fallback.")
        L = C.CDLL(path)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(L, name)
            fn.restype, fn.argtypes = res, args
        _lib = L
    return _lib


def ptr(a):
    """numpy array (C-contiguous in its last dim) or int address -> void*"""
    if a is None:
        return None
    if isinstance(a, int):
        return C.c_void_p(a)
    return C.c_void_p(a.ctypes.data)


def check(status, handle=None):
    if status != OK:
        msg = lib().msdr_last_error(handle)
        raise MsdrError(status, msg.decode() if msg else "")
    return status


def snapshot_info(blob):
    """msdr_snapshot_info on a host copy of (at least the first 256 bytes of) a snapshot: {n_channels, max_taps_needed, flags}.
    Needs no device; raises MsdrError for a bad magic, a short header or another format version."""
    b = np.ascontiguousarray(blob, np.uint8).reshape(-1)
    n, t, f = C.c_uint32(0), C.c_uint32(0), C.c_uint32(0)
    st = lib().msdr_snapshot_info(ptr(b), b.size, C.byref(n), C.byref(t), C.byref(f))
    if st != OK:
        raise MsdrError(st, "msdr_snapshot_info")
    return {"n_channels": n.value, "max_taps_needed": t.value, "flags": f.value}


class PinnedBuffer:
    """Pinned host memory from msdr_host_alloc, viewed as a numpy array (`.array`).  Keep the object alive while the
    array is in use; freed by `.free()` or on collection."""

    def __init__(self, shape, dtype=np.int16):
        self.nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
        self.ptr = lib().msdr_host_alloc(max(self.nbytes, 16))
        if not self.ptr:
            raise MemoryError("msdr_host_alloc failed")
        self._buf = (C.c_char * self.nbytes).from_address(self.ptr)
        self.array = np.frombuffer(self._buf, dtype=dtype).reshape(shape)

    def free(self):
        if self.ptr:
            self.array = None
            self._buf = None
            lib().msdr_host_free(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass
