"""Host-side mirror of the reference's receive chain objects, on top of the C ABI.

`ReceiveChain` is `demodulation()` + `biquad1_dac` + `biquad2_dac` (Minimal-SDR.ino:66-81,518-775) for a batch of
independent channels.  Method names follow the reference: `init_FIR()` (.ino:901-930), `tune()` (.ino:328-368),
`setCoefficients`/`setLowpass`/`setNotch` (filter_biquad.h:43-149), `update()`.
"""
import ctypes as C
import json
import os

import numpy as np

from . import capi, design

_HERE = os.path.dirname(os.path.abspath(__file__))


def load_ref_constants():
    """Numeric constants of the sketch (tap tables, tap counts, rates); see tools/extract_ref_constants.py."""
    with open(os.path.join(_HERE, "data", "ref_constants.json")) as f:
        return json.load(f)


class ReceiveChain:
    def __init__(self, n_channels, device=0, max_taps=0, am_q31=False):
        self._L = capi.lib()
        self.n_channels = int(n_channels)
        self.device = device
        h = C.c_void_p()
        st = self._L.msdr_chain_create(C.byref(h), device, self.n_channels, max_taps, capi.FLAG_AM_Q31 if am_q31 else 0)
        if st != capi.OK:
            msg = self._L.msdr_last_error(None)
            raise capi.MsdrError(st, msg.decode() if msg else "")
        self.h = h
        self.K = load_ref_constants()

    # -- lifetime ------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "h", None):
            self._L.msdr_chain_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _rng(self, ch0, nch):
        return int(ch0), int(self.n_channels - ch0 if nch is None else nch)

    def _ck(self, st):
        return capi.check(st, self.h)

    # -- configuration -------------------------------------------------------------------------
    def set_mode(self, mode, ch0=0, nch=None):
        ch0, nch = self._rng(ch0, nch)
        return self._ck(self._L.msdr_chain_set_mode(self.h, ch0, nch, int(mode)))

    def fir_init(self, cI, cQ, ch0=0, nch=None, check=True):
        """arm_fir_init_q15 on the I and Q instances; returns the arm_status-like code when check=False."""
        ch0, nch = self._rng(ch0, nch)
        cI = np.ascontiguousarray(cI, np.int16)
        cQ = np.ascontiguousarray(cQ, np.int16)
        assert cI.size == cQ.size
        st = self._L.msdr_fir_init_q15(self.h, ch0, nch, cI.size, capi.ptr(cI), capi.ptr(cQ))
        return self._ck(st) if check else st

    def set_mode_list(self, mode, channels):
        ch = np.ascontiguousarray(channels, np.uint32)
        return self._ck(self._L.msdr_chain_set_mode_list(self.h, capi.ptr(ch), ch.size, int(mode)))

    def fir_init_list(self, cI, cQ, channels):
        ch = np.ascontiguousarray(channels, np.uint32)
        cI = np.ascontiguousarray(cI, np.int16)
        cQ = np.ascontiguousarray(cQ, np.int16)
        assert cI.size == cQ.size
        return self._ck(self._L.msdr_fir_init_q15_list(self.h, capi.ptr(ch), ch.size, cI.size, capi.ptr(cI), capi.ptr(cQ)))

    def fir_taps(self, ch=0):
        """numTaps of the FIR pair bound to channel ch (0 = not initialised)."""
        return int(self._L.msdr_chain_fir_taps(self.h, int(ch)))

    def fir_set_coefficients(self, cI, cQ, ch0=0, nch=None):
        ch0, nch = self._rng(ch0, nch)
        cI = np.ascontiguousarray(cI, np.int16)
        cQ = np.ascontiguousarray(cQ, np.int16)
        T = self.fir_taps(ch0)  # the C ABI reads the bound tap count from both arrays, like the reference's borrowed pointer
        if T > 0 and not (cI.size == cQ.size == T):
            raise capi.MsdrError(capi.ERR_LENGTH, f"fir_set_coefficients: {cI.size}/{cQ.size} taps given, {T} bound")
        return self._ck(self._L.msdr_fir_set_coefficients(self.h, ch0, nch, capi.ptr(cI), capi.ptr(cQ)))

    def tables_for_mode(self, mode, am_table=None):
        """FIR tables init_FIR() binds for `mode` (Minimal-SDR.ino:904-929)."""
        K = self.K
        if mode in (capi.MODE_USB, capi.MODE_LSB):
            return K["FIR_SSB_I_coeffs"], K["FIR_SSB_Q_coeffs"]
        if mode == capi.MODE_CW:
            return K["FIR_CW_I_coeffs"], K["FIR_CW_Q_coeffs"]
        am = K["FIR_AM_coeffs_bw2800_fs24000"] if am_table is None else am_table
        return am, am

    def init_FIR(self, mode, ch0=0, nch=None, am_table=None):
        cI, cQ = self.tables_for_mode(mode, am_table)
        return self.fir_init(cI, cQ, ch0, nch)

    def tune(self, mode, ch0=0, nch=None, am_table=None, notch=True):
        """The DSP-relevant part of tune() (.ino:328-368): mode, init_FIR(), biquad2 notch at fs/8 (.ino:355-356)."""
        self.set_mode(mode, ch0, nch)
        self.init_FIR(mode, ch0, nch, am_table)
        if notch:
            self.biquad_set_coefficients(1, 0, self.K["biquad2_notch_coef"], ch0, nch)

    def setup_like_sketch(self, mode=capi.MODE_AM, ch0=0, nch=None):
        """setup() (.ino:372-411): biquad1 low-pass at 0.9*IF, Q 0.54 (.ino:391-393), then tune()."""
        self.biquad_set_coefficients(0, 0, self.K["biquad1_lowpass_coef"], ch0, nch)
        self.tune(mode, ch0, nch)

    def biquad_set_coefficients(self, obj, stage, coef, ch0=0, nch=None):
        """AudioFilterBiquad::setCoefficients(stage, const int*) on object obj (0 = biquad1_dac, 1 = biquad2_dac)."""
        ch0, nch = self._rng(ch0, nch)
        coef = np.ascontiguousarray(coef, np.int32)
        assert coef.size == 5
        return self._ck(self._L.msdr_biquad_set_coefficients(self.h, int(obj), ch0, nch, int(stage), capi.ptr(coef)))

    def biquad_set_coefficients_double(self, obj, stage, coef, ch0=0, nch=None):
        """setCoefficients(stage, const double*) (filter_biquad.h:44-52)."""
        return self.biquad_set_coefficients(obj, stage, design.biquad_double_to_int(coef), ch0, nch)

    def setLowpass(self, obj, stage, frequency, q=0.7071, ch0=0, nch=None, fs=None):
        return self.biquad_set_coefficients(obj, stage, design.biquad_lowpass(frequency, q, fs or self.K["AUDIO_SAMPLE_RATE_EXACT"]), ch0, nch)

    def setNotch(self, obj, stage, frequency, q=1.0, ch0=0, nch=None, fs=None):
        return self.biquad_set_coefficients(obj, stage, design.biquad_notch(frequency, q, fs or self.K["AUDIO_SAMPLE_RATE_EXACT"]), ch0, nch)

    def set_anr(self, anr_on, ch0=0, nch=None):
        """ANR_on of the sketch (Minimal-SDR.ino:99): 0 off, 1 LMS notch, 2 LMS noise reduction, between demodulation and the biquads."""
        ch0, nch = self._rng(ch0, nch)
        return self._ck(self._L.msdr_chain_set_anr(self.h, ch0, nch, int(anr_on)))

    def get_anr_state(self, ch):
        st = capi.AnrState()
        self._ck(self._L.msdr_chain_get_anr_state(self.h, int(ch), C.byref(st)))
        return st

    def set_anr_state(self, ch, st):
        return self._ck(self._L.msdr_chain_set_anr_state(self.h, int(ch), C.byref(st)))

    def set_option(self, key, value):
        return self._ck(self._L.msdr_chain_set_option(self.h, key.encode(), int(value)))

    def set_stream(self, cuda_stream_handle):
        """cudaStream_t handle as an int.  0 is what torch reports for its default stream: it is passed on as cudaStreamLegacy
        (handle 1), so the chain's kernels are ordered with work queued there; None = the chain's own non-blocking stream."""
        h = 0 if cuda_stream_handle is None else (int(cuda_stream_handle) or 1)
        return self._ck(self._L.msdr_chain_set_stream(self.h, C.c_void_p(h)))

    # -- the hot path ----------------------------------------------------------------------------
    def update(self, x, out=None):
        """x: int16 [n_channels, n_blocks*128] in HOST memory -> demodulated, biquad-filtered audio, same shape."""
        x = np.asarray(x)
        assert x.dtype == np.int16 and x.ndim == 2 and x.shape[0] == self.n_channels and x.shape[1] % capi.BLOCK == 0
        assert x.strides[1] == 2 and x.strides[0] % 2 == 0
        if out is None:
            out = np.empty((self.n_channels, x.shape[1]), np.int16)
        assert out.dtype == np.int16 and out.shape == x.shape and out.strides[1] == 2
        assert out.strides[0] == x.strides[0], "in/out must share the row stride"
        self._ck(self._L.msdr_chain_update(self.h, capi.ptr(x), capi.ptr(out), x.shape[1] // capi.BLOCK, x.strides[0] // 2))
        return out

    def update_device(self, d_in, d_out, n_blocks, stride):
        """Device pointers (ints), asynchronous on the chain's stream."""
        return self._ck(self._L.msdr_chain_update_device(self.h, C.c_void_p(int(d_in)), C.c_void_p(int(d_out)), int(n_blocks), int(stride)))

    def update_range_device(self, ch0, nch, d_in, d_out, n_blocks, stride):
        """Only channels [ch0, ch0+nch); the buffers hold nch rows."""
        return self._ck(self._L.msdr_chain_update_range_device(self.h, int(ch0), int(nch), C.c_void_p(int(d_in)), C.c_void_p(int(d_out)),
                                                               int(n_blocks), int(stride)))

    def update_list(self, channels, x, out=None):
        """Only the listed chain channels, in list order: row i of x (int16 [len(channels), n_blocks*128], HOST memory) is
        channel channels[i]; returns the audio of those rows, same shape."""
        ch = np.ascontiguousarray(channels, np.uint32).ravel()
        x = np.asarray(x)
        assert x.dtype == np.int16 and x.ndim == 2 and x.shape[0] == ch.size and x.shape[1] % capi.BLOCK == 0
        assert x.strides[1] == 2 and x.strides[0] % 2 == 0
        if out is None:
            out = np.empty(x.shape, np.int16)
        assert out.dtype == np.int16 and out.shape == x.shape and out.strides[1] == 2
        assert out.strides[0] == x.strides[0], "in/out must share the row stride"
        self._ck(self._L.msdr_chain_update_list(self.h, capi.ptr(ch), ch.size, capi.ptr(x), capi.ptr(out), x.shape[1] // capi.BLOCK,
                                                x.strides[0] // 2))
        return out

    def update_list_device(self, channels, d_in, d_out, n_blocks, stride):
        """Only the listed chain channels (host array, any order); device buffers of len(channels) rows, row i = channels[i]."""
        ch = np.ascontiguousarray(channels, np.uint32).ravel()
        return self._ck(self._L.msdr_chain_update_list_device(self.h, capi.ptr(ch), ch.size, C.c_void_p(int(d_in)), C.c_void_p(int(d_out)),
                                                              int(n_blocks), int(stride)))

    # -- raw ADC codes in: the front end (frontend.Frontend) per channel in front of the chain -----------------------------------
    def enable_frontend(self, agc_start=0.25, agc_max=40.0, agc_on=True):
        """(Re)initialise every channel's front end like frontend.Frontend(...): DC-block state 0, AGC at agc_start."""
        return self._ck(self._L.msdr_chain_enable_frontend(self.h, float(agc_start), float(agc_max), int(bool(agc_on))))

    def frontend_preset(self, first_reading, ch0=0, nch=None):
        """AudioInputAnalog::init: hpf_x1 = first ADC reading << 14, hpf_y1 = 0 (input_adc.cpp:59-63)."""
        ch0, nch = self._rng(ch0, nch)
        return self._ck(self._L.msdr_chain_frontend_preset(self.h, ch0, nch, int(first_reading)))

    def frontend_preset_list(self, first_reading, channels):
        """frontend_preset for the listed chain channels (any order) in one call."""
        ch = np.ascontiguousarray(channels, np.uint32).ravel()
        return self._ck(self._L.msdr_chain_frontend_preset_list(self.h, capi.ptr(ch), ch.size, int(first_reading)))

    def update_adc(self, adc, out=None):
        """adc: uint16 raw codes [n_channels, n_blocks*128] in HOST memory -> audio, as frontend.Frontend.update then update()."""
        adc = np.asarray(adc)
        assert adc.dtype == np.uint16 and adc.ndim == 2 and adc.shape[0] == self.n_channels and adc.shape[1] % capi.BLOCK == 0
        assert adc.strides[1] == 2 and adc.strides[0] % 2 == 0
        if out is None:
            out = np.empty((self.n_channels, adc.shape[1]), np.int16)
        assert out.dtype == np.int16 and out.shape == adc.shape and out.strides[1] == 2
        assert out.strides[0] == adc.strides[0], "in/out must share the row stride"
        self._ck(self._L.msdr_chain_update_adc(self.h, capi.ptr(adc), capi.ptr(out), adc.shape[1] // capi.BLOCK, adc.strides[0] // 2))
        return out

    def update_adc_device(self, d_adc, d_out, n_blocks, stride):
        """Device pointers (ints), asynchronous on the chain's stream."""
        return self._ck(self._L.msdr_chain_update_adc_device(self.h, C.c_void_p(int(d_adc)), C.c_void_p(int(d_out)), int(n_blocks), int(stride)))

    def update_adc_range_device(self, ch0, nch, d_adc, d_out, n_blocks, stride):
        """Only channels [ch0, ch0+nch); the buffers hold nch rows."""
        return self._ck(self._L.msdr_chain_update_adc_range_device(self.h, int(ch0), int(nch), C.c_void_p(int(d_adc)), C.c_void_p(int(d_out)),
                                                                   int(n_blocks), int(stride)))

    def update_adc_list(self, channels, adc, out=None):
        """Only the listed chain channels, in list order: row i of adc (uint16 raw codes [len(channels), n_blocks*128], HOST memory)
        is channel channels[i]; returns the audio of those rows, same shape."""
        ch = np.ascontiguousarray(channels, np.uint32).ravel()
        adc = np.asarray(adc)
        assert adc.dtype == np.uint16 and adc.ndim == 2 and adc.shape[0] == ch.size and adc.shape[1] % capi.BLOCK == 0
        assert adc.strides[1] == 2 and adc.strides[0] % 2 == 0
        if out is None:
            out = np.empty(adc.shape, np.int16)
        assert out.dtype == np.int16 and out.shape == adc.shape and out.strides[1] == 2
        assert out.strides[0] == adc.strides[0], "in/out must share the row stride"
        self._ck(self._L.msdr_chain_update_adc_list(self.h, capi.ptr(ch), ch.size, capi.ptr(adc), capi.ptr(out), adc.shape[1] // capi.BLOCK,
                                                    adc.strides[0] // 2))
        return out

    def update_adc_list_device(self, channels, d_adc, d_out, n_blocks, stride):
        """Only the listed chain channels (host array, any order); device buffers of len(channels) rows, row i = channels[i]."""
        ch = np.ascontiguousarray(channels, np.uint32).ravel()
        return self._ck(self._L.msdr_chain_update_adc_list_device(self.h, capi.ptr(ch), ch.size, C.c_void_p(int(d_adc)), C.c_void_p(int(d_out)),
                                                                  int(n_blocks), int(stride)))

    def get_frontend_state(self, ch):
        st = capi.FrontendState()
        self._ck(self._L.msdr_chain_get_frontend_state(self.h, int(ch), C.byref(st)))
        return st

    def set_frontend_state(self, ch, st):
        return self._ck(self._L.msdr_chain_set_frontend_state(self.h, int(ch), C.byref(st)))

    def synchronize(self):
        return self._ck(self._L.msdr_chain_synchronize(self.h))

    def last_update_ms(self):
        ms = C.c_float(0)
        self._ck(self._L.msdr_chain_last_update_ms(self.h, C.byref(ms)))
        return ms.value

    def processor_usage(self, sample_rate_hz):
        """(last, max) load in percent of the block period at sample_rate_hz: AudioProcessorUsage / AudioProcessorUsageMax."""
        a, b = C.c_float(0), C.c_float(0)
        self._ck(self._L.msdr_chain_processor_usage(self.h, float(sample_rate_hz), C.byref(a), C.byref(b)))
        return a.value, b.value

    def processor_usage_max_reset(self):
        return self._ck(self._L.msdr_chain_processor_usage_max_reset(self.h))

    def plan_build_count(self):
        return int(self._L.msdr_chain_plan_build_count(self.h))

    def last_kernel(self):
        return (self._L.msdr_chain_last_kernel(self.h) or b"").decode()

    def launch_count(self):
        return int(self._L.msdr_chain_launch_count(self.h))

    # -- state -------------------------------------------------------------------------------------
    def get_state(self, ch):
        st = capi.ChannelState()
        self._ck(self._L.msdr_chain_get_state(self.h, int(ch), C.byref(st)))
        return st

    def set_state(self, ch, st):
        return self._ck(self._L.msdr_chain_set_state(self.h, int(ch), C.byref(st)))

    # -- snapshots: checkpoint / resume / migration / re-sharding of channel ranges (include/msdr.h, DESIGN.md 7) -----------------
    def snapshot_bytes(self, nch=None):
        return int(self._L.msdr_chain_snapshot_bytes(self.h, int(self.n_channels if nch is None else nch)))

    def snapshot(self, ch0=0, nch=None, out=None):
        """Channels [ch0, ch0+nch) as a uint8 array (tables, modes, ANR switches and all device state).  `out`: a host uint8 array of at
        least snapshot_bytes(nch) bytes to write into, e.g. capi.PinnedBuffer(...).array for PCIe-rate copies."""
        ch0, nch = self._rng(ch0, nch)
        size = self.snapshot_bytes(nch)
        if out is None:
            out = np.empty(size, np.uint8)
        assert out.dtype == np.uint8 and out.flags.c_contiguous and out.size >= size
        self._ck(self._L.msdr_chain_snapshot(self.h, ch0, nch, capi.ptr(out), out.size))
        return out[:size]

    def restore(self, blob, ch0=0, first=0, n=None):
        """Chain channels [ch0, ch0+n) take the state of snapshot channels [first, first+n) (n = None: the rest of the snapshot)."""
        blob = np.ascontiguousarray(blob, np.uint8).reshape(-1)
        if n is None:
            n = capi.snapshot_info(blob)["n_channels"] - int(first)
        return self._ck(self._L.msdr_chain_restore(self.h, int(ch0), capi.ptr(blob), blob.size, int(first), int(n)))

    @staticmethod
    def _device_bytes(tensor):
        assert tensor.is_cuda and str(tensor.dtype) == "torch.uint8" and tensor.is_contiguous(), "a contiguous CUDA uint8 tensor"
        return C.c_void_p(tensor.data_ptr()), tensor.numel()

    def snapshot_device(self, ch0, nch, tensor):
        """Into a CUDA uint8 tensor on the chain's device, asynchronous on the chain's stream (after every earlier update)."""
        p, size = self._device_bytes(tensor)
        return self._ck(self._L.msdr_chain_snapshot_device(self.h, int(ch0), int(nch), p, size))

    def restore_device(self, tensor, ch0=0, first=0, n=None):
        """From a CUDA uint8 tensor on the chain's device; keep the tensor alive until the chain's stream has passed."""
        p, size = self._device_bytes(tensor)
        if n is None:
            n = capi.snapshot_info(tensor[:256].cpu().numpy())["n_channels"] - int(first)
        return self._ck(self._L.msdr_chain_restore_device(self.h, int(ch0), p, size, int(first), int(n)))
