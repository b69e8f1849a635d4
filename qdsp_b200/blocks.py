"""Host-side mirror of the reference's ``dsp::`` block interface over the C ABI.

Class names, constructor/`init` argument order and setter names follow the reference headers
(``src/dsp/{window,filter,resampling,processing,demodulator,pll,vfo}.h``); the thread-per-block
`start()/stop()` machinery is not reproduced here — a block's `run()` body is `process(...)`, which
enqueues sm_100a kernels on a CUDA stream. (The C++ mirror with `stream<T>`/`generic_block` lives in
``include/dsp``.)  Two calling styles:

* ``process(x, block=...)``            numpy in -> numpy out (H2D, kernels, D2H; convenience / tests)
* ``process_device(in_ptr, out_ptr, n, ...)``  raw device pointers, asynchronous (bench / pipelines)
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import lib as _lib
from . import synth as _synth
from .lib import CF32, F32, QdspError, check


def _L():
    return _lib.load()


def _fptr(a: np.ndarray):
    return a.ctypes.data_as(C.POINTER(C.c_float))


def _iptr(a):
    return None if a is None else a.ctypes.data_as(C.POINTER(C.c_int))


class DevBuf:
    """A device allocation owned by Python (cudaMalloc through the C ABI)."""

    def __init__(self, nbytes: int):
        _lib.require_device()
        self.nbytes = int(nbytes)
        self.ptr = check(_L().qdsp_malloc_device(max(self.nbytes, 16)), "qdsp_malloc_device")

    @classmethod
    def from_numpy(cls, a: np.ndarray, stream=None) -> "DevBuf":
        a = np.ascontiguousarray(a)
        b = cls(a.nbytes)
        if a.nbytes:
            check(_L().qdsp_copy_h2d(b.ptr, a.ctypes.data, a.nbytes, stream), "h2d")
            check(_L().qdsp_stream_sync(stream), "sync")
        return b

    def to_numpy(self, dtype, count: int, stream=None, offset_bytes: int = 0) -> np.ndarray:
        out = np.empty(count, dtype)
        if out.nbytes:
            check(_L().qdsp_stream_sync(stream), "sync")
            check(_L().qdsp_copy_d2h(out.ctypes.data, self.ptr + offset_bytes, out.nbytes, stream), "d2h")
            check(_L().qdsp_stream_sync(stream), "sync")
        return out

    def free(self):
        if getattr(self, "ptr", None):
            _L().qdsp_free_device(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def _iq_format(fmt, scale=None, offset=None):
    """'cs16' / 'cs8' / 'cu8' (or the QDSP_* code), with the usual scale / offset unless given -> (name, code, s, o)."""
    names = {v: k for k, v in _synth.IQ_CODES.items()}
    name = names.get(fmt, fmt)
    if name not in _synth.IQ_FORMATS:
        raise ValueError(f"unknown integer IQ format {fmt!r}: one of {sorted(_synth.IQ_FORMATS)}")
    _, s0, o0 = _synth.IQ_FORMATS[name]
    return name, _synth.IQ_CODES[name], float(s0 if scale is None else scale), float(o0 if offset is None else offset)


def _iq_input(x, name):
    """The caller's input for the handle's input format: complex64 samples (name None) or interleaved integer pairs."""
    if name is None:
        x = np.ascontiguousarray(x, np.complex64)
        return x, len(x)
    x = np.ascontiguousarray(x).reshape(-1)
    return _iq_input_checked(x, name)


def _iq_input_checked(x, name):
    """As _iq_input, without a copy: for caller-owned (pinned) buffers, which must already have the right type."""
    want = np.dtype(np.complex64 if name is None else _synth.IQ_FORMATS[name][0])
    if x.dtype != want or not x.flags.c_contiguous or (name is not None and x.size % 2):
        raise TypeError(f"{name or 'cf32'} input is a contiguous {want} array" + (" of (re, im) pairs" if name else ""))
    return x, (x.size if name is None else x.size // 2)


class _InputFormat:
    """set_input_format() of the handles that read integer IQ (qdsp_*_set_input_format)."""

    _in_fmt = None   # None = cf32, else the format name

    def set_input_format(self, fmt, scale=None, offset=None):
        """fmt: 'cs16' / 'cs8' / 'cu8' (scale / offset default to the usual ones, synth.IQ_FORMATS), or 'cf32' / CF32."""
        if fmt in ("cf32", CF32):
            check(getattr(_L(), self._set_fmt)(self.h, CF32, 1.0, 0.0), self._set_fmt)
            self._in_fmt = None
            return
        name, code, sc, off = _iq_format(fmt, scale, offset)
        check(getattr(_L(), self._set_fmt)(self.h, code, sc, off), self._set_fmt)
        self._in_fmt = name


def _blocks_arg(n: int, block):
    """block: None/int -> uniform partition (block_size); list/array -> explicit sizes."""
    if block is None:
        return None, 0, 0
    if np.isscalar(block):
        return None, 0, int(block)
    b = np.ascontiguousarray(block, dtype=np.int32)
    if int(b.sum()) != n:
        raise ValueError("block sizes must sum to the input length")
    return b, len(b), 0


def _nblocks(n: int, block) -> int:
    if block is None:
        return 1 if n else 0
    if np.isscalar(block):
        return (n + int(block) - 1) // int(block)
    return len(block)


# ---------------------------------------------------------------------------------------------
# windows (reference src/dsp/window.h)
# ---------------------------------------------------------------------------------------------
class generic_window:
    def getTapCount(self) -> int:  # noqa: N802 (reference naming)
        raise NotImplementedError

    def createTaps(self, tapCount: int | None = None, factor: float = 1.0) -> np.ndarray:  # noqa: N802
        raise NotImplementedError


class BlackmanWindow(generic_window):
    """filter_window::BlackmanWindow (window.h:13-76): init(cutoff, transWidth, sampleRate)."""

    def __init__(self, cutoff: float, transWidth: float, sampleRate: float):
        self.init(cutoff, transWidth, sampleRate)

    def init(self, cutoff, transWidth, sampleRate):
        self._cutoff, self._transWidth, self._sampleRate = float(cutoff), float(transWidth), float(sampleRate)

    def setSampleRate(self, v):
        self._sampleRate = float(v)

    def setCutoff(self, v):
        self._cutoff = float(v)

    def setTransWidth(self, v):
        self._transWidth = float(v)

    def getTapCount(self) -> int:
        return int(_L().qdsp_blackman_tap_count(self._cutoff, self._transWidth, self._sampleRate))

    def createTaps(self, tapCount=None, factor=1.0) -> np.ndarray:
        n = self.getTapCount() if tapCount is None else int(tapCount)
        t = np.empty(n, np.float32)
        _L().qdsp_blackman_taps(self._cutoff, self._transWidth, self._sampleRate, _fptr(t), n, float(factor))
        return t


class BlackmanBandpassWindow(BlackmanWindow):
    """filter_window::BlackmanBandpassWindow (window.h:78-148)."""

    def __init__(self, cutoff, transWidth, offset, sampleRate):
        self.init(cutoff, transWidth, offset, sampleRate)

    def init(self, cutoff, transWidth, offset, sampleRate):
        super().init(cutoff, transWidth, sampleRate)
        self._offset = float(offset)

    def setOffset(self, v):
        self._offset = float(v)

    def createTaps(self, tapCount=None, factor=1.0) -> np.ndarray:
        n = self.getTapCount() if tapCount is None else int(tapCount)
        t = np.empty(n, np.float32)
        _L().qdsp_blackman_bandpass_taps(self._cutoff, self._transWidth, self._offset, self._sampleRate, _fptr(t), n,
                                         float(factor))
        return t


class RRCTaps(generic_window):
    """filter_window::RRCTaps (window.h:150-231): init(tapCount, sampleRate, baudRate, alpha)."""

    def __init__(self, tapCount, sampleRate, baudRate, alpha):
        self._tapCount, self._sampleRate, self._baudRate, self._alpha = int(tapCount), float(sampleRate), float(baudRate), float(alpha)

    def getTapCount(self) -> int:
        return self._tapCount

    def createTaps(self, tapCount=None, factor=1.0) -> np.ndarray:
        n = self._tapCount if tapCount is None else int(tapCount)
        t = np.zeros(n | 1, np.float32)
        _L().qdsp_rrc_taps(n, self._sampleRate, self._baudRate, self._alpha, _fptr(t))
        return t[:n] if n == (n | 1) else t


class _TapsWindow(generic_window):
    """Adapter: a fixed tap vector presented as a window (tests, custom designs)."""

    def __init__(self, taps):
        self.taps = np.ascontiguousarray(taps, np.float32)

    def getTapCount(self):
        return len(self.taps)

    def createTaps(self, tapCount=None, factor=1.0):
        return (self.taps * np.float32(factor)).astype(np.float32)


def rates_to_ratio(inSampleRate: float, outSampleRate: float) -> tuple[int, int]:
    i, d = C.c_int(), C.c_int()
    _L().qdsp_rates_to_ratio(float(inSampleRate), float(outSampleRate), C.byref(i), C.byref(d))
    return i.value, d.value


def resamp_schedule(interp: int, decim: int, count: int):
    n = (count * interp) // decim
    ph, ix = np.empty(n, np.int32), np.empty(n, np.int32)
    _L().qdsp_resamp_schedule(interp, decim, count, _iptr(ph), _iptr(ix))
    return ph, ix


# ---------------------------------------------------------------------------------------------
# base class for stream blocks
# ---------------------------------------------------------------------------------------------
class _Block:
    in_dtype = np.complex64
    out_dtype = np.complex64
    _destroy = None

    def __init__(self):
        self.h = None
        self.stream = None

    def _out_capacity(self, n: int, block) -> int:
        return n

    def _run(self, in_ptr, out_ptr, n, block):
        raise NotImplementedError

    def process_device(self, in_ptr, out_ptr, n, block=None, stream=None) -> int:
        self.stream = stream
        return int(check(self._run(in_ptr, out_ptr, int(n), block), type(self).__name__))

    def process(self, x, block=None) -> np.ndarray:
        x = np.ascontiguousarray(x, dtype=self.in_dtype)
        n = len(x)
        din = DevBuf.from_numpy(x)
        cap = self._out_capacity(n, block)
        dout = DevBuf(max(cap, 1) * np.dtype(self.out_dtype).itemsize)
        self.stream = None
        m = int(check(self._run(din.ptr, dout.ptr, n, block), type(self).__name__))
        y = dout.to_numpy(self.out_dtype, m)
        din.free()
        dout.free()
        return y

    def close(self):
        if self.h and self._destroy:
            getattr(_L(), self._destroy)(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# ---------------------------------------------------------------------------------------------
# FIR / resampling (reference filter.h, resampling.h)
# ---------------------------------------------------------------------------------------------
class FIR(_Block):
    """dsp::FIR<T>: init(in, window). `dtype` is np.complex64 (complex_t) or np.float32."""

    _destroy = "qdsp_fir_destroy"

    def __init__(self, window: generic_window, dtype=np.complex64):
        super().__init__()
        _lib.require_device()
        self.in_dtype = self.out_dtype = np.dtype(dtype).type
        # an even RRC count is rounded up inside createTaps (window.h:186); like the reference's FIR, use the first
        # getTapCount() taps of what it wrote
        self.taps = np.ascontiguousarray(window.createTaps(window.getTapCount())[:window.getTapCount()])
        kind = CF32 if self.in_dtype is np.complex64 else F32
        self.h = check(_L().qdsp_fir_create(kind, _fptr(self.taps), len(self.taps)), "qdsp_fir_create")

    def updateWindow(self, window: generic_window):  # noqa: N802
        self.taps = np.ascontiguousarray(window.createTaps(window.getTapCount())[:window.getTapCount()])
        check(_L().qdsp_fir_set_taps(self.h, _fptr(self.taps), len(self.taps)), "qdsp_fir_set_taps")

    def set_variant(self, v: int):
        _L().qdsp_fir_set_variant(self.h, v)

    def history_len(self) -> int:
        return _L().qdsp_fir_history_len(self.h)

    def import_tail(self, tail_ptr, src_device=-1, stream=None):
        check(_L().qdsp_fir_import_tail(self.h, tail_ptr, src_device, stream), "qdsp_fir_import_tail")

    def process_halo_device(self, halo_ptr, in_ptr, out_ptr, n, stream=None) -> int:
        """One call whose (tapCount-1)-sample history is read straight from `halo_ptr` (may be peer-mapped); None = zeros."""
        return int(check(_L().qdsp_fir_process_halo(self.h, halo_ptr, in_ptr, out_ptr, int(n), stream), "qdsp_fir_process_halo"))

    def set_history(self, hist: np.ndarray):
        hist = np.ascontiguousarray(hist, self.in_dtype)
        assert len(hist) == self.history_len()
        check(_L().qdsp_fir_set_history(self.h, hist.ctypes.data), "qdsp_fir_set_history")

    def get_history(self) -> np.ndarray:
        out = np.empty(self.history_len(), self.in_dtype)
        check(_L().qdsp_fir_get_history(self.h, out.ctypes.data), "qdsp_fir_get_history")
        return out

    def reset(self):
        check(_L().qdsp_fir_reset(self.h))

    def _run(self, in_ptr, out_ptr, n, block):
        return _L().qdsp_fir_process(self.h, in_ptr, out_ptr, n, self.stream)


class PolyphaseResampler(_Block):
    """dsp::PolyphaseResampler<T>: init(in, window, inSampleRate, outSampleRate)."""

    _destroy = "qdsp_resamp_destroy"

    def __init__(self, window: generic_window, inSampleRate: float, outSampleRate: float, dtype=np.complex64):
        super().__init__()
        _lib.require_device()
        self.in_dtype = self.out_dtype = np.dtype(dtype).type
        self._interp, self._decim = rates_to_ratio(inSampleRate, outSampleRate)
        self.taps = window.createTaps(window.getTapCount(), float(self._interp))
        kind = CF32 if self.in_dtype is np.complex64 else F32
        self.h = check(_L().qdsp_resamp_create(kind, _fptr(self.taps), len(self.taps), self._interp, self._decim),
                       "qdsp_resamp_create")
        self.last_out_counts = None

    def getInterpolation(self):  # noqa: N802
        return self._interp

    def getDecimation(self):  # noqa: N802
        return self._decim

    def updateWindow(self, window: generic_window):  # noqa: N802
        self.taps = window.createTaps(window.getTapCount(), float(self._interp))
        check(_L().qdsp_resamp_set_taps(self.h, _fptr(self.taps), len(self.taps)), "qdsp_resamp_set_taps")

    def calcOutSize(self, n: int) -> int:  # noqa: N802
        return int(_L().qdsp_resamp_out_count(self.h, n))

    def tapsPerPhase(self) -> int:  # noqa: N802
        return _L().qdsp_resamp_taps_per_phase(self.h)

    def set_variant(self, v: int):
        _L().qdsp_resamp_set_variant(self.h, v)

    def reset(self):
        check(_L().qdsp_resamp_reset(self.h))

    def _out_capacity(self, n, block):
        return (n * self._interp) // self._decim + 16

    def _run(self, in_ptr, out_ptr, n, block):
        b, nb, bs = _blocks_arg(n, block)
        oc = np.zeros(max(_nblocks(n, block), 1), np.int32)
        r = _L().qdsp_resamp_process(self.h, in_ptr, out_ptr, n, _iptr(b), nb, bs, _iptr(oc), self.stream)
        self.last_out_counts = oc[: _nblocks(n, block)]
        return r

    def schedule_device(self, n: int, block=None):
        """(phase, index) of every output as computed on the device."""
        b, nb, bs = _blocks_arg(n, block)
        cap = self._out_capacity(n, block)
        dp, di = DevBuf(cap * 4), DevBuf(cap * 8)
        m = int(check(_L().qdsp_resamp_schedule_device(self.h, n, _iptr(b), nb, bs, dp.ptr, di.ptr, None)))
        return dp.to_numpy(np.int32, m), di.to_numpy(np.int64, m)


class PowerDecimator(_Block):
    """dsp::PowerDecimator: init(in, power)."""

    def __init__(self, power: int):
        super().__init__()
        _lib.require_device()
        self._power = int(power)

    def setPower(self, power):  # noqa: N802
        self._power = int(power)

    def _run(self, in_ptr, out_ptr, n, block):
        return _L().qdsp_power_decim_process(self._power, in_ptr, out_ptr, n, self.stream)


# ---------------------------------------------------------------------------------------------
# processing / demodulation (reference processing.h, demodulator.h, vfo.h)
# ---------------------------------------------------------------------------------------------
class FrequencyXlator(_Block):
    """dsp::FrequencyXlator<complex_t>: init(in, sampleRate, freq)."""

    _destroy = "qdsp_xlator_destroy"

    def __init__(self, sampleRate: float, freq: float):
        super().__init__()
        _lib.require_device()
        self._sampleRate, self._freq = float(sampleRate), float(freq)
        self.h = check(_L().qdsp_xlator_create(self._sampleRate, self._freq), "qdsp_xlator_create")

    def setSampleRate(self, v):  # noqa: N802
        self._sampleRate = float(v)
        _L().qdsp_xlator_set_frequency(self.h, self._sampleRate, self._freq)

    def setFrequency(self, v):  # noqa: N802
        self._freq = float(v)
        _L().qdsp_xlator_set_frequency(self.h, self._sampleRate, self._freq)

    def getFrequency(self):  # noqa: N802
        return self._freq

    def phase_delta(self) -> complex:
        re, im = C.c_float(), C.c_float()
        _L().qdsp_xlator_get_phase_delta(self.h, C.byref(re), C.byref(im))
        return complex(re.value, im.value)

    def get_phase(self) -> complex:
        re, im = C.c_float(), C.c_float()
        _L().qdsp_xlator_get_phase(self.h, C.byref(re), C.byref(im))
        return complex(re.value, im.value)

    def set_phase(self, p: complex):
        _L().qdsp_xlator_set_phase(self.h, float(p.real), float(p.imag))

    def _run(self, in_ptr, out_ptr, n, block):
        return _L().qdsp_xlator_process(self.h, in_ptr, out_ptr, n, self.stream)


class FloatFMDemod(_Block):
    """dsp::FloatFMDemod: init(in, sampleRate, deviation) -> float audio."""

    _destroy = "qdsp_fmdemod_destroy"
    out_dtype = np.float32
    _stereo = 0

    def __init__(self, sampleRate: float, deviation: float):
        super().__init__()
        _lib.require_device()
        self.h = check(_L().qdsp_fmdemod_create(float(sampleRate), float(deviation), self._stereo))

    def get_phase(self) -> float:
        return float(_L().qdsp_fmdemod_get_phase(self.h))

    def set_phase(self, v: float):
        check(_L().qdsp_fmdemod_set_phase(self.h, float(v)))

    def _run(self, in_ptr, out_ptr, n, block):
        return _L().qdsp_fmdemod_process(self.h, in_ptr, out_ptr, n, self.stream)


class FMDemod(FloatFMDemod):
    """dsp::FMDemod: same demodulator writing stereo_t {l = r = audio} (viewed as complex64)."""

    out_dtype = np.complex64
    _stereo = 1


class StereoFMDemod(_Block):
    """dsp::StereoFMDemod: init(in, sampleRate, deviation) -> stereo_t (viewed as complex64: l = re, r = im)."""

    _destroy = "qdsp_stereofm_destroy"

    def __init__(self, sampleRate: float, deviation: float):
        super().__init__()
        _lib.require_device()
        self.h = check(_L().qdsp_stereofm_create(float(sampleRate), float(deviation)), "qdsp_stereofm_create")

    def _run(self, in_ptr, out_ptr, n, block):
        b, nb, bs = _blocks_arg(n, block)
        return _L().qdsp_stereofm_process(self.h, in_ptr, out_ptr, n, _iptr(b), nb, bs, self.stream)


class VFO:
    """dsp::VFO (vfo.h): FrequencyXlator(-offset) -> PolyphaseResampler with the auto-designed window,
    run block by block as two kernels (the unfused composition; `VFOFM` is the fused pass)."""

    def __init__(self, offset, inSampleRate, outSampleRate, bandWidth):
        self.init(offset, inSampleRate, outSampleRate, bandWidth)

    def init(self, offset, inSampleRate, outSampleRate, bandWidth):
        self._offset, self._in, self._out, self._bw = float(offset), float(inSampleRate), float(outSampleRate), float(bandWidth)
        cutoff = min(self._bw, min(self._in, self._out)) / 2.0
        self.xlator = FrequencyXlator(self._in, -self._offset)
        self.win = BlackmanWindow(cutoff, cutoff, self._in)
        interp, _ = rates_to_ratio(self._in, self._out)
        self.win.setSampleRate(np.float32(self._in) * np.float32(interp))
        self.resamp = PolyphaseResampler(self.win, self._in, self._out)

    def setOffset(self, offset):  # noqa: N802
        self._offset = float(offset)
        self.xlator.setFrequency(-self._offset)

    def process(self, x, block=None) -> np.ndarray:
        x = np.ascontiguousarray(x, np.complex64)
        return self.resamp.process(self.xlator.process(x), block)


class VFOFM(_InputFormat, _Block):
    """Fused VFO -> FloatFMDemod (one kernel; translated and resampled IQ stay on chip). After set_input_format('cs16' |
    'cs8' | 'cu8'), process / process_host take interleaved integer pairs (converted to cf32 on the GPU)."""

    _destroy = "qdsp_vfofm_destroy"
    _set_fmt = "qdsp_vfofm_set_input_format"
    out_dtype = np.float32

    def __init__(self, offset, inSampleRate, outSampleRate, bandWidth, deviation):
        super().__init__()
        _lib.require_device()
        self.h = check(_L().qdsp_vfofm_create(float(offset), float(inSampleRate), float(outSampleRate),
                                              float(bandWidth), float(deviation)), "qdsp_vfofm_create")
        t, i, d = C.c_int(), C.c_int(), C.c_int()
        _L().qdsp_vfofm_design(self.h, C.byref(t), C.byref(i), C.byref(d))
        self.tapCount, self._interp, self._decim = t.value, i.value, d.value
        self.want_iq = False
        self.last_iq = None
        self.last_out_counts = None

    def setOffset(self, offset):  # noqa: N802
        check(_L().qdsp_vfofm_set_offset(self.h, float(offset)))

    def set_variant(self, v: int):
        _L().qdsp_vfofm_set_variant(self.h, v)

    def get_phase(self) -> complex:
        re, im = C.c_float(), C.c_float()
        _L().qdsp_vfofm_get_phase(self.h, C.byref(re), C.byref(im))
        return complex(re.value, im.value)

    def set_phase(self, p: complex):
        check(_L().qdsp_vfofm_set_phase(self.h, float(p.real), float(p.imag)))

    def reset(self):
        check(_L().qdsp_vfofm_reset(self.h))

    def seek(self, start: int):
        check(_L().qdsp_vfofm_seek(self.h, int(start)))

    def history_len(self) -> int:
        return _L().qdsp_vfofm_history_len(self.h)

    def import_tail(self, tail_ptr, src_device=-1, stream=None):
        check(_L().qdsp_vfofm_import_tail(self.h, tail_ptr, src_device, stream))

    def out_count(self, n, block=None) -> int:
        b, nb, bs = _blocks_arg(n, block)
        return int(check(_L().qdsp_vfofm_out_count(self.h, n, _iptr(b), nb, bs)))

    def process_replay(self, x, block, ckpt: np.ndarray, want_iq=False):
        """DEBUG: the chain with the reference's recursive float32 NCO replayed from per-512-sample phase checkpoints
        (`ckpt`: complex64, one per 512-sample run of every run() block). Returns audio (and the resampled IQ)."""
        x = np.ascontiguousarray(x, np.complex64)
        n = len(x)
        ck = np.ascontiguousarray(ckpt, np.complex64).view(np.float32)
        din = DevBuf.from_numpy(x)
        cap = self._out_capacity(n, block)
        dout = DevBuf(max(cap, 1) * 4)
        diq = DevBuf(max(cap, 1) * 8) if want_iq else None
        b, nb, bs = _blocks_arg(n, block)
        m = int(check(_L().qdsp_vfofm_process_replay(self.h, din.ptr, dout.ptr, diq.ptr if diq else None, n, _iptr(b), nb, bs,
                                                     _fptr(ck), len(ck) // 2, None), "qdsp_vfofm_process_replay"))
        y = dout.to_numpy(np.float32, m)
        iq = diq.to_numpy(np.complex64, m) if diq else None
        din.free()
        dout.free()
        if diq:
            diq.free()
        return (y, iq) if want_iq else y

    def process_host(self, x: np.ndarray, block: int) -> np.ndarray:
        """The host-buffer entry point (qdsp_vfofm_process_host): pinned host in / out, chunked H2D | kernel | D2H."""
        x, n = _iq_input(x, self._in_fmt)
        L = _L()
        hin = L.qdsp_malloc_pinned(max(x.nbytes, 1))
        cap = self._out_capacity(n, block)
        hout = L.qdsp_malloc_pinned(max(cap, 1) * 4)
        try:
            C.memmove(hin, x.ctypes.data, x.nbytes)
            m = int(check(L.qdsp_vfofm_process_host(self.h, hin, hout, n, int(block), None), "qdsp_vfofm_process_host"))
            y = np.empty(m, np.float32)
            C.memmove(y.ctypes.data, hout, m * 4)
        finally:
            L.qdsp_free_pinned(hin)
            L.qdsp_free_pinned(hout)
        return y

    def _out_capacity(self, n, block):
        return (n * self._interp) // self._decim + 16

    def _run(self, in_ptr, out_ptr, n, block, iq_ptr=None):
        b, nb, bs = _blocks_arg(n, block)
        oc = np.zeros(max(_nblocks(n, block), 1), np.int32)
        r = _L().qdsp_vfofm_process(self.h, in_ptr, out_ptr, iq_ptr, n, _iptr(b), nb, bs, _iptr(oc), self.stream)
        self.last_out_counts = oc[: _nblocks(n, block)]
        return r

    def process(self, x, block=None) -> np.ndarray:
        if not self.want_iq and self._in_fmt is None:
            return super().process(x, block)
        x, n = _iq_input(x, self._in_fmt)
        din = DevBuf.from_numpy(x)
        cap = self._out_capacity(n, block)
        dout, diq = DevBuf(cap * 4), (DevBuf(cap * 8) if self.want_iq else None)
        self.stream = None
        m = int(check(self._run(din.ptr, dout.ptr, n, block, diq.ptr if diq else None), "VFOFM"))
        if diq:
            self.last_iq = diq.to_numpy(np.complex64, m)
        return dout.to_numpy(np.float32, m)

    def process_host_into(self, x: np.ndarray, out: np.ndarray, block_size: int, stream=None) -> int:
        """End-to-end call with caller-owned HOST buffers (pinned for real overlap): chunked H2D/compute/D2H inside.
        `x` is complex64, or interleaved integer pairs after set_input_format."""
        x, n = _iq_input_checked(x, self._in_fmt)
        return int(check(_L().qdsp_vfofm_process_host(self.h, x.ctypes.data, out.ctypes.data, n, int(block_size),
                                                      stream), "qdsp_vfofm_process_host"))


class Channelizer(_InputFormat, _Block):
    """nch x [VFO -> FloatFMDemod] fed by one Splitter (routing.h:47-57): every channel reads the same
    device-resident wideband buffer; output is [nch, n_out] float32. set_input_format as VFOFM (the channelizer's
    kernels read the input converted to cf32). process_iq also returns every channel's complex baseband."""

    _destroy = "qdsp_channelizer_destroy"
    _set_fmt = "qdsp_channelizer_set_input_format"
    out_dtype = np.float32

    def __init__(self, offsets, inSampleRate, outSampleRate, bandWidth, deviation):
        super().__init__()
        _lib.require_device()
        self.offsets = np.ascontiguousarray(offsets, np.float32)
        self.nch = len(self.offsets)
        self.h = check(_L().qdsp_channelizer_create(self.nch, _fptr(self.offsets), float(inSampleRate),
                                                    float(outSampleRate), float(bandWidth), float(deviation)))
        t, i, d = C.c_int(), C.c_int(), C.c_int()
        _L().qdsp_channelizer_design(self.h, C.byref(t), C.byref(i), C.byref(d))
        self.tapCount, self._interp, self._decim = t.value, i.value, d.value

    def set_variant(self, v: int):
        _L().qdsp_channelizer_set_variant(self.h, v)

    def seek(self, start: int):
        """Time-sharding: the next call's first sample is sample `start` of the stream (include/qdsp_b200.h)."""
        check(_L().qdsp_channelizer_seek(self.h, int(start)))

    def reset(self):
        check(_L().qdsp_channelizer_reset(self.h))

    def set_offsets(self, offsets):
        """VFO::setOffset for every channel, from the next call on: each NCO's phase is continuous at the current stream
        position, a channel whose offset is unchanged keeps its NCO bit for bit, and every other piece of state carries
        on. Synchronises the device. Raises QdspError (handle unchanged) for a wrong length or a non-finite offset."""
        offs = np.ascontiguousarray(offsets, np.float32)
        if offs.shape != (self.nch,):
            raise ValueError(f"set_offsets takes {self.nch} offsets, got shape {offs.shape}")
        check(_L().qdsp_channelizer_set_offsets(self.h, _fptr(offs)), "qdsp_channelizer_set_offsets")
        self.offsets = offs

    @property
    def fft_form(self) -> bool:
        """True if the next call with a suitable partition takes the FFT polyphase form (the offsets form the uniform
        256-channel comb and the variant is 0)."""
        return bool(_L().qdsp_channelizer_fft_form(self.h))

    def process_device(self, in_ptr, out_ptr, n, out_stride, block=None, stream=None) -> int:
        b, nb, bs = _blocks_arg(n, block)
        return int(check(_L().qdsp_channelizer_process(self.h, in_ptr, out_ptr, int(out_stride), int(n), _iptr(b), nb,
                                                       bs, stream), "qdsp_channelizer_process"))

    def process(self, x, block=None) -> np.ndarray:
        x, n = _iq_input(x, self._in_fmt)
        stride = (n * self._interp) // self._decim + 16
        din, dout = DevBuf.from_numpy(x), DevBuf(self.nch * stride * 4)
        m = self.process_device(din.ptr, dout.ptr, n, stride, block)
        y = dout.to_numpy(np.float32, self.nch * stride).reshape(self.nch, stride)[:, :m].copy()
        return y

    def process_device_iq(self, in_ptr, iq_ptr, audio_ptr, n, out_stride, block=None, stream=None) -> int:
        """As process_device, and also every channel's complex baseband (the VFO output, before the FM demodulator):
        channel c at iq_ptr + c * out_stride complex64 elements. audio_ptr may be None (no audio stored; the demodulator
        state advances as if it had been)."""
        b, nb, bs = _blocks_arg(n, block)
        return int(check(_L().qdsp_channelizer_process_iq(self.h, in_ptr, iq_ptr, audio_ptr, int(out_stride), int(n), _iptr(b),
                                                          nb, bs, stream), "qdsp_channelizer_process_iq"))

    def process_iq(self, x, block=None, audio=True):
        """Complex baseband of every channel, [nch, n_out] complex64 -- the input of any complex-baseband block (AMDemod,
        SSBDemod, Squelch, ComplexAGC, CostasLoop, ...). With audio=True returns (iq, audio [nch, n_out] float32)."""
        x, n = _iq_input(x, self._in_fmt)
        stride = (n * self._interp) // self._decim + 16
        din, diq = DevBuf.from_numpy(x), DevBuf(self.nch * stride * 8)
        dout = DevBuf(self.nch * stride * 4) if audio else None
        m = self.process_device_iq(din.ptr, diq.ptr, dout.ptr if audio else None, n, stride, block)
        iq = diq.to_numpy(np.complex64, self.nch * stride).reshape(self.nch, stride)[:, :m].copy()
        if not audio:
            return iq
        return iq, dout.to_numpy(np.float32, self.nch * stride).reshape(self.nch, stride)[:, :m].copy()


class IQConverter(_Block):
    """Integer IQ from a radio front end -> complex_t (qdsp_iq_convert_process): y = (float(x) + offset) * scale per
    component. Feeds any cf32 block (VFO, PSKDemod, ...). process() takes interleaved integer pairs."""

    out_dtype = np.complex64

    def __init__(self, fmt, scale=None, offset=None):
        super().__init__()
        self.fmt, self.code, self.scale, self.offset = _iq_format(fmt, scale, offset)
        self.in_dtype = _synth.IQ_FORMATS[self.fmt][0]

    def _run(self, in_ptr, out_ptr, n, block):
        return _L().qdsp_iq_convert_process(self.code, self.scale, self.offset, in_ptr, out_ptr, n, self.stream)

    def process(self, x, block=None) -> np.ndarray:
        x, n = _iq_input(x, self.fmt)
        din, dout = DevBuf.from_numpy(x), DevBuf(max(n, 1) * 8)
        self.stream = None
        m = int(check(self._run(din.ptr, dout.ptr, n, None), "IQConverter"))
        return dout.to_numpy(np.complex64, m)


class Spectrum(_InputFormat, _Block):
    """Welch power spectrum of a complex64 stream (qdsp_spectrum_*; an addition, the reference has none). Row r is the
    mean of |FFT(window * frame)|^2 over frames r*average .. r*average + average - 1, frame f = samples
    [f*hop, f*hop + fftSize), FFT-shifted (column 0 is -fs/2), linear float32 power. hop defaults to fftSize, window to
    rectangular. Rows are a pure function of the stream: samples of rows not yet complete stay in the handle.
    After set_input_format('cs16' | 'cs8' | 'cu8'), process takes interleaved integer pairs (read and converted by the
    frames kernel itself) and process_device a pointer to them."""

    _destroy = "qdsp_spectrum_destroy"
    _set_fmt = "qdsp_spectrum_set_input_format"
    out_dtype = np.float32

    def __init__(self, fftSize, window=None, hop=None, average=1):
        super().__init__()
        _lib.require_device()
        self.fftSize = int(fftSize)
        self.hop = self.fftSize if hop is None else int(hop)
        self.average = int(average)
        w = None
        if window is not None:
            w = np.ascontiguousarray(window, np.float32)
            if w.shape != (self.fftSize,):
                raise ValueError(f"window must hold fftSize = {self.fftSize} values")
        self.h = check(_L().qdsp_spectrum_create(self.fftSize, None if w is None else _fptr(w), self.hop, self.average),
                       "qdsp_spectrum_create")

    def out_rows(self, n) -> int:
        """Rows the next call of n samples completes (host arithmetic)."""
        return int(check(_L().qdsp_spectrum_out_rows(self.h, int(n)), "qdsp_spectrum_out_rows"))

    def process_device(self, in_ptr, out_ptr, n, stream=None) -> int:
        """in_ptr: n complex64 samples (8-byte aligned), or n integer pairs after set_input_format (aligned to the pair);
        out_ptr: room for out_rows(n) rows of fftSize floats."""
        return int(check(_L().qdsp_spectrum_process(self.h, in_ptr, out_ptr, int(n), stream), "qdsp_spectrum_process"))

    def process(self, x) -> np.ndarray:
        x, n = _iq_input(x, self._in_fmt)
        rows = self.out_rows(n)
        din, dout = DevBuf.from_numpy(x), DevBuf(max(rows, 1) * self.fftSize * 4)
        m = self.process_device(din.ptr, dout.ptr, n)
        return dout.to_numpy(np.float32, m * self.fftSize).reshape(m, self.fftSize)

    def reset(self):
        check(_L().qdsp_spectrum_reset(self.h), "qdsp_spectrum_reset")


# ---------------------------------------------------------------------------------------------
# recurrent blocks (reference filter.h BFMDeemp, processing.h AGCs, pll.h CostasLoop)
# ---------------------------------------------------------------------------------------------
class BFMDeemp(_Block):
    """dsp::BFMDeemp: init(in, sampleRate, tau); stereo_t stream viewed as complex64 (l=re, r=im)."""

    _destroy = "qdsp_deemp_destroy"

    def __init__(self, sampleRate, tau):
        super().__init__()
        _lib.require_device()
        self.h = check(_L().qdsp_deemp_create(float(sampleRate), float(tau)))

    def get_state(self):
        l, r = C.c_float(), C.c_float()
        check(_L().qdsp_deemp_get_state(self.h, C.byref(l), C.byref(r)))
        return l.value, r.value

    def set_state(self, l, r):
        check(_L().qdsp_deemp_set_state(self.h, float(l), float(r)))

    def _run(self, in_ptr, out_ptr, n, block):
        return _L().qdsp_deemp_process(self.h, in_ptr, out_ptr, n, self.stream)


class AGC(_Block):
    """dsp::AGC: init(in, fallRate, sampleRate); float stream; result depends on the run() partition."""

    _destroy = "qdsp_agc_destroy"
    in_dtype = np.float32
    out_dtype = np.float32

    def __init__(self, fallRate, sampleRate):
        super().__init__()
        _lib.require_device()
        self.h = check(_L().qdsp_agc_create(float(fallRate), float(sampleRate)))

    def get_state(self) -> float:
        v = C.c_float()
        check(_L().qdsp_agc_get_state(self.h, C.byref(v)))
        return v.value

    def _run(self, in_ptr, out_ptr, n, block):
        b, nb, bs = _blocks_arg(n, block)
        return _L().qdsp_agc_process(self.h, in_ptr, out_ptr, n, _iptr(b), nb, bs, self.stream)


class ComplexAGC(_Block):
    """dsp::ComplexAGC: init(in, setPoint, maxGain, rate)."""

    _destroy = "qdsp_cagc_destroy"

    def __init__(self, setPoint, maxGain, rate):
        super().__init__()
        _lib.require_device()
        self.h = check(_L().qdsp_cagc_create(float(setPoint), float(maxGain), float(rate)))

    def get_state(self) -> float:
        v = C.c_float()
        check(_L().qdsp_cagc_get_state(self.h, C.byref(v)))
        return v.value

    def set_state(self, g):
        check(_L().qdsp_cagc_set_state(self.h, float(g)))

    def _run(self, in_ptr, out_ptr, n, block):
        return _L().qdsp_cagc_process(self.h, in_ptr, out_ptr, n, self.stream)


class FeedForwardAGC(_Block):
    """dsp::FeedForwardAGC<T>: init(in); returns the valid (toProcess) outputs of each call."""

    _destroy = "qdsp_ffagc_destroy"

    def __init__(self, dtype=np.complex64):
        super().__init__()
        _lib.require_device()
        self.in_dtype = self.out_dtype = np.dtype(dtype).type
        self.h = check(_L().qdsp_ffagc_create(CF32 if self.in_dtype is np.complex64 else F32))

    def _run(self, in_ptr, out_ptr, n, block):
        return _L().qdsp_ffagc_process(self.h, in_ptr, out_ptr, n, self.stream)


class CostasLoop(_Block):
    """dsp::CostasLoop<ORDER>: init(in, loopBandwidth)."""

    _destroy = "qdsp_costas_destroy"

    def __init__(self, order: int, loopBandwidth: float):
        super().__init__()
        _lib.require_device()
        self.h = check(_L().qdsp_costas_create(int(order), float(loopBandwidth)))

    def set_chunking(self, chunk: int, warmup: int):
        _L().qdsp_costas_set_chunking(self.h, int(chunk), int(warmup))

    def get_state(self) -> np.ndarray:
        st = np.zeros(4, np.float32)
        check(_L().qdsp_costas_get_state(self.h, _fptr(st)))
        return st

    def set_state(self, st):
        st = np.ascontiguousarray(st, np.float32)
        check(_L().qdsp_costas_set_state(self.h, _fptr(st)))

    def last_residual(self) -> float:
        return float(_L().qdsp_costas_last_residual(self.h))

    def _run(self, in_ptr, out_ptr, n, block):
        return _L().qdsp_costas_process(self.h, in_ptr, out_ptr, n, self.stream)


__all__ = [n for n in dir() if not n.startswith("_")]


# ---------------------------------------------------------------------------------------------
# element-wise / layout / per-block-statistic blocks (reference math.h, audio.h, convertion.h,
# processing.h Volume / DelayImag / Squelch / Threshold, demodulator.h AMDemod / SSBDemod)
# stereo_t streams are viewed as complex64 (l = re, r = im), like everywhere else in this module.
# ---------------------------------------------------------------------------------------------
MATH_ADD, MATH_SUB, MATH_MUL = 0, 1, 2
(LAYOUT_MONO_TO_STEREO, LAYOUT_CHANNELS_TO_STEREO, LAYOUT_STEREO_TO_MONO, LAYOUT_STEREO_TO_CHANNELS,
 LAYOUT_COMPLEX_TO_STEREO, LAYOUT_COMPLEX_TO_REAL, LAYOUT_COMPLEX_TO_IMAG, LAYOUT_REAL_TO_COMPLEX) = range(8)


class _Binary:
    """Two-input block (math.h): process(a, b) -> out. Mismatched lengths produce nothing, like the reference's
    `if (a_count != b_count) { flush; return 0; }` (math.h:26-30)."""

    _op = MATH_ADD

    def __init__(self, dtype=np.complex64):
        _lib.require_device()
        self.dtype = np.dtype(dtype)
        self._code = CF32 if self.dtype == np.complex64 else F32
        self.stream = None

    def process_device(self, a_ptr, b_ptr, out_ptr, n, stream=None) -> int:
        return int(check(_L().qdsp_math_process(self._op, self._code, a_ptr, b_ptr, out_ptr, int(n), stream), type(self).__name__))

    def process(self, a, b) -> np.ndarray:
        a = np.ascontiguousarray(a, dtype=self.dtype)
        b = np.ascontiguousarray(b, dtype=self.dtype)
        if len(a) != len(b):
            return np.empty(0, self.dtype)
        da, db = DevBuf.from_numpy(a), DevBuf.from_numpy(b)
        do = DevBuf(max(a.nbytes, 16))
        m = self.process_device(da.ptr, db.ptr, do.ptr, len(a))
        y = do.to_numpy(self.dtype, m)
        for d in (da, db, do):
            d.free()
        return y


class Add(_Binary):
    """dsp::Add<T>: init(a, b)."""
    _op = MATH_ADD


class Substract(_Binary):
    """dsp::Substract<T> (sic): init(a, b)."""
    _op = MATH_SUB


class Multiply(_Binary):
    """dsp::Multiply<T>: init(a, b); complex product for complex_t."""
    _op = MATH_MUL


class _Layout(_Block):
    _op = 0

    def __init__(self):
        super().__init__()
        _lib.require_device()

    def _run(self, in_ptr, out_ptr, n, block):
        return _L().qdsp_layout_process(self._op, in_ptr, None, out_ptr, None, n, self.stream)


class MonoToStereo(_Layout):
    """dsp::MonoToStereo (audio.h:5-42)."""
    _op, in_dtype, out_dtype = LAYOUT_MONO_TO_STEREO, np.float32, np.complex64


class StereoToMono(_Layout):
    """dsp::StereoToMono (audio.h:96-145)."""
    _op, in_dtype, out_dtype = LAYOUT_STEREO_TO_MONO, np.complex64, np.float32


class ComplexToStereo(_Layout):
    """dsp::ComplexToStereo (convertion.h:5-44)."""
    _op, in_dtype, out_dtype = LAYOUT_COMPLEX_TO_STEREO, np.complex64, np.complex64


class ComplexToReal(_Layout):
    """dsp::ComplexToReal (convertion.h:46-83)."""
    _op, in_dtype, out_dtype = LAYOUT_COMPLEX_TO_REAL, np.complex64, np.float32


class ComplexToImag(_Layout):
    """dsp::ComplexToImag (convertion.h:85-122)."""
    _op, in_dtype, out_dtype = LAYOUT_COMPLEX_TO_IMAG, np.complex64, np.float32


class RealToComplex(_Layout):
    """dsp::RealToComplex (convertion.h:125-170)."""
    _op, in_dtype, out_dtype = LAYOUT_REAL_TO_COMPLEX, np.float32, np.complex64


class ChannelsToStereo:
    """dsp::ChannelsToStereo (audio.h:44-94): process(left, right) -> stereo_t."""

    def __init__(self):
        _lib.require_device()

    def process(self, left, right) -> np.ndarray:
        left = np.ascontiguousarray(left, np.float32)
        right = np.ascontiguousarray(right, np.float32)
        n = len(left)   # the reference interleaves count_l elements whatever count_r is (audio.h:76-80)
        dl, dr, do = DevBuf.from_numpy(left), DevBuf.from_numpy(right), DevBuf(max(n * 8, 16))
        m = int(check(_L().qdsp_layout_process(LAYOUT_CHANNELS_TO_STEREO, dl.ptr, dr.ptr, do.ptr, None, n, None)))
        y = do.to_numpy(np.complex64, m)
        for d in (dl, dr, do):
            d.free()
        return y


class StereoToChannels:
    """dsp::StereoToChannels (audio.h:147-187): process(stereo) -> (left, right)."""

    def __init__(self):
        _lib.require_device()

    def process(self, x):
        x = np.ascontiguousarray(x, np.complex64)
        n = len(x)
        di, dl, dr = DevBuf.from_numpy(x), DevBuf(max(n * 4, 16)), DevBuf(max(n * 4, 16))
        m = int(check(_L().qdsp_layout_process(LAYOUT_STEREO_TO_CHANNELS, di.ptr, None, dl.ptr, dr.ptr, n, None)))
        out = dl.to_numpy(np.float32, m), dr.to_numpy(np.float32, m)
        for d in (di, dl, dr):
            d.free()
        return out


class Volume(_Block):
    """dsp::Volume<T>: init(in, volume). As in the reference, the constructor stores `volume` but leaves the applied
    level at 1.0 until setVolume() is called (processing.h:355-359 vs :371-374)."""

    def __init__(self, volume: float = 1.0, dtype=np.float32):
        super().__init__()
        _lib.require_device()
        self.in_dtype = self.out_dtype = np.dtype(dtype)
        self._code = CF32 if self.in_dtype == np.complex64 else F32
        self._volume, self._level, self._muted = float(volume), 1.0, False

    def setVolume(self, volume):  # noqa: N802
        self._volume = float(volume)
        self._level = float(_L().qdsp_volume_level(self._volume))

    def getVolume(self):  # noqa: N802
        return self._volume

    def setMuted(self, muted):  # noqa: N802
        self._muted = bool(muted)

    def getMuted(self):  # noqa: N802
        return self._muted

    def _run(self, in_ptr, out_ptr, n, block):
        return _L().qdsp_volume_process(self._code, self._level, int(self._muted), in_ptr, out_ptr, n, self.stream)


class Threshold(_Block):
    """dsp::Threshold (processing.h:554-610): uint8 stream of (x > 0)."""
    in_dtype, out_dtype = np.float32, np.uint8

    def __init__(self):
        super().__init__()
        _lib.require_device()

    def _run(self, in_ptr, out_ptr, n, block):
        return _L().qdsp_threshold_process(in_ptr, out_ptr, n, self.stream)


class DelayImag(_Block):
    """dsp::DelayImag (processing.h:300-346)."""
    _destroy = "qdsp_delayimag_destroy"

    def __init__(self):
        super().__init__()
        _lib.require_device()
        self.h = check(_L().qdsp_delayimag_create(), "qdsp_delayimag_create")

    def get_state(self) -> float:
        v = C.c_float()
        check(_L().qdsp_delayimag_get_state(self.h, C.byref(v)))
        return v.value

    def _run(self, in_ptr, out_ptr, n, block):
        return _L().qdsp_delayimag_process(self.h, in_ptr, out_ptr, n, self.stream)


class AMDemod(_Block):
    """dsp::AMDemod (demodulator.h:332-378): |x| minus its mean over the run() block."""
    _destroy = "qdsp_amdemod_destroy"
    out_dtype = np.float32

    def __init__(self):
        super().__init__()
        _lib.require_device()
        self.h = check(_L().qdsp_amdemod_create(), "qdsp_amdemod_create")

    def _run(self, in_ptr, out_ptr, n, block):
        b, nb, bs = _blocks_arg(n, block)
        return _L().qdsp_amdemod_process(self.h, in_ptr, out_ptr, n, _iptr(b), nb, bs, self.stream)


class Squelch(_Block):
    """dsp::Squelch: init(in, level) (processing.h:424-489)."""
    _destroy = "qdsp_squelch_destroy"

    def __init__(self, level: float = -50.0):
        super().__init__()
        _lib.require_device()
        self.h = check(_L().qdsp_squelch_create(float(level)), "qdsp_squelch_create")

    def setLevel(self, level):  # noqa: N802
        _L().qdsp_squelch_set_level(self.h, float(level))

    def getLevel(self):  # noqa: N802
        return float(_L().qdsp_squelch_get_level(self.h))

    def _run(self, in_ptr, out_ptr, n, block):
        b, nb, bs = _blocks_arg(n, block)
        return _L().qdsp_squelch_process(self.h, in_ptr, out_ptr, n, _iptr(b), nb, bs, self.stream)


class SSBDemod(_Block):
    """dsp::SSBDemod: init(in, sampleRate, bandWidth, mode) (demodulator.h:380-497)."""
    _destroy = "qdsp_ssbdemod_destroy"
    out_dtype = np.float32
    MODE_USB, MODE_LSB, MODE_DSB = 0, 1, 2

    def __init__(self, sampleRate: float, bandWidth: float, mode: int):
        super().__init__()
        _lib.require_device()
        self._sampleRate, self._bandWidth, self._mode = float(sampleRate), float(bandWidth), int(mode)
        self.h = check(_L().qdsp_ssbdemod_create(self._sampleRate, self._bandWidth, self._mode), "qdsp_ssbdemod_create")

    def _reconf(self):
        _L().qdsp_ssbdemod_configure(self.h, self._sampleRate, self._bandWidth, self._mode)

    def setSampleRate(self, v):  # noqa: N802
        self._sampleRate = float(v)
        self._reconf()

    def setBandWidth(self, v):  # noqa: N802
        self._bandWidth = float(v)
        self._reconf()

    def setMode(self, v):  # noqa: N802
        self._mode = int(v)
        self._reconf()

    def phase_delta(self) -> complex:
        re, im = C.c_float(), C.c_float()
        _L().qdsp_ssbdemod_get_phase_delta(self.h, C.byref(re), C.byref(im))
        return complex(re.value, im.value)

    def get_phase(self) -> complex:
        re, im = C.c_float(), C.c_float()
        _L().qdsp_ssbdemod_get_phase(self.h, C.byref(re), C.byref(im))
        return complex(re.value, im.value)

    def set_phase(self, p: complex):
        _L().qdsp_ssbdemod_set_phase(self.h, float(p.real), float(p.imag))

    def _run(self, in_ptr, out_ptr, n, block):
        return _L().qdsp_ssbdemod_process(self.h, in_ptr, out_ptr, n, self.stream)


class SineSource:
    """dsp::SineSource: init(blockSize, sampleRate, freq) (source.h:5-71); generate() is one run() call."""

    def __init__(self, blockSize: int, sampleRate: float, freq: float):
        _lib.require_device()
        self._blockSize, self._sampleRate, self._freq = int(blockSize), float(sampleRate), float(freq)
        self.h = check(_L().qdsp_sinesource_create(self._sampleRate, self._freq), "qdsp_sinesource_create")

    def setBlockSize(self, n):  # noqa: N802
        self._blockSize = int(n)

    def getBlockSize(self):  # noqa: N802
        return self._blockSize

    def setSampleRate(self, v):  # noqa: N802
        self._sampleRate = float(v)
        _L().qdsp_sinesource_configure(self.h, self._sampleRate, self._freq)

    def setFrequency(self, v):  # noqa: N802
        self._freq = float(v)
        _L().qdsp_sinesource_configure(self.h, self._sampleRate, self._freq)

    def getFrequency(self):  # noqa: N802
        return self._freq

    def generate_device(self, out_ptr, stream=None) -> int:
        return int(check(_L().qdsp_sinesource_process(self.h, out_ptr, self._blockSize, stream), "SineSource"))

    def generate(self) -> np.ndarray:
        d = DevBuf(max(self._blockSize * 8, 16))
        m = self.generate_device(d.ptr)
        y = d.to_numpy(np.complex64, m)
        d.free()
        return y

    def close(self):
        if self.h:
            _L().qdsp_sinesource_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# ---------------------------------------------------------------------------------------------
# symbol-timing recovery and the PSK / MSK hier blocks (reference clock_recovery.h:68-243, demodulator.h:499-682)
# ---------------------------------------------------------------------------------------------
class MMClockRecovery:
    """dsp::MMClockRecovery<T>: init(in, omega, gainOmega, muGain, omegaRelLimit). `interp_taps` is the reference's
    INTERP_TAPS[129][8] table (src/dsp/interpolation_taps.h), supplied by the caller. process() returns the recovered
    symbols; `last_out_counts` holds the per-run()-block counts."""

    def __init__(self, omega, gainOmega, muGain, omegaRelLimit, interp_taps, dtype=np.complex64):
        _lib.require_device()
        self.dtype = np.dtype(dtype)
        t = np.ascontiguousarray(interp_taps, np.float32)
        if t.shape != (129, 8):
            raise ValueError("interp_taps must be the 129 x 8 INTERP_TAPS table")
        self.h = check(_L().qdsp_mm_create(CF32 if self.dtype == np.complex64 else F32, float(omega), float(gainOmega),
                                           float(muGain), float(omegaRelLimit), _fptr(t)), "qdsp_mm_create")
        self.last_out_counts = None

    def setOmega(self, omega, omegaRelLimit):  # noqa: N802
        check(_L().qdsp_mm_set_omega(self.h, float(omega), float(omegaRelLimit)))

    def setGains(self, omegaGain, muGain):  # noqa: N802
        check(_L().qdsp_mm_set_gains(self.h, float(omegaGain), float(muGain)))

    def setOmegaRelLimit(self, v):  # noqa: N802
        check(_L().qdsp_mm_set_omega_rel_limit(self.h, float(v)))

    def get_state(self) -> np.ndarray:
        st = np.zeros(44, np.float32)
        check(_L().qdsp_mm_get_state(self.h, _fptr(st)))
        return st

    def set_state(self, st):
        st = np.ascontiguousarray(st, np.float32)
        check(_L().qdsp_mm_set_state(self.h, _fptr(st)))

    def max_out(self, n: int) -> int:
        return int(_L().qdsp_mm_max_out(self.h, int(n)))

    def process_device(self, in_ptr, out_ptr, n, block=None, stream=None) -> int:
        b, nb, bs = _blocks_arg(n, block)
        oc = np.zeros(max(_nblocks(n, block), 1), np.int32)
        m = int(check(_L().qdsp_mm_process(self.h, in_ptr, out_ptr, int(n), _iptr(b), nb, bs, _iptr(oc), stream), "MMClockRecovery"))
        self.last_out_counts = oc[:_nblocks(n, block)]
        return m

    def process(self, x, block=None) -> np.ndarray:
        x = np.ascontiguousarray(x, dtype=self.dtype)
        din = DevBuf.from_numpy(x)
        dout = DevBuf(max(self.max_out(len(x)), 1) * self.dtype.itemsize)
        m = self.process_device(din.ptr, dout.ptr, len(x), block)
        y = dout.to_numpy(self.dtype, m)
        din.free()
        dout.free()
        return y

    def close(self):
        if self.h:
            _L().qdsp_mm_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class MSKDemod:
    """dsp::MSKDemod hier block (demodulator.h:499-565): FloatFMDemod -> MMClockRecovery<float>."""

    def __init__(self, sampleRate, deviation, baudRate, interp_taps, omegaGain=(0.01 * 0.01) / 4, muGain=0.01, omegaRelLimit=0.005):
        # like the reference constructor, which forwards only (sampleRate, deviation, baudRate) to init() (:503-505)
        self.demod = FloatFMDemod(sampleRate, deviation)
        self.recov = MMClockRecovery(np.float32(sampleRate) / np.float32(baudRate), (0.01 * 0.01) / 4, 0.01, 0.005, interp_taps, np.float32)

    def process(self, x, block=None) -> np.ndarray:
        x = np.ascontiguousarray(x, np.complex64)
        sizes = [len(x)] if block is None else (list(_as_sizes(len(x), block)))
        off, parts = 0, []
        for s in sizes:
            parts.append(self.demod.process(x[off:off + s]))
            off += s
        y = self.recov.process(np.concatenate(parts) if parts else np.empty(0, np.float32), block)
        self.last_out_counts = self.recov.last_out_counts
        return y


class PSKDemod:
    """dsp::PSKDemod<ORDER, OFFSET> hier block (demodulator.h:567-682):
    ComplexAGC(1, 65535, agcRate) -> FIR<complex_t>(RRCTaps) -> CostasLoop<ORDER> [-> DelayImag] -> MMClockRecovery<complex_t>."""

    def __init__(self, order, offset, sampleRate, baudRate, interp_taps, RRCTapCount=32, RRCAlpha=0.32, agcRate=10e-4,
                 costasLoopBw=0.004, omegaGain=(0.01 * 0.01) / 4, muGain=0.01, omegaRelLimit=0.005):
        self.agc = ComplexAGC(1.0, 65535.0, agcRate)
        self.rrc = FIR(RRCTaps(RRCTapCount, sampleRate, baudRate, RRCAlpha))
        self.demod = CostasLoop(order, costasLoopBw)
        self.delay = DelayImag() if offset else None
        self.recov = MMClockRecovery(np.float32(sampleRate) / np.float32(baudRate), omegaGain, muGain, omegaRelLimit, interp_taps)

    def process(self, x, block=None) -> np.ndarray:
        x = np.ascontiguousarray(x, np.complex64)
        sizes = [len(x)] if block is None else (list(_as_sizes(len(x), block)))
        off, parts = 0, []
        for s in sizes:   # one run() call per block through the sample-rate stages (their state carries in the handles)
            y = self.demod.process(self.rrc.process(self.agc.process(x[off:off + s])))
            if self.delay is not None:
                y = self.delay.process(y)
            parts.append(y)
            off += s
        y = self.recov.process(np.concatenate(parts) if parts else np.empty(0, np.complex64), block)
        self.last_out_counts = self.recov.last_out_counts
        return y


def _as_sizes(n: int, block):
    if np.isscalar(block):
        b = int(block)
        return [b] * (n // b) + ([n % b] if n % b else [])
    return [int(v) for v in block]

