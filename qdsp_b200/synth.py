"""Counter-based synthetic IQ generators (SURVEY.md §8d).

Random-access: sample n depends only on (seed, n), so the CPU oracle, the parity tests and the
device generator (csrc/synth.cu, same integer recipe) can materialise any window of a stream
independently and byte-identically. Host-side numpy only; nothing here is on the timed path.
"""
from __future__ import annotations

import numpy as np

_M64 = np.uint64(0xFFFFFFFFFFFFFFFF)


def _splitmix64(z: np.ndarray) -> np.ndarray:
    with np.errstate(over="ignore"):
        z = z + np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z = z ^ (z >> np.uint64(31))
    return z


def uniform_cf32(seed: int, start: int, count: int) -> np.ndarray:
    """U(seed, n): cf32 uniform in [-1,1)^2; re from bits 0..23, im from bits 24..47 of
    splitmix64((seed << 40) ^ n); value = k * 2^-23 - 1 (exact in fp32)."""
    n = np.arange(start, start + count, dtype=np.uint64)
    z = _splitmix64((np.uint64(seed) << np.uint64(40)) ^ n)
    re = (z & np.uint64(0xFFFFFF)).astype(np.float32) * np.float32(2.0 ** -23) - np.float32(1.0)
    im = ((z >> np.uint64(24)) & np.uint64(0xFFFFFF)).astype(np.float32) * np.float32(2.0 ** -23) - np.float32(1.0)
    out = np.empty(count, np.complex64)
    out.real = re
    out.imag = im
    return out


def uniform_f32(seed: int, start: int, count: int) -> np.ndarray:
    return uniform_cf32(seed, start, count).real.copy()


def _frac(n: np.ndarray, f_hz: int, fs_hz: int) -> np.ndarray:
    """frac(n * f / fs) in float64 from exact integer arithmetic (n*f fits int64 for our sizes)."""
    r = (n.astype(np.int64) * np.int64(f_hz)) % np.int64(fs_hz)
    return r.astype(np.float64) / float(fs_hz)


def fm_cf32(start: int, count: int, fs: int, fc: int, fm: int, dev: float, amp: float) -> np.ndarray:
    """FM(n; fc, fm, dev, A) = A * exp(j(2*pi*frac(n*fc/fs) + (dev/fm)*sin(2*pi*frac(n*fm/fs)))),
    float64 evaluation, cast to cf32."""
    n = np.arange(start, start + count, dtype=np.int64)
    ph = 2.0 * np.pi * _frac(n, fc, fs) + (dev / fm) * np.sin(2.0 * np.pi * _frac(n, fm, fs))
    return (amp * np.exp(1j * ph)).astype(np.complex64)


def cfg2_input(start: int, count: int) -> np.ndarray:
    """BASELINE config 2 input: FM(fc=250 kHz, fm=1 kHz, dev=5 kHz, A=0.5) + 0.005*U(2,n) at 2.4 MS/s."""
    return fm_cf32(start, count, 2_400_000, 250_000, 1_000, 5e3, 0.5) + np.float32(0.005) * uniform_cf32(2, start, count)


def cfg4_input(start: int, count: int, nch: int = 256, fs: int = 61_440_000, spacing: int = 240_000) -> np.ndarray:
    """BASELINE config 4 wideband input: sum of nch FM carriers at (k-(nch-1)/2)*spacing,
    fm = 300+10k Hz, dev 5 kHz, A = 1/64, + 0.001*U(4,n)."""
    acc = np.zeros(count, np.complex128)
    n = np.arange(start, start + count, dtype=np.int64)
    for k in range(nch):
        fc = (2 * k - (nch - 1)) * spacing // 2
        fm = 300 + 10 * k
        ph = 2.0 * np.pi * _frac(n, fc, fs) + (5e3 / fm) * np.sin(2.0 * np.pi * _frac(n, fm, fs))
        acc += (1.0 / 64.0) * np.exp(1j * ph)
    return acc.astype(np.complex64) + np.float32(0.001) * uniform_cf32(4, start, count)


def cfg4_offsets(nch: int = 256, spacing: int = 240_000) -> np.ndarray:
    return np.asarray([(2 * k - (nch - 1)) * spacing / 2 for k in range(nch)], dtype=np.float32)


def qpsk_cf32(seed: int, start: int, count: int, sps: int = 4, freq_off: float = 0.01, sigma: float = 0.07,
              am_depth: float = 0.0, am_period: int = 50_000) -> np.ndarray:
    """QPSK symbols held for `sps` samples, rotated by freq_off rad/sample, + sigma*U noise;
    optional slow amplitude modulation (for the AGC cases). Config 5 input."""
    n = np.arange(start, start + count, dtype=np.int64)
    sym = _splitmix64((np.uint64(seed + 77) << np.uint64(40)) ^ (n // sps).astype(np.uint64))
    bits = (sym & np.uint64(3)).astype(np.int64)
    const = np.exp(1j * (np.pi / 4 + np.pi / 2 * bits))
    amp = 1.0 + am_depth * np.sin(2.0 * np.pi * (n % am_period) / am_period)
    sig = amp * const * np.exp(1j * freq_off * n.astype(np.float64))
    return sig.astype(np.complex64) + np.float32(sigma) * uniform_cf32(seed, start, count)


def bpsk_cf32(seed: int, start: int, count: int, sps: int = 4, freq_off: float = 0.01, sigma: float = 0.07) -> np.ndarray:
    """BPSK (+-1) symbols held for `sps` samples, rotated by freq_off rad/sample, + sigma*U noise."""
    n = np.arange(start, start + count, dtype=np.int64)
    sym = _splitmix64((np.uint64(seed + 77) << np.uint64(40)) ^ (n // sps).astype(np.uint64))
    const = 1.0 - 2.0 * (sym & np.uint64(1)).astype(np.float64)
    sig = const * np.exp(1j * freq_off * n.astype(np.float64))
    return sig.astype(np.complex64) + np.float32(sigma) * uniform_cf32(seed, start, count)


def stereo_mpx_fm_cf32(start: int, count: int, fs: int = 240_000, dev: float = 75e3, fl: int = 700, fr: int = 1_100,
                       amp: float = 0.8) -> np.ndarray:
    """Broadcast-FM style baseband: stereo multiplex (L+R, 19 kHz pilot, (L-R) on 38 kHz DSB-SC) frequency-modulated
    with peak deviation `dev` at sample rate `fs`. The phase integral is evaluated in closed form, so any window
    of the stream can be generated independently."""
    n = np.arange(start, start + count, dtype=np.int64)

    def cosint(f, scale=1.0):   # integral of scale*sin(2*pi*f*t) dt, sampled at n/fs (closed form)
        return -scale * np.cos(2.0 * np.pi * _frac(n, f, fs)) / (2.0 * np.pi * f)

    # mpx = 0.45*(L+R) + 0.1*pilot + 0.45*(L-R)*sin(2*pi*38k t), L = sin(2*pi*fl t), R = sin(2*pi*fr t)
    # products of sines expand into sum/difference tones, each integrated in closed form
    integ = 0.45 * (cosint(fl) + cosint(fr)) + 0.1 * cosint(19_000)
    for fa, sgn in ((fl, 1.0), (fr, -1.0)):
        # sin(a) * sin(b) = 0.5*(cos(a-b) - cos(a+b)); integral of cos(2*pi*f t) = sin(2*pi*f t)/(2*pi*f)
        for fb, s2 in ((38_000 - fa, 1.0), (38_000 + fa, -1.0)):
            integ += sgn * 0.45 * 0.5 * s2 * np.sin(2.0 * np.pi * _frac(n, fb, fs)) / (2.0 * np.pi * fb)
    ph = 2.0 * np.pi * dev * integ
    return (amp * np.exp(1j * ph)).astype(np.complex64)


# ---- integer IQ (include/qdsp_b200.h, QDSP_CS16 / QDSP_CS8 / QDSP_CU8) ----------------------------------------------
# format -> (numpy dtype of a component, the usual (scale, offset)); the conversion is y = (float(x) + offset) * scale
IQ_FORMATS = {
    "cs16": (np.int16, 1.0 / 32768, 0.0),
    "cs8": (np.int8, 1.0 / 128, 0.0),
    "cu8": (np.uint8, 1.0 / 128, -127.5),
}
IQ_CODES = {"cs16": 2, "cs8": 3, "cu8": 4}


def iq_to_cf32(raw: np.ndarray, scale: float, offset: float) -> np.ndarray:
    """The library's conversion rule on the host: interleaved integer pairs -> complex64, each step rounded to float32."""
    y = (np.asarray(raw).reshape(-1).astype(np.float32) + np.float32(offset)) * np.float32(scale)
    return y.view(np.complex64)


def quantize_iq(x: np.ndarray, fmt: str, scale: float | None = None, offset: float | None = None) -> np.ndarray:
    """cf32 -> interleaved integer pairs of `fmt` (round to nearest, saturate): the inverse of iq_to_cf32 up to the
    quantisation step. Test inputs as a radio front end would deliver them."""
    dt, s0, o0 = IQ_FORMATS[fmt]
    scale = s0 if scale is None else scale
    offset = o0 if offset is None else offset
    info = np.iinfo(dt)
    f = np.asarray(x, np.complex64).view(np.float32).astype(np.float64)
    return np.clip(np.rint(f / scale - offset), info.min, info.max).astype(dt)
