"""The overlapped-call harness: back-to-back calls of one handle whose consecutive grids may overlap on the GPU
(programmatic dependent launch, the history advance folded into the kernel: DESIGN.md §6.0f) -- the FIR on its
constant-bank kernels, the resampler in config 1b's geometry (row-per-lane and sliding-window kernels) and the fused
VFO -> FM chain, on cf32 and integer input. runs() plays every sequence twice, in this process (overlap allowed) and in
a subprocess with QDSP_PDL=0 (every launch serialized), once per test process; the tests that read it
(test_vfofm_overlapped_calls.py, test_iq_formats.py, test_gpu_parity.py) require the two to be bit-identical and check
the streams against the oracle."""
import ctypes as C
import functools
import os
import subprocess
import sys
import tempfile

import numpy as np

from oracle import loader
from tests.test_iq_formats import BLOCK, CHAIN, FMTS, K1, N1, SIZES2, TABLE, _quantized

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIR_TAPS = [127, 601]                      # fir_cplx_kernel, fir_longcplx_kernel
FIR_SIZES = [1 << 18, 1 << 18, 100, 1 << 18, 4 * 288 + 7, 1 << 18, 1 << 18, 2304 * 3, 1 << 18, 1 << 17]
RS_NCALL, RS_N, RS_BLK = 12, 1 << 19, 1 << 17       # resampler, fir_rowcplx_kernel
SL_NCALL, SL_N = 3, 1 << 25                          # resampler, fir_slide4_kernel (calls of >= 2^25 samples)


def _process(L, h, in_ptr, audio_ptr, n, block=BLOCK, iq_ptr=None):
    if np.isscalar(block):
        b, nb, bs = None, 0, int(block)
    else:
        b = np.ascontiguousarray(block, np.int32)
        nb, bs = len(b), 0
    m = L.qdsp_vfofm_process(h, in_ptr, audio_ptr, iq_ptr, n, None if b is None else b.ctypes.data_as(C.POINTER(C.c_int)),
                             nb, bs, None, None)
    assert m >= 0
    return m


def _fir_taps(ntaps):
    rng = np.random.default_rng(ntaps)
    return (rng.standard_normal(ntaps) * np.hanning(ntaps + 2)[1:-1] / np.sqrt(ntaps)).astype(np.float32)


def _resampler_taps():
    return loader.port().blackman_taps(300e3, 4 * 2.4e6 / 127, 2.4e6)


def _vfofm_sequences(L, out):
    from qdsp_b200 import blocks as B, synth

    # 1. the benchmark's pattern: the same input and the same audio buffer for every call
    x1 = synth.cfg2_input(0, N1)
    xin = B.DevBuf.from_numpy(x1)
    v = B.VFOFM(*CHAIN)
    m1 = v.out_count(N1, BLOCK)
    aud = B.DevBuf((m1 + 64) * 4)
    for _ in range(K1):
        assert _process(L, v.h, xin.ptr, aud.ptr, N1) == m1
    out["same_buffers_last"] = aud.to_numpy(np.float32, m1)
    _process(L, v.h, xin.ptr, aud.ptr, N1)           # a 9th call after the read-back: demod state + history carried
    out["same_buffers_next"] = aud.to_numpy(np.float32, m1)
    # 2. distinct buffers per call, a call shorter than the history, calls that end off the decimation grid
    x2 = synth.cfg2_input(0, sum(SIZES2))
    offs = np.concatenate([[0], np.cumsum(SIZES2)])
    ins = [B.DevBuf.from_numpy(x2[offs[i]:offs[i + 1]]) for i in range(len(SIZES2))]
    v2 = B.VFOFM(*CHAIN)
    cnt = [v2.out_count(s, BLOCK) for s in SIZES2]
    auds = [B.DevBuf((c + 64) * 4) for c in cnt]
    for i, s in enumerate(SIZES2):
        assert _process(L, v2.h, ins[i].ptr, auds[i].ptr, s) == cnt[i]
    out["distinct"] = np.concatenate([a.to_numpy(np.float32, c) for a, c in zip(auds, cnt)])
    # 3a. refused: a call's input overlaps the previous call's audio (read after write)
    n3 = 4 * BLOCK
    xa, xb = synth.cfg2_input(0, n3), synth.cfg2_input(n3, n3)
    ina, inb = B.DevBuf.from_numpy(xa), B.DevBuf.from_numpy(xb)
    big = B.DevBuf.from_numpy(synth.cfg2_input(2 * n3, n3))    # call 2 writes its audio over the head of call 3's input
    m3 = v.out_count(n3, BLOCK)
    a1, a3 = B.DevBuf((m3 + 64) * 4), B.DevBuf((m3 + 64) * 4)
    v3 = B.VFOFM(*CHAIN)
    _process(L, v3.h, ina.ptr, a1.ptr, n3)
    _process(L, v3.h, inb.ptr, big.ptr, n3)
    _process(L, v3.h, big.ptr, a3.ptr, n3)
    out["raw_a1"] = a1.to_numpy(np.float32, m3)
    out["raw_big"] = big.to_numpy(np.float32, 2 * n3)
    out["raw_a3"] = a3.to_numpy(np.float32, m3)
    # 3b. refused: a table partition (explicit run() blocks), same buffers
    nt = sum(TABLE)
    intab = B.DevBuf.from_numpy(synth.cfg2_input(0, nt))
    mt = v.out_count(nt, TABLE)
    at = B.DevBuf((mt + 64) * 4)
    v4 = B.VFOFM(*CHAIN)
    for _ in range(3):
        assert _process(L, v4.h, intab.ptr, at.ptr, nt, TABLE) == mt
    out["table_last"] = at.to_numpy(np.float32, mt)
    # 3c. refused: the resampled IQ is wanted, same buffers
    iq = B.DevBuf((m3 + 64) * 8)
    v5 = B.VFOFM(*CHAIN)
    for _ in range(3):
        _process(L, v5.h, ina.ptr, a1.ptr, n3, iq_ptr=iq.ptr)
    out["iq_audio"] = a1.to_numpy(np.float32, m3)
    out["iq_iq"] = iq.to_numpy(np.complex64, m3)
    # 3d. refused: another library kernel between two calls of the handle, same buffers
    xl = B.FrequencyXlator(2.4e6, 100e3)
    xo = B.DevBuf(n3 * 8)
    v6 = B.VFOFM(*CHAIN)
    _process(L, v6.h, ina.ptr, a1.ptr, n3)
    assert L.qdsp_xlator_process(xl.h, inb.ptr, xo.ptr, n3, None) == n3
    _process(L, v6.h, ina.ptr, a1.ptr, n3)
    out["between_audio"] = a1.to_numpy(np.float32, m3)
    # 4. integer input: the first two sequences again
    for fmt in FMTS:
        q1, _ = _quantized(fmt, 0, N1)
        xin = B.DevBuf.from_numpy(q1)
        v = B.VFOFM(*CHAIN)
        v.set_input_format(fmt)
        aud = B.DevBuf((m1 + 64) * 4)
        for _ in range(K1):
            assert _process(L, v.h, xin.ptr, aud.ptr, N1) == m1
        out[fmt + "_same_last"] = aud.to_numpy(np.float32, m1)
        q2, _ = _quantized(fmt, 0, sum(SIZES2))
        ins = [B.DevBuf.from_numpy(q2[2 * offs[i]:2 * offs[i + 1]]) for i in range(len(SIZES2))]
        v2 = B.VFOFM(*CHAIN)
        v2.set_input_format(fmt)
        auds = [B.DevBuf((c + 64) * 4) for c in cnt]
        for i, s in enumerate(SIZES2):
            assert _process(L, v2.h, ins[i].ptr, auds[i].ptr, s) == cnt[i]
        out[fmt + "_distinct"] = np.concatenate([a.to_numpy(np.float32, c) for a, c in zip(auds, cnt)])


def _fir_sequences(out, ntaps):
    # the constant-bank FIR kernels advance the history themselves (one launch per call): 10 back-to-back calls on distinct
    # buffers incl. one shorter than the filter, then the refused case (one output buffer for every call, read back
    # after each call)
    from qdsp_b200 import blocks as B, synth

    taps = _fir_taps(ntaps)
    x = synth.uniform_cf32(13, 0, sum(FIR_SIZES))
    offs = np.concatenate([[0], np.cumsum(FIR_SIZES)])
    ins = [B.DevBuf.from_numpy(x[offs[i]:offs[i + 1]]) for i in range(len(FIR_SIZES))]
    outs = [B.DevBuf(max(s, 2) * 8) for s in FIR_SIZES]
    f = B.FIR(B._TapsWindow(taps))
    for i, s in enumerate(FIR_SIZES):
        assert f.process_device(ins[i].ptr, outs[i].ptr, s) == s
    out[f"fir{ntaps}_distinct"] = np.concatenate([outs[i].to_numpy(np.complex64, s) for i, s in enumerate(FIR_SIZES)])
    big = B.DevBuf(max(FIR_SIZES) * 8)
    f2 = B.FIR(B._TapsWindow(taps))
    parts = []
    for i, s in enumerate(FIR_SIZES):
        f2.process_device(ins[i].ptr, big.ptr, s)
        parts.append(big.to_numpy(np.complex64, s))
    out[f"fir{ntaps}_one_out"] = np.concatenate(parts)
    out[f"fir{ntaps}_history"] = f.get_history()
    for b in ins + outs + [big]:
        b.free()


def _resampler_sequences(out):
    from qdsp_b200 import blocks as B, synth

    win = B.BlackmanWindow(300e3, 4 * 2.4e6 / 127, 2.4e6)
    # 12 back-to-back calls on preloaded distinct device buffers, nothing in between; then the same stream with ONE output
    # buffer for every call (refused: write-after-write), read back after each call, and without any read-back: the last
    # call's result must be the one that stays
    x = synth.uniform_cf32(11, 0, RS_NCALL * RS_N)
    ins = [B.DevBuf.from_numpy(x[i * RS_N:(i + 1) * RS_N]) for i in range(RS_NCALL)]
    outs = [B.DevBuf(RS_N // 4 * 8) for _ in range(RS_NCALL)]
    r = B.PolyphaseResampler(win, 2.4e6, 0.6e6)
    for i in range(RS_NCALL):
        assert r.process_device(ins[i].ptr, outs[i].ptr, RS_N, RS_BLK) == RS_N // 4
    out["resamp_distinct"] = np.concatenate([o.to_numpy(np.complex64, RS_N // 4) for o in outs])
    r2 = B.PolyphaseResampler(win, 2.4e6, 0.6e6)
    parts = []
    for i in range(RS_NCALL):
        r2.process_device(ins[i].ptr, outs[0].ptr, RS_N, RS_BLK)
        parts.append(outs[0].to_numpy(np.complex64, RS_N // 4))
    out["resamp_one_out"] = np.concatenate(parts)
    r3 = B.PolyphaseResampler(win, 2.4e6, 0.6e6)
    for i in range(RS_NCALL):
        r3.process_device(ins[i].ptr, outs[1].ptr, RS_N, RS_BLK)
    out["resamp_one_out_last"] = outs[1].to_numpy(np.complex64, RS_N // 4)
    for b in ins + outs:
        b.free()
    # calls of >= 2^25 samples take the sliding-window kernel: back-to-back calls on distinct buffers
    x2 = synth.uniform_cf32(19, 0, SL_NCALL * SL_N)
    ins = [B.DevBuf.from_numpy(x2[i * SL_N:(i + 1) * SL_N]) for i in range(SL_NCALL)]
    outs = [B.DevBuf(SL_N // 4 * 8) for _ in range(SL_NCALL)]
    r4 = B.PolyphaseResampler(win, 2.4e6, 0.6e6)
    for i in range(SL_NCALL):
        assert r4.process_device(ins[i].ptr, outs[i].ptr, SL_N, SL_N) == SL_N // 4
    out["slide_distinct"] = np.concatenate([o.to_numpy(np.complex64, SL_N // 4) for o in outs])
    for b in ins + outs:
        b.free()


def _sequences():
    """Runs every sequence once; returns {name: array}. Nothing is read back between the calls of a sequence unless
    said so."""
    from qdsp_b200 import lib

    out = {}
    _vfofm_sequences(lib.load(), out)
    for ntaps in FIR_TAPS:
        _fir_sequences(out, ntaps)
    _resampler_sequences(out)
    return out


def _dump(path):
    np.savez(path, **_sequences())


@functools.cache
def runs():
    """(this process's results, the serialized subprocess's results) of _sequences(), computed once per process."""
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "serial.npz")
        env = dict(os.environ, QDSP_PDL="0", PYTHONPATH=ROOT)
        code = f"from tests.overlapped import _dump; _dump({path!r}); print('ok')"
        r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=env, capture_output=True, text=True, timeout=1800)
        assert r.returncode == 0 and "ok" in r.stdout, r.stdout + r.stderr
        with np.load(path) as z:
            serial = dict(z)
    return _sequences(), serial
