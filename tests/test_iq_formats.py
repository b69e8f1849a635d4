"""Integer IQ input (cs16 / cs8 / cu8): qdsp_iq_convert_process, and the fused VFO -> FM chain, the channelizer,
process_host and the dsp:: example taking integer input (converted on the GPU, then the cf32 kernels). The reference for
every integer run is the cf32 path fed with the host conversion of the same integers (synth.iq_to_cf32): bit for bit."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

from oracle import loader

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BLOCK = 819_200
CHAIN = (250e3, 2.4e6, 48e3, 48e3, 5e3)
AUDIO_TOL = 1e-4
FMTS = ["cs16", "cs8", "cu8"]
NEW_SYMBOLS = ["qdsp_iq_convert_process", "qdsp_vfofm_set_input_format", "qdsp_channelizer_set_input_format"]
N1, K1 = 20 * BLOCK, 8                     # the benchmark's geometry: 819 200-sample blocks, 20 per call
SIZES2 = [2 * BLOCK, 2 * BLOCK, 200, 2 * BLOCK + 37, BLOCK, 3 * BLOCK + 13, 2 * BLOCK, 50_000]
TABLE = [409_600, 409_600, 100_000]
TABLE_OFF_GRID = [409_626, 409_574, 100_000]   # the second block's leading angle comes from off its row grid


def _bits_equal(a, b):
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


def _quantized(fmt, start, n):
    from qdsp_b200 import synth

    _, sc, off = synth.IQ_FORMATS[fmt]
    q = synth.quantize_iq(synth.cfg2_input(start, n), fmt)
    return q, synth.iq_to_cf32(q, sc, off)


# ---- CPU ---------------------------------------------------------------------------------------------------------
def test_new_symbols_exported_and_declared(qlib):
    from qdsp_b200 import lib

    for s in NEW_SYMBOLS:
        assert s in lib.header_symbols() and s in lib.SIGNATURES and hasattr(qlib, s), s
    assert (lib.CS16, lib.CS8, lib.CU8) == (2, 3, 4)


def test_conversion_rule_extremes():
    from qdsp_b200 import synth

    cases = {
        "cs16": ([-32768, 32767, 0, -1], [-1.0, 32767 / 32768, 0.0, -1 / 32768]),
        "cs8": ([-128, 127, 0, -1], [-1.0, 127 / 128, 0.0, -1 / 128]),
        "cu8": ([0, 255, 127, 128], [-127.5 / 128, 127.5 / 128, -0.5 / 128, 0.5 / 128]),
    }
    for fmt, (xs, want) in cases.items():
        dt, sc, off = synth.IQ_FORMATS[fmt]
        y = synth.iq_to_cf32(np.asarray(xs, dt), sc, off)
        assert np.array_equal(y.view(np.float32), np.asarray(want, np.float32)), fmt
        # the rule, step by step in float32
        for x, v in zip(xs, y.view(np.float32)):
            assert v == np.float32(np.float32(np.float32(x) + np.float32(off)) * np.float32(sc))
        # quantising the converted values gives the integers back; out-of-range values saturate
        assert np.array_equal(synth.quantize_iq(y, fmt), np.asarray(xs, dt))
        info = np.iinfo(dt)
        big = np.asarray([10 + 10j, -10 - 10j], np.complex64)
        assert np.array_equal(synth.quantize_iq(big, fmt), np.asarray([info.max] * 2 + [info.min] * 2, dt))


def test_bad_formats_and_parameters_rejected(qlib):
    # every check below runs before any device work
    from qdsp_b200 import lib

    buf = (C.c_char * 64)()
    p = C.addressof(buf)
    for fmt, scale, off in [(1, 1.0, 0.0), (0, 1.0, 0.0), (5, 1.0, 0.0), (2, 0.0, 0.0), (2, math.inf, 0.0),
                            (3, math.nan, 0.0), (4, 1.0, math.inf), (4, 1.0, math.nan)]:
        assert qlib.qdsp_iq_convert_process(fmt, scale, off, p, p, 4, None) == -1, (fmt, scale, off)
    assert qlib.qdsp_iq_convert_process(2, 1.0, 0.0, p + 2, p, 4, None) == -1      # cs16 needs 4-byte pairs
    assert "aligned" in lib.last_error()
    taps = (C.c_float * 4)(1, 2, 3, 4)
    for fmt in (lib.CS16, lib.CS8, lib.CU8):
        assert not qlib.qdsp_fir_create(fmt, taps, 4)
        assert not qlib.qdsp_resamp_create(fmt, taps, 4, 1, 2)
        assert not qlib.qdsp_ffagc_create(fmt)
        assert qlib.qdsp_math_process(0, fmt, p, p, p, 4, None) == -1
        assert qlib.qdsp_volume_process(fmt, 1.0, 0, p, p, 4, None) == -1


def _build_example(out):
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-I" + os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "examples", "iq_chain.cpp"), "-L" + os.path.join(ROOT, "qdsp_b200"),
                           "-lqdsp_b200", "-lpthread", "-Wl,-rpath," + os.path.join(ROOT, "qdsp_b200"), "-o", str(out)])


def test_iq_example_compiles(qlib, tmp_path):
    _build_example(tmp_path / "iq_chain")
    assert os.path.exists(tmp_path / "iq_chain")


# ---- GPU: the converter ------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("fmt", FMTS)
def test_convert_bit_exact(fmt):
    from qdsp_b200 import blocks as B, lib, synth

    L = lib.load()
    dt, sc, off = synth.IQ_FORMATS[fmt]
    E = 2 * np.dtype(dt).itemsize
    info = np.iinfo(dt)
    rng = np.random.default_rng(7)
    for n in (1, 7, 1001, 1 << 16):
        raw = rng.integers(info.min, info.max + 1, 2 * n, dtype=np.int64).astype(dt)
        raw[:4] = [info.min, info.max, 0, info.max][:min(4, 2 * n)]
        for scale, offset in ((sc, off), (1 / 2048, 0.0), (0.37, 3.25)):
            want = synth.iq_to_cf32(raw, scale, offset)
            for in_off in (0, E, 3 * E, 16):           # pointers aligned only to the pair
                for out_off in (0, 8):
                    din, dout = B.DevBuf(raw.nbytes + 64), B.DevBuf(n * 8 + 64)
                    assert L.qdsp_copy_h2d(din.ptr + in_off, raw.ctypes.data, raw.nbytes, None) == 0
                    assert L.qdsp_iq_convert_process(synth.IQ_CODES[fmt], scale, offset, din.ptr + in_off,
                                                     dout.ptr + out_off, n, None) == n
                    got = dout.to_numpy(np.complex64, n, offset_bytes=out_off)
                    assert _bits_equal(got.view(np.float32), want.view(np.float32)), (n, scale, in_off, out_off)
    # the converter block
    raw = synth.quantize_iq(synth.cfg2_input(0, 5000), fmt)
    assert _bits_equal(B.IQConverter(fmt).process(raw).view(np.float32), synth.iq_to_cf32(raw, sc, off).view(np.float32))


# ---- GPU: the fused chain ----------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("fmt", FMTS)
def test_fused_benchmark_geometry(fmt):
    from qdsp_b200 import blocks as B, lib

    L = lib.load()
    q, xc = _quantized(fmt, 0, N1)
    ref = B.VFOFM(*CHAIN).process(xc, BLOCK)
    v = B.VFOFM(*CHAIN)
    v.set_input_format(fmt)
    din = B.DevBuf.from_numpy(q)
    m = v.out_count(N1, BLOCK)
    aud = B.DevBuf((m + 64) * 4)
    before = L.qdsp_launch_count()
    assert v.process_device(din.ptr, aud.ptr, N1, BLOCK) == m
    assert L.qdsp_launch_count() - before == 2                  # the conversion, then the row-per-lane kernel
    assert _bits_equal(aud.to_numpy(np.float32, m), ref)


def _process_raw(L, h, in_ptr, audio_ptr, n, block=BLOCK):
    if np.isscalar(block):
        b, nb, bs = None, 0, int(block)
    else:
        b = np.ascontiguousarray(block, np.int32)
        nb, bs = len(b), 0
    m = L.qdsp_vfofm_process(h, in_ptr, audio_ptr, None, n, None if b is None else b.ctypes.data_as(C.POINTER(C.c_int)),
                             nb, bs, None, None)
    assert m >= 0, m
    return m


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", FMTS)
def test_fused_ragged_table_unaligned_calls(fmt):
    """One handle: calls off the decimation grid, a call shorter than the history, a table partition and an input
    pointer that is not 16-byte aligned, against the cf32 path call by call and the oracle."""
    from qdsp_b200 import blocks as B, lib

    L = lib.load()
    calls = [(s, BLOCK, 0) for s in SIZES2] + [(sum(TABLE), TABLE, 0), (sum(TABLE_OFF_GRID), TABLE_OFF_GRID, 0),
                                               (BLOCK + 50, BLOCK, 4), (2 * BLOCK, BLOCK, 0)]
    total = sum(c[0] for c in calls)
    q, xc = _quantized(fmt, 0, total)
    v, r = B.VFOFM(*CHAIN), B.VFOFM(*CHAIN)
    v.set_input_format(fmt)
    got, want, sizes = [], [], []
    pos = 0
    for n, blk, misalign in calls:
        qi = np.ascontiguousarray(q[2 * pos:2 * (pos + n)])
        din = B.DevBuf(qi.nbytes + 64)
        assert L.qdsp_copy_h2d(din.ptr + misalign, qi.ctypes.data, qi.nbytes, None) == 0
        m = v.out_count(n, blk)
        aud = B.DevBuf((m + 64) * 4)
        assert _process_raw(L, v.h, din.ptr + misalign, aud.ptr, n, blk) == m
        got.append(aud.to_numpy(np.float32, m))
        want.append(r.process(xc[pos:pos + n], blk))
        assert _bits_equal(got[-1], want[-1]), (n, blk, misalign)
        sizes += [int(b) for b in loader.as_blocks(n, blk)]
        pos += n
    a64, _ = loader.port().vfo_fm(*CHAIN, xc, sizes, nco_f64=True)
    audio = np.concatenate(got)
    assert audio.shape == a64.shape
    assert np.abs(audio[16:] - a64[16:]).max() <= AUDIO_TOL


@pytest.fixture(scope="module")
def overlap_runs():
    # the back-to-back sequences of test_vfofm_overlapped_calls.py on integer input, overlapped and serialized
    from tests import overlapped

    return overlapped.runs()


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", FMTS)
def test_overlapped_calls_same_buffers(overlap_runs, fmt):
    from qdsp_b200 import blocks as B

    ours, serial = overlap_runs
    assert _bits_equal(ours[fmt + "_same_last"], serial[fmt + "_same_last"])
    _, xc = _quantized(fmt, 0, N1)
    r = B.VFOFM(*CHAIN)
    for _ in range(K1):
        y = r.process(xc, BLOCK)
    assert _bits_equal(ours[fmt + "_same_last"], y)


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", FMTS)
def test_overlapped_calls_distinct_buffers(overlap_runs, fmt):
    from qdsp_b200 import blocks as B

    ours, serial = overlap_runs
    assert _bits_equal(ours[fmt + "_distinct"], serial[fmt + "_distinct"])
    _, xc = _quantized(fmt, 0, sum(SIZES2))
    r = B.VFOFM(*CHAIN)
    offs = np.concatenate([[0], np.cumsum(SIZES2)])
    want = np.concatenate([r.process(xc[offs[i]:offs[i + 1]], BLOCK) for i in range(len(SIZES2))])
    assert _bits_equal(ours[fmt + "_distinct"], want)


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", FMTS)
def test_process_host_matches_device(fmt):
    # process_host stages ~8 M samples per chunk: 20 blocks of 819 200 cross two chunk seams
    from qdsp_b200 import blocks as B

    q, xc = _quantized(fmt, 0, N1)
    h = B.VFOFM(*CHAIN)
    h.set_input_format(fmt)
    d = B.VFOFM(*CHAIN)
    d.set_input_format(fmt)
    yh, yd = h.process_host(q, BLOCK), d.process(q, BLOCK)
    assert _bits_equal(yh, yd)
    # caller-owned buffers must already hold the handle's format
    with pytest.raises(TypeError):
        h.process_host_into(np.zeros(16, np.complex64), np.zeros(16, np.float32), BLOCK)
    assert _bits_equal(yd, B.VFOFM(*CHAIN).process(xc, BLOCK))


@pytest.mark.gpu
def test_formats_mixed_call_by_call():
    from qdsp_b200 import blocks as B, synth

    n = 3 * BLOCK
    x = synth.cfg2_input(0, 4 * n)
    q16 = synth.quantize_iq(x[n:2 * n], "cs16")
    qu8 = synth.quantize_iq(x[2 * n:3 * n], "cu8")
    stream = [x[:n], synth.iq_to_cf32(q16, 1 / 32768, 0.0), synth.iq_to_cf32(qu8, 1 / 128, -127.5), x[3 * n:]]
    v, r = B.VFOFM(*CHAIN), B.VFOFM(*CHAIN)
    got = [v.process(x[:n], BLOCK)]
    v.set_input_format("cs16")
    got.append(v.process(q16, BLOCK))
    v.set_input_format("cu8")
    got.append(v.process(qu8, BLOCK))
    v.set_input_format("cf32")
    got.append(v.process(x[3 * n:], BLOCK))
    for g, s in zip(got, stream):
        assert _bits_equal(g, r.process(s, BLOCK))
    # debug replay reads cf32 only
    v.set_input_format("cs8")
    with pytest.raises(Exception):
        v.process_replay(synth.quantize_iq(x[:1000], "cs8"), 1000, np.ones(2, np.complex64))


# ---- GPU: the channelizer ----------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("variant", [0, 2], ids=["fft", "direct"])
def test_channelizer_cs16(variant):
    from qdsp_b200 import blocks as B, synth

    n, blk = 1 << 18, 81920
    offs = synth.cfg4_offsets(256)
    q = synth.quantize_iq(synth.cfg4_input(0, n, nch=256), "cs16", scale=1 / 4096)
    xc = synth.iq_to_cf32(q, 1 / 4096, 0.0)
    a, b = B.Channelizer(offs, 61.44e6, 48e3, 48e3, 5e3), B.Channelizer(offs, 61.44e6, 48e3, 48e3, 5e3)
    a.set_variant(variant)
    b.set_variant(variant)
    a.set_input_format("cs16", scale=1 / 4096)
    ya, yb = a.process(q, blk), b.process(xc, blk)
    assert ya.shape == (256, n // 1280)
    assert _bits_equal(ya, yb)


# ---- GPU: the dsp:: example --------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("fmt", FMTS)
def test_iq_example_matches_oracle(qlib, tmp_path, fmt):
    exe = tmp_path / "iq_chain"
    _build_example(exe)
    n, blk = 4 * 81920 + 1000, 81920
    q, xc = _quantized(fmt, 0, n)
    fin = tmp_path / "in.raw"
    q.tofile(fin)
    sizes = [int(b) for b in loader.as_blocks(n, blk)]
    a64, _ = loader.port().vfo_fm(*CHAIN, xc, sizes, nco_f64=True)
    for mode in ([], ["convert"]):
        fout = tmp_path / "out.f32"
        subprocess.check_call([str(exe), fmt, str(fin), str(fout), str(blk)] + mode)
        y = np.fromfile(fout, np.float32)
        assert y.shape == a64.shape, mode
        assert np.abs(y[16:] - a64[16:]).max() <= AUDIO_TOL, mode
