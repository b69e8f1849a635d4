"""Integer IQ input (cs16, cs8, cu8) for the power spectrum (qdsp_spectrum_set_input_format, blocks.Spectrum,
dsp::SpectrumT<T>): the frames kernel reads the integer pairs itself.

CPU: the new symbol is declared, exported and typed; the integer-input example graph compiles.
GPU: rows bit-identical to a cf32 handle fed the host-converted samples (synth.iq_to_cf32, pinned to the GPU conversion
by test_iq_formats.py::test_convert_bit_exact) over the whole parity grid; one case per format against numpy's float64 FFT;
bit-identical rows under ragged calls that start at every alignment the format allows, and under a format change from call
to call; rejections; the dsp:: graph; one 2^28-sample call."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

from tests.test_spectrum import (FS4, GRID_N, MAX_LEN, NCH4, SPACING4, assert_rows_close, comb_device, frames_complete,
                                 hann, ragged_calls, ref_rows, rows_complete, slice_len)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FMTS = ["cs16", "cs8", "cu8"]
HOPS = {"N": lambda N: N, "N/2": lambda N: N // 2, "N/4+3": lambda N: N // 4 + 3, "3N": lambda N: 3 * N}


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _example(tmp_path):
    exe = tmp_path / "spectrum_iq_chain"
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-I" + os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "examples", "spectrum_iq_chain.cpp"), "-L" + os.path.join(ROOT, "qdsp_b200"),
                           "-lqdsp_b200", "-lpthread", "-Wl,-rpath," + os.path.join(ROOT, "qdsp_b200"), "-o", str(exe)])
    return exe


# ---- CPU --------------------------------------------------------------------------------------------------------
def test_spectrum_set_input_format_declared_exported_and_typed(qlib):
    from qdsp_b200 import lib

    n = "qdsp_spectrum_set_input_format"
    assert n in lib.header_symbols() and hasattr(qlib, n)
    assert lib.SIGNATURES[n] == lib.SIGNATURES["qdsp_vfofm_set_input_format"]
    assert lib.SIGNATURES[n][0] is C.c_int


def test_spectrum_iq_example_compiles(qlib, tmp_path):
    assert _example(tmp_path).exists()


# ---- GPU fixtures -----------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def quantized():
    """The comb and the config-2 stream of test_spectrum.py, quantised to each format: {(signal, fmt): (raw, cf32)},
    cf32 being the host conversion of raw with the format's usual scale and offset."""
    from qdsp_b200 import synth

    _, comb = comb_device(MAX_LEN)
    out = {}
    for name, x in {"cfg2": synth.cfg2_input(0, MAX_LEN), "comb": comb}.items():
        for fmt in FMTS:
            _, sc, off = synth.IQ_FORMATS[fmt]
            raw = synth.quantize_iq(x, fmt)
            out[(name, fmt)] = (raw, synth.iq_to_cf32(raw, sc, off))
    return out


def _int_handle(fmt, *args):
    from qdsp_b200 import blocks as B

    h = B.Spectrum(*args)
    h.set_input_format(fmt)
    return h


# ---- GPU: bit-identity to the cf32 path -------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("fmt", FMTS)
@pytest.mark.parametrize("N", GRID_N)
@pytest.mark.parametrize("hop_kind", list(HOPS))
def test_spectrum_iq_bit_identical_to_cf32(qlib, quantized, fmt, N, hop_kind):
    from qdsp_b200 import blocks as B

    hop = HOPS[hop_kind](N)
    w = hann(N)
    for A in (1, 7, 64):
        n = (2 * A + 1) * hop + N + 5          # two full rows and part of a third
        for name in ("cfg2", "comb"):
            raw, xc = quantized[(name, fmt)]
            raw, xc = raw[:2 * n], xc[:n]
            got = _int_handle(fmt, N, w, hop, A).process(raw)
            want = B.Spectrum(N, w, hop, A).process(xc)
            assert got.shape == want.shape and len(got) >= 2, (name, A)
            assert np.array_equal(_bits(got), _bits(want)), f"{name} {fmt} N={N} hop={hop} A={A}"


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", FMTS)
def test_spectrum_iq_matches_numpy(qlib, quantized, fmt):
    N, A = 4096, 7
    hop = N // 4 + 3
    n = (2 * A + 1) * hop + N + 5
    for name in ("cfg2", "comb"):
        raw, xc = quantized[(name, fmt)]
        got = _int_handle(fmt, N, hann(N), hop, A).process(raw[:2 * n])
        assert_rows_close(got, ref_rows(xc[:n], N, hop, A, hann(N)), f"{name} {fmt}")


# ---- GPU: split invariance --------------------------------------------------------------------------------------
def _ragged(n, N, hop, A, seed):
    """test_spectrum.ragged_calls with three more one-sample calls after its first one, so that calls start at four
    consecutive sample offsets (every offset mod 4)."""
    sizes = ragged_calls(n - 3, N, hop, A, seed)
    assert sizes[4] == 1
    return sizes[:5] + [1, 1, 1] + sizes[5:]


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", FMTS)
@pytest.mark.parametrize("N,hop,A", [
    (64, 19, 64),        # 32 frames side by side per CTA, one slice per row
    (256, 100, 300),     # two slices per row, 8 frames side by side
    (1024, 259, 7),
    (4096, 3 * 4096, 7),  # gaps between frames
    (16384, 8192, 7),    # two slices per row (4 + 3 frames), frames overlap
])
def test_spectrum_iq_partition_invariant(qlib, quantized, fmt, N, hop, A):
    from qdsp_b200 import blocks as B

    E = 4 if fmt == "cs16" else 2                        # bytes per pair
    n = (3 * A + 2) * hop + N + 17
    raw, xc = quantized[("cfg2", fmt)]
    raw, xc = raw[:2 * n], xc[:n]
    din = B.DevBuf.from_numpy(raw)
    rows_total = rows_complete(n, N, hop, A)
    whole = _int_handle(fmt, N, hann(N), hop, A)
    dout = B.DevBuf(rows_total * N * 4)
    assert whole.process_device(din.ptr, dout.ptr, n) == rows_total
    want = dout.to_numpy(np.float32, rows_total * N)
    # the one call equals the cf32 path
    assert np.array_equal(_bits(want), _bits(B.Spectrum(N, hann(N), hop, A).process(xc).reshape(-1)))

    sizes = _ragged(n, N, hop, A, seed=N + hop + A)
    S = slice_len(N, A)
    ends = np.cumsum(sizes)
    starts = ends - np.asarray(sizes)
    F = np.asarray([frames_complete(int(e), N, hop) for e in ends])
    tail_start = F * hop
    assert 0 in sizes and any(0 < s < hop for s in sizes) and any(0 < s < N for s in sizes)
    assert np.any((tail_start < ends) & (tail_start + N > ends)), "no call ends mid-frame"
    assert np.any((F % A) % S != 0), "no call ends mid-slice"
    assert np.any(F % A != 0), "no call ends mid-row"
    # every byte alignment the pair allows within 8 bytes: offsets 0..3 mod 4 (8-bit) or 0..1 mod 2 (cs16)
    assert set((starts * E) % 8) == set(range(0, 8, E)), "a pair alignment is missing"

    h = _int_handle(fmt, N, hann(N), hop, A)
    got = B.DevBuf(max(rows_total, 1) * N * 4)
    done = 0
    for s0, c in zip(starts, sizes):
        pred = h.out_rows(c)
        r = h.process_device(din.ptr + E * int(s0), got.ptr + 4 * N * done, c)
        assert r == pred == rows_complete(int(s0) + c, N, hop, A) - rows_complete(int(s0), N, hop, A)
        done += r
    assert done == rows_total
    assert np.array_equal(_bits(got.to_numpy(np.float32, rows_total * N)), _bits(want))

    # after reset the handle equals a fresh one, and keeps its format
    h.reset()
    assert h.process_device(din.ptr, got.ptr, n) == rows_total
    assert np.array_equal(_bits(got.to_numpy(np.float32, rows_total * N)), _bits(want))


@pytest.mark.gpu
@pytest.mark.parametrize("N,hop,A", [(1024, 700, 3), (64, 19, 64), (16384, 8192, 2)])
def test_spectrum_format_changes_call_to_call(qlib, N, hop, A):
    """cf32 -> cs16 -> cu8 -> cs8 -> cf32 on one handle, every call ending mid-frame: the rows of a cf32 handle fed the
    host-converted stream."""
    from qdsp_b200 import blocks as B, synth

    n = (4 * A + 1) * hop + N
    x = synth.cfg2_input(0, n)
    cuts = [0] + [int(n * k / 5) + 3 * k for k in range(1, 5)] + [n]
    h, ref = B.Spectrum(N, hann(N), hop, A), B.Spectrum(N, hann(N), hop, A)
    got, want = [], []
    for fmt, a, b in zip(["cf32", "cs16", "cu8", "cs8", "cf32"], cuts[:-1], cuts[1:]):
        if b < n:
            F = frames_complete(b, N, hop)
            assert F * hop < b < F * hop + N, f"the {fmt} call does not end mid-frame"
        h.set_input_format(fmt)
        if fmt == "cf32":
            seg = xc = x[a:b]
        else:
            _, sc, off = synth.IQ_FORMATS[fmt]
            seg = synth.quantize_iq(x[a:b], fmt)
            xc = synth.iq_to_cf32(seg, sc, off)
        got.append(h.process(seg))
        want.append(ref.process(xc))
    got, want = np.concatenate(got), np.concatenate(want)
    assert len(got) == rows_complete(n, N, hop, A) > 0
    assert np.array_equal(_bits(got), _bits(want))


# ---- GPU: rejections --------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_spectrum_iq_rejections(qlib, quantized):
    from qdsp_b200 import blocks as B

    N, hop, A = 1024, 512, 2
    n = (2 * A + 1) * hop + N
    v = B.VFOFM(250e3, 2.4e6, 48e3, 48e3, 5e3)
    for fmt in FMTS:
        raw, xc = quantized[("cfg2", fmt)]
        raw, xc = raw[:2 * n], xc[:n]
        want = B.Spectrum(N, None, hop, A).process(xc)
        E = raw.itemsize * 2
        h = _int_handle(fmt, N, None, hop, A)
        # bad format codes and conversions: rejected as the fused chain rejects them, the format unchanged
        for code, sc, off in [(0, 1.0, 0.0), (5, 1.0, 0.0), (-1, 1.0, 0.0), (2, 0.0, 0.0), (2, math.inf, 0.0),
                              (3, math.nan, 0.0), (4, 1.0, math.inf), (4, 1.0, math.nan), (4, -math.inf, 0.0)]:
            assert qlib.qdsp_vfofm_set_input_format(v.h, code, sc, off) == -1
            assert qlib.qdsp_spectrum_set_input_format(h.h, code, sc, off) == -1, (code, sc, off)
        assert np.array_equal(_bits(h.process(raw)), _bits(want)), fmt
        # a pointer not aligned to the pair: -1 and nothing consumed
        h.reset()
        din = B.DevBuf(raw.nbytes + 64)
        assert qlib.qdsp_copy_h2d(din.ptr + 8, raw.ctypes.data, raw.nbytes, None) == 0
        out = B.DevBuf(8 * N * 4)
        bad = [din.ptr + 8 + 2] if fmt == "cs16" else [din.ptr + 8 + 1, din.ptr + 8 + 3]
        for p in bad:
            assert qlib.qdsp_spectrum_process(h.h, p, out.ptr, n, None) == -1
        assert h.process_device(din.ptr + 8, out.ptr, n) == len(want)
        assert np.array_equal(_bits(out.to_numpy(np.float32, len(want) * N).reshape(-1, N)), _bits(want))
        # a pointer aligned to the pair but not to 8 bytes is valid integer input
        h.reset()
        assert qlib.qdsp_copy_h2d(din.ptr + E, raw.ctypes.data, raw.nbytes, None) == 0
        assert h.process_device(din.ptr + E, out.ptr, n) == len(want)
        assert np.array_equal(_bits(out.to_numpy(np.float32, len(want) * N).reshape(-1, N)), _bits(want))
    # back to cf32: the 8-byte rule again
    h = B.Spectrum(N, None, hop, A)
    h.set_input_format("cs8")
    h.set_input_format("cf32")
    x = B.DevBuf(n * 8 + 16)
    assert qlib.qdsp_spectrum_process(h.h, x.ptr + 4, x.ptr, n, None) == -1


# ---- GPU: the dsp:: graph ---------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["cu8", "cs16"])
@pytest.mark.parametrize("N,hop,A,block", [(1024, 512, 8, 300_000), (16384, 16384, 1, 1_000_000)])
def test_spectrum_iq_cpp_graph_matches_numpy(qlib, tmp_path, fmt, N, hop, A, block):
    from qdsp_b200 import synth

    exe = _example(tmp_path)
    _, sc, off = synth.IQ_FORMATS[fmt]
    raw = synth.quantize_iq(synth.cfg2_input(0, 2_500_000), fmt)
    fin, fout = tmp_path / "in.raw", tmp_path / "out.f32"
    raw.tofile(fin)
    subprocess.check_call([str(exe), fmt, str(fin), str(fout), str(N), str(hop), str(A), str(block)], timeout=120)
    got = np.fromfile(fout, np.float32)
    assert got.size % N == 0 and got.size > 0
    assert_rows_close(got.reshape(-1, N), ref_rows(synth.iq_to_cf32(raw, sc, off), N, hop, A, hann(N)),
                      f"dsp::SpectrumT<{fmt}> graph")


# ---- GPU: one full-size call ------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_spectrum_iq_full_size_call(qlib):
    from qdsp_b200 import blocks as B, lib, synth

    n, N, A = 1 << 28, 4096, 64
    _, sc, off = synth.IQ_FORMATS["cu8"]
    d = B.DevBuf(n * 8)
    lib.check(lib.load().qdsp_synth_comb_cf32(d.ptr, 0, n, FS4, NCH4, SPACING4, 5e3, 1.0 / 64.0, 0.001, 4, None))
    raw = np.empty(2 * n, np.uint8)
    chunk = 1 << 24
    for c0 in range(0, n, chunk):
        raw[2 * c0:2 * (c0 + chunk)] = synth.quantize_iq(d.to_numpy(np.complex64, chunk, offset_bytes=8 * c0), "cu8")
    dq = B.DevBuf.from_numpy(raw)
    h = _int_handle("cu8", N, hann(N), N, A)
    R = h.out_rows(n)
    assert R == n // (N * A)
    out = B.DevBuf(R * N * 4)
    assert h.process_device(dq.ptr, out.ptr, n) == R
    rows = out.to_numpy(np.float32, R * N).reshape(R, N)
    for r in np.linspace(0, R - 1, 64).astype(int):
        x = synth.iq_to_cf32(raw[2 * int(r) * A * N:2 * (int(r) + 1) * A * N], sc, off)
        assert_rows_close(rows[r:r + 1], ref_rows(x, N, N, A, hann(N)), f"row {r}")
    # and every row equals the cf32 path on the GPU-converted stream
    assert lib.load().qdsp_iq_convert_process(synth.IQ_CODES["cu8"], sc, off, dq.ptr, d.ptr, n, None) == n
    ref = B.Spectrum(N, hann(N), N, A)
    out2 = B.DevBuf(R * N * 4)
    assert ref.process_device(d.ptr, out2.ptr, n) == R
    assert np.array_equal(_bits(out2.to_numpy(np.float32, R * N)), _bits(rows.reshape(-1)))
