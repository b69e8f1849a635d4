"""The channelizer's complex baseband (qdsp_channelizer_process_iq, Channelizer.process_iq): every channel's VFO output
(resampling.h:99-132 after the translator, before FloatFMDemod) from the FFT polyphase form and from every direct-form
kernel. Bars: rel-L2 <= 1e-5 per channel against the oracle with the drift-free (float64) rotator, from output 16 on (the
first outputs come from an all-zero history); the audio of an IQ call is bit-identical to a process() call's."""
import numpy as np
import pytest

from oracle import loader

IQ_TOL = 1e-5
FS4, BLK4 = 61.44e6, 81920
N4 = 1 << 18
PICKS = (0, 1, 100, 128, 255)
CUTS = [0, BLK4, 2 * BLK4 + 1280 * 3 + 700, N4]   # the third call starts off the decimation grid


def _rel(a, b):
    return float(np.linalg.norm(a - b) / np.linalg.norm(b))


def _worst_rel(y, yr, start=16):
    return max(_rel(y[c, start:], yr[c, start:]) for c in range(y.shape[0]))


def _bits_equal(a, b):
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


def _comb(shift=0):
    """config 4's comb moved by `shift` Hz: 0 = the half-bin grid, 120 kHz = the bin grid, 50 kHz = neither (pre-rotated)."""
    from qdsp_b200 import synth

    x = synth.cfg4_input(0, N4, nch=256)
    offs = synth.cfg4_offsets(256)
    if shift:
        sh = np.exp(2j * np.pi * synth._frac(np.arange(N4, dtype=np.int64), shift, 61_440_000))
        x = (x.astype(np.complex128) * sh).astype(np.complex64)
        offs = (offs + np.float32(shift)).astype(np.float32)
    return x, offs


def _chan(offs, variant=0, in_sr=FS4, out_sr=48e3, bw=48e3):
    from qdsp_b200 import blocks as B

    ch = B.Channelizer(offs, in_sr, out_sr, bw, 5e3)
    ch.set_variant(variant)
    return ch


# ---- CPU ---------------------------------------------------------------------------------------------------------
def test_process_iq_symbol_declared_exported_and_bound(qlib):
    from qdsp_b200 import lib

    s = "qdsp_channelizer_process_iq"
    assert s in lib.header_symbols() and s in lib.SIGNATURES and hasattr(qlib, s)


# ---- GPU: FFT polyphase form -------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("shift", [0, 120_000, 50_000], ids=["half_bin", "bin", "rotated"])
def test_fft_form_iq_matches_oracle(shift):
    # the absolute channel phase (row phase in 64-bit turns, pad, half-bin twist and tap signs, pre-rotation, dt0), which
    # the FM audio cannot see, on all three comb placements
    P = loader.port()
    x, offs = _comb(shift)
    iq, audio = _chan(offs).process_iq(x, BLK4)
    assert iq.shape == audio.shape == (256, N4 // 1280) and iq.dtype == np.complex64
    for c in PICKS:
        _, _, iq64 = P.vfo_fm(float(offs[c]), FS4, 48e3, 48e3, 5e3, x, BLK4, nco_f64=True, want_iq=True)
        assert iq[c].shape == iq64.shape
        assert _rel(iq[c][16:], iq64[16:]) <= IQ_TOL, (shift, c, _rel(iq[c][16:], iq64[16:]))


@pytest.mark.gpu
def test_fft_form_iq_matches_direct_form_on_every_channel():
    x, offs = _comb()
    iq = _chan(offs).process_iq(x, BLK4, audio=False)
    iqd = _chan(offs, 2).process_iq(x, BLK4, audio=False)
    assert iq.shape == iqd.shape == (256, N4 // 1280)
    assert _worst_rel(iq, iqd) <= IQ_TOL, _worst_rel(iq, iqd)


@pytest.mark.gpu
@pytest.mark.parametrize("variant", [0, 2, 1], ids=["fft", "direct", "generic"])
def test_audio_of_iq_calls_is_bit_identical(variant):
    from qdsp_b200 import synth

    n = 1 << 17
    x = synth.cfg4_input(0, n, nch=256)
    offs = synth.cfg4_offsets(256)
    a, b = _chan(offs, variant), _chan(offs, variant)
    cuts = [0, BLK4, n]
    ya = np.concatenate([a.process(x[lo:hi], BLK4) for lo, hi in zip(cuts[:-1], cuts[1:])], axis=1)
    yb = np.concatenate([b.process_iq(x[lo:hi], BLK4)[1] for lo, hi in zip(cuts[:-1], cuts[1:])], axis=1)
    assert ya.shape == (256, n // 1280)
    assert _bits_equal(ya, yb)


@pytest.mark.gpu
def test_fft_form_streamed_iq_matches_direct_form():
    x, offs = _comb()
    s, d = _chan(offs), _chan(offs, 2)
    parts = [s.process_iq(x[lo:hi], BLK4, audio=False) for lo, hi in zip(CUTS[:-1], CUTS[1:])]
    partsd = [d.process_iq(x[lo:hi], BLK4, audio=False) for lo, hi in zip(CUTS[:-1], CUTS[1:])]
    y, yd = np.concatenate(parts, axis=1), np.concatenate(partsd, axis=1)
    assert y.shape == yd.shape == (256, N4 // 1280)
    assert _worst_rel(y, yd) <= IQ_TOL, _worst_rel(y, yd)


@pytest.mark.gpu
@pytest.mark.parametrize("variant", [0, 2], ids=["fft", "direct"])
def test_iq_only_calls_advance_the_demodulator_state(variant):
    # IQ-only calls (no audio buffer) between audio calls: the audio after them, and their IQ, equal a run that stored
    # audio throughout, bit for bit
    x, offs = _comb()
    a, b = _chan(offs, variant), _chan(offs, variant)
    cuts = [0, BLK4, BLK4 + 1280 * 7, 2 * BLK4 + 1280 * 3 + 700, N4]
    for i, (lo, hi) in enumerate(zip(cuts[:-1], cuts[1:])):
        iqa, ya = a.process_iq(x[lo:hi], BLK4)
        if i in (1, 2):
            iqb = b.process_iq(x[lo:hi], BLK4, audio=False)
            assert _bits_equal(iqa.view(np.float32), iqb.view(np.float32)), i
        else:
            assert _bits_equal(ya, b.process(x[lo:hi], BLK4)), i


# ---- GPU: direct-form kernels with more than one channel (and the one-channel row-per-lane kernel) ---------------
DIRECT = {
    # non-comb offsets at D = 1280: channel-per-lane kernel (k_chan.cu) + slice reduction
    "k_chan": dict(offs=[-30.6e6, 120e3, 17.88e6], in_sr=FS4, out_sr=48e3, bw=48e3, n=1 << 18, blk=BLK4),
    # 2.4 MS/s -> 48 kS/s, 4 channels: the decimating FIR (k_decim.cu)
    "k_decim": dict(offs=[-600e3, -250e3, 250e3, 700e3], in_sr=2.4e6, out_sr=48e3, bw=48e3, n=204800, blk=81920),
    # 250 kS/s -> 48 kS/s (I = 24, D = 125): the generic kernel (k_generic.cu)
    "generic": dict(offs=[-60e3, 10e3, 75e3], in_sr=250e3, out_sr=48e3, bw=24e3, n=100_000, blk=25_000),
    # one channel, 2.4 MS/s -> 48 kS/s: the row-per-lane kernel (k_rowlane.cu)
    "rowlane": dict(offs=[250e3], in_sr=2.4e6, out_sr=48e3, bw=48e3, n=204800, blk=81920),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(DIRECT))
def test_direct_form_iq_matches_oracle(name):
    from qdsp_b200 import synth

    c = DIRECT[name]
    P = loader.port()
    x = synth.cfg2_input(0, c["n"]) + synth.uniform_cf32(9, 0, c["n"]) * np.float32(0.1)
    ch = _chan(np.asarray(c["offs"], np.float32), 0, c["in_sr"], c["out_sr"], c["bw"])
    iq, audio = ch.process_iq(x, c["blk"])
    y = _chan(np.asarray(c["offs"], np.float32), 0, c["in_sr"], c["out_sr"], c["bw"]).process(x, c["blk"])
    assert _bits_equal(audio, y)
    for k, off in enumerate(c["offs"]):
        _, _, iq64 = P.vfo_fm(float(np.float32(off)), c["in_sr"], c["out_sr"], c["bw"], 5e3, x, c["blk"], nco_f64=True,
                              want_iq=True)
        assert iq[k].shape == iq64.shape
        assert _rel(iq[k][16:], iq64[16:]) <= IQ_TOL, (name, k, _rel(iq[k][16:], iq64[16:]))


# ---- GPU: integer input, seek, rejections ------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("variant", [0, 2], ids=["fft", "direct"])
def test_cs16_input_iq_is_bit_identical_to_cf32(variant):
    from qdsp_b200 import synth

    x, offs = _comb()
    q = synth.quantize_iq(x, "cs16", scale=1 / 4096)
    xc = synth.iq_to_cf32(q, 1 / 4096, 0.0)
    a, b = _chan(offs, variant), _chan(offs, variant)
    a.set_input_format("cs16", scale=1 / 4096)
    iqa, ya = a.process_iq(q, BLK4)
    iqb, yb = b.process_iq(xc, BLK4)
    assert iqa.shape == (256, N4 // 1280)
    assert _bits_equal(iqa.view(np.float32), iqb.view(np.float32)) and _bits_equal(ya, yb)


@pytest.mark.gpu
def test_seek_shard_with_lead_in_matches_unsharded_run():
    # as bench.py's cfg4 shards the stream: seek to the shard's start minus 16 rows, drop the outputs of the lead-in
    D = 1280
    x, offs = _comb()
    full = _chan(offs).process_iq(x, BLK4, audio=False)
    lo, lead = 64 * D, 16 * D
    sh = _chan(offs)
    sh.seek(lo - lead)
    part = sh.process_iq(x[lo - lead:], BLK4, audio=False)
    got, want = part[:, lead // D:], full[:, lo // D:]
    assert got.shape == want.shape
    assert _worst_rel(got, want, 0) <= IQ_TOL, _worst_rel(got, want, 0)


@pytest.mark.gpu
def test_process_iq_rejects_bad_arguments():
    from qdsp_b200 import blocks as B, lib

    L = lib.load()
    x, offs = _comb()
    ch = _chan(offs)
    n = 4 * BLK4
    din, diq, dout = B.DevBuf.from_numpy(x[:n]), B.DevBuf(256 * (n // 1280 + 16) * 8 + 8), B.DevBuf(256 * (n // 1280 + 16) * 4)
    stride = n // 1280 + 16
    call = lambda iq, cnt: L.qdsp_channelizer_process_iq(ch.h, din.ptr, iq, dout.ptr, stride, cnt, None, 0, BLK4, None)
    assert call(None, n) == -1 and "iq_out_dev" in lib.last_error()
    assert call(diq.ptr + 4, n) == -1 and "aligned" in lib.last_error()
    assert call(diq.ptr, -1) == -1
    assert call(diq.ptr, n) == n // 1280
    with pytest.raises(lib.QdspError):
        ch.process_device_iq(din.ptr, None, dout.ptr, n, stride, BLK4)
