"""Retuning a live channelizer (qdsp_channelizer_set_offsets, Channelizer.set_offsets) and the FFT form's bookkeeping
(qdsp_channelizer_fft_form). A retune keeps every channel's NCO phase continuous at the current stream position and
carries the history (untranslated), the demodulator phases and the position on; the FFT polyphase form stays while the
offsets form the comb. The oracle below is the f64-rotator VFO chain of oracle/windows.py with the translator's frequency
changing at the retune sample P, phase continuous there; because the history is kept untranslated, the outputs computed
after the retune see the samples before P at the new frequency as well, and the oracle models exactly that."""
import math
import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest

from oracle import loader

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FS4, BLK4, D4 = 61.44e6, 81920, 1280
CUTS = [0, 2 * BLK4, 4 * BLK4, 6 * BLK4]        # three calls; retunes before calls 2 and 3
N4 = CUTS[-1]
AUDIO_TOL, IQ_TOL = 1e-4, 1e-5
NEW_SYMBOLS = ["qdsp_channelizer_set_offsets", "qdsp_channelizer_fft_form", "qdsp_scatter_rows"]
GOLDEN_VFOFM = os.path.join(ROOT, "tests", "golden", "vfofm_set_offset.npz")
CHAIN = (250e3, 2.4e6, 48e3, 48e3, 5e3)


def _bits_equal(a, b):
    return a.shape == b.shape and np.array_equal(np.ascontiguousarray(a).view(np.uint32), np.ascontiguousarray(b).view(np.uint32))


def _rel(a, b):
    return float(np.linalg.norm(a - b) / np.linalg.norm(b))


def _input(shift=0):
    """config 4's comb (carriers on the half-bin grid), or moved by `shift` Hz (120 kHz: the bin grid)."""
    from qdsp_b200 import synth

    x = synth.cfg4_input(0, N4, nch=256)
    offs = synth.cfg4_offsets(256)
    if shift:
        sh = np.exp(2j * np.pi * synth._frac(np.arange(N4, dtype=np.int64), shift, 61_440_000))
        x = (x.astype(np.complex128) * sh).astype(np.complex64)
        offs = (offs + np.float32(shift)).astype(np.float32)
    return x, offs


def _moved(offs, hz):
    return (offs.astype(np.float64) + hz).astype(np.float32)


def _off_grid(offs):
    o = offs.copy()
    o[77] = np.float32(float(o[77]) + 9e3)
    return o


# name -> (input comb shift, offsets of calls 1, 2, 3 from the input's offsets, fft_form before each call at variant 0)
SCENARIOS = {
    "off_grid_and_back": (0, lambda o: [o, _off_grid(o), o], [1, 0, 1]),
    "half_bin_then_rotated": (0, lambda o: [o, _moved(o, 720e3), _moved(o, 713e3)], [1, 1, 1]),
    "bin_then_rotated": (120_000, lambda o: [o, _moved(o, -720e3), _moved(o, -715e3)], [1, 1, 1]),
}


def _chan(offs, variant=0, in_sr=FS4, out_sr=48e3, bw=48e3):
    from qdsp_b200 import blocks as B

    ch = B.Channelizer(offs, in_sr, out_sr, bw, 5e3)
    ch.set_variant(variant)
    return ch


def _run(ch, x, offs_calls, cuts=CUTS, block=BLK4, audio=True, forms=None):
    """One call per [cuts[j], cuts[j+1]) with the offsets of call j set before it; returns (iq, audio) [nch, n_out]."""
    iqs, auds = [], []
    for j, (lo, hi) in enumerate(zip(cuts[:-1], cuts[1:])):
        if j > 0:
            ch.set_offsets(offs_calls[j])
        if forms is not None:
            forms.append(int(ch.fft_form))
        r = ch.process_iq(x[lo:hi], block, audio=audio)
        if audio:
            iqs.append(r[0])
            auds.append(r[1])
        else:
            iqs.append(r)
    iq = np.concatenate(iqs, axis=1)
    return (iq, np.concatenate(auds, axis=1)) if audio else iq


def _oracle(x, offs_calls, c, cuts=CUTS, in_sr=FS4, out_sr=48e3, bw=48e3, dev=5e3):
    """Channel c of the retuned chain: call j's outputs are the VFO over the raw stream mixed at call j's frequency,
    with the phase continuous at every retune sample; float64 rotator, the reference's resampler and FM demodulator."""
    P = loader.port()
    taps, I, D = P.vfo_design(in_sr, out_sr, bw)
    lead = (len(taps) // D + 3) * D
    iqs = []
    const, prev_th = 0.0, None
    for j, (lo, hi) in enumerate(zip(cuts[:-1], cuts[1:])):
        inc = P.xlator_phase_delta(in_sr, -float(offs_calls[j][c]))
        th = math.atan2(inc.imag, inc.real)              # in float64, of the float32 phaseDelta (as the NCO)
        if prev_th is not None:
            const += (prev_th - th) * lo                 # phase continuous at sample lo
        prev_th = th
        w0 = max(0, lo - lead)
        n = np.arange(w0, hi, dtype=np.float64)
        ang = np.mod(const + th * n, 2 * np.pi)
        mixed = (x[w0:hi].astype(np.complex128) * np.exp(1j * ang)).astype(np.complex64)
        y, _ = P.resamp_cf32(taps, I, D, mixed, hi - w0)
        iqs.append(y[(lo - w0) // D:(hi - w0) // D])
    iq = np.concatenate(iqs)
    return P.fm_demod(out_sr, dev, iq), iq


# ---- CPU ---------------------------------------------------------------------------------------------------------
def test_new_symbols_declared_exported_and_bound(qlib):
    from qdsp_b200 import lib

    for s in NEW_SYMBOLS:
        assert s in lib.header_symbols() and s in lib.SIGNATURES and hasattr(qlib, s), s


# ---- GPU: against the oracle -------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("variant", [0, 2], ids=["auto", "direct"])
@pytest.mark.parametrize("name", list(SCENARIOS))
def test_retune_matches_oracle(name, variant):
    shift, make, want_forms = SCENARIOS[name]
    x, offs = _input(shift)
    offs_calls = make(offs)
    forms = []
    iq, audio = _run(_chan(offs, variant), x, offs_calls, forms=forms)
    assert forms == (want_forms if variant == 0 else [0, 0, 0]), forms
    assert iq.shape == audio.shape == (256, N4 // D4)
    worst_a, worst_q = 0.0, 0.0
    for c in range(256):
        a64, q64 = _oracle(x, offs_calls, c)
        assert q64.shape == iq[c].shape
        worst_a = max(worst_a, float(np.abs(audio[c, 16:] - a64[16:]).max()))
        worst_q = max(worst_q, _rel(iq[c, 16:], q64[16:]))
    assert worst_a <= AUDIO_TOL and worst_q <= IQ_TOL, (name, variant, worst_a, worst_q)


# ---- GPU: bit-exact invariants -----------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("variant", [0, 2], ids=["fft", "direct"])
def test_unchanged_offsets_are_a_bit_exact_no_op(variant):
    x, offs = _input()
    a = _run(_chan(offs, variant), x, [offs, offs, offs])
    ch = _chan(offs, variant)
    b = [ch.process_iq(x[lo:hi], BLK4) for lo, hi in zip(CUTS[:-1], CUTS[1:])]
    assert _bits_equal(a[0].view(np.float32), np.concatenate([r[0] for r in b], axis=1).view(np.float32))
    assert _bits_equal(a[1], np.concatenate([r[1] for r in b], axis=1))


@pytest.mark.gpu
def test_direct_form_retune_leaves_other_channels_bit_identical():
    x, offs = _input()
    moved = offs.copy()
    moved[5] = np.float32(float(moved[5]) + 3.3e3)
    iq_a, au_a = _run(_chan(offs, 2), x, [offs, moved, moved])
    iq_b, au_b = _run(_chan(offs, 2), x, [offs, offs, offs])
    keep = np.arange(256) != 5
    assert _bits_equal(iq_a[keep].view(np.float32), iq_b[keep].view(np.float32)) and _bits_equal(au_a[keep], au_b[keep])
    assert not np.array_equal(iq_a[5], iq_b[5])


def vfofm_retune_sequence():
    """The one-channel handle's retune sequence whose audio tests/golden/vfofm_set_offset.npz holds from the commit before
    qdsp_vfofm_set_offset went through the channelizer's set_offsets (row-per-lane kernel; then the generic kernel)."""
    from qdsp_b200 import blocks as B, synth

    x = synth.cfg2_input(0, 6 * 81920)
    out = {}
    for variant in (0, 1):
        v = B.VFOFM(*CHAIN)
        v.set_variant(variant)
        parts = [v.process(x[:2 * 81920], 81920)]
        v.setOffset(262.5e3)
        parts.append(v.process(x[2 * 81920:4 * 81920 + 700], 81920))
        v.setOffset(-13e3)
        v.setOffset(250e3)
        parts.append(v.process(x[4 * 81920 + 700:], 81920))
        out[f"variant{variant}"] = np.concatenate(parts)
    return out


@pytest.mark.gpu
def test_vfofm_set_offset_audio_unchanged():
    with np.load(GOLDEN_VFOFM) as g:
        want = dict(g)
    got = vfofm_retune_sequence()
    assert sorted(got) == sorted(want)
    for k in got:
        assert _bits_equal(got[k], want[k]), k


# ---- GPU: composition with the rest of the handle's state --------------------------------------------------------
@pytest.mark.gpu
def test_retune_then_seek_keeps_the_closed_form_phase():
    # a shard that retunes and then seeks: its NCOs stay continuous at the retune sample P in the closed form, so from S on
    # its IQ is a fresh handle's (tuned to the new offsets, seeked to S) times e^{j (theta_old - theta_new) P}
    P_ = loader.port()
    x, offs = _input()
    new = _moved(offs, 720e3)
    P0, S, lead = 2 * BLK4, 4 * BLK4, 16 * D4
    a = _chan(offs)
    a.process_iq(x[:P0], BLK4)
    a.set_offsets(new)
    a.seek(S)
    iq_a, au_a = a.process_iq(x[S:], BLK4)
    b = _chan(new)
    b.seek(S - lead)
    iq_b, au_b = b.process_iq(x[S - lead:], BLK4)
    iq_b, au_b = iq_b[:, lead // D4:], au_b[:, lead // D4:]
    assert iq_a.shape == iq_b.shape
    for c in range(256):
        th = [math.atan2(i.imag, i.real) for i in
              (P_.xlator_phase_delta(FS4, -float(offs[c])), P_.xlator_phase_delta(FS4, -float(new[c])))]
        rot = np.exp(1j * np.mod((th[0] - th[1]) * P0, 2 * np.pi))
        y = (iq_b[c] * rot).astype(np.complex64)
        assert _rel(iq_a[c, 16:], y[16:]) <= IQ_TOL, c
        # fast_arctan2 is not invariant under a constant rotation: the audio is checked against the reference demodulator
        # on the rotated samples
        assert np.abs(au_a[c, 16:] - P_.fm_demod(48e3, 5e3, y[15:])[1:]).max() <= AUDIO_TOL, c


@pytest.mark.gpu
@pytest.mark.parametrize("variant", [0, 2], ids=["fft", "direct"])
def test_retune_with_cs16_input_is_bit_identical_to_cf32(variant):
    from qdsp_b200 import synth

    x, offs = _input()
    q = synth.quantize_iq(x, "cs16", scale=1 / 4096)
    xc = synth.iq_to_cf32(q, 1 / 4096, 0.0)
    calls = [offs, _moved(offs, 720e3), _off_grid(_moved(offs, 720e3))]
    a, b = _chan(offs, variant), _chan(offs, variant)
    a.set_input_format("cs16", scale=1 / 4096)
    qa = q.reshape(-1, 2)
    iqs_a, aus_a = [], []
    for j, (lo, hi) in enumerate(zip(CUTS[:-1], CUTS[1:])):
        if j:
            a.set_offsets(calls[j])
        r = a.process_iq(qa[lo:hi].reshape(-1), BLK4)
        iqs_a.append(r[0])
        aus_a.append(r[1])
    iq_b, au_b = _run(b, xc, calls)
    assert _bits_equal(np.concatenate(iqs_a, axis=1).view(np.float32), iq_b.view(np.float32))
    assert _bits_equal(np.concatenate(aus_a, axis=1), au_b)


@pytest.mark.gpu
@pytest.mark.parametrize("variant", [0, 2], ids=["fft", "direct"])
def test_iq_only_calls_across_a_retune(variant):
    x, offs = _input()
    calls = [offs, _off_grid(offs), _moved(offs, 713e3)]
    iq_a = _run(_chan(offs, variant), x, calls, audio=False)
    iq_b, _ = _run(_chan(offs, variant), x, calls)
    assert _bits_equal(iq_a.view(np.float32), iq_b.view(np.float32))


def _rowlane_retune_sequence():
    """The fused chain's row-per-lane kernel, back-to-back calls on device buffers with a retune between calls 2 and 3
    (and between 3 and 4): the call after a retune never overlaps the one before it."""
    from qdsp_b200 import blocks as B, lib, synth
    from tests.overlapped import _process
    from tests.test_iq_formats import BLOCK

    L = lib.load()
    n = 4 * BLOCK
    x = synth.cfg2_input(0, 5 * n)
    ins = [B.DevBuf.from_numpy(x[i * n:(i + 1) * n]) for i in range(5)]
    v = B.VFOFM(*CHAIN)
    m = v.out_count(n, BLOCK)
    auds = [B.DevBuf((m + 64) * 4) for _ in range(5)]
    for i in range(5):
        if i in (2, 3):
            v.setOffset(250e3 + 1.7e3 * i)
        assert _process(L, v.h, ins[i].ptr, auds[i].ptr, n) == m
    return np.concatenate([a.to_numpy(np.float32, m) for a in auds])


def _dump_rowlane(path):
    np.save(path, _rowlane_retune_sequence())


@pytest.mark.gpu
def test_rowlane_retune_between_back_to_back_calls_matches_serialized():
    here = _rowlane_retune_sequence()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "serial.npy")
        env = dict(os.environ, QDSP_PDL="0", PYTHONPATH=ROOT)
        code = f"from tests.test_channelizer_retune import _dump_rowlane; _dump_rowlane({path!r}); print('ok')"
        r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
        assert r.returncode == 0 and "ok" in r.stdout, r.stdout + r.stderr
        serial = np.load(path)
    assert _bits_equal(here, serial)


# ---- GPU: rejections ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_set_offsets_rejects_bad_arguments_and_leaves_the_handle_unchanged():
    import ctypes as C

    from qdsp_b200 import lib

    L = lib.load()
    x, offs = _input()
    a, b = _chan(offs), _chan(offs)
    ya = a.process_iq(x[:CUTS[1]], BLK4)
    yb = b.process_iq(x[:CUTS[1]], BLK4)
    assert L.qdsp_channelizer_set_offsets(None, offs.ctypes.data_as(C.POINTER(C.c_float))) == -1
    assert L.qdsp_channelizer_set_offsets(a.h, None) == -1 and "NULL" in lib.last_error()
    for bad in (np.nan, np.inf, -np.inf):
        o = _off_grid(offs)
        o[200] = bad
        assert L.qdsp_channelizer_set_offsets(a.h, o.ctypes.data_as(C.POINTER(C.c_float))) == -1
        assert "finite" in lib.last_error()
        with pytest.raises(lib.QdspError):
            a.set_offsets(o)
    with pytest.raises(ValueError):
        a.set_offsets(offs[:-1])
    assert a.fft_form
    za = a.process_iq(x[CUTS[1]:], BLK4)
    zb = b.process_iq(x[CUTS[1]:], BLK4)
    assert _bits_equal(ya[1], yb[1]) and _bits_equal(za[0].view(np.float32), zb[0].view(np.float32)) and _bits_equal(za[1], zb[1])
