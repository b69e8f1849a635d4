"""Back-to-back calls of the fused VFO -> FM chain on one handle: consecutive grids may overlap on the GPU (programmatic
dependent launch, k_rowlane.cu). Every sequence here runs twice -- in this process (overlap allowed) and in a subprocess
with QDSP_PDL=0 (every launch serialized) -- and the audio must be bit-identical; the streams are also checked against
the oracle (oracle/port.c, float64 NCO) across the call seams."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import loader, windows

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BLOCK = 819_200
CHAIN = (250e3, 2.4e6, 48e3, 48e3, 5e3)
AUDIO_TOL = 1e-4
N1, K1 = 20 * BLOCK, 8                     # the benchmark's pattern: > one wave of CTAs per call
SIZES2 = [2 * BLOCK, 2 * BLOCK, 200, 2 * BLOCK + 37, BLOCK, 3 * BLOCK + 13, 2 * BLOCK, 50_000]
TABLE = [409_600, 409_600, 100_000]


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


def _sequences():
    """Runs every sequence once; returns {name: array}. Nothing is read back between the calls of a sequence unless
    said so."""
    from qdsp_b200 import blocks as B, lib, synth

    L = lib.load()
    out = {}
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
    return out


def _dump(path):
    np.savez(path, **_sequences())


@pytest.fixture(scope="module")
def runs(tmp_path_factory):
    path = str(tmp_path_factory.mktemp("serial") / "serial.npz")
    env = dict(os.environ, QDSP_PDL="0", PYTHONPATH=ROOT)
    code = f"from tests.test_vfofm_overlapped_calls import _dump; _dump({path!r}); print('ok')"
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "ok" in r.stdout, r.stdout + r.stderr
    serial = dict(np.load(path))
    return _sequences(), serial


def _bits_equal(a, b):
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


@pytest.mark.gpu
def test_same_buffers_every_call(runs):
    ours, serial = runs
    assert _bits_equal(ours["same_buffers_last"], serial["same_buffers_last"])
    assert _bits_equal(ours["same_buffers_next"], serial["same_buffers_next"])
    # the stream is x repeated K1 + 1 times; calls K1 and K1 + 1 against the oracle, their seam included
    from qdsp_b200 import synth

    x1 = synth.cfg2_input(0, N1)
    total = (K1 + 1) * N1
    m1 = N1 // 50
    audio = np.zeros(total // 50, np.float32)
    audio[(K1 - 1) * m1:K1 * m1] = ours["same_buffers_last"]
    audio[K1 * m1:] = ours["same_buffers_next"]

    def get_in(lo, hi):
        return np.take(x1, np.arange(lo, hi) % N1)

    span = 65536
    centres = [K1 * N1, (K1 - 1) * N1 + span, (K1 - 1) * N1 + N1 // 2, K1 * N1 + N1 // 2, total - span]
    err, cmp = windows.check_vfofm_windows(get_in, audio, total, BLOCK, centres, span, *CHAIN, 50, 401)
    assert cmp > 0 and err <= AUDIO_TOL, err


@pytest.mark.gpu
def test_distinct_buffers_ragged_calls(runs):
    ours, serial = runs
    assert _bits_equal(ours["distinct"], serial["distinct"])
    from qdsp_b200 import synth

    x2 = synth.cfg2_input(0, sum(SIZES2))
    sizes = []
    for s in SIZES2:
        sizes += [int(b) for b in loader.as_blocks(s, BLOCK)]
    a64, _ = loader.port().vfo_fm(*CHAIN, x2, sizes, nco_f64=True)
    assert ours["distinct"].shape == a64.shape
    assert np.abs(ours["distinct"][16:] - a64[16:]).max() <= AUDIO_TOL


@pytest.mark.gpu
@pytest.mark.parametrize("case", [("raw_a1", "raw_big", "raw_a3"), ("table_last",), ("iq_audio", "iq_iq"), ("between_audio",)],
                         ids=["input_overlaps_previous_audio", "table_partition", "want_iq", "kernel_in_between"])
def test_refused_overlap_cases(runs, case):
    ours, serial = runs
    for k in case:
        assert _bits_equal(ours[k], serial[k]), k
