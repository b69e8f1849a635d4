"""Back-to-back calls of the fused VFO -> FM chain on one handle: consecutive grids may overlap on the GPU (programmatic
dependent launch, k_rowlane.cu). Every sequence here runs twice (tests/overlapped.py) -- in this process (overlap
allowed) and in a subprocess with QDSP_PDL=0 (every launch serialized) -- and the audio must be bit-identical; the
streams are also checked against the oracle (oracle/port.c, float64 NCO) across the call seams."""
import numpy as np
import pytest

from oracle import loader, windows
from tests import overlapped

BLOCK = 819_200
CHAIN = (250e3, 2.4e6, 48e3, 48e3, 5e3)
AUDIO_TOL = 1e-4
N1, K1 = 20 * BLOCK, 8                     # the benchmark's pattern: > one wave of CTAs per call
SIZES2 = [2 * BLOCK, 2 * BLOCK, 200, 2 * BLOCK + 37, BLOCK, 3 * BLOCK + 13, 2 * BLOCK, 50_000]


@pytest.fixture(scope="module")
def runs():
    return overlapped.runs()


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
