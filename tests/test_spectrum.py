"""Welch power spectrum (qdsp_spectrum_*, blocks.Spectrum, dsp::Spectrum).

CPU: the C-ABI surface, the example graph compiles, the row-count arithmetic.
GPU: rows against numpy's float64 FFT on the same float32 samples; rows bit-identical under any split of the stream into
calls; one 2^28-sample call; the dsp:: graph example."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FS4, NCH4, SPACING4 = 61_440_000, 256, 240_000


# ---- the row-count arithmetic, restated --------------------------------------------------------------------------
def frames_complete(P, N, hop):
    """Frames f (samples [f*hop, f*hop + N)) that lie inside the first P samples of the stream."""
    return (P - N) // hop + 1 if P >= N else 0


def rows_complete(P, N, hop, A):
    return frames_complete(P, N, hop) // A


def slice_len(N, A):
    """Frames per slice: the kernel's spectrum_slice_len."""
    return min(A, 65536 // N)


def test_spectrum_symbols_declared_exported_and_typed(qlib):
    from qdsp_b200 import lib

    names = ["qdsp_spectrum_create", "qdsp_spectrum_destroy", "qdsp_spectrum_out_rows", "qdsp_spectrum_process",
             "qdsp_spectrum_reset"]
    declared = lib.header_symbols()
    for n in names:
        assert n in declared and n in lib.SIGNATURES and hasattr(qlib, n), n
    assert lib.SIGNATURES["qdsp_spectrum_process"][0] is C.c_longlong
    assert lib.SIGNATURES["qdsp_spectrum_out_rows"][0] is C.c_longlong


def test_spectrum_example_compiles(qlib, tmp_path):
    exe = tmp_path / "spectrum_chain"
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-I" + os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "examples", "spectrum_chain.cpp"), "-L" + os.path.join(ROOT, "qdsp_b200"),
                           "-lqdsp_b200", "-lpthread", "-Wl,-rpath," + os.path.join(ROOT, "qdsp_b200"), "-o", str(exe)])
    assert exe.exists()


@pytest.mark.parametrize("N,hop,A,cases", [
    # contiguous frames: one row per N samples
    (4, 4, 1, [(0, 0), (3, 0), (4, 1), (7, 1), (8, 2), (12, 3)]),
    # gaps: frame 1 is samples 10..13, samples 4..9 are never read
    (4, 10, 1, [(4, 1), (9, 1), (13, 1), (14, 2), (23, 2), (24, 3)]),
    # overlap: frames end at 8, 10, 12, ...
    (8, 2, 1, [(7, 0), (8, 1), (9, 1), (10, 2), (16, 5)]),
    # A > 1 with overlap: frames end at 4, 6, 8, 10, 12, 14; rows after 3 and 6 frames
    (4, 2, 3, [(7, 0), (8, 1), (13, 1), (14, 2), (19, 2), (20, 3)]),
    # A > 1 with gaps: frames end at 4, 9, 14, 19; rows after 2 and 4 frames
    (4, 5, 2, [(8, 0), (9, 1), (18, 1), (19, 2)]),
])
def test_spectrum_row_count_arithmetic(N, hop, A, cases):
    for P, rows in cases:
        assert rows_complete(P, N, hop, A) == rows, (P, rows)
    # rows a call completes depend on where it ends only
    for p0 in range(0, 30):
        for c in range(0, 30):
            got = rows_complete(p0 + c, N, hop, A) - rows_complete(p0, N, hop, A)
            assert got == sum(1 for r in range(64) if p0 < (r * A + A - 1) * hop + N <= p0 + c)


# ---- GPU helpers ---------------------------------------------------------------------------------------------------
def ref_rows(x, N, hop, A, w=None):
    """numpy float64 FFT of the same float32 samples, the mean of A frames per row, FFT-shifted."""
    R = frames_complete(len(x), N, hop) // A
    idx = np.arange(R * A, dtype=np.int64)[:, None] * hop + np.arange(N)[None, :]
    fr = x[idx].astype(np.complex128)
    if w is not None:
        fr = fr * np.asarray(w, np.float32).astype(np.float64)
    P = np.abs(np.fft.fft(fr, axis=1)) ** 2
    return np.fft.fftshift(P.reshape(R, A, N).mean(axis=1), axes=1)


def assert_rows_close(got, want, what=""):
    assert got.shape == want.shape, (what, got.shape, want.shape)
    for r in range(len(want)):
        d = got[r].astype(np.float64) - want[r]
        rel = np.linalg.norm(d) / np.linalg.norm(want[r])
        assert rel <= 1e-5, f"{what} row {r}: rel-L2 {rel:.3e}"
        worst = np.abs(d).max() / want[r].max()
        assert worst <= 1e-5, f"{what} row {r}: max |err| / row max {worst:.3e}"


def hann(N):
    return (0.5 - 0.5 * np.cos(2 * np.pi * np.arange(N) / N)).astype(np.float32)


def comb_device(n):
    """config 4's wideband comb generated on the device: (DevBuf, host copy)."""
    from qdsp_b200 import blocks as B, lib

    d = B.DevBuf(n * 8)
    lib.check(lib.load().qdsp_synth_comb_cf32(d.ptr, 0, n, FS4, NCH4, SPACING4, 5e3, 1.0 / 64.0, 0.001, 4, None))
    return d, d.to_numpy(np.complex64, n)


GRID_N = [64, 256, 1024, 4096, 16384]
MAX_LEN = (2 * 64 + 1) * 3 * 16384 + 16384


@pytest.fixture(scope="module")
def signals():
    from qdsp_b200 import synth

    _, comb = comb_device(MAX_LEN)
    return {"cfg2": synth.cfg2_input(0, MAX_LEN), "comb": comb}


@pytest.mark.gpu
@pytest.mark.parametrize("N", GRID_N)
@pytest.mark.parametrize("hop_kind", ["N", "N/2", "N/4+3", "3N"])
def test_spectrum_matches_numpy(qlib, signals, N, hop_kind):
    from qdsp_b200 import blocks as B

    hop = {"N": N, "N/2": N // 2, "N/4+3": N // 4 + 3, "3N": 3 * N}[hop_kind]
    w = hann(N)
    for A in (1, 7, 64):
        n = (2 * A + 1) * hop + N + 5          # two full rows and part of a third
        for name, x in signals.items():
            x = x[:n]
            got = B.Spectrum(N, w, hop, A).process(x)
            assert_rows_close(got, ref_rows(x, N, hop, A, w), f"{name} N={N} hop={hop} A={A}")


@pytest.mark.gpu
@pytest.mark.parametrize("N,b", [(64, 5), (1024, 100), (1024, 1000), (16384, 12345)])
def test_spectrum_pure_tone_peaks_at_shifted_bin(qlib, N, b):
    from qdsp_b200 import blocks as B

    n = np.arange(8 * N)
    x = np.exp(2j * np.pi * ((b * n) % N) / N).astype(np.complex64)
    rows = B.Spectrum(N, None, N // 2, 3).process(x)
    assert len(rows) == frames_complete(len(x), N, N // 2) // 3
    assert np.all(np.argmax(rows, axis=1) == (b + N // 2) % N)


@pytest.mark.gpu
@pytest.mark.parametrize("N", [64, 4096])
def test_spectrum_null_window_equals_ones(qlib, signals, N):
    from qdsp_b200 import blocks as B

    x = signals["comb"][:20 * N]
    a = B.Spectrum(N, None, N // 4 + 3, 7).process(x)
    b = B.Spectrum(N, np.ones(N, np.float32), N // 4 + 3, 7).process(x)
    assert len(a) > 0 and np.array_equal(a.view(np.uint32), b.view(np.uint32))


def ragged_calls(n, N, hop, A, seed):
    """Call sizes summing to n: an empty call, calls shorter than hop and than N, then seeded sizes from 1 sample to a
    few rows, with calls that start an odd number of samples in (8 bytes off a 16-byte boundary)."""
    rng = np.random.default_rng(seed)
    sizes = [0, max(1, hop // 2), max(1, N // 3), 0, 1]
    row = A * hop
    while sum(sizes) < n:
        scale = [1, hop, N, row, 3 * row][int(rng.integers(0, 5))]
        sizes.append(int(rng.integers(1, max(2, scale) + 1)))
    sizes[-1] -= sum(sizes) - n
    return [s for s in sizes if s >= 0]


@pytest.mark.gpu
@pytest.mark.parametrize("N,hop,A", [
    (64, 19, 64),        # 32 frames side by side per CTA, one slice per row
    (256, 100, 300),     # two slices per row, 8 frames side by side
    (1024, 259, 7),
    (4096, 3 * 4096, 7),  # gaps between frames
    (16384, 8192, 7),    # two slices per row (4 + 3 frames), frames overlap
])
def test_spectrum_partition_invariant(qlib, signals, N, hop, A):
    from qdsp_b200 import blocks as B

    n = (3 * A + 2) * hop + N + 17
    x = signals["cfg2"][:n]
    din = B.DevBuf.from_numpy(x)
    rows_total = rows_complete(n, N, hop, A)
    whole = B.Spectrum(N, hann(N), hop, A)
    dout = B.DevBuf(rows_total * N * 4)
    assert whole.out_rows(n) == rows_total
    assert whole.process_device(din.ptr, dout.ptr, n) == rows_total
    want = dout.to_numpy(np.float32, rows_total * N)
    assert_rows_close(want.reshape(-1, N), ref_rows(x, N, hop, A, hann(N)), "single call")

    sizes = ragged_calls(n, N, hop, A, seed=N + hop + A)
    S = slice_len(N, A)
    ends = np.cumsum(sizes)
    starts = ends - np.asarray(sizes)
    F = np.asarray([frames_complete(int(e), N, hop) for e in ends])
    tail_start = F * hop                                 # where the first incomplete frame begins
    assert 0 in sizes and any(0 < s < hop for s in sizes) and any(0 < s < N for s in sizes)
    assert np.any((tail_start < ends) & (tail_start + N > ends)), "no call ends mid-frame"
    assert np.any((F % A) % S != 0), "no call ends mid-slice"
    assert np.any(F % A != 0), "no call ends mid-row"
    assert np.any(starts % 2 == 1), "no call starts 8 bytes off a 16-byte boundary"

    h = B.Spectrum(N, hann(N), hop, A)
    got = B.DevBuf(max(rows_total, 1) * N * 4)
    done = 0
    for s0, c in zip(starts, sizes):
        pred = h.out_rows(c)
        assert pred == rows_complete(int(s0) + c, N, hop, A) - rows_complete(int(s0), N, hop, A)
        r = h.process_device(din.ptr + 8 * int(s0), got.ptr + 4 * N * done, c)
        assert r == pred
        done += r
    assert done == rows_total
    out = got.to_numpy(np.float32, rows_total * N)
    assert np.array_equal(out.view(np.uint32), want.view(np.uint32))

    # after reset the handle equals a fresh one
    h.reset()
    assert h.out_rows(n) == rows_total
    assert h.process_device(din.ptr, got.ptr, n) == rows_total
    assert np.array_equal(got.to_numpy(np.float32, rows_total * N).view(np.uint32), want.view(np.uint32))


@pytest.mark.gpu
def test_spectrum_rejects_bad_parameters(qlib):
    from qdsp_b200 import blocks as B
    from qdsp_b200.lib import QdspError

    for args in [(100, None, 100, 1), (32, None, 32, 1), (32768, None, 32768, 1), (1024, None, 0, 1), (1024, None, 1024, 0)]:
        with pytest.raises(QdspError):
            B.Spectrum(*args)
    w = np.ones(1024, np.float32)
    w[5] = np.nan
    with pytest.raises(QdspError):
        B.Spectrum(1024, w)
    h = B.Spectrum(1024)
    x = B.DevBuf(4096 * 8)
    assert qlib.qdsp_spectrum_process(h.h, x.ptr, x.ptr, -1, None) == -1
    assert qlib.qdsp_spectrum_process(h.h, x.ptr + 4, x.ptr, 1024, None) == -1
    assert h.out_rows(0) == 0 and h.process_device(x.ptr, x.ptr, 0) == 0


@pytest.mark.gpu
def test_spectrum_full_size_call(qlib):
    from qdsp_b200 import blocks as B, lib

    n, N, A = 1 << 28, 4096, 64
    d = B.DevBuf(n * 8)
    lib.check(lib.load().qdsp_synth_comb_cf32(d.ptr, 0, n, FS4, NCH4, SPACING4, 5e3, 1.0 / 64.0, 0.001, 4, None))
    h = B.Spectrum(N, hann(N), N, A)
    R = h.out_rows(n)
    assert R == n // (N * A)
    out = B.DevBuf(R * N * 4)
    assert h.process_device(d.ptr, out.ptr, n) == R
    rows = out.to_numpy(np.float32, R * N).reshape(R, N)
    for r in np.linspace(0, R - 1, 64).astype(int):
        x = d.to_numpy(np.complex64, A * N, offset_bytes=8 * int(r) * A * N)
        assert_rows_close(rows[r:r + 1], ref_rows(x, N, N, A, hann(N)), f"row {r}")


@pytest.mark.gpu
@pytest.mark.parametrize("N,hop,A,block", [(1024, 512, 8, 300_000), (16384, 16384, 1, 1_000_000)])
def test_spectrum_cpp_graph_matches_numpy(qlib, tmp_path, N, hop, A, block):
    from qdsp_b200 import synth

    exe = tmp_path / "spectrum_chain"
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-I" + os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "examples", "spectrum_chain.cpp"), "-L" + os.path.join(ROOT, "qdsp_b200"),
                           "-lqdsp_b200", "-lpthread", "-Wl,-rpath," + os.path.join(ROOT, "qdsp_b200"), "-o", str(exe)])
    x = synth.cfg2_input(0, 2_500_000)
    fin, fout, fw = tmp_path / "in.cf32", tmp_path / "out.f32", tmp_path / "w.f32"
    x.tofile(fin)
    hann(N).tofile(fw)
    subprocess.check_call([str(exe), str(fin), str(fout), str(N), str(hop), str(A), str(block), str(fw)], timeout=120)
    got = np.fromfile(fout, np.float32)
    assert got.size % N == 0
    assert_rows_close(got.reshape(-1, N), ref_rows(x, N, hop, A, hann(N)), "dsp::Spectrum graph")


@pytest.mark.gpu
def test_spectrum_cpp_block_says_why_it_has_no_handle(qlib, tmp_path):
    exe = tmp_path / "spectrum_chain"
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-I" + os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "examples", "spectrum_chain.cpp"), "-L" + os.path.join(ROOT, "qdsp_b200"),
                           "-lqdsp_b200", "-lpthread", "-Wl,-rpath," + os.path.join(ROOT, "qdsp_b200"), "-o", str(exe)])
    fin = tmp_path / "in.cf32"
    np.zeros(4096, np.complex64).tofile(fin)
    for args, msg in [(["1024", "100", "1"], "average * hop"), (["1000", "1000", "1"], "power of two")]:
        p = subprocess.run([str(exe), str(fin), str(tmp_path / "out.f32")] + args, capture_output=True, text=True, timeout=60)
        assert p.returncode == 2 and msg in p.stderr, (args, p.returncode, p.stderr)
