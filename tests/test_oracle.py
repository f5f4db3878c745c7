"""CPU tests of the oracle (the checker the GPU parity tests lean on).

Pinning, in order of strength:
  1. golden fixtures produced by the reference's OWN dsp headers (tests/golden/reference_path.npz, made by
     tools/make_golden.py from oracle/_ref) -- the restatement must reproduce them bit for bit;
  2. SHA-256 fingerprints of the reference build's outputs, block by block on seeded random inputs
     (tests/golden/oracle_vs_ref.npz): the restatement must match every one (test_oracle_vs_ref.py);
  3. analytic known answers (impulse -> taps, tone -> bin and level, DC gain of the decimation cascade,
     constant-frequency FM -> constant audio) and a float64 numpy FFT bound the leaf arithmetic, which is the part
     no reference artefact pins (VOLK / FFTW are external and absent: SURVEY.md section 8c).
"""
import os

import numpy as np
import pytest

from golden_cases import run_cases
from util import noise_iq

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_path.npz")


def test_restatement_reproduces_reference_golden(oracle):
    want = np.load(GOLDEN)
    got = run_cases(oracle)
    assert set(got) == set(want.files)
    for k in want.files:
        a, b = np.asarray(got[k]), want[k]
        assert a.shape == b.shape, k
        if a.dtype == np.float32:
            assert np.array_equal(a.view(np.uint32), b.view(np.uint32)), "golden mismatch (bitwise): " + k
        else:
            assert np.array_equal(a, b), "golden mismatch: " + k


@pytest.mark.parametrize("N", [8, 16, 32, 64, 128, 1024, 4096, 65536, 1 << 18])
def test_fft_against_float64_numpy(oracle, N):
    x = noise_iq(N, N, 1.0)
    X = oracle.fft_raw(N, N, 0, x)
    w = np.where(np.arange(N) % 2, -1.0, 1.0)                  # rectangular window carries the (-1)^n pre-twist
    ref = np.fft.fft(x.astype(np.complex128) * w)
    err = np.linalg.norm(X - ref) / np.linalg.norm(ref)
    assert err < 3e-7, err


def test_tone_lands_on_expected_bin_with_expected_level(oracle):
    N = 65536
    A, b = 0.25, 1234                                           # bin offset from the centre (DC sits at N/2)
    n = np.arange(N)
    x = (A * np.exp(2j * np.pi * b * n / N)).astype(np.complex64)
    line = oracle.fft_frame(N, N, 2, x)
    assert int(np.argmax(line)) == N // 2 + b
    wsum = np.sum(np.abs(oracle.window_buf(2, N)).astype(np.float64))
    want = 20 * np.log10(A * wsum / N)                          # SURVEY 8c: 20 log10(A * sum(w) / N)
    assert abs(float(line[N // 2 + b]) - want) < 1e-3


def test_impulse_through_each_decimation_stage_returns_its_taps(oracle):
    for ratio in (2, 8, 256):
        plan = oracle.decim_plan(ratio)
        d0, t0 = plan[0]
        taps = oracle.decim_taps(ratio, 0)
        # an impulse at index t0-1 + k*d0 makes output k+... walk the taps; simplest: feed an impulse and a plain
        # decimating FIR with decimation 1 returns the reversed (here symmetric) tap table
        imp = np.zeros(2 * (t0 + 8), np.float32)
        imp[0] = 1.0
        y = oracle.decfir_cr(taps, 1).process(imp).view(np.complex64)
        assert np.array_equal(y.real[:t0], taps[::-1])
        assert np.allclose(taps, taps[::-1], atol=1e-9)          # all plan tables are symmetric (SURVEY App. A 18)


def test_decimation_cascade_dc_gain(oracle):
    # plan_256 = (32,143)(4,27)(2,69): DC gain = product of the per-table tap sums (SURVEY App. A 18: ~1.0083)
    g = 1.0
    for s in range(3):
        g *= float(np.sum(oracle.decim_taps(256, s).astype(np.float64)))
    x = np.ones(2 * 400000, np.float32)
    x[1::2] = 0.0
    y = oracle.decim(256).process(x).view(np.complex64)
    assert abs(y[-1].real - g) < 2e-5 and abs(y[-1].imag) < 1e-6
    assert abs(g - 1.0083) < 2e-3


def test_xlator_of_dc_is_a_pure_phasor(oracle):
    fs, off, n = 2.4e6, -300e3, 4096
    x = np.zeros(2 * n, np.float32)
    x[0::2] = 1.0
    b = oracle.xlator(off, fs)
    y = b.process(x).view(np.complex64)
    _, dl = oracle.xlator_phase(b)
    w = np.arctan2(np.float64(dl[1]), np.float64(dl[0]))
    assert np.max(np.abs(y - np.exp(1j * w * np.arange(n)))) < 2e-6
    assert abs(w - 2 * np.pi * off / fs) < 1e-7


def test_constant_frequency_fm_demodulates_to_a_constant(oracle):
    fs, dev, f = 250e3, 75e3, 10e3
    n = 5000
    x = np.exp(2j * np.pi * f * np.arange(n) / fs).astype(np.complex64)
    y = oracle.quad(dev, fs).process(x.view(np.float32))
    assert np.max(np.abs(y[1:] - f / dev)) < 2e-6
    a = oracle.wfm(dev, fs, False, True).process(x.view(np.float32)).reshape(-1, 2)
    assert np.array_equal(a[:, 0], a[:, 1])
    lp_gain = float(np.sum(oracle.lowpass(15000.0, 4000.0, fs).astype(np.float64)))
    assert abs(a[-1, 0] - lp_gain * f / dev) < 5e-6


def test_chunking_does_not_change_linear_blocks(oracle):
    """Delay lines / offsets / polyphase phase are carried exactly: any chunking gives bit-identical output."""
    fs, n = 2.4e6, 120000
    x = noise_iq(n, 99, 0.5).view(np.float32)
    a = oracle.rxvfo(fs, 250e3, 150e3, 300e3).process_chunks(x, 12000)
    b = oracle.rxvfo(fs, 250e3, 150e3, 300e3).process_chunks(x, 12000 * 5)
    assert a.size == b.size
    # the rotator renormalises per call (every 512 samples counted from the start of each call): chunking moves the
    # renormalisation points, so equality is to fp32 rounding, not bitwise
    assert np.linalg.norm(a - b) / np.linalg.norm(b) < 1e-6
    c = oracle.decim(8).process_chunks(x, 7777)
    d = oracle.decim(8).process_chunks(x, 12000)
    assert np.array_equal(c, d)


def test_agc_depends_on_chunk_boundaries_like_the_reference(oracle):
    """AGC clip look-ahead scans to the end of the current chunk (agc.h:93-101): documented quirk, kept."""
    sr, n = 24e3, 4800
    t = np.arange(n)
    x = (0.01 * np.exp(2j * np.pi * 0.03 * t)).astype(np.complex64)
    x[2400:] *= 400.0                                           # a jump that clips ...
    x[3000:] *= 3.0                                             # ... and a larger level the look-ahead sees only if it is in the same chunk
    a = oracle.ssb(2, 4600.0, sr, 50 / sr, 5 / sr).process_chunks(x.view(np.float32), 4800)
    b = oracle.ssb(2, 4600.0, sr, 50 / sr, 5 / sr).process_chunks(x.view(np.float32), 2450)
    assert a.shape == b.shape and not np.array_equal(a, b)


def test_zoom_right_edge_and_hold_start_index(oracle):
    line = np.arange(1000, dtype=np.float32)
    z = oracle.zoom(900, 200, 50, line)                          # window runs off the right edge: clipped, last pixels -inf
    assert z[0] == 903.0 and np.isneginf(z[-1])
    h = oracle.hold(np.zeros(8, np.float32), np.full(8, 5.0, np.float32), 1.0)
    assert h[0] == 0.0 and np.all(h[1:] == 5.0)                  # the reference's hold loop starts at i = 1
