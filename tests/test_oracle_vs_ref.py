"""The plain-C restatement must be BIT-IDENTICAL to the reference's own dsp headers over the restated leaf layer, block by
block.  tools/make_golden.py ran every case of golden_cases.VS_REF on the reference build and stored a SHA-256 of each output
(dtype, shape and bytes) in tests/golden/oracle_vs_ref.npz; these tests run the same cases on the restatement."""
import os

import numpy as np
import pytest

from golden_cases import VS_REF, rds_group_signal, sha256
from util import rds_baseband, rds_decode_ps

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "oracle_vs_ref.npz")


@pytest.fixture(scope="module")
def golden():
    return np.load(GOLDEN)


def _same_as_reference(golden, case, got):
    want = sorted(k.split("__", 1)[1] for k in golden.files if k.startswith(case + "__") and not k.endswith(("_full", "_branch")))
    assert sorted(got) == want
    for name, a in got.items():
        assert np.array_equal(sha256(a), golden[case + "__" + name]), "differs from the reference build: %s/%s" % (case, name)


@pytest.mark.parametrize("seed", [1, 2])
def test_blocks_bit_identical(oracle, golden, seed):
    case = "blocks_seed%d" % seed
    got = VS_REF[case](oracle)
    _same_as_reference(golden, case, got)
    # RDS side output of BroadcastFM (rdsOut): one sample per 50 of the 250 kS/s VFO; the reference's stereo branch gave the
    # same output as its mono branch (the same three blocks behind the same discriminator)
    assert abs(got["wfm_rds"].size // 2 - (got["vfo_in"].size // 2) // 50) <= 1
    assert np.array_equal(golden[case + "__wfm_rds_stereo_branch"], golden[case + "__wfm_rds"])


def test_design_and_spectrum_bit_identical(oracle, golden):
    _same_as_reference(golden, "design", VS_REF["design"](oracle))


def test_packet_and_export_formats_bit_identical(oracle, golden):
    """compressed sample stream (sample_stream_compressor.h / _decompressor.h) and the recorder conversions: the
    restatement against the reference's own code, plus known answers."""
    got = VS_REF["formats"](oracle)
    _same_as_reference(golden, "formats", got)
    from util import noise_iq, fm_carrier
    x = (noise_iq(5000, 3, 0.4) + fm_carrier(5000, 2.4e6, 300e3)).astype(np.complex64)
    for t in (0, 1, 2):
        ps = got["pcm_packet%d" % t]
        y = oracle.pcm_decompress(ps)
        # the scaler is the largest sample VALUE (not magnitude): samples inside (-max, max) come back within half a
        # step, more negative ones saturate -- the reference's behaviour, kept
        xf, yf = x.view(np.float32), y.view(np.float32)
        mx = float(np.max(xf))
        step = {0: mx / 128.0, 1: mx / 32768.0, 2: 0.0}[t]
        inside = np.abs(xf) < mx * (1.0 - 1.0 / 128.0)
        assert np.max(np.abs(yf[inside] - xf[inside])) <= step * 0.51 + 1e-9
        assert ps.size == 8 + x.size * {0: 2, 1: 4, 2: 8}[t]
        assert int(ps[2]) + 256 * int(ps[3]) == t and int(ps[0]) == 0 and int(ps[1]) == 0
    a = np.array([0.0, 0.5, -0.5, 1.0, -1.0, 2.0, -2.0, 1.5e-5, 0.25000763], np.float32)
    assert list(oracle.export_convert(a, 1)[:7]) == [0, 16384, -16384, 32767, -32767, 32767, -32768]     # rintf: ties to even, saturation
    assert list(oracle.export_convert(a[:5], 0)) == [128, 191, 64, 255, 1]


def test_rds_demod_bit_identical(oracle, golden):
    """RDSDemod (decoder_modules/radio/src/rds_demod.h: FastAGC, two Costas loops, band-pass, M&M clock recovery, slicer,
    differential decoder): the restatement against the reference's own class, tap sets, soft values and bits, across chunk
    sizes and a reset; the loops lock and the bits come back."""
    got = VS_REF["rds_demod"](oracle)
    _same_as_reference(golden, "rds_demod", got)
    x, bits = rds_baseband(3000, 11)
    assert got["bandpass_taps"].size == 2 * 190
    for chunk in (x.size, 839, 25, 1):
        n = x.size if chunk > 1 else 1500
        assert got["soft_chunk%d" % chunk].size == got["hard_chunk%d" % chunk].size
        assert abs(got["soft_chunk%d" % chunk].size - n * 1187.5 / 5000.0) <= 4
    # same start state after a reset, apart from the samples MM::reset leaves in its work buffer
    assert np.array_equal(got["hard_reset"][8:], got["hard_chunk839"][8:])
    # the decoded stream carries the transmitted bits (after the loops have settled), at some fixed delay
    _, hard = oracle.rds_demod().process_chunks(x, 1000)
    tail = hard[600:]
    best = max(np.mean(tail[: 2000] == bits[d: d + 2000]) for d in range(560, 640))
    assert best > 0.99, best


def test_rds_bits_are_what_the_reference_group_decoder_reads(oracle, golden):
    """An RDS subcarrier carrying four type-0A groups (PI 0xB200, PS name 'B200 DSP', checkwords per IEC 62106) on an FM
    carrier -> rdsOut branch -> RDSDemod: the restatement's bits are the reference's, from which the reference's OWN group
    decoder (decoder_modules/radio/src/rds.cpp) read the PI code and the name; the group decoder of the tests reads the same."""
    bits, _ = rds_group_signal()
    got = VS_REF["rds_groups"](oracle)
    _same_as_reference(golden, "rds_groups", got)
    assert np.array_equal(got["hard"], golden["rds_groups__hard_full"])
    assert np.array_equal(got["soft"].view(np.uint32), golden["rds_groups__soft_full"].view(np.uint32))
    for what, b in (("generator", bits), ("chain", got["hard"])):
        want = (int(golden["rds_decoder__%s_pi" % what]), str(golden["rds_decoder__%s_ps" % what]))
        assert want == (0xB200, "B200 DSP"), (what, want)
        assert rds_decode_ps(b) == want, what
