"""GPU parity of RDSDemod (decoder_modules/radio/src/rds_demod.h:64-73), the symbol-rate half of the RDS path: FastAGC, two
Costas loops, complex band-pass, Mueller & Mueller clock recovery, slicer, differential decoder -- b200_rds_demod_* against the
oracle's restatement (itself bit-identical to the reference's own class, tests/test_oracle_vs_ref.py).

Three feedback loops: the device follows the reference statement by statement in fp32, the only difference left is the last
bit of sinf / cosf (CUDA's vs the host libm's).  The loops are contracting, so the soft symbols agree to ~1e-6; what a
last-bit difference CAN do, rarely, is move the clock recovery's phase across one of its 128 interpolator boundaries for a
symbol -- a 1/128-sample timing step on that symbol, absorbed by the loop.  The gate therefore is: relative RMS error of the
soft symbols below 1e-5 on all but at most 0.5 % of them, below 1e-3 over all of them, decoded bits identical wherever the soft
value is not within 1e-3 of the decision threshold, and the same symbol count (+-1 at the very end)."""
import numpy as np
import pytest

from util import rel_rms, rds_baseband, rds_mpx_iq

pytestmark = pytest.mark.gpu
TOL = 1e-5


@pytest.fixture(scope="module")
def sb():
    import sdrplusplus_b200 as m
    from sdrplusplus_b200 import lib
    L = lib.load()
    assert L.b200_device_count() > 0
    assert L.b200_init(0) == 0
    return m


def _gate(soft, hard, so, ho):
    assert abs(soft.size - so.size) <= 1, (soft.size, so.size)
    n = min(soft.size, so.size)
    soft, hard, so, ho = soft[:n], hard[:n], so[:n], ho[:n]
    scale = float(np.sqrt(np.mean(so.astype(np.float64) ** 2)))
    err = np.abs(soft.astype(np.float64) - so.astype(np.float64)) / scale
    cut = np.sort(err)[int(0.995 * (n - 1))]
    e_all = rel_rms(soft, so)
    # a bit may differ only where a soft value (this symbol's or the previous one's: the decoder is differential) sits on the threshold
    near = np.abs(so) < 1e-3 * scale
    near = near | np.concatenate([[False], near[:-1]])
    bad = int(np.count_nonzero((hard != ho) & ~near))
    return {"symbols": int(n), "p99_5_rel_err": float(cut), "max_rel_err": float(err.max()), "rel_rms_all": e_all,
            "bit_mismatches": int(np.count_nonzero(hard != ho)), "bit_mismatches_off_threshold": bad}


@pytest.mark.parametrize("chunk", [839, 25, 5000])
def test_rds_demod_block_vs_oracle(sb, oracle, report, chunk):
    x, bits = rds_baseband(4000, 21)
    d = sb.RdsDemod()
    soft, hard = d.process_chunks(x, chunk)
    so, ho = oracle.rds_demod().process_chunks(x, chunk)
    r = _gate(soft, hard, so, ho)
    r["launches"] = d.launch_count()
    report["rds_demod_block_chunk%d" % chunk] = r
    assert r["launches"] == (x.size + chunk - 1) // chunk                 # the kernel ran, once per chunk
    assert r["p99_5_rel_err"] < TOL, r
    assert r["rel_rms_all"] < 1e-3, r
    assert r["bit_mismatches_off_threshold"] == 0, r
    # and the transmitted bits come back once the loops have locked
    tail = hard[600:2600]
    best = max(np.mean(tail == bits[k: k + tail.size]) for k in range(560, 640))
    assert best > 0.99, best
    # reset: the same input gives the same symbols again (apart from the clock recovery's 7-sample tail, which reset keeps)
    d.reset()
    s2, h2 = d.process_chunks(x, chunk)
    assert s2.size == soft.size and np.array_equal(h2[8:], hard[8:])
    d.close()


def test_rds_chain_from_fm_carrier(sb, oracle, report):
    """The whole RDS path behind the VFO: FM carrier with a 57 kHz biphase subcarrier -> BroadcastFM's rdsOut
    (b200_wfm_rds_create: discriminator, -57 kHz, 5 kS/s) -> b200_rds_demod; the oracle runs the same two blocks."""
    x, bits = rds_mpx_iq(1500, 3)
    xf = x.view(np.float32)
    y = sb.Block.wfm_rds(75e3, 250e3).process_chunks(xf, 12500).view(np.complex64)
    soft, hard = sb.RdsDemod().process_chunks(y, 250)
    oracle.set_rotator_mode(1)
    try:
        yo = oracle.wfm_rds(75e3, 250e3).process_chunks(xf, 12500).view(np.complex64)
    finally:
        oracle.set_rotator_mode(0)
    assert y.shape == yo.shape
    so, ho = oracle.rds_demod().process_chunks(yo, 250)
    r = _gate(soft, hard, so, ho)
    r["rds_out_rel_rms"] = rel_rms(y[100:], yo[100:])
    report["rds_chain_from_fm_carrier"] = r
    assert r["rds_out_rel_rms"] < TOL, r
    # the demodulator's input already differs by the rdsOut error (~1e-6): the same gate, one decade wider
    assert r["p99_5_rel_err"] < 1e-4, r
    assert r["bit_mismatches_off_threshold"] == 0, r
    best = max(np.mean(hard[300:1300] == bits[k: k + 1000]) for k in range(200, 400))
    assert best == 1.0, best


def test_rds_demod_reads_device_memory(sb, oracle):
    """`in` may be a device pointer: the 5 kS/s stream of a front-end VFO can be handed over without a host round trip"""
    import torch
    x, _ = rds_baseband(800, 4)
    t = torch.from_numpy(x.view(np.float32).copy()).cuda()
    d = sb.RdsDemod()
    s_dev, h_dev = d.process(t)
    d2 = sb.RdsDemod()
    s_host, h_host = d2.process(x)
    assert np.array_equal(s_dev.view(np.uint32), s_host.view(np.uint32)) and np.array_equal(h_dev, h_host)
    so, ho = oracle.rds_demod().process(x)
    assert abs(so.size - s_host.size) <= 1
    assert d.process(np.empty(0, np.complex64))[0].size == 0


def test_rds_chain_feeds_the_reference_group_decoder(sb):
    """FM carrier whose RDS subcarrier carries PI 0xB200 / PS 'B200 DSP' -> b200_wfm_rds -> b200_rds_demod -> the group decoder
    of the tests (util.rds_decode_ps, which reads from this signal what the reference's own group decoder rds.cpp read:
    tests/test_oracle_vs_ref.py): the programme identification and the name come out."""
    from golden_cases import rds_group_signal
    from util import rds_decode_ps
    _, x = rds_group_signal()
    y = sb.Block.wfm_rds(75e3, 250e3).process_chunks(x.view(np.float32), 12500).view(np.complex64)
    _, hard = sb.RdsDemod().process_chunks(y, 250)
    assert rds_decode_ps(hard) == (0xB200, "B200 DSP")
