"""The golden cases: one function that drives an oracle implementation (reference-header build or plain-C
restatement) over seeded inputs and returns {name: array}.  tools/make_golden.py runs it on the reference build
and commits the result; tests/test_oracle.py runs it on the restatement and demands bit-identical arrays."""
import hashlib

import numpy as np

from util import noise_iq, fm_carrier, am_carrier, ssb_tone, rds_baseband, rds_mpx_iq, rds_group_bits

FS = 2.4e6


def signal(n, seed):
    x = noise_iq(n, seed, 0.02).copy()
    x += fm_carrier(n, FS, 300e3)
    x += fm_carrier(n, FS, -650e3, tones=((3000.0, 0.6),))
    x += am_carrier(n, FS, -400e3)
    x += ssb_tone(n, FS, 600e3, 1000.0)
    return x


def digest(a):
    """order-sensitive checksum of a float32 array: [count, sum a[i]*(1 + i mod 251), sum |a|] in float64"""
    a = np.asarray(a, np.float32).reshape(-1).astype(np.float64)
    w = 1.0 + (np.arange(a.size) % 251)
    return np.array([a.size, float(np.sum(a * w)), float(np.sum(np.abs(a)))])


def stereo_mpx_iq(n, fs, seed=5):
    """FM carrier modulated with a stereo multiplex: L+R, 19 kHz pilot, L-R on the 38 kHz subcarrier (+ a little noise)."""
    t = np.arange(n, dtype=np.float64) / fs
    lpr = 0.4 * np.sin(2 * np.pi * 1000.0 * t) + 0.1 * np.sin(2 * np.pi * 3300.0 * t)
    lmr = 0.3 * np.sin(2 * np.pi * 700.0 * t)
    mpx = lpr + 0.1 * np.sin(2 * np.pi * 19000.0 * t) + lmr * np.sin(2 * np.pi * 38000.0 * t)
    ph = 2 * np.pi * 75e3 * np.cumsum(mpx) / fs
    rng = np.random.default_rng(seed)
    x = 0.5 * np.exp(1j * ph) + 0.001 * (rng.uniform(-1, 1, n) + 1j * rng.uniform(-1, 1, n))
    return x.astype(np.complex64)


def run_cases(R):
    g = {}
    # ---- host-side design ----
    g["lowpass_wfm_audio"] = R.lowpass(15000.0, 4000.0, 250000.0)
    g["lowpass_vfo_150k"] = R.lowpass(75000.0, 7500.0, 250000.0)
    g["lowpass_odd"] = R.lowpass(1400.0, 140.0, 24000.0, True)
    g["highpass_300_48k"] = R.highpass(300.0, 100.0, 48000.0)
    g["window_nuttall_4096"] = R.window_buf(2, 4096)
    g["window_blackman_1000"] = R.window_buf(1, 1000)
    for rates in ((2.4e6, 250e3), (100e6, 250e3), (1.024e9, 250e3), (2.4e6, 15e3), (250e3, 48e3)):
        p = R.resamp_plan(*rates)
        g["plan_%g_%g" % rates] = np.array([p[k] for k in ("mode", "predec_ratio", "interp", "decim", "ntaps", "taps_per_phase")])
    g["resamp_taps_2.4M_250k"] = R.resamp_taps(2.4e6, 250e3)
    g["decim_plan_256"] = np.array(R.decim_plan(256)).reshape(-1)
    g["decim_taps_256_0_digest"] = digest(R.decim_taps(256, 0))
    g["fft_params"] = np.array([R.fft_params(2.4e6, 65536, 20.0), R.fft_params(100e6, 1 << 20, 20.0)]).reshape(-1)
    # ---- streaming blocks on a seeded signal, chunked like file_source (fs/200) ----
    n, chunk = 240000, 12000
    x = signal(n, 0x5D12)
    xf = x.view(np.float32)
    g["seed"] = np.array([0x5D12, n, chunk])
    y = R.xlator(-300e3, FS).process_chunks(xf, chunk)
    g["xlator_head"] = y[:256]
    g["xlator_digest"] = digest(y)
    y = R.decim(8).process_chunks(xf, chunk)
    g["decim8_head"] = y[:256]
    g["decim8_digest"] = digest(y)
    y = R.resamp(FS, 250e3).process_chunks(xf, chunk)
    g["resamp_head"] = y[:256]
    g["resamp_digest"] = digest(y)
    vfo = R.rxvfo(FS, 250e3, 150e3, 300e3).process_chunks(xf, chunk)
    g["rxvfo_tail"] = vfo[-512:]
    g["rxvfo_digest"] = digest(vfo)
    a = R.wfm(75e3, 250e3).process_chunks(vfo, 1250)
    g["wfm_tail"] = a[-512:]
    g["wfm_digest"] = digest(a)
    g["quad_digest"] = digest(R.quad(75e3, 250e3).process_chunks(vfo, 1250))
    v = R.rxvfo(FS, 50e3, 12500.0, 300e3).process_chunks(xf, chunk)
    g["nfm_digest"] = digest(R.nfm(50e3, 12500.0, True).process_chunks(v, 250))
    v = R.rxvfo(FS, 15e3, 10e3, -400e3).process_chunks(xf, chunk)
    a = R.am(1, 10e3, 50 / 15e3, 5 / 15e3, 100 / 15e3, 15e3).process_chunks(v, 75)
    g["am_audio_tail"] = a[-128:]
    g["am_audio_digest"] = digest(a)
    g["am_carrier_digest"] = digest(R.am(0, 10e3, 50 / 15e3, 5 / 15e3, 100 / 15e3, 15e3).process_chunks(v, 75))
    v = R.rxvfo(FS, 24e3, 2800.0, 600e3).process_chunks(xf, chunk)
    a = R.ssb(0, 2800.0, 24e3, 50 / 24e3, 5 / 24e3).process_chunks(v, 120)
    g["usb_tail"] = a[-128:]
    g["usb_digest"] = digest(a)
    g["lsb_digest"] = digest(R.ssb(1, 2800.0, 24e3, 50 / 24e3, 5 / 24e3).process_chunks(v, 120))
    g["deemph_digest"] = digest(R.deemph(50e-6, 48e3).process_chunks(a, 480))
    # stereo branch of BroadcastFM (pilot band-pass -> PLL -> L-R recovery) on a synthetic stereo multiplex; power squelch
    ws = stereo_mpx_iq(100000, 250e3)
    a = R.wfm(75e3, 250e3, True, True).process_chunks(ws.view(np.float32), 1250)
    g["wfm_stereo_tail"] = a[-512:]
    g["wfm_stereo_digest"] = digest(a)
    g["squelch_digest"] = digest(R.squelch(-27.0).process_chunks((ws * np.linspace(0.02, 0.2, ws.size).astype(np.float32)).astype(np.complex64).view(np.float32), 1250))
    # RDS side output of BroadcastFM: discriminator -> -57 kHz -> 5 kS/s
    a = R.wfm_rds(75e3, 250e3).process_chunks(ws.view(np.float32), 1250)
    g["wfm_rds_tail"] = a[-256:]
    g["wfm_rds_digest"] = digest(a)
    # RDSDemod of the radio module (rds_demod.h): AGC, two Costas loops, band-pass, M&M clock recovery, slicer, differential
    # decoder -- on a synthetic 5 kS/s RDS baseband and behind the rdsOut branch of an FM carrier with a 57 kHz subcarrier
    xr, _ = rds_baseband(1500, 31)
    soft, hard = R.rds_demod().process_chunks(xr, 839)
    g["rds_demod_soft_tail"] = soft[-256:]
    g["rds_demod_soft_digest"] = digest(soft)
    g["rds_demod_bits"] = np.packbits(hard)
    xm, _ = rds_mpx_iq(400, 7)
    rds_if = R.wfm_rds(75e3, 250e3).process_chunks(xm.view(np.float32), 12500).view(np.complex64)
    soft, hard = R.rds_demod().process_chunks(rds_if, 250)
    g["rds_chain_soft_digest"] = digest(soft)
    g["rds_chain_bits"] = np.packbits(hard)
    bp, bank = R.rds_demod_taps()
    g["rds_bandpass_taps"] = bp.view(np.float32).copy()
    g["rds_interp_bank_digest"] = digest(bank)
    # IF chain of the radio module: noise blanker (impulses on top of the FM signal), FM IF noise reduction (32 and 15 bins)
    imp = ws[:30000].copy()
    imp[::997] *= np.float32(12.0)
    a = R.noise_blanker(500.0 / 250e3, 3.0).process_chunks(imp.view(np.float32), 1250)
    g["noise_blanker_tail"] = a[-256:]
    g["noise_blanker_digest"] = digest(a)
    wn = (ws[:30000] + noise_iq(30000, 9, 0.2)).astype(np.complex64)
    a = R.fm_if(32).process_chunks(wn.view(np.float32), 1250)
    g["fm_if32_tail"] = a[-256:]
    g["fm_if32_digest"] = digest(a)
    g["fm_if15_digest"] = digest(R.fm_if(15).process_chunks(wn.view(np.float32), 999))
    # radio AF chain behind WFM: 250 k -> 48 k stereo resampler, 300 Hz high-pass, 50 us deemphasis
    w = R.wfm(75e3, 250e3).process_chunks(vfo, 1250)
    af = R.resamp_stereo(250e3, 48e3).process_chunks(w, 1250)
    af = R.fir_cr(R.highpass(300.0, 100.0, 48000.0)).process_chunks(af, 240)
    af = R.deemph(50e-6, 48e3).process_chunks(af, 240)
    g["af_chain_tail"] = af[-256:]
    g["af_chain_digest"] = digest(af)
    # ---- spectrum branch ----
    line = R.fft_frame(65536, 65536, 2, x[:65536])
    g["fft_65536_stride"] = line[::64]
    g["fft_65536_digest"] = digest(line)
    g["fft_65536_argmax"] = np.array([int(np.argmax(line))])
    g["fft_4096_3000"] = R.fft_frame(4096, 3000, 1, x[:3000])
    g["zoom_1280"] = R.zoom(1000, 60000, 1280, line)
    g["zoom_edge"] = R.zoom(60000, 8000, 777, line)
    g["hold"] = R.hold(np.full(1280, -200.0, np.float32), g["zoom_1280"], 0.5)
    i16 = np.random.default_rng(3).integers(-32768, 32767, 512).astype(np.int16)
    g["i16_in"] = i16
    g["i16_out"] = R.i16_to_f32(i16)
    # ---- data formats either side of the path (compressed sample stream; recorder sample types) ----
    xs = signal(4096, 77).astype(np.complex64)
    for t, name in ((0, "i8"), (1, "i16"), (2, "f32")):
        pkt = R.pcm_compress(xs, t)
        g["pcm_packet_%s_head" % name] = pkt[:72].copy()
        g["pcm_packet_%s_digest" % name] = digest(pkt.astype(np.float32))
        g["pcm_roundtrip_%s_digest" % name] = digest(R.pcm_decompress(pkt).view(np.float32))
    a = np.concatenate([xs.view(np.float32) * 3.0, np.array([1.0, -1.0, 0.5, -0.5, 2.5e-5], np.float32)])
    g["export_i16_digest"] = digest(R.export_convert(a, 1).astype(np.float32))
    g["export_i32_head"] = R.export_convert(a[:64], 2)
    g["export_u8_head"] = R.export_convert(np.clip(a[:64], -1.0, 1.0), 0)
    return g


# ---- the block-by-block cases of test_oracle_vs_ref.py: tools/make_golden.py stores a SHA-256 of every output of the
# reference build, the tests recompute them on the restatement.  Each function returns {name: array}.

def sha256(a):
    """bit-exact fingerprint of an array: dtype, shape and bytes"""
    a = np.ascontiguousarray(a)
    h = hashlib.sha256(("%s%s" % (a.dtype.str, a.shape)).encode())
    h.update(a.tobytes())
    return np.frombuffer(h.digest(), np.uint8).copy()


def vs_ref_blocks(O, seed):
    n = 120000
    x = (noise_iq(n, seed, 0.3) + fm_carrier(n, FS, 300e3)).astype(np.complex64).view(np.float32)
    mk = [
        (lambda o: o.xlator(-300e3, FS), 12000), (lambda o: o.decim(2), 7777), (lambda o: o.decim(16), 12000),
        (lambda o: o.decim(128), 12000), (lambda o: o.resamp(FS, 250e3), 12000), (lambda o: o.resamp(FS, 24e3), 12000),
        (lambda o: o.resamp(48e3, 250e3), 3000), (lambda o: o.rxvfo(FS, 250e3, 150e3, 300e3), 12000),
        (lambda o: o.rxvfo(FS, 250e3, 250e3, -123456.0), 11999), (lambda o: o.rxvfo(FS, 15e3, 10e3, 1e5), 12000),
        (lambda o: o.dcblock_c(50.0 / FS), 12000),
    ]
    g = {"iq%02d" % k: f(O).process_chunks(x, ch) for k, (f, ch) in enumerate(mk)}
    y = O.rxvfo(FS, 250e3, 150e3, 300e3).process_chunks(x, 12000)
    g["vfo_in"] = y
    # RDS side output of BroadcastFM (rdsOut), mono branch
    g["wfm_rds"] = O.wfm_rds(75e3, 250e3).process_chunks(y, 1250)
    mk2 = [
        (lambda o: o.quad(75e3, 250e3), 1250), (lambda o: o.wfm(75e3, 250e3), 1250), (lambda o: o.wfm(75e3, 250e3, False, False), 999),
        (lambda o: o.nfm(250e3, 12500.0, True), 1250), (lambda o: o.am(1, 10e3, 2e-4, 2e-5, 4e-4, 250e3), 1250),
        (lambda o: o.am(0, 10e3, 2e-4, 2e-5, 4e-4, 250e3), 1250), (lambda o: o.ssb(0, 2800.0, 250e3, 2e-4, 2e-5), 1250),
        (lambda o: o.ssb(1, 2800.0, 250e3, 2e-4, 2e-5), 1250), (lambda o: o.ssb(2, 4600.0, 250e3, 2e-4, 2e-5), 1250),
        (lambda o: o.deemph(50e-6, 48e3), 480), (lambda o: o.resamp_stereo(250e3, 48e3), 1250),
        (lambda o: o.wfm(75e3, 250e3, True, True), 1250), (lambda o: o.wfm(75e3, 250e3, True, False), 777),      # stereo branch: pilot PLL
        (lambda o: o.squelch(-20.0), 1250), (lambda o: o.squelch(-60.0), 999),
        # IF chain of the radio module (radio_module.h:90-96): noise blanker, FM IF noise reduction at its four presets
        (lambda o: o.noise_blanker(500.0 / 24000.0, 2.0), 1250), (lambda o: o.noise_blanker(500.0 / 250e3, 1.2), 999),
        (lambda o: o.fm_if(32), 1250), (lambda o: o.fm_if(9), 999), (lambda o: o.fm_if(15), 1250), (lambda o: o.fm_if(31), 640),
    ]
    for k, (f, ch) in enumerate(mk2):
        g["vfo%02d" % k] = f(O).process_chunks(y, ch)
    return g


def vs_ref_design(O):
    g = {}
    for k, a in enumerate(((15000.0, 4000.0, 250000.0, False), (5000.0, 500.0, 15000.0, False), (3125.0, 312.5, 50000.0, True))):
        g["lowpass%d" % k] = O.lowpass(*a)
    g["highpass"] = O.highpass(300.0, 100.0, 48000.0)
    g["bandpass_c"] = O.bandpass_c(18750, 19250, 3000, 250000, True).view(np.float32)
    for r in (2, 4, 8, 16, 32, 64, 128, 256, 512, 1024, 2048, 4096, 8192):
        plan = O.decim_plan(r)
        g["decim_plan_%d" % r] = np.array(plan, np.int64).reshape(-1)
        for st in range(len(plan)):
            g["decim_taps_%d_%d" % (r, st)] = O.decim_taps(r, st)
    for rates in ((2.4e6, 250e3), (100e6, 250e3), (1.024e9, 50e3), (8e6, 24e3), (44100.0, 48000.0)):
        p = O.resamp_plan(*rates)
        g["resamp_plan_%g_%g" % rates] = np.array([p[k] for k in ("mode", "predec_ratio", "interp", "decim", "ntaps", "taps_per_phase")], np.int64)
        g["resamp_taps_%g_%g" % rates] = O.resamp_taps(*rates)
    x = noise_iq(65536, 7, 1.0)
    for N, nz, w in ((1024, 1024, 0), (65536, 65536, 2), (4096, 3000, 1)):
        g["fft_%d_%d_%d" % (N, nz, w)] = O.fft_frame(N, nz, w, x[:nz])
    line = O.fft_frame(65536, 65536, 2, x)
    for args in ((0, 65536, 1000), (1000, 60000, 1280), (60000, 8000, 777)):
        g["zoom_%d_%d_%d" % args] = O.zoom(args[0], args[1], args[2], line)
    return g


def vs_ref_formats(O):
    """compressed sample stream (sample_stream_compressor.h / _decompressor.h) and the recorder conversions"""
    g = {}
    x = (noise_iq(5000, 3, 0.4) + fm_carrier(5000, FS, 300e3)).astype(np.complex64)
    for t in (0, 1, 2):
        g["pcm_packet%d" % t] = O.pcm_compress(x, t)
        g["pcm_roundtrip%d" % t] = O.pcm_decompress(g["pcm_packet%d" % t]).view(np.uint32)
    a = np.array([0.0, 0.5, -0.5, 1.0, -1.0, 2.0, -2.0, 1.5e-5, 0.25000763], np.float32)
    for t in (0, 1, 2):
        g["export%d" % t] = O.export_convert(a[:5] if t == 0 else a, t)
    return g


def vs_ref_rds_demod(O):
    """RDSDemod: tap sets, then soft values and bits across chunk sizes and a reset"""
    bp, bank = O.rds_demod_taps()
    g = {"bandpass_taps": bp.view(np.float32), "interp_bank": bank}
    x, _ = rds_baseband(3000, 11)
    for chunk in (x.size, 839, 25, 1):
        xs = x if chunk > 1 else x[:1500]
        d = O.rds_demod()
        g["soft_chunk%d" % chunk], g["hard_chunk%d" % chunk] = d.process_chunks(xs, chunk)
        if chunk == 839:
            d.reset()
            g["soft_reset"], g["hard_reset"] = d.process_chunks(xs, chunk)
    return g


def rds_group_signal():
    """bits of six cycles of the type-0A groups carrying PI 0xB200 / PS 'B200 DSP', and an FM carrier whose 57 kHz RDS
    subcarrier carries them"""
    bits = rds_group_bits(0xB200, "B200 DSP", 6)
    x, _ = rds_mpx_iq(0, 3, bits=bits)
    return bits, x


def vs_ref_rds_groups(O):
    """the RDS groups behind the rdsOut branch of BroadcastFM and RDSDemod"""
    _, x = rds_group_signal()
    y = O.wfm_rds(75e3, 250e3).process_chunks(x.view(np.float32), 12500)
    soft, hard = O.rds_demod().process_chunks(y.view(np.complex64), 250)
    return {"rds_if": y, "soft": soft, "hard": hard}


VS_REF = {"blocks_seed1": lambda O: vs_ref_blocks(O, 1), "blocks_seed2": lambda O: vs_ref_blocks(O, 2), "design": vs_ref_design,
          "formats": vs_ref_formats, "rds_demod": vs_ref_rds_demod, "rds_groups": vs_ref_rds_groups}
