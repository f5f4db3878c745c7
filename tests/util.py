"""Shared helpers of the parity tests: seeded signals and error metrics."""
import numpy as np


def rel_rms(a, b):
    """||a-b||_2 / ||b||_2  (RMS-normalised relative error; b is the oracle)."""
    a = np.asarray(a, np.float64).reshape(-1) if not np.iscomplexobj(a) else np.asarray(a, np.complex128).reshape(-1)
    b = np.asarray(b, np.float64).reshape(-1) if not np.iscomplexobj(b) else np.asarray(b, np.complex128).reshape(-1)
    assert a.shape == b.shape, (a.shape, b.shape)
    den = np.linalg.norm(b)
    return float(np.linalg.norm(a - b) / den) if den > 0 else float(np.linalg.norm(a - b))


def max_rel(a, b):
    """max |a-b| / max |b|"""
    a = np.asarray(a).reshape(-1)
    b = np.asarray(b).reshape(-1)
    assert a.shape == b.shape, (a.shape, b.shape)
    den = np.max(np.abs(b))
    return float(np.max(np.abs(a - b)) / den) if den > 0 else float(np.max(np.abs(a - b)))


def noise_iq(n, seed, amp=1.0):
    """i.i.d. uniform[-amp, amp) re/im -- the SpeedTester distribution (core/src/dsp/bench/speed_tester.h:37-41)."""
    rng = np.random.default_rng(seed)
    x = np.empty(2 * n, np.float32)
    x[:] = rng.uniform(-amp, amp, 2 * n)
    return x.view(np.complex64)


def fm_carrier(n, fs, offset, dev=75000.0, tones=((1000.0, 0.5), (5000.0, 0.3)), amp=0.05, start=0):
    """FM carrier at `offset` Hz: instantaneous frequency offset + dev * sum(a_i sin(2 pi f_i t))."""
    t = (np.arange(n, dtype=np.float64) + start) / fs
    phase = 2 * np.pi * offset * t
    for f, a in tones:
        phase += -(dev * a / f) * np.cos(2 * np.pi * f * t)
    return (amp * np.exp(1j * phase)).astype(np.complex64)


def am_carrier(n, fs, offset, tone=1000.0, depth=0.5, amp=0.05):
    t = np.arange(n, dtype=np.float64) / fs
    env = 1.0 + depth * np.sin(2 * np.pi * tone * t)
    return (amp * env * np.exp(2j * np.pi * offset * t)).astype(np.complex64)


def ssb_tone(n, fs, offset, tone=1000.0, amp=0.05):
    t = np.arange(n, dtype=np.float64) / fs
    return (amp * np.exp(2j * np.pi * (offset + tone) * t)).astype(np.complex64)


def test_signal(n, fs, carriers, seed=0x5D12, noise_amp=0.01):
    """noise + FM carriers at the given (offset, ...) list."""
    x = noise_iq(n, seed, noise_amp).copy()
    for c in carriers:
        x += fm_carrier(n, fs, c)
    return x


def to_i16(x):
    """complex64 in [-1,1) -> interleaved int16 IQ (file_source format)."""
    v = np.clip(np.round(x.view(np.float32) * 32768.0), -32768, 32767).astype(np.int16)
    return v


def rds_baseband(nbits, seed, fs=5000.0, amp=0.02, cfo_hz=1.5, phase0=0.7, noise_amp=0.002):
    """An RDS-like complex baseband at `fs` (what BroadcastFM's rdsOut carries): random bits, differentially encoded, biphase
    symbols at 1187.5 Bd (two half-symbols of opposite sign) with raised-cosine edges, a small residual carrier offset and
    phase, uniform noise.  Returns (complex64 samples, the bits)."""
    rng = np.random.default_rng(seed)
    bits = rng.integers(0, 2, nbits)
    enc = np.cumsum(bits) % 2                                   # differential encoding
    chips = np.repeat(2.0 * enc - 1.0, 2) * np.tile([1.0, -1.0], nbits)
    chip_rate = 2375.0
    n = int(nbits * 2 * fs / chip_rate)
    t = np.arange(n, dtype=np.float64) / fs
    k = t * chip_rate
    idx = np.minimum(k.astype(np.int64), chips.size - 1)
    frac = k - idx
    nxt = chips[np.minimum(idx + 1, chips.size - 1)]
    # raised-cosine transition over the last 40 % of a chip
    w = np.clip((frac - 0.6) / 0.4, 0.0, 1.0)
    base = chips[idx] + (nxt - chips[idx]) * 0.5 * (1.0 - np.cos(np.pi * w))
    x = amp * base * np.exp(1j * (2 * np.pi * cfo_hz * t + phase0))
    x = x + (rng.uniform(-noise_amp, noise_amp, n) + 1j * rng.uniform(-noise_amp, noise_amp, n))
    return x.astype(np.complex64), bits


def rds_checkword(info16, offset):
    """the 10-bit checkword of an RDS block: remainder of info(x) x^10 by g(x) = x^10 + x^8 + x^7 + x^5 + x^4 + x^3 + 1,
    plus the block's offset word (IEC 62106; the syndromes the decoders look for follow from it)"""
    reg = info16 << 10
    for i in range(25, 9, -1):
        if reg & (1 << i):
            reg ^= 0x5B9 << (i - 10)
    return (reg & 0x3FF) ^ offset


RDS_OFFSET_WORDS = {0x0FC: "A", 0x198: "B", 0x168: "C", 0x350: "C'", 0x1B4: "D"}


def rds_decode_ps(bits):
    """Programme identification and service name from an RDS bit stream, per IEC 62106 without error correction: a group
    counts where four consecutive 26-bit blocks carry the offset words A, B, C (or C'), D; type-0 groups give the name two
    characters at a time.  Returns (PI or None, the 8-character name or None while a segment is missing)."""
    b = np.asarray(bits, np.int64)

    def block(p):
        w = int("".join(map(str, b[p:p + 26])), 2)
        info = w >> 10
        return info, RDS_OFFSET_WORDS.get(rds_checkword(info, 0) ^ (w & 0x3FF))

    pi, segs, p = None, {}, 0
    while p + 104 <= b.size:
        blocks = [block(p + 26 * k) for k in range(4)]
        if [t for _, t in blocks] in (["A", "B", "C", "D"], ["A", "B", "C'", "D"]):
            pi = blocks[0][0]
            if blocks[1][0] >> 12 == 0:
                segs[blocks[1][0] & 3] = blocks[3][0]
            p += 104
        else:
            p += 1
    name = "".join(chr(segs[s] >> 8) + chr(segs[s] & 0xFF) for s in range(4)) if len(segs) == 4 else None
    return pi, name


def rds_group_bits(pi, ps_name, repeats):
    """bit stream of `repeats` cycles of the four type-0A groups that carry the 8-character programme service name"""
    OFF = {"A": 0x0FC, "B": 0x198, "C": 0x168, "D": 0x1B4}
    ps = (ps_name + " " * 8)[:8]
    bits = []
    for _ in range(repeats):
        for seg in range(4):
            blocks = [("A", pi),
                      ("B", (0 << 12) | (0 << 11) | (0 << 10) | (10 << 5) | (0 << 4) | (1 << 3) | (0 << 2) | seg),   # group 0A, PTY 10, music
                      ("C", 0xE0CD),                                                                                # AF: "1 AF follows", 107.9 MHz
                      ("D", (ord(ps[2 * seg]) << 8) | ord(ps[2 * seg + 1]))]
            for name, info in blocks:
                word = (info << 10) | rds_checkword(info, OFF[name])
                bits.extend((word >> k) & 1 for k in range(25, -1, -1))
    return np.array(bits, np.int64)


def rds_mpx_iq(nbits, seed, fs=250e3, bits=None):
    """FM carrier at `fs` whose multiplex carries programme audio, the 19 kHz pilot and a biphase RDS subcarrier at 57 kHz
    (1187.5 Bd, differentially encoded).  Returns (complex64 IQ, bits)."""
    rng = np.random.default_rng(seed)
    if bits is None:
        bits = rng.integers(0, 2, nbits)
    else:
        bits = np.asarray(bits, np.int64)
        nbits = bits.size
    enc = np.cumsum(bits) % 2
    chips = np.repeat(2.0 * enc - 1.0, 2) * np.tile([1.0, -1.0], nbits)
    n = int(nbits * fs / 1187.5)
    t = np.arange(n, dtype=np.float64) / fs
    k = t * 2375.0
    idx = np.minimum(k.astype(np.int64), chips.size - 1)
    frac = k - idx
    nxt = chips[np.minimum(idx + 1, chips.size - 1)]
    w = np.clip((frac - 0.5) / 0.5, 0.0, 1.0)
    base = chips[idx] + (nxt - chips[idx]) * 0.5 * (1.0 - np.cos(np.pi * w))
    mpx = 0.4 * np.sin(2 * np.pi * 1000 * t) + 0.1 * np.sin(2 * np.pi * 19000 * t) + 0.06 * base * np.sin(2 * np.pi * 57000 * t + 0.4)
    ph = 2 * np.pi * 75000.0 * np.cumsum(mpx) / fs
    x = 0.5 * np.exp(1j * ph) + 0.001 * (rng.uniform(-1, 1, n) + 1j * rng.uniform(-1, 1, n))
    return x.astype(np.complex64), bits
