"""Deterministic test streams shared by tests/golden/make_golden.py (which runs the unmodified reference on
them, in the build container) and by the parity tests (which regenerate them from the seed anywhere).

Every case is a dict: name, fs, oversample, fmt ('u8'|'s16'), centerfreq, freqs, chunk (bytes) and iq (numpy
array of uint8 / int16, interleaved I,Q).  Shapes follow BASELINE.json configs / SURVEY.md §8(d), scaled so
that the CPU oracle finishes in seconds.
"""
import hashlib
import lzma
import os
import numpy as np
from dumpvdl2_b200 import synth

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden")
CENTER = 136975000


def _mk(name, fs, fmt, freqs, iq, chunk=320000, bursts=None, centerfreq=CENTER, max_ppm=0.0):
    return dict(name=name, fs=fs, oversample=fs // 105000, fmt=fmt, centerfreq=centerfreq,
                freqs=[int(f) for f in freqs], iq=iq, chunk=chunk, bursts=bursts or [], max_ppm=max_ppm)


def iq_sha256(case):
    return hashlib.sha256(np.ascontiguousarray(case["iq"]).view(np.uint8).tobytes()).hexdigest()


def case_wav():
    """BASELINE config 1: the reference's own fixture, whole file incl. the 44-byte RIFF header fed as samples
    (src/dumpvdl2.c:353-356 does not skip it), S16_LE, oversample 10, one channel on the centre frequency."""
    raw = lzma.decompress(open(os.path.join(GOLDEN, "vdl2_model_16b_1050kHz.wav.xz"), "rb").read())
    iq = np.frombuffer(raw[:len(raw) // 2 * 2], dtype="<i2").copy()
    c = _mk("wav", 1050000, "s16", [CENTER], iq)
    c["raw_bytes"] = raw
    return c


def case_cfg2(duration=1.0):
    """BASELINE config 2: 2.1 Msps cu8, 8 offset-tuned channels, one burst each, Es/N0 30 dB, -10 dBFS."""
    fs = 2100000
    offs = [-100e3, -75e3, -50e3, -25e3, 25e3, 50e3, 75e3, 100e3]
    rng = np.random.default_rng(0x56444C32)
    bursts = [synth.BurstSpec(0.05 + 0.1 * i, offs[i], synth.random_frames(rng), power_dbfs=-10.0) for i in range(8)]
    iq = synth.synth_stream(fs, duration, bursts, es_n0_db=30, fmt="u8", seed=0x56444C32)
    return _mk("cfg2", fs, "u8", [CENTER + o for o in offs], iq, bursts=bursts)


def case_mixed_s16():
    """cs16 at 1.05 Msps (oversample 10): centre channel + 4 offset channels, two bursts per channel,
    small carrier offsets, odd chunk size (not a multiple of the oversample factor)."""
    fs = 1050000
    offs = [0.0, -50e3, 25e3, 150e3, -200e3]
    rng = np.random.default_rng(77)
    bursts = []
    for i, o in enumerate(offs):
        for k in range(2):
            bursts.append(synth.BurstSpec(0.01 + 0.03 * i + 0.2 * k, o, synth.random_frames(rng, lo=11, hi=300),
                                          power_dbfs=-14.0, freq_err_hz=float(rng.uniform(-300, 300))))
    iq = synth.synth_stream(fs, 0.45, bursts, es_n0_db=22, fmt="s16", seed=78)
    return _mk("mixed_s16", fs, "s16", [CENTER + o for o in offs], iq, chunk=4 * 33331, bursts=bursts)


def case_mirics_os13():
    """1.365 Msps cs16 (Mirics front-end rate, src/mirics.h:23: oversample 13): a decimation factor without a
    specialised K1, i.e. the generic per-sample kernel in production use; centre channel + offsets, odd chunks."""
    fs = 1365000
    offs = [0.0, -125e3, 100e3, 300e3]
    rng = np.random.default_rng(1365)
    bursts = []
    for i, o in enumerate(offs):
        for k in range(2):
            bursts.append(synth.BurstSpec(0.015 + 0.05 * i + 0.22 * k, o, synth.random_frames(rng), power_dbfs=-13.0,
                                          freq_err_hz=float(rng.uniform(-200, 200))))
    iq = synth.synth_stream(fs, 0.5, bursts, es_n0_db=26, fmt="s16", seed=1366)
    return _mk("mirics_os13", fs, "s16", [CENTER + o for o in offs], iq, chunk=4 * 50001, bursts=bursts)


def case_fec():
    """RS error correction, header bit errors, multi-block and short-last-block bursts (paths no reference
    fixture pins; pinned here by running the reference itself)."""
    fs = 2100000
    offs = [-75e3 * k for k in range(-4, 5) if k != 0]
    rng = np.random.default_rng(4242)
    specs = [
        dict(frames=[synth.random_avlc_frame(rng, 600)], corrupt=[(0, 3, 0x55), (1, 100, 0x01), (2, 7, 0xFF)]),      # 3 blocks, 1 err each
        dict(frames=[synth.random_avlc_frame(rng, 255)], corrupt=[(0, 10, 1), (0, 20, 2), (0, 30, 4)]),              # 3 errors in a full block (t=3)
        dict(frames=[synth.random_avlc_frame(rng, 245)], corrupt=[(0, 1, 9), (0, 2, 9), (0, 3, 9), (0, 4, 9)]),      # 4 errors: uncorrectable
        dict(frames=[synth.random_avlc_frame(rng, 20)], corrupt=[(0, 5, 0x80)]),                                     # short block, 2 parity octets
        dict(frames=[synth.random_avlc_frame(rng, 60)], corrupt=[(0, 0, 0x11)], hdr=(7,)),                           # 4 parity octets + header bit error
        dict(frames=[synth.random_avlc_frame(rng, 11), synth.random_avlc_frame(rng, 11), synth.random_avlc_frame(rng, 40)], hdr=(24,)),
        dict(frames=[synth.random_avlc_frame(rng, 249 * 2 - 3)], corrupt=[(1, 248, 3)]),                             # last block exactly ... see test
        dict(frames=[synth.random_avlc_frame(rng, 1200)], corrupt=[(0, 0, 1), (4, 200, 0x7e)]),
    ]
    bursts, t = [], 0.02
    for i, sp in enumerate(specs):                      # one after the other: no adjacent-channel overlap
        b = synth.BurstSpec(t, offs[i], sp["frames"], power_dbfs=-12.0, corrupt_octets=sp.get("corrupt"),
                            header_bit_errors=sp.get("hdr", ()))
        bursts.append(b)
        t += synth.burst_duration_s(sp["frames"]) + 0.012
    iq = synth.synth_stream(fs, t + 0.02, bursts, es_n0_db=32, fmt="u8", seed=4243)
    return _mk("fec", fs, "u8", [CENTER + o for o in offs], iq, bursts=bursts)


def case_hdlc_edge():
    """Crafted payloads (src/bitstream.c:109-150 corner cases, pinned by running the reference itself): repeated
    flags, back-to-back flags, abort (seven ones), a frame that is not a whole number of octets after a good one,
    a missing closing flag, trailing bits after the last flag, frames shorter than an AVLC header."""
    fs = 2100000
    rng = np.random.default_rng(31337)
    F = "01111110"

    def st(n):
        return "".join(format(b, "08b")[::-1] for b in rng.integers(0, 256, n, dtype=np.uint8)).replace("11111", "111110")

    def fr(n):
        return "".join(format(b, "08b")[::-1] for b in synth.random_avlc_frame(rng, n)).replace("11111", "111110")
    payloads = [
        F + F + F + fr(40) + F,                          # repeated opening flags
        F + fr(30) + F + F + fr(25) + F,                 # back-to-back flags between frames
        F + fr(30) + F + st(10) + "1111111" + st(4) + F, # abort in the second frame: the first stays pushed
        F + fr(22) + F + st(9) + "010" + F,              # second frame not octet aligned
        F + fr(50),                                      # no closing flag
        F + fr(35) + F + "0101",                         # trailing bits after the closing flag
        F + st(3) + F + st(1) + F + fr(20) + F,          # frames shorter than an AVLC header
        F + fr(270) + F + fr(260) + F,                   # three RS blocks
        "0110" + F + fr(20) + F,                         # garbage before the opening flag (< 7 bits: error)
        F + fr(12) + F + F,                              # trailing flag: zero-length last frame
    ]
    offs = [75e3 * k for k in range(-5, 6) if k != 0]
    bursts, t = [], 0.02
    for i, pl in enumerate(payloads):
        bursts.append(synth.BurstSpec(t, offs[i], [], power_dbfs=-12.0, payload=pl))
        t += synth.burst_duration_s(None, payload=pl) + 0.012
    iq = synth.synth_stream(fs, t + 0.02, bursts, es_n0_db=32, fmt="u8", seed=31338)
    return _mk("hdlc_edge", fs, "u8", [CENTER + o for o in offs], iq, bursts=bursts)


def case_maxlen():
    """Size corners of src/decode.c:45-48,124-133,222-297 on the air: the longest transmission the header can carry
    within the reference's limit (2047 octets, 9 RS blocks, 54 FEC octets), a burst whose last block is full
    (3 x 249 octets) and one whose last block is too short to carry FEC octets (249 + 2)."""
    fs = 2100000
    rng = np.random.default_rng(2047)
    F = "01111110"

    def fr(n):
        return "".join(format(b, "08b")[::-1] for b in synth.random_avlc_frame(rng, n)).replace("11111", "111110")

    def fill(frames, n_octets):
        pl = F + F.join(fr(n) for n in frames) + F
        assert len(pl) <= 8 * n_octets
        return (pl + F * 64)[:8 * n_octets]              # pad with flags up to the exact transmission length
    payloads = [(fill([240] * 8, 2047), 100e3), (fill([240, 240, 230], 747), -100e3), (fill([235], 251), -100e3)]
    bursts, t = [], {100e3: 0.02, -100e3: 0.02}
    for pl, off in payloads:
        bursts.append(synth.BurstSpec(t[off], off, [], power_dbfs=-12.0, payload=pl))
        t[off] += synth.burst_duration_s(None, payload=pl) + 0.015
    iq = synth.synth_stream(fs, max(t.values()) + 0.02, bursts, es_n0_db=32, fmt="u8", seed=2048)
    return _mk("maxlen", fs, "u8", [CENTER + 100e3, CENTER - 100e3], iq, chunk=524288, bursts=bursts)


def case_stress():
    """Impairments the goldens do not carry (CPU-only differential case, not a golden): carrier offsets up to
    +-900 Hz (beyond and within the sync range), powers from -45 dBFS to clipping, bursts following each other
    after 0.3-2 ms (the sample after a burst, the 150 samples after a reset), two bursts overlapping on one
    channel, cu8 quantisation at low level."""
    fs = 2100000
    offs = [-150e3, -75e3, 50e3, 125e3, 300e3, -425e3]
    rng = np.random.default_rng(4711)
    bursts = []
    for i, o in enumerate(offs):
        t = 0.005 + 0.003 * i
        for k in range(5):
            fr = synth.random_frames(rng, lo=11, hi=120)
            pw = float(rng.choice([-45.0, -30.0, -18.0, -9.0, -2.0, 1.5]))
            bursts.append(synth.BurstSpec(t, o, fr, power_dbfs=pw, freq_err_hz=float(rng.uniform(-900, 900))))
            gap = float(rng.choice([0.0003, 0.001, 0.002, 0.015]))
            t += synth.burst_duration_s(fr) + gap
            if k == 3 and i % 2 == 0:
                t -= 0.004                                # the next burst starts before this one has ended
    iq = synth.synth_stream(fs, 0.6, bursts, noise_power=10 ** (-38 / 10), fmt="u8", seed=4712)
    return _mk("stress", fs, "u8", [CENTER + o for o in offs], iq, chunk=2 * 77777, bursts=bursts)


def case_noisy():
    """Low SNR (Es/N0 19.5 dB): symbol errors, RS corrections and failures, false syncs on noise."""
    fs = 2100000
    offs = [50e3 * k for k in range(-4, 5) if k != 0]
    rng = np.random.default_rng(99)
    bursts = []
    for i, o in enumerate(offs):
        for k in range(3):
            bursts.append(synth.BurstSpec(0.01 + 0.02 * i + 0.22 * k, o, synth.random_frames(rng), power_dbfs=-16.0))
    iq = synth.synth_stream(fs, 0.7, bursts, es_n0_db=19.5, fmt="u8", seed=100)
    return _mk("noisy", fs, "u8", [CENTER + o for o in offs], iq, bursts=bursts)


def case_replicas(n_slots=16, n_rep=4, duration=0.5, seed=0x56444C33, es_n0_db=20, rate_hz=6.0):
    """BASELINE config 3 shape (scaled): n_slots 25 kHz slots x n_rep replicas, Poisson bursts per slot."""
    fs = 2100000
    slots = [25e3 * (k - n_slots // 2) for k in range(n_slots)]
    slots = [s if s != 0 else 25e3 * (n_slots // 2) for s in slots]
    rng = np.random.default_rng(seed)
    bursts = []
    for s in slots:
        t = float(rng.exponential(1.0 / rate_hz))
        while t < duration - 0.12:
            bursts.append(synth.BurstSpec(t, s, synth.random_frames(rng), power_dbfs=-20.0))
            t += 0.12 + float(rng.exponential(1.0 / rate_hz))
    iq = synth.synth_stream(fs, duration, bursts, es_n0_db=es_n0_db, fmt="u8", seed=seed + 1)
    freqs = [CENTER + s for s in slots for _ in range(n_rep)]
    return _mk(f"replicas_{n_slots}x{n_rep}", fs, "u8", freqs, iq, chunk=524288, bursts=bursts)


def case_fuzz():
    """Differential fuzz of the burst decoder: transmissions whose payloads are random bits, or stuffed frames cut at a
    random bit, some with corrupted code words and header bits, on two channels."""
    rng = np.random.default_rng(0x7E7E)
    F = "01111110"

    def stuffed(n):
        return "".join(format(b, "08b")[::-1] for b in rng.integers(0, 256, n, dtype=np.uint8)).replace("11111", "111110")
    fs, offs = 2100000, [100e3, -100e3]
    bursts, t = [], [0.02, 0.02]
    for k in range(18):
        nbits = int(rng.integers(40, 5000))
        if k % 3 == 0:
            pl = "".join("01"[b] for b in rng.integers(0, 2, nbits, dtype=np.uint8))
        else:
            pl = F
            while len(pl) < nbits:
                pl += stuffed(int(rng.integers(0, 200))) + F * int(rng.integers(1, 3))
            if k % 3 == 1:
                pl = pl[:nbits]
        n_oct = -(-len(pl) // 8)
        nblk = -(-n_oct // 249)
        corrupt = [(int(rng.integers(0, nblk)), int(rng.integers(0, min(249, n_oct - (nblk - 1) * 249))), int(rng.integers(1, 256)))
                   for _ in range(int(rng.integers(0, 5)) if k % 2 else 0)]
        hdr = (int(rng.integers(0, 25)),) if k % 5 == 4 else ()
        ch = k % 2
        try:
            synth.burst_bits_from_payload(pl, corrupt)
        except ValueError:
            continue
        bursts.append(synth.BurstSpec(t[ch], offs[ch], [], power_dbfs=-12.0, payload=pl, corrupt_octets=corrupt, header_bit_errors=hdr))
        t[ch] += synth.burst_duration_s(None, payload=pl) + 0.012
    iq = synth.synth_stream(fs, max(t) + 0.02, bursts, es_n0_db=32, fmt="u8", seed=0x7E7F)
    return _mk("fuzz", fs, "u8", [CENTER + o for o in offs], iq, chunk=524288, bursts=bursts)


ALL_GOLDEN = {"wav": case_wav, "cfg2": case_cfg2, "mixed_s16": case_mixed_s16, "fec": case_fec, "noisy": case_noisy,
              "hdlc_edge": case_hdlc_edge, "mirics_os13": case_mirics_os13, "maxlen": case_maxlen}
# streams whose reference output is stored too, but which only the CPU oracle is compared with (test_oracle.py)
ORACLE_GOLDEN = {"replicas_8x2": lambda: case_replicas(n_slots=8, n_rep=2, duration=0.4), "stress": case_stress, "fuzz": case_fuzz}
