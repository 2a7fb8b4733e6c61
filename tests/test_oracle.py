"""CPU: the oracle restatement against the reference's own fixture and against what the unmodified reference
produced, stored in tests/golden by tests/golden/make_golden.py: its output on the streams of tests/cases.py and
its table literals."""
import hashlib
import numpy as np
import pytest
from oracle import pyoracle as po
from tests import cases, util


@pytest.mark.parametrize("name", list(cases.ALL_GOLDEN))
def test_oracle_matches_reference_golden(name):
    c = cases.ALL_GOLDEN[name]()
    gold = util.load_golden(name)
    assert cases.iq_sha256(c) == gold["iq_sha256"], "stream regenerated from the seed differs from the golden's"
    o = util.run_oracle(c)
    util.assert_matches_golden(o.frames(), gold, "strict", f"oracle vs reference(strict) [{name}]")
    util.assert_matches_golden(o.frames(), gold, "fast", f"oracle vs reference(-ffast-math) [{name}]")


def test_golden_wav_is_the_reference_fixture():
    """SURVEY.md §8c: 1 burst -> 2 frames (314 + 186 octets), both FCS-good, sha256 ee98da53...; the CI of the
    reference greps for the two tails below (.github/workflows/build.yml:17)."""
    c = cases.case_wav()
    assert len(c["raw_bytes"]) == 1582220
    fr = util.run_oracle(c).frames()
    h = "".join(f.data.hex() + "\n" for f in fr)
    assert hashlib.sha256(h.encode()).hexdigest() == "ee98da5344ee2b0167508c2f4e7efc95eb931217ce86b47472a0297c27415477"
    assert [len(f.data) for f in fr] == [314, 186] and all(f.fcs_ok for f in fr)
    assert fr[0].data.endswith(bytes.fromhex("202d5241204252204f56433030350a44bf"))
    assert fr[1].data.endswith(bytes.fromhex("20534c503133350a3ef9"))
    assert fr[0].sync_dec_index == 11975 and fr[0].datalen_octets == 504 and fr[0].num_fec_corrections == 0


def test_chunking_invariance_of_oracle():
    c = cases.case_cfg2(0.4)
    a = util.run_oracle(c, chunk=320000).frames()
    b = util.run_oracle(c, chunk=2 * 9973).frames()
    util.assert_frames_equal(a, b, "oracle chunk 320000 vs 19946")


def test_injected_frames_come_back():
    """generator <-> decoder round trip at high SNR (SURVEY.md §7 step 2)"""
    c = cases.case_cfg2()
    got = {f.data for f in util.run_oracle(c).frames()}
    want = {fr for b in c["bursts"] for fr in b.frames}
    assert want <= got and len(want) == 12


def _oracle_and_reference(name, flavour):
    """the oracle's frames on a stored stream (sorted by key) and the reference's output on it (tests/golden, per
    channel in push order)"""
    c = cases.ORACLE_GOLDEN[name]()
    gold = util.load_golden(name)
    assert cases.iq_sha256(c) == gold["iq_sha256"], "stream regenerated from the seed differs from the golden's"
    return sorted(util.run_oracle(c).frames(), key=lambda f: f.key()), gold[flavour]


@pytest.mark.parametrize("flavour", ["strict", "fast"])
def test_oracle_matches_live_reference_on_replicas(flavour):
    fr, ref = _oracle_and_reference("replicas_8x2", flavour)
    assert len(fr) == len(ref) and len(fr) > 4
    for a, b in zip(fr, ref):
        assert (a.channel, a.idx, a.data.hex()) == (b["channel"], b["idx"], b["hex"])
        if flavour == "strict":     # the -ffast-math build may slice a marginal symbol differently (RS then repairs it)
            assert a.num_fec_corrections == b["num_fec_corrections"]


def test_oracle_matches_live_reference_on_stress_stream():
    """Demodulator-side differential: carrier offsets, clipping / very weak bursts, back-to-back and overlapping
    bursts (cases.case_stress) - frames and printed metadata identical to the strictly compiled reference."""
    fr, ref = _oracle_and_reference("stress", "strict")
    assert len(fr) == len(ref) and len(fr) > 15, (len(fr), len(ref))
    for a, b in zip(fr, ref):
        assert (a.channel, a.idx, a.data.hex(), a.num_fec_corrections, a.synd_weight) == (b["channel"], b["idx"], b["hex"], b["num_fec_corrections"], b["synd_weight"])
        assert abs(a.frame_pwr_dbfs - b["frame_pwr_dbfs"]) < 2e-3 and abs(a.nf_pwr_dbfs - b["nf_pwr_dbfs"]) < 2e-3
        assert abs(a.ppm_error - b["ppm_error"]) < 2e-3


def test_oracle_matches_live_reference_on_fuzzed_payloads():
    """Differential fuzz of the burst decoder against the reference itself (cases.case_fuzz): random-bit payloads and
    stuffed frames cut at a random bit, some with corrupted code words and header bits, decoded by the unmodified
    src/decode.c, bitstream.c, rs.c and by the restatement."""
    fr, ref = _oracle_and_reference("fuzz", "strict")
    assert len(fr) == len(ref) and len(fr) > 20
    for a, b in zip(fr, ref):
        assert (a.channel, a.idx, a.data.hex(), a.num_fec_corrections, a.synd_weight) == (b["channel"], b["idx"], b["hex"], b["num_fec_corrections"], b["synd_weight"])


def test_tables_against_reference_literals():
    """header syndrome weights and error patterns (src/decode.c) and the CRC-16 table (src/crc.c), as stored from the
    reference's literals in tests/golden/ref_tables.json"""
    t = util.load_golden("ref_tables")
    pats, weights, crc_tab = t["syndrome_patterns"], t["synd_weight"], t["crc16_table"]
    assert len(t["syndrome_rows"]) == 5 and len(pats) == 32 and len(weights) == 32 and len(crc_tab) == 256
    import ctypes as C
    L = po.lib()
    for syn in range(32):
        assert L.vo_synd_weight(syn) == weights[syn]
    for bit in range(25):                   # single-bit errors decode back to the clean word
        w = C.c_uint32(po.lib().vo_header_encode(4029) ^ (1 << bit))
        L.vo_header_decode(C.byref(w))
        assert w.value == 0x2f7c0e
    # every syndrome maps to the reference's error pattern
    for pat in pats:
        w = C.c_uint32(pat)
        s = L.vo_header_decode(C.byref(w))
        assert w.value == 0 and pats[s] == pat
    for b in range(256):
        assert po.crc16(bytes([b]), init=0) == crc_tab[b]


def test_rs_codec_properties():
    rng = np.random.default_rng(0)
    for trial in range(300):
        msg = rng.integers(0, 256, 249, dtype=np.uint8)
        cw = po.rs_encode(msg)
        assert po.rs_verify(cw, 6)[0] == 0
        nerr = int(rng.integers(0, 6))
        bad = cw.copy()
        pos = rng.choice(255, nerr, replace=False)
        for p in pos:
            bad[p] ^= int(rng.integers(1, 256))
        ret, fixed = po.rs_verify(bad, 6)
        if nerr <= 3:
            assert ret == nerr and np.array_equal(fixed, cw)
        else:
            assert ret == -1 or not np.array_equal(fixed, cw)      # beyond capacity: failure or miscorrection, never silent success
    # shortened last block: trailing zero fill, untransmitted parity declared erased (src/rs.c:36-47)
    for nfec, nerr_ok in ((4, 2), (2, 1)):
        msg = np.zeros(249, np.uint8); msg[:40] = rng.integers(0, 256, 40, dtype=np.uint8)
        cw = po.rs_encode(msg); rx = cw.copy(); rx[249 + nfec:] = 0
        ret, fixed = po.rs_verify(rx, nfec)
        assert ret == 6 - nfec and np.array_equal(fixed, cw)
        rx[3] ^= 0x40
        if nerr_ok >= 1:
            ret, fixed = po.rs_verify(rx, nfec)
            assert ret == 6 - nfec + 1 and np.array_equal(fixed, cw)


def test_empty_and_ragged_inputs():
    o = po.Oracle(2100000, 20, po.FMT_U8, cases.CENTER, [cases.CENTER + 25000])
    o.process(np.zeros(0, np.uint8))
    o.process(np.full(2 * 7, 128, np.uint8))
    o.process(np.full(2 * 13 + 1, 127, np.uint8))      # trailing unpaired component ignored
    assert o.frames() == [] and o.counters().sum() == 0
