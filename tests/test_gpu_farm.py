"""-m gpu: receiver-farm contexts (vdl2gpu_create_streams / Vdl2Channels.from_streams).  Every stream carries its own
traffic around its own centre frequency; each stream's channels must equal the oracle run on that stream alone, with
that stream's centre: frames, metadata and counters bit for bit, trace events and decimated samples too."""
import numpy as np
import pytest
import dumpvdl2_b200 as vd
from dumpvdl2_b200 import synth
from oracle import pyoracle as po
from tests import cases, util

pytestmark = pytest.mark.gpu
CENTER = cases.CENTER


def _streams(counts, centres, os, fmt, seconds, seed):
    """[(centre, freqs, iq)]: stream s is traffic on max(count, 1) slots around its own centre, its channels the first
    `count` slots"""
    fs = 105000 * os
    out = []
    for s, (n, c) in enumerate(zip(counts, centres)):
        iq, offs, _ = synth.traffic_stream(fs, seconds, max(n, 1), 8.0, 22.0, -20.0, seed + s, fmt)
        out.append((c, [c + int(o) for o in offs[:n]], iq))
    return out


def _oracles(streams, os, fmt, chunk_bytes, trace=False, dec_tap=False):
    fs = 105000 * os
    code = po.FMT_S16 if fmt == "s16" else po.FMT_U8
    out = []
    for c, fr, iq in streams:
        o = None
        if fr:
            o = po.Oracle(fs, os, code, c, fr, trace=trace, dec_tap=dec_tap)
            o.process_chunked(iq, chunk_bytes)
        out.append(o)
    return out


def _farm(streams, os, fmt, chunk_bytes, flags=0):
    return vd.Vdl2Channels.from_streams(105000 * os, os, vd.FMT_S16 if fmt == "s16" else vd.FMT_U8,
                                        [(c, fr) for c, fr, _ in streams], max_chunk_bytes=chunk_bytes, flags=flags)


def _feed(g, streams, chunk_bytes, device=False):
    """chunk k of every stream, back to back (submit: host buffer; submit_device: one device buffer per chunk)"""
    raw = [np.ascontiguousarray(iq).view(np.uint8).reshape(-1) for _, _, iq in streams]
    n = min(r.size for r in raw)
    keep = []
    for off in range(0, n, chunk_bytes):
        buf = np.concatenate([r[off:off + chunk_bytes] for r in raw])
        if device:
            import torch
            t = torch.from_numpy(buf).cuda()
            keep.append(t)
            g.submit_device(t.data_ptr(), buf.size // len(raw), torch.cuda.current_stream().cuda_stream)
        else:
            g.submit(buf)
    frames = g.flush()
    del keep
    return frames


def _check_against_oracles(g, frames, streams, oracles, what):
    cnt = g.channel_counters()
    st = g.stats()
    assert st["pool_overflows"] == 0 and st["out_overflows"] == 0
    base, total = 0, 0
    for s, ((c, fr, _), o) in enumerate(zip(streams, oracles)):
        n = len(fr)
        assert (g.stream_of_channel[base:base + n] == s).all()
        mine = [f for f in frames if base <= f.channel < base + n]
        for f in mine:
            assert f.freq == fr[f.channel - base]
            f.channel -= base
        if o is not None:
            util.assert_frames_equal(mine, o.frames(), f"{what}: stream {s}")
            assert np.array_equal(cnt[base:base + n], o.counters()), f"{what}: counters of stream {s}"
        total += len(mine)
        base += n
    assert base == g.n_channels
    return total


def test_heterogeneous_layout_cu8_os20():
    """7 streams with 1, 3, 8, 14, 0, 31 and 40 channels on three centre frequencies: warps and K1 blocks straddle
    streams, one stream is empty.  With the trace on (no graphs) and off (graph replay)."""
    counts = [1, 3, 8, 14, 0, 31, 40]
    centres = [CENTER, CENTER + 3000000, CENTER - 2000000, CENTER, CENTER + 3000000, CENTER - 2000000, CENTER + 3000000]
    chunk = 262144
    streams = _streams(counts, centres, 20, "u8", 0.6, 0x56444C60)
    oracles = _oracles(streams, 20, "u8", chunk, trace=True)
    g = _farm(streams, 20, "u8", chunk, flags=vd.FLAG_TRACE)
    assert g.n_streams == 7 and list(g.centerfreqs) == centres
    frames = _feed(g, streams, chunk)
    total = _check_against_oracles(g, frames, streams, oracles, "trace on")
    assert total > 60
    ev = g.read_events()
    base = 0
    for s, ((_, fr, _), o) in enumerate(zip(streams, oracles)):
        mine = [dict(e, channel=e["channel"] - base) for e in ev if base <= e["channel"] < base + len(fr)]
        if o is not None:
            util.assert_events_equal(mine, o.events(), f"events of stream {s}")
        base += len(fr)
    g.close()
    g = _farm(streams, 20, "u8", chunk)
    assert _check_against_oracles(g, _feed(g, streams, chunk), streams, oracles, "graphs") == total
    g.close()


@pytest.mark.parametrize("os, fmt", [(10, "s16"), (13, "s16"), (13, "u8")])
def test_other_rates_and_formats(os, fmt):
    counts = [2, 0, 9, 5, 1]
    centres = [CENTER, CENTER + 1000000, CENTER - 500000, CENTER + 1000000, CENTER]
    chunk = 131072 if fmt == "u8" else 262144
    streams = _streams(counts, centres, os, fmt, 0.8, 0x56444C70 + os)
    oracles = _oracles(streams, os, fmt, chunk)
    g = _farm(streams, os, fmt, chunk)
    assert _check_against_oracles(g, _feed(g, streams, chunk), streams, oracles, f"os {os} {fmt}") > 10
    g.close()


@pytest.mark.parametrize("os, fmt", [(20, "u8"), (10, "s16"), (13, "u8")])
def test_k1_decimated_samples_bit_exact(os, fmt):
    counts = [3, 0, 7, 1, 12]
    centres = [CENTER, CENTER + 2000000, CENTER - 1000000, CENTER, CENTER + 2000000]
    chunk = 100002 if fmt == "u8" else 200004          # odd pair counts: every decimation phase, unaligned segments
    streams = _streams(counts, centres, os, fmt, 0.3, 0x56444C80 + os)
    oracles = _oracles(streams, os, fmt, chunk, dec_tap=True)
    odec = [o.dec_samples() if o is not None else None for o in oracles]
    g = _farm(streams, os, fmt, chunk, flags=vd.FLAG_KEEP_DEC)
    raw = [np.ascontiguousarray(iq).view(np.uint8).reshape(-1) for _, _, iq in streams]
    bpp = 4 if fmt == "s16" else 2
    max_dec = chunk // bpp // os + 2
    pos = 0
    for off in range(0, raw[0].size, chunk):
        g.submit(np.concatenate([r[off:off + chunk] for r in raw]))
        d = g.read_dec(max_dec)
        base = 0
        for s, (_, fr, _) in enumerate(streams):
            if fr:
                want = odec[s][pos:pos + d.shape[0]]
                got = np.ascontiguousarray(d[:, base:base + len(fr)])
                assert got.shape == want.shape
                assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), f"stream {s}: K1 output differs in chunk at byte {off}"
            base += len(fr)
        pos += d.shape[0]
    assert pos == odec[0].shape[0]
    g.flush()
    g.close()


def _collect(g, iqs, chunk):
    """frames, counters and every chunk's decimated samples"""
    n = min(x.size for x in iqs)
    decs = []
    for off in range(0, n, chunk):
        g.submit(np.concatenate([x[off:off + chunk] for x in iqs]))
        decs.append(g.read_dec(chunk // 2 // 20 + 2))
    frames = sorted(g.flush(), key=lambda f: f.key())
    return frames, g.channel_counters(), decs


def _assert_same(a, b, what):
    fa, ca, da = a
    fb, cb, db = b
    util.assert_frames_equal(fa, fb, what)
    assert [f.freq for f in fa] == [f.freq for f in fb]
    assert np.array_equal(ca, cb), what
    assert len(da) == len(db) and all(np.array_equal(x.view(np.uint32), y.view(np.uint32)) for x, y in zip(da, db)), what


def test_uniform_layout_equals_the_independent_streams_mode():
    S, Cn, chunk = 4, 32, 262144
    offs = synth.slot_offsets(Cn, 25e3)
    freqs_one = [CENTER + int(o) for o in offs]
    iqs = [synth.traffic_stream(2100000, 0.5, Cn, 6.0, 22.0, -20.0, 0x56444C90 + s, "u8")[0] for s in range(S)]
    g = vd.Vdl2Channels(2100000, 20, vd.FMT_U8, CENTER, freqs_one * S, max_chunk_bytes=chunk, n_streams=S, flags=vd.FLAG_KEEP_DEC)
    want = _collect(g, iqs, chunk)
    g.close()
    g = vd.Vdl2Channels.from_streams(2100000, 20, vd.FMT_U8, [(CENTER, freqs_one)] * S, max_chunk_bytes=chunk, flags=vd.FLAG_KEEP_DEC)
    got = _collect(g, iqs, chunk)
    g.close()
    assert len(want[0]) > 30
    _assert_same(got, want, "4 x 32 farm vs n_streams = 4")


def test_all_ones_layout_equals_one_stream_per_channel():
    S, chunk = 40, 131072
    base, offs, _ = synth.traffic_stream(2100000, 0.5, 8, 8.0, 24.0, -20.0, 0x56444CA0, "u8")
    iqs = [np.roll(base, 2 * 7919 * s) for s in range(S)]
    freqs = [CENTER + int(offs[s % len(offs)]) for s in range(S)]
    g = vd.Vdl2Channels(2100000, 20, vd.FMT_U8, CENTER, freqs, max_chunk_bytes=chunk, n_streams=S, flags=vd.FLAG_KEEP_DEC)
    want = _collect(g, iqs, chunk)
    g.close()
    g = vd.Vdl2Channels.from_streams(2100000, 20, vd.FMT_U8, [(CENTER, [f]) for f in freqs], max_chunk_bytes=chunk, flags=vd.FLAG_KEEP_DEC)
    got = _collect(g, iqs, chunk)
    g.close()
    assert len(want[0]) > 20
    _assert_same(got, want, "all-ones farm vs one stream per channel")


@pytest.mark.parametrize("chunk", [262144, 65538, 100006])          # 65538 and 100006: len not a multiple of 16 bytes
def test_chunkings_submit_paths_and_graphs(chunk):
    counts = [5, 11, 0, 2, 30]
    centres = [CENTER, CENTER - 1500000, CENTER, CENTER + 2500000, CENTER - 1500000]
    streams = _streams(counts, centres, 20, "u8", 0.5, 0x56444CB0)
    oracles = _oracles(streams, 20, "u8", chunk)
    results = []
    for device in (False, True):
        for flags in (0, vd.FLAG_NO_GRAPH):
            g = _farm(streams, 20, "u8", chunk, flags=flags)
            g.enable_timing(True)
            frames = _feed(g, streams, chunk, device=device)
            total = _check_against_oracles(g, frames, streams, oracles, f"chunk {chunk} device={device} flags={flags}")
            km = g.kernel_ms()
            assert km["K0"][1] == 0 and km["K1"][1] > 0            # no conversion pass: the farm K1 reads the raw bytes
            st = g.stats()
            assert (st["graph_launches"] > 0) == (flags == 0)
            results.append(sorted(util.frame_tuple(f) + (f.sync_dec_index,) for f in frames))
            g.close()
    assert total > 20 and all(r == results[0] for r in results)


def test_balanced_slot_mapping_with_1400_streams():
    """1400 receivers with 4-14 channels each (about 12 600 channels, more than half a machine's worth: dealt over all 592
    warps), three centre frequencies, streams built on the device from one synthetic stream shifted in time and fed
    through submit_device; streams at warp, block and end boundaries are checked against the oracle."""
    import torch
    fs, pairs, n_chunks = 2100000, 65536, 3
    base, offs, _ = synth.traffic_stream(fs, 0.3, 32, 12.0, 24.0, -20.0, 0x56444CC0, "u8")
    rng = np.random.default_rng(0x56444CC1)
    S = 1400
    counts = rng.integers(4, 15, S)
    centres = [CENTER + (0, 2000000, -3000000)[s % 3] for s in range(S)]
    picks = [np.sort(rng.choice(len(offs), int(n), replace=False)) for n in counts]
    layout = [(centres[s], [centres[s] + int(offs[k]) for k in picks[s]]) for s in range(S)]
    n_ch = int(counts.sum())
    assert 9472 < n_ch <= 18944
    L = base.size // 2
    b2 = torch.from_numpy(base[:2 * L].reshape(L, 2)).cuda()
    ar = torch.arange(n_chunks * pairs, device="cuda", dtype=torch.int64)
    raw = torch.empty(n_chunks, S, pairs, 2, dtype=torch.uint8, device="cuda")
    for s0 in range(0, S, 128):
        sh = (torch.arange(s0, min(s0 + 128, S), device="cuda", dtype=torch.int64) * 7919) % L
        blk = b2[(ar[None, :] + sh[:, None]) % L]
        for c in range(n_chunks):
            raw[c, s0:s0 + blk.shape[0]] = blk[:, c * pairs:(c + 1) * pairs]
    g = vd.Vdl2Channels.from_streams(fs, 20, vd.FMT_U8, layout, max_chunk_bytes=2 * pairs)
    st = torch.cuda.current_stream()
    for c in range(n_chunks):
        g.submit_device(raw[c].data_ptr(), 2 * pairs, st.cuda_stream)
    got = {}
    for f in g.flush():
        got.setdefault(f.channel, []).append(f)
    cnt = g.channel_counters()
    stats = g.stats()
    soc = g.stream_of_channel.copy()
    g.close()
    assert stats["pool_overflows"] == 0 and stats["out_overflows"] == 0
    lanes = -(-n_ch // 592)
    first = np.concatenate([[0], np.cumsum(counts)])
    sample = {0, S - 1, int(soc[n_ch // 2])}
    for k in (lanes - 1, lanes, 4 * lanes - 1, 4 * lanes, 8 * lanes, n_ch - 1):      # warp and block boundaries
        sample.add(int(soc[k]))
    checked = 0
    for s in sorted(sample):
        iq = np.roll(base[:2 * L], -2 * ((7919 * s) % L))[:2 * n_chunks * pairs]
        o = po.Oracle(fs, 20, po.FMT_U8, centres[s], layout[s][1])
        o.process_chunked(iq, 2 * pairs)
        mine = []
        for k in range(first[s], first[s + 1]):
            for f in got.get(k, []):
                f.channel = k - first[s]
                mine.append(f)
        util.assert_frames_equal(mine, o.frames(), f"stream {s}")
        assert np.array_equal(cnt[first[s]:first[s + 1]], o.counters())
        checked += len(mine)
    assert checked > 5
