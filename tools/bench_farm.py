#!/usr/bin/env python
"""tools/bench_farm.py — a receiver farm (vdl2gpu_create_streams) against the two ways the n_streams modes can express it.

Shape (default): 2048 receivers x 8 channels = 16384 channels, 262144-pair cu8 chunks.  Receiver s is the bench stream
(bench.make_stream) started 7919 s samples later, tuned to one of three centre frequencies; its 8 channels are its own
pick of the 64 traffic slots, so the lanes of a warp carry different signals.  Streams are built on the GPU and fed with
submit_device: host-to-device bandwidth is not part of the question.  Measured in one process, A-B-A-B:

  farm  Vdl2Channels.from_streams: 2048 streams, 8 channels each, no conversion pass
  A     one stream per channel: every receiver's buffer replicated 8x (16384 streams, n_streams = n_channels)
  B     n_streams = 2048 with C = 32: 24 padding channels per stream (65536 channels, a quarter of them useful)

For each: serial kernel ms per stage (enable_timing, FLAG_NO_OVERLAP), pipelined ms per chunk, USEFUL channel-samples/s
(the 16384 real channels) and channels at real time, and the HBM bytes per chunk the mode has to move up to K1 (computed
from shapes).  Afterwards a fixed sample of the farm's streams (first, last, warp and block boundaries) is checked
against the oracle over the first chunks; any mismatch exits with status 3.

    python tools/bench_farm.py [--streams 2048] [--per-stream 8] [--chunks 6] [--out farm.json]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch
import bench
import dumpvdl2_b200 as vd

CENTRES = (bench.CENTER, bench.CENTER + 2000000, bench.CENTER - 3000000)
PARITY_CHUNKS = 3


def card():
    name = torch.cuda.get_device_name()
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(torch.cuda.current_device())
        return dict(name=name, power_limit_w=pynvml.nvmlDeviceGetPowerManagementLimit(h) / 1000.0)
    except Exception:
        pass
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", str(torch.cuda.current_device())],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return dict(name=name, power_limit_w=float(out))
    except Exception:
        return dict(name=name, power_limit_w=None)


def measure(make, raws, nbytes, chunks):
    """serial stage times (FLAG_NO_OVERLAP) and pipelined ms per chunk of one mode; raws are device buffers fed in turn"""
    stream = torch.cuda.current_stream()
    res = {}
    for overlap in (False, True):
        g = make(0 if overlap else vd.FLAG_NO_OVERLAP)
        for i in range(2):
            g.submit_device(raws[i % len(raws)].data_ptr(), nbytes, stream.cuda_stream)
        g.flush_count()
        if not overlap:
            g.enable_timing(True)
        k0 = g.kernel_ms()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        frames = 0
        for i in range(chunks):
            g.submit_device(raws[i % len(raws)].data_ptr(), nbytes, stream.cuda_stream)
            frames += g.poll_count()
        frames += g.flush_count()
        g.stream_wait(stream.cuda_stream)
        e1.record(stream)
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / chunks
        st = g.stats()
        assert st["pool_overflows"] == 0 and st["out_overflows"] == 0, st
        if overlap:
            res["pipelined_ms_per_chunk"] = ms
            res["frames_per_chunk"] = frames / chunks
        else:
            k1 = g.kernel_ms()
            res["kernel_ms"] = {k: (k1[k][0] - k0[k][0]) / max(k1[k][1] - k0[k][1], 1) for k in k1}
            res["kernel_launches"] = {k: k1[k][1] - k0[k][1] for k in k1}
            res["serial_ms_per_chunk"] = ms
        g.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=2048)
    ap.add_argument("--per-stream", type=int, default=8)
    ap.add_argument("--chunks", type=int, default=6)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--chunk-pairs", type=int, default=bench.CHUNK_PAIRS)
    ap.add_argument("--out")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_farm.py needs a CUDA device")
    S, C, P = a.streams, a.per_stream, a.chunk_pairs
    n_ch, nbytes, pad_c = S * C, 2 * P, -(-C // 32) * 32
    chunks, offs, _ = bench.make_stream(2.0)
    base = torch.from_numpy(chunks.reshape(-1)).cuda()
    L = base.numel() // 2
    base2 = base.view(L, 2)
    rng = np.random.default_rng(0x56444C33)
    picks = [np.sort(rng.choice(len(offs), C, replace=False)) for _ in range(S)]
    centres = [CENTRES[s % 3] for s in range(S)]
    layout = [(centres[s], [centres[s] + int(offs[k]) for k in picks[s]]) for s in range(S)]
    # receiver s = the bench stream started 7919 s samples later (wrapping); PARITY_CHUNKS consecutive chunks of it
    raw = torch.empty(PARITY_CHUNKS, S, P, 2, dtype=torch.uint8, device="cuda")
    ar = torch.arange(PARITY_CHUNKS * P, device="cuda", dtype=torch.int64)
    for s0 in range(0, S, 64):
        sh = (torch.arange(s0, min(s0 + 64, S), device="cuda", dtype=torch.int64) * 7919) % L
        blk = base2[(ar[None, :] + sh[:, None]) % L]
        for c in range(PARITY_CHUNKS):
            raw[c, s0:s0 + blk.shape[0]] = blk[:, c * P:(c + 1) * P]
    del blk
    torch.cuda.synchronize()
    farm_raws = [raw[c] for c in range(PARITY_CHUNKS)]
    # the workarounds express every receiver with the common centre: channel offsets from the centre are what K1 sees
    rel = [[bench.CENTER + int(offs[k]) for k in picks[s]] for s in range(S)]
    freqs_a = np.array([f for r in rel for f in r], np.uint32)
    pad = [[bench.CENTER + int(offs[k]) for k in range(len(offs)) if k not in set(picks[s])][:pad_c - C] for s in range(S)]
    freqs_b = np.array([f for s in range(S) for f in rel[s] + pad[s]], np.uint32)

    def make_farm(flags):
        return vd.Vdl2Channels.from_streams(bench.FS, 20, vd.FMT_U8, layout, max_chunk_bytes=nbytes, flags=flags)

    def make_a(flags):
        return vd.Vdl2Channels(bench.FS, 20, vd.FMT_U8, bench.CENTER, freqs_a, max_chunk_bytes=nbytes, n_streams=n_ch, flags=flags)

    def make_b(flags):
        return vd.Vdl2Channels(bench.FS, 20, vd.FMT_U8, bench.CENTER, freqs_b, max_chunk_bytes=nbytes, n_streams=S, flags=flags)

    modes = dict(farm=(make_farm, farm_raws, n_ch), A=(make_a, None, n_ch), B=(make_b, farm_raws[:1], S * pad_c))
    rounds = {k: [] for k in modes}
    for r in range(a.rounds):
        for name, (make, raws, _) in modes.items():
            if name == "A":
                raws = [raw[0].repeat_interleave(C, dim=0)]           # every receiver's buffer once per channel
            rounds[name].append(measure(make, raws, nbytes, a.chunks))
            del raws
            torch.cuda.empty_cache()
    dec_bytes = lambda ch: ch * (P // 20) * 8
    hbm = dict(farm=dict(k1_raw_read=S * P * 2, dec_write=dec_bytes(n_ch)),
               A=dict(k0_raw_read=n_ch * P * 2, k0_plane_write=n_ch * P * 8, k1_plane_read=n_ch * P * 8, dec_write=dec_bytes(n_ch)),
               B=dict(k0_raw_read=S * P * 2, k0_plane_write=S * P * 8, k1_plane_read=S * P * 8, dec_write=dec_bytes(S * pad_c)))
    res = dict(card=card(), streams=S, channels_per_stream=C, useful_channels=n_ch, chunk_pairs=P, sample_fmt="cu8", chunks_timed=a.chunks,
               order=" -> ".join(list(modes) * a.rounds), modes={})
    for name, (_, _, total_ch) in modes.items():
        rr = rounds[name]
        ms = float(np.median([x["pipelined_ms_per_chunk"] for x in rr]))
        useful = n_ch * P / (ms * 1e-3)
        res["modes"][name] = dict(channels_total=total_ch, rounds=rr, pipelined_ms_per_chunk=ms, useful_channel_samples_per_s=useful,
                                  useful_channels_at_realtime=useful / bench.FS,
                                  hbm_bytes_per_chunk=dict(hbm[name], total=sum(hbm[name].values())))
    res["hbm_note"] = "bytes each mode must move per chunk up to and including K1's output, computed from shapes (not measured)"
    # ---- parity: a fixed sample of farm streams against the oracle over PARITY_CHUNKS chunks ----
    from oracle import pyoracle as po
    g = make_farm(0)
    stream = torch.cuda.current_stream()
    for c in range(PARITY_CHUNKS):
        g.submit_device(farm_raws[c].data_ptr(), nbytes, stream.cuda_stream)
    by = {}
    for f in g.flush():
        by.setdefault(f.channel, []).append(f)
    cnt = g.channel_counters()
    soc = g.stream_of_channel.copy()
    g.close()
    wa = 4 * torch.cuda.get_device_properties(0).multi_processor_count              # the slot mapping of create_impl
    lanes = -(-n_ch // wa) if 16 * wa < n_ch <= 32 * wa else 32
    sample = {0, S - 1, S // 2}
    for k in (lanes - 1, lanes, 4 * lanes - 1, 4 * lanes, 40 * lanes, n_ch - 1):
        if 0 <= k < n_ch:
            sample.add(int(soc[k]))
    base_np = chunks.reshape(-1)[:2 * L]
    mism, frames_checked = 0, 0
    for s in sorted(sample):
        iq = np.roll(base_np, -2 * ((7919 * s) % L))[:2 * PARITY_CHUNKS * P]
        o = po.Oracle(bench.FS, 20, po.FMT_U8, centres[s], layout[s][1])
        o.process_chunked(iq, nbytes)
        oby = {}
        for f in o.frames():
            oby.setdefault(f.channel, []).append(f)
        ocnt = o.counters()
        for i in range(C):
            k = s * C + i
            mine = by.get(k, [])
            frames_checked += len(mine)
            if bench.digest_frames(mine, cnt[k]) != bench.digest_frames(oby.get(i, []), ocnt[i]):
                mism += 1
    res["parity"] = dict(streams_checked=sorted(sample), channels_checked=len(sample) * C, frames_checked=frames_checked, mismatches=mism,
                         seconds=PARITY_CHUNKS * P / bench.FS,
                         what="per-channel (burst, idx, frame octets, FEC corrections, syndrome weight) lists + 9 counters vs the oracle run on that stream alone")
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt + "\n")
    if mism:
        sys.exit(3)


if __name__ == "__main__":
    main()
